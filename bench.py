#!/usr/bin/env python
"""bench.py — boosting-iteration throughput of the B200-native hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W [--impl reference]

Workload (config.workload): one GBMRegressor boosting iteration, squared loss, on N_rows x 128 fp32
synthetic rows per GPU (default 100 M x 128, the configuration the metric is quoted on):
    line search  (Brent, commons-math3 semantics, over the one-pass sufficient statistics  — K2, 8 B/row:
                  the residual r = y - F left by the previous fused update, and h)
  + F += lr*alpha*h fused with next-round pseudo-residuals and train loss                  — K1, 20 B/row
i.e. regression/GBMRegressor.scala:398-442 + :368-385 of the reference, per round.
`value`  = rows/s with y, F, h (and the 128-column feature matrix) resident in HBM.
`e2e`    = the same round through the host-side mirror with HOST (pinned) buffers: the direction h is
           copied host->device and the pseudo-residuals device->host inside the timed region.
`roofline` is for the dominant kernel K1 (fused update+residual+loss), timed with CUDA events on the
library's own stream, against MEASURED_PEAKS.json's HBM copy bandwidth.
`extras.strong_scaling`: the SAME round on a fixed GLOBAL dataset (--strong-rows, default 100 M rows) split over
the ranks (12.5 M rows per GPU at N=8), measured in the same run after the weak-scaling figure; `extras.strong_c3`:
BASELINE config 3 (bernoulli, 50 M rows global, Brent line search + update per round) split the same way.
`parity_ok` / `parity`: after all timed regions every rank downloads its shard, runs one more round on the GPU
and the fp64 CPU oracle (checker only) on the same data; the GPU's GLOBAL alpha / Σloss (summed across GPUs inside
the kernels) are compared with the oracle's sums all-reduced over torch.distributed, F / r row by row (1e-5).
`cpu_baseline` / `--impl reference`: the reference algorithm's CPU restatement (oracle/, OpenMP, fp64:
one full pass per Brent evaluation as RDDLossFunction does) on the host cores, bounded sample.
The reference itself is Scala/Spark and cannot run here (no JVM): kind = "port".
`--dump-outputs DIR`: after the timed steps, rank 0 writes what the last timed round returned (see dump_outputs) as
DIR/<name>.npy; the inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import atexit
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "boosting-iter rows/sec (grad+update)"
BYTES_K1 = 20  # y,F,h read + F',r written, fp32 (SURVEY.md §8d)
BYTES_K2 = 8   # squared-loss statistics read the current residual r = y - F and h (12 when r is stale: y,F,h)
BYTES_ROUND = BYTES_K1 + BYTES_K2  # the one-launch round runs both passes inside one kernel


def _ncu_traffic(rows: int, bytes_per_row: int):
    """DRAM bytes per launch of the roofline kernel from the committed `ncu --set full` capture (profiles/), if it
    was taken at this row count for this kernel."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        d = json.load(open(p))
        key = "fused_round" if bytes_per_row == BYTES_ROUND else "k1"
        if int(d[key]["rows"]) == int(rows):
            return float(d[key]["dram_bytes_per_launch"])
    except Exception:
        pass
    return None


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu, self.proc, self.path = gpu_index, None, None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "200"], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
            atexit.register(self.proc.kill)  # nvidia-smi -lms never exits by itself: not even when bench.py fails
        except Exception:
            self.proc = None

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.path):
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        os.unlink(self.path)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def _pinned_array(n: int):
    """float32[n] over page-locked memory from the library (se_host_alloc)."""
    import ctypes as C
    from spark_ensemble_b200 import _native as N
    lib = N.load()
    p = C.c_void_p()
    N.check(lib.se_host_alloc(4 * n, C.byref(p)))
    buf = (C.c_float * n).from_address(p.value)
    arr = np.frombuffer(buf, dtype=np.float32)
    return arr, p


# ------------------------------------------------------------------ CPU arm (oracle port)
def cpu_reference_round(orc, y, F, h, r_buf, lr=0.1, tol=1e-6, max_iter=100):
    """One reference round on the CPU: Brent with a full pass per evaluation (GBMLoss.scala:50-74 via
    RDDLossFunction), F update, next pseudo-residuals, mean loss."""
    from oracle import oracle as O
    f = lambda a: orc.linesearch_eval(O.SQUARED, 0.0, y, None, F, h, [a])[0]
    alpha, n_eval, _ = orc.brent(f, 0.0, 100.0, 1.0, tol, tol, max_iter)
    orc.update(F, h, [lr * alpha])
    orc.pseudo_residuals(O.SQUARED, 0.0, 1, y, None, F, False, out_r=r_buf, want_weights=False)
    orc.mean_loss(O.SQUARED, 0.0, 1, y, F)
    return alpha, n_eval


def _usable_cpus() -> int:
    """CPUs this process may actually use: affinity mask capped by the cgroup CPU quota (a container can
    see 128 cores and be allowed 16; oversubscribed OpenMP spin-waits are then catastrophically slow)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period) + 0.5)))
    except Exception:
        pass
    return n


def run_cpu_arm(sample_rows: int, steps: int, warmup: int) -> dict:
    from oracle import oracle as O
    from oracle.oracle import Oracle
    orc = Oracle(omp=True)
    rng = np.random.default_rng(1)
    y = rng.standard_normal(sample_rows)
    F = np.zeros((1, sample_rows))
    h = (0.5 * y + 0.5 * rng.standard_normal(sample_rows)).reshape(1, -1)
    r_buf = np.zeros((1, sample_rows))
    # "all the host threads it can use": pick the fastest thread count among powers of two up to the
    # usable CPUs, measured on one line-search evaluation (memory-bound: more threads is not always faster)
    cap = _usable_cpus()
    cands = sorted({c for c in (1, 2, 4, 8, 16, 32, 64, 128, 256, cap) if c <= cap})
    best_t, best_dt = cands[0], float("inf")
    for t in cands:
        orc.lib.orc_set_num_threads(t)
        orc.linesearch_eval(O.SQUARED, 0.0, y, None, F, h, [1.0])
        dt = float("inf")
        for _ in range(3):
            t0 = time.perf_counter()
            orc.linesearch_eval(O.SQUARED, 0.0, y, None, F, h, [1.0])
            dt = min(dt, time.perf_counter() - t0)
        if dt < best_dt:
            best_t, best_dt = t, dt
    orc.lib.orc_set_num_threads(best_t)
    evals = []
    for _ in range(warmup):
        cpu_reference_round(orc, y, F, h, r_buf)
    t0 = time.perf_counter()
    for _ in range(steps):
        _, ne = cpu_reference_round(orc, y, F, h, r_buf)
        evals.append(ne)
    dt = time.perf_counter() - t0
    return {"value": sample_rows * steps / dt, "ms_per_step": 1e3 * dt / steps, "cores": best_t,
            "usable_cpus": cap, "brent_evals_per_round": float(np.mean(evals)), "sample_rows": sample_rows}


# ------------------------------------------------------------------ self-check against the oracle (checker only)
def parity_check(ctx, n, lr, tol, max_iter, world, rank, dist, label):
    """One extra round on the current device state, replayed by the fp64 oracle on this rank's shard; the
    line-search objective is summed over ALL ranks' shards through torch.distributed (an independent channel), so
    the GPU's global alpha / Σloss (in-kernel cross-GPU sums) are checked against the concatenated data."""
    from oracle import oracle as O
    from oracle.oracle import Oracle
    from spark_ensemble_b200 import _native as N
    t_start = time.perf_counter()
    orc = Oracle(omp=True)
    orc.lib.orc_set_num_threads(max(1, _usable_cpus() // max(world, 1)))
    y32 = ctx.download(N.SLOT_Y)[:n]
    F32 = ctx.download(N.SLOT_F)[:n]
    h32 = ctx.download(N.SLOT_H)[:n]
    alpha_g, loss_g, ne_g = ctx.gbm_round(lr, True, tol, max_iter, residual=True)
    fused = int(ctx.get_option("last_round_fused"))
    Fg = ctx.download(N.SLOT_F)[:n]
    rg = ctx.download(N.SLOT_R)[:n]
    y = y32.astype(np.float64); F = F32.astype(np.float64).reshape(1, -1); h = h32.astype(np.float64).reshape(1, -1)

    def allsum(vals):
        v = np.asarray(vals, dtype=np.float64)
        if dist is None:
            return v
        import torch
        t = torch.tensor(v, dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return t.cpu().numpy()

    n_glob = float(allsum([n])[0])

    def objective(a):  # RDDLossFunction over the concatenated shards: Σ lossSum / Σ weightSum (GBMLoss.scala:50-74)
        l_local = orc.linesearch_eval(O.SQUARED, 0.0, y, None, F, h, [a])[0] * n
        return float(allsum([l_local])[0]) / n_glob

    alpha_o, ne_o, st = orc.brent(objective, 0.0, 100.0, 1.0, tol, tol, max_iter)
    orc.update(F, h, [lr * alpha_g])  # the GPU's step: row-level parity is not blurred by the optimiser tolerance
    loss_o = float(allsum([orc.mean_loss(O.SQUARED, 0.0, 1, y, F) * n])[0])
    r_o, _, _ = orc.pseudo_residuals(O.SQUARED, 0.0, 1, y, None, F, False, want_weights=False)
    f_scale = max(1.0, float(np.abs(F).max()))
    r_scale = max(1.0, float(np.abs(r_o).max()))
    f_err = float(np.max(np.abs(Fg - F[0]))) / f_scale
    r_err = float(np.max(np.abs(rg - r_o[0]))) / r_scale
    if dist is not None:
        import torch
        t = torch.tensor([f_err, r_err], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        f_err, r_err = float(t[0]), float(t[1])
    a_err = abs(alpha_g - alpha_o)
    l_err = abs(loss_g - loss_o) / abs(loss_o)
    ok = bool(st == 0 and a_err <= 1e-5 * max(abs(alpha_o), 1e-3) + 4 * tol and l_err <= 1e-5 and f_err <= 1e-5
              and r_err <= 1e-5)
    return {"case": label, "ok": ok, "rows_global": int(n_glob), "rows_per_gpu": int(n), "fused_round": fused,
            "alpha_gpu": alpha_g, "alpha_oracle": alpha_o, "brent_evals_gpu": ne_g, "brent_evals_oracle": ne_o,
            "loss_sum_gpu": loss_g, "loss_sum_oracle": loss_o, "loss_rel_err": l_err, "F_max_rel_err": f_err,
            "r_max_rel_err": r_err, "tolerance": 1e-5, "seconds": time.perf_counter() - t_start}


# ------------------------------------------------------------------ --dump-outputs
DUMP_ROWS = 1 << 21  # sampled rows: F and r in fp32 + the row indices in fp64 = 32 MB


def dump_outputs(out_dir, ctx, n, alpha, loss_sum, n_eval):
    """What a caller of the timed round receives after the last timed step: the line-search minimiser alpha, the train
    loss sum and the number of Brent evaluations, and the round's per-row outputs — the updated predictions F and the
    next pseudo-residuals r — over every row, or over a fixed seeded sample of DUMP_ROWS rows (`row_index`) when
    there are more."""
    from spark_ensemble_b200 import _native as N
    idx = np.arange(n) if n <= DUMP_ROWS else np.sort(np.random.default_rng(0).choice(n, DUMP_ROWS, replace=False))
    out = {"alpha": np.array([alpha]), "loss_sum": np.array([loss_sum]), "brent_evals": np.array([float(n_eval)]),
           "row_index": idx.astype(np.float64),
           "F": ctx.download(N.SLOT_F)[:n][idx], "r": ctx.download(N.SLOT_R)[:n][idx]}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ------------------------------------------------------------------ main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rows", type=int, default=int(os.environ.get("SE_BENCH_ROWS", 100_000_000)),
                    help="rows per GPU (weak scaling)")
    ap.add_argument("--features", type=int, default=128)
    ap.add_argument("--cpu-rows", type=int, default=16_000_000, help="bounded CPU sample per step")
    ap.add_argument("--no-features", action="store_true", help="do not materialise the feature matrix")
    ap.add_argument("--strong-rows", type=int, default=int(os.environ.get("SE_BENCH_STRONG_ROWS", 100_000_000)),
                    help="GLOBAL rows of the strong-scaling measurement (split over the ranks); 0 disables")
    ap.add_argument("--no-parity", action="store_true", help="skip the oracle self-check after the timed regions")
    ap.add_argument("--no-extras", action="store_true", help="skip the tree / async / config-3 extras")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed round's outputs (rank 0) as DIR/<name>.npy, at most 32 MB")
    args = ap.parse_args()
    if args.impl == "ours" and args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    workload = (f"GBMRegressor boosting iteration (Brent line search + fused F update / next pseudo-residuals / "
                f"loss), squared loss, {args.rows} rows x {args.features} features fp32 per GPU, synthetic; "
                f"direction h = 0.5*y + 0.5*N(0,1) (a base learner correlated with the label), learningRate 0.1")

    if args.impl == "reference":
        if rank != 0:
            return 0
        res = run_cpu_arm(args.cpu_rows, max(args.steps, 1), max(args.warmup, 1))
        sample = f"{args.cpu_rows} rows per step (of {args.rows}), fp64, OpenMP restatement of the reference round"
        print(json.dumps({
            "impl": "reference", "metric": METRIC, "value": res["value"], "unit": "rows/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": res["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload, "note": "reference is Scala/Spark (no JVM in this image): oracle port timed"},
            "cpu_baseline": {"value": res["value"], "unit": "rows/s", "cores": res["cores"], "kind": "port",
                             "sample": sample, "brent_evals_per_round": res["brent_evals_per_round"],
                             "usable_cpus": res["usable_cpus"]},
            "e2e": {"value": res["value"], "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }))
        return 0

    # ---------------- ours
    from spark_ensemble_b200 import _native as N
    from spark_ensemble_b200.context import Context
    from spark_ensemble_b200.gbm_engine import GBMEngine

    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    ctx = Context(local_rank)
    if world > 1:
        import torch
        uid = torch.zeros(N.COMM_ID_BYTES, dtype=torch.uint8, device="cuda")
        if rank == 0:
            uid = torch.frombuffer(bytearray(Context.comm_unique_id()), dtype=torch.uint8).cuda()
        dist.broadcast(uid, 0)
        ctx.comm_init(world, rank, bytes(uid.cpu().numpy().tobytes()))

    # clocks are sampled from here (before the inputs are generated: nvidia-smi's own start-up — NVML attaching to every
    # GPU of the box — is over long before the first timed step, so only its periodic light queries overlap the timed
    # region) to the end of the e2e loop: the device-resident timed region alone lasts only ~K x 0.5 ms, shorter than
    # one sampling period
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    n, d = args.rows, args.features
    eng = GBMEngine(ctx, n, 0, 1, "squared", 0.0, has_weights=False)
    seed = 1000 * (rank + 1)
    ctx.fill_synthetic(N.SLOT_Y, "normal", seed + 1, 0.0, 1.0)

    def make_direction():
        """h = 0.5*y + 0.5*N(0,1) built on the device with ABI calls only (same law as the CPU arm's direction):
        F <- N(0, 0.5); H <- y; F <- F + 0.5*H; H <- F; F <- 0."""
        ctx.fill_synthetic(N.SLOT_F, "normal", seed + 2, 0.0, 0.5)
        ctx.copy_slot(N.SLOT_H, N.SLOT_Y)
        ctx.gbm_update([0.5], residual=False, loss=False)
        ctx.copy_slot(N.SLOT_H, N.SLOT_F)
        ctx.fill(N.SLOT_F, 0.0)

    make_direction()
    have_x = not args.no_features
    if have_x:
        ctx.alloc(N.SLOT_X, d, n)
        ctx.fill_synthetic(N.SLOT_X, "normal", seed + 3, 0.0, 1.0)
    ctx.gbm_pseudo_residuals(False)
    ctx.sync()
    lr, tol, max_iter = 0.1, 1e-6, 100

    def barrier():
        ctx.sync()
        if dist is not None:
            dist.barrier()
        ctx.sync()

    def step():
        # Brent line search + fused update/residual/loss: one call through the C ABI (se_gbm_round)
        return ctx.gbm_round(lr, True, tol, max_iter, residual=True)

    for _ in range(args.warmup):
        step()
    barrier()
    ctx.kernel_timing(True)
    ctx.kernel_times_reset()
    launches0 = ctx.launch_count
    barrier()
    ctx.timer_start()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        last = step()
    ms_dev = ctx.timer_stop()
    ctx.sync()
    ms_wall = 1e3 * (time.perf_counter() - t0)
    barrier()
    launches = ctx.launch_count - launches0
    ktimes = ctx.kernel_times()
    ctx.kernel_timing(False)
    ms = max(ms_dev, ms_wall)  # device events and host clock bracket the same region; host syncs are inside
    if dist is not None:
        import torch
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, ctx, n, *last)

    # ---------------- e2e: host buffers through the host-side mirror's round body
    h_host, hp = _pinned_array(n)
    r_host, rp = _pinned_array(n)
    ctx.download(N.SLOT_H, out=h_host)
    for _ in range(2):
        eng.boost_round(h_host, lr, tol, max_iter, r_host)
    barrier()
    e2e_steps = max(3, min(args.steps, 10))
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        eng.boost_round(h_host, lr, tol, max_iter, r_host)
    ctx.sync()
    e2e_ms = 1e3 * (time.perf_counter() - t0)
    clocks = sampler.stop() if rank == 0 else None
    if dist is not None:
        import torch
        t = torch.tensor([e2e_ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = float(t.item())

    # ---------------- extras: device-resident async round, on-device tree direction over X
    extras = {}
    ctx.kernel_timing(False)
    if args.no_extras:
        have_x = False
    for _ in range(2):
        ctx.gbm_round_squared_async(lr)
    barrier()
    ctx.timer_start()
    for _ in range(args.steps):
        ctx.gbm_round_squared_async(lr)
    ams = ctx.timer_stop()
    extras["async_round_rows_per_s_per_gpu"] = n * args.steps / (ams * 1e-3)
    if have_x:
        depth = 6
        nn = 2 ** (depth + 1) - 1
        idx = np.arange(nn)
        leaf = idx >= 2 ** depth - 1
        tree = {"feature": np.where(leaf, -1, (idx * 37) % d), "threshold": np.where(leaf, 0.0, ((idx * 13) % 7 - 3) * 0.2),
                "left": np.where(leaf, 0, 2 * idx + 1), "right": np.where(leaf, 0, 2 * idx + 2),
                "value": np.linspace(-1, 1, nn)}
        ctx.tree_predict(tree, N.SLOT_H, 0)
        ctx.sync()
        ctx.kernel_timing(True)
        ctx.kernel_times_reset()
        for _ in range(5):
            ctx.tree_predict(tree, N.SLOT_H, 0)
        kt = ctx.kernel_times().get("tree", {"ms": float("nan"), "launches": 1})
        ctx.kernel_timing(False)
        extras["tree_direction"] = {"depth": depth, "ms": kt["ms"] / kt["launches"],
                                    "rows_per_s_per_gpu": n / (kt["ms"] / kt["launches"] * 1e-3),
                                    "note": "on-device base-model predict over column-major X; reported separately"}

        # e2e with the base model evaluated on device: only the tree (bytes) goes host->device per round
        for _ in range(2):
            ctx.tree_predict(tree, N.SLOT_H, 0)
            a_, _, _ = ctx.gbm_linesearch_brent(0.0, 100.0, 1.0, tol, tol, max_iter)
            ctx.gbm_update([lr * a_], residual=True, loss=True)
            ctx.download(N.SLOT_R, out=r_host)
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            ctx.tree_predict(tree, N.SLOT_H, 0)
            a_, _, _ = ctx.gbm_linesearch_brent(0.0, 100.0, 1.0, tol, tol, max_iter)
            ctx.gbm_update([lr * a_], residual=True, loss=True)
            ctx.download(N.SLOT_R, out=r_host)
        ctx.sync()
        dt_ms = 1e3 * (time.perf_counter() - t0)
        extras["e2e_device_tree"] = {"rows_per_s_per_gpu": n * e2e_steps / (dt_ms * 1e-3), "ms_per_step": dt_ms / e2e_steps,
                                     "h2d_bytes_per_step": 20 * nn, "d2h_bytes_per_step": 4 * n + 32,
                                     "note": "direction = depth-6 tree evaluated on device over the resident feature matrix; "
                                             "pseudo-residuals still go device->host for the (host) base-learner fit"}

    # ---------------- strong scaling: a fixed GLOBAL dataset split over the ranks (same buffers, first rows)
    def timed_rounds(n_rows, steps, loss="squared"):
        ctx.gbm_configure(n_rows, 0, 1, loss, 0.0, False)   # re-uses the resident slots (no reallocation)
        if loss != "squared":
            # labels ~ Bernoulli(0.4); direction h = y + N(0, 0.5): correlated with the label like a fitted base learner
            ctx.fill_synthetic(N.SLOT_Y, "bernoulli", seed + 7, 0.4, 1.0)
            ctx.fill_synthetic(N.SLOT_F, "normal", seed + 8, 0.0, 0.5)
            ctx.copy_slot(N.SLOT_H, N.SLOT_Y)
            ctx.set_option("fused_round", 0)
            ctx.gbm_update([1.0], residual=False, loss=False)
            ctx.set_option("fused_round", -1)
            ctx.copy_slot(N.SLOT_H, N.SLOT_F)
        else:
            make_direction()   # the tree extras overwrote H
        ctx.fill(N.SLOT_F, 0.0)
        ctx.gbm_pseudo_residuals(False)
        for _ in range(3):
            ctx.gbm_round(lr if loss == "squared" else 0.1, True, tol, max_iter, residual=True)
        barrier()
        ctx.timer_start()
        t0 = time.perf_counter()
        evals = 0
        for _ in range(steps):
            _, _, ne = ctx.gbm_round(lr if loss == "squared" else 0.1, True, tol, max_iter, residual=True)
            evals += ne
        ms_d = ctx.timer_stop()
        ctx.sync()
        ms_w = 1e3 * (time.perf_counter() - t0)
        barrier()
        m = max(ms_d, ms_w)
        if dist is not None:
            import torch
            t = torch.tensor([m], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            m = float(t.item())
        return m / steps, evals / steps

    strong = strong_c3 = None
    if args.strong_rows > 0:
        ns = min(n, (args.strong_rows // world) // 4 * 4)
        ms_s, ne_s = timed_rounds(ns, max(args.steps, 20))
        strong = {"rows_global": ns * world, "rows_per_gpu": ns, "ms_per_step": ms_s, "value": ns * world / (ms_s * 1e-3),
                  "unit": "rows/s", "one_launch_round": int(ctx.get_option("last_round_fused")),
                  "brent_evals_per_round": ne_s, "scaling": "strong",
                  "note": "same round as `value` on a fixed global dataset split over the ranks"}
    parity = []
    if not args.no_parity and args.strong_rows > 0:
        parity.append(parity_check(ctx, ns, lr, tol, max_iter, world, rank, dist, "strong shard (global rows / N per GPU)"))
    if args.strong_rows > 0 and not args.no_extras:
        nc3 = min(n, (min(args.strong_rows, 50_000_000) // world) // 4 * 4)
        ms_c, ne_c = timed_rounds(nc3, 5, loss="bernoulli")
        strong_c3 = {"rows_global": nc3 * world, "rows_per_gpu": nc3, "ms_per_round": ms_c, "value": nc3 * world / (ms_c * 1e-3),
                     "unit": "rows/s", "brent_evals_per_round": ne_c, "loss": "bernoulli",
                     "line_search": {0: "one launch per evaluation", 1: "one persistent launch (device Brent)",
                                     2: "host Brent over the persistent kernel"}[int(ctx.get_option("ls_mode"))],
                     "ls_workers": int(ctx.get_option("last_ls_workers")), "l2_hit_ratio_requested": ctx.get_option("last_ls_hit_ratio")}
    if not args.no_parity:
        # the weak-scaling configuration itself (full shard per GPU, the round `value` was timed on)
        ctx.gbm_configure(n, 0, 1, "squared", 0.0, False)
        ctx.fill_synthetic(N.SLOT_Y, "normal", seed + 1, 0.0, 1.0)
        make_direction()
        ctx.gbm_pseudo_residuals(False)
        ctx.gbm_round(lr, True, tol, max_iter, residual=True)
        parity.append(parity_check(ctx, n, lr, tol, max_iter, world, rank, dist, "weak shard (the timed configuration)"))
    p2p_active = bool(ctx.comm_p2p_active()) if world > 1 else None

    if rank != 0:
        ctx.close()
        if dist is not None:
            dist.destroy_process_group()
        return 0

    peak, peak_src = _peaks()
    k1 = ktimes.get("update", {"ms": float("nan"), "launches": 1})
    k2 = ktimes.get("sq_stats", None)
    k1_ms = k1["ms"] / max(k1["launches"], 1)
    if k2 is None:
        # one cooperative launch per round: statistics pass (8 B/row) + update pass (20 B/row) inside ONE kernel
        roof_kernel = ("gbm_round_sq_fused_kernel (whole round in one launch: statistics r,h -> Brent -> "
                       "F update + residual; 8 + 20 B/row)")
        roof_bytes = BYTES_ROUND
        extras["kernel_ms_share_of_step"] = k1["ms"] / ms_dev if ms_dev > 0 else None
    else:
        roof_kernel = "gbm_scalar_kernel<squared, UPDATE_RESID> (K1: F update + residual + loss)"
        roof_bytes = BYTES_K1
        k2_ms = k2["ms"] / max(k2["launches"], 1)
        extras["k2_stats_kernel"] = {"ms": k2_ms, "achieved_gbs": BYTES_K2 * n / (k2_ms * 1e-3) / 1e9,
                                     "frac": BYTES_K2 * n / (k2_ms * 1e-3) / 1e9 / peak}
        extras["kernel_ms_share_of_step"] = (k1["ms"] + k2["ms"]) / ms_dev if ms_dev > 0 else None
    achieved = roof_bytes * n / (k1_ms * 1e-3) / 1e9
    extras["device_ms_per_step"] = ms_dev / args.steps
    extras["wall_ms_per_step"] = ms_wall / args.steps
    extras["strong_scaling"] = strong
    extras["strong_c3"] = strong_c3

    cpu = None
    if world == 1:
        cpu_steps = 3
        c = run_cpu_arm(args.cpu_rows, cpu_steps, 1)
        cpu = {"value": c["value"], "unit": "rows/s", "cores": c["cores"], "usable_cpus": c["usable_cpus"], "kind": "port",
               "sample": f"{cpu_steps} reference rounds on {args.cpu_rows} rows (fp64 OpenMP restatement; "
                         f"{c['brent_evals_per_round']:.1f} full-pass Brent evaluations per round)"}

    out = {
        "metric": METRIC, "value": world * n * args.steps / (ms * 1e-3), "unit": "rows/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload, "rows_per_gpu": n, "features": d, "loss": "squared",
                   "l2": "inputs (1.2 GB of y/F/h per GPU) are larger than L2 (126 MB); no flush needed",
                   "features_resident": have_x,
                   "parallelism": (f"rows sharded x{world}; the <=3 fp64 sums of every reduction are exchanged over NVLink peer "
                                   f"memory by the reducing kernel's last CTA (fused all-reduce, p2p_active={p2p_active}; NCCL only "
                                   f"bootstraps the IPC handles and is the fallback)") if world > 1 else "single GPU"},
        "clocks": clocks,
        "e2e": {"value": world * n * e2e_steps / (e2e_ms * 1e-3), "unit": "rows/s",
                "h2d_bytes_per_step": 4 * n, "d2h_bytes_per_step": 4 * n + 8 * 4, "steps": e2e_steps,
                "ms_per_step": e2e_ms / e2e_steps,
                "note": "direction h host->device and pseudo-residuals device->host (pinned) every round"},
        "gpu_launches": int(launches),
        "parity_ok": (all(p["ok"] for p in parity) if parity else None), "parity": parity, "p2p_active": p2p_active,
        "roofline": {"kernel": roof_kernel,
                     "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": _ncu_traffic(n, roof_bytes), "peak_source": peak_src, "bytes_per_row": roof_bytes, "ms_per_launch": k1_ms,
                     "launches_timed": k1["launches"]},
        "cpu_baseline": cpu,
        "extras": extras,
    }
    print(json.dumps(out))
    ctx.close()
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
