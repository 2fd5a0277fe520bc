#!/usr/bin/env python
"""AdaBoost.R2 median transform for tree members: se_forest_weighted_median (one pass over the rank matrix, the weighted
median fused with the forest walk, no member outputs) vs the member route (one se_tree_predict per member into
SE_SLOT_P, then se_agg_run(SE_AGG_BOOSTING_REG_MEDIAN)).

    python benchmarks/forest_median_time.py [--rows 10000000] [--out profiles/r04_forest_median.json]

Full trees of depth 5 and 6 over 64 columns with 31 candidate thresholds each (Spark's default maxBins 32), M in
{10, 32, 64} members, generic weights (fast path with the rounding margin, mode 1) and equal weights (mode 2).  Times are
host clocks around work that ends in a device synchronise, after one warm-up call of each route, best of --repeat.  The
outputs of both routes are compared bit for bit on every row.
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

from spark_ensemble_b200 import _native as N  # noqa: E402
from spark_ensemble_b200.context import Context  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--rows", type=int, default=10_000_000)
ap.add_argument("--repeat", type=int, default=3)
ap.add_argument("--out", default=None)
args = ap.parse_args()

d = 64
grid = (np.arange(-15, 16) * 0.1).astype(np.float32)


def make_forest(rng, depth, n_trees):
    nn = 2 ** (depth + 1) - 1
    idx = np.arange(nn)
    leaf = idx >= 2 ** depth - 1
    return [{"feature": np.where(leaf, -1, rng.integers(0, d, nn)).astype(np.int32),
             "threshold": np.where(leaf, 0.0, grid[rng.integers(0, grid.size, nn)]).astype(np.float32),
             "left": np.where(leaf, 0, 2 * idx + 1).astype(np.int32), "right": np.where(leaf, 0, 2 * idx + 2).astype(np.int32),
             "value": rng.standard_normal(nn).astype(np.float32)} for _ in range(n_trees)]


def member_route(ctx, trees, w, n):
    ctx.agg_configure(N.AGG_BOOSTING_REG_MEDIAN, len(trees), 0, 1, 0, n)
    for m, tr in enumerate(trees):
        ctx.tree_predict(tr, N.SLOT_P, m)
    ctx.agg_run(w)


def timed(fn, ctx):
    best = float("inf")
    for _ in range(args.repeat):
        ctx.sync()
        t0 = time.perf_counter()
        fn()
        ctx.sync()
        best = min(best, time.perf_counter() - t0)
    return 1e3 * best


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()
        name, plim = [s.strip() for s in q[0].split(",")]
        return {"gpu": name, "power_limit": plim}
    except Exception as e:  # the numbers still stand; say what is missing
        return {"gpu": f"unknown ({e})", "power_limit": "unknown"}


rng = np.random.default_rng(7)
n = args.rows
res = {"rows": n, "columns": d, "thresholds_per_column": int(grid.size), **gpu_info(), "cases": []}
ctx = Context(0)
ctx.alloc(N.SLOT_X, d, n)
ctx.fill_synthetic(N.SLOT_X, "normal", 3, 0, 1)
for depth in (5, 6):
    for M in (10, 32, 64):
        trees = make_forest(rng, depth, M)
        for wkind in ("generic", "equal"):
            w = 0.1 + rng.random(M) if wkind == "generic" else np.full(M, 0.25)
            ctx.free(N.SLOT_P)
            ctx.alloc(N.SLOT_F, 1, n)
            one = lambda: ctx.forest_weighted_median(trees, N.SLOT_F, w)  # noqa: E731
            one()
            forest_ms = timed(one, ctx)
            mode = int(ctx.get_option("last_wm_mode"))
            deferred = int(ctx.get_option("last_wm_deferred"))
            out_f = ctx.download(N.SLOT_F)
            members = lambda: member_route(ctx, trees, w, n)  # noqa: E731
            members()
            member_ms = timed(members, ctx)
            member_deferred = int(ctx.get_option("last_wm_deferred"))
            out_m = ctx.download(N.SLOT_RAW)
            r = {"depth": depth, "members": M, "weights": wkind, "wm_mode": mode, "forest_ms": forest_ms,
                 "member_route_ms": member_ms, "speedup": member_ms / forest_ms,
                 "last_wm_deferred": deferred, "member_route_deferred": member_deferred,
                 "intermediate_bytes_avoided": 4 * M * n,
                 "bit_equal_rows": int(np.sum(out_f.view(np.uint32) == out_m.view(np.uint32))),
                 "bit_equal": bool(np.array_equal(out_f.view(np.uint32), out_m.view(np.uint32)))}
            res["cases"].append(r)
            print(json.dumps(r), flush=True)
ctx.close()
print(json.dumps({k: v for k, v in res.items() if k != "cases"}))
if args.out:
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    json.dump(res, open(args.out, "w"), indent=1)
