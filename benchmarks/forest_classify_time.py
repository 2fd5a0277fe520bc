#!/usr/bin/env python
"""Classifier-ensemble transform for tree members: se_forest_classify (one pass over the rank matrix, no member outputs)
vs the member route (one se_tree_predict / se_tree_predict_multi per member into SE_SLOT_P, then se_agg_run).

    python benchmarks/forest_classify_time.py [--rows 10000000] [--check-rows 1000000] [--out profiles/r03_forest_classify.json]

Depth-6 trees over 64 columns with 31 candidate thresholds each (Spark's default maxBins 32).  Times are host clocks
around work that ends in a device synchronise, after one warm-up call of each route, best of --repeat.

se_tree_predict_multi writes rows 0..K-1 of its output slot, so the timed member route of the probability kinds
evaluates every member into the first K rows of P: the same kernels and bytes as the real route, only the destination
rows differ.  The RAW comparison therefore runs separately on the first --check-rows rows, where each member's
probabilities are copied into their own rows of P through the host.
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
ap.add_argument("--check-rows", type=int, default=1_000_000)
ap.add_argument("--repeat", type=int, default=3)
ap.add_argument("--out", default=None)
args = ap.parse_args()

d, depth = 64, 6
grid = (np.arange(-15, 16) * 0.1).astype(np.float32)
CASES = [("soft", N.AGG_BAGGING_SOFT, 50, 26, 1), ("real", N.AGG_BOOSTING_REAL, 50, 26, 1),
         ("hard", N.AGG_BAGGING_HARD, 100, 26, 1), ("gbm", N.AGG_GBM_CLASSIFIER, 20, 26, 26),
         ("gbm_binary", N.AGG_GBM_CLASSIFIER, 100, 2, 1)]


def make_forest(rng, kind, n_trees, K):
    nn = 2 ** (depth + 1) - 1
    idx = np.arange(nn)
    leaf = idx >= 2 ** depth - 1
    trees = []
    for _ in range(n_trees):
        t = {"feature": np.where(leaf, -1, rng.integers(0, d, nn)).astype(np.int32),
             "threshold": np.where(leaf, 0.0, grid[rng.integers(0, grid.size, nn)]).astype(np.float32),
             "left": np.where(leaf, 0, 2 * idx + 1).astype(np.int32), "right": np.where(leaf, 0, 2 * idx + 2).astype(np.int32)}
        if kind in ("soft", "real"):
            p = rng.random((nn, K)).astype(np.float64) + 1e-3
            t["values"] = (p / p.sum(1, keepdims=True)).astype(np.float32)
        elif kind == "hard":
            t["value"] = rng.integers(0, K, nn).astype(np.float32)
        else:
            t["value"] = (0.1 * rng.standard_normal(nn)).astype(np.float32)
        trees.append(t)
    return trees


def member_route(ctx, trees, kid, M, K, dim, w, init, n, exact):
    """se_tree_predict* per member into P, then se_agg_run.  exact: every member into its own rows of P."""
    ctx.agg_configure(kid, M, K, dim, "logloss" if dim > 1 else "bernoulli", n)
    for m, tr in enumerate(trees):
        if "values" not in tr:
            ctx.tree_predict(tr, N.SLOT_P, m)
        elif exact:
            ctx.tree_predict_multi(tr, N.SLOT_PROBA)
            ctx.upload(N.SLOT_P, ctx.download(N.SLOT_PROBA).reshape(-1), offset=m * K * n)
        else:
            ctx.tree_predict_multi(tr, N.SLOT_P)
    ctx.agg_run(w, init)


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
res = {"rows": args.rows, "columns": d, "depth": depth, "check_rows": args.check_rows, **gpu_info(), "cases": []}
big, small = Context(0), Context(0)
for ctx, n in ((big, args.rows), (small, args.check_rows)):
    ctx.alloc(N.SLOT_X, d, n)
    ctx.fill_synthetic(N.SLOT_X, "normal", 3, 0, 1)
for name, kid, M, K, dim in CASES:
    n_trees = M * dim
    trees = make_forest(rng, name, n_trees, K)
    w = init = None
    if kid == N.AGG_GBM_CLASSIFIER:
        w = 0.5 + rng.random((M, dim))
        init = 0.1 * rng.standard_normal(dim)
    loss = "logloss" if dim > 1 else "bernoulli"
    n = args.rows
    one = lambda: big.forest_classify(trees, kid, K, dim=dim, loss=loss, weights=w, init=init)  # noqa: E731
    one()
    forest_ms = timed(one, big)
    chunks = int(big.get_option("last_forest_chunks"))
    members = lambda: member_route(big, trees, kid, M, K, dim, w, init, n, exact=False)  # noqa: E731
    members()
    member_ms = timed(members, big)
    width = K if name in ("soft", "real") else 1
    big.free(N.SLOT_P)
    # RAW of both routes on the first check rows (the members in their own rows of P)
    small.alloc(N.SLOT_PROBA, K, args.check_rows)
    small.forest_classify(trees, kid, K, dim=dim, loss=loss, weights=w, init=init)
    raw_f = small.download(N.SLOT_RAW).astype(np.float64)
    lab_f = small.download(N.SLOT_LABEL)
    member_route(small, trees, kid, M, K, dim, w, init, args.check_rows, exact=True)
    raw_m = small.download(N.SLOT_RAW).astype(np.float64)
    lab_m = small.download(N.SLOT_LABEL)
    small.free(N.SLOT_P)
    r = {"case": name, "members": M, "classes": K, "dim": dim, "trees": n_trees, "forest_ms": forest_ms,
         "forest_chunks": chunks, "member_route_ms": member_ms, "speedup": member_ms / forest_ms,
         "intermediate_bytes_avoided": 4 * M * dim * width * n,
         "raw_max_rel_diff": float(np.max(np.abs(raw_f - raw_m)) / max(np.max(np.abs(raw_m)), 1e-30)),
         "label_mismatch_rows": int(np.sum(lab_f != lab_m))}
    res["cases"].append(r)
    print(json.dumps(r), flush=True)
big.close()
small.close()
print(json.dumps({k: v for k, v in res.items() if k != "cases"}))
if args.out:
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    json.dump(res, open(args.out, "w"), indent=1)
