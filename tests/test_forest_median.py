"""se_forest_weighted_median: AdaBoost.R2's weighted median of tree members in one pass over the rank matrix, bit for bit
against the device member route (tree_predict of every member + agg_run(AGG_BOOSTING_REG_MEDIAN)) and against the fp64
oracle over a plain numpy walk of every member; its failure modes; Params residentFeatures and forestTransform of
BoostingRegressor / BoostingRegressionModel; ShardedContext.  GPU tests are marked `gpu`, the rest run anywhere."""
import os
import re
import zlib

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WEIGHTS = ["random", "equal", "integers", "one_heavy", "zeros", "negative"]
LEAF_POOL = np.array([0.0, -0.0, 1e30, -1e30, 1.5, -2.25, 0.5], dtype=np.float32)


@pytest.fixture(scope="module")
def ctx():
    from spark_ensemble_b200.context import Context
    c = Context(0)
    yield c
    c.close()


def _walk(tree, X):
    """Plain numpy walk: x <= threshold goes left (Spark ContinuousSplit.shouldGoLeft)."""
    node = np.zeros(X.shape[0], dtype=np.int64)
    for _ in range(1024):
        f = tree["feature"][node]
        live = f >= 0
        if not live.any():
            break
        x = X[np.arange(X.shape[0]), np.maximum(f, 0)]
        nxt = np.where(x <= tree["threshold"][node], tree["left"][node], tree["right"][node])
        node = np.where(live, nxt, node)
    return node


def _random_unbalanced_tree(rng, n_internal, d, candidates):
    """Random binary tree grown by splitting a random leaf n_internal times; node ids in creation order (not a heap).
    Leaf values: ties from a small pool (±0, ±1e30 included) mixed with distinct values."""
    feat, thr, left, right = [-1], [0.0], [0], [0]
    leaves = [0]
    for _ in range(n_internal):
        i = leaves.pop(int(rng.integers(0, len(leaves))))
        f = int(rng.integers(0, d))
        feat[i], thr[i] = f, float(candidates[f][rng.integers(0, len(candidates[f]))])
        left[i], right[i] = len(feat), len(feat) + 1
        for _c in range(2):
            feat.append(-1); thr.append(0.0); left.append(0); right.append(0)
        leaves += [left[i], right[i]]
    nn = len(feat)
    value = np.where(rng.random(nn) < 0.5, LEAF_POOL[rng.integers(0, LEAF_POOL.size, nn)],
                     rng.standard_normal(nn).astype(np.float32)).astype(np.float32)
    return {"feature": np.array(feat, np.int32), "threshold": np.array(thr, np.float32), "left": np.array(left, np.int32),
            "right": np.array(right, np.int32), "value": value}


def _weights(rng, kind, M):
    ints = rng.integers(1, 4, M).astype(np.float64)
    if ints.sum() % 2:
        ints[0] += 1.0  # even total: sorted prefixes DO hit the half-weight exactly
    return {"random": rng.random(M) + 0.05, "equal": np.full(M, 0.3), "integers": ints,
            "one_heavy": np.where(np.arange(M) == M // 2, 1e6, 1e-3), "zeros": np.zeros(M),
            "negative": np.where(np.arange(M) == 0, -0.5, 1.0) * (rng.random(M) + 0.05)}[kind]


def _expected_mode(a):
    if np.any(a < 0) or not np.all(np.isfinite(a)):
        return 0
    return 2 if np.all(a == a[0]) else 1


def _bits(v):
    return np.asarray(v, dtype=np.float32).view(np.uint32)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 777, 30_011, 200_003])
@pytest.mark.parametrize("weights", WEIGHTS)
@pytest.mark.parametrize("M", [1, 2, 3, 10, 33, 64])
def test_forest_weighted_median_matches_member_route(ctx, oracle, M, weights, n):
    from spark_ensemble_b200 import _native as N
    rng = np.random.default_rng(zlib.crc32(repr((M, weights, n)).encode()))
    d = 24
    X = rng.standard_normal((n, d)).astype(np.float32)
    cand = [np.unique(np.concatenate([rng.standard_normal(12).astype(np.float32), X[rng.integers(0, n, 3), f]]))
            for f in range(d)]
    trees = [_random_unbalanced_tree(rng, int(rng.integers(1, 41)), d, cand) for _ in range(M)]
    a = _weights(rng, weights, M)
    P = np.stack([tr["value"][_walk(tr, X)] for tr in trees]).astype(np.float32)
    ref = oracle.agg_weighted_median(P, a).astype(np.float32)
    mode = _expected_mode(a)
    try:
        for validation, slot in ((False, N.SLOT_X), (True, N.SLOT_VX)):
            ctx.alloc(slot, d, n)
            ctx.upload_rowmajor(slot, X)
            ctx.alloc(N.SLOT_RAW, 1, n)
            ctx.forest_weighted_median(trees, N.SLOT_RAW, a, validation=validation)
            got = ctx.download(N.SLOT_RAW)
            assert ctx.get_option("last_forest_chunks") == 1
            assert ctx.get_option("last_tree_binned") == 1
            assert ctx.get_option("last_wm_mode") == mode
            deferred = ctx.get_option("last_wm_deferred")
            np.testing.assert_array_equal(got, ref)
            if mode == 1 and weights == "random":
                assert deferred == 0
            if mode == 1 and weights == "integers" and M >= 5 and n >= 30_011:
                assert deferred > 0
            # the exact pick for every row: the same bits
            try:
                ctx.set_option("wm_fast", 0)
                ctx.forest_weighted_median(trees, N.SLOT_RAW, a, validation=validation)
                assert ctx.get_option("last_wm_mode") == 0
                np.testing.assert_array_equal(_bits(ctx.download(N.SLOT_RAW)), _bits(got))
            finally:
                ctx.set_option("wm_fast", 1)
        # the device member route: every member into P (X), then se_agg_run over the same weights
        ctx.agg_configure(N.AGG_BOOSTING_REG_MEDIAN, M, 0, 1, 0, n)
        for t, tr in enumerate(trees):
            ctx.tree_predict(tr, N.SLOT_P, t)
        ctx.agg_run(a)
        assert ctx.get_option("last_wm_mode") == mode
        if mode == 1:  # the same rows fail the same margin test
            assert ctx.get_option("last_wm_deferred") == deferred
        np.testing.assert_array_equal(_bits(ctx.download(N.SLOT_RAW)), _bits(got))
    finally:
        ctx.free(N.SLOT_X)
        ctx.free(N.SLOT_VX)
        ctx.free(N.SLOT_P)


@pytest.mark.gpu
def test_forest_weighted_median_failure_modes(ctx):
    from spark_ensemble_b200 import _native as N
    rng = np.random.default_rng(7)
    n, d = 1000, 6
    X = rng.standard_normal((n, d)).astype(np.float32)
    cand = [np.sort(rng.standard_normal(10).astype(np.float32)) for _ in range(d)]
    trees = [_random_unbalanced_tree(rng, 12, d, cand) for _ in range(5)]
    a = rng.random(5) + 0.1
    ctx.free(N.SLOT_X)
    ctx.alloc(N.SLOT_RAW, 1, n)
    with pytest.raises(N.NativeError) as e:  # no feature slot
        ctx.forest_weighted_median(trees, N.SLOT_RAW, a)
    assert e.value.code == N.SE_ERR_STATE
    ctx.alloc(N.SLOT_X, d, n)
    ctx.upload_rowmajor(N.SLOT_X, X)
    try:
        def ok(oracle_trees=trees, w=a):
            from oracle.oracle import Oracle
            ctx.alloc(N.SLOT_RAW, 1, n)
            ctx.forest_weighted_median(oracle_trees, N.SLOT_RAW, w)
            P = np.stack([tr["value"][_walk(tr, X)] for tr in oracle_trees]).astype(np.float32)
            np.testing.assert_array_equal(ctx.download(N.SLOT_RAW), Oracle(omp=False).agg_weighted_median(P, w).astype(np.float32))

        ok()
        many = [_random_unbalanced_tree(rng, 6, d, cand) for _ in range(65)]  # more than 64 members
        with pytest.raises(N.NativeError) as e:
            ctx.forest_weighted_median(many, N.SLOT_RAW, np.ones(65))
        assert e.value.code == N.SE_ERR_STATE
        ok(many[:64], np.ones(64))
        big = [_random_unbalanced_tree(rng, 1000, d, cand) for _ in range(10)]  # 20 010 nodes: beyond one chunk
        with pytest.raises(N.NativeError) as e:
            ctx.forest_weighted_median(big, N.SLOT_RAW, np.ones(10))
        assert e.value.code == N.SE_ERR_STATE
        ok()
        wide = np.sort(rng.standard_normal(400).astype(np.float32))  # > 255 thresholds in one column
        wide_col = [_random_unbalanced_tree(rng, 60, d, [wide] * d) for _ in range(8)]
        for tr in wide_col:
            tr["feature"] = np.where(tr["feature"] >= 0, 5, -1).astype(np.int32)
        with pytest.raises(N.NativeError) as e:
            ctx.forest_weighted_median(wide_col, N.SLOT_RAW, np.ones(8))
        assert e.value.code == N.SE_ERR_STATE
        ok()
        ctx.alloc(N.SLOT_RAW, 1, n + 1)  # output columns != feature columns
        with pytest.raises(N.NativeError) as e:
            ctx.forest_weighted_median(trees, N.SLOT_RAW, a)
        assert e.value.code == N.SE_ERR_STATE
        ok()
        internal = int(np.argmax(trees[0]["feature"] >= 0))
        b = dict(trees[0]); b["left"] = b["left"].copy(); b["left"][internal] = internal  # its own child
        with pytest.raises(ValueError):
            ctx.forest_weighted_median([b] + trees[1:], N.SLOT_RAW, a)
        ok()
        b = dict(trees[0]); b["feature"] = b["feature"].copy(); b["feature"][internal] = d + 3  # column outside X
        with pytest.raises(ValueError):
            ctx.forest_weighted_median([b] + trees[1:], N.SLOT_RAW, a)
        ok()
        with pytest.raises(ValueError):  # missing weights
            ctx.forest_weighted_median(trees, N.SLOT_RAW, None)
        ok()
    finally:
        ctx.free(N.SLOT_X)


def _cpusmall(rows=4000):
    z = np.load(os.path.join(ROOT, "tests", "golden", "cpusmall.npz"))
    return np.asarray(z["X"], np.float32)[:rows], np.asarray(z["y"], np.float64)[:rows]


@pytest.mark.gpu
@pytest.mark.parametrize("voting", ["median", "mean"])
def test_mirror_boosting_regressor_forest_transform_and_resident_features(voting):
    from spark_ensemble_b200.ensemble import DataFrame
    from spark_ensemble_b200.learners import DecisionTreeRegressor
    from spark_ensemble_b200.regression import BoostingRegressionModel, BoostingRegressor
    X, y = _cpusmall()
    df = DataFrame(features=X, label=y)

    def est(resident):
        return (BoostingRegressor().set("baseLearner", DecisionTreeRegressor(maxDepth=5)).set("numBaseLearners", 10)
                .set("votingStrategy", voting).set("residentFeatures", resident))

    host, dev = est(False).fit(df), est(True).fit(df)
    assert dev("residentFeatures") is True and host.numModels == dev.numModels >= 2
    np.testing.assert_array_equal(dev.weights, host.weights)
    assert dev.trainingHistory == host.trainingHistory
    feats = DataFrame(features=X)
    base = np.asarray(host.transform(feats)["prediction"])
    np.testing.assert_array_equal(np.asarray(dev.transform(feats)["prediction"]), base)
    fast = np.asarray(host.copy().set("forestTransform", True).transform(feats)["prediction"])
    if voting == "median":
        np.testing.assert_array_equal(_bits(fast), _bits(base))
    else:
        scale = float(np.abs(base).max())
        assert np.all(np.abs(fast - base) <= 1e-5 * np.maximum(np.abs(base), scale))
    # 70 tree members: the median is beyond the kernel's 64 and takes the member route with identical output; the mean
    # (se_forest_predict) has no member limit
    rng = np.random.default_rng(5)
    members = [host.models[i % host.numModels] for i in range(70)]
    big = BoostingRegressionModel(rng.random(70) + 0.1, members)
    big.set("votingStrategy", voting)
    off = np.asarray(big.transform(feats)["prediction"])
    on = np.asarray(big.copy().set("forestTransform", True).transform(feats)["prediction"])
    if voting == "median":
        np.testing.assert_array_equal(on, off)
    else:
        scale = float(np.abs(off).max())
        assert np.all(np.abs(on - off) <= 1e-5 * np.maximum(np.abs(off), scale))


@pytest.mark.gpu
def test_sharded_forest_weighted_median_equals_one_context():
    from spark_ensemble_b200 import _native as N
    from spark_ensemble_b200.context import Context
    from spark_ensemble_b200.sharded import ShardedContext
    if N.device_count() < 2:
        pytest.skip("needs two GPUs")
    rng = np.random.default_rng(11)
    n, d, M = 50_001, 10, 12
    X = rng.standard_normal((n, d)).astype(np.float32)
    cand = [np.sort(rng.standard_normal(12).astype(np.float32)) for _ in range(d)]
    trees = [_random_unbalanced_tree(rng, 30, d, cand) for _ in range(M)]
    a = _weights(rng, "integers", M)
    with Context(0) as c:
        c.alloc(N.SLOT_X, d, n)
        c.upload_rowmajor(N.SLOT_X, X)
        c.alloc(N.SLOT_RAW, 1, n)
        c.forest_weighted_median(trees, N.SLOT_RAW, a)
        want = c.download(N.SLOT_RAW)
    with ShardedContext([0, 1]) as sc:
        sc.gbm_configure(n, 0, 1, "squared")
        sc.alloc(N.SLOT_X, d, n)
        sc.upload_rowmajor(N.SLOT_X, X)
        sc.alloc(N.SLOT_F, 1, n)
        sc.forest_weighted_median(trees, N.SLOT_F, a)
        got = sc.download(N.SLOT_F)
    np.testing.assert_array_equal(_bits(np.asarray(got).reshape(-1)), _bits(want))


# ------------------------------------------------------------------ CPU
@pytest.mark.parametrize("name", ["BoostingRegressor", "BoostingRegressionModel"])
@pytest.mark.parametrize("param", ["forestTransform", "residentFeatures"])
def test_boosting_regressor_params_default_off(name, param):
    from spark_ensemble_b200 import regression
    cls = getattr(regression, name)
    assert cls._params[param].name == param
    assert cls._defaults[param] is False


def test_boosting_regressor_params_are_copied_to_the_model():
    from spark_ensemble_b200.regression import BoostingRegressionModel, BoostingRegressor
    est = BoostingRegressor().set("forestTransform", True).set("residentFeatures", True)
    m = est._copyValues(BoostingRegressionModel([], []))
    assert m("forestTransform") is True
    assert m("residentFeatures") is True


class _FakeCtx:
    def __init__(self, device):
        self.device, self.calls = device, []

    def close(self):
        pass

    def sync(self):
        pass

    def comm_destroy(self):
        pass

    def gbm_configure(self, n, nv, dim, loss, param=0.0, has_weights=False):
        self.n = n

    def forest_weighted_median(self, trees, out_slot, weights, out_row=0, validation=False):
        self.calls.append(("median", len(trees), out_slot, tuple(weights), out_row, validation))


def test_sharded_forest_weighted_median_reaches_every_shard():
    from spark_ensemble_b200 import _native as N
    from spark_ensemble_b200.sharded import ShardedContext
    sc = ShardedContext([0, 1, 2], context_factory=_FakeCtx, join=False)
    sc.gbm_configure(101, 0, 1, "squared")
    sc.forest_weighted_median([{"feature": [-1]}] * 4, N.SLOT_F, [1.0, 2.0, 3.0, 4.0], validation=True)
    assert all(c.calls == [("median", 4, N.SLOT_F, (1.0, 2.0, 3.0, 4.0), 0, True)] for c in sc.ctxs)
    sc.close()


def test_boosting_regression_model_native_uses_existing_natives():
    natives = set(re.findall(r"@native def (\w+)\(", open(os.path.join(ROOT, "scala", "org", "apache", "spark", "ml", "se",
                                                                       "SeNative.scala")).read()))
    src = open(os.path.join(ROOT, "scala", "org", "apache", "spark", "ml", "regression",
                            "BoostingRegressionModelNative.scala")).read()
    used = set(re.findall(r"SeNative\.(\w+)\(", src))
    assert used and used <= natives, used - natives
    for call in ("forestWeightedMedian", "forestPredict", "aggConfigure", "aggRun", "uploadRowmajor", "download",
                 "ctxDestroy"):
        assert call in used


def test_forest_wmedian_kernel_compiles_without_spills(tmp_path):
    import shutil
    import subprocess
    from spark_ensemble_b200 import build
    nvcc = build._nvcc() if (shutil.which("nvcc") or os.path.exists("/usr/local/cuda/bin/nvcc")) else None
    if nvcc is None:
        pytest.skip("nvcc not available")
    r = subprocess.run([nvcc] + build.NVCC_FLAGS + ["-Xptxas", "-v", "-c", os.path.join(build.CSRC, "se_models.cu"),
                                                    "-o", str(tmp_path / "m.o")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = r.stderr.splitlines()
    found = set()
    for i, line in enumerate(lines):
        m = re.search(r"Function properties for .*forest_wmedian_kernelILi(\d+)E", line)
        if m:
            mp = int(m.group(1))
            found.add(mp)
            assert "0 bytes spill stores, 0 bytes spill loads" in lines[i + 1], (mp, lines[i + 1])
            regs = int(re.search(r"Used (\d+) registers", lines[i + 2]).group(1))
            assert regs * 256 * (1 if mp >= 32 else 2) <= 65536, (mp, regs)  # the kernel's __launch_bounds__
    assert found == {1, 2, 4, 8, 16, 32, 64}
