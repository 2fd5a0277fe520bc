"""se_forest_classify: a classifier ensemble of trees in one pass over the rank matrix (GBM, bagging soft / hard, SAMME.R,
SAMME), against the fp64 oracle aggregation of a plain numpy walk of every member and against the device member route
(tree_predict* + agg_run); its failure modes; Param forestTransform of the mirror models; ShardedContext.  GPU tests are
marked `gpu`, the rest run anywhere."""
import os
import re
import zlib

import numpy as np
import pytest

from oracle import oracle as O

RTOL = 1e-5
KINDS = ["gbm", "soft", "hard", "real", "discrete"]
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def ctx():
    from spark_ensemble_b200.context import Context
    c = Context(0)
    yield c
    c.close()


def close(a, b, rtol=RTOL, scale=None):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    if scale is None:
        scale = float(np.sqrt(np.mean(b * b))) if b.size else 1.0
    bad = np.abs(a - b) > rtol * np.maximum(np.abs(b), scale)
    assert not bad.any(), (f"{bad.sum()} / {b.size} mismatches; worst rel "
                           f"{np.max(np.abs(a - b) / np.maximum(np.abs(b), scale)):.3e}")


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
    """Random binary tree grown by splitting a random leaf n_internal times; node ids in creation order (not a heap)."""
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
    return {"feature": np.array(feat, np.int32), "threshold": np.array(thr, np.float32), "left": np.array(left, np.int32),
            "right": np.array(right, np.int32), "value": rng.standard_normal(len(feat)).astype(np.float32)}


def _agg_kind(N, kind):
    return {"gbm": N.AGG_GBM_CLASSIFIER, "soft": N.AGG_BAGGING_SOFT, "hard": N.AGG_BAGGING_HARD,
            "real": N.AGG_BOOSTING_REAL, "discrete": N.AGG_BOOSTING_DISCRETE}[kind]


def _forest(rng, kind, K, dim, d, cand, n_trees):
    """Trees of 150..250 internal nodes (several chunks of trees per call) with the leaves `kind` takes."""
    trees, subs = [], []
    for t in range(n_trees):
        sub = None
        if kind in ("soft", "hard", "gbm") and t % 3 == 1:  # per-member subspaces (HasSubBag)
            sub = np.sort(rng.choice(d, size=d // 2, replace=False)).astype(np.int32)
        cc = cand if sub is None else [cand[c] for c in sub]
        tr = _random_unbalanced_tree(rng, int(rng.integers(150, 251)), d if sub is None else sub.size, cc)
        nn = tr["feature"].size
        if kind in ("soft", "real"):
            p = rng.random((nn, K)) * (rng.random((nn, K)) < 0.7)   # zeros: SAMME.R clamps them to eps
            p[:, 0] += 1e-3
            tr["values"] = (p / p.sum(1, keepdims=True)).astype(np.float32)
        elif kind in ("hard", "discrete"):
            tr["value"] = rng.integers(0, K, nn).astype(np.float32)
        trees.append(tr)
        subs.append(sub)
    return trees, subs


def _member_outputs(trees, subs, X, kind):
    """[M][width][n] member outputs of the numpy walk (width K for probability leaves, else 1)."""
    key = "values" if kind in ("soft", "real") else "value"
    out = []
    for tr, sub in zip(trees, subs):
        leaf = _walk(tr, X if sub is None else X[:, sub])
        v = np.asarray(tr[key])[leaf]
        out.append(v.T if v.ndim == 2 else v[None, :])
    return np.stack(out).astype(np.float32)


def _oracle(oracle, kind, P, K, dim, loss, w, init):
    """(raw, prob) of the fp64 oracle over member outputs P."""
    if kind == "gbm":
        M = P.shape[0] // dim
        raw = oracle.agg_gbm_classifier_raw(P.reshape(M, dim, -1), w.reshape(M, dim), init, K)
        return raw, oracle.gbm_raw2prob(O.LOSS_IDS[loss], raw)
    if kind == "soft":
        return oracle.agg_bagging_soft(P)
    if kind == "real":
        return oracle.agg_boosting_real(P)
    if kind == "hard":
        return oracle.agg_bagging_hard(P[:, 0], K)
    return oracle.agg_boosting_discrete(P[:, 0], w, K)


def _cases():
    for kind in KINDS:
        for K in (2, 3, 8, 26, 65):
            if kind == "gbm":
                yield kind, K, K, "logloss"
                if K == 2:
                    yield kind, 2, 1, "bernoulli"
                    yield kind, 2, 1, "exponential"
            else:
                yield kind, K, 1, "logloss"


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 777, 30_011, 200_003])
@pytest.mark.parametrize("kind,K,dim,loss", list(_cases()))
def test_forest_classify_matches_member_route(ctx, oracle, kind, K, dim, loss, n):
    from spark_ensemble_b200 import _native as N
    rng = np.random.default_rng(zlib.crc32(repr((kind, K, dim, loss, n)).encode()))
    d = 24
    X = rng.standard_normal((n, d)).astype(np.float32)
    cand = [np.unique(np.concatenate([rng.standard_normal(12).astype(np.float32), X[rng.integers(0, n, 3), f]]))
            for f in range(d)]
    M = max(2, 24 // dim) if kind == "gbm" else 24
    trees, subs = _forest(rng, kind, K, dim, d, cand, M * dim if kind == "gbm" else M)
    w = init = None
    if kind == "gbm":
        w = (rng.random((M, dim)) + 0.1).astype(np.float32).astype(np.float64)
        init = rng.standard_normal(dim).astype(np.float32).astype(np.float64)
    elif kind == "discrete":
        w = (rng.random(M) + 0.1).astype(np.float32).astype(np.float64)
    kid = _agg_kind(N, kind)
    P = _member_outputs(trees, subs, X, kind)
    raw_o, prob_o = _oracle(oracle, kind, P, K, dim, loss, w, init)
    C = raw_o.shape[0]
    ctx.free(N.SLOT_P)
    try:
        for validation, slot in ((False, N.SLOT_X), (True, N.SLOT_VX)):
            ctx.alloc(slot, d, n)
            ctx.upload_rowmajor(slot, X)
            ctx.forest_classify(trees, kid, K, dim=dim, loss=loss, weights=w, init=init, validation=validation,
                                subspaces=subs)
            chunks = ctx.get_option("last_forest_chunks")
            assert chunks > 1
            assert ctx.device_ptr(N.SLOT_P) == 0  # no member outputs
            raw = ctx.download(N.SLOT_RAW).reshape(C, n)
            prob = ctx.download(N.SLOT_PROB).reshape(C, n)
            lab = ctx.download(N.SLOT_LABEL).reshape(n)
            tol = RTOL * chunks
            if kind == "hard":
                np.testing.assert_array_equal(raw, raw_o)
                np.testing.assert_array_equal(lab, oracle.argmax(raw_o))
                close(prob, prob_o)
                continue
            rscale = float(np.abs(raw_o).max()) + 1.0
            close(raw, raw_o, rtol=tol, scale=rscale)
            if kind in ("real", "discrete"):
                close(prob, prob_o, rtol=tol * max(1.0, 2.0 * rscale / (K - 1)), scale=1e-3)
                assert np.max(np.abs(raw.astype(np.float64).sum(0))) <= tol * np.abs(raw).sum(0).max()  # zero sum
            elif kind == "gbm":
                close(prob, prob_o, rtol=tol * max(1.0, 2.0 * rscale), scale=1e-3)
            else:
                close(prob, prob_o, rtol=tol)
            srt = np.sort(raw_o, axis=0)
            clear = (srt[-1] - srt[-2]) > 2 * tol * rscale if C > 1 else np.ones(n, bool)
            np.testing.assert_array_equal(lab[clear], oracle.argmax(raw_o)[clear])
        # the device member route over the same context: every member into P, then se_agg_run
        ctx.agg_configure(kid, M, K, dim, loss, n)
        width = P.shape[1]
        if width == 1:
            for t, (tr, sub) in enumerate(zip(trees, subs)):
                ctx.tree_predict(tr, N.SLOT_P, t, subspace=sub)
        else:
            ctx.alloc(N.SLOT_PROBA, K, n)
            for t, (tr, sub) in enumerate(zip(trees, subs)):
                ctx.tree_predict_multi(tr, N.SLOT_PROBA, subspace=sub)
                ctx.upload(N.SLOT_P, ctx.download(N.SLOT_PROBA).reshape(-1), offset=t * K * n)
        ctx.agg_run(w, init)
        raw_m = ctx.download(N.SLOT_RAW).reshape(C, n)
        if kind == "hard":
            np.testing.assert_array_equal(raw, raw_m)
        else:
            close(raw, raw_m, rtol=RTOL * chunks, scale=float(np.abs(raw_o).max()) + 1.0)
    finally:
        ctx.free(N.SLOT_X)
        ctx.free(N.SLOT_VX)
        ctx.free(N.SLOT_P)


@pytest.mark.gpu
def test_forest_classify_failure_modes(ctx):
    from spark_ensemble_b200 import _native as N
    rng = np.random.default_rng(7)
    n, d, K = 1000, 6, 5
    X = rng.standard_normal((n, d)).astype(np.float32)
    cand = [np.sort(rng.standard_normal(10).astype(np.float32)) for _ in range(d)]
    trees = [_random_unbalanced_tree(rng, 12, d, cand) for _ in range(4)]
    for tr in trees:
        tr["value"] = rng.integers(0, K, tr["feature"].size).astype(np.float32)
    ctx.free(N.SLOT_X)
    with pytest.raises(N.NativeError) as e:  # no feature slot
        ctx.forest_classify(trees, N.AGG_BAGGING_HARD, K)
    assert e.value.code == N.SE_ERR_STATE
    ctx.alloc(N.SLOT_X, d, n)
    ctx.upload_rowmajor(N.SLOT_X, X)
    try:
        def ok():
            ctx.forest_classify(trees, N.AGG_BAGGING_HARD, K)
            want = np.zeros((K, n))
            for tr in trees:
                want[tr["value"][_walk(tr, X)].astype(int), np.arange(n)] += 1
            np.testing.assert_array_equal(ctx.download(N.SLOT_RAW).reshape(K, n), want)

        ok()
        leaf = int(np.argmax(trees[0]["feature"] < 0))
        for bad in (K, -1, 2.5):  # label leaves must be classes
            b = dict(trees[0]); b["value"] = b["value"].copy(); b["value"][leaf] = bad
            with pytest.raises(ValueError):
                ctx.forest_classify([b] + trees[1:], N.AGG_BAGGING_HARD, K)
            ok()
        for kind in (N.AGG_GBM_REGRESSOR, N.AGG_BAGGING_REGRESSOR, N.AGG_BOOSTING_REG_MEDIAN):  # regressor kinds
            with pytest.raises(ValueError):
                ctx.forest_classify(trees, kind, K, weights=np.ones(4))
        wide = [dict(t, value=np.repeat(t["value"][:, None], 2, 1)) for t in trees]  # leaf width 2 for label leaves
        with pytest.raises(ValueError):
            ctx.forest_classify(wide, N.AGG_BAGGING_HARD, K)
        with pytest.raises(ValueError):  # probability leaves of width K for K + 1 classes
            ctx.forest_classify([dict(t, values=np.ones((t["feature"].size, K), np.float32)) for t in trees],
                                N.AGG_BAGGING_SOFT, K + 1)
        internal = int(np.argmax(trees[0]["feature"] >= 0))
        b = dict(trees[0]); b["left"] = b["left"].copy(); b["left"][internal] = internal  # its own child
        with pytest.raises(ValueError):
            ctx.forest_classify([b] + trees[1:], N.AGG_BAGGING_HARD, K)
        b = dict(trees[0]); b["feature"] = b["feature"].copy(); b["feature"][internal] = d + 3  # column outside X
        with pytest.raises(ValueError):
            ctx.forest_classify([b] + trees[1:], N.AGG_BAGGING_HARD, K)
        ok()
        many = np.sort(rng.standard_normal(400).astype(np.float32))  # > 255 thresholds in one column
        wide_col = [_random_unbalanced_tree(rng, 60, 1, [many]) for _ in range(8)]
        for tr in wide_col:
            tr["value"] = np.zeros(tr["feature"].size, np.float32)
        with pytest.raises(N.NativeError) as e:
            ctx.forest_classify(wide_col, N.AGG_BAGGING_HARD, K, subspaces=[np.array([5], np.int32)] * 8)
        assert e.value.code == N.SE_ERR_STATE
        ok()
    finally:
        ctx.free(N.SLOT_X)


def _golden(name):
    z = np.load(os.path.join(ROOT, "tests", "golden", name + ".npz"))
    return z


def _mirror_pair(model, X):
    from spark_ensemble_b200.ensemble import DataFrame
    df = DataFrame(features=X)
    base = model.copy().set("forestTransform", False).transform(df)
    fast = model.copy().set("forestTransform", True).transform(df)
    return base, fast


def _assert_classifier_outputs(base, fast, K):
    raw_b, raw_f = np.asarray(base["rawPrediction"]), np.asarray(fast["rawPrediction"])
    scale = float(np.abs(raw_b).max()) + 1.0
    close(raw_f, raw_b, rtol=RTOL * 4, scale=scale)
    close(np.asarray(fast["probability"]), np.asarray(base["probability"]), rtol=RTOL * 4 * max(1.0, 2 * scale), scale=1e-3)
    srt = np.sort(raw_b, axis=1)
    clear = (srt[:, -1] - srt[:, -2]) > 8 * RTOL * scale
    np.testing.assert_array_equal(np.asarray(fast["prediction"])[clear], np.asarray(base["prediction"])[clear])


@pytest.mark.gpu
@pytest.mark.parametrize("fixture", ["letter", "adult8k"])
def test_mirror_classifiers_forest_transform(fixture):
    from spark_ensemble_b200.classification import BaggingClassifier, BoostingClassifier, GBMClassifier
    from spark_ensemble_b200.ensemble import DataFrame
    from spark_ensemble_b200.learners import DecisionTreeClassifier, DecisionTreeRegressor, LinearRegression
    z = _golden(fixture)
    X, y = np.asarray(z["X"], np.float32)[:3000], np.asarray(z["y"], np.float64)[:3000]
    K = int(y.max()) + 1
    df = DataFrame(features=X, label=y)
    models = [
        GBMClassifier().set("baseLearner", DecisionTreeRegressor(maxDepth=4)).set("numBaseLearners", 3)
        .set("optimizedWeights", False).set("loss", "logloss" if K > 2 else "bernoulli").fit(df),
        BaggingClassifier().set("baseLearner", DecisionTreeClassifier(maxDepth=5)).set("numBaseLearners", 6)
        .set("subspaceRatio", 0.7).set("votingStrategy", "soft").fit(df),
        BaggingClassifier().set("baseLearner", DecisionTreeClassifier(maxDepth=5)).set("numBaseLearners", 6)
        .set("votingStrategy", "hard").fit(df),
        BoostingClassifier().set("baseLearner", DecisionTreeClassifier(maxDepth=3)).set("numBaseLearners", 4)
        .set("algorithm", "real").fit(df),
        BoostingClassifier().set("baseLearner", DecisionTreeClassifier(maxDepth=3)).set("numBaseLearners", 4)
        .set("algorithm", "discrete").fit(df),
    ]
    for m in models:
        base, fast = _mirror_pair(m, X)
        _assert_classifier_outputs(base, fast, K)
    # a member that is not a tree: the member route, identical output
    g = GBMClassifier().set("baseLearner", LinearRegression()).set("numBaseLearners", 2).set("optimizedWeights", False) \
        .set("loss", "logloss" if K > 2 else "bernoulli").fit(df)
    base, fast = _mirror_pair(g, X)
    for col in ("rawPrediction", "probability", "prediction"):
        np.testing.assert_array_equal(np.asarray(fast[col]), np.asarray(base[col]))


@pytest.mark.gpu
def test_mirror_regressors_forest_transform():
    from spark_ensemble_b200.ensemble import DataFrame
    from spark_ensemble_b200.learners import DecisionTreeRegressor
    from spark_ensemble_b200.regression import BaggingRegressor, GBMRegressor
    z = _golden("cpusmall")
    X, y = np.asarray(z["X"], np.float32)[:4000], np.asarray(z["y"], np.float64)[:4000]
    df = DataFrame(features=X, label=y)
    for m in (GBMRegressor().set("baseLearner", DecisionTreeRegressor(maxDepth=5)).set("numBaseLearners", 5).fit(df),
              BaggingRegressor().set("baseLearner", DecisionTreeRegressor(maxDepth=5)).set("numBaseLearners", 6)
              .set("subspaceRatio", 0.6).fit(df)):
        base, fast = _mirror_pair(m, X)
        b = np.asarray(base["prediction"])
        close(np.asarray(fast["prediction"]), b, rtol=RTOL, scale=float(np.abs(b).max()))
    # a column with more than 255 distinct thresholds: the member route, identical output
    rng = np.random.default_rng(3)
    Xw = np.concatenate([X, rng.standard_normal((X.shape[0], 1)).astype(np.float32)], axis=1)
    yw = 100.0 * Xw[:, -1] + 0.01 * y  # deep trees split the new column at far more than 255 places
    dfw = DataFrame(features=Xw, label=yw)
    m = BaggingRegressor().set("baseLearner", DecisionTreeRegressor(maxDepth=14)).set("numBaseLearners", 3).fit(dfw)
    assert len(np.unique(m.models[0].tree_arrays()["threshold"][m.models[0].tree_arrays()["feature"] == 12])) > 255
    base, fast = _mirror_pair(m, Xw)
    np.testing.assert_array_equal(np.asarray(fast["prediction"]), np.asarray(base["prediction"]))


@pytest.mark.gpu
def test_sharded_forest_classify_equals_one_context():
    from spark_ensemble_b200 import _native as N
    from spark_ensemble_b200.context import Context
    from spark_ensemble_b200.sharded import ShardedContext
    if N.device_count() < 2:
        pytest.skip("needs two GPUs")
    rng = np.random.default_rng(11)
    n, d, K = 50_001, 10, 7
    X = rng.standard_normal((n, d)).astype(np.float32)
    cand = [np.sort(rng.standard_normal(12).astype(np.float32)) for _ in range(d)]
    trees, subs = _forest(rng, "soft", K, 1, d, cand, 12)
    with Context(0) as c:
        c.alloc(N.SLOT_X, d, n)
        c.upload_rowmajor(N.SLOT_X, X)
        c.forest_classify(trees, N.AGG_BAGGING_SOFT, K, subspaces=subs)
        want = [c.download(s) for s in (N.SLOT_RAW, N.SLOT_PROB, N.SLOT_LABEL)]
    with ShardedContext([0, 1]) as sc:
        sc.gbm_configure(n, 0, 1, "squared")
        sc.alloc(N.SLOT_X, d, n)
        sc.upload_rowmajor(N.SLOT_X, X)
        sc.forest_classify(trees, N.AGG_BAGGING_SOFT, K, subspaces=subs)
        got = [sc.download(s) for s in (N.SLOT_RAW, N.SLOT_PROB, N.SLOT_LABEL)]
    for g, w in zip(got, want):
        np.testing.assert_array_equal(np.asarray(g).reshape(-1), np.asarray(w).reshape(-1))


# ------------------------------------------------------------------ CPU
@pytest.mark.parametrize("module,name", [("classification", c) for c in (
    "GBMClassifier", "GBMClassificationModel", "BaggingClassifier", "BaggingClassificationModel", "BoostingClassifier",
    "BoostingClassificationModel")] + [("regression", c) for c in (
    "GBMRegressor", "GBMRegressionModel", "BaggingRegressor", "BaggingRegressionModel")])
def test_forest_transform_param_defaults_off(module, name):
    import importlib
    cls = getattr(importlib.import_module("spark_ensemble_b200." + module), name)
    assert cls._params["forestTransform"].name == "forestTransform"
    assert cls._defaults["forestTransform"] is False


def test_forest_transform_param_is_copied_to_the_model():
    from spark_ensemble_b200.classification import BaggingClassificationModel, BaggingClassifier
    est = BaggingClassifier().set("forestTransform", True)
    m = est._copyValues(BaggingClassificationModel(2, [], []))
    assert m("forestTransform") is True


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

    def forest_classify(self, trees, kind, num_classes, **kw):
        self.calls.append(("classify", len(trees), kind, num_classes, kw.get("validation")))
        self.out = np.arange(num_classes * self.n, dtype=np.float32).reshape(num_classes, self.n) + 1000 * self.device

    def layout(self, slot):
        return self.out.shape[0], self.out.shape[1], self.out.shape[1]

    def download(self, slot, scale=None):
        return self.out.copy()


def test_sharded_forest_classify_reaches_every_shard():
    from spark_ensemble_b200 import _native as N
    from spark_ensemble_b200.ensemble import row_partition
    from spark_ensemble_b200.sharded import ShardedContext
    sc = ShardedContext([0, 1, 2], context_factory=_FakeCtx, join=False)
    n, K = 101, 3
    sc.gbm_configure(n, 0, 1, "squared")
    sc.forest_classify([{"feature": [-1]}] * 4, N.AGG_BAGGING_SOFT, K)
    assert all(c.calls == [("classify", 4, N.AGG_BAGGING_SOFT, K, False)] for c in sc.ctxs)
    raw = sc.download(N.SLOT_RAW)
    assert raw.shape == (K, n)
    for r, c in enumerate(sc.ctxs):
        s0, s1 = row_partition(n, 3, r)
        np.testing.assert_array_equal(raw[:, s0:s1], c.out)
    sc.close()


def test_gbm_classification_model_native_uses_existing_natives():
    natives = set(re.findall(r"@native def (\w+)\(", open(os.path.join(ROOT, "scala", "org", "apache", "spark", "ml", "se",
                                                                       "SeNative.scala")).read()))
    src = open(os.path.join(ROOT, "scala", "org", "apache", "spark", "ml", "classification",
                            "GBMClassificationModelNative.scala")).read()
    used = set(re.findall(r"SeNative\.(\w+)\(", src))
    assert used and used <= natives, used - natives
    for call in ("forestClassify", "uploadRowmajor", "aggConfigure", "aggRun", "download", "ctxDestroy"):
        assert call in used


def test_forest_classify_kernel_compiles_without_spills(tmp_path):
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
    found = 0
    for i, line in enumerate(lines):
        if "Function properties for" in line and "forest_classify_kernel" in line:
            found += 1
            assert "0 bytes spill stores, 0 bytes spill loads" in lines[i + 1], lines[i + 1]
            regs = int(re.search(r"Used (\d+) registers", lines[i + 2]).group(1))
            assert regs * 256 * 2 <= 65536  # two 256-thread CTAs per SM
    assert found == 3
