"""GPU parity tests: every kernel of the hot path, called through the C ABI, against the CPU oracle on
the same seeded fp32-representable inputs.  Tolerance: 1e-5 relative (north_star) on predictions and
per-iteration loss / reduction scalars; written next to each assertion.  Integer outputs are exact."""
import numpy as np
import pytest

from oracle import np_oracle as NP
from oracle import oracle as O

pytestmark = pytest.mark.gpu

RTOL = 1e-5  # north_star: fp32 predictions and per-iteration loss within 1e-5 relative
PARAM = {"huber": 0.9, "quantile": 0.9, "scaledlogcosh": 0.9}
SCALAR = ["squared", "absolute", "huber", "quantile", "logcosh", "scaledlogcosh", "bernoulli",
          "exponential"]
HESS = ["squared", "logcosh", "scaledlogcosh", "bernoulli", "exponential"]


@pytest.fixture(scope="module")
def ctx():
    from spark_ensemble_b200.context import Context
    c = Context(0)
    yield c
    c.close()


def f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def labels(name, rng, n, K=5):
    if name in ("bernoulli", "exponential"):
        return f32(rng.random(n) < 0.4)
    if name == "logloss":
        return f32(rng.integers(0, K, n))
    return f32(rng.standard_normal(n))


def close(a, b, rtol=RTOL, scale=None):
    """|a-b| <= rtol * max(|b|, scale) elementwise; scale defaults to the rms magnitude of b."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    if scale is None:
        scale = float(np.sqrt(np.mean(b * b))) if b.size else 1.0
    tol = rtol * np.maximum(np.abs(b), scale)
    bad = np.abs(a - b) > tol
    assert not bad.any(), (f"{bad.sum()} / {b.size} mismatches; worst rel "
                           f"{np.max(np.abs(a - b) / np.maximum(np.abs(b), scale)):.3e}")


def setup_gbm(ctx, rng, name, n, weighted=False, K=5, nv=0):
    from spark_ensemble_b200 import _native as N
    dim = K if name == "logloss" else 1
    par = PARAM.get(name, 0.0)
    y = labels(name, rng, n, K)
    F = f32(rng.standard_normal((dim, n)) * 0.7)
    h = f32(rng.standard_normal((dim, n)))
    w = f32(rng.random(n) + 0.5) if weighted else None
    ctx.gbm_configure(n, nv, dim, name, par, weighted)
    ctx.upload(N.SLOT_Y, y)
    ctx.upload(N.SLOT_F, F)
    ctx.upload(N.SLOT_H, h)
    if weighted:
        ctx.upload(N.SLOT_W, w)
    return dim, par, y, F, h, w


@pytest.mark.parametrize("name", SCALAR + ["logloss"])
@pytest.mark.parametrize("n,weighted", [(1, False), (3, True), (1023, False), (40961, True)])
def test_linesearch_eval(ctx, oracle, rng, name, n, weighted):
    dim, par, y, F, h, w = setup_gbm(ctx, rng, name, n, weighted)
    for alpha in (np.ones(dim), rng.random(dim) * 3.0, np.zeros(dim)):
        lg, gg = ctx.gbm_linesearch_eval(alpha)
        lo, go = oracle.linesearch_eval(O.LOSS_IDS[name], par, y, w, F, h, alpha)
        assert lg == pytest.approx(lo, rel=RTOL, abs=1e-7)
        scale = float(np.mean(np.abs(h))) * 1e-1  # gradient sums cancel: scale by typical |h·g|/n
        close(gg, go, rtol=RTOL, scale=max(scale, float(np.max(np.abs(go)))))


@pytest.mark.parametrize("name", SCALAR + ["logloss"])
@pytest.mark.parametrize("K", [2, 3, 7, 13, 26, 32])
def test_pseudo_residuals_gradient(ctx, oracle, rng, name, K):
    from spark_ensemble_b200 import _native as N
    if name != "logloss" and K != 2:
        pytest.skip("K only varies for logloss")
    n = 5003
    dim, par, y, F, h, w = setup_gbm(ctx, rng, name, n, False, K=K)
    ctx.gbm_pseudo_residuals(newton=False)
    r = ctx.download(N.SLOT_R).reshape(dim, n)
    ro, _, _ = oracle.pseudo_residuals(O.LOSS_IDS[name], par, dim, y, None, F, False)
    close(r, ro, rtol=RTOL, scale=1.0)


@pytest.mark.parametrize("name", HESS + ["logloss"])
@pytest.mark.parametrize("weighted", [False, True])
def test_pseudo_residuals_newton(ctx, oracle, rng, name, weighted):
    from spark_ensemble_b200 import _native as N
    n, K = 4099, 6
    dim, par, y, F, h, w = setup_gbm(ctx, rng, name, n, weighted, K=K)
    S = ctx.gbm_pseudo_residuals(newton=True)
    r = ctx.download(N.SLOT_R).reshape(dim, n)
    wo = ctx.download(N.SLOT_WOUT).reshape(dim, n)
    ro, woo, So = oracle.pseudo_residuals(O.LOSS_IDS[name], par, dim, y, w, F, True)
    close(S, So, rtol=RTOL)
    close(r, ro, rtol=RTOL, scale=1.0)
    close(wo, woo, rtol=RTOL)


def test_newton_rejected_without_hessian(ctx, rng):
    setup_gbm(ctx, rng, "absolute", 64)
    with pytest.raises(ValueError):
        ctx.gbm_pseudo_residuals(newton=True)


@pytest.mark.parametrize("name", SCALAR + ["logloss"])
@pytest.mark.parametrize("mode", ["plain", "residual", "newton"])
def test_update_fused(ctx, oracle, rng, name, mode):
    """K1: F' = F + step·h fused with next-round residual and Σloss(F')."""
    from spark_ensemble_b200 import _native as N
    if mode == "newton" and name not in HESS + ["logloss"]:
        pytest.skip("no hessian")
    n, K = 30011, 4
    dim, par, y, F, h, w = setup_gbm(ctx, rng, name, n, mode == "newton", K=K)
    step = rng.random(dim) * 0.8 + 0.1
    ls, S = ctx.gbm_update(step, residual=(mode == "residual"), newton=(mode == "newton"), loss=True)
    Fg = ctx.download(N.SLOT_F).reshape(dim, n)
    Fo = F.astype(np.float64).copy()
    oracle.update(Fo, h, step)
    close(Fg, Fo, rtol=RTOL)  # predictions within 1e-5 relative
    lid = O.LOSS_IDS[name]
    assert ls / n == pytest.approx(oracle.mean_loss(lid, par, dim, y, Fo), rel=RTOL, abs=1e-7)
    if mode != "plain":
        ro, woo, So = oracle.pseudo_residuals(lid, par, dim, y, w, Fo, mode == "newton")
        close(ctx.download(N.SLOT_R).reshape(dim, n), ro, rtol=RTOL, scale=1.0)
        if mode == "newton":
            close(S, So, rtol=RTOL)
            close(ctx.download(N.SLOT_WOUT).reshape(dim, n), woo, rtol=RTOL)


def test_mean_loss_and_validation(ctx, oracle, rng):
    from spark_ensemble_b200 import _native as N
    n, nv = 7001, 1999
    for name in ("squared", "bernoulli", "logloss"):
        dim, par, y, F, h, w = setup_gbm(ctx, rng, name, n, False, K=3, nv=nv)
        vy = labels(name, rng, nv, 3)
        vF = f32(rng.standard_normal((dim, nv)))
        vh = f32(rng.standard_normal((dim, nv)))
        ctx.upload(N.SLOT_VY, vy); ctx.upload(N.SLOT_VF, vF); ctx.upload(N.SLOT_VH, vh)
        lid = O.LOSS_IDS[name]
        assert ctx.gbm_mean_loss(False) == pytest.approx(oracle.mean_loss(lid, par, dim, y, F), rel=RTOL)
        assert ctx.gbm_mean_loss(True) == pytest.approx(oracle.mean_loss(lid, par, dim, vy, vF), rel=RTOL)
        step = rng.random(dim)
        lv = ctx.gbm_update_validation(step)
        vFo = vF.astype(np.float64).copy()
        oracle.update(vFo, vh, step)
        assert lv == pytest.approx(oracle.mean_loss(lid, par, dim, vy, vFo), rel=RTOL)
        close(ctx.download(N.SLOT_VF).reshape(dim, nv), vFo)


def test_squared_stats_brent_and_async_round(ctx, oracle, rng):
    from spark_ensemble_b200 import _native as N
    n = 100003
    dim, par, y, F, h, w = setup_gbm(ctx, rng, "squared", n, True)
    h = f32((y - F[0]) * 0.6 + 0.2 * rng.standard_normal(n)).reshape(1, n)
    ctx.upload(N.SLOT_H, h)
    s = ctx.gbm_linesearch_stats()
    d = (y.astype(np.float64) - F[0]); hh = h[0].astype(np.float64)
    close(s, [np.sum(d * d), np.sum(hh * d), np.sum(hh * hh), np.sum(w.astype(np.float64))], rtol=RTOL)
    # native Brent over the one-pass parabola == oracle Brent over full-pass evaluations
    a, l, ne = ctx.gbm_linesearch_brent()
    f = lambda x: oracle.linesearch_eval(O.SQUARED, 0.0, y, w, F, h, [x])[0]
    ao, neo, st = oracle.brent(f)
    assert st == 0
    assert a == pytest.approx(ao, rel=1e-5, abs=2e-6)  # optimiser tolerance tol=1e-6
    assert l == pytest.approx(f(ao), rel=RTOL)
    # device-resident round: closed-form alpha, no host round trip
    ctx.gbm_configure(n, 0, 1, "squared", 0.0, False)
    ctx.upload(N.SLOT_Y, y); ctx.upload(N.SLOT_F, F); ctx.upload(N.SLOT_H, h)
    ctx.gbm_round_squared_async(0.5)
    alpha, loss_sum = ctx.gbm_round_result()
    star = float(np.clip(np.sum(hh * d) / np.sum(hh * hh), 0, 100))
    assert alpha == pytest.approx(star, rel=RTOL)
    Fo = F.astype(np.float64).copy()
    oracle.update(Fo, h, [0.5 * star])
    close(ctx.download(N.SLOT_F), Fo[0])
    assert loss_sum / n == pytest.approx(oracle.mean_loss(O.SQUARED, 0.0, 1, y, Fo), rel=RTOL)
    ro, _, _ = oracle.pseudo_residuals(O.SQUARED, 0.0, 1, y, None, Fo, False)
    close(ctx.download(N.SLOT_R), ro[0], scale=1.0)


@pytest.mark.parametrize("name", ["bernoulli", "absolute", "logcosh"])
def test_native_brent_line_search(ctx, oracle, rng, name):
    from spark_ensemble_b200 import _native as N
    n = 20011
    dim, par, y, F, h, w = setup_gbm(ctx, rng, name, n)
    lid = O.LOSS_IDS[name]
    r, _, _ = oracle.pseudo_residuals(lid, par, 1, y, None, F, False)
    h = f32(r * 0.8 + 0.1 * rng.standard_normal((1, n)))
    ctx.upload(N.SLOT_H, h)
    a, l, ne = ctx.gbm_linesearch_brent()
    f = lambda x: oracle.linesearch_eval(lid, par, y, None, F, h, [x])[0]
    ao, neo, st = oracle.brent(f)
    assert st == 0 and 3 <= ne <= 100
    # the minimiser is defined to optimiser tolerance; the objective value is the parity quantity
    assert l == pytest.approx(f(ao), rel=RTOL)
    assert f(a) <= f(ao) * (1 + 1e-5)


def test_multi_round_drift(ctx, oracle, rng):
    """200 fused rounds of fp32 state against the fp64 oracle: predictions and per-iteration loss stay
    within 1e-5 relative (SURVEY.md §7 'hard parts')."""
    from spark_ensemble_b200 import _native as N
    n = 20000
    for name in ("squared", "bernoulli"):
        dim, par, y, F, h, w = setup_gbm(ctx, rng, name, n)
        lid = O.LOSS_IDS[name]
        Fo = F.astype(np.float64).copy()
        worst = 0.0
        for t in range(200):
            ro, _, _ = oracle.pseudo_residuals(lid, par, 1, y, None, Fo, False)
            ht = f32(ro * 0.5 + 0.05 * rng.standard_normal((1, n)))
            ctx.upload(N.SLOT_H, ht)
            step = 0.1
            ls, _ = ctx.gbm_update([step], residual=True, loss=True)
            oracle.update(Fo, ht, [step])
            lo = oracle.mean_loss(lid, par, 1, y, Fo)
            worst = max(worst, abs(ls / n - lo) / lo)
        assert worst < RTOL, worst
        close(ctx.download(N.SLOT_F), Fo[0])


# ------------------------------------------------------------------ BoostingClassifier
@pytest.mark.parametrize("K", [2, 3, 5, 9, 26])
@pytest.mark.parametrize("n", [2, 255, 256, 257, 4097, 50001])
def test_samme_r_update(ctx, oracle, rng, K, n):
    """K < 5: register-streaming kernel; K >= 5: TMA-tiled kernel (256-row tiles, tails included)."""
    from spark_ensemble_b200 import _native as N
    y = f32(rng.integers(0, K, n))
    Z = rng.standard_normal((K, n))
    Z[y.astype(int), np.arange(n)] += 2.0
    P = f32(NP.softmax_cols(Z))
    P[0, : min(n, 5)] = 0.0  # exercises max(p, EPSILON)
    w = f32(rng.random(n) + 0.1)
    ctx.boost_configure(n, K, True)
    ctx.upload(N.SLOT_Y, y); ctx.upload(N.SLOT_BW, w); ctx.upload(N.SLOT_PROBA, P)
    sw = ctx.slot_sum(N.SLOT_BW)
    assert sw == pytest.approx(oracle.sum(w), rel=1e-12)  # fp64 accumulation of fp32 values
    e, s = ctx.boost_real_update(sw)
    out, eo, so = oracle.samme_r_update(K, y, w, sw, P)
    assert e == pytest.approx(eo, rel=RTOL, abs=1e-9)
    assert s == pytest.approx(so, rel=RTOL)
    close(ctx.download(N.SLOT_BW), out, rtol=RTOL, scale=float(np.min(out)))


def test_samme_discrete(ctx, oracle, rng):
    from spark_ensemble_b200 import _native as N
    n, K = 33333, 7
    y = f32(rng.integers(0, K, n))
    pred = f32(np.where(rng.random(n) < 0.7, y, rng.integers(0, K, n)))
    w = f32(rng.random(n))
    ctx.boost_configure(n, K, False)
    ctx.upload(N.SLOT_Y, y); ctx.upload(N.SLOT_BW, w); ctx.upload(N.SLOT_PRED, pred)
    sw = ctx.slot_sum(N.SLOT_BW)
    e = ctx.boost_discrete_error(sw)
    eo = oracle.samme_error(y, w, sw, pred)
    assert e == pytest.approx(eo, rel=RTOL)
    beta = eo / ((1 - eo) * (K - 1))
    s = ctx.boost_discrete_update(sw, beta)
    out, so = oracle.samme_update(y, w, sw, pred, beta)
    assert s == pytest.approx(so, rel=RTOL)
    close(ctx.download(N.SLOT_BW), out, rtol=RTOL, scale=1e-12)


# ------------------------------------------------------------------ aggregation
@pytest.mark.parametrize("M,n", [(1, 5), (10, 4099), (512, 2051)])
def test_agg_regressors(ctx, oracle, rng, M, n):
    from spark_ensemble_b200 import _native as N
    P = f32(rng.standard_normal((M, n)) + 3.0)
    a = rng.random(M)
    ctx.agg_configure(N.AGG_GBM_REGRESSOR, M, 0, 1, 0, n)
    ctx.upload(N.SLOT_P, P)
    ctx.agg_run(a, [0.25])
    close(ctx.download(N.SLOT_RAW), oracle.agg_weighted_sum(P, a.astype(np.float32).astype(np.float64), 0.25))
    ctx.agg_configure(N.AGG_BAGGING_REGRESSOR, M, 0, 1, 0, n)
    ctx.upload(N.SLOT_P, P)
    ctx.agg_run()
    close(ctx.download(N.SLOT_RAW), oracle.agg_mean(P))


@pytest.mark.parametrize("loss,dim,K", [("bernoulli", 1, 2), ("exponential", 1, 2), ("logloss", 2, 2),
                                        ("logloss", 5, 5), ("logloss", 26, 26)])
def test_agg_gbm_classifier(ctx, oracle, rng, loss, dim, K):
    from spark_ensemble_b200 import _native as N
    M, n = 9, 3001
    P = f32(rng.standard_normal((M, dim, n)))
    a = f32(rng.random((M, dim))).astype(np.float64)
    init = f32(rng.standard_normal(dim)).astype(np.float64)
    ctx.agg_configure(N.AGG_GBM_CLASSIFIER, M, K, dim, loss, n)
    ctx.upload(N.SLOT_P, P)
    ctx.agg_run(a, init)
    raw = oracle.agg_gbm_classifier_raw(P, a, init, K)
    close(ctx.download(N.SLOT_RAW), raw, scale=1.0)
    close(ctx.download(N.SLOT_PROB), oracle.gbm_raw2prob(O.LOSS_IDS[loss], raw), scale=1e-3)
    lab = ctx.download(N.SLOT_LABEL)
    srt = np.sort(raw, axis=0)
    clear = (srt[-1] - srt[-2]) > 1e-4  # argmax is only defined up to fp32 ties
    np.testing.assert_array_equal(lab[clear], oracle.argmax(raw)[clear])


@pytest.mark.parametrize("K", [2, 26])
def test_agg_bagging_classifier(ctx, oracle, rng, K):
    from spark_ensemble_b200 import _native as N
    M, n = 11, 2999
    Pk = f32(rng.random((M, K, n)))
    ctx.agg_configure(N.AGG_BAGGING_SOFT, M, K, 1, 0, n)
    ctx.upload(N.SLOT_P, Pk)
    ctx.agg_run()
    raw, prob = oracle.agg_bagging_soft(Pk)
    close(ctx.download(N.SLOT_RAW), raw)
    close(ctx.download(N.SLOT_PROB), prob)
    votes = f32(rng.integers(0, K, (M, n)))
    ctx.agg_configure(N.AGG_BAGGING_HARD, M, K, 1, 0, n)
    ctx.upload(N.SLOT_P, votes)
    ctx.agg_run()
    raw, prob = oracle.agg_bagging_hard(votes, K)
    np.testing.assert_array_equal(ctx.download(N.SLOT_RAW), raw)  # vote counts: exact
    close(ctx.download(N.SLOT_PROB), prob)
    np.testing.assert_array_equal(ctx.download(N.SLOT_LABEL), oracle.argmax(raw))


@pytest.mark.parametrize("K", [2, 5, 26])
def test_agg_boosting_classifier_and_zero_sum(ctx, oracle, rng, K):
    """Parity + the reference's invariant (BoostingClassifierSuite.scala:126-154): rawPrediction rows
    sum to 0 (here to fp32 rounding of the row's magnitude)."""
    from spark_ensemble_b200 import _native as N
    M, n = 7, 2500
    P = f32(NP.softmax_cols(rng.standard_normal((M * K, n)).reshape(M, K, n).reshape(M * K, n)).reshape(M, K, n))
    P = f32(P / P.sum(axis=1, keepdims=True))
    ctx.agg_configure(N.AGG_BOOSTING_REAL, M, K, 1, 0, n)
    ctx.upload(N.SLOT_P, P)
    ctx.agg_run()
    raw, prob = oracle.agg_boosting_real(P)
    g = ctx.download(N.SLOT_RAW)
    close(g, raw, scale=float(np.abs(raw).max()))
    assert np.max(np.abs(g.sum(axis=0))) <= 1e-5 * np.abs(g).sum(axis=0).max()
    close(ctx.download(N.SLOT_PROB), prob, scale=1e-3)
    votes = f32(rng.integers(0, K, (M, n)))
    a = f32(rng.random(M) + 0.1).astype(np.float64)
    ctx.agg_configure(N.AGG_BOOSTING_DISCRETE, M, K, 1, 0, n)
    ctx.upload(N.SLOT_P, votes)
    ctx.agg_run(a)
    raw, prob = oracle.agg_boosting_discrete(votes, a, K)
    g = ctx.download(N.SLOT_RAW)
    close(g, raw, scale=float(np.abs(raw).max()))
    assert np.max(np.abs(g.sum(axis=0))) <= 1e-5 * np.abs(g).sum(axis=0).max()
    close(ctx.download(N.SLOT_PROB), prob, scale=1e-3)


@pytest.mark.parametrize("n", [1, 255, 256, 257, 1030])
@pytest.mark.parametrize("M,K", [(1, 2), (40, 2), (5, 7), (70, 3), (3, 40)])
def test_agg_classifier_shapes(ctx, oracle, rng, n, M, K):
    """Every classifier aggregation kind over awkward shapes: single rows, 4-row group tails, one model, more models
    than one load batch, binary and > 32 classes.

    Probabilities are soft-maxes of raw/(K-1): a raw vector that matches to RTOL·max|raw| (the fp32 output format
    cannot do better) pins them to 2·RTOL·max|raw|/(K-1) relative, which is the tolerance used for them here."""
    def ptol(raw):
        return RTOL * max(1.0, 2.0 * float(np.abs(raw).max()) / (K - 1))

    from spark_ensemble_b200 import _native as N
    Pk = f32(rng.random((M, K, n)) + 0.01)
    Pk = f32(Pk / Pk.sum(axis=1, keepdims=True))
    ctx.agg_configure(N.AGG_BAGGING_SOFT, M, K, 1, 0, n)
    ctx.upload(N.SLOT_P, Pk)
    ctx.agg_run()
    raw, prob = oracle.agg_bagging_soft(Pk)
    close(ctx.download(N.SLOT_RAW).reshape(K, n), raw)
    close(ctx.download(N.SLOT_PROB).reshape(K, n), prob)
    ctx.agg_configure(N.AGG_BOOSTING_REAL, M, K, 1, 0, n)
    ctx.upload(N.SLOT_P, Pk)
    ctx.agg_run()
    raw, prob = oracle.agg_boosting_real(Pk)
    close(ctx.download(N.SLOT_RAW).reshape(K, n), raw, scale=float(np.abs(raw).max()))
    close(ctx.download(N.SLOT_PROB).reshape(K, n), prob, rtol=ptol(raw), scale=1e-3)
    votes = f32(rng.integers(0, K, (M, n)))
    a = f32(rng.random(M) + 0.1).astype(np.float64)
    ctx.agg_configure(N.AGG_BAGGING_HARD, M, K, 1, 0, n)
    ctx.upload(N.SLOT_P, votes)
    ctx.agg_run()
    raw, prob = oracle.agg_bagging_hard(votes, K)
    np.testing.assert_array_equal(ctx.download(N.SLOT_RAW).reshape(K, n), raw)
    np.testing.assert_array_equal(ctx.download(N.SLOT_LABEL), oracle.argmax(raw))
    ctx.agg_configure(N.AGG_BOOSTING_DISCRETE, M, K, 1, 0, n)
    ctx.upload(N.SLOT_P, votes)
    ctx.agg_run(a)
    raw, prob = oracle.agg_boosting_discrete(votes, a, K)
    close(ctx.download(N.SLOT_RAW).reshape(K, n), raw, scale=float(np.abs(raw).max()))
    close(ctx.download(N.SLOT_PROB).reshape(K, n), prob, rtol=ptol(raw), scale=1e-3)
    dim = K
    P = f32(rng.standard_normal((M, dim, n)))
    aw = f32(rng.random((M, dim))).astype(np.float64)
    init = f32(rng.standard_normal(dim)).astype(np.float64)
    ctx.agg_configure(N.AGG_GBM_CLASSIFIER, M, K, dim, O.LOSS_IDS["logloss"], n)
    ctx.upload(N.SLOT_P, P)
    ctx.agg_run(aw, init)
    raw = oracle.agg_gbm_classifier_raw(P, aw, init, K)
    close(ctx.download(N.SLOT_RAW).reshape(dim, n), raw, scale=1.0)
    close(ctx.download(N.SLOT_PROB).reshape(dim, n), oracle.gbm_raw2prob(O.LOSS_IDS["logloss"], raw),
          rtol=RTOL * max(1.0, 2.0 * float(np.abs(raw).max())), scale=1e-3)

# ------------------------------------------------------------------ on-device base models
def test_tree_and_linear_predict(ctx, rng):
    from sklearn.tree import DecisionTreeRegressor
    from spark_ensemble_b200 import _native as N
    n, d = 10007, 12
    X = f32(rng.standard_normal((n, d)))
    yv = X[:, 0] * 2 + np.sin(X[:, 3]) + 0.1 * rng.standard_normal(n)
    sub = np.array([0, 2, 3, 5, 7, 11], dtype=np.int32)
    t = DecisionTreeRegressor(max_depth=6, random_state=0).fit(X[:, sub], yv)
    tr = t.tree_
    tree = {"feature": np.where(tr.children_left < 0, -1, tr.feature), "threshold": tr.threshold,
            "left": np.maximum(tr.children_left, 0), "right": np.maximum(tr.children_right, 0),
            "value": tr.value.reshape(-1)}
    ctx.alloc(N.SLOT_X, d, n)
    ctx.upload(N.SLOT_X, np.ascontiguousarray(X.T))
    ctx.alloc(N.SLOT_H, 1, n)
    ctx.tree_predict(tree, N.SLOT_H, 0, subspace=sub)
    # sklearn thresholds are fp64 midpoints; the fp32 rounding of a threshold can only flip rows whose
    # feature equals it to ~1 ulp — none with continuous random data
    np.testing.assert_allclose(ctx.download(N.SLOT_H), t.predict(X[:, sub]).astype(np.float32), rtol=1e-6)
    coef = f32(rng.standard_normal(len(sub)))
    ctx.linear_predict(coef, 0.5, N.SLOT_H, 0, subspace=sub)
    ref = 0.5 + X[:, sub].astype(np.float64) @ coef.astype(np.float64)
    close(ctx.download(N.SLOT_H), ref, scale=1.0)


def test_synthetic_fill_statistics(ctx):
    from spark_ensemble_b200 import _native as N
    n = 1 << 20
    ctx.alloc(N.SLOT_Y, n)
    ctx.fill_synthetic(N.SLOT_Y, "normal", 7, 1.0, 2.0)
    v = ctx.download(N.SLOT_Y).astype(np.float64)
    assert abs(v.mean() - 1.0) < 0.01 and abs(v.std() - 2.0) < 0.01
    ctx.fill_synthetic(N.SLOT_Y, "randint", 8, 0, 26)
    v = ctx.download(N.SLOT_Y)
    assert v.min() == 0 and v.max() == 25 and np.all(v == np.floor(v))
    ctx.fill_synthetic(N.SLOT_Y, "bernoulli", 9, 0.3, 0)
    assert abs(ctx.download(N.SLOT_Y).mean() - 0.3) < 0.01
    # chunked fills are index-addressed: same stream regardless of how the range is split
    ctx.fill_synthetic(N.SLOT_Y, "uniform", 10, 0, 1)
    whole = ctx.download(N.SLOT_Y).copy()
    ctx.fill_synthetic(N.SLOT_Y, "uniform", 10, 0, 1, count=1000, offset=0)
    ctx.fill_synthetic(N.SLOT_Y, "uniform", 10, 0, 1, count=n - 1000, offset=1000)
    np.testing.assert_array_equal(ctx.download(N.SLOT_Y), whole)


def test_multi_gpu_sharded_parity():
    """Row-sharded run over NCCL (one rank per GPU, torchrun): skipped on single-GPU boxes."""
    import os
    import subprocess
    import sys
    from spark_ensemble_b200 import _native as N
    g = N.device_count()
    if g < 2:
        pytest.skip("needs >= 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    world = 2
    # once with the fused peer-memory all-reduce (default), once forcing the NCCL fallback
    for port, p2p in ((29533, "1"), (29537, "0")):
        env = dict(os.environ, SE_P2P_ALLREDUCE=p2p, SE_REQUIRE_P2P="1")
        out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
                              "--master-addr", "127.0.0.1", "--master-port", str(port),
                              os.path.join(root, "tests", "mgpu_check.py")], capture_output=True, text=True,
                             timeout=600, env=env)
        assert out.returncode == 0 and "MGPU_PARITY_OK" in out.stdout, out.stdout[-2000:] + out.stderr[-4000:]
        assert f"p2p_allreduce={p2p == '1'}" in out.stdout


def test_bench_dump_outputs_repeat(tmp_path):
    """`bench.py --dump-outputs`: the last timed round's outputs over a seeded row sample, fp32 / fp64, within the
    64 MB budget, and the same from one run to the next (the inputs are seeded)."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    n, steps = 3_000_001, 2
    dumps = []
    for run in range(2):
        d = tmp_path / f"run{run}"
        out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--steps", str(steps), "--warmup", "3",
                              "--rows", str(n), "--no-features", "--no-extras", "--no-parity", "--strong-rows", "0",
                              "--cpu-rows", "20000", "--dump-outputs", str(d)], capture_output=True, text=True,
                             timeout=600)
        assert out.returncode == 0, out.stderr[-4000:]
        res = json.loads(out.stdout.strip().splitlines()[-1])
        assert res["steps"] == steps and res["value"] > 0
        files = sorted(os.listdir(d))
        assert files == sorted(f"{k}.npy" for k in ("alpha", "loss_sum", "brent_evals", "row_index", "F", "r"))
        assert sum(os.path.getsize(d / f) for f in files) <= 64 << 20
        dumps.append({f[:-4]: np.load(d / f) for f in files})
    a, b = dumps
    for k, v in a.items():
        assert v.dtype in (np.float32, np.float64), k
    idx = a["row_index"]
    assert idx.size == 1 << 21 and np.all(np.diff(idx) > 0) and idx[-1] < n and np.all(idx == np.floor(idx))
    assert a["F"].shape == a["r"].shape == idx.shape and np.all(np.isfinite(a["F"])) and np.all(np.isfinite(a["r"]))
    assert a["alpha"][0] > 0 and a["loss_sum"][0] > 0 and a["brent_evals"][0] >= 1
    np.testing.assert_array_equal(a["row_index"], b["row_index"])
    for k in ("alpha", "loss_sum", "F", "r"):
        np.testing.assert_allclose(a[k], b[k], rtol=RTOL, atol=RTOL * float(np.abs(a[k]).max()), err_msg=k)


@pytest.mark.parametrize("K", [9, 26, 32, 33, 64, 65, 200, 1000])
@pytest.mark.parametrize("n", [1, 127, 129, 255, 256, 257, 40961])
def test_logloss_wide_k_tiled_kernels(ctx, oracle, rng, K, n):
    """LogLoss with K >= 5 runs through the TMA-tiled kernels (se_gbm_tiled.cu, 256-row tiles): every mode,
    tile tails included."""
    from spark_ensemble_b200 import _native as N
    dim, par, y, F, h, w = setup_gbm(ctx, rng, "logloss", n, True, K=K)
    lid = O.LOGLOSS
    alpha = rng.random(K) * 2.0
    lg, gg = ctx.gbm_linesearch_eval(alpha)
    lo, go = oracle.linesearch_eval(lid, 0.0, y, w, F, h, alpha)
    assert lg == pytest.approx(lo, rel=RTOL)
    close(gg, go, rtol=RTOL, scale=float(np.max(np.abs(go))))
    assert ctx.gbm_mean_loss(False) == pytest.approx(oracle.mean_loss(lid, 0.0, K, y, F), rel=RTOL)
    S = ctx.gbm_pseudo_residuals(newton=True)
    ro, woo, So = oracle.pseudo_residuals(lid, 0.0, K, y, w, F, True)
    close(S, So, rtol=RTOL)
    close(ctx.download(N.SLOT_R).reshape(K, n), ro, rtol=RTOL, scale=1.0)
    close(ctx.download(N.SLOT_WOUT).reshape(K, n), woo, rtol=RTOL)
    ctx.gbm_pseudo_residuals(newton=False)
    rg, _, _ = oracle.pseudo_residuals(lid, 0.0, K, y, None, F, False)
    close(ctx.download(N.SLOT_R).reshape(K, n), rg, rtol=RTOL, scale=1.0)
    step = rng.random(K) * 0.5
    for mode in ("residual", "newton", "plain"):
        ls, S = ctx.gbm_update(step, residual=(mode == "residual"), newton=(mode == "newton"), loss=True)
        Fo = F.astype(np.float64).copy() if mode == "residual" else Fo
        oracle.update(Fo, h, step)
        close(ctx.download(N.SLOT_F).reshape(K, n), Fo, rtol=RTOL, scale=1.0)
        assert ls / n == pytest.approx(oracle.mean_loss(lid, 0.0, K, y, Fo), rel=RTOL, abs=1e-7)
        if mode != "plain":
            ro, woo, So = oracle.pseudo_residuals(lid, 0.0, K, y, w, Fo, mode == "newton")
            close(ctx.download(N.SLOT_R).reshape(K, n), ro, rtol=RTOL, scale=1.0)
            if mode == "newton":
                close(S, So, rtol=RTOL)
                close(ctx.download(N.SLOT_WOUT).reshape(K, n), woo, rtol=RTOL)


def test_abi_utilities(ctx, rng):
    """Slots, uploads (fp32/fp64, logical offsets over padded rows), scaled download, copy, fill, timers,
    launch counter, error paths: every remaining exported entry point is exercised."""
    from spark_ensemble_b200 import _native as N
    n, rows = 1003, 3
    ctx.alloc(N.SLOT_P, rows, n)
    r, c, ld = ctx.layout(N.SLOT_P)
    assert (r, c) == (rows, n) and ld % 32 == 0 and ld >= n  # padded, 128-byte aligned rows
    a = f32(rng.standard_normal((rows, n)))
    ctx.upload(N.SLOT_P, a)
    np.testing.assert_array_equal(ctx.download(N.SLOT_P), a)
    # logical offsets crossing a row boundary
    patch = f32(rng.standard_normal(50))
    ctx.upload(N.SLOT_P, patch, offset=n - 20)
    a.reshape(-1)[n - 20:n + 30] = patch
    np.testing.assert_array_equal(ctx.download(N.SLOT_P), a)
    np.testing.assert_array_equal(ctx.download(N.SLOT_P, count=100, offset=2 * n - 50), a.reshape(-1)[2 * n - 50:2 * n + 50])
    # fp64 upload narrows on the host
    d = rng.standard_normal(n)
    ctx.alloc(N.SLOT_Y, n)
    ctx.upload(N.SLOT_Y, d)
    np.testing.assert_array_equal(ctx.download(N.SLOT_Y), d.astype(np.float32))
    np.testing.assert_allclose(ctx.download(N.SLOT_Y, scale=0.25), d.astype(np.float32) * np.float32(0.25), rtol=1e-7)
    ctx.alloc(N.SLOT_W, n)
    ctx.copy_slot(N.SLOT_W, N.SLOT_Y)
    np.testing.assert_array_equal(ctx.download(N.SLOT_W), d.astype(np.float32))
    ctx.fill(N.SLOT_W, 2.5, 10, 5)
    w = ctx.download(N.SLOT_W)
    assert np.all(w[5:15] == 2.5) and w[4] == np.float32(d[4]) and w[15] == np.float32(d[15])
    assert ctx.slot_sum(N.SLOT_W) == pytest.approx(float(np.sum(w.astype(np.float64))), rel=1e-12)
    # timers and counters
    before = ctx.launch_count
    ctx.timer_start()
    ctx.fill(N.SLOT_W, 1.0)
    ms = ctx.timer_stop()
    assert ms >= 0.0 and ctx.launch_count == before + 1
    ctx.kernel_timing(True); ctx.kernel_times_reset()
    ctx.slot_sum(N.SLOT_W)
    ctx.kernel_timing(False)
    assert ctx.comm_info() == (1, 0)
    np.testing.assert_array_equal(ctx.allreduce_host([1.0, 2.0]), [1.0, 2.0])  # no communicator: identity
    # error paths: bad slot, range outside slot, state errors -> exceptions, never a crash
    with pytest.raises(ValueError):
        ctx.alloc(99, 4)
    with pytest.raises(ValueError):
        ctx.upload(N.SLOT_W, np.zeros(n + 1, dtype=np.float32))
    ctx.free(N.SLOT_VY)
    with pytest.raises(N.NativeError):
        ctx.download(N.SLOT_VY, count=1)
    with pytest.raises(ValueError):
        ctx.gbm_configure(10, 0, 3, "squared")  # scalar losses have dim 1
    ctx.gbm_configure(10, 0, 65, "logloss")  # beyond 64 classes: the general kernels (no cap short of 16384)
    with pytest.raises(ValueError):
        ctx.gbm_configure(10, 0, 20000, "logloss")


@pytest.mark.parametrize("loss_type", ["exponential", "linear", "squared"])
@pytest.mark.parametrize("n", [3, 4097, 60001])
def test_adaboost_r2_kernels(ctx, oracle, rng, loss_type, n):
    """BoostingRegressor (AdaBoost.R2) weight recursion, SURVEY.md §8f-2."""
    from spark_ensemble_b200 import _native as N
    y = f32(rng.standard_normal(n))
    pred = f32(y + 0.4 * rng.standard_normal(n))
    w = f32(rng.random(n) + 0.1)
    ctx.boostreg_configure(n)
    ctx.upload(N.SLOT_Y, y); ctx.upload(N.SLOT_PRED, pred); ctx.upload(N.SLOT_BW, w)
    sw = ctx.slot_sum(N.SLOT_BW)
    mx = ctx.boostreg_max_error()
    assert mx == pytest.approx(oracle.r2_max_error(y, pred), rel=1e-6)  # fp32 subtraction rounds once
    e = ctx.boostreg_error(sw, loss_type, mx)
    eo = oracle.r2_estimator_error(loss_type, y, pred, w, sw, mx)
    assert e == pytest.approx(eo, rel=RTOL)
    beta = eo / (1 - eo)
    s = ctx.boostreg_update(sw, loss_type, mx, beta)
    out, so = oracle.r2_update(loss_type, y, pred, w, sw, mx, beta)
    assert s == pytest.approx(so, rel=RTOL)
    close(ctx.download(N.SLOT_BW), out, rtol=RTOL, scale=float(np.min(out)))
    # maxError == 0 branch: losses are loss(err) (all zero) and every weight is multiplied by beta
    ctx.upload(N.SLOT_PRED, y); ctx.upload(N.SLOT_BW, w)
    assert ctx.boostreg_max_error() == 0.0
    assert ctx.boostreg_error(sw, loss_type, 0.0) == 0.0


@pytest.mark.parametrize("M,n", [(1, 5), (10, 4099), (64, 1001), (200, 300), (257, 77), (1000, 131), (3000, 9)])
def test_agg_boosting_regressor(ctx, oracle, rng, M, n):
    from spark_ensemble_b200 import _native as N
    P = f32(rng.standard_normal((M, n)))
    P[:, : n // 3] = np.round(P[:, : n // 3], 1)  # ties between members
    a = rng.random(M) + 0.05
    ctx.agg_configure(N.AGG_BOOSTING_REG_MEDIAN, M, 0, 1, 0, n)
    ctx.upload(N.SLOT_P, P)
    ctx.agg_run(a)
    np.testing.assert_array_equal(ctx.download(N.SLOT_RAW), oracle.agg_weighted_median(P, a).astype(np.float32))
    ctx.agg_configure(N.AGG_BOOSTING_REG_MEAN, M, 0, 1, 0, n)
    ctx.upload(N.SLOT_P, P)
    ctx.agg_run(a)
    close(ctx.download(N.SLOT_RAW), oracle.agg_weighted_mean(P, a.astype(np.float32).astype(np.float64)), scale=0.1)


@pytest.mark.parametrize("M", [1, 2, 3, 5, 8, 13, 16, 20, 32, 33, 50, 64])
@pytest.mark.parametrize("weights", ["random", "equal", "integers", "one_heavy", "zeros", "negative", "tiny_list"])
def test_weighted_median_fast_path_is_exact(ctx, oracle, rng, M, weights):
    """M <= 64 and weights >= 0: 32-bit keys sorted alone, the half-weight crossing found by bisection on sums taken
    in MODEL order, and every row whose crossing lies within the rounding margin of the two summation orders redone by
    the exact kernel ((key, model) words, sorted-order fp64 sums, ensemble/Utils.scala:31-38).  Bit-exact against
    the oracle for generic weights (no deferred rows), equal weights (no margin needed), small integers (exact
    half-weight ties: many deferred rows), a list too small for the deferred rows (exact pass over all rows),
    all-zero and negative weights (exact kernel only), values with ties / +-0 / huge magnitudes."""
    from spark_ensemble_b200 import _native as N
    n = 20_011
    P = f32(rng.standard_normal((M, n)))
    P[:, : n // 3] = np.round(P[:, : n // 3], 1)          # ties between members, zeros of both signs
    P[:, n // 3: n // 3 + 50] *= 1e30
    P[:, n // 3 + 50: n // 3 + 100] = 0.0
    if M > 1:
        P[1, n // 3 + 50: n // 3 + 100] = -0.0
    ints = rng.integers(1, 4, M).astype(np.float64)
    if ints.sum() % 2:
        ints[0] += 1.0                                    # even total: sorted prefixes DO hit the half-weight exactly
    a = {"random": rng.random(M) + 0.05, "equal": np.full(M, 0.3), "integers": ints,
         "one_heavy": np.where(np.arange(M) == M // 2, 1e6, 1e-3), "zeros": np.zeros(M),
         "negative": np.where(np.arange(M) == 0, -0.5, 1.0) * (rng.random(M) + 0.05), "tiny_list": ints}[weights]
    ctx.agg_configure(N.AGG_BOOSTING_REG_MEDIAN, M, 0, 1, 0, n)
    ctx.upload(N.SLOT_P, P)
    ref = oracle.agg_weighted_median(P, a).astype(np.float32)
    try:
        ctx.set_option("wm_list_cap", 7 if weights == "tiny_list" else n if weights == "integers" else 0)
        ctx.agg_run(a)
        got = ctx.download(N.SLOT_RAW)
        np.testing.assert_array_equal(got, ref)
        mode = ctx.get_option("last_wm_mode")
        deferred = ctx.get_option("last_wm_deferred")
        if weights == "negative":
            assert mode == 0
        elif weights in ("equal", "zeros") or M == 1 or len(set(a.tolist())) == 1:
            assert mode == 2 and deferred == 0
        else:
            assert mode == 1
            if weights == "random":
                assert deferred == 0                      # generic weights: nothing lands within 8 M 2^-53 of the half-weight
            if weights in ("integers", "tiny_list") and M >= 5:
                assert deferred > (7 if weights == "tiny_list" else 0)   # exact half-weight ties do occur; tiny list overflows
        ctx.set_option("wm_fast", 0)
        ctx.agg_run(a)
        assert ctx.get_option("last_wm_mode") == 0
        np.testing.assert_array_equal(ctx.download(N.SLOT_RAW), ref)
    finally:
        ctx.set_option("wm_fast", 1)
        ctx.set_option("wm_list_cap", 0)


@pytest.mark.parametrize("n", [1, 2, 1000, 100003])
def test_exact_quantile_radix_select(ctx, rng, n):
    """se_quantile == the ceil(q·N)-th smallest value, bit-exact (SURVEY.md §8f-3)."""
    from spark_ensemble_b200 import _native as N
    from spark_ensemble_b200.ensemble import exact_quantile
    v = f32(rng.standard_normal(n) * 3)
    v[: n // 5] = np.round(v[: n // 5])  # many duplicates, zeros of both signs
    if n > 10:
        v[3], v[4] = 0.0, -0.0
    ctx.alloc(N.SLOT_Y, n)
    ctx.upload(N.SLOT_Y, v)
    for q in (0.0, 0.1, 0.5, 0.9, 0.999, 1.0):
        assert ctx.quantile(N.SLOT_Y, q) == exact_quantile(v, q), (n, q)
    F = f32(rng.standard_normal(n))
    ctx.gbm_configure(n, 0, 1, "huber", 1.0, False)
    ctx.upload(N.SLOT_Y, v); ctx.upload(N.SLOT_F, F)
    for q in (0.5, 0.9):
        assert ctx.gbm_abs_residual_quantile(q) == exact_quantile(np.abs(v - F), q)


@pytest.mark.parametrize("name", ["squared", "bernoulli", "logloss2", "logloss9"])
def test_bag_multiplicities(ctx, oracle, rng, name):
    """Row sub-sampling (SURVEY.md §8f-4): with bag counts c_i the line-search sums and newton's Σh equal the
    reference's sums over the materialised bag (rows repeated c_i times); update/residuals stay on all rows."""
    from spark_ensemble_b200 import _native as N
    n = 20011
    K = int(name[7:]) if name.startswith("logloss") else 5
    lname = "logloss" if name.startswith("logloss") else name
    dim, par, y, F, h, w = setup_gbm(ctx, rng, lname, n, True, K=K)
    c = rng.poisson(1.0, n).astype(np.float32)
    ctx.gbm_set_bag(c)
    rep = np.repeat(np.arange(n), c.astype(int))  # the materialised bag
    yb, wb, Fb, hb = y[rep], w[rep], np.ascontiguousarray(F[:, rep]), np.ascontiguousarray(h[:, rep])
    lid = O.LOSS_IDS[lname]
    alpha = rng.random(dim) + 0.3
    lg, gg = ctx.gbm_linesearch_eval(alpha)
    lo, go = oracle.linesearch_eval(lid, par, yb, wb, Fb, hb, alpha)
    assert lg == pytest.approx(lo, rel=RTOL)
    close(gg, go, rtol=RTOL, scale=float(np.max(np.abs(go))))
    if lname == "squared":
        st = ctx.gbm_linesearch_stats()
        d = yb.astype(np.float64) - Fb[0]
        close(st, [np.sum(d * d), np.sum(hb[0] * d), np.sum(hb[0].astype(np.float64) ** 2), np.sum(wb.astype(np.float64))])
    S = ctx.gbm_pseudo_residuals(newton=True)
    _, _, So = oracle.pseudo_residuals(lid, par, dim, yb, wb, Fb, True)
    close(S, So, rtol=RTOL)
    ro, _, _ = oracle.pseudo_residuals(lid, par, dim, y, w, F, True)  # residuals themselves: every row
    close(ctx.download(N.SLOT_R).reshape(dim, n), ro, rtol=RTOL, scale=1.0)
    step = rng.random(dim) * 0.3
    ls, _ = ctx.gbm_update(step, residual=True, loss=True)
    Fo = F.astype(np.float64).copy()
    oracle.update(Fo, h, step)
    assert ls / n == pytest.approx(oracle.mean_loss(lid, par, dim, y, Fo), rel=RTOL)  # full train set
    ctx.gbm_set_bag(None)
    lg2, _ = ctx.gbm_linesearch_eval(alpha)
    assert lg2 == pytest.approx(oracle.linesearch_eval(lid, par, y, w, Fo, h, alpha)[0], rel=RTOL)


def test_empty_and_tiny_inputs(ctx, oracle):
    """Edge cases the domain has: empty shards (a rank may own zero rows), single rows, zero models."""
    from spark_ensemble_b200 import _native as N
    # empty GBM shard: every entry point runs, sums are 0, nothing crashes
    ctx.gbm_configure(0, 0, 1, "squared", 0.0, False)
    ctx.gbm_pseudo_residuals(False)
    ls, _ = ctx.gbm_update([0.5], residual=True, loss=True)
    assert ls == 0.0
    s = ctx.gbm_linesearch_stats()
    assert list(s[:3]) == [0.0, 0.0, 0.0]
    ctx.gbm_configure(0, 0, 3, "logloss", 0.0, False)
    ls, _ = ctx.gbm_update(np.ones(3), residual=True, loss=True)
    assert ls == 0.0
    ctx.gbm_configure(0, 0, 9, "logloss", 0.0, False)  # TMA-tiled kernel with no tiles
    ls, _ = ctx.gbm_update(np.ones(9), residual=True, loss=True)
    assert ls == 0.0
    # empty boosting shard
    ctx.boost_configure(0, 3, True)
    assert ctx.slot_sum(N.SLOT_BW) == 0.0
    e, s2 = ctx.boost_real_update(1.0)
    assert (e, s2) == (0.0, 0.0)
    # single row through every GBM loss
    for name in ("squared", "absolute", "huber", "quantile", "bernoulli", "exponential"):
        ctx.gbm_configure(1, 0, 1, name, 0.5, False)
        ctx.upload(N.SLOT_Y, [1.0]); ctx.upload(N.SLOT_F, [0.25]); ctx.upload(N.SLOT_H, [0.5])
        l, g = ctx.gbm_linesearch_eval([2.0])
        lo, go = oracle.linesearch_eval(O.LOSS_IDS[name], 0.5, np.array([1.0]), None, np.array([[0.25]]),
                                        np.array([[0.5]]), [2.0])
        assert l == pytest.approx(lo, rel=RTOL) and g[0] == pytest.approx(go[0], rel=RTOL, abs=1e-7)
    # aggregation over zero rows
    ctx.agg_configure(N.AGG_GBM_REGRESSOR, 3, 0, 1, 0, 0)
    ctx.agg_run([1.0, 1.0, 1.0], [0.0])
    assert ctx.download(N.SLOT_RAW).size == 0


@pytest.mark.parametrize("name", ["squared", "bernoulli", "exponential", "logcosh"])
def test_newton_line_search_matches_brent(ctx, oracle, rng, name):
    """Opt-in curvature line search: derivatives of the objective match the oracle (finite differences of the
    fp64 objective), and the minimiser agrees with Brent's to optimiser tolerance in far fewer passes."""
    from spark_ensemble_b200 import _native as N
    n = 50021
    dim, par, y, F, h, w = setup_gbm(ctx, rng, name, n, True)
    lid = O.LOSS_IDS[name]
    r, _, _ = oracle.pseudo_residuals(lid, par, 1, y, None, F, False)
    h = f32(0.7 * r + 0.2 * rng.standard_normal((1, n)))
    ctx.upload(N.SLOT_H, h)
    f = lambda a: oracle.linesearch_eval(lid, par, y, w, F, h, [a])
    l, d1, d2 = ctx.gbm_linesearch_eval2(0.8)
    lo, go = f(0.8)
    assert l == pytest.approx(lo, rel=RTOL) and d1 == pytest.approx(go[0], rel=1e-4, abs=1e-8)
    eps = 1e-4
    fd2 = (f(0.8 + eps)[1][0] - f(0.8 - eps)[1][0]) / (2 * eps)
    assert d2 == pytest.approx(fd2, rel=1e-3)
    an, ln, nn = ctx.gbm_linesearch_newton()
    ab, lb, nb = ctx.gbm_linesearch_brent()
    # the fp32-evaluated objective is flat to ~1e-7 relative around its minimum, so Brent's abscissa is only
    # defined to ~sqrt(noise/curvature); compare the objective reached (fp64 oracle) and the abscissa loosely
    assert f(an)[0] <= f(ab)[0] * (1 + 1e-7)
    assert abs(an - ab) <= 2e-3 * max(1.0, abs(ab))
    assert abs(f(an)[1][0]) <= 1e-4 * max(1.0, abs(f(0.0)[1][0]))  # stationary point of the oracle objective
    assert ln == pytest.approx(lb, rel=1e-6)
    assert nn <= 12 and nn < nb  # quadratic convergence, then a few steps at the fp32 noise floor of the slope
    ctx.gbm_configure(64, 0, 1, "absolute", 0.0, False)
    with pytest.raises(ValueError):
        ctx.gbm_linesearch_newton()


@pytest.mark.parametrize("n,d", [(1, 1), (33, 12), (1000, 128), (300_001, 64)])
def test_rowmajor_ingest(ctx, rng, n, d):
    """se_upload_rowmajor: row-major feature partitions land transposed in the column-major slot (bit-exact),
    including appends at a row offset and chunk boundaries (the 300k x 64 case spans three 32 MB chunks)."""
    from spark_ensemble_b200 import _native as N
    X = f32(rng.standard_normal((n, d)))
    ctx.alloc(N.SLOT_X, d, n)
    ctx.fill(N.SLOT_X, -7.0)
    split = n // 3
    ctx.upload_rowmajor(N.SLOT_X, X[:split], 0)          # two Spark partitions appended one after the other
    ctx.upload_rowmajor(N.SLOT_X, X[split:], split)
    got = ctx.download(N.SLOT_X).reshape(d, n)
    np.testing.assert_array_equal(got, X.T)
    with pytest.raises(ValueError):
        ctx.upload_rowmajor(N.SLOT_X, X, 1)  # runs past the slot


def test_gbm_round_single_call(ctx, oracle, rng):
    """se_gbm_round == se_gbm_linesearch_brent + se_gbm_update."""
    from spark_ensemble_b200 import _native as N
    n = 30011
    ctx.set_option("fused_round", 0)  # the one-launch round has its own test (different reduction grids)
    for name in ("squared", "bernoulli"):
        dim, par, y, F, h, w = setup_gbm(ctx, rng, name, n)
        a1, l1, ne1 = ctx.gbm_round(0.5, True, 1e-6, 100, residual=True)
        F1, r1 = ctx.download(N.SLOT_F).copy(), ctx.download(N.SLOT_R).copy()
        ctx.upload(N.SLOT_F, F)
        a2, _, ne2 = ctx.gbm_linesearch_brent()
        l2, _ = ctx.gbm_update([0.5 * a2], residual=True, loss=True)
        assert (a1, ne1) == (a2, ne2) and l1 == l2
        np.testing.assert_array_equal(F1, ctx.download(N.SLOT_F))
        np.testing.assert_array_equal(r1, ctx.download(N.SLOT_R))
        a3, l3, ne3 = ctx.gbm_round(0.5, False)
        assert (a3, ne3) == (1.0, 0)
    ctx.set_option("fused_round", -1)


def test_device_brent_matches_host_brent(oracle, rng, monkeypatch):
    """Squared loss: with SE_DEVICE_BRENT=1 se_gbm_round runs Brent on the device over the parabola of the sufficient
    statistics (se_brent.cu: the same template as the host line search, compiled without multiply-add contraction).
    alpha, the evaluation count, the train loss and the updated F / R must equal the host line search bit for bit,
    for interior minima, both interval ends and several tolerances."""
    from spark_ensemble_b200 import _native as N
    from spark_ensemble_b200.context import Context
    monkeypatch.setenv("SE_ALTERNATE_PASSES", "0")  # one tile direction: sums do not depend on the call history
    c = Context(0)
    c.set_option("fused_round", 0)  # compare the three-launch device search with the two-launch host search
    try:
        n = 50021
        for case, (scale, shift, tol) in enumerate([(1.0, 0.0, 1e-6), (0.01, 0.0, 1e-6), (-1.0, 0.0, 1e-6),
                                                    (3.0, 0.5, 1e-9), (1e-3, 0.0, 1e-4), (0.3, -2.0, 1e-12)]):
            y = f32(rng.standard_normal(n))
            F = f32(0.3 * rng.standard_normal(n) + shift)
            h = f32(scale * (y - F) + 0.1 * rng.standard_normal(n))
            out = []
            for host in (False, True):
                c.gbm_configure(n, 0, 1, "squared", 0.0, False)
                c.upload(N.SLOT_Y, y); c.upload(N.SLOT_F, F); c.upload(N.SLOT_H, h)
                if host:
                    monkeypatch.delenv("SE_DEVICE_BRENT", raising=False)
                else:
                    monkeypatch.setenv("SE_DEVICE_BRENT", "1")
                a, l, ne = c.gbm_round(0.7, True, tol, 100, residual=True)
                out.append((a, l, ne, c.download(N.SLOT_F).copy(), c.download(N.SLOT_R).copy()))
            monkeypatch.delenv("SE_DEVICE_BRENT", raising=False)
            (a1, l1, ne1, F1, r1), (a2, l2, ne2, F2, r2) = out
            assert (a1, ne1, l1) == (a2, ne2, l2), (case, a1, a2, ne1, ne2, l1, l2)
            np.testing.assert_array_equal(F1, F2)
            np.testing.assert_array_equal(r1, r2)
            assert ne1 >= 3
        # MaxEval exceeded: both paths raise (commons-math: TooManyEvaluationsException)
        for host in (False, True):
            c.gbm_configure(n, 0, 1, "squared", 0.0, False)
            c.upload(N.SLOT_Y, y); c.upload(N.SLOT_F, F); c.upload(N.SLOT_H, h)
            if not host:
                monkeypatch.setenv("SE_DEVICE_BRENT", "1")
            with pytest.raises(N.NativeError):
                c.gbm_round(0.7, True, 1e-12, 2, residual=True)
        monkeypatch.delenv("SE_DEVICE_BRENT", raising=False)
    finally:
        c.close()

def test_squared_stats_from_residual_slot(ctx, oracle, rng):
    """Squared loss: when R holds the current residual (after pseudo_residuals or a fused update) the line-search
    statistics are read from (r, h) — 8 B/row — and are bit-identical to the (y, F, h) pass; any write to
    Y/F/R falls back to the 12 B/row pass."""
    from spark_ensemble_b200 import _native as N
    n = 100003
    dim, par, y, F, h, w = setup_gbm(ctx, rng, "squared", n, True)
    s_yfh = ctx.gbm_linesearch_stats()           # R stale: y, F, h
    ctx.gbm_pseudo_residuals(False)
    s_r = ctx.gbm_linesearch_stats()             # R current: r, h
    np.testing.assert_array_equal(s_r, s_yfh)
    ls, _ = ctx.gbm_update([0.3], residual=True, loss=True)
    s_r2 = ctx.gbm_linesearch_stats()            # fused update refreshed R
    Fo = F.astype(np.float64).copy(); oracle.update(Fo, h, [0.3])
    d = y.astype(np.float64) - Fo[0]; hh = h[0].astype(np.float64)
    close(s_r2[:3], [np.sum(d * d), np.sum(hh * d), np.sum(hh * hh)])
    Fnow = ctx.download(N.SLOT_F)
    ctx.upload(N.SLOT_F, Fnow)                   # same values, but the write invalidates the cache
    np.testing.assert_array_equal(ctx.gbm_linesearch_stats(), s_r2)
    ctx.gbm_update([0.1], residual=False, loss=True)   # plain update: R is stale again
    s3 = ctx.gbm_linesearch_stats()
    oracle.update(Fo, h, [0.1]); d = y.astype(np.float64) - Fo[0]
    close(s3[:3], [np.sum(d * d), np.sum(hh * d), np.sum(hh * hh)])


@pytest.mark.parametrize("name", ["bernoulli", "exponential"])
@pytest.mark.parametrize("weighted_bag", [False, True])
def test_brent_packed_line_search_view_is_bit_identical(oracle, rng, name, weighted_bag, monkeypatch):
    """se_gbm_linesearch_brent evaluates the binary losses on the signed view u=(2y-1)F, v=(2y-1)h (8 B/row):
    same alpha, objective and evaluation count as the plain (y, F, h) evaluations, bit for bit.

    Consecutive passes normally walk the tiles in alternating directions (L2 reuse), which changes which CTA owns
    which tile and therefore the last bits of the fp64 sums; the comparison runs in its own context with the
    alternation switched off (SE_ALTERNATE_PASSES=0, read at context creation) so both searches see one direction."""
    from spark_ensemble_b200 import _native as N
    from spark_ensemble_b200.context import Context
    monkeypatch.setenv("SE_ALTERNATE_PASSES", "0")
    ctx = Context(0)
    ctx.set_option("ls_mode", 0)  # the one-launch-per-evaluation path (the persistent search has its own test)
    try:
        _packed_vs_plain(ctx, oracle, rng, name, weighted_bag, monkeypatch, N)
    finally:
        ctx.close()


def _packed_vs_plain(ctx, oracle, rng, name, weighted_bag, monkeypatch, N):
    n = 40013
    dim, par, y, F, h, w = setup_gbm(ctx, rng, name, n, weighted_bag)
    r, _, _ = oracle.pseudo_residuals(O.LOSS_IDS[name], par, 1, y, None, F, False)
    h = f32(0.6 * r + 0.2 * rng.standard_normal((1, n)))
    ctx.upload(N.SLOT_H, h)
    if weighted_bag:
        ctx.gbm_set_bag(rng.poisson(1.0, n).astype(np.float32))
    packed = ctx.gbm_linesearch_brent()
    monkeypatch.setenv("SE_NO_LS_PACK", "1")
    plain = ctx.gbm_linesearch_brent()
    monkeypatch.delenv("SE_NO_LS_PACK")
    assert packed == plain
    assert packed[2] >= 8


def test_tree_predict_multi_class_probabilities(ctx, rng):
    """Classification trees on device: leaf class-probability vectors -> SE_SLOT_PROBA, leaf labels -> SE_SLOT_PRED."""
    from spark_ensemble_b200 import _native as N
    from spark_ensemble_b200.learners import DecisionTreeClassifier
    n, d, K = 20011, 10, 7
    X = f32(rng.standard_normal((n, d)))
    yv = (np.abs(X[:, 0] * 2 + X[:, 3]).astype(int) % K).astype(np.float64)
    yv[yv == 5] = 4  # class 5 never occurs: sklearn's classes_ is a subset
    m = DecisionTreeClassifier(maxDepth=7).fit(X, yv, None, num_classes=K)
    t = m.tree_arrays()
    ctx.alloc(N.SLOT_X, d, n)
    ctx.upload_rowmajor(N.SLOT_X, X)
    ctx.alloc(N.SLOT_PROBA, K, n)
    ctx.tree_predict_multi(t, N.SLOT_PROBA)
    np.testing.assert_allclose(ctx.download(N.SLOT_PROBA), m.predictProbability(X).T.astype(np.float32), rtol=1e-6)
    ctx.alloc(N.SLOT_PRED, n)
    ctx.tree_predict(t, N.SLOT_PRED, 0)
    np.testing.assert_array_equal(ctx.download(N.SLOT_PRED), m.predict(X).astype(np.float32))


def test_libsvm_to_device_ingest(ctx, rng, tmp_path):
    """LIBSVM file -> row blocks -> se_upload_rowmajor -> column-major X in HBM, block boundaries not 32-aligned."""
    from spark_ensemble_b200 import _native as N
    from spark_ensemble_b200.io import load_libsvm_to_device
    n, d = 1003, 12
    X = np.where(rng.random((n, d)) < 0.6, rng.standard_normal((n, d)), 0.0).astype(np.float32)
    y = rng.integers(0, 3, n).astype(np.float64)
    p = tmp_path / "x.svm"
    with open(p, "w") as fh:
        for i in range(n):
            fh.write(f"{float(y[i])!r} " + " ".join(f"{j + 1}:{float(X[i, j])!r}" for j in range(d) if X[i, j] != 0.0) + "\n")
    labels = load_libsvm_to_device(ctx, N.SLOT_X, str(p), d, block_rows=250)
    np.testing.assert_array_equal(labels, y)
    np.testing.assert_array_equal(ctx.download(N.SLOT_X).reshape(d, n), X.T)


# ------------------------------------------------------------------ cooperative whole-round / whole-search kernels
def _host_brent(fn, rel=1e-6, abs_tol=1e-6, max_eval=100):
    """The product's host Brent (se_brent_minimize) over a Python objective."""
    import ctypes
    from spark_ensemble_b200 import _native as N
    lib = N.load()
    cb = N.FN1(lambda x, _u: float(fn(x)))
    x, f, ne = ctypes.c_double(), ctypes.c_double(), ctypes.c_int()
    rc = lib.se_brent_minimize(cb, None, 0.0, 100.0, 1.0, rel, abs_tol, max_eval, ctypes.byref(x), ctypes.byref(f),
                               ctypes.byref(ne))
    return rc, x.value, f.value, ne.value


@pytest.mark.parametrize("n", [1, 5, 1023, 4096, 100003, 1200007])
@pytest.mark.parametrize("weighted", [False, True])
def test_fused_squared_round(ctx, oracle, rng, n, weighted):
    """se_gbm_round as ONE cooperative launch (statistics -> Brent on the device -> update + residual + loss):
    statistics, F, r and the loss against the fp64 oracle (1e-5), and the in-kernel Brent against the host Brent
    (same template) on the kernel's own statistics: alpha and the evaluation count bit for bit."""
    from spark_ensemble_b200 import _native as N
    dim, par, y, F, h, w = setup_gbm(ctx, rng, "squared", n, weighted)
    h = f32((y - F[0]) * 0.6 + 0.2 * rng.standard_normal(n)).reshape(1, n)
    ctx.upload(N.SLOT_H, h)
    ws = float(np.sum(w.astype(np.float64))) if weighted else float(n)
    ws_dev = ctx.gbm_linesearch_stats()[3]
    assert ws_dev == pytest.approx(ws, rel=1e-12)
    ctx.set_option("fused_round", 1)
    try:
        Fo = F.astype(np.float64).copy()
        hh = h[0].astype(np.float64)
        for rnd in range(3):  # round 0 reads (y, F, h); later rounds read the residual slot (8 B/row)
            a, ls, ne = ctx.gbm_round(0.7, True, 1e-6, 100, residual=True)
            assert ctx.get_option("last_round_fused") == 1
            s = [ctx.get_option(f"last_round_stat{i}") for i in range(3)]
            d = y.astype(np.float64) - Fo[0]
            # rounds >= 1 read the fp32 residual slot: each d carries (|y| + |F|) 2^-23 of the fp32 state's rounding
            dtol = 1.2e-7 * (np.abs(y) + np.abs(Fo[0]))
            want = np.array([np.sum(d * d), np.sum(hh * d), np.sum(hh * hh)])
            slack = np.array([2.0 * np.sum(np.abs(d) * dtol), np.sum(np.abs(hh) * dtol), 0.0])
            assert np.all(np.abs(np.array(s) - want) <= RTOL * np.abs(want) + slack), (s, want, slack)
            inv = 1.0 / (2.0 * ws_dev)  # se_brent.h BrentParabola: one reciprocal, then multiplications
            rc, xh, fh, neh = _host_brent(lambda x: (s[0] - 2.0 * x * s[1] + x * x * s[2]) * inv)
            assert rc == 0 and (a, ne) == (xh, neh), (rnd, a, xh, ne, neh)
            oracle.update(Fo, h, [0.7 * a])
            close(ctx.download(N.SLOT_F), Fo[0])
            ro, _, _ = oracle.pseudo_residuals(O.SQUARED, 0.0, 1, y, None, Fo, False)
            close(ctx.download(N.SLOT_R), ro[0], scale=1.0)
            # F lives in fp32: a residual d = y - F carries |F| 2^-24 of rounding, the loss d^2 / 2 therefore
            # |d| |F| 2^-24 — invisible next to 1e-5 except when a row's residual has shrunk far below |F| (n = 1)
            dd = y.astype(np.float64) - Fo[0]
            atol = 5e-7 * float(np.mean(np.abs(dd) * (np.abs(Fo[0]) + np.abs(y))))
            assert ls / n == pytest.approx(oracle.mean_loss(O.SQUARED, 0.0, 1, y, Fo), rel=RTOL, abs=atol)
        # the two-launch path on the same state agrees to rounding of the fp64 sums
        Fnow = ctx.download(N.SLOT_F).copy()
        a1, l1, ne1 = ctx.gbm_round(0.7, True, 1e-6, 100, residual=True)
        F1 = ctx.download(N.SLOT_F).copy()
        ctx.upload(N.SLOT_F, Fnow)
        ctx.set_option("fused_round", 0)
        a2, l2, ne2 = ctx.gbm_round(0.7, True, 1e-6, 100, residual=True)
        assert ctx.get_option("last_round_fused") == 0
        assert a1 == pytest.approx(a2, rel=1e-9, abs=1e-12)
        assert l1 == pytest.approx(l2, rel=RTOL, abs=atol * n)  # closed form over the fp64 statistics vs the sum of the fp32 rows
        close(F1, ctx.download(N.SLOT_F), rtol=1e-6)
        # the in-kernel row reduction of the loss (the path bags use) agrees with the closed form
        ctx.upload(N.SLOT_F, Fnow)
        ctx.set_option("fused_round", 1)
        ctx.set_option("fused_loss_reduce", 1)
        a3, l3, ne3 = ctx.gbm_round(0.7, True, 1e-6, 100, residual=True)
        ctx.set_option("fused_loss_reduce", 0)
        assert (a3, ne3) == (a1, ne1) and l3 == pytest.approx(l1, rel=RTOL, abs=atol * n)
        np.testing.assert_array_equal(F1, ctx.download(N.SLOT_F))
        # MaxEval exceeded: SE_ERR_OPT (TooManyEvaluationsException in the reference) and F is left untouched
        ctx.set_option("fused_round", 1)
        Fbefore = ctx.download(N.SLOT_F).copy()
        if n > 5:
            with pytest.raises(N.ConvergenceError):
                ctx.gbm_round(0.7, True, 1e-12, 2, residual=True)
            np.testing.assert_array_equal(Fbefore, ctx.download(N.SLOT_F))
    finally:
        ctx.set_option("fused_round", -1)


def test_fused_squared_round_with_bag(ctx, oracle, rng):
    from spark_ensemble_b200 import _native as N
    n = 50007
    dim, par, y, F, h, w = setup_gbm(ctx, rng, "squared", n, True)
    bag = rng.poisson(1.0, n).astype(np.float32)
    ctx.gbm_set_bag(bag)
    ctx.set_option("fused_round", 1)
    try:
        a, ls, ne = ctx.gbm_round(0.5, True, 1e-6, 100, residual=True)
    finally:
        ctx.set_option("fused_round", -1)
    c = bag.astype(np.float64); d = y.astype(np.float64) - F[0]; hh = h[0].astype(np.float64)
    star = float(np.clip(np.sum(c * hh * d) / np.sum(c * hh * hh), 0, 100))  # the line search runs on the bag (quirk 4)
    assert a == pytest.approx(star, rel=1e-5, abs=2e-6)
    Fo = F.astype(np.float64).copy(); oracle.update(Fo, h, [0.5 * a])
    close(ctx.download(N.SLOT_F), Fo[0])                                      # the update on all rows
    assert ls / n == pytest.approx(oracle.mean_loss(O.SQUARED, 0.0, 1, y, Fo), rel=RTOL)
    ctx.gbm_configure(4, 0, 1, "squared", 0.0, False)  # drops the bag for the tests that follow


LS_LOSSES = ["absolute", "huber", "quantile", "logcosh", "scaledlogcosh", "bernoulli", "exponential"]


@pytest.mark.parametrize("name", LS_LOSSES)
@pytest.mark.parametrize("n,ctas,resident,ring", [(3, 4, 1, 0), (2049, 4, 1, 0), (40013, 4, 1, 0), (700001, 1, 0, 3),
                                                  (700001, 1, 0, 0), (700001, 1, 1, 0), (2000003, 2, 1, 0),
                                                  (2000003, 4, 0, 2), (2000003, 4, 0, 4), (5000011, 4, 1, 3)])
def test_device_line_search_matches_host_brent(ctx, oracle, rng, name, n, ctas, resident, ring):
    """Brent's whole line search in ONE persistent launch (workers + coordinator warp, tiles resident in shared
    memory, the first evaluation builds the signed view of the binary losses).  ls_mode 2 runs the HOST Brent over
    single-evaluation launches of the same kernel: alpha, the objective and the evaluation count must be identical
    bit for bit.  Tiles that do not stay resident stream through a per-thread cp.async ring (`ls_ring` stages; 0 = the
    register prefetch).  Against the oracle: the objective value at the minimiser within 1e-5."""
    from spark_ensemble_b200 import _native as N
    dim, par, y, F, h, w = setup_gbm(ctx, rng, name, n, weighted=(n % 2 == 0))
    lid = O.LOSS_IDS[name]
    r, _, _ = oracle.pseudo_residuals(lid, par, 1, y, None, F, False)
    h = f32(0.6 * r + 0.2 * rng.standard_normal((1, n)))
    ctx.upload(N.SLOT_H, h)
    ctx.set_option("ls_ctas_per_sm", ctas)
    ctx.set_option("ls_resident", resident)
    ctx.set_option("ls_ring", ring)
    try:
        ctx.set_option("ls_mode", 1)
        dev = ctx.gbm_linesearch_brent()
        passes = ctx.get_option("last_ls_passes")
        assert passes == dev[2] and ctx.get_option("last_ls_workers") >= 1
        dev_again = ctx.gbm_linesearch_brent()
        assert dev_again == dev  # deterministic: fixed tile ownership, fixed reduction order
        ctx.set_option("ls_mode", 2)
        host = ctx.gbm_linesearch_brent()
        assert dev == host, (dev, host)
        ctx.set_option("ls_mode", 0)
        old = ctx.gbm_linesearch_brent()
        assert old[1] == pytest.approx(dev[1], rel=1e-6)
        if n <= 700001:
            f = lambda x: oracle.linesearch_eval(lid, par, y, w, F, h, [x])[0]
            ao, neo, st = oracle.brent(f)
            assert st == 0
            assert dev[1] == pytest.approx(f(ao), rel=RTOL)
            assert f(dev[0]) <= f(ao) * (1 + 1e-5) + 1e-12
        ctx.set_option("ls_mode", 1)
        if n > 3:
            with pytest.raises(N.ConvergenceError):
                ctx.gbm_linesearch_brent(0.0, 100.0, 1.0, 1e-12, 1e-12, 3)
            assert ctx.gbm_linesearch_brent() == dev  # the failed search left the rendezvous state clean
        # the update that follows must see untouched (y, F, h)
        ls, _ = ctx.gbm_update([0.5 * dev[0]], residual=True, loss=True)
        Fo = F.astype(np.float64).copy(); oracle.update(Fo, h, [0.5 * dev[0]])
        assert ls / n == pytest.approx(oracle.mean_loss(lid, par, 1, y, Fo), rel=RTOL)
    finally:
        ctx.set_option("ls_mode", 1)
        ctx.set_option("ls_ctas_per_sm", 4)
        ctx.set_option("ls_resident", 1)
        ctx.set_option("ls_ring", 0)


def test_options_roundtrip(ctx):
    from spark_ensemble_b200 import _native as N
    for key, val in (("fused_round", 1), ("ls_mode", 2), ("peer_timeout_ms", 2500.0), ("l2_persist_frac", 0.5)):
        old = ctx.get_option(key)
        ctx.set_option(key, val)
        assert ctx.get_option(key) == val
        ctx.set_option(key, old)
    with pytest.raises(ValueError):
        ctx.set_option("no_such_option", 1)
    with pytest.raises(ValueError):
        ctx.set_option("last_round_fused", 1)  # read-only
    assert ctx.get_option("l2_persist_max_bytes") >= 0


@pytest.mark.parametrize("bad", [-1.0, "K", 2.5, float("nan")])
@pytest.mark.parametrize("K", [3, 9, 40])
def test_bad_labels_fail_loudly(ctx, rng, K, bad):
    """A label that is not an integer class index in [0, K) makes the reference throw on the JVM
    (GBMLoss.scala:200-204 `res(label.toInt) = 1.0`; Classifier.validateLabel).  Here: SE_ERR_ARG from the call that
    observes it, never an out-of-bounds access (run under compute-sanitizer in profiles/r02_sanitizer.md), and the
    context stays usable."""
    from spark_ensemble_b200 import _native as N
    n = 5003
    badv = float(K) if bad == "K" else bad
    y = f32(rng.integers(0, K, n))
    F = f32(rng.standard_normal((K, n)))
    h = f32(rng.standard_normal((K, n)))
    yb = y.copy(); yb[n // 2] = badv; yb[n - 1] = badv
    # LogLoss: line-search evaluation, fused update (register kernel K <= 4, TMA-tiled kernel K >= 5)
    ctx.gbm_configure(n, 0, K, "logloss", 0.0, False)
    ctx.upload(N.SLOT_F, F); ctx.upload(N.SLOT_H, h)
    ctx.upload(N.SLOT_Y, yb)
    with pytest.raises(ValueError, match="class index"):
        ctx.gbm_linesearch_eval(np.ones(K))
    with pytest.raises(ValueError, match="class index"):
        ctx.gbm_update(np.full(K, 0.1), residual=True, loss=True)
    with pytest.raises(ValueError, match="class index"):
        ctx.gbm_pseudo_residuals(False)
        ctx.sync()
    ctx.upload(N.SLOT_Y, y); ctx.upload(N.SLOT_F, F)
    l, g = ctx.gbm_linesearch_eval(np.ones(K))
    assert np.isfinite(l) and np.all(np.isfinite(g))
    # SAMME.R (register kernel K < 5, TMA-tiled K >= 5)
    P = rng.random((K, n)); P = f32(P / P.sum(0))
    ctx.boost_configure(n, K, True)
    ctx.upload(N.SLOT_PROBA, P); ctx.fill(N.SLOT_BW, 1.0)
    ctx.upload(N.SLOT_Y, yb)
    with pytest.raises(ValueError, match="class index"):
        ctx.boost_real_update(float(n))
    ctx.upload(N.SLOT_Y, y); ctx.fill(N.SLOT_BW, 1.0)
    e, s = ctx.boost_real_update(float(n))
    assert 0.0 <= e <= 1.0 and s > 0
    # hard votes
    M = 7
    votes = f32(rng.integers(0, K, (M, n)))
    vb = votes.copy(); vb[3, 17] = badv
    ctx.agg_configure(N.AGG_BAGGING_HARD, M, K, 1, 0, n)
    ctx.upload(N.SLOT_P, vb)
    ctx.agg_run()
    with pytest.raises(ValueError, match="class index"):
        ctx.sync()
    ctx.upload(N.SLOT_P, votes)
    ctx.agg_run()
    ctx.sync()
    raw = ctx.download(N.SLOT_RAW)
    assert np.all(raw.reshape(K, n).sum(0) == M)


def _random_tree(rng, depth, d, candidates, n_out=1):
    """Complete binary tree in array form; thresholds drawn from per-feature candidate lists (like Spark's findSplits)."""
    nn = 2 ** (depth + 1) - 1
    idx = np.arange(nn)
    leaf = idx >= 2 ** depth - 1
    feat = rng.integers(0, d, nn)
    thr = np.array([candidates[f][rng.integers(0, len(candidates[f]))] for f in feat], dtype=np.float32)
    t = {"feature": np.where(leaf, -1, feat).astype(np.int32), "threshold": np.where(leaf, 0.0, thr).astype(np.float32),
         "left": np.where(leaf, 0, 2 * idx + 1).astype(np.int32), "right": np.where(leaf, 0, 2 * idx + 2).astype(np.int32),
         "value": rng.standard_normal(nn).astype(np.float32)}
    if n_out > 1:
        t["values"] = rng.random((nn, n_out)).astype(np.float32)
    return t


def _walk(tree, X):
    """Plain numpy walk: x <= threshold goes left (Spark ContinuousSplit.shouldGoLeft)."""
    node = np.zeros(X.shape[0], dtype=np.int64)
    for _ in range(256):
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


@pytest.mark.parametrize("n,d,n_internal", [(5, 3, 1), (4099, 11, 17), (100_003, 40, 64), (100_003, 40, 65), (33_333, 5, 120)])
def test_shallow_tree_all_nodes_kernel(ctx, rng, n, d, n_internal):
    """Trees of <= 64 internal nodes go through the all-nodes kernel (every node's comparison from coalesced column
    reads of the rank matrix, then a walk over bits); larger ones walk.  Arbitrary shapes / node orders, rows ON
    thresholds, every row count modulo the vector width: the leaf must be the fp32 walk's."""
    from spark_ensemble_b200 import _native as N
    X = rng.standard_normal((n, d)).astype(np.float32)
    cand = [np.unique(np.concatenate([rng.standard_normal(15).astype(np.float32), X[rng.integers(0, n, 4), f]])) for f in range(d)]
    ctx.alloc(N.SLOT_X, d, n)
    ctx.upload_rowmajor(N.SLOT_X, X)
    ctx.alloc(N.SLOT_H, 1, n)
    ctx.set_option("tree_bins", 1)
    try:
        for mask in (1, 0, 1):
            ctx.set_option("tree_mask", mask)
            tree = _random_unbalanced_tree(rng, n_internal, d, cand)
            ctx.tree_predict(tree, N.SLOT_H, 0)
            assert ctx.get_option("last_tree_binned") == 1
            assert ctx.get_option("last_tree_mask") == (1 if mask and n_internal <= 64 else 0)
            np.testing.assert_array_equal(ctx.download(N.SLOT_H), tree["value"][_walk(tree, X)])
        single = {"feature": [-1], "threshold": [0.0], "left": [0], "right": [0], "value": [2.5]}   # a root-only tree
        ctx.tree_predict(single, N.SLOT_H, 0)
        np.testing.assert_array_equal(ctx.download(N.SLOT_H), np.full(n, 2.5, np.float32))
    finally:
        ctx.set_option("tree_mask", 1)
        ctx.free(N.SLOT_X)


@pytest.mark.parametrize("n,d,T,max_internal", [(1, 3, 1, 2), (777, 5, 2, 6), (30_011, 20, 7, 40), (30_011, 20, 41, 63),
                                                (9_001, 150, 300, 60)])
def test_forest_predict_matches_member_sum(ctx, n, d, T, max_internal):
    """se_forest_predict: init + sum_t w_t * tree_t(x) (GBMRegressionModel.predict, GBMRegressor.scala:531-539) in one
    pass over the rank matrix per chunk of trees, fp64 accumulation in model order.  Against a plain numpy walk of every
    member (leaf choice exact; the sum within one fp32 rounding per chunk), with per-tree subspaces, on the validation
    slot, for forests that need several chunks, and the failure modes (not a tree, bad column, > 255 thresholds)."""
    from spark_ensemble_b200 import _native as N
    rng = np.random.default_rng(1000 + n + T)
    X = rng.standard_normal((n, d)).astype(np.float32)
    cand = [np.unique(np.concatenate([rng.standard_normal(12).astype(np.float32), X[rng.integers(0, n, 3), f]])) for f in range(d)]
    trees, subs = [], []
    for t in range(T):
        if t % 3 == 0 and d >= 3:
            sub = np.sort(rng.choice(d, size=max(2, d // 2), replace=False)).astype(np.int32)
        else:
            sub = None
        dd = d if sub is None else sub.size
        cc = cand if sub is None else [cand[c] for c in sub]
        trees.append(_random_unbalanced_tree(rng, int(rng.integers(0, max_internal + 1)), dd, cc))
        subs.append(sub)
    w = rng.random(T) + 0.1
    init = 0.37
    want = np.full(n, init)
    for tr, sub, wt in zip(trees, subs, w):
        Xs = X if sub is None else X[:, sub]
        want = want + wt * tr["value"][_walk(tr, Xs)].astype(np.float64)
    for validation, slot in ((False, N.SLOT_X), (True, N.SLOT_VX)):
        ctx.alloc(slot, d, n)
        ctx.upload_rowmajor(slot, X)
        out = N.SLOT_VH if validation else N.SLOT_H
        ctx.alloc(out, 1, n)
        ctx.forest_predict(trees, out, weights=w, init=init, validation=validation, subspaces=subs)
        chunks = ctx.get_option("last_forest_chunks")
        assert chunks >= 1 and (T < 300 or chunks > 1)
        got = ctx.download(out).astype(np.float64)
        scale = float(np.max(np.abs(want))) + 1.0
        assert np.max(np.abs(got - want)) <= 1.5e-7 * scale * chunks, (np.max(np.abs(got - want)), chunks)
        if not validation:   # the per-tree path agrees row by row on the leaf of every member
            ctx.tree_predict(trees[0], out, 0, subspace=subs[0])
            Xs = X if subs[0] is None else X[:, subs[0]]
            np.testing.assert_array_equal(ctx.download(out), trees[0]["value"][_walk(trees[0], Xs)])
    # weights None == all ones, init 0
    ctx.forest_predict(trees, N.SLOT_H, subspaces=subs)
    ones = np.zeros(n)
    for tr, sub in zip(trees, subs):
        ones = ones + tr["value"][_walk(tr, X if sub is None else X[:, sub])].astype(np.float64)
    assert np.max(np.abs(ctx.download(N.SLOT_H).astype(np.float64) - ones)) <= 1.5e-7 * (np.max(np.abs(ones)) + 1.0) * chunks
    if T >= 2 and n > 1:
        bad = dict(trees[0]); bad_trees = [bad] + trees[1:]
        if np.any(np.asarray(bad["feature"]) >= 0):
            i = int(np.argmax(np.asarray(bad["feature"]) >= 0))
            bad["left"] = np.array(bad["left"]).copy(); bad["left"][i] = i        # a node that is its own child
            with pytest.raises(ValueError):
                ctx.forest_predict(bad_trees, N.SLOT_H, subspaces=subs)
            bad2 = dict(trees[0]); bad2["feature"] = np.array(bad2["feature"]).copy(); bad2["feature"][i] = d + 5
            with pytest.raises(ValueError):
                ctx.forest_predict([bad2] + trees[1:], N.SLOT_H, subspaces=[None] + subs[1:])
        # a column with more than 255 distinct thresholds cannot be ranked in a byte: SE_ERR_STATE, fall back per tree
        many = np.sort(rng.standard_normal(400).astype(np.float32))
        wide = [_random_unbalanced_tree(rng, 60, 1, [many]) for _ in range(8)]
        with pytest.raises(N.NativeError):
            ctx.forest_predict(wide, N.SLOT_H, subspaces=[np.array([0], np.int32)] * 8)
    ctx.free(N.SLOT_X)
    ctx.free(N.SLOT_VX)


@pytest.mark.parametrize("n,d,depth", [(1, 3, 2), (1027, 7, 4), (200_003, 33, 6), (50_001, 9, 8)])
def test_tree_walk_over_binned_features_is_exact(ctx, rng, n, d, depth):
    """The tree walk over the uint8 RANK matrix (bin(x) = #{thresholds < x}; `x <= t_j` <=> `bin <= j`) must pick the
    same leaf as the fp32 walk for every row — including rows sitting exactly ON a threshold —, keep doing so as new
    trees add thresholds (columns are re-ranked), after the feature matrix is rewritten, through a subspace map, and
    for leaf vectors; a column that needs more than 255 thresholds sends the tree to the fp32 walk."""
    from spark_ensemble_b200 import _native as N
    X = rng.standard_normal((n, d)).astype(np.float32)
    cand = [np.unique(np.concatenate([rng.standard_normal(31).astype(np.float32), X[rng.integers(0, n, 4), f]])) for f in range(d)]
    ctx.alloc(N.SLOT_X, d, n)
    ctx.upload_rowmajor(N.SLOT_X, X)
    ctx.alloc(N.SLOT_H, 1, n)
    ctx.set_option("tree_bins", 1)
    rebinned = 0
    for k in range(6):
        tree = _random_tree(rng, depth, d, cand)
        leaf = _walk(tree, X)
        ctx.tree_predict(tree, N.SLOT_H, 0)
        assert ctx.get_option("last_tree_binned") == 1
        rebinned += ctx.get_option("last_tree_rebinned_cols")
        np.testing.assert_array_equal(ctx.download(N.SLOT_H), tree["value"][leaf])
    assert rebinned >= 1
    # once every candidate threshold has been seen nothing is re-ranked any more (the steady state of a Spark fit)
    for f in range(d):
        for t0 in range(0, len(cand[f]), 3):
            ts = list(cand[f][t0:t0 + 3]) + [cand[f][0]] * 3
            stump = {"feature": [f, f, f, -1, -1, -1, -1], "threshold": [ts[0], ts[1], ts[2], 0, 0, 0, 0],
                     "left": [1, 3, 5, 0, 0, 0, 0], "right": [2, 4, 6, 0, 0, 0, 0], "value": [0, 0, 0, 1.0, 2.0, 3.0, 4.0]}
            ctx.tree_predict(stump, N.SLOT_H, 0)
    tree = _random_tree(rng, depth, d, cand)
    ctx.tree_predict(tree, N.SLOT_H, 0)
    assert ctx.get_option("last_tree_binned") == 1 and ctx.get_option("last_tree_rebinned_cols") == 0
    np.testing.assert_array_equal(ctx.download(N.SLOT_H), tree["value"][_walk(tree, X)])
    # rewriting the feature matrix invalidates the ranks
    X2 = rng.standard_normal((n, d)).astype(np.float32)
    ctx.upload_rowmajor(N.SLOT_X, X2)
    tree = _random_tree(rng, depth, d, cand)
    ctx.tree_predict(tree, N.SLOT_H, 0)
    assert ctx.get_option("last_tree_binned") == 1 and ctx.get_option("last_tree_rebinned_cols") >= 1
    np.testing.assert_array_equal(ctx.download(N.SLOT_H), tree["value"][_walk(tree, X2)])
    # fp32 walk on the same tree: identical
    ctx.set_option("tree_bins", 0)
    ctx.tree_predict(tree, N.SLOT_H, 0)
    assert ctx.get_option("last_tree_binned") == 0
    np.testing.assert_array_equal(ctx.download(N.SLOT_H), tree["value"][_walk(tree, X2)])
    ctx.set_option("tree_bins", 1)
    # subspace map + leaf vectors
    if d >= 3:
        sub = np.sort(rng.choice(d, size=max(2, d // 2), replace=False)).astype(np.int32)
        tr = _random_tree(rng, depth, len(sub), [cand[c] for c in sub], n_out=3)
        ctx.alloc(N.SLOT_PROBA, 3, n)
        ctx.tree_predict_multi(tr, N.SLOT_PROBA, subspace=sub)
        assert ctx.get_option("last_tree_binned") == 1
        np.testing.assert_array_equal(ctx.download(N.SLOT_PROBA).reshape(3, n), tr["values"][_walk(tr, X2[:, sub])].T)
    # a column with more than 255 distinct thresholds cannot be ranked in a byte: fp32 walk, still exact
    many = [np.sort(rng.standard_normal(400).astype(np.float32))]
    seen_fallback = False
    for k in range(200):
        tr = _random_tree(rng, 6, d, [many[0]] * d)
        ctx.tree_predict(tr, N.SLOT_H, 0)
        seen_fallback |= ctx.get_option("last_tree_binned") == 0
        np.testing.assert_array_equal(ctx.download(N.SLOT_H), tr["value"][_walk(tr, X2)])
        if seen_fallback:
            break
    assert seen_fallback
    ctx.free(N.SLOT_X)
