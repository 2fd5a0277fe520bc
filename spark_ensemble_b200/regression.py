"""Host-side mirror of the reference's regression ensembles for the hot path:
GBMRegressor / GBMRegressionModel (regression/GBMRegressor.scala) and BaggingRegressionModel.predict
(regression/BaggingRegressor.scala:221-228) — same class names, UID prefixes, Params and defaults; the
per-row RDD closures of train()/predict() are replaced by calls into libse_b200 (sm_100a kernels).

On a JVM host the same substitution is made in Scala (scala/ + jni/se_jni.cpp, see INTEGRATION.md).
"""
from __future__ import annotations

import numpy as np

from . import _native as N
from .context import Context
from .ensemble import (DataFrame, exact_quantile, fit_dummy_regressor, java_string_hash, subspace)
from .gbm_engine import GBMEngine
from .params import (Param, Params, ParamValidators, boosting_params, gbm_params, random_uid,
                     shared_predictor_params, subbag_params)

_REG_LOSSES = ("squared", "absolute", "huber", "quantile")  # GBMRegressor.scala:119-120
_REG_INIT = ("constant", "zero", "base")                     # :121-123


def _extract_instances(est: Params, dataset: DataFrame):
    """Predictor.extractInstances: label cast to double, weight = weightCol if set and non-empty else 1."""
    X = np.asarray(dataset[est("featuresCol")])
    y = np.asarray(dataset[est("labelCol")], dtype=np.float64)
    wc = est("weightCol") if est.isDefined("weightCol") else ""
    w = np.asarray(dataset[wc], dtype=np.float64) if wc else None
    return X, y, w


def bag_counts(n: int, subsample_ratio: float, replacement: bool, seed: int):
    """Multiplicity of every train row in `RDD.sample(replacement, ratio, seed)`; None when the bag is the
    whole set.  Drawn once, because the reference passes the same seed every round (quirk 3).
    Without replacement: Spark's own algorithm for rows in ONE partition (java.util.Random -> per-partition seed ->
    XORShiftRandom -> BernoulliSampler with gap sampling below 0.4), restated in the native library
    (se_spark_bernoulli_sample; unpinned: no Spark here).  With replacement Spark uses commons-math3's
    PoissonDistribution over a Well19937c generator, which is not restated: numpy draws Poisson(ratio).
    On a Spark host the multiplicities come from Spark itself (GBMRegressorNative.scala)."""
    if subsample_ratio == 1.0 and not replacement:
        return None
    if not replacement:
        import ctypes as C
        lib = N.load()
        c = np.zeros(n, dtype=np.float32)
        s64 = int(seed) & 0xFFFFFFFFFFFFFFFF
        s64 = s64 - (1 << 64) if s64 >= (1 << 63) else s64
        N.check(lib.se_spark_bernoulli_sample(C.c_int64(s64), float(subsample_ratio), n, 0, N.fptr(c)))
        return c
    rng = np.random.default_rng(seed & 0xFFFFFFFF)
    return rng.poisson(subsample_ratio, n).astype(np.float32)


def _split_validation(est: Params, dataset: DataFrame):
    vc = est("validationIndicatorCol") if est.isDefined("validationIndicatorCol") else ""
    if vc:
        mask = np.asarray(dataset[vc], dtype=bool)
        return dataset.filter(~mask), dataset.filter(mask)
    return dataset, None


# Param `forestTransform` of the tree-ensemble models: transform evaluates the whole forest in one pass over the
# feature matrix on the device (se_forest_predict / se_forest_classify / se_forest_weighted_median) instead of
# predicting every member on the host and aggregating the stacked outputs.  Off by default.
_pforest = [Param("forestTransform", "transform tree ensembles in one pass over the device-resident features", convert=bool)]


def _member_trees(models):
    """tree_arrays() of every member, or None when there is none or one is not a tree."""
    trees = [m.tree_arrays() for m in models]
    return trees if trees and all(t is not None for t in trees) else None


def _forest_transform(device: int, X, run):
    """Uploads X column-major once and returns run(ctx); None when the rank matrix cannot hold the forest (SE_ERR_STATE:
    a column with more than 255 distinct thresholds), so that the caller takes the member-by-member route."""
    X = np.asarray(X, dtype=np.float32)
    with Context(device) as ctx:
        ctx.alloc(N.SLOT_X, X.shape[1], X.shape[0])
        ctx.upload_rowmajor(N.SLOT_X, X)
        try:
            return run(ctx)
        except N.NativeError as e:
            if e.code != N.SE_ERR_STATE:
                raise
            return None


def _forest_predict(ctx: Context, trees, subspaces, weights, init: float) -> np.ndarray:
    n = ctx.layout(N.SLOT_X)[1]
    ctx.alloc(N.SLOT_RAW, 1, n)
    ctx.forest_predict(trees, N.SLOT_RAW, weights=weights, init=init, subspaces=subspaces)
    return ctx.download(N.SLOT_RAW).astype(np.float64)


class GBMRegressor(Params):
    """regression/GBMRegressor.scala:164-476.  UID prefix "GBMRegressor2" (sic, :229)."""

    def __init__(self, uid: str | None = None, device: int = 0):
        super().__init__(uid or random_uid("GBMRegressor2"))
        self.device = device

    def copy(self, extra=None):
        c = super().copy(extra)
        if c.isDefined("baseLearner"):
            c.set("baseLearner", c("baseLearner").copy(extra))  # :230-234
        return c

    def fit(self, dataset: DataFrame) -> "GBMRegressionModel":
        return self._train(dataset)

    # -- GBMRegressor.train :237-476
    def _train(self, dataset: DataFrame) -> "GBMRegressionModel":
        train_df, valid_df = _split_validation(self, dataset)
        with_validation = valid_df is not None
        X, y, w = _extract_instances(self, train_df)
        Xv, yv, _ = _extract_instances(self, valid_df) if with_validation else (None, None, None)
        n, nv = y.shape[0], (yv.shape[0] if with_validation else 0)
        num_features = X.shape[1]
        loss = self("loss").lower()
        updates = self("updates").lower()
        learner = self("baseLearner")
        num_learners = self("numBaseLearners")
        seed = self("seed")
        counts = bag_counts(n, self("subsampleRatio"), self("replacement"), seed)  # same bag every round (:357-359)
        subspaces = [subspace(self("subspaceRatio"), num_features, seed + i) for i in range(num_learners)]  # :282-284

        # init model :287-303
        init_strategy = self("initStrategy").lower()
        if init_strategy == "base":
            init = learner.fit(X, y, w)
        elif init_strategy == "zero":
            init = fit_dummy_regressor("constant", y, constant=0.0)
        else:
            strat = {"squared": "mean", "absolute": "median", "huber": "median", "quantile": "quantile"}[loss]
            init = fit_dummy_regressor(strat, y, quantile=self("alpha"))

        # huber delta / quantile parameter :305-308
        param = exact_quantile(y, self("alpha")) if loss == "huber" else self("alpha")
        newton = updates == "newton" and loss == "squared"  # HasScalarHessian among selectable losses :369

        # Param `devices` with two or more GPUs: rows are sharded over one context per GPU (sharded.ShardedContext),
        # the per-round scalars are summed across GPUs inside the kernels; everything below is unchanged
        from .sharded import make_context
        ctx = make_context(self.device, self("devices"))
        try:
            eng = GBMEngine(ctx, n, nv, 1, loss, param, has_weights=w is not None)
            const_init = hasattr(init, "prediction")  # Dummy model: broadcast the constant on device
            F0 = init.prediction if const_init else init.predict(X)
            vF0 = (init.prediction if const_init else init.predict(Xv)) if with_validation else None
            eng.load(y, w, F0, yv, vF0)
            on_device_models = bool(self("residentFeatures"))
            if on_device_models:
                eng.load_features(X, Xv)
            if counts is not None:
                ctx.gbm_set_bag(counts)
                in_bag = counts > 0
            best = ctx.gbm_mean_loss(validation=True) if with_validation else 0.0  # :330-335

            models, weights = [], []
            history = []
            eng.residuals(newton)  # residuals of F0; later rounds get them fused with the update
            i = v = 0
            while i < num_learners and v < self("numRounds"):  # :340
                if loss == "huber":  # :342-353: δ = α-quantile of |y − F| (approxQuantile -> exact radix select on device)
                    param = ctx.gbm_abs_residual_quantile(self("alpha"))
                    ctx.gbm_set_loss_param(param)
                    eng.residuals(False)
                sub = subspaces[i]
                r, wout = eng.fetch_residuals(newton)
                fit_w = wout[0] if newton else w
                if counts is None:
                    model = learner.fit(X[:, sub], r[0], fit_w)  # third party :387-396
                else:  # the base learner sees the bag: row i with multiplicity c_i (== weight c_i·w_i)
                    bw = counts[in_bag] if fit_w is None else counts[in_bag] * fit_w[in_bag]
                    model = learner.fit(X[in_bag][:, sub], r[0][in_bag], bw)
                eng.set_direction_from_model(0, model, sub, X)
                if self("optimizedWeights"):  # :398-425
                    if self("lineSearch") == "newton" and loss == "squared":
                        alpha, _, _ = eng.line_search_newton(self("tol"), self("maxIter"))
                    else:
                        alpha, _, _ = eng.line_search_brent(self("tol"), self("maxIter"))
                else:
                    alpha = 1.0
                weight = self("learningRate") * alpha  # :427
                loss_sum, _ = eng.update(weight, residual=(not newton and loss != "huber"), newton=newton)
                models.append(model)
                weights.append(weight)
                history.append({"alpha": alpha, "trainLoss": loss_sum / n if n else float("nan")})
                if with_validation:  # :444-465
                    eng.set_direction_from_model(0, model, sub, Xv, validation=True)
                    err = eng.update_validation(weight)
                    history[-1]["validationLoss"] = err
                    if best - err < self("validationTol") * max(err, 0.01):
                        v += 1
                    elif err < best:
                        best = err
                        v = 0
                i += 1
            keep = i - v  # :474
            model = GBMRegressionModel(weights[:keep], subspaces[:keep], models[:keep], init,
                                       device=self.device)
            self._copyValues(model)
            model.parent = self
            model.trainingHistory = history
            return model
        finally:
            ctx.close()


_p, _d = shared_predictor_params()
_ps, _ds = subbag_params()
_pb, _db = boosting_params()
_pg, _dg = gbm_params()
_preg = [
    Param("loss", "loss function, (case-insensitive). Supported options:" + ",".join(_REG_LOSSES),
          lambda v: v.lower() in _REG_LOSSES, str),
    Param("alpha", "The alpha-quantile of the loss function. Only for huber and quantile loss.", convert=float),
    Param("initStrategy", "strategy for the init predictions (constant, zero, base)",
          lambda v: v in _REG_INIT, str),
    # the one new expert Param (SURVEY.md §5): keep the column-major feature matrix in HBM and evaluate
    # fitted trees / linear models on device instead of model.predict on the host
    Param("residentFeatures", "evaluate base models on device over the HBM-resident feature matrix", convert=bool),
    # expert Param: "brent" = the reference's optimiser (default); "newton" = curvature-based line search on
    # the same objective (dim 1, losses with a hessian): same minimiser within tol, ~6x fewer data passes
    Param("lineSearch", "line-search optimiser for dim 1: brent (reference) or newton", lambda v: v in ("brent", "newton"), str),
    # expert Param: GPUs to shard the rows of a fit over (one context per GPU, contiguous row blocks); [] = `device`
    Param("devices", "CUDA device ordinals to shard the training rows over", lambda v: all(int(d) >= 0 for d in v),
          lambda v: [int(d) for d in v]),
]
_GBM_REG_DEFAULTS = {**_d, **_ds, **_db, **_dg, "loss": "squared", "alpha": 0.9, "initStrategy": "constant", "residentFeatures": False, "lineSearch": "brent",
                     "devices": [], "forestTransform": False,
                     "seed": java_string_hash("org.apache.spark.ml.regression.GBMRegressor")}
GBMRegressor._declare(_p + _ps + _pb + _pg + _preg + _pforest, _GBM_REG_DEFAULTS)


def _stack_model_outputs(models, subspaces, X, extra=None) -> np.ndarray:
    rows = [] if extra is None else [extra]
    for m, s in zip(models, subspaces):
        rows.append(m.predict(X[:, s]))
    if not rows:
        return np.zeros((0, X.shape[0]), dtype=np.float32)
    return np.ascontiguousarray(np.stack(rows), dtype=np.float32)


class GBMRegressionModel(Params):
    """regression/GBMRegressor.scala:512-556; predict :531-539 = init + Σ_i w_i·m_i(x[S_i])."""

    def __init__(self, weights, subspaces, models, init, uid: str | None = None, device: int = 0):
        super().__init__(uid or random_uid("GBMRegressionModel"))
        self.weights = np.asarray(weights, dtype=np.float64)
        self.subspaces = list(subspaces)
        self.models = list(models)
        self.init = init
        self.numModels = len(self.models)
        self.device = device
        self.parent = None

    def _aggregate(self, X) -> np.ndarray:
        n = X.shape[0]
        const_init = hasattr(self.init, "prediction")
        trees = _member_trees(self.models) if self("forestTransform") and const_init else None
        if trees is not None:
            out = _forest_transform(self.device, X, lambda ctx: _forest_predict(ctx, trees, self.subspaces, self.weights,
                                                                                self.init.prediction))
            if out is not None:
                return out
        P = _stack_model_outputs(self.models, self.subspaces, X,
                                 None if const_init else self.init.predict(X))
        a = self.weights if const_init else np.concatenate([[1.0], self.weights])
        with Context(self.device) as ctx:
            ctx.agg_configure(N.AGG_GBM_REGRESSOR, P.shape[0], 0, 1, 0, n)
            if P.shape[0]:
                ctx.upload(N.SLOT_P, P)
            ctx.agg_run(a, [self.init.prediction if const_init else 0.0])
            return ctx.download(N.SLOT_RAW).astype(np.float64)

    def transform(self, dataset: DataFrame) -> DataFrame:
        X = np.asarray(dataset[self("featuresCol")])
        return dataset.withColumn(self("predictionCol"), self._aggregate(X))

    def predict(self, features) -> float:
        return float(self._aggregate(np.asarray(features).reshape(1, -1))[0])


GBMRegressionModel._declare(_p + _ps + _pb + _pg + _preg + _pforest, _GBM_REG_DEFAULTS)


# ---- Bagging (train is out of the hot path: embarrassingly parallel base-learner fits) ---------------
class BaggingRegressor(Params):
    """regression/BaggingRegressor.scala:77-172.  Only the model's predict is on the hot path; train
    here is the minimal host loop (one base learner per bootstrap bag)."""

    def __init__(self, uid: str | None = None, device: int = 0):
        super().__init__(uid or random_uid("BaggingRegressor"))
        self.device = device

    def fit(self, dataset: DataFrame) -> "BaggingRegressionModel":
        X, y, w = _extract_instances(self, dataset)
        n, d = X.shape
        seed = self("seed")
        M = self("numBaseLearners")
        subs = [subspace(self("subspaceRatio"), d, seed + i) for i in range(M)]
        models = []
        rng = np.random.default_rng(seed & 0xFFFFFFFF)  # same sample for every bag: reference quirk 3
        if self("replacement"):
            counts = rng.poisson(self("subsampleRatio"), n).astype(np.float64)
        else:
            counts = (rng.random(n) < self("subsampleRatio")).astype(np.float64)
        bw = counts if w is None else counts * w
        keep = bw > 0
        for i in range(M):
            models.append(self("baseLearner").fit(X[keep][:, subs[i]], y[keep], bw[keep]))
        m = BaggingRegressionModel(subs, models, device=self.device)
        self._copyValues(m)
        m.parent = self
        return m


_pbag = [Param("numBaseLearners", "number of base learners", ParamValidators.gtEq(1), int),
         Param("baseLearner", "base learner"),
         Param("parallelism", "the number of threads to use when running parallel algorithms (>= 1)",
               ParamValidators.gtEq(1), int)]
_BAG_REG_DEFAULTS = {**_d, **_ds, "numBaseLearners": 10, "parallelism": 1, "forestTransform": False,
                     "seed": java_string_hash("org.apache.spark.ml.regression.BaggingRegressor")}
BaggingRegressor._declare(_p + _ps + _pbag + _pforest, _BAG_REG_DEFAULTS)


class BaggingRegressionModel(Params):
    """regression/BaggingRegressor.scala:208-235; predict :221-228 = (Σ_i m_i(x[S_i])) / numModels."""

    def __init__(self, subspaces, models, uid: str | None = None, device: int = 0):
        super().__init__(uid or random_uid("BaggingRegressionModel"))
        self.subspaces, self.models = list(subspaces), list(models)
        self.numModels = len(self.models)
        self.device = device
        self.parent = None

    def _aggregate(self, X) -> np.ndarray:
        trees = _member_trees(self.models) if self("forestTransform") else None
        if trees is not None:  # (Σ_i m_i) / M as Σ_i m_i / M
            out = _forest_transform(self.device, X, lambda ctx: _forest_predict(
                ctx, trees, self.subspaces, np.full(len(trees), 1.0 / len(trees)), 0.0))
            if out is not None:
                return out
        P = _stack_model_outputs(self.models, self.subspaces, X)
        with Context(self.device) as ctx:
            ctx.agg_configure(N.AGG_BAGGING_REGRESSOR, P.shape[0], 0, 1, 0, X.shape[0])
            ctx.upload(N.SLOT_P, P)
            ctx.agg_run()
            return ctx.download(N.SLOT_RAW).astype(np.float64)

    def transform(self, dataset: DataFrame) -> DataFrame:
        return dataset.withColumn(self("predictionCol"), self._aggregate(np.asarray(dataset[self("featuresCol")])))

    def predict(self, features) -> float:
        return float(self._aggregate(np.asarray(features).reshape(1, -1))[0])


BaggingRegressionModel._declare(_p + _ps + _pbag + _pforest, _BAG_REG_DEFAULTS)


# ---- BoostingRegressor (AdaBoost.R2, Drucker 1997): SURVEY.md §8f-2 -----------------------------------
class BoostingRegressor(Params):
    """regression/BoostingRegressor.scala:138-282.  Per round: maxError, estimatorError = Σ wₙ·loss, weight
    update wₙ·β^(1-loss), Σw' — three streaming passes on the device instead of four RDD jobs."""

    def __init__(self, uid: str | None = None, device: int = 0):
        super().__init__(uid or random_uid("BoostingRegressor"))
        self.device = device

    def fit(self, dataset: DataFrame) -> "BoostingRegressionModel":
        X, y, w = _extract_instances(self, dataset)
        n = y.shape[0]
        loss_type = self("lossType").lower()
        learner = self("baseLearner")
        models, est_weights, history = [], [], []
        ctx = Context(self.device)
        try:
            ctx.boostreg_configure(n)
            resident = bool(self("residentFeatures"))
            if resident:  # column-major X in HBM: fitted trees / linear models are evaluated on device (no upload per round)
                ctx.alloc(N.SLOT_X, X.shape[1], n)
                ctx.upload_rowmajor(N.SLOT_X, X)
            ctx.upload(N.SLOT_Y, y)
            ctx.upload(N.SLOT_BW, np.ones(n) if w is None else w)  # :205
            sum_w = ctx.slot_sum(N.SLOT_BW)                          # :212
            i, best, done = 0, 0, False
            while i < self("numBaseLearners") and not done and sum_w > 0:  # :218
                wn = ctx.download(N.SLOT_BW, scale=1.0 / sum_w)     # :222-225
                model = learner.fit(X, y, wn)                        # third party :231-233
                _predict_into(ctx, model, X, resident)
                max_error = ctx.boostreg_max_error()                 # :235-238
                if max_error == 0:                                   # :240-243
                    best, done = i, True
                est_err = ctx.boostreg_error(sum_w, loss_type, max_error)  # :248-254
                if est_err >= 0.5:                                   # :256
                    best, done = i - 1, True
                beta = est_err / (1 - est_err)
                est_weight = 1.0 if beta == 0.0 else float(np.log(1.0 / beta))
                sum_w = ctx.boostreg_update(sum_w, loss_type, max_error, beta) if beta > 0 else 0.0  # :261-268
                est_weights.append(est_weight)
                models.append(model)
                history.append({"maxError": max_error, "estimatorError": est_err, "sumWeights": sum_w})
                best = i
                i += 1
            best += 1
            m = BoostingRegressionModel(est_weights[:best], models[:best], device=self.device)
            self._copyValues(m)
            m.parent = self
            m.trainingHistory = history
            return m
        finally:
            ctx.close()


def _predict_into(ctx: Context, model, X, resident: bool):
    """The member's predictions in SLOT_PRED: on the device over the resident X for a tree or a linear model, otherwise
    model.predict on the host + upload (the reference's path)."""
    t = model.tree_arrays() if resident else None
    if t is not None:
        ctx.tree_predict(t, N.SLOT_PRED, 0)
        return
    lin = model.linear_arrays() if resident else None
    if lin is not None:
        ctx.linear_predict(lin["coef"], float(lin["intercept"]), N.SLOT_PRED, 0)
        return
    ctx.upload(N.SLOT_PRED, model.predict(X))


def _forest_median(ctx: Context, trees, weights) -> np.ndarray:
    n = ctx.layout(N.SLOT_X)[1]
    ctx.alloc(N.SLOT_RAW, 1, n)
    ctx.forest_weighted_median(trees, N.SLOT_RAW, weights)
    return ctx.download(N.SLOT_RAW).astype(np.float64)


_pbr = [Param("lossType", "loss function, exponential by default (case-insensitive). Supported: exponential,squared,linear",
              lambda v: v.lower() in ("exponential", "squared", "linear"), str),
        Param("votingStrategy", "voting strategy, (case-insensitive). Supported options: median,mean",
              lambda v: v.lower() in ("median", "mean"), str),
        Param("seed", "random seed", convert=int),
        Param("residentFeatures", "evaluate base models on device over the HBM-resident feature matrix", convert=bool)]
_BOOST_REG_DEFAULTS = {**_d, **_db, "lossType": "exponential", "votingStrategy": "median", "residentFeatures": False,
                       "forestTransform": False, "seed": java_string_hash("org.apache.spark.ml.regression.BoostingRegressor")}
BoostingRegressor._declare(_p + _pb + _pbr + _pforest, _BOOST_REG_DEFAULTS)


class BoostingRegressionModel(Params):
    """regression/BoostingRegressor.scala:318-360: weighted median (ensemble/Utils.scala:26-40) or weighted
    mean of the members' predictions."""

    def __init__(self, weights, models, uid: str | None = None, device: int = 0):
        super().__init__(uid or random_uid("BoostingRegressionModel"))
        self.weights = np.asarray(weights, dtype=np.float64)
        self.models = list(models)
        self.numModels = len(self.models)
        self.device = device
        self.parent = None

    def _aggregate(self, X) -> np.ndarray:
        median = self("votingStrategy").lower() == "median"
        trees = _member_trees(self.models) if self("forestTransform") else None
        if trees is not None:
            if median:  # the weighted median of the leaves, fused with the forest walk (se_forest_weighted_median)
                run = lambda ctx: _forest_median(ctx, trees, self.weights)
            else:  # dot(predictions, weights) / Σ weights (BoostingRegressor.scala:339-342) as Σ_i (w_i / Σw) · m_i
                sum_w = 0.0
                for a in self.weights:  # fp64, model order
                    sum_w += float(a)
                run = lambda ctx: _forest_predict(ctx, trees, None, self.weights / sum_w, 0.0)
            # None: more than 64 members, a forest beyond one chunk or a column with > 255 thresholds (member route)
            out = _forest_transform(self.device, X, run)
            if out is not None:
                return out
        P = np.ascontiguousarray(np.stack([m.predict(X) for m in self.models]), dtype=np.float32)
        kind = N.AGG_BOOSTING_REG_MEDIAN if median else N.AGG_BOOSTING_REG_MEAN
        with Context(self.device) as ctx:
            ctx.agg_configure(kind, P.shape[0], 0, 1, 0, X.shape[0])
            ctx.upload(N.SLOT_P, P)
            ctx.agg_run(self.weights)
            return ctx.download(N.SLOT_RAW).astype(np.float64)

    def transform(self, dataset: DataFrame) -> DataFrame:
        return dataset.withColumn(self("predictionCol"), self._aggregate(np.asarray(dataset[self("featuresCol")])))

    def predict(self, features) -> float:
        return float(self._aggregate(np.asarray(features).reshape(1, -1))[0])


BoostingRegressionModel._declare(_p + _pb + _pbr + _pforest, _BOOST_REG_DEFAULTS)
