"""Host-side mirror of the reference's classification ensembles for the hot path:
GBMClassifier (classification/GBMClassifier.scala), BoostingClassifier SAMME / SAMME.R
(classification/BoostingClassifier.scala) and the predictRaw/probability aggregation of
GBM / Boosting / Bagging classification models — same names, UID prefixes, Params and defaults, with
the per-row RDD closures replaced by calls into libse_b200.
"""
from __future__ import annotations

import math

import numpy as np

from . import _native as N
from .context import Context
from .ensemble import DataFrame, fit_dummy_classifier, java_string_hash, subspace
from .gbm_engine import GBMEngine
from .params import (Param, Params, ParamValidators, boosting_params, gbm_params, random_uid,
                     shared_classifier_params, shared_predictor_params, subbag_params)
from .regression import (_extract_instances, _forest_transform, _member_trees, _pforest, _split_validation,
                         bag_counts)

_CLS_LOSSES = ("logloss", "exponential", "bernoulli")  # GBMClassifier.scala:102-103
_CLS_INIT = ("uniform", "prior")                        # :104-106


def _num_classes(y: np.ndarray) -> int:
    """Classifier.getNumClasses: max label + 1 (labels are 0..K-1 doubles)."""
    return int(np.max(y)) + 1 if y.size else 0


def _validate_labels(y: np.ndarray, num_classes: int):
    """Classifier.validateLabel: non-negative integers below numClasses."""
    if y.size and (np.any(y < 0) or np.any(y != np.floor(y)) or np.any(y >= num_classes)):
        raise ValueError(f"Classifier was given dataset with invalid label; labels must be integers in [0, {num_classes})")


class _ClassifierModelBase(Params):
    """ProbabilisticClassificationModel.transform: rawPrediction, probability, prediction columns."""

    numClasses: int

    def _raw_prob_label(self, X):  # -> (raw [n,C], prob [n,C], label [n])
        raise NotImplementedError

    def transform(self, dataset: DataFrame) -> DataFrame:
        X = np.asarray(dataset[self("featuresCol")])
        raw, prob, label = self._raw_prob_label(X)
        out = dataset
        if self("rawPredictionCol"):
            out = out.withColumn(self("rawPredictionCol"), raw)
        if self("probabilityCol"):
            out = out.withColumn(self("probabilityCol"), prob)
        if self("predictionCol"):
            out = out.withColumn(self("predictionCol"), label)
        return out

    def predictRaw(self, features) -> np.ndarray:
        return self._raw_prob_label(np.asarray(features).reshape(1, -1))[0][0]

    def predictProbability(self, features) -> np.ndarray:
        return self._raw_prob_label(np.asarray(features).reshape(1, -1))[1][0]

    def predict(self, features) -> float:
        return float(self._raw_prob_label(np.asarray(features).reshape(1, -1))[2][0])

    def _fetch(self, ctx: Context):
        raw = ctx.download(N.SLOT_RAW).astype(np.float64)
        prob = ctx.download(N.SLOT_PROB).astype(np.float64)
        label = ctx.download(N.SLOT_LABEL).astype(np.float64)
        C = self._out_classes
        return raw.reshape(C, -1).T, prob.reshape(C, -1).T, label

    def _forest(self, X, trees, kind, subspaces=None, dim=1, loss=0, weights=None, init=None):
        """Param forestTransform: the members' trees in one pass over X on the device (se_forest_classify).  None when
        it is off, a member is not a tree, or the rank matrix cannot hold the forest: the member route runs then."""
        if not self("forestTransform") or trees is None:
            return None

        def run(ctx):
            ctx.forest_classify(trees, kind, self.numClasses, dim=dim, loss=loss, weights=weights, init=init,
                                subspaces=subspaces)
            return self._fetch(ctx)
        return _forest_transform(self.device, X, run)


# ================================================================================ GBMClassifier
class GBMClassifier(Params):
    """classification/GBMClassifier.scala:146-496.  UID prefix "GBMClassifier" (:211)."""

    def __init__(self, uid: str | None = None, device: int = 0):
        super().__init__(uid or random_uid("GBMClassifier"))
        self.device = device

    def copy(self, extra=None):
        c = super().copy(extra)
        if c.isDefined("baseLearner"):
            c.set("baseLearner", c("baseLearner").copy(extra))
        return c

    def fit(self, dataset: DataFrame) -> "GBMClassificationModel":
        train_df, valid_df = _split_validation(self, dataset)
        with_validation = valid_df is not None
        X, y, w = _extract_instances(self, train_df)
        Xv, yv, _ = _extract_instances(self, valid_df) if with_validation else (None, None, None)
        n, nv = y.shape[0], (yv.shape[0] if with_validation else 0)
        num_features = X.shape[1]
        num_classes = _num_classes(np.asarray(dataset[self("labelCol")], dtype=np.float64))
        _validate_labels(y, num_classes)
        loss = self("loss").lower()
        dim = num_classes if loss == "logloss" else 1  # GBMLoss.scala:198,270,295
        if dim == 1 and num_classes != 2:
            raise ValueError(f"loss {loss} is binary; got numClasses={num_classes}")
        learner = self("baseLearner")
        num_learners = self("numBaseLearners")
        seed = self("seed")
        counts = bag_counts(n, self("subsampleRatio"), self("replacement"), seed)  # :329-331
        subspaces = [subspace(self("subspaceRatio"), num_features, seed + i) for i in range(num_learners)]
        newton = self("updates").lower() == "newton"  # every classification loss HasHessian (:338)

        # init :275-288 — binary "prior" with dim 1 stores the FULL log-odds (reference quirk 5)
        init_strategy = self("initStrategy").lower()
        if init_strategy == "prior" and dim == 1 and num_classes == 2:
            p1 = float(np.mean(y == 1.0))
            logodds = math.log(p1 / (1 - p1))
            init_raw = np.array([logodds])
        else:
            init_raw = fit_dummy_classifier(init_strategy, y, num_classes).rawPrediction
            if init_raw.shape[0] != dim:
                raise ValueError("prior init needs every class present in the training labels")

        from .sharded import make_context
        ctx = make_context(self.device, self("devices"))  # Param `devices`: rows sharded over several GPUs
        try:
            eng = GBMEngine(ctx, n, nv, dim, loss, 0.0, has_weights=w is not None)
            eng.load(y, w, init_raw, yv, init_raw if with_validation else None)
            if bool(self("residentFeatures")):
                eng.load_features(X, Xv)
            if counts is not None:
                ctx.gbm_set_bag(counts)
                in_bag = counts > 0
            best = ctx.gbm_mean_loss(validation=True) if with_validation else 0.0  # :315-320
            models, weights, history = [], [], []
            eng.residuals(newton)
            i = v = 0
            while i < num_learners and v < self("numRounds"):  # :325
                sub = subspaces[i]
                r, wout = eng.fetch_residuals(newton)
                imodels = []
                for j in range(dim):  # one regressor per dimension (:377-411; Futures in the reference)
                    fit_w = wout[j] if newton else w
                    if counts is None:
                        imodels.append(learner.fit(X[:, sub], r[j], fit_w))
                    else:
                        bw = counts[in_bag] if fit_w is None else counts[in_bag] * fit_w[in_bag]
                        imodels.append(learner.fit(X[in_bag][:, sub], r[j][in_bag], bw))
                for j in range(dim):
                    eng.set_direction_from_model(j, imodels[j], sub, X)
                if self("optimizedWeights"):  # :413-431
                    if self("lineSearch") == "newton" and dim == 1:
                        a1, _, _ = eng.line_search_newton(self("tol"), self("maxIter"))
                        alpha = np.array([a1])
                    else:
                        alpha, _, _ = eng.line_search_lbfgsb(self("tol"), self("maxIter"))
                else:
                    alpha = np.ones(dim)
                iweights = np.asarray(alpha) * self("learningRate")  # :432
                loss_sum, _ = eng.update(iweights, residual=not newton, newton=newton)
                models.append(imodels)
                weights.append(iweights)
                history.append({"alpha": np.asarray(alpha).copy(), "trainLoss": loss_sum / n if n else float("nan")})
                if with_validation:  # :451-479
                    for j in range(dim):
                        eng.set_direction_from_model(j, imodels[j], sub, Xv, validation=True)
                    err = eng.update_validation(iweights)
                    history[-1]["validationLoss"] = err
                    if best - err < self("validationTol") * max(err, 0.01):
                        v += 1
                    elif err < best:
                        best = err
                        v = 0
                i += 1
            keep = i - v  # :488-494
            model = GBMClassificationModel(num_classes, weights[:keep], subspaces[:keep], models[:keep],
                                           init_raw, dim, device=self.device)
            self._copyValues(model)
            model.parent = self
            model.trainingHistory = history
            return model
        finally:
            ctx.close()


_p, _d = shared_predictor_params()
_pc, _dc = shared_classifier_params()
_ps, _ds = subbag_params()
_pb, _db = boosting_params()
_pg, _dg = gbm_params()
_pcls = [
    Param("loss", "loss function, (case-insensitive). Supported options:" + ",".join(_CLS_LOSSES),
          lambda v: v.lower() in _CLS_LOSSES, str),
    Param("initStrategy", "strategy for the init predictions (uniform, prior)", lambda v: v in _CLS_INIT, str),
    Param("residentFeatures", "evaluate base models on device over the HBM-resident feature matrix", convert=bool),
    # expert Param: "brent" = the reference's optimiser (default); "newton" = curvature-based line search on
    # the same objective (dim 1, losses with a hessian): same minimiser within tol, ~6x fewer data passes
    Param("lineSearch", "line-search optimiser for dim 1: brent (reference) or newton", lambda v: v in ("brent", "newton"), str),
    Param("devices", "CUDA device ordinals to shard the training rows over", lambda v: all(int(d) >= 0 for d in v),
          lambda v: [int(d) for d in v]),
]
_GBM_CLS_DEFAULTS = {**_d, **_dc, **_ds, **_db, **_dg, "loss": "logloss", "initStrategy": "prior",
                     "residentFeatures": False, "lineSearch": "brent", "devices": [], "forestTransform": False,
                     "seed": java_string_hash("org.apache.spark.ml.classification.GBMClassifier")}
GBMClassifier._declare(_p + _pc + _ps + _pb + _pg + _pcls + _pforest, _GBM_CLS_DEFAULTS)


class GBMClassificationModel(_ClassifierModelBase):
    """classification/GBMClassifier.scala:532-612; predictRaw :567-589, raw2probability :564-565."""

    def __init__(self, numClasses, weights, subspaces, models, init_raw, dim, uid=None, device: int = 0):
        super().__init__(uid or random_uid("GBMClassificationModel"))
        self.numClasses = int(numClasses)
        self.weights = [np.asarray(wt, dtype=np.float64) for wt in weights]
        self.subspaces, self.models = list(subspaces), [list(m) for m in models]
        self.init = np.asarray(init_raw, dtype=np.float64)
        self.dim = int(dim)
        self.numModels = len(self.models)
        self.device = device
        self.parent = None
        self._out_classes = 2 if (self.dim == 1 and self.numClasses == 2) else self.dim

    def _raw_prob_label(self, X):
        n, M, dim = X.shape[0], self.numModels, self.dim
        if self("forestTransform"):  # tree t = models(t // dim)(t % dim)
            trees = _member_trees([m for ms in self.models for m in ms])
            res = self._forest(X, trees, N.AGG_GBM_CLASSIFIER, [s for s in self.subspaces for _ in range(dim)], dim,
                               self("loss").lower(), np.stack(self.weights) if M else None, self.init)
            if res is not None:
                return res
        P = np.zeros((max(M, 1), dim, n), dtype=np.float32)
        for i in range(M):
            Xs = X[:, self.subspaces[i]]
            for j in range(dim):
                P[i, j] = self.models[i][j].predict(Xs)
        a = np.stack(self.weights) if M else np.zeros((1, dim))
        with Context(self.device) as ctx:
            ctx.agg_configure(N.AGG_GBM_CLASSIFIER, max(M, 1), self.numClasses, dim, self("loss").lower(), n)
            ctx.upload(N.SLOT_P, P)
            ctx.agg_run(a, self.init)
            return self._fetch(ctx)


GBMClassificationModel._declare(_p + _pc + _ps + _pb + _pg + _pcls + _pforest, _GBM_CLS_DEFAULTS)


# ================================================================================ BoostingClassifier
class BoostingClassifier(Params):
    """classification/BoostingClassifier.scala:105-282: AdaBoost SAMME ("discrete") / SAMME.R ("real")."""

    def __init__(self, uid: str | None = None, device: int = 0):
        super().__init__(uid or random_uid("BoostingClassifier"))
        self.device = device

    def fit(self, dataset: DataFrame) -> "BoostingClassificationModel":
        X, y, w = _extract_instances(self, dataset)
        n = y.shape[0]
        K = _num_classes(y)
        _validate_labels(y, K)
        real = self("algorithm").lower() == "real"
        learner = self("baseLearner")
        models, est_weights, history = [], [], []
        ctx = Context(self.device)
        try:
            ctx.boost_configure(n, K, real)
            resident = bool(self("residentFeatures"))
            if resident:  # column-major X in HBM: fitted trees are evaluated on device (no K x n upload per round)
                ctx.alloc(N.SLOT_X, X.shape[1], n)
                ctx.upload_rowmajor(N.SLOT_X, X)
            ctx.upload(N.SLOT_Y, y)
            ctx.upload(N.SLOT_BW, np.ones(n) if w is None else w)  # boostingWeights = instances.map(_.weight) :168
            sum_w = ctx.slot_sum(N.SLOT_BW)  # :175
            i, done = 0, False
            while i < self("numBaseLearners") and not done and sum_w > 0:  # :180
                wn = ctx.download(N.SLOT_BW, scale=1.0 / sum_w)  # weight = boostingWeight / sumWeights :184-187
                model = learner.fit(X, y, wn, num_classes=K)    # third party :189-195
                if real:  # SAMME.R :198-230
                    if not hasattr(model, "predictProbability"):
                        raise RuntimeError('algorithm "real" is not compatible with base learner')  # :261-263
                    t = model.tree_arrays() if resident else None
                    if t is not None:
                        ctx.tree_predict_multi(t, N.SLOT_PROBA)
                    else:
                        P = model.predictProbability(X)
                        ctx.upload(N.SLOT_PROBA, np.ascontiguousarray(P.T, dtype=np.float32))
                    err, new_sum = ctx.boost_real_update(sum_w)
                    if err <= 0:
                        done = True
                    est_weights.append(1.0)  # :212
                    models.append(model)
                else:  # SAMME :231-260
                    t = model.tree_arrays() if resident else None
                    if t is not None:
                        ctx.tree_predict(t, N.SLOT_PRED, 0)
                    else:
                        ctx.upload(N.SLOT_PRED, model.predict(X))
                    err = ctx.boost_discrete_error(sum_w)
                    if err <= 0:
                        done = True
                    beta = err / ((1 - err) * (K - 1))
                    est_weights.append(1.0 if beta == 0.0 else math.log(1.0 / beta))
                    models.append(model)
                    if err >= 1.0 - (1.0 / K):  # :252 drop this model and stop
                        i -= 1
                        done = True
                    new_sum = ctx.boost_discrete_update(sum_w, beta if beta != 0.0 else 0.0)
                history.append({"estimatorError": err, "sumWeights": new_sum})
                sum_w = new_sum  # :269
                i += 1
            keep = max(i, 0)
            model = BoostingClassificationModel(K, est_weights[:keep], models[:keep], device=self.device)
            self._copyValues(model)
            model.parent = self
            model.trainingHistory = history
            return model
        finally:
            ctx.close()


_pboost = [Param("algorithm", "algorithm, (case-insensitive). Supported options: discrete,real",
                 lambda v: v.lower() in ("discrete", "real"), str),
           Param("residentFeatures", "evaluate base models on device over the HBM-resident feature matrix", convert=bool)]
_BOOST_DEFAULTS = {**_d, **_dc, **_db, "algorithm": "discrete", "residentFeatures": False, "forestTransform": False,
                   "seed": java_string_hash("org.apache.spark.ml.classification.BoostingClassifier")}
BoostingClassifier._declare(_p + _pc + _pb + _pboost + _pforest + [Param("seed", "random seed", convert=int)], _BOOST_DEFAULTS)


class BoostingClassificationModel(_ClassifierModelBase):
    """classification/BoostingClassifier.scala:318-404; predictRawReal :348-364, predictRawDiscrete
    :366-382, raw2probabilityInPlace :342-346."""

    def __init__(self, numClasses, weights, models, uid=None, device: int = 0):
        super().__init__(uid or random_uid("BoostingClassificationModel"))
        self.numClasses = int(numClasses)
        self.weights = np.asarray(weights, dtype=np.float64)
        self.models = list(models)
        self.numModels = len(self.models)
        self.device = device
        self.parent = None
        self._out_classes = self.numClasses

    def _raw_prob_label(self, X):
        n, M, K = X.shape[0], self.numModels, self.numClasses
        real = self("algorithm").lower() == "real"
        res = self._forest(X, _member_trees(self.models) if self("forestTransform") else None,
                           N.AGG_BOOSTING_REAL if real else N.AGG_BOOSTING_DISCRETE,
                           weights=None if real else self.weights)
        if res is not None:
            return res
        with Context(self.device) as ctx:
            if real:
                P = np.zeros((max(M, 1), K, n), dtype=np.float32)
                for i, m in enumerate(self.models):
                    P[i] = m.predictProbability(X).T
                if M == 0:
                    P[:] = 1.0
                ctx.agg_configure(N.AGG_BOOSTING_REAL, max(M, 1), K, 1, 0, n)
                ctx.upload(N.SLOT_P, P)
                ctx.agg_run()
            else:
                V = np.zeros((max(M, 1), n), dtype=np.float32)
                for i, m in enumerate(self.models):
                    V[i] = m.predict(X)
                ctx.agg_configure(N.AGG_BOOSTING_DISCRETE, max(M, 1), K, 1, 0, n)
                ctx.upload(N.SLOT_P, V)
                ctx.agg_run(self.weights if M else np.zeros(1))
            return self._fetch(ctx)


BoostingClassificationModel._declare(_p + _pc + _pb + _pboost + _pforest + [Param("seed", "random seed", convert=int)], _BOOST_DEFAULTS)


# ================================================================================ BaggingClassifier
class BaggingClassifier(Params):
    """classification/BaggingClassifier.scala:106-207. Only the model's predictRaw is on the hot path."""

    def __init__(self, uid: str | None = None, device: int = 0):
        super().__init__(uid or random_uid("BaggingClassifier"))
        self.device = device

    def fit(self, dataset: DataFrame) -> "BaggingClassificationModel":
        X, y, w = _extract_instances(self, dataset)
        n, d = X.shape
        K = _num_classes(y)
        seed, M = self("seed"), self("numBaseLearners")
        subs = [subspace(self("subspaceRatio"), d, seed + i) for i in range(M)]
        rng = np.random.default_rng(seed & 0xFFFFFFFF)
        counts = (rng.poisson(self("subsampleRatio"), n) if self("replacement")
                  else (rng.random(n) < self("subsampleRatio"))).astype(np.float64)
        bw = counts if w is None else counts * w
        keep = bw > 0
        models = [self("baseLearner").fit(X[keep][:, subs[i]], y[keep], bw[keep], num_classes=K) for i in range(M)]
        m = BaggingClassificationModel(K, subs, models, device=self.device)
        self._copyValues(m)
        m.parent = self
        return m


_pbagc = [Param("numBaseLearners", "number of base learners", ParamValidators.gtEq(1), int),
          Param("baseLearner", "base learner"),
          Param("votingStrategy", "voting strategy, (case-insensitive). Supported options: soft,hard",
                lambda v: v.lower() in ("soft", "hard"), str),
          Param("parallelism", "threads", ParamValidators.gtEq(1), int)]
_BAG_CLS_DEFAULTS = {**_d, **_dc, **_ds, "numBaseLearners": 10, "votingStrategy": "hard", "parallelism": 1,
                     "forestTransform": False,
                     "seed": java_string_hash("org.apache.spark.ml.classification.BaggingClassifier")}
BaggingClassifier._declare(_p + _pc + _ps + _pbagc + _pforest, _BAG_CLS_DEFAULTS)


class BaggingClassificationModel(_ClassifierModelBase):
    """classification/BaggingClassifier.scala:243-300; predictRaw :260-283, raw2probability :285-287."""

    def __init__(self, numClasses, subspaces, models, uid=None, device: int = 0):
        super().__init__(uid or random_uid("BaggingClassificationModel"))
        self.numClasses = int(numClasses)
        self.subspaces, self.models = list(subspaces), list(models)
        self.numModels = len(self.models)
        self.device = device
        self.parent = None
        self._out_classes = self.numClasses

    def _raw_prob_label(self, X):
        n, M, K = X.shape[0], self.numModels, self.numClasses
        soft = self("votingStrategy").lower() == "soft"
        res = self._forest(X, _member_trees(self.models) if self("forestTransform") else None,
                           N.AGG_BAGGING_SOFT if soft else N.AGG_BAGGING_HARD, self.subspaces)
        if res is not None:
            return res
        with Context(self.device) as ctx:
            if soft:
                P = np.zeros((M, K, n), dtype=np.float32)
                for i, m in enumerate(self.models):
                    P[i] = m.predictProbability(X[:, self.subspaces[i]]).T
                ctx.agg_configure(N.AGG_BAGGING_SOFT, M, K, 1, 0, n)
            else:
                P = np.zeros((M, n), dtype=np.float32)
                for i, m in enumerate(self.models):
                    P[i] = m.predict(X[:, self.subspaces[i]])
                ctx.agg_configure(N.AGG_BAGGING_HARD, M, K, 1, 0, n)
            ctx.upload(N.SLOT_P, P)
            ctx.agg_run()
            return self._fetch(ctx)


BaggingClassificationModel._declare(_p + _pc + _ps + _pbagc + _pforest, _BAG_CLS_DEFAULTS)
