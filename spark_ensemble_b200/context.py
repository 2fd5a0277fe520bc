"""One GPU == one row shard: a thin, numpy-friendly wrapper over the se_ctx C ABI.

Every method is one call into libse_b200 (include/se_abi.h); no arithmetic of the hot path happens
in Python.  Host arrays are fp32 (the device storage type); scalars come back as Python floats (fp64).
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _native as N


def _flatten_trees(trees, subspaces, leaf_key):
    """Concatenated node arrays of a forest (offsets, feature, threshold, left, right, leaf) as se_forest_predict /
    se_forest_classify take them: tree-local children, features mapped through each tree's subspace to GLOBAL columns,
    tree[leaf_key] flattened per node ([n_nodes] or [n_nodes, width])."""
    offs = np.zeros(len(trees) + 1, dtype=np.int32)
    f, t, l, r, v = [], [], [], [], []
    for i, tr in enumerate(trees):
        fi = np.asarray(tr["feature"], dtype=np.int32)
        if subspaces is not None and subspaces[i] is not None:
            sub = np.asarray(subspaces[i], dtype=np.int32)
            if np.any(fi >= sub.size):
                raise ValueError(f"tree {i}: feature index outside its subspace")
            fi = np.where(fi >= 0, sub[np.maximum(fi, 0)], fi).astype(np.int32)
        f.append(fi)
        t.append(np.asarray(tr["threshold"], dtype=np.float32))
        l.append(np.asarray(tr["left"], dtype=np.int32))
        r.append(np.asarray(tr["right"], dtype=np.int32))
        v.append(np.asarray(tr[leaf_key], dtype=np.float32).reshape(-1))
        offs[i + 1] = offs[i] + fi.size
    return (offs,) + tuple(np.ascontiguousarray(np.concatenate(a)) for a in (f, t, l, r, v))


class Context:
    def __init__(self, device: int = 0):
        self._lib = N.load()
        self._h = C.c_void_p()
        N.check(self._lib.se_ctx_create(int(device), C.byref(self._h)))
        self.device = int(device)

    # ---- lifecycle
    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self._lib.se_ctx_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _ck(self, rc):
        N.check(rc, self._h)

    def sync(self):
        self._ck(self._lib.se_ctx_sync(self._h))

    @property
    def launch_count(self) -> int:
        v = C.c_int64()
        self._ck(self._lib.se_ctx_launch_count(self._h, C.byref(v)))
        return v.value

    def set_timing(self, on: bool):
        self._ck(self._lib.se_ctx_set_timing(self._h, int(on)))

    def last_ms(self) -> float:
        v = C.c_double()
        self._ck(self._lib.se_ctx_last_ms(self._h, C.byref(v)))
        return v.value

    def timer_start(self):
        self._ck(self._lib.se_ctx_timer_start(self._h))

    def timer_stop(self) -> float:
        v = C.c_double()
        self._ck(self._lib.se_ctx_timer_stop(self._h, C.byref(v)))
        return v.value

    def kernel_timing(self, on: bool):
        self._ck(self._lib.se_ctx_kernel_timing(self._h, int(on)))

    def kernel_times(self) -> dict:
        out = {}
        for i, name in enumerate(N.KERNEL_FAMILIES):
            ms, cnt = C.c_double(), C.c_int64()
            self._ck(self._lib.se_ctx_kernel_time(self._h, i, C.byref(ms), C.byref(cnt)))
            if cnt.value:
                out[name] = {"ms": ms.value, "launches": cnt.value}
        return out

    def kernel_times_reset(self):
        self._ck(self._lib.se_ctx_kernel_time_reset(self._h))

    def set_option(self, key: str, value: float):
        """Tunables by name (se_ctx_set_option): fused_round, ls_mode, l2_persist, peer_timeout_ms, ..."""
        self._ck(self._lib.se_ctx_set_option(self._h, key.encode(), float(value)))

    def get_option(self, key: str) -> float:
        v = C.c_double()
        self._ck(self._lib.se_ctx_get_option(self._h, key.encode(), C.byref(v)))
        return v.value

    # ---- communicator
    @staticmethod
    def comm_unique_id() -> bytes:
        buf = C.create_string_buffer(N.COMM_ID_BYTES)
        N.check(N.load().se_comm_unique_id(buf, N.COMM_ID_BYTES))
        return buf.raw

    def comm_init(self, nranks: int, rank: int, uid: bytes | None):
        buf = C.create_string_buffer(uid, N.COMM_ID_BYTES) if uid is not None else None
        self._ck(self._lib.se_comm_init(self._h, nranks, rank, buf, N.COMM_ID_BYTES if uid else 0))

    def comm_p2p_active(self) -> bool:
        v = C.c_int()
        self._ck(self._lib.se_comm_p2p_active(self._h, C.byref(v)))
        return bool(v.value)

    def comm_clear_error(self):
        self._ck(self._lib.se_comm_clear_error(self._h))

    def comm_destroy(self):
        self._ck(self._lib.se_comm_destroy(self._h))

    def comm_info(self):
        a, b = C.c_int(), C.c_int()
        self._ck(self._lib.se_comm_info(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def allreduce_host(self, values) -> np.ndarray:
        v = np.ascontiguousarray(values, dtype=np.float64).copy()
        self._ck(self._lib.se_comm_allreduce_host(self._h, N.dptr(v), v.size))
        return v

    # ---- slots
    def alloc(self, slot: int, rows: int, cols: int | None = None):
        if cols is None:
            self._ck(self._lib.se_slot_alloc(self._h, slot, rows))
        else:
            self._ck(self._lib.se_slot_alloc2d(self._h, slot, rows, cols))

    def free(self, slot: int):
        self._ck(self._lib.se_slot_free(self._h, slot))

    def layout(self, slot: int):
        r, c, ld = C.c_int64(), C.c_int64(), C.c_int64()
        self._ck(self._lib.se_slot_layout(self._h, slot, C.byref(r), C.byref(c), C.byref(ld)))
        return r.value, c.value, ld.value

    def device_ptr(self, slot: int) -> int:
        p, n = C.c_void_p(), C.c_int64()
        self._ck(self._lib.se_slot_info(self._h, slot, C.byref(p), C.byref(n)))
        return p.value or 0

    def upload(self, slot: int, host, offset: int = 0):
        if isinstance(host, np.ndarray) and host.dtype == np.float64:
            a = np.ascontiguousarray(host)
            self._ck(self._lib.se_upload_f64(self._h, slot, N.dptr(a.reshape(-1)), a.size, offset))
            return
        a = N.as_f32(host)
        self._ck(self._lib.se_upload(self._h, slot, N.fptr(a.reshape(-1)), a.size, offset))

    def upload_rowmajor(self, slot: int, features, row_offset: int = 0):
        """Row-major [n_rows, d] partition -> rows [row_offset, ...) of the column-major [d][n] slot."""
        a = N.as_f32(features)
        assert a.ndim == 2
        self._ck(self._lib.se_upload_rowmajor(self._h, slot, N.fptr(a.reshape(-1)), a.shape[0], a.shape[1], row_offset))

    def download(self, slot: int, count: int | None = None, offset: int = 0, scale: float | None = None,
                 out: np.ndarray | None = None) -> np.ndarray:
        r, c, _ = self.layout(slot)
        shape = (r, c) if (count is None and r > 1) else None
        if count is None:
            count = r * c - offset
        if out is None:
            out = np.empty(count, dtype=np.float32)
        if scale is None:
            self._ck(self._lib.se_download(self._h, slot, N.fptr(out.reshape(-1)), count, offset))
        else:
            self._ck(self._lib.se_download_scaled(self._h, slot, float(scale), N.fptr(out.reshape(-1)),
                                                  count, offset))
        return out.reshape(shape) if (shape is not None and offset == 0) else out

    def fill(self, slot: int, value: float, count: int | None = None, offset: int = 0):
        if count is None:
            r, c, _ = self.layout(slot)
            count = r * c - offset
        self._ck(self._lib.se_fill(self._h, slot, float(value), count, offset))

    def fill_synthetic(self, slot: int, kind: str, seed: int, a: float, b: float, count: int | None = None,
                       offset: int = 0):
        k = {"uniform": 0, "normal": 1, "randint": 2, "bernoulli": 3}[kind]
        if count is None:
            r, c, _ = self.layout(slot)
            count = r * c - offset
        self._ck(self._lib.se_fill_synthetic(self._h, slot, k, int(seed), float(a), float(b), count, offset))

    def copy_slot(self, dst: int, src: int):
        self._ck(self._lib.se_copy_slot(self._h, dst, src))

    def slot_sum(self, slot: int, count: int | None = None) -> float:
        if count is None:
            _, count, _ = self.layout(slot)
        v = C.c_double()
        self._ck(self._lib.se_slot_sum(self._h, slot, count, C.byref(v)))
        return v.value

    def quantile(self, slot: int, q: float, count: int | None = None) -> float:
        """Exact q-quantile (ceil(q·N)-th smallest, global) of a [n] slot."""
        if count is None:
            _, count, _ = self.layout(slot)
        v = C.c_double()
        self._ck(self._lib.se_quantile(self._h, 0, slot, count, float(q), C.byref(v)))
        return v.value

    def gbm_abs_residual_quantile(self, q: float) -> float:
        """Exact q-quantile of |y − F| over the train rows (huber δ)."""
        v = C.c_double()
        self._ck(self._lib.se_quantile(self._h, 1, 0, 0, float(q), C.byref(v)))
        return v.value

    # ---- GBM
    def gbm_configure(self, n_train: int, n_valid: int, dim: int, loss, param: float = 0.0,
                      has_weights: bool = False):
        lid = N.LOSS[loss] if isinstance(loss, str) else int(loss)
        self._ck(self._lib.se_gbm_configure(self._h, n_train, n_valid, dim, lid, float(param),
                                            int(has_weights)))
        self.dim = dim

    def gbm_set_loss_param(self, param: float):
        self._ck(self._lib.se_gbm_set_loss_param(self._h, float(param)))

    def gbm_set_bag(self, counts):
        """Upload bag multiplicities (row sub-sampling); None disables."""
        if counts is None:
            self._ck(self._lib.se_gbm_set_bag(self._h, 0))
            return
        self._ck(self._lib.se_gbm_set_bag(self._h, 1))
        self.upload(N.SLOT_BAG, np.ascontiguousarray(counts, dtype=np.float32))

    def gbm_pseudo_residuals(self, newton: bool = False):
        sh = np.zeros(max(self.dim, 1))
        self._ck(self._lib.se_gbm_pseudo_residuals(self._h, int(newton), N.dptr(sh)))
        return sh if newton else None

    def gbm_linesearch_eval(self, alpha, want_grad: bool = True):
        a = np.ascontiguousarray(np.atleast_1d(alpha), dtype=np.float64)
        loss = C.c_double()
        g = np.zeros(a.size)
        self._ck(self._lib.se_gbm_linesearch_eval(self._h, N.dptr(a), C.byref(loss),
                                                  N.dptr(g) if want_grad else None))
        return loss.value, g

    def gbm_linesearch_stats(self) -> np.ndarray:
        s = np.zeros(4)
        self._ck(self._lib.se_gbm_linesearch_stats(self._h, N.dptr(s)))
        return s

    def gbm_update(self, step, residual: bool = False, newton: bool = False, loss: bool = True):
        s = np.ascontiguousarray(np.atleast_1d(step), dtype=np.float64)
        flags = (N.UPD_RESIDUAL if residual else 0) | (N.UPD_NEWTON if newton else 0) | (N.UPD_LOSS if loss else 0)
        ls = C.c_double(float("nan"))
        sh = np.zeros(max(self.dim, 1))
        self._ck(self._lib.se_gbm_update(self._h, N.dptr(s), flags, C.byref(ls), N.dptr(sh)))
        return ls.value, (sh if newton else None)

    def gbm_mean_loss(self, validation: bool = False) -> float:
        v = C.c_double()
        self._ck(self._lib.se_gbm_mean_loss(self._h, int(validation), C.byref(v)))
        return v.value

    def gbm_update_validation(self, step) -> float:
        s = np.ascontiguousarray(np.atleast_1d(step), dtype=np.float64)
        v = C.c_double()
        self._ck(self._lib.se_gbm_update_validation(self._h, N.dptr(s), C.byref(v)))
        return v.value

    def gbm_linesearch_brent(self, lo=0.0, hi=100.0, start=1.0, rel=1e-6, abs_tol=1e-6, max_eval=100):
        a, l, ne = C.c_double(), C.c_double(), C.c_int()
        self._ck(self._lib.se_gbm_linesearch_brent(self._h, lo, hi, start, rel, abs_tol, max_eval,
                                                   C.byref(a), C.byref(l), C.byref(ne)))
        return a.value, l.value, ne.value

    def gbm_round(self, learning_rate: float, optimized: bool = True, tol: float = 1e-6, max_iter: int = 100,
                  residual: bool = True, newton: bool = False):
        """Line search + update in one native call (dim 1). Returns (alpha, train_loss_sum, n_eval)."""
        flags = (N.UPD_RESIDUAL if residual else 0) | (N.UPD_NEWTON if newton else 0) | N.UPD_LOSS
        a, l, ne = C.c_double(), C.c_double(), C.c_int()
        self._ck(self._lib.se_gbm_round(self._h, float(learning_rate), int(optimized), float(tol), int(max_iter), flags,
                                        C.byref(a), C.byref(l), C.byref(ne)))
        return a.value, l.value, ne.value

    def gbm_linesearch_eval2(self, alpha: float):
        l, d1, d2 = C.c_double(), C.c_double(), C.c_double()
        self._ck(self._lib.se_gbm_linesearch_eval2(self._h, float(alpha), C.byref(l), C.byref(d1), C.byref(d2)))
        return l.value, d1.value, d2.value

    def gbm_linesearch_newton(self, lo=0.0, hi=100.0, start=1.0, rel=1e-6, abs_tol=1e-6, max_eval=100):
        a, l, ne = C.c_double(), C.c_double(), C.c_int()
        self._ck(self._lib.se_gbm_linesearch_newton(self._h, lo, hi, start, rel, abs_tol, max_eval,
                                                    C.byref(a), C.byref(l), C.byref(ne)))
        return a.value, l.value, ne.value

    def gbm_round_squared_async(self, learning_rate: float = 1.0):
        self._ck(self._lib.se_gbm_round_squared_async(self._h, float(learning_rate)))

    def gbm_round_result(self):
        a, l = C.c_double(), C.c_double()
        self._ck(self._lib.se_gbm_round_result(self._h, C.byref(a), C.byref(l)))
        return a.value, l.value

    # ---- Boosting
    def boost_configure(self, n: int, num_classes: int, real: bool):
        self._ck(self._lib.se_boost_configure(self._h, n, num_classes, int(real)))

    def boost_real_update(self, sum_w: float):
        e, s = C.c_double(), C.c_double()
        self._ck(self._lib.se_boost_real_update(self._h, float(sum_w), C.byref(e), C.byref(s)))
        return e.value, s.value

    def boost_discrete_error(self, sum_w: float) -> float:
        e = C.c_double()
        self._ck(self._lib.se_boost_discrete_error(self._h, float(sum_w), C.byref(e)))
        return e.value

    def boost_discrete_update(self, sum_w: float, beta: float) -> float:
        s = C.c_double()
        self._ck(self._lib.se_boost_discrete_update(self._h, float(sum_w), float(beta), C.byref(s)))
        return s.value

    # ---- BoostingRegressor (AdaBoost.R2)
    def boostreg_configure(self, n: int):
        self._ck(self._lib.se_boostreg_configure(self._h, n))

    def boostreg_max_error(self) -> float:
        v = C.c_double()
        self._ck(self._lib.se_boostreg_max_error(self._h, C.byref(v)))
        return v.value

    def boostreg_error(self, sum_w: float, loss_type: str, max_error: float) -> float:
        v = C.c_double()
        self._ck(self._lib.se_boostreg_error(self._h, float(sum_w), N.R2_LOSS[loss_type], float(max_error), C.byref(v)))
        return v.value

    def boostreg_update(self, sum_w: float, loss_type: str, max_error: float, beta: float) -> float:
        v = C.c_double()
        self._ck(self._lib.se_boostreg_update(self._h, float(sum_w), N.R2_LOSS[loss_type], float(max_error),
                                              float(beta), C.byref(v)))
        return v.value

    # ---- aggregation
    def agg_configure(self, kind: int, num_models: int, num_classes: int, dim: int, loss, n: int):
        lid = N.LOSS[loss] if isinstance(loss, str) else int(loss)
        self._ck(self._lib.se_agg_configure(self._h, kind, num_models, num_classes, dim, lid, n))

    def agg_run(self, weights=None, init=None):
        w = None if weights is None else np.ascontiguousarray(weights, dtype=np.float64).reshape(-1)
        i = None if init is None else np.ascontiguousarray(np.atleast_1d(init), dtype=np.float64)
        self._ck(self._lib.se_agg_run(self._h, None if w is None else N.dptr(w),
                                      None if i is None else N.dptr(i)))

    # ---- on-device base models
    def tree_predict(self, tree: dict, out_slot: int, out_row: int = 0, validation: bool = False,
                     subspace=None):
        f = np.ascontiguousarray(tree["feature"], dtype=np.int32)
        t = np.ascontiguousarray(tree["threshold"], dtype=np.float32)
        l = np.ascontiguousarray(tree["left"], dtype=np.int32)
        r = np.ascontiguousarray(tree["right"], dtype=np.int32)
        v = np.ascontiguousarray(tree["value"], dtype=np.float32)
        sub = None if subspace is None else np.ascontiguousarray(subspace, dtype=np.int32)
        self._ck(self._lib.se_tree_predict(self._h, int(validation), f.size, N.iptr(f), N.fptr(t), N.iptr(l),
                                           N.iptr(r), N.fptr(v), None if sub is None else N.iptr(sub),
                                           0 if sub is None else sub.size, out_slot, out_row))

    def tree_predict_multi(self, tree: dict, out_slot: int, validation: bool = False, subspace=None):
        """Classification tree: tree["values"] is [n_nodes, K] (leaf class probabilities) -> K rows of out_slot."""
        f = np.ascontiguousarray(tree["feature"], dtype=np.int32)
        t = np.ascontiguousarray(tree["threshold"], dtype=np.float32)
        l = np.ascontiguousarray(tree["left"], dtype=np.int32)
        r = np.ascontiguousarray(tree["right"], dtype=np.int32)
        v = np.ascontiguousarray(tree["values"], dtype=np.float32)
        sub = None if subspace is None else np.ascontiguousarray(subspace, dtype=np.int32)
        self._ck(self._lib.se_tree_predict_multi(self._h, int(validation), f.size, N.iptr(f), N.fptr(t), N.iptr(l),
                                                 N.iptr(r), N.fptr(v.reshape(-1)), v.shape[1],
                                                 None if sub is None else N.iptr(sub), 0 if sub is None else sub.size,
                                                 out_slot))

    def forest_predict(self, trees, out_slot: int, weights=None, init: float = 0.0, out_row: int = 0,
                       validation: bool = False, subspaces=None):
        """out = init + sum_t weights[t] * tree_t(x) for a list of regression trees (dicts as in tree_predict) in one
        pass over the resident feature matrix (se_forest_predict: GBMRegressionModel.predict,
        regression/GBMRegressor.scala:531-539).  `subspaces[t]` maps tree t's feature indices to columns of X."""
        offs, f, t, l, r, v = _flatten_trees(trees, subspaces, "value")
        w = None if weights is None else np.ascontiguousarray(weights, dtype=np.float64)
        if w is not None and w.size != len(trees):
            raise ValueError("one weight per tree")
        self._ck(self._lib.se_forest_predict(self._h, int(validation), len(trees), N.iptr(offs), N.iptr(f), N.fptr(t),
                                             N.iptr(l), N.iptr(r), N.fptr(v), None if w is None else N.dptr(w),
                                             float(init), out_slot, out_row))

    def forest_classify(self, trees, kind: int, num_classes: int, dim: int = 1, loss=0, weights=None, init=None,
                        validation: bool = False, subspaces=None):
        """RAW, PROB and LABEL of a classifier ensemble of trees in one pass over the resident feature matrix
        (se_forest_classify): what agg_configure + agg_run would give from the members' outputs, without them.
        Leaves: tree["values"] ([n_nodes, K] class probabilities) for AGG_BAGGING_SOFT / AGG_BOOSTING_REAL,
        tree["value"] (regression value or predicted label) for the others.  GBM: tree t = models(t // dim)(t % dim),
        weights [M][dim], init [dim]; SAMME: weights [M].  `subspaces[t]` maps tree t's features to columns of X."""
        vector = kind in (N.AGG_BAGGING_SOFT, N.AGG_BOOSTING_REAL)
        offs, f, t, l, r, v = _flatten_trees(trees, subspaces, "values" if vector else "value")
        width = v.size // max(int(offs[-1]), 1)
        lid = N.LOSS[loss] if isinstance(loss, str) else int(loss)
        w = None if weights is None else np.ascontiguousarray(weights, dtype=np.float64).reshape(-1)
        if w is not None and w.size != len(trees):
            raise ValueError("one weight per tree")
        i = None if init is None else np.ascontiguousarray(np.atleast_1d(init), dtype=np.float64)
        self._ck(self._lib.se_forest_classify(self._h, int(validation), int(kind), int(num_classes), int(dim), lid,
                                              len(trees), N.iptr(offs), N.iptr(f), N.fptr(t), N.iptr(l), N.iptr(r),
                                              N.fptr(v), int(width), None if w is None else N.dptr(w),
                                              None if i is None else N.dptr(i)))

    def forest_weighted_median(self, trees, out_slot: int, weights, out_row: int = 0, validation: bool = False):
        """out = Utils.weightedMedian([tree_t(x)]_t, weights) for a list of at most 64 regression trees (dicts as in
        tree_predict, features = columns of X, model order) in one pass over the resident feature matrix
        (se_forest_weighted_median: BoostingRegressionModel.predict, regression/BoostingRegressor.scala:333-337).  The
        same bits as tree_predict of every member + agg_run(AGG_BOOSTING_REG_MEDIAN); NativeError SE_ERR_STATE when
        the forest is beyond the kernel (more than 64 trees, more than one chunk, a column with > 255 thresholds)."""
        offs, f, t, l, r, v = _flatten_trees(trees, None, "value")
        w = None if weights is None else np.ascontiguousarray(weights, dtype=np.float64).reshape(-1)
        if w is not None and w.size != len(trees):
            raise ValueError("one weight per tree")
        self._ck(self._lib.se_forest_weighted_median(self._h, int(validation), len(trees), N.iptr(offs), N.iptr(f),
                                                     N.fptr(t), N.iptr(l), N.iptr(r), N.fptr(v),
                                                     None if w is None else N.dptr(w), out_slot, out_row))

    def linear_predict(self, coef, intercept: float, out_slot: int, out_row: int = 0,
                       validation: bool = False, subspace=None):
        c = np.ascontiguousarray(coef, dtype=np.float32)
        sub = None if subspace is None else np.ascontiguousarray(subspace, dtype=np.int32)
        self._ck(self._lib.se_linear_predict(self._h, int(validation), c.size, N.fptr(c), float(intercept),
                                             None if sub is None else N.iptr(sub), out_slot, out_row))
