"""Row-sharded GBM fit over several GPUs from ONE host process: N contexts (one per GPU), rows split into contiguous
blocks (ensemble.row_partition), every C-ABI call issued on all contexts at once (one host thread per GPU; ctypes
releases the GIL during the call).  The contexts are joined by se_comm_init, so the scalars each call returns are
already GLOBAL — summed across GPUs inside the reducing kernels over NVLink peer memory (or by NCCL as the fallback)
exactly where the reference calls treeAggregate/treeReduce — and rank 0's values are handed back.

ShardedContext exposes the subset of Context that gbm_engine.GBMEngine and the estimator mirrors use for a fit, with
the same signatures: host arrays are passed / returned WHOLE (the [dim][n_total] layout of the single-GPU path) and
are split / concatenated here, so the estimator code is unchanged (Param `devices`, regression.GBMRegressor).
"""
from __future__ import annotations

import concurrent.futures as cf

import numpy as np

from . import _native as N
from .context import Context
from .ensemble import row_partition

_TRAIN_SLOTS = {N.SLOT_Y, N.SLOT_W, N.SLOT_F, N.SLOT_H, N.SLOT_R, N.SLOT_WOUT, N.SLOT_BAG, N.SLOT_X}
_VALID_SLOTS = {N.SLOT_VY, N.SLOT_VF, N.SLOT_VH, N.SLOT_VX}
_OUT_SLOTS = {N.SLOT_RAW, N.SLOT_PROB, N.SLOT_LABEL}


class ShardedContext:
    def __init__(self, devices, context_factory=Context, join: bool = True):
        devices = [int(d) for d in devices]
        if len(devices) < 2:
            raise ValueError("ShardedContext needs at least two devices")
        self.devices = devices
        self.world = len(devices)
        self.ctxs = [context_factory(d) for d in devices]
        self._pool = cf.ThreadPoolExecutor(max_workers=self.world)
        self.n = self.nv = self._n_out = 0
        self.dim = 1
        if join:
            uid = Context.comm_unique_id()
            self._all(lambda r, c: c.comm_init(self.world, r, uid))  # collective: all ranks at once

    # ---- plumbing
    def _all(self, fn):
        futs = [self._pool.submit(fn, r, c) for r, c in enumerate(self.ctxs)]
        return [f.result() for f in futs]

    def _total(self, slot: int) -> int:
        if slot in _TRAIN_SLOTS:
            return self.n
        if slot in _VALID_SLOTS:
            return self.nv
        if slot in _OUT_SLOTS:  # the outputs of forest_classify: one column per row of the feature slot it read
            return self._n_out
        raise ValueError(f"slot {slot} is not row-sharded by ShardedContext")

    def close(self):
        if not self.ctxs:
            return
        # every rank leaves the communicator at the same time, each from its own thread (NCCL tears a communicator
        # down collectively), and only then are the contexts (and the mailboxes their peers map) released
        try:
            self._all(lambda r, c: c.sync())
            self._all(lambda r, c: c.comm_destroy())
        finally:
            for c in self.ctxs:
                c.close()
            self.ctxs = []
            self._pool.shutdown(wait=True)

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def sync(self):
        self._all(lambda r, c: c.sync())

    def comm_p2p_active(self) -> bool:
        return all(self._all(lambda r, c: c.comm_p2p_active()))

    def set_option(self, key, value):
        self._all(lambda r, c: c.set_option(key, value))

    def get_option(self, key):
        return self.ctxs[0].get_option(key)

    # ---- slots: host arrays are whole, [k][n_total]
    def gbm_configure(self, n_train, n_valid, dim, loss, param=0.0, has_weights=False):
        self.n, self.nv, self.dim = int(n_train), int(n_valid), int(dim)

        def f(r, c):
            s0, s1 = row_partition(self.n, self.world, r)
            v0, v1 = row_partition(self.nv, self.world, r)
            c.gbm_configure(s1 - s0, v1 - v0, dim, loss, param, has_weights)
        self._all(f)

    def alloc(self, slot, rows, cols=None):
        if cols is None:
            raise ValueError("sharded alloc takes (rows, total columns)")
        tot = self._total(slot)
        assert cols == tot, (cols, tot)
        self._all(lambda r, c: c.alloc(slot, rows, (lambda s: s[1] - s[0])(row_partition(tot, self.world, r))))

    def upload(self, slot, host, offset: int = 0):
        tot = self._total(slot)
        a = np.asarray(host)
        if tot == 0:
            return
        assert a.size % tot == 0 and offset % tot == 0, (a.size, offset, tot)
        a2 = a.reshape(a.size // tot, tot)
        row0 = offset // tot

        def f(r, c):
            s0, s1 = row_partition(tot, self.world, r)
            if s1 > s0:
                c.upload(slot, np.ascontiguousarray(a2[:, s0:s1]), offset=row0 * (s1 - s0))
        self._all(f)

    def upload_rowmajor(self, slot, features, row_offset: int = 0):
        tot = self._total(slot)
        X = np.asarray(features)
        assert row_offset == 0 and X.shape[0] == tot

        def f(r, c):
            s0, s1 = row_partition(tot, self.world, r)
            if s1 > s0:
                c.upload_rowmajor(slot, X[s0:s1])
        self._all(f)

    def fill(self, slot, value, count=None, offset: int = 0):
        tot = self._total(slot)
        if count is None:
            self._all(lambda r, c: c.fill(slot, value))
            return
        assert count == tot and offset % max(tot, 1) == 0
        row0 = offset // max(tot, 1)

        def f(r, c):
            s0, s1 = row_partition(tot, self.world, r)
            if s1 > s0:
                c.fill(slot, value, s1 - s0, row0 * (s1 - s0))
        self._all(f)

    def download(self, slot, count=None, offset: int = 0, scale=None, out=None):
        assert count is None and offset == 0, "sharded download returns the whole slot"
        tot = self._total(slot)

        def f(r, c):
            s0, s1 = row_partition(tot, self.world, r)
            if s1 == s0:
                return None
            rows, cols, _ = c.layout(slot)
            return np.asarray(c.download(slot, scale=scale)).reshape(rows, cols)
        parts = [p for p in self._all(f) if p is not None]
        whole = np.concatenate(parts, axis=1) if parts else np.zeros((self.dim, 0), dtype=np.float32)
        res = whole if whole.shape[0] > 1 else whole.reshape(-1)
        if out is not None:
            out.reshape(-1)[:] = res.reshape(-1)
            return out
        return res

    # ---- GBM entry points: scalars are global on every rank; rank 0's are returned
    def gbm_set_loss_param(self, p):
        self._all(lambda r, c: c.gbm_set_loss_param(p))

    def gbm_set_bag(self, counts):
        if counts is None:
            self._all(lambda r, c: c.gbm_set_bag(None))
            return
        counts = np.asarray(counts, dtype=np.float32)

        def f(r, c):
            s0, s1 = row_partition(self.n, self.world, r)
            c.gbm_set_bag(counts[s0:s1])
        self._all(f)

    def gbm_pseudo_residuals(self, newton=False):
        return self._all(lambda r, c: c.gbm_pseudo_residuals(newton))[0]

    def gbm_linesearch_eval(self, alpha):
        return self._all(lambda r, c: c.gbm_linesearch_eval(alpha))[0]

    def gbm_linesearch_stats(self):
        return self._all(lambda r, c: c.gbm_linesearch_stats())[0]

    def gbm_update(self, step, residual=False, newton=False, loss=True):
        return self._all(lambda r, c: c.gbm_update(step, residual=residual, newton=newton, loss=loss))[0]

    def gbm_mean_loss(self, validation=False):
        return self._all(lambda r, c: c.gbm_mean_loss(validation))[0]

    def gbm_update_validation(self, step):
        return self._all(lambda r, c: c.gbm_update_validation(step))[0]

    def gbm_linesearch_brent(self, *a, **k):
        res = self._all(lambda r, c: c.gbm_linesearch_brent(*a, **k))
        assert all(x == res[0] for x in res), "ranks disagree on the line search (sums must be bit-identical)"
        return res[0]

    def gbm_linesearch_newton(self, *a, **k):
        return self._all(lambda r, c: c.gbm_linesearch_newton(*a, **k))[0]

    def gbm_round(self, *a, **k):
        res = self._all(lambda r, c: c.gbm_round(*a, **k))
        assert all(x[0] == res[0][0] for x in res), "ranks disagree on alpha"
        return res[0]

    def gbm_abs_residual_quantile(self, q):
        return self._all(lambda r, c: c.gbm_abs_residual_quantile(q))[0]

    def tree_predict(self, tree, out_slot, out_row=0, validation=False, subspace=None):
        self._all(lambda r, c: c.tree_predict(tree, out_slot, out_row, validation=validation, subspace=subspace))

    def tree_predict_multi(self, tree, out_slot, validation=False, subspace=None):
        self._all(lambda r, c: c.tree_predict_multi(tree, out_slot, validation=validation, subspace=subspace))

    def forest_predict(self, trees, out_slot, weights=None, init=0.0, out_row=0, validation=False, subspaces=None):
        self._all(lambda r, c: c.forest_predict(trees, out_slot, weights=weights, init=init, out_row=out_row,
                                                validation=validation, subspaces=subspaces))

    def forest_classify(self, trees, kind, num_classes, dim=1, loss=0, weights=None, init=None, validation=False,
                        subspaces=None):
        """Every shard classifies its own rows (no reduction): RAW / PROB / LABEL reassemble through `download`."""
        self._n_out = self.nv if validation else self.n
        self._all(lambda r, c: c.forest_classify(trees, kind, num_classes, dim=dim, loss=loss, weights=weights, init=init,
                                                 validation=validation, subspaces=subspaces))

    def forest_weighted_median(self, trees, out_slot, weights, out_row=0, validation=False):
        """Every shard takes the weighted median over its own rows (no reduction)."""
        self._all(lambda r, c: c.forest_weighted_median(trees, out_slot, weights, out_row=out_row, validation=validation))

    def linear_predict(self, coef, intercept, out_slot, out_row=0, validation=False, subspace=None):
        self._all(lambda r, c: c.linear_predict(coef, intercept, out_slot, out_row, validation=validation, subspace=subspace))


def make_context(device: int = 0, devices=None):
    """One Context, or a ShardedContext when `devices` lists two or more GPUs (Param `devices` of the estimators)."""
    devices = list(devices or [])
    if len(devices) >= 2:
        return ShardedContext(devices)
    return Context(devices[0] if devices else device)
