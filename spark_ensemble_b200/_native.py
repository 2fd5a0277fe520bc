"""ctypes binding of libse_b200.so — the C ABI declared in include/se_abi.h.

This is the same boundary the Scala/JNI shim binds (jni/se_jni.cpp).  There is NO fallback: if the
CUDA library is missing or no device works, importing/using the hot path raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libse_b200.so")

SE_OK, SE_ERR_ARG, SE_ERR_CUDA, SE_ERR_NCCL, SE_ERR_STATE, SE_ERR_OPT = 0, -1, -2, -3, -4, -5
COMM_ID_BYTES = 128

# enum se_loss
LOSS = {"squared": 0, "absolute": 1, "huber": 2, "quantile": 3, "logcosh": 4, "scaledlogcosh": 5,
        "bernoulli": 6, "exponential": 7, "logloss": 8}
# enum se_slot
(SLOT_Y, SLOT_W, SLOT_F, SLOT_H, SLOT_R, SLOT_WOUT, SLOT_VY, SLOT_VF, SLOT_VH, SLOT_BW, SLOT_PROBA,
 SLOT_PRED, SLOT_P, SLOT_RAW, SLOT_PROB, SLOT_LABEL, SLOT_X, SLOT_VX, SLOT_BAG) = range(19)
NUM_SLOTS = 19
# se_gbm_update flags
UPD_RESIDUAL, UPD_NEWTON, UPD_LOSS = 1, 2, 4
# enum se_agg_kind
(AGG_GBM_REGRESSOR, AGG_BAGGING_REGRESSOR, AGG_GBM_CLASSIFIER, AGG_BAGGING_SOFT, AGG_BAGGING_HARD,
 AGG_BOOSTING_REAL, AGG_BOOSTING_DISCRETE, AGG_BOOSTING_REG_MEDIAN, AGG_BOOSTING_REG_MEAN) = range(9)
R2_LOSS = {"exponential": 0, "linear": 1, "squared": 2}

# enum se_kernel_family
KERNEL_FAMILIES = ["sq_stats", "eval", "update", "resid", "mean_loss", "boost_real", "boost_err",
                   "boost_upd", "agg", "tree", "linear", "other"]

FN1 = C.CFUNCTYPE(C.c_double, C.c_double, C.c_void_p)

_i32, _i64, _u64, _d, _f = C.c_int, C.c_int64, C.c_uint64, C.c_double, C.c_float
_vp = C.c_void_p
_dp, _fp, _ip = C.POINTER(C.c_double), C.POINTER(C.c_float), C.POINTER(C.c_int32)

# name -> argtypes (restype is int unless listed in _RESTYPES); mirrors include/se_abi.h one-to-one
PROTOTYPES = {
    "se_abi_version": [],
    "se_last_error": [_vp],
    "se_device_count": [C.POINTER(_i32)],
    "se_ctx_create": [_i32, C.POINTER(_vp)],
    "se_ctx_destroy": [_vp],
    "se_ctx_sync": [_vp],
    "se_ctx_device": [_vp, C.POINTER(_i32)],
    "se_ctx_launch_count": [_vp, C.POINTER(_i64)],
    "se_ctx_last_ms": [_vp, _dp],
    "se_ctx_set_timing": [_vp, _i32],
    "se_ctx_timer_start": [_vp],
    "se_ctx_timer_stop": [_vp, _dp],
    "se_ctx_kernel_timing": [_vp, _i32],
    "se_ctx_kernel_time": [_vp, _i32, _dp, C.POINTER(_i64)],
    "se_ctx_kernel_time_reset": [_vp],
    "se_ctx_set_option": [_vp, C.c_char_p, _d],
    "se_ctx_get_option": [_vp, C.c_char_p, _dp],
    "se_host_alloc": [_i64, C.POINTER(_vp)],
    "se_host_free": [_vp],
    "se_comm_unique_id": [_vp, _i32],
    "se_comm_init": [_vp, _i32, _i32, _vp, _i32],
    "se_comm_p2p_active": [_vp, C.POINTER(_i32)],
    "se_comm_clear_error": [_vp],
    "se_comm_destroy": [_vp],
    "se_comm_info": [_vp, C.POINTER(_i32), C.POINTER(_i32)],
    "se_comm_allreduce_host": [_vp, _dp, _i32],
    "se_slot_alloc": [_vp, _i32, _i64],
    "se_slot_alloc2d": [_vp, _i32, _i64, _i64],
    "se_slot_layout": [_vp, _i32, C.POINTER(_i64), C.POINTER(_i64), C.POINTER(_i64)],
    "se_slot_free": [_vp, _i32],
    "se_slot_info": [_vp, _i32, C.POINTER(_vp), C.POINTER(_i64)],
    "se_upload": [_vp, _i32, _fp, _i64, _i64],
    "se_upload_f64": [_vp, _i32, _dp, _i64, _i64],
    "se_upload_rowmajor": [_vp, _i32, _fp, _i64, _i32, _i64],
    "se_download": [_vp, _i32, _fp, _i64, _i64],
    "se_download_scaled": [_vp, _i32, _d, _fp, _i64, _i64],
    "se_fill": [_vp, _i32, _f, _i64, _i64],
    "se_copy_slot": [_vp, _i32, _i32],
    "se_fill_synthetic": [_vp, _i32, _i32, _u64, _d, _d, _i64, _i64],
    "se_slot_sum": [_vp, _i32, _i64, _dp],
    "se_quantile": [_vp, _i32, _i32, _i64, _d, _dp],
    "se_gbm_configure": [_vp, _i64, _i64, _i32, _i32, _d, _i32],
    "se_gbm_set_loss_param": [_vp, _d],
    "se_gbm_set_bag": [_vp, _i32],
    "se_gbm_pseudo_residuals": [_vp, _i32, _dp],
    "se_gbm_linesearch_eval": [_vp, _dp, _dp, _dp],
    "se_gbm_linesearch_stats": [_vp, _dp],
    "se_gbm_update": [_vp, _dp, _i32, _dp, _dp],
    "se_gbm_mean_loss": [_vp, _i32, _dp],
    "se_gbm_update_validation": [_vp, _dp, _dp],
    "se_gbm_linesearch_brent": [_vp, _d, _d, _d, _d, _d, _i32, _dp, _dp, C.POINTER(_i32)],
    "se_gbm_round": [_vp, _d, _i32, _d, _i32, _i32, _dp, _dp, C.POINTER(_i32)],
    "se_gbm_linesearch_eval2": [_vp, _d, _dp, _dp, _dp],
    "se_gbm_linesearch_newton": [_vp, _d, _d, _d, _d, _d, _i32, _dp, _dp, C.POINTER(_i32)],
    "se_gbm_round_squared_async": [_vp, _d],
    "se_gbm_round_result": [_vp, _dp, _dp],
    "se_brent_minimize": [FN1, _vp, _d, _d, _d, _d, _d, _i32, _dp, _dp, C.POINTER(_i32)],
    "se_boost_configure": [_vp, _i64, _i32, _i32],
    "se_boost_real_update": [_vp, _d, _dp, _dp],
    "se_boost_discrete_error": [_vp, _d, _dp],
    "se_boost_discrete_update": [_vp, _d, _d, _dp],
    "se_boostreg_configure": [_vp, _i64],
    "se_boostreg_max_error": [_vp, _dp],
    "se_boostreg_error": [_vp, _d, _i32, _d, _dp],
    "se_boostreg_update": [_vp, _d, _i32, _d, _d, _dp],
    "se_agg_configure": [_vp, _i32, _i32, _i32, _i32, _i32, _i64],
    "se_agg_run": [_vp, _dp, _dp],
    "se_spark_bernoulli_sample": [_i64, _d, _i64, _i32, _fp],
    "se_tree_predict": [_vp, _i32, _i32, _ip, _fp, _ip, _ip, _fp, _ip, _i32, _i32, _i32],
    "se_tree_predict_multi": [_vp, _i32, _i32, _ip, _fp, _ip, _ip, _fp, _i32, _ip, _i32, _i32],
    "se_forest_predict": [_vp, _i32, _i32, _ip, _ip, _fp, _ip, _ip, _fp, _dp, _d, _i32, _i32],
    "se_forest_classify": [_vp, _i32, _i32, _i32, _i32, _i32, _i32, _ip, _ip, _fp, _ip, _ip, _fp, _i32, _dp, _dp],
    "se_forest_weighted_median": [_vp, _i32, _i32, _ip, _ip, _fp, _ip, _ip, _fp, _dp, _i32, _i32],
    "se_linear_predict": [_vp, _i32, _i32, _fp, _f, _ip, _i32, _i32],
}
_RESTYPES = {"se_last_error": C.c_char_p}


class NativeError(RuntimeError):
    """Non-zero status from libse_b200 (maps to RuntimeException / IllegalArgumentException in Scala)."""

    def __init__(self, code: int, message: str):
        super().__init__(f"libse_b200 error {code}: {message}")
        self.code = code
        self.message = message


class ConvergenceError(NativeError):
    """SE_ERR_OPT: optimiser exceeded MaxEval (TooManyEvaluationsException in the reference)."""


_lib = None


def load():
    """Load the CUDA library. Raises if it has not been built — there is no CPU fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -m spark_ensemble_b200.build` "
            "(nvcc, sm_100a). The boosting hot path has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, argtypes in PROTOTYPES.items():
        fn = getattr(lib, name)  # AttributeError here == ABI mismatch: fail loudly
        fn.argtypes = argtypes
        fn.restype = _RESTYPES.get(name, C.c_int)
    _lib = lib
    return lib


def last_error(handle=None) -> str:
    msg = load().se_last_error(handle)
    return msg.decode("utf-8", "replace") if msg else ""


def check(rc: int, handle=None) -> None:
    if rc == SE_OK:
        return
    msg = last_error(handle)
    if rc == SE_ERR_OPT:
        raise ConvergenceError(rc, msg)
    if rc == SE_ERR_ARG:
        raise ValueError(f"libse_b200: {msg}")
    raise NativeError(rc, msg)


def device_count() -> int:
    n = C.c_int(0)
    rc = load().se_device_count(C.byref(n))
    return n.value if rc == SE_OK else 0


def as_f32(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.float32)


def fptr(a: np.ndarray):
    assert a.dtype == np.float32 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(_fp)


def dptr(a: np.ndarray):
    assert a.dtype == np.float64 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(_dp)


def iptr(a: np.ndarray):
    assert a.dtype == np.int32 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(_ip)
