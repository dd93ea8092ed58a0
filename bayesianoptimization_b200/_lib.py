"""ctypes binding of include/b200bo.h.  Fails loudly when the CUDA library is missing - there is
no CPU fallback behind this module."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libb200bo.so")

OK, ERR_CUDA, ERR_ARG, ERR_NOT_PD, ERR_UNSUPPORTED, ERR_STATE = 0, -1, -2, -3, -4, -5
KERNEL_MATERN, KERNEL_RBF = 0, 1
NU_05, NU_15, NU_25, NU_INF = 0, 1, 2, 3
ACQ_UCB, ACQ_EI, ACQ_POI, ACQ_NONE = 0, 1, 2, 3
MAX_GPS, MAX_DIM, MAX_TOPK = 8, 64, 64
XFORM_IDENTITY, XFORM_ROUND = 0, 1
GET_L, GET_ALPHA, GET_YSTATS, GET_K, GET_LINV = 0, 1, 2, 3, 4
PRECISION_FP64, PRECISION_FP32 = 0, 1
PATH_AUTO, PATH_STABLE = 0, 1

EXPORTS = [
    "b200bo_version", "b200bo_last_error", "b200bo_device_count", "b200bo_launch_count",
    "b200bo_gp_create", "b200bo_gp_destroy", "b200bo_gp_set_precision", "b200bo_gp_set_private_stream",
    "b200bo_gp_set_transform", "b200bo_gp_fit",
    "b200bo_gp_set_data", "b200bo_gp_append", "b200bo_gp_lml", "b200bo_gp_get", "b200bo_gp_n", "b200bo_gp_dim",
    "b200bo_gp_predict", "b200bo_gp_predict_cov", "b200bo_acq_eval", "b200bo_acq_argmin_topk", "b200bo_acq_eval_dev",
    "b200bo_last_kernel_ms", "b200bo_last_select_stats",
    "b200bo_acq_argmin_topk_philox", "b200bo_acq_select_philox_dev", "b200bo_philox_rows",
    "b200bo_gp_replicate", "b200bo_multi_gpu_acq_argmin_topk", "b200bo_multi_gpu_acq_argmin_topk_philox",
    "b200bo_multi_gpu_acq_eval",
]


class KernelSpec(C.Structure):
    _fields_ = [
        ("family", C.c_int32), ("nu", C.c_int32), ("n_length_scale", C.c_int32),
        ("reserved", C.c_int32), ("const_value", C.c_double),
        ("length_scale", C.POINTER(C.c_double)), ("noise_level", C.c_double),
    ]


class AcqSpec(C.Structure):
    _fields_ = [
        ("kind", C.c_int32), ("n_gps", C.c_int32), ("path", C.c_int32), ("reserved", C.c_int32),
        ("kappa", C.c_double), ("xi", C.c_double),
        ("y_max", C.c_double), ("gps", C.c_void_p * MAX_GPS), ("lb", C.c_double * MAX_GPS),
        ("ub", C.c_double * MAX_GPS),
    ]


class B200Error(RuntimeError):
    pass


_lib = None


def lib():
    """Load libb200bo.so (once).  Raises ImportError with build instructions if absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: the sm_100a CUDA library has not been built. Run "
            "`python -c 'import __graft_entry__ as g; g.build()'` (needs nvcc). "
            "bayesianoptimization_b200 has no CPU fallback."
        )
    L = C.CDLL(LIB_PATH)
    dp = C.POINTER(C.c_double)
    i64p = C.POINTER(C.c_int64)
    L.b200bo_version.restype = C.c_int
    L.b200bo_last_error.restype = C.c_char_p
    L.b200bo_device_count.restype = C.c_int
    L.b200bo_launch_count.restype = C.c_int64
    L.b200bo_gp_create.argtypes = [C.POINTER(C.c_void_p), C.c_int]
    L.b200bo_gp_destroy.argtypes = [C.c_void_p]
    L.b200bo_gp_destroy.restype = None
    L.b200bo_gp_set_precision.argtypes = [C.c_void_p, C.c_int]
    L.b200bo_gp_set_private_stream.argtypes = [C.c_void_p, C.c_int]
    L.b200bo_gp_set_transform.argtypes = [C.c_void_p, C.POINTER(C.c_int32), C.c_int]
    L.b200bo_gp_fit.argtypes = [C.c_void_p, dp, dp, C.c_int64, C.c_int, C.POINTER(KernelSpec),
                                C.c_double, C.c_int, i64p]
    L.b200bo_gp_set_data.argtypes = [C.c_void_p, dp, dp, C.c_int64, C.c_int, C.c_int]
    L.b200bo_gp_append.argtypes = [C.c_void_p, dp, C.c_double, i64p]
    L.b200bo_gp_lml.argtypes = [C.c_void_p, C.POINTER(KernelSpec), C.c_double, C.c_int, dp, dp]
    L.b200bo_gp_get.argtypes = [C.c_void_p, C.c_int, dp, C.c_int64]
    L.b200bo_gp_n.argtypes = [C.c_void_p]
    L.b200bo_gp_n.restype = C.c_int64
    L.b200bo_gp_dim.argtypes = [C.c_void_p]
    L.b200bo_gp_predict.argtypes = [C.c_void_p, dp, C.c_int64, dp, dp, i64p]
    L.b200bo_gp_predict_cov.argtypes = [C.c_void_p, dp, C.c_int64, dp, dp]
    L.b200bo_acq_eval.argtypes = [C.POINTER(AcqSpec), dp, C.c_int64, dp]
    L.b200bo_acq_argmin_topk.argtypes = [C.POINTER(AcqSpec), dp, C.c_int64, C.c_int, dp, i64p, dp,
                                         i64p, dp]
    L.b200bo_acq_eval_dev.argtypes = [C.POINTER(AcqSpec), C.c_void_p, C.c_int64, C.c_void_p,
                                      C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int64,
                                      C.c_void_p]
    L.b200bo_last_kernel_ms.argtypes = [C.POINTER(C.c_float)]
    L.b200bo_last_select_stats.argtypes = [i64p, i64p]
    philox_outs = [dp, i64p, dp, dp, i64p, dp]
    L.b200bo_acq_argmin_topk_philox.argtypes = [C.POINTER(AcqSpec), C.c_uint64, dp, dp, C.c_int64, C.c_int64,
                                                C.c_int, *philox_outs]
    L.b200bo_acq_select_philox_dev.argtypes = [C.POINTER(AcqSpec), C.c_uint64, dp, dp, C.c_int64, C.c_int64,
                                               C.c_int, C.c_void_p, C.c_void_p]
    L.b200bo_philox_rows.argtypes = [C.c_int, C.c_uint64, dp, dp, C.c_int, i64p, C.c_int64, dp]
    L.b200bo_gp_replicate.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_void_p)]
    L.b200bo_multi_gpu_acq_argmin_topk.argtypes = [C.POINTER(AcqSpec), C.c_int, dp, C.c_int64, C.c_int, dp,
                                                   i64p, dp, i64p]
    L.b200bo_multi_gpu_acq_argmin_topk_philox.argtypes = [C.POINTER(AcqSpec), C.c_int, C.c_uint64, dp, dp,
                                                          C.c_int64, C.c_int64, C.c_int, *philox_outs]
    L.b200bo_multi_gpu_acq_eval.argtypes = [C.POINTER(AcqSpec), C.c_int, dp, C.c_int64, i64p, dp]
    _lib = L
    return L


def check(rc: int, info: int | None = None):
    """Map C-ABI error codes onto the exception types the reference's callers expect."""
    if rc == OK:
        return
    msg = lib().b200bo_last_error().decode("utf-8", "replace")
    if rc == ERR_NOT_PD:
        raise np.linalg.LinAlgError(msg)
    if rc == ERR_UNSUPPORTED:
        raise NotImplementedError(msg)
    if rc == ERR_ARG:
        raise ValueError(msg)
    raise B200Error(f"b200bo error {rc}: {msg}")


def as_dp(a: np.ndarray):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def c_f64(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.float64)
