"""ctypes binding of include/gprb200.h - one Python method per exported symbol, nothing else.
Same ABI a Julia ``ccall((:gprb_eval, libgprb200), Cint, ...)`` would hit (see INTEGRATION.md)."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))

EXPORTS = [
    "gprb_version", "gprb_last_error", "gprb_init", "gprb_init_multi", "gprb_destroy", "gprb_device_info",
    "gprb_dataset_create", "gprb_datasets_create", "gprb_dataset_update", "gprb_datasets_update", "gprb_dataset_destroy",
    "gprb_batch_create", "gprb_batch_set_targets", "gprb_batch_set_diag_offset", "gprb_batch_destroy", "gprb_batch_append",
    "gprb_eval", "gprb_eval_mixed", "gprb_eval_device", "gprb_lbfgs_default_opts", "gprb_optimize", "gprb_lbfgs_selftest",
    "gprb_predict", "gprb_predict_async", "gprb_predict_wait", "gprb_last_predict_ms",
    "gprb_predict_cov", "gprb_sample_posterior", "gprb_eval_loo", "gprb_predict_grad",
    "gprb_get_K", "gprb_get_chol", "gprb_get_alpha", "gprb_get_Kinv",
    "gprb_comm_unique_id", "gprb_comm_init_rank", "gprb_gather", "gprb_gather_multi",
    "gprb_set_profiling", "gprb_last_stage_ms", "gprb_last_gemm_launch_ms", "gprb_launch_count",
]


class GprbError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libgprb200 error {code}: {msg}")
        self.code = code


class LbfgsOpts(C.Structure):
    _fields_ = [("m", C.c_int32), ("iterations", C.c_int32), ("max_evals", C.c_int32), ("ls_iterations", C.c_int32),
                ("g_abstol", C.c_double), ("time_limit", C.c_double),
                ("c_1", C.c_double), ("rho_hi", C.c_double), ("rho_lo", C.c_double),
                ("cost_value", C.c_double), ("cost_grad", C.c_double)]


class OptResult(C.Structure):
    _fields_ = [("mll", C.c_double), ("g_norm", C.c_double), ("iterations", C.c_int32), ("f_calls", C.c_int32),
                ("fg_calls", C.c_int32), ("converged", C.c_int32), ("ls_failed", C.c_int32), ("info", C.c_int32)]


def library_path() -> str:
    return os.environ.get("GPRB200_LIB", os.path.join(_HERE, "libgprb200.so"))


_dp = C.POINTER(C.c_double)
_vp = C.c_void_p


def _d(a):
    return a.ctypes.data_as(_dp) if a is not None else None


class Library:
    """Loaded libgprb200.so with typed prototypes.  Loading needs no GPU; ``init`` does."""

    def __init__(self, path: str | None = None):
        path = path or library_path()
        if not os.path.exists(path):
            raise GprbError(-3, f"{path} not found - build it with gpr.jl_b200/csrc/build.sh "
                                "(there is no CPU fallback for this path)")
        self.path = path
        self.dll = C.CDLL(path)
        L = self.dll
        L.gprb_version.restype = C.c_int
        L.gprb_last_error.restype = C.c_char_p
        L.gprb_init.argtypes = [C.POINTER(_vp), C.c_int]
        L.gprb_init_multi.argtypes = [C.POINTER(_vp), C.c_int32, C.POINTER(C.c_int)]
        L.gprb_destroy.argtypes = [_vp]
        L.gprb_device_info.argtypes = [_vp, C.POINTER(C.c_int64)]
        L.gprb_dataset_create.argtypes = [_vp, C.c_int64, C.c_int32, _dp, C.c_int64, C.POINTER(_vp)]
        L.gprb_datasets_create.argtypes = [_vp, C.c_int32, C.c_int64, C.c_int32, C.POINTER(_dp), C.c_int64, C.POINTER(_vp)]
        L.gprb_dataset_update.argtypes = [_vp, _dp, C.c_int64]
        L.gprb_datasets_update.argtypes = [_vp, C.c_int32, C.POINTER(_vp), C.POINTER(_dp), C.c_int64]
        L.gprb_dataset_destroy.argtypes = [_vp]
        L.gprb_batch_create.argtypes = [_vp, C.c_int32, C.POINTER(_vp), _dp, C.c_int32, C.POINTER(_vp)]
        L.gprb_batch_set_targets.argtypes = [_vp, _dp]
        L.gprb_batch_set_diag_offset.argtypes = [_vp, _dp]
        L.gprb_batch_destroy.argtypes = [_vp]
        L.gprb_batch_append.argtypes = [_vp, C.c_int64, C.POINTER(_dp), C.c_int64, _dp, _dp, C.POINTER(C.c_int32)]
        L.gprb_eval.argtypes = [_vp, _dp, C.POINTER(C.c_uint8), _dp, _dp, C.POINTER(C.c_int32)]
        L.gprb_eval_mixed.argtypes = [_vp, _dp, C.POINTER(C.c_uint8), _dp, _dp, C.POINTER(C.c_int32)]
        L.gprb_eval_device.argtypes = [_vp, _vp, _vp, _vp, _vp, _vp]
        L.gprb_lbfgs_default_opts.argtypes = [C.POINTER(LbfgsOpts)]
        L.gprb_lbfgs_default_opts.restype = None
        L.gprb_optimize.argtypes = [_vp, _dp, C.POINTER(LbfgsOpts), C.POINTER(OptResult)]
        L.gprb_lbfgs_selftest.argtypes = [C.c_int32, C.c_int32, _dp, C.POINTER(LbfgsOpts), C.c_double, C.POINTER(OptResult)]
        L.gprb_predict.argtypes = [_vp, C.c_int64, _dp, C.c_int64, _dp, _dp, _dp]
        L.gprb_predict_async.argtypes = [_vp, C.c_int32, C.c_int32, C.c_int32, C.c_int64, _dp, C.c_int64, C.c_int32, _dp, C.c_int32]
        L.gprb_predict_wait.argtypes = [_vp, C.c_int32, _dp, _dp]
        L.gprb_last_predict_ms.argtypes = [_vp, C.c_int32, _dp]
        L.gprb_predict_cov.argtypes = [_vp, C.c_int64, _dp, C.c_int64, _dp, C.c_int32, _dp, _dp]
        L.gprb_sample_posterior.argtypes = [_vp, C.c_int64, _dp, C.c_int64, _dp, C.c_int32, _dp, _dp, C.POINTER(C.c_int32)]
        L.gprb_predict_grad.argtypes = [_vp, C.c_int64, _dp, C.c_int64, _dp, _dp, _dp, _dp, _dp, _dp]
        L.gprb_eval_loo.argtypes = [_vp, _dp, C.POINTER(C.c_uint8), _dp, _dp, _dp, _dp, _dp, _dp, C.POINTER(C.c_int32)]
        L.gprb_comm_unique_id.argtypes = [C.c_void_p]
        L.gprb_comm_init_rank.argtypes = [_vp, C.c_int32, C.c_int32, C.c_void_p]
        _ip = C.POINTER(C.c_int32)
        L.gprb_gather.argtypes = [_vp, C.c_int32, C.c_int32, C.c_int32, _ip, _dp, _dp]
        L.gprb_gather_multi.argtypes = [C.POINTER(_vp), C.c_int32, C.c_int32, C.c_int32, _ip, C.POINTER(_ip), C.POINTER(_dp), _dp]
        for f in ("gprb_get_K", "gprb_get_chol", "gprb_get_alpha", "gprb_get_Kinv"):
            getattr(L, f).argtypes = [_vp, C.c_int32, _dp]
        L.gprb_set_profiling.argtypes = [_vp, C.c_int32]
        L.gprb_last_stage_ms.argtypes = [_vp, _dp]
        L.gprb_last_gemm_launch_ms.argtypes = [_vp, _dp, C.c_int32]
        L.gprb_launch_count.argtypes = [_vp]
        L.gprb_launch_count.restype = C.c_int64

    def check(self, rc: int):
        if rc != 0:
            raise GprbError(rc, self.dll.gprb_last_error().decode())

    def has_symbol(self, name: str) -> bool:
        try:
            getattr(self.dll, name)
            return True
        except AttributeError:
            return False


_LIB = None


def load_library() -> Library:
    global _LIB
    if _LIB is None:
        _LIB = Library()
    return _LIB


def as_f64(a, order="C"):
    return np.require(a, dtype=np.float64, requirements=["C_CONTIGUOUS" if order == "C" else "F_CONTIGUOUS", "ALIGNED"])
