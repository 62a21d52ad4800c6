"""ctypes binding of ``libkfb200.so`` (C ABI in ``include/kfb200.h``).

There is NO fallback: if the CUDA library is missing or a call fails this module raises.
"""
from __future__ import annotations

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("KFB_LIB") or os.path.join(_HERE, "libkfb200.so")  # KFB_LIB: developer override (A/B builds)

KFB_STANDARD, KFB_UNIVARIATE, KFB_STEADY_STATE, KFB_SINGLE, KFB_CHOLESKY = range(5)
FILTER_KIND = {
    "standard": KFB_STANDARD,
    "univariate": KFB_UNIVARIATE,
    "steady_state": KFB_STEADY_STATE,
    "single": KFB_SINGLE,
    "cholesky": KFB_CHOLESKY,
}
KFB_FLAG_CORRECTED = 1
KFB_FLAG_FORCE_COOP = 2
KFB_FLAG_GENERIC_ADJOINT = 4
KFB_FLAG_Z_UNIT0 = 8
KFB_FLAG_H_ZERO = 16
KFB_FLAG_T_COMPANION = 32
KFB_FLAG_NO_MISSING = 64
KFB_FLAG_TIME_PARALLEL = 128
KFB_FLAG_PARTIAL_ROWS = 256
KFB_INFO_DARE_FAILED = 0x40000001
KFB_INFO_NOT_STATIONARY = 0x40000002
KFB_INFO_BAD_STRUCTURE = 0x40000003
KFB_INFO_NOT_PSD = 0x40000004
KFB_SHOCK_UNIT, KFB_SHOCK_STD, KFB_SHOCK_CHOLESKY = range(3)  # kfb_impulse_response: S = I, diag(sqrt(diag Q)), chol(Q)
SHOCK_KIND = {"unit": KFB_SHOCK_UNIT, "std": KFB_SHOCK_STD, "cholesky": KFB_SHOCK_CHOLESKY}

KFB_OK, KFB_ERR_INVALID_ARG, KFB_ERR_UNSUPPORTED, KFB_ERR_WORKSPACE, KFB_ERR_CUDA = range(5)

_c_i32, _c_i64, _c_u32, _vp = ctypes.c_int32, ctypes.c_int64, ctypes.c_uint32, ctypes.c_void_p


class KfbDesc(ctypes.Structure):
    _fields_ = (
        [("filter_kind", _c_i32), ("flags", _c_u32), ("n_draws", _c_i64), ("n_series", _c_i64)]
        + [(k, _c_i32) for k in ("n", "m", "p", "r")]
        + [(k + "_bs", _c_i64) for k in ("y", "a0", "P0", "T", "Z", "R", "H", "Q", "c", "d")]
        + [(k + "_ts", _c_i64) for k in ("T", "Z", "R", "H", "Q", "c", "d")]
    )


class KfbInputs(ctypes.Structure):
    _fields_ = [(k, _vp) for k in ("y", "a0", "P0", "T", "Z", "R", "H", "Q", "c", "d")]


class KfbOutputs(ctypes.Structure):
    _fields_ = [(k, _vp) for k in ("loglik", "ll_obs", "filtered_states", "predicted_states", "filtered_covs",
                                  "predicted_covs", "info")]


class KfbCotangents(ctypes.Structure):
    _fields_ = [(k, _vp) for k in ("g_loglik", "g_ll_obs")]


class KfbGrads(ctypes.Structure):
    _fields_ = [(k, _vp) for k in ("a0", "P0", "T", "Z", "R", "H", "Q", "c", "d")]


KFB_MAX_SCATTER_SEGMENTS = 8


class KfbScatterSeg(ctypes.Structure):
    _fields_ = [("block", _c_i32), ("n_map", _c_i32), ("base", _vp), ("src_idx", _vp), ("dst_idx", _vp), ("data", _vp)]


EXPORTS = {
    "kfb_version": (_c_i32, []),
    "kfb_status_string": (ctypes.c_char_p, [_c_i32]),
    "kfb_last_cuda_error": (ctypes.c_char_p, []),
    "kfb_launch_count": (_c_i64, []),
    "kfb_workspace_bytes": (_c_i32, [ctypes.POINTER(KfbDesc), _c_i32, ctypes.POINTER(ctypes.c_size_t)]),
    "kfb_forward": (_c_i32, [ctypes.POINTER(KfbDesc), ctypes.POINTER(KfbInputs), ctypes.POINTER(KfbOutputs), _vp,
                             ctypes.c_size_t, _c_i32, _vp]),
    "kfb_backward": (_c_i32, [ctypes.POINTER(KfbDesc), ctypes.POINTER(KfbInputs), ctypes.POINTER(KfbCotangents),
                              ctypes.POINTER(KfbGrads), _vp, ctypes.c_size_t, _vp]),
    "kfb_smoother": (_c_i32, [_c_i64, _c_i64, _c_i32, _c_i32, _c_i32, _vp, _c_i64, _vp, _c_i64, _vp, _c_i64, _vp, _vp, _vp, _vp,
                              _vp, ctypes.c_size_t, _vp]),
    "kfb_smoother_ex": (_c_i32, [_c_i64, _c_i64, _c_i32, _c_i32, _c_i32, _vp, _c_i64, _vp, _c_i64, _vp, _c_i64, _vp, _vp, _vp,
                                 _vp, _vp, ctypes.c_size_t, ctypes.c_uint32, _vp]),
    "kfb_lyapunov_forward": (_c_i32, [_c_i64, _c_i32, _c_i32, _vp, _c_i64, _vp, _c_i64, _vp, _c_i64, _vp, _vp, _vp]),
    "kfb_lyapunov_backward": (_c_i32, [_c_i64, _c_i32, _c_i32, _vp, _c_i64, _vp, _c_i64, _vp, _c_i64, _vp, _vp, _vp,
                                       _vp, _vp, _vp]),
    "kfb_scatter_forward": (_c_i32, [_c_i64, _c_i32, _c_i32, _c_i32, _vp, _vp, _vp, _vp, _vp, _vp]),
    "kfb_scatter_backward": (_c_i32, [_c_i64, _c_i32, _c_i32, _c_i32, _vp, _vp, _vp, _vp, _vp]),
    "kfb_scatter_forward_multi": (_c_i32, [_c_i64, _c_i32, _c_i32, ctypes.POINTER(KfbScatterSeg), _vp, _vp]),
    "kfb_scatter_backward_multi": (_c_i32, [_c_i64, _c_i32, _c_i32, ctypes.POINTER(KfbScatterSeg), _vp, _vp]),
    "kfb_simulate": (_c_i32, [_c_i64, _c_i64, _c_i32, _c_i32, _c_i32, _c_i32, _vp, _c_i64, _vp, _c_i64, _vp, _c_i64, _vp, _c_i64,
                              _vp, _c_i64, _vp, _c_i64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "kfb_mvn_draws": (_c_i32, [_c_i64, _c_i64, _c_i32, _c_i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "kfb_simulation_smoother_workspace_bytes": (_c_i32, [ctypes.POINTER(KfbDesc), _c_i64, ctypes.POINTER(ctypes.c_size_t)]),
    "kfb_simulation_smoother": (_c_i32, [ctypes.POINTER(KfbDesc), ctypes.POINTER(KfbInputs), _vp, _c_i64, _vp, _vp, _vp, _vp,
                                         _vp, _vp, ctypes.c_size_t, _vp]),
    "kfb_forecast_paths_workspace_bytes": (_c_i32, [ctypes.POINTER(KfbDesc), _c_i64, ctypes.POINTER(ctypes.c_size_t)]),
    "kfb_forecast_paths": (_c_i32, [ctypes.POINTER(KfbDesc), ctypes.POINTER(KfbInputs), _vp, _vp, _c_i32, _c_i64, _vp, _vp,
                                    _vp, _vp, _vp, _vp, _vp, ctypes.c_size_t, _vp]),
    "kfb_conditional_forecast_workspace_bytes": (_c_i32, [ctypes.POINTER(KfbDesc), _c_i32, _c_i64,
                                                          ctypes.POINTER(ctypes.c_size_t)]),
    "kfb_conditional_forecast": (_c_i32, [ctypes.POINTER(KfbDesc), ctypes.POINTER(KfbInputs), _vp, _vp, _c_i32, _vp, _c_i64,
                                          _c_i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, ctypes.c_size_t,
                                          _vp]),
    "kfb_masked_filter_workspace_bytes": (_c_i32, [ctypes.POINTER(KfbDesc), ctypes.POINTER(ctypes.c_size_t)]),
    "kfb_masked_filter": (_c_i32, [ctypes.POINTER(KfbDesc), ctypes.POINTER(KfbInputs), _vp, _vp, _vp, _vp, ctypes.c_size_t,
                                   _vp]),
    "kfb_impulse_response": (_c_i32, [ctypes.POINTER(KfbDesc), ctypes.POINTER(KfbInputs), _c_i32, _c_i32, _vp, _vp, _vp,
                                      _vp]),
    "kfb_fp64_peak": (_c_i32, [_c_i32, _c_i32, _c_i32, _vp, ctypes.POINTER(ctypes.c_double), _vp]),
    "kfb_fp64_peak_distinct": (_c_i32, [_c_i32, _c_i32, _c_i32, _vp, ctypes.POINTER(ctypes.c_double), _vp]),
}

_lib = None


class KfbError(RuntimeError):
    def __init__(self, status, where):
        self.status = status
        lib = load()
        msg = lib.kfb_status_string(status).decode()
        if status == KFB_ERR_CUDA:
            msg += ": " + lib.kfb_last_cuda_error().decode()
        super().__init__(f"{where}: {msg} (kfb_status={status})")


def load():
    """dlopen libkfb200.so and declare every prototype.  Raises if the library was not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(make -C pymc_statespace_b200/csrc).  pymc_statespace_b200 has no CPU fallback."
        )
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in EXPORTS.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is missing
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(status, where):
    if status != KFB_OK:
        raise KfbError(status, where)
