"""ctypes binding of libpgmuvi_b200.so (the C ABI in include/pgmuvi_b200.h).

This is the binding a pgmuvi maintainer would add (INTEGRATION.md).  There is no CPU
fallback: if the shared library is missing the import of any compute entry point raises.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_double, c_int, c_int32, c_size_t, c_void_p, POINTER

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libpgmuvi_b200.so")

# constants mirrored from include/pgmuvi_b200.h
KIND_SM1D, KIND_SM_ARD_PRODSUM, KIND_SM_ARD_SUMPROD = 0, 1, 2
KIND_SEP_RBF, KIND_SEP_MATERN15, KIND_SEP_RQ, KIND_SEP_CONST = 3, 4, 5, 6
SEP_KINDS = (KIND_SEP_RBF, KIND_SEP_MATERN15, KIND_SEP_RQ, KIND_SEP_CONST)
NUM_LAM = {KIND_SEP_RBF: 2, KIND_SEP_MATERN15: 2, KIND_SEP_RQ: 3, KIND_SEP_CONST: 1}
# N3 stationary time kernels: kind = 8 + 5 * TK + WK (TK 0 RBF / 1 Matern-1.5 / 2 QP; WK 0 none,
# 1 RBF, 2 Matern-1.5, 3 RQ, 4 Constant), no mixtures (Q = 0)
KIND_STAT_BASE = 8


def stat_kind(tk, wk):
    return KIND_STAT_BASE + 5 * tk + wk


def is_stat(kind):
    return KIND_STAT_BASE <= kind <= stat_kind(5, 0)


def stat_num_lam(kind):
    tk, wk = divmod(kind - KIND_STAT_BASE, 5)
    return (2, 2, 4, 6, 2, 2)[tk] + (0, 2, 2, 3, 1)[wk]


def param_count(Q: int, d: int, learn_noise: bool, kind: int = -1) -> int:
    """P of the packed layout ``[mean | w | mu | sigma | (noise) | lam]`` (pgmuvi_b200.h)."""
    if is_stat(kind):            # stationary time kernels: no mixtures (Q = 0)
        return 1 + (1 if learn_noise else 0) + stat_num_lam(kind)
    if kind in SEP_KINDS:
        return 1 + 3 * Q + (1 if learn_noise else 0) + NUM_LAM[kind]
    return 1 + Q + 2 * Q * d + (1 if learn_noise else 0)


CON_NONE, CON_SOFTPLUS, CON_INTERVAL, CON_RSOFTPLUS = 0, 1, 2, 3
FLAG_GRAD, FLAG_LEARN_NOISE, FLAG_BOUNDS_PER_LC, FLAG_JITTER_F32, FLAG_TF32X3, FLAG_TF32X3_CHOL, FLAG_NOSYNC = (
    1, 2, 4, 8, 16, 32, 64)
OPT_SGD, OPT_ADAM, OPT_ADAMW = 0, 1, 2

# every exported symbol: name -> (restype, argtypes); device pointers travel as integers
_dp = _ip = _vp = c_void_p
_MLL_GRAD = [_dp, _ip, _dp, _dp, _dp, _ip, _dp, _dp, c_int, c_int, c_int, c_int, c_int, c_int,
             _dp, _dp, _ip, _vp, c_size_t, _vp]
_MLL_GRAD_ALPHA = [_dp, _ip, _dp, _dp, _dp, _ip, _dp, _dp, c_int, c_int, c_int, c_int, c_int,
                   c_int, _dp, _dp, _dp, _ip, _vp, c_size_t, _vp]
_FIT = [_dp, _ip, _dp, _dp, _dp, _ip, _dp, _dp, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
        c_double, c_double, c_double, c_double, c_double, c_int, c_int, c_double, c_int, _dp, _dp,
        _ip, _ip]
PROTOTYPES = {
    "pgm_version": (c_int, []),
    "pgm_last_error": (c_char_p, []),
    "pgm_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_int, c_int]),
    "pgm_sm_mll_grad_f64": (c_int, _MLL_GRAD),
    "pgm_sm_kernel_dense_f64": (c_int, [_dp, _ip, _dp, _dp, _ip, _dp, _dp, c_int, c_int, c_int,
                                        c_int, c_int, c_int, _dp, _vp]),
    "pgm_optim_step_f64": (c_int, [_dp, _dp, _dp, _dp, _ip, c_int, c_int, c_int, c_double,
                                   c_double, c_double, c_double, c_double, c_int, _vp]),
    "pgm_sm_fit_f64": (c_int, _FIT + [_dp, _vp, c_size_t, _vp]),
    "pgm_peak_probe": (c_int, [c_int, c_int, POINTER(c_double), _vp]),
    "pgm_staged_workspace_bytes": (c_size_t, [c_int, c_int]),
    "pgm_sm_mll_grad_staged_f64": (c_int, _MLL_GRAD),
    "pgm_predict_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "pgm_sm_predict_f64": (c_int, [_dp, _ip, _dp, _dp, _dp, _ip, _dp, _dp, c_int, c_int, c_int,
                                   c_int, c_int, c_int, _dp, c_int, _dp, _dp, _ip, _vp, c_size_t,
                                   _vp]),
    "pgm_f32_staging_bytes": (c_size_t, [c_int] * 8),
    "pgm_sm_mll_grad_f32": (c_int, _MLL_GRAD),
    "pgm_sm_fit_f32": (c_int, _FIT + [_vp, c_size_t, _vp]),
    "pgm_lombscargle_f64": (c_int, [_dp, _ip, _dp, _dp, c_int, c_int, _dp, _dp, _ip, c_int, c_int,
                                    _dp, _vp]),
    "pgm_ls_peaks_f64": (c_int, [_dp, _ip, c_int, c_int, c_int, c_int, _ip, _dp, _vp, c_size_t,
                                 _vp]),
    "pgm_sm_mll_grad_alpha_f64": (c_int, _MLL_GRAD_ALPHA),
    "pgm_sm_mll_grad_staged_alpha_f64": (c_int, _MLL_GRAD_ALPHA),
    "pgm_sm_psd_peak_f64": (c_int, [_dp, _dp, _dp, _dp, _dp, c_int, c_int, c_int, _dp, _dp, _ip,
                                    _dp, _dp, _ip, _vp]),
    "pgm_staged_tf32x3_workspace_bytes": (c_size_t, [c_int, c_int]),
    "pgm_sm_mll_grad_staged_tf32x3_f64": (c_int, _MLL_GRAD),
    "pgm_sm_mll_grad_tf32x3_f32": (c_int, _MLL_GRAD),
    "pgm_fused_grid": (c_int, [c_int, c_int, c_int]),
    "pgm_fisher_workspace_bytes": (c_size_t, [c_int] * 6),
    "pgm_sm_fisher_f64": (c_int, [_dp, _ip, _dp, _dp, _dp, _ip, _dp, _dp, c_int, c_int, c_int,
                                  c_int, c_int, c_int, _dp, _ip, _vp, c_size_t, _vp]),
}
EXPORTS = tuple(PROTOTYPES)

_lib = None


class EngineError(RuntimeError):
    """The CUDA engine rejected the call (bad argument or launch failure)."""


def load():
    """Load the shared library (once) and declare the prototypes.  Fails loudly."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: build it with `python -m pgmuvi_b200.build` "
            "(pgmuvi_b200 has no CPU fallback)")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (restype, argtypes) in PROTOTYPES.items():
        fn = getattr(lib, name)
        fn.restype = restype
        fn.argtypes = argtypes
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise EngineError(f"pgmuvi_b200 C ABI error {rc}: {load().pgm_last_error().decode()}")


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()
