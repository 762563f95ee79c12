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


CON_NONE, CON_SOFTPLUS, CON_INTERVAL, CON_RSOFTPLUS = 0, 1, 2, 3
FLAG_GRAD, FLAG_LEARN_NOISE, FLAG_BOUNDS_PER_LC, FLAG_JITTER_F32, FLAG_TF32X3, FLAG_TF32X3_CHOL, FLAG_NOSYNC = (
    1, 2, 4, 8, 16, 32, 64)
OPT_SGD, OPT_ADAM, OPT_ADAMW = 0, 1, 2

EXPORTS = (
    "pgm_version", "pgm_last_error", "pgm_workspace_bytes", "pgm_sm_mll_grad_f64",
    "pgm_sm_kernel_dense_f64", "pgm_optim_step_f64", "pgm_sm_fit_f64", "pgm_peak_probe",
    "pgm_staged_workspace_bytes", "pgm_sm_mll_grad_staged_f64",
    "pgm_predict_workspace_bytes", "pgm_sm_predict_f64",
    "pgm_f32_staging_bytes", "pgm_sm_mll_grad_f32", "pgm_sm_fit_f32",
    "pgm_lombscargle_f64", "pgm_ls_peaks_f64",
    "pgm_sm_mll_grad_alpha_f64", "pgm_sm_mll_grad_staged_alpha_f64",
    "pgm_sm_psd_peak_f64",
    "pgm_staged_tf32x3_workspace_bytes", "pgm_sm_mll_grad_staged_tf32x3_f64",
    "pgm_sm_mll_grad_tf32x3_f32", "pgm_fused_grid",
    "pgm_fisher_workspace_bytes", "pgm_sm_fisher_f64",
)

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
    dp, ip, vp = c_void_p, c_void_p, c_void_p  # device pointers travel as integers
    lib.pgm_version.restype = c_int
    lib.pgm_last_error.restype = c_char_p
    lib.pgm_workspace_bytes.restype = c_size_t
    lib.pgm_workspace_bytes.argtypes = [c_int, c_int, c_int, c_int, c_int]
    lib.pgm_sm_mll_grad_f64.restype = c_int
    lib.pgm_sm_mll_grad_f64.argtypes = [dp, ip, dp, dp, dp, ip, dp, dp, c_int, c_int, c_int,
                                        c_int, c_int, c_int, dp, dp, ip, vp, c_size_t, vp]
    lib.pgm_sm_kernel_dense_f64.restype = c_int
    lib.pgm_sm_kernel_dense_f64.argtypes = [dp, ip, dp, dp, ip, dp, dp, c_int, c_int, c_int,
                                            c_int, c_int, c_int, dp, vp]
    lib.pgm_optim_step_f64.restype = c_int
    lib.pgm_optim_step_f64.argtypes = [dp, dp, dp, dp, ip, c_int, c_int, c_int, c_double,
                                       c_double, c_double, c_double, c_double, c_int, vp]
    lib.pgm_sm_fit_f64.restype = c_int
    lib.pgm_sm_fit_f64.argtypes = [dp, ip, dp, dp, dp, ip, dp, dp, c_int, c_int, c_int, c_int,
                                   c_int, c_int, c_int, c_double, c_double, c_double, c_double,
                                   c_double, c_int, c_int, c_double, c_int, dp, dp, ip, ip, dp,
                                   vp, c_size_t, vp]
    lib.pgm_staged_workspace_bytes.restype = c_size_t
    lib.pgm_staged_workspace_bytes.argtypes = [c_int, c_int]
    lib.pgm_sm_mll_grad_staged_f64.restype = c_int
    lib.pgm_sm_mll_grad_staged_f64.argtypes = lib.pgm_sm_mll_grad_f64.argtypes
    lib.pgm_fused_grid.restype = c_int
    lib.pgm_fused_grid.argtypes = [c_int, c_int, c_int]
    lib.pgm_staged_tf32x3_workspace_bytes.restype = c_size_t
    lib.pgm_staged_tf32x3_workspace_bytes.argtypes = [c_int, c_int]
    lib.pgm_sm_mll_grad_staged_tf32x3_f64.restype = c_int
    lib.pgm_sm_mll_grad_staged_tf32x3_f64.argtypes = lib.pgm_sm_mll_grad_f64.argtypes
    lib.pgm_sm_mll_grad_tf32x3_f32.restype = c_int
    lib.pgm_sm_mll_grad_tf32x3_f32.argtypes = lib.pgm_sm_mll_grad_f64.argtypes
    lib.pgm_predict_workspace_bytes.restype = c_size_t
    lib.pgm_predict_workspace_bytes.argtypes = [c_int, c_int, c_int]
    lib.pgm_sm_predict_f64.restype = c_int
    lib.pgm_sm_predict_f64.argtypes = [dp, ip, dp, dp, dp, ip, dp, dp, c_int, c_int, c_int, c_int,
                                       c_int, c_int, dp, c_int, dp, dp, ip, vp, c_size_t, vp]
    lib.pgm_f32_staging_bytes.restype = c_size_t
    lib.pgm_f32_staging_bytes.argtypes = [c_int] * 8
    lib.pgm_sm_mll_grad_f32.restype = c_int
    lib.pgm_sm_mll_grad_f32.argtypes = lib.pgm_sm_mll_grad_f64.argtypes
    lib.pgm_sm_fit_f32.restype = c_int
    lib.pgm_sm_fit_f32.argtypes = [dp, ip, dp, dp, dp, ip, dp, dp, c_int, c_int, c_int, c_int,
                                   c_int, c_int, c_int, c_double, c_double, c_double, c_double,
                                   c_double, c_int, c_int, c_double, c_int, dp, dp, ip, ip,
                                   vp, c_size_t, vp]
    lib.pgm_lombscargle_f64.restype = c_int
    lib.pgm_lombscargle_f64.argtypes = [dp, ip, dp, dp, c_int, c_int, dp, dp, ip, c_int, c_int,
                                        dp, vp]
    lib.pgm_ls_peaks_f64.restype = c_int
    lib.pgm_ls_peaks_f64.argtypes = [dp, ip, c_int, c_int, c_int, c_int, ip, dp, vp, c_size_t, vp]
    lib.pgm_sm_mll_grad_alpha_f64.restype = c_int
    lib.pgm_sm_mll_grad_alpha_f64.argtypes = [dp, ip, dp, dp, dp, ip, dp, dp, c_int, c_int, c_int,
                                              c_int, c_int, c_int, dp, dp, dp, ip, vp, c_size_t, vp]
    lib.pgm_sm_mll_grad_staged_alpha_f64.restype = c_int
    lib.pgm_sm_mll_grad_staged_alpha_f64.argtypes = lib.pgm_sm_mll_grad_alpha_f64.argtypes
    lib.pgm_sm_psd_peak_f64.restype = c_int
    lib.pgm_sm_psd_peak_f64.argtypes = [dp, dp, dp, dp, dp, c_int, c_int, c_int, dp, dp, ip, dp, dp,
                                        ip, vp]
    lib.pgm_fisher_workspace_bytes.restype = c_size_t
    lib.pgm_fisher_workspace_bytes.argtypes = [c_int] * 6
    lib.pgm_sm_fisher_f64.restype = c_int
    lib.pgm_sm_fisher_f64.argtypes = [dp, ip, dp, dp, dp, ip, dp, dp, c_int, c_int, c_int, c_int,
                                      c_int, c_int, dp, ip, vp, c_size_t, vp]
    lib.pgm_peak_probe.restype = c_int
    lib.pgm_peak_probe.argtypes = [c_int, c_int, POINTER(c_double), vp]
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise EngineError(f"pgmuvi_b200 C ABI error {rc}: {load().pgm_last_error().decode()}")


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()
