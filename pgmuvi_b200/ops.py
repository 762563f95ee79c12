"""Torch custom ops over the C ABI (device memory, streams: torch is plumbing only).

``pgmuvi_b200::sm_mll_grad``, ``::sm_kernel_dense``, ``::optim_step``, ``::sm_fit`` take CUDA
tensors, run on the current torch CUDA stream and never fall back to the CPU.
"""
from __future__ import annotations

from typing import Optional, Tuple

import torch
from torch import Tensor

from . import _lib
from ._lib import (FLAG_BOUNDS_PER_LC, FLAG_GRAD, FLAG_LEARN_NOISE, KIND_SM1D,
                   KIND_SM_ARD_PRODSUM, KIND_SM_ARD_SUMPROD, KIND_STAT_BASE, check, is_stat,
                   param_count, ptr)

_workspaces = {}
_staged_ws = {}


def _require_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("pgmuvi_b200 ops need CUDA tensors (there is no CPU fallback)")


def _cached_ws(cache, device, need):
    """A workspace of at least `need` bytes, kept per device and grown on demand."""
    ws = cache.get(device.index)
    if ws is None or ws.numel() < need:
        cache.pop(device.index, None)   # free the old one before the larger allocation
        ws = None
        ws = torch.empty(need, dtype=torch.uint8, device=device)
        cache[device.index] = ws
    return ws


def _device_index(device):
    return device.index if device.index is not None else torch.cuda.current_device()


def _workspace(device, n_max, d, Q, extra=0):
    need = _lib.load().pgm_workspace_bytes(8, n_max, d, Q, _device_index(device))
    if extra:   # fp32 entry points: fp64 staging area behind the (256-aligned) base workspace
        need = ((need + 255) & ~255) + extra
    return _cached_ws(_workspaces, device, need)


def _n_valid(n_valid):
    return None if n_valid is None else n_valid.to(torch.int32).contiguous()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _prep(x, y, fixed_noise, raw, con_kind, con_lb, con_ub, kind, Q, learn_noise):
    _require_cuda(x, y, fixed_noise, raw, con_kind, con_lb, con_ub)
    if x.dtype not in (torch.float64, torch.float32):
        raise RuntimeError("pgmuvi_b200 ops take float64 or float32 tensors")
    for t in (y, fixed_noise, raw, con_lb, con_ub):
        if t is not None and t.dtype != x.dtype:
            raise RuntimeError(f"all floating tensors must share one dtype ({x.dtype}), "
                               f"got {t.dtype}")
    B, n = y.shape
    d = 1 if (kind == KIND_SM1D or (is_stat(kind) and (kind - KIND_STAT_BASE) % 5 == 0)) else 2
    if is_stat(kind) and Q != 0:
        raise RuntimeError("stationary kinds have no mixtures: pass Q = 0")
    if x.shape != (B, n, d):
        raise RuntimeError(f"x must be [B, n, {d}], got {tuple(x.shape)}")
    P = param_count(Q, d, learn_noise, kind)
    if raw.shape != (B, P):
        raise RuntimeError(f"raw must be [B, {P}], got {tuple(raw.shape)}")
    flags = FLAG_LEARN_NOISE if learn_noise else 0
    if con_lb.dim() == 2:
        flags |= FLAG_BOUNDS_PER_LC
        if con_lb.shape != (B, P) or con_ub.shape != (B, P):
            raise RuntimeError("per-light-curve bounds must be [B, P]")
    elif con_lb.shape != (P,) or con_ub.shape != (P,):
        raise RuntimeError("shared bounds must be [P]")
    if con_kind.shape != (P,) or con_kind.dtype != torch.int32:
        raise RuntimeError("con_kind must be int32 [P]")
    c = lambda t: None if t is None else t.contiguous()
    return (c(x), c(y), c(fixed_noise), c(raw), c(con_kind), c(con_lb), c(con_ub), B, n, d, P,
            flags)


@torch.library.custom_op("pgmuvi_b200::sm_mll_grad", mutates_args=(), device_types="cuda")
def sm_mll_grad(x: Tensor, y: Tensor, fixed_noise: Optional[Tensor], raw: Tensor,
                con_kind: Tensor, con_lb: Tensor, con_ub: Tensor, n_valid: Optional[Tensor],
                kind: int, Q: int, learn_noise: bool, want_grad: bool
                ) -> Tuple[Tensor, Tensor, Tensor]:
    """Per-datum exact MLL, d MLL / d raw and Cholesky info for B light curves."""
    (x, y, fixed_noise, raw, con_kind, con_lb, con_ub, B, n, d, P, flags) = _prep(
        x, y, fixed_noise, raw, con_kind, con_lb, con_ub, kind, Q, learn_noise)
    n_valid = _n_valid(n_valid)
    if want_grad:
        flags |= FLAG_GRAD
    mll = torch.empty(B, dtype=x.dtype, device=x.device)
    grad = torch.zeros(B, P, dtype=x.dtype, device=x.device)
    info = torch.zeros(B, dtype=torch.int32, device=x.device)
    lib = _lib.load()
    f32 = x.dtype == torch.float32
    extra = lib.pgm_f32_staging_bytes(B, n, d, Q, kind, flags, 0, 0) if f32 else 0
    ws = _workspace(x.device, n, d, Q, extra)
    entry = lib.pgm_sm_mll_grad_f32 if f32 else lib.pgm_sm_mll_grad_f64
    with torch.cuda.device(x.device):
        check(entry(
            ptr(x), ptr(n_valid), ptr(y), ptr(fixed_noise), ptr(raw), ptr(con_kind), ptr(con_lb),
            ptr(con_ub), B, n, d, Q, kind, flags, ptr(mll), ptr(grad), ptr(info), ptr(ws),
            ws.numel(), _stream()))
    return mll, grad, info


@sm_mll_grad.register_fake
def _(x, y, fixed_noise, raw, con_kind, con_lb, con_ub, n_valid, kind, Q, learn_noise,
      want_grad):
    B = y.shape[0]
    return (y.new_empty(B), torch.empty_like(raw), y.new_empty(B, dtype=torch.int32))


@torch.library.custom_op("pgmuvi_b200::sm_mll_grad_alpha", mutates_args=(), device_types="cuda")
def sm_mll_grad_alpha(x: Tensor, y: Tensor, fixed_noise: Optional[Tensor], raw: Tensor,
                      con_kind: Tensor, con_lb: Tensor, con_ub: Tensor,
                      n_valid: Optional[Tensor], kind: int, Q: int, learn_noise: bool,
                      staged: bool) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    """As :func:`sm_mll_grad` (float64, with gradient), additionally returning
    ``alpha = K~^-1 (y - c)`` [B, n]: ``d mll / d y = -alpha / n`` (the hook for non-constant
    mean functions).  ``staged`` selects the whole-device engine (long light curves)."""
    (x, y, fixed_noise, raw, con_kind, con_lb, con_ub, B, n, d, P, flags) = _prep(
        x, y, fixed_noise, raw, con_kind, con_lb, con_ub, kind, Q, learn_noise)
    n_valid = _n_valid(n_valid)
    if x.dtype != torch.float64:
        raise RuntimeError("sm_mll_grad_alpha takes float64 tensors")
    flags |= FLAG_GRAD
    mll = torch.empty(B, dtype=x.dtype, device=x.device)
    grad = torch.zeros(B, P, dtype=x.dtype, device=x.device)
    alpha = torch.zeros(B, n, dtype=x.dtype, device=x.device)
    info = torch.zeros(B, dtype=torch.int32, device=x.device)
    lib = _lib.load()
    if staged:
        ws = _cached_ws(_staged_ws, x.device, lib.pgm_staged_workspace_bytes(n, B))
        entry = lib.pgm_sm_mll_grad_staged_alpha_f64
    else:
        ws = _workspace(x.device, n, d, Q)
        entry = lib.pgm_sm_mll_grad_alpha_f64
    with torch.cuda.device(x.device):
        check(entry(ptr(x), ptr(n_valid), ptr(y), ptr(fixed_noise), ptr(raw), ptr(con_kind),
                    ptr(con_lb), ptr(con_ub), B, n, d, Q, kind, flags, ptr(mll), ptr(grad),
                    ptr(alpha), ptr(info), ptr(ws), ws.numel(), _stream()))
    return mll, grad, info, alpha


@sm_mll_grad_alpha.register_fake
def _(x, y, fixed_noise, raw, con_kind, con_lb, con_ub, n_valid, kind, Q, learn_noise, staged):
    B = y.shape[0]
    return (y.new_empty(B), torch.empty_like(raw), y.new_empty(B, dtype=torch.int32),
            torch.empty_like(y))


@torch.library.custom_op("pgmuvi_b200::sm_kernel_dense", mutates_args=(), device_types="cuda")
def sm_kernel_dense(x: Tensor, fixed_noise: Optional[Tensor], raw: Tensor, con_kind: Tensor,
                    con_lb: Tensor, con_ub: Tensor, n_valid: Optional[Tensor], kind: int, Q: int,
                    learn_noise: bool) -> Tensor:
    """Dense K + D [B, n, n] from the same device builder the fused path uses."""
    B, n = x.shape[0], x.shape[1]
    y = x.new_empty(B, n)
    (x, _, fixed_noise, raw, con_kind, con_lb, con_ub, B, n, d, P, flags) = _prep(
        x, y, fixed_noise, raw, con_kind, con_lb, con_ub, kind, Q, learn_noise)
    n_valid = _n_valid(n_valid)
    if x.dtype != torch.float64:
        raise RuntimeError("sm_kernel_dense takes float64 tensors")
    K = torch.zeros(B, n, n, dtype=x.dtype, device=x.device)
    with torch.cuda.device(x.device):
        check(_lib.load().pgm_sm_kernel_dense_f64(
            ptr(x), ptr(n_valid), ptr(fixed_noise), ptr(raw), ptr(con_kind), ptr(con_lb),
            ptr(con_ub), B, n, d, Q, kind, flags, ptr(K), _stream()))
    return K


@sm_kernel_dense.register_fake
def _(x, fixed_noise, raw, con_kind, con_lb, con_ub, n_valid, kind, Q, learn_noise):
    return x.new_empty(x.shape[0], x.shape[1], x.shape[1])


@torch.library.custom_op("pgmuvi_b200::optim_step", mutates_args=("raw", "exp_avg", "exp_avg_sq"),
                         device_types="cuda")
def optim_step(raw: Tensor, grad_mll: Tensor, exp_avg: Tensor, exp_avg_sq: Tensor,
               active: Optional[Tensor], optim_kind: int, lr: float, beta1: float, beta2: float,
               eps: float, weight_decay: float, step: int) -> None:
    """In-place SGD / Adam / AdamW step on packed raw parameters [B, P] (minimises -MLL)."""
    _require_cuda(raw, grad_mll, exp_avg, exp_avg_sq, active)
    B, P = raw.shape
    for t in (raw, grad_mll, exp_avg, exp_avg_sq):
        if not t.is_contiguous() or t.dtype != torch.float64:
            raise RuntimeError("optim_step needs contiguous float64 tensors")
    with torch.cuda.device(raw.device):
        check(_lib.load().pgm_optim_step_f64(
            ptr(raw), ptr(grad_mll), ptr(exp_avg), ptr(exp_avg_sq), ptr(active), B, P, optim_kind,
            lr, beta1, beta2, eps, weight_decay, step, _stream()))


@optim_step.register_fake
def _(raw, grad_mll, exp_avg, exp_avg_sq, active, optim_kind, lr, beta1, beta2, eps, weight_decay,
      step):
    return None


@torch.library.custom_op("pgmuvi_b200::sm_fit", mutates_args=("raw",), device_types="cuda")
def sm_fit(x: Tensor, y: Tensor, fixed_noise: Optional[Tensor], raw: Tensor, con_kind: Tensor,
           con_lb: Tensor, con_ub: Tensor, n_valid: Optional[Tensor], kind: int, Q: int,
           learn_noise: bool, optim_kind: int, lr: float, beta1: float, beta2: float, eps: float,
           weight_decay: float, maxiter: int, miniter: int, stop: float, stopavg: int,
           keep_history: bool) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    """Whole optimisation loop on device.  Returns (loss_hist [maxiter,B],
    raw_hist [maxiter+1,B,P] or empty, n_iter [B], info [B]); ``raw`` is updated in place."""
    (x, y, fixed_noise, raw_c, con_kind, con_lb, con_ub, B, n, d, P, flags) = _prep(
        x, y, fixed_noise, raw, con_kind, con_lb, con_ub, kind, Q, learn_noise)
    n_valid = _n_valid(n_valid)
    if not raw.is_contiguous():
        raise RuntimeError("raw must be contiguous (updated in place)")
    loss_hist = torch.empty(maxiter, B, dtype=x.dtype, device=x.device)
    raw_hist = torch.empty((maxiter + 1, B, P) if keep_history else (0,), dtype=x.dtype,
                           device=x.device)
    n_iter = torch.zeros(B, dtype=torch.int32, device=x.device)
    info = torch.zeros(B, dtype=torch.int32, device=x.device)
    lib = _lib.load()
    if x.dtype == torch.float32:
        extra = lib.pgm_f32_staging_bytes(B, n, d, Q, kind, flags, maxiter, int(keep_history))
        ws = _workspace(x.device, n, d, Q, extra)
        with torch.cuda.device(x.device):
            check(lib.pgm_sm_fit_f32(
                ptr(x), ptr(n_valid), ptr(y), ptr(fixed_noise), ptr(raw), ptr(con_kind),
                ptr(con_lb), ptr(con_ub), B, n, d, Q, kind, flags, optim_kind, lr, beta1, beta2,
                eps, weight_decay, maxiter, miniter, stop, stopavg, ptr(loss_hist),
                ptr(raw_hist) if keep_history else None, ptr(n_iter), ptr(info), ptr(ws),
                ws.numel(), _stream()))
        return loss_hist, raw_hist, n_iter, info
    ws = _workspace(x.device, n, d, Q)
    with torch.cuda.device(x.device):
        check(lib.pgm_sm_fit_f64(
            ptr(x), ptr(n_valid), ptr(y), ptr(fixed_noise), ptr(raw), ptr(con_kind), ptr(con_lb),
            ptr(con_ub), B, n, d, Q, kind, flags, optim_kind, lr, beta1, beta2, eps, weight_decay,
            maxiter, miniter, stop, stopavg, ptr(loss_hist),
            ptr(raw_hist) if keep_history else None, ptr(n_iter), ptr(info), None, ptr(ws),
            ws.numel(), _stream()))
    return loss_hist, raw_hist, n_iter, info


@sm_fit.register_fake
def _(x, y, fixed_noise, raw, con_kind, con_lb, con_ub, n_valid, kind, Q, learn_noise, optim_kind,
      lr, beta1, beta2, eps, weight_decay, maxiter, miniter, stop, stopavg, keep_history):
    B, P = raw.shape
    return (y.new_empty(maxiter, B),
            y.new_empty((maxiter + 1, B, P) if keep_history else (0,)),
            y.new_empty(B, dtype=torch.int32), y.new_empty(B, dtype=torch.int32))


def sm_mll_grad_staged(x: Tensor, y: Tensor, fixed_noise: Optional[Tensor], raw: Tensor,
                       con_kind: Tensor, con_lb: Tensor, con_ub: Tensor,
                       n_valid: Optional[Tensor], kind: int, Q: int, learn_noise: bool,
                       want_grad: bool = True, tf32x3: bool = False, tf32x3_chol: bool = False,
                       nosync: bool = False) -> Tuple[Tensor, Tensor, Tensor]:
    """Same contract as :func:`sm_mll_grad`, through the staged whole-device engine
    (``pgm_sm_mll_grad_staged_f64``): every light curve's K~ lives in HBM as 64x64 tiles and
    the batch advances stage by stage.  Blocking.

    ``tf32x3=True``: the K~^-1 = X^T X products of the gradient run on the Blackwell tensor cores
    (tcgen05, 3xTF32; ``pgm_sm_mll_grad_staged_tf32x3_f64`` for float64 tensors,
    ``pgm_sm_mll_grad_tf32x3_f32`` for float32 tensors - the reference's default dtype).
    ``tf32x3_chol=True`` (implied for float32 tensors): the trailing updates of the panel-schedule
    Cholesky run there too.
    ``nosync=True``: no host synchronisation (``PGM_FLAG_NOSYNC``; single GPs up to n = 12800 and small
    batches): ``info`` is final once the stream has drained."""
    (x, y, fixed_noise, raw, con_kind, con_lb, con_ub, B, n, d, P, flags) = _prep(
        x, y, fixed_noise, raw, con_kind, con_lb, con_ub, kind, Q, learn_noise)
    n_valid = _n_valid(n_valid)
    f32 = x.dtype == torch.float32
    if f32 and not tf32x3:
        raise RuntimeError("the staged engine takes float64 tensors (float32: tf32x3=True)")
    if want_grad:
        flags |= FLAG_GRAD
    if nosync:
        flags |= _lib.FLAG_NOSYNC
    if tf32x3_chol:
        if not tf32x3:
            raise RuntimeError("tf32x3_chol needs tf32x3=True")
        flags |= _lib.FLAG_TF32X3_CHOL
    lib = _lib.load()
    if tf32x3:
        need = lib.pgm_staged_tf32x3_workspace_bytes(n, B)
        if f32:
            need = ((need + 255) & ~255) + lib.pgm_f32_staging_bytes(B, n, d, Q, kind, flags, 0, 0)
    else:
        need = lib.pgm_staged_workspace_bytes(n, B)
    ws = _cached_ws(_staged_ws, x.device, need)
    mll = torch.empty(B, dtype=x.dtype, device=x.device)
    grad = torch.zeros(B, P, dtype=x.dtype, device=x.device)
    info = torch.zeros(B, dtype=torch.int32, device=x.device)
    entry = (lib.pgm_sm_mll_grad_tf32x3_f32 if f32 else lib.pgm_sm_mll_grad_staged_tf32x3_f64
             if tf32x3 else lib.pgm_sm_mll_grad_staged_f64)
    with torch.cuda.device(x.device):
        check(entry(
            ptr(x), ptr(n_valid), ptr(y), ptr(fixed_noise), ptr(raw), ptr(con_kind), ptr(con_lb),
            ptr(con_ub), B, n, d, Q, kind, flags, ptr(mll), ptr(grad), ptr(info), ptr(ws),
            ws.numel(), _stream()))
    return mll, grad, info


def sm_predict(x: Tensor, y: Tensor, fixed_noise: Optional[Tensor], raw: Tensor,
               con_kind: Tensor, con_lb: Tensor, con_ub: Tensor, n_valid: Optional[Tensor],
               xstar: Tensor, kind: int, Q: int, learn_noise: bool
               ) -> Tuple[Tensor, Tensor, Tensor]:
    """Exact posterior mean and latent variance at ``xstar [B, m, d]`` for B light curves
    (``pgm_sm_predict_f64``).  Returns (mean [B, m], var [B, m], info [B]); blocking."""
    (x, y, fixed_noise, raw, con_kind, con_lb, con_ub, B, n, d, P, flags) = _prep(
        x, y, fixed_noise, raw, con_kind, con_lb, con_ub, kind, Q, learn_noise)
    n_valid = _n_valid(n_valid)
    _require_cuda(xstar)
    if xstar.dim() == 2:
        xstar = xstar.unsqueeze(-1)
    if xstar.shape[0] != B or xstar.shape[2] != d or xstar.dtype != torch.float64:
        raise RuntimeError(f"xstar must be float64 [B, m, {d}]")
    xstar = xstar.contiguous()
    m = xstar.shape[1]
    lib = _lib.load()
    ws = _cached_ws(_staged_ws, x.device,
                    lib.pgm_predict_workspace_bytes(n, B, _device_index(x.device)))
    mean = torch.empty(B, m, dtype=x.dtype, device=x.device)
    var = torch.empty(B, m, dtype=x.dtype, device=x.device)
    info = torch.zeros(B, dtype=torch.int32, device=x.device)
    with torch.cuda.device(x.device):
        check(lib.pgm_sm_predict_f64(
            ptr(x), ptr(n_valid), ptr(y), ptr(fixed_noise), ptr(raw), ptr(con_kind), ptr(con_lb),
            ptr(con_ub), B, n, d, Q, kind, flags, ptr(xstar), m, ptr(mean), ptr(var), ptr(info),
            ptr(ws), ws.numel(), _stream()))
    return mean, var, info


def sm_mll_grad_large(x: Tensor, y: Tensor, fixed_noise: Optional[Tensor], raw: Tensor,
                      con_kind: Tensor, con_lb: Tensor, con_ub: Tensor, kind: int, Q: int,
                      learn_noise: bool, want_grad: bool = True, nosync: bool = False):
    """ONE large GP (x [n, d], y [n], raw [P]) factored by the whole device: the staged engine
    with B = 1.  Returns (mll 0-d tensor, grad [P], info int); blocking.
    ``nosync=True`` (n <= 12800): nothing is synchronised and ``info`` comes back as a 0-d DEVICE
    tensor - the caller reads it when it has to."""
    if x.dim() == 1:
        x = x.unsqueeze(-1)
    mll, grad, info = sm_mll_grad_staged(
        x.unsqueeze(0), y.unsqueeze(0), None if fixed_noise is None else fixed_noise.unsqueeze(0),
        raw.reshape(1, -1), con_kind, con_lb.reshape(-1), con_ub.reshape(-1), None, kind, Q,
        learn_noise, want_grad, nosync=nosync)
    return mll[0], grad[0], (info[0] if nosync else int(info.item()))


@torch.library.custom_op("pgmuvi_b200::sm_fisher", mutates_args=(), device_types="cuda")
def sm_fisher(x: Tensor, y: Tensor, fixed_noise: Optional[Tensor], raw: Tensor, con_kind: Tensor,
              con_lb: Tensor, con_ub: Tensor, n_valid: Optional[Tensor], kind: int, Q: int,
              learn_noise: bool) -> Tuple[Tensor, Tensor]:
    """Expected (Fisher) information of the exact log-likelihood ``n * mll`` in the constrained
    parameters, ``fisher [B, P, P]``, and the Cholesky ``info [B]`` (``pgm_sm_fisher_f64``: the
    staged engine's P and T phases, then the Fisher kernels).  Rows of a light curve with
    ``info < 0`` are NaN.  float64 only; blocking."""
    (x, y, fixed_noise, raw, con_kind, con_lb, con_ub, B, n, d, P, flags) = _prep(
        x, y, fixed_noise, raw, con_kind, con_lb, con_ub, kind, Q, learn_noise)
    n_valid = _n_valid(n_valid)
    if x.dtype != torch.float64:
        raise RuntimeError("sm_fisher takes float64 tensors")
    fisher = torch.empty(B, P, P, dtype=x.dtype, device=x.device)
    info = torch.zeros(B, dtype=torch.int32, device=x.device)
    lib = _lib.load()
    # not cached between calls: a batch's workspace can take most of the device memory
    ws = torch.empty(lib.pgm_fisher_workspace_bytes(n, B, d, Q, kind, flags), dtype=torch.uint8,
                     device=x.device)
    with torch.cuda.device(x.device):
        check(lib.pgm_sm_fisher_f64(
            ptr(x), ptr(n_valid), ptr(y), ptr(fixed_noise), ptr(raw), ptr(con_kind), ptr(con_lb),
            ptr(con_ub), B, n, d, Q, kind, flags, ptr(fisher), ptr(info), ptr(ws), ws.numel(),
            _stream()))
    return fisher, info


@sm_fisher.register_fake
def _(x, y, fixed_noise, raw, con_kind, con_lb, con_ub, n_valid, kind, Q, learn_noise):
    B, P = raw.shape
    return y.new_empty(B, P, P), y.new_empty(B, dtype=torch.int32)


def fisher_workspace_bytes(n_max: int, B: int, d: int, Q: int, kind: int, learn_noise: bool) -> int:
    """Device bytes one :func:`sm_fisher` call of B light curves of up to n_max points needs."""
    return int(_lib.load().pgm_fisher_workspace_bytes(n_max, B, d, Q, kind,
                                                      FLAG_LEARN_NOISE if learn_noise else 0))


def peak_probe(kind: int, iters: int = 4096) -> float:
    """Self-measured FP64 DMMA (0) / DFMA (1) / FP32 FFMA (2) throughput in TFLOP/s."""
    import ctypes
    out = ctypes.c_double(0.0)
    check(_lib.load().pgm_peak_probe(kind, iters, ctypes.byref(out), _stream()))
    return out.value


__all__ = ["sm_mll_grad", "sm_fisher", "sm_mll_grad_alpha", "sm_mll_grad_large", "sm_mll_grad_staged", "sm_predict", "sm_kernel_dense", "optim_step", "sm_fit",
           "peak_probe", "param_count",
           "KIND_SM1D", "KIND_SM_ARD_PRODSUM", "KIND_SM_ARD_SUMPROD"]
