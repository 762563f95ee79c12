"""Torch-CPU restatement of the reference hot path (oracle + CPU baseline).

TEST INFRASTRUCTURE - see ``oracle/__init__.py`` (parity unpinned at the GPyTorch
boundary).  Every function cites what it follows.  Reference paths are relative to
``/root/reference``; "A.n" is SURVEY.md Appendix A (restated GPyTorch maths, whose source
is not vendored in the reference tree).

The path (pgmuvi/trainers.py:177-182):

    output = model(train_x)              # gps.py:217-220 ConstantMean + SpectralMixtureKernel
    loss   = -ExactMLL(output, train_y)  # trainers.py:119,180  (Cholesky, per-datum)
    loss.backward()                      # trainers.py:181
    optimizer.step()                     # trainers.py:141-147,182 (SGD/Adam/AdamW on RAW params)

Packed raw-parameter layout used by the oracle, the C ABI and the golden files
(``P = 1 + Q + 2*Q*ds (+1) + NL``)::

    [ mean | w[0..Q) | mu[q*ds + k] | sigma[q*ds + k] | (learned noise) | lam[0..NL) ]

``ds`` = dims the spectral mixture acts on (= d, or 1 for the separable kinds whose
wavelength factor has the ``NL`` parameters ``lam``).
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import numpy as np
import torch

# kernel kinds -------------------------------------------------------------------------
KIND_SM1D = 0              # gps.py:208  SMK(num_mixtures=Q)                       (d = 1)
KIND_SM_ARD_PRODSUM = 1    # gps.py:305  SMK(ard_num_dims=2): prod_d sum_q (GPyTorch; F7)
KIND_SM_ARD_SUMPROD = 2    # switchable variant: sum_q w_q prod_d (notebook tinygp cell; F7)
# separable 2-D models (gps.py:1327-1336  covar = time_kernel * wavelength_kernel with
# active_dims [0] / [1]); time kernel = SMK(Q, ard_num_dims=1) (gps.py:990-1002)
KIND_SEP_RBF = 3           # x ScaleKernel(RBFKernel())          gps.py:1045-1048, 1063-1064
KIND_SEP_MATERN15 = 4      # x ScaleKernel(MaternKernel(nu=1.5)) gps.py:1049-1052
KIND_SEP_RQ = 5            # x ScaleKernel(RQKernel())           gps.py:1053-1056
KIND_SEP_CONST = 6         # x ConstantKernel()                  gps.py:1414-1415 (Achromatic)
SEP_KINDS = (KIND_SEP_RBF, KIND_SEP_MATERN15, KIND_SEP_RQ, KIND_SEP_CONST)
NUM_LAM = {KIND_SEP_RBF: 2, KIND_SEP_MATERN15: 2, KIND_SEP_RQ: 3, KIND_SEP_CONST: 1}
# N3: stationary time kernels instead of the spectral mixture (gps.py:985-990, 1131-1184,
# 1316-1319): kind = 8 + 5 * TK + WK, TK 0 ScaleKernel(RBF) / 1 ScaleKernel(Matern-1.5) in time,
# WK 0 none (1-D) / 1 RBF / 2 Matern-1.5 / 3 RQ / 4 Constant in wavelength; Q = 0.
KIND_STAT_BASE = 8
ATOM_QP = 100      # time atom 2: quasi-periodic ScaleKernel(PeriodicKernel * RBFKernel), gps.py:915-935
ATOM_QP_RBF = 101  # time atom 3: AdditiveKernel(QP, ScaleKernel(RBFKernel)), gps.py:1187-1236 (1-D only)
ATOM_M12, ATOM_M25 = 102, 103   # time atoms 4 / 5: ScaleKernel(MaternKernel(0.5 | 2.5)), gps.py:1166-1179


def stat_kind(tk: int, wk: int) -> int:
    return KIND_STAT_BASE + 5 * tk + wk


def stat_atoms(kind: int):
    """(time atom, wavelength atom or None) as separable-kind codes."""
    tk, wk = divmod(kind - KIND_STAT_BASE, 5)
    return ((KIND_SEP_RBF, KIND_SEP_MATERN15, ATOM_QP, ATOM_QP_RBF, ATOM_M12, ATOM_M25)[tk],
            None if wk == 0 else (KIND_SEP_RBF, KIND_SEP_MATERN15, KIND_SEP_RQ, KIND_SEP_CONST)[wk - 1])

# constraint kinds (A.2) ---------------------------------------------------------------
CON_NONE = 0       # value = raw
CON_SOFTPLUS = 1   # Positive / GreaterThan(lb): value = softplus(raw) + lb
CON_RSOFTPLUS = 3  # value = ub / (softplus(raw) + lb)  (flicker term: sigma = 1 / (2 pi lengthscale))
CON_INTERVAL = 2   # Interval(lb, ub):           value = lb + (ub - lb) * sigmoid(raw)

TWO_PI = 2.0 * math.pi


@dataclass(frozen=True)
class ModelSpec:
    """Static description of one model family on the path."""

    d: int = 1                 # input dims (1: time; 2: time, wavelength)
    Q: int = 4                 # num_mixtures (gps.py:205 default 4)
    kind: int = KIND_SM1D
    learn_noise: bool = False  # GaussianLikelihood / FixedNoise(learn_additional_noise)
    # fixed per-point noise is a data argument (None -> absent)

    @property
    def ds(self) -> int:
        """dims the spectral mixture acts on (separable kinds: time only)."""
        return 1 if (self.kind in SEP_KINDS or self.kind >= KIND_STAT_BASE) else self.d

    @property
    def NL(self) -> int:
        """parameters behind the mixture: wavelength kernel of the separable kinds; time +
        wavelength kernel of the stationary kinds."""
        if self.kind >= KIND_STAT_BASE:
            ta, wl = stat_atoms(self.kind)
            return {ATOM_QP: 4, ATOM_QP_RBF: 6}.get(ta, 2) + (0 if wl is None else NUM_LAM[wl])
        return NUM_LAM.get(self.kind, 0)

    @property
    def P(self) -> int:
        return 1 + self.Q + 2 * self.Q * self.ds + (1 if self.learn_noise else 0) + self.NL

    # slot offsets in the packed layout
    @property
    def o_w(self):
        return 1

    @property
    def o_mu(self):
        return 1 + self.Q

    @property
    def o_sigma(self):
        return 1 + self.Q + self.Q * self.ds

    @property
    def o_noise(self):
        return 1 + self.Q + 2 * self.Q * self.ds

    @property
    def o_lam(self):
        return self.o_noise + (1 if self.learn_noise else 0)


# ---------------------------------------------------------------------------------------
# constraints (A.2; chosen by lightcurve.py:3817-4008, SMK defaults Positive)
# ---------------------------------------------------------------------------------------
def constrain(raw, kinds, lb, ub):
    """raw -> constrained value, elementwise.  kinds int tensor/array [P]."""
    kinds = torch.as_tensor(kinds)
    sp = torch.nn.functional.softplus(raw) + lb
    iv = lb + (ub - lb) * torch.sigmoid(raw)
    out = torch.where(kinds == CON_SOFTPLUS, sp, raw)
    out = torch.where(kinds == CON_INTERVAL, iv, out)
    # CON_RSOFTPLUS: ub / (softplus(raw) + lb) - a lengthscale seen as an SM frequency scale
    out = torch.where(kinds == CON_RSOFTPLUS, ub / sp, out)
    return out


def unconstrain(val, kinds, lb, ub):
    """Inverse of :func:`constrain` (A.2: log(expm1(v-lb)); logit((v-lb)/(ub-lb)))."""
    kinds = torch.as_tensor(kinds)
    val = torch.as_tensor(val)
    lb = torch.as_tensor(lb, dtype=val.dtype)
    ub = torch.as_tensor(ub, dtype=val.dtype)
    v = val - lb
    # inv softplus: x + log(-expm1(-x)), stable for large x
    sp = torch.where(v > 30, v, v + torch.log(-torch.expm1(-v.clamp(min=1e-300))))
    u = (v / (ub - lb)).clamp(1e-300, 1 - 1e-16)
    iv = torch.log(u) - torch.log1p(-u)
    out = torch.where(kinds == CON_SOFTPLUS, sp, val)
    out = torch.where(kinds == CON_INTERVAL, iv, out)
    return out


def unpack_params(theta, spec: ModelSpec):
    """Split a packed (constrained or raw) vector [..., P] into named pieces."""
    Q, d = spec.Q, spec.ds
    mean = theta[..., 0]
    w = theta[..., spec.o_w:spec.o_w + Q]
    mu = theta[..., spec.o_mu:spec.o_mu + Q * d].reshape(*theta.shape[:-1], Q, d)
    sigma = theta[..., spec.o_sigma:spec.o_sigma + Q * d].reshape(*theta.shape[:-1], Q, d)
    noise = theta[..., spec.o_noise] if spec.learn_noise else None
    return mean, w, mu, sigma, noise


# ---------------------------------------------------------------------------------------
# kernel (A.3: gpytorch.kernels.SpectralMixtureKernel.forward, instantiated gps.py:208,305)
# ---------------------------------------------------------------------------------------
def sm_kernel_dense(x1, x2, w, mu, sigma, kind=KIND_SM1D):
    """Dense spectral-mixture covariance, following GPyTorch's op order.

    x1 [..., n, d], x2 [..., m, d]; w [..., Q]; mu, sigma [..., Q, d].
    tau is formed as ``x1*p - x2*p`` (scale, then subtract) as GPyTorch does (F8).
    Returns [..., n, m].
    """
    x1_ = x1.unsqueeze(-3)                         # [..., 1, n, d]
    x2_ = x2.unsqueeze(-3)
    sc = sigma.unsqueeze(-2)                       # [..., Q, 1, d]
    mn = mu.unsqueeze(-2)
    x1e, x2e = x1_ * sc, x2_ * sc                  # [..., Q, n, d]
    x1c, x2c = x1_ * mn, x2_ * mn
    exp_term = (x1e.unsqueeze(-2) - x2e.unsqueeze(-3)).pow(2).mul(-2 * math.pi ** 2)
    cos_term = (x1c.unsqueeze(-2) - x2c.unsqueeze(-3)).mul(TWO_PI)
    res = exp_term.exp() * cos_term.cos()          # [..., Q, n, m, d]
    if kind in (KIND_SM1D, KIND_SM_ARD_PRODSUM):
        # "Sum over mixtures" then "Product over dimensions" (F7 / A.3)
        ww = w.unsqueeze(-1).unsqueeze(-1).unsqueeze(-1)
        return (res * ww).sum(-4).prod(-1)
    if kind == KIND_SM_ARD_SUMPROD:
        ww = w.unsqueeze(-1).unsqueeze(-1)
        return (res.prod(-1) * ww).sum(-3)
    raise ValueError(f"unknown kernel kind {kind}")


def unpack_lam(theta, spec: ModelSpec):
    """Wavelength-kernel parameters [..., NL] of the separable kinds."""
    return theta[..., spec.o_lam:spec.o_lam + spec.NL]


def wavelength_kernel_dense(l1, l2, lam, kind):
    """Wavelength factor of the separable kinds, following GPyTorch's kernels (A.3):
    ScaleKernel: outputscale * base;  RBF exp(-tau^2 / (2 l^2));  Matern-1.5
    (1 + sqrt3 r) exp(-sqrt3 r), r = |tau| / l;  RQ (1 + tau^2 / (2 alpha l^2))^-alpha;
    ConstantKernel: constant.   l1 [..., n], l2 [..., m]; lam [..., NL]."""
    tau = l1.unsqueeze(-1) - l2.unsqueeze(-2)
    ex = lambda t: t.unsqueeze(-1).unsqueeze(-1)
    if kind == KIND_SEP_CONST:
        return ex(lam[..., 0]) * torch.ones_like(tau)
    os_, ell = ex(lam[..., 0]), ex(lam[..., 1])
    if kind == KIND_SEP_RBF:
        return os_ * torch.exp(-0.5 * (tau / ell) ** 2)
    if kind == KIND_SEP_MATERN15:
        r = math.sqrt(3.0) * (tau / ell).abs()
        return os_ * (1.0 + r) * torch.exp(-r)
    if kind == ATOM_M12:      # MaternKernel(nu=0.5): exp(-|tau| / l)
        return os_ * torch.exp(-(tau / ell).abs())
    if kind == ATOM_M25:      # MaternKernel(nu=2.5): (1 + sqrt5 d + 5/3 d^2) exp(-sqrt5 d)
        r = math.sqrt(5.0) * (tau / ell).abs()
        return os_ * (1.0 + r + r * r / 3.0) * torch.exp(-r)
    if kind == KIND_SEP_RQ:
        al = ex(lam[..., 2])
        return os_ * (1.0 + (tau / ell) ** 2 / (2.0 * al)) ** (-al)
    raise ValueError(f"not a separable kind: {kind}")


def kernel_dense(x1, x2, theta, spec: ModelSpec):
    """Dense covariance of any kind from a constrained packed vector theta [..., P].
    Separable kinds: ProductKernel restricted by active_dims (gps.py:1319-1336), i.e. the
    elementwise product K_t(x[:, 0]) * K_l(x[:, 1])  (tests/test_kernels.py:130-139)."""
    mean, w, mu, sigma, noise = unpack_params(theta, spec)
    if spec.kind >= KIND_STAT_BASE:
        # ScaleKernel(time atom)(x[:, 0]) [* wavelength kernel (x[:, 1])]: the same GPyTorch
        # kernels as the wavelength factors, acting on the time column
        lam = unpack_lam(theta, spec)
        ta, wa = stat_atoms(spec.kind)
        if ta in (ATOM_QP, ATOM_QP_RBF):
            # GPyTorch PeriodicKernel: exp(-2 sin^2(pi tau / p) / lengthscale) (the lengthscale
            # is NOT squared in gpytorch >= 1.x), times RBFKernel, inside one ScaleKernel
            nt = 4
            ex = lambda t: t.unsqueeze(-1).unsqueeze(-1)
            tau = x1[..., 0].unsqueeze(-1) - x2[..., 0].unsqueeze(-2)
            os_, lmb, per, ell = (ex(lam[..., k]) for k in range(4))
            K = os_ * torch.exp(-2.0 * torch.sin(math.pi * tau / per) ** 2 / lmb) \
                * torch.exp(-0.5 * (tau / ell) ** 2)
            if ta == ATOM_QP_RBF:       # + stochastic ScaleKernel(RBFKernel)
                nt = 6
                K = K + wavelength_kernel_dense(x1[..., 0], x2[..., 0], lam[..., 4:6], KIND_SEP_RBF)
        else:
            nt = 2
            K = wavelength_kernel_dense(x1[..., 0], x2[..., 0], lam[..., :2], ta)
        if wa is not None:
            K = K * wavelength_kernel_dense(x1[..., 1], x2[..., 1], lam[..., nt:], wa)
        return K
    if spec.kind in SEP_KINDS:
        Kt = sm_kernel_dense(x1[..., :1], x2[..., :1], w, mu, sigma, KIND_SM1D)
        Kl = wavelength_kernel_dense(x1[..., 1], x2[..., 1], unpack_lam(theta, spec), spec.kind)
        return Kt * Kl
    return sm_kernel_dense(x1, x2, w, mu, sigma, spec.kind)


def noise_diag(n, fixed_noise, learned_noise, dtype):
    """A.4: D = diag(fixed) (+ sigma^2 I).  fixed_noise is already squared/clamped by the
    host layer (lightcurve.py:2780-2784; GPyTorch min_fixed_noise clamp)."""
    dvec = torch.zeros(n, dtype=dtype)
    if fixed_noise is not None:
        dvec = dvec + fixed_noise
    if learned_noise is not None:
        dvec = dvec + learned_noise.unsqueeze(-1)
    return dvec


# ---------------------------------------------------------------------------------------
# Cholesky with GPyTorch's jitter ladder (A.5: linear_operator psd_safe_cholesky)
# ---------------------------------------------------------------------------------------
def default_jitter(dtype):
    """First rung of the ladder: GPyTorch's cholesky_jitter, 1e-6 for float32 and 1e-8 for float64."""
    return 1e-6 if dtype == torch.float32 else 1e-8


def jitter_rung(info, jitter):
    """Diagonal jitter that rung `info` (1..3) adds: jitter * 10^(info - 1)."""
    return jitter * 10 ** (int(info) - 1)


def psd_safe_cholesky(A, max_tries=3, jitter=None):
    """Try plain; on failure add jitter*10^i to failed members only.  `jitter` is the first rung,
    None: default_jitter(A.dtype).  jitter=1e-6 on float64 input gives the float32 ladder
    (PGM_FLAG_JITTER_F32) in float64 arithmetic.

    Returns (L, info) with info[b] = 0 ok without jitter, k>0 = succeeded at jitter try k,
    -1 = NaN input (NanError), -2 = not PD after max_tries (NotPSDError).
    """
    batch = A.shape[:-2]
    Af = A.reshape(-1, *A.shape[-2:]).clone()
    info_out = torch.zeros(Af.shape[0], dtype=torch.int32)
    nan = torch.isnan(Af).flatten(1).any(1)
    info_out[nan] = -1
    L, info = torch.linalg.cholesky_ex(Af)
    bad = (info > 0) & ~nan
    if jitter is None:
        jitter = default_jitter(A.dtype)
    prev = 0.0
    for i in range(max_tries):
        if not bad.any():
            break
        jn = jitter * (10 ** i)
        idx = torch.nonzero(bad).flatten()
        Aj = Af[idx]
        Aj.diagonal(dim1=-2, dim2=-1).add_(jn - prev)
        Af[idx] = Aj
        prev = jn
        Lj, ij = torch.linalg.cholesky_ex(Aj)
        L[idx] = Lj
        ok = ij == 0
        info_out[idx[ok]] = i + 1
        bad[idx[ok]] = False
    info_out[bad] = -2
    return L.reshape(*batch, *A.shape[-2:]), info_out.reshape(batch)


# ---------------------------------------------------------------------------------------
# exact MLL (A.5: ExactMarginalLogLikelihood.forward -> MVN.log_prob, per datum)
# ---------------------------------------------------------------------------------------
def _mll_from_theta(x, y, fixed_noise, theta, spec: ModelSpec, jitter=None):
    """Per-datum MLL from constrained theta.  x [n,d], y [n], theta [P]."""
    n = y.shape[-1]
    if jitter is None:
        jitter = default_jitter(y.dtype)
    mean, w, mu, sigma, noise = unpack_params(theta, spec)
    K = kernel_dense(x, x, theta, spec)
    Kt = K + torch.diag_embed(noise_diag(n, fixed_noise, noise, y.dtype))
    L, info = psd_safe_cholesky(Kt.detach(), jitter=jitter)
    if int(info) > 0:  # re-apply the jitter that made it succeed, keeping the graph
        Kt = Kt + jitter_rung(info, jitter) * torch.eye(n, dtype=y.dtype)
    if int(info) < 0:
        return torch.full((), float("nan"), dtype=y.dtype), info
    L = torch.linalg.cholesky(Kt)
    r = (y - mean).unsqueeze(-1)
    z = torch.linalg.solve_triangular(L, r, upper=False)
    inv_quad = (z * z).sum()
    logdet = 2.0 * torch.log(torch.diagonal(L)).sum()
    mll = -0.5 * (inv_quad + logdet + n * math.log(TWO_PI)) / n
    return mll, info


def mll_and_grad_autograd(x, y, fixed_noise, raw, kinds, lb, ub, spec: ModelSpec, jitter=None):
    """One light curve through GPyTorch's op sequence with torch autograd
    (trainers.py:179-181).  Returns (mll, dmll/draw [P], info)."""
    raw = raw.detach().clone().requires_grad_(True)
    theta = constrain(raw, kinds, lb, ub)
    mll, info = _mll_from_theta(x, y, fixed_noise, theta, spec, jitter)
    if int(info) < 0:
        return mll.detach(), torch.full_like(raw, float("nan")).detach(), info
    (g,) = torch.autograd.grad(mll, raw)
    return mll.detach(), g, info


def constraint_jacobian(raw, kinds, lb, ub):
    """d value / d raw (A.2)."""
    kinds = torch.as_tensor(kinds)
    s = torch.sigmoid(raw)
    j = torch.ones_like(raw)
    j = torch.where(kinds == CON_SOFTPLUS, s, j)
    j = torch.where(kinds == CON_INTERVAL, (ub - lb) * s * (1 - s), j)
    v = torch.nn.functional.softplus(raw) + lb
    j = torch.where(kinds == CON_RSOFTPLUS, -ub * s / (v * v), j)
    return j


def mll_and_grad_analytic(x, y, fixed_noise, raw, kinds, lb, ub, spec: ModelSpec, jitter=None):
    """Same quantity via the closed form of A.5 (what the CUDA gradient kernel computes):

        W = alpha alpha^T - Kt^-1,  dMLL/dtheta = (1/2n) sum_ij W_ij dK_ij/dtheta,
        dMLL/dnoise = (1/2n) tr W,  dMLL/dc = (1/n) sum_i alpha_i,   then x Jacobian.

    `jitter`: first rung of the Cholesky's jitter ladder (psd_safe_cholesky)."""
    dt = y.dtype
    n = y.shape[-1]
    Q, d = spec.Q, spec.ds
    if spec.kind >= KIND_STAT_BASE:
        # stationary kinds: the closed form is d K / d theta by autograd of the dense kernel,
        # contracted with W (the Cholesky part is still the explicit one below)
        return _mll_and_grad_stat(x, y, fixed_noise, raw, kinds, lb, ub, spec, jitter)
    theta = constrain(raw, kinds, lb, ub)
    mean, w, mu, sigma, noise = unpack_params(theta, spec)
    K = kernel_dense(x, x, theta, spec)
    Kt = K + torch.diag_embed(noise_diag(n, fixed_noise, noise, dt))
    L, info = psd_safe_cholesky(Kt, jitter=jitter)
    if int(info) < 0:
        nanv = torch.full((), float("nan"), dtype=dt)
        return nanv, torch.full_like(raw, float("nan")), info
    r = (y - mean).unsqueeze(-1)
    alpha = torch.cholesky_solve(r, L)
    Kinv = torch.cholesky_inverse(L)
    inv_quad = (r * alpha).sum()
    logdet = 2.0 * torch.log(torch.diagonal(L)).sum()
    mll = -0.5 * (inv_quad + logdet + n * math.log(TWO_PI)) / n
    W = alpha @ alpha.T - Kinv

    sep = spec.kind in SEP_KINDS
    if sep:
        # K = Kt o Kl: the time-kernel parameters see W o Kl, the wavelength ones W o Kt
        lam = unpack_lam(theta, spec)
        Kl = wavelength_kernel_dense(x[:, 1], x[:, 1], lam, spec.kind)
        Ktime = K / Kl
        W_full = W
        W = W * Kl
        x_full, x = x, x[:, :1]
    tau = x.unsqueeze(-2) - x.unsqueeze(-3)                     # [n, n, ds]
    E = torch.exp(-2 * math.pi ** 2 * (tau.unsqueeze(0) * sigma[:, None, None, :]) ** 2)
    ph = TWO_PI * tau.unsqueeze(0) * mu[:, None, None, :]       # [Q, n, n, d]
    C, S = torch.cos(ph), torch.sin(ph)
    EC = E * C
    g = torch.zeros(spec.P, dtype=dt)
    g[0] = alpha.sum() / n
    half = 0.5 / n
    if spec.kind in (KIND_SM1D, KIND_SM_ARD_PRODSUM) or sep:
        Sd = (w[:, None, None, None] * EC).sum(0)               # [n, n, d]
        for k in range(d):
            R = torch.ones(n, n, dtype=dt)
            for k2 in range(d):
                if k2 != k:
                    R = R * Sd[..., k2]
            WR = W * R
            for q in range(Q):
                g[spec.o_w + q] += half * (WR * EC[q, ..., k]).sum()
                g[spec.o_mu + q * d + k] = half * (
                    WR * (-TWO_PI * tau[..., k] * w[q] * E[q, ..., k] * S[q, ..., k])).sum()
                g[spec.o_sigma + q * d + k] = half * (
                    WR * (-4 * math.pi ** 2 * tau[..., k] ** 2 * sigma[q, k] * w[q]
                          * EC[q, ..., k])).sum()
    else:  # sum over q of w_q prod_d
        for q in range(Q):
            Pq = EC[q].prod(-1)
            g[spec.o_w + q] = half * (W * Pq).sum()
            for k in range(d):
                Rq = torch.ones(n, n, dtype=dt)
                for k2 in range(d):
                    if k2 != k:
                        Rq = Rq * EC[q, ..., k2]
                g[spec.o_mu + q * d + k] = half * (
                    W * Rq * (-TWO_PI * tau[..., k] * w[q] * E[q, ..., k] * S[q, ..., k])).sum()
                g[spec.o_sigma + q * d + k] = half * (
                    W * Rq * (-4 * math.pi ** 2 * tau[..., k] ** 2 * sigma[q, k] * w[q]
                              * EC[q, ..., k])).sum()
    if sep:
        W = W_full
        tl = x_full[:, 1].unsqueeze(-1) - x_full[:, 1].unsqueeze(-2)
        WK = W * Ktime
        if spec.kind == KIND_SEP_CONST:
            g[spec.o_lam] = half * WK.sum()
        else:
            os_, ell = lam[0], lam[1]
            f = Kl / os_
            g[spec.o_lam] = half * (WK * f).sum()
            if spec.kind == KIND_SEP_RBF:
                dfdl = f * tl ** 2 / ell ** 3
            elif spec.kind == KIND_SEP_MATERN15:
                u = math.sqrt(3.0) * tl.abs() / ell
                dfdl = u ** 2 * torch.exp(-u) / ell
            else:
                al = lam[2]
                u = tl ** 2 / (2.0 * al * ell ** 2)
                dfdl = 2.0 * al * f * u / ((1.0 + u) * ell)
                g[spec.o_lam + 2] = half * (WK * os_ * f * (u / (1.0 + u) - torch.log1p(u))).sum()
            g[spec.o_lam + 1] = half * (WK * os_ * dfdl).sum()
    if spec.learn_noise:
        g[spec.o_noise] = half * torch.diagonal(W).sum()
    g = g * constraint_jacobian(raw, kinds, lb, ub)
    return mll, g, info


def _mll_and_grad_stat(x, y, fixed_noise, raw, kinds, lb, ub, spec: ModelSpec, jitter=None):
    """mll_and_grad_analytic for the stationary kinds: W from the explicit Cholesky, then
    g_theta = (1/2n) sum_ij W_ij dK_ij/dtheta with dK/dtheta from autograd of kernel_dense."""
    dt = y.dtype
    n = y.shape[-1]
    rawg = raw.detach().clone().requires_grad_(True)
    theta = constrain(rawg, kinds, lb, ub)
    mean, w, mu, sigma, noise = unpack_params(theta, spec)
    K = kernel_dense(x, x, theta, spec)
    Kt = K + torch.diag_embed(noise_diag(n, fixed_noise, noise, dt))
    if jitter is None:
        jitter = default_jitter(dt)
    L, info = psd_safe_cholesky(Kt.detach(), jitter=jitter)
    if int(info) < 0:
        nanv = torch.full((), float("nan"), dtype=dt)
        return nanv, torch.full_like(raw, float("nan")), info
    if int(info) > 0:
        Kt = Kt + jitter_rung(info, jitter) * torch.eye(n, dtype=dt)
    r = (y - mean.detach()).unsqueeze(-1)
    alpha = torch.cholesky_solve(r, L)
    Kinv = torch.cholesky_inverse(L)
    mll = -0.5 * ((r * alpha).sum() + 2.0 * torch.log(torch.diagonal(L)).sum()
                  + n * math.log(TWO_PI)) / n
    W = (alpha @ alpha.T - Kinv).detach()
    surrogate = (0.5 / n) * (W * Kt).sum() + (alpha.detach().sum() / n) * mean
    (g,) = torch.autograd.grad(surrogate, rawg)
    return mll.detach(), g.detach(), info


# ---------------------------------------------------------------------------------------
# N1: posterior prediction (GPyTorch ExactGP eval mode: ExactPredictionStrategy, exact form)
# ---------------------------------------------------------------------------------------
def predict(x, y, fixed_noise, raw, kinds, lb, ub, spec: ModelSpec, xstar, jitter=None):
    """Posterior mean and LATENT variance at xstar [m, d] (what ``model(x*)`` returns in eval
    mode, pgmuvi/lightcurve.py:9862; the likelihood then adds its homoskedastic noise):
        mean* = c + K*^T Kt^-1 (y - c),   var* = k** - K*^T Kt^-1 K*      (Cholesky solves).
    The reference computes the variance under ``fast_pred_var`` (LOVE, approximate,
    lightcurve.py:9607); this is the exact quantity it approximates."""
    n = y.shape[-1]
    theta = constrain(raw, kinds, lb, ub)
    mean, w, mu, sigma, noise = unpack_params(theta, spec)
    Kt = kernel_dense(x, x, theta, spec) + torch.diag_embed(noise_diag(n, fixed_noise, noise, y.dtype))
    L, info = psd_safe_cholesky(Kt, jitter=jitter)
    Ks = kernel_dense(x, xstar, theta, spec)                    # [n, m]
    alpha = torch.cholesky_solve((y - mean).unsqueeze(-1), L)
    v = torch.linalg.solve_triangular(L, Ks, upper=False)
    kss = torch.diagonal(kernel_dense(xstar, xstar, theta, spec))
    return mean + (Ks.T @ alpha).squeeze(-1), kss - (v * v).sum(0), info


# ---------------------------------------------------------------------------------------
# batched CPU baseline (torch batch mode; same op sequence, autograd) - BASELINE.md section 3
# ---------------------------------------------------------------------------------------
def batched_mll_and_grad(x, y, fixed_noise, raw, kinds, lb, ub, spec: ModelSpec):
    """x [B,n,d], y [B,n], fixed_noise [B,n] or None, raw/lb/ub [B,P].  No jitter ladder
    (used for timing and for well-conditioned parity cases).  Returns (mll [B], grad [B,P])."""
    raw = raw.detach().clone().requires_grad_(True)
    theta = constrain(raw, kinds, lb, ub)
    mean, w, mu, sigma, noise = unpack_params(theta, spec)
    n = y.shape[-1]
    K = kernel_dense(x, x, theta, spec)
    dvec = torch.zeros_like(y)
    if fixed_noise is not None:
        dvec = dvec + fixed_noise
    if noise is not None:
        dvec = dvec + noise.unsqueeze(-1)
    Kt = K + torch.diag_embed(dvec)
    L = torch.linalg.cholesky(Kt)
    r = (y - mean.unsqueeze(-1)).unsqueeze(-1)
    z = torch.linalg.solve_triangular(L, r, upper=False)
    inv_quad = (z * z).sum((-2, -1))
    logdet = 2.0 * torch.log(torch.diagonal(L, dim1=-2, dim2=-1)).sum(-1)
    mll = -0.5 * (inv_quad + logdet + n * math.log(TWO_PI)) / n
    (g,) = torch.autograd.grad(mll.sum(), raw)
    return mll.detach(), g


# ---------------------------------------------------------------------------------------
# optimisers (A.7: torch.optim defaults as used at trainers.py:141-147)
# ---------------------------------------------------------------------------------------
def adam_step(p, g, m, v, step, lr, b1=0.9, b2=0.999, eps=1e-8, weight_decay=0.0,
              decoupled=False):
    """One Adam (decoupled=False, wd added to grad) / AdamW (decoupled=True) step, torch
    semantics.  ``g`` is the gradient of the LOSS (= -MLL).  step counts from 1.
    Works on numpy arrays or torch tensors; returns (p, m, v)."""
    if decoupled:
        p = p * (1.0 - lr * weight_decay)
    elif weight_decay != 0.0:
        g = g + weight_decay * p
    m = b1 * m + (1 - b1) * g
    v = b2 * v + (1 - b2) * g * g
    bc1 = 1 - b1 ** step
    bc2 = 1 - b2 ** step
    denom = (v ** 0.5) / math.sqrt(bc2) + eps
    p = p - (lr / bc1) * (m / denom)
    return p, m, v


def train_loop(x, y, fixed_noise, raw0, kinds, lb, ub, spec: ModelSpec, maxiter=100,
               miniter=10, stop=None, lr=1e-4, optim="SGD", eps=1e-8, stopavg=9,
               use_torch_optim=True, jitter=None, on_failure="raise"):
    """trainers.py:167-209 restated for one light curve on packed raw parameters.

    Returns dict(loss=[...], delta_loss=[...], raw=[P-vectors, initial first]).  The loss
    recorded at iteration i is evaluated BEFORE that iteration's step (trainers.py:179-188);
    parameters are recorded AFTER it (trainers.py:190-192).

    `jitter`: first rung of the Cholesky's jitter ladder (psd_safe_cholesky).
    on_failure="raise" raises when an evaluation's Cholesky fails, as the reference does;
    on_failure="stop" ends the loop there instead, the rule of the engine's fit kernel: the failed
    evaluation's loss (NaN) is recorded and no step is taken.  The result then also has
    info=[per-iteration Cholesky info].
    """
    if on_failure not in ("raise", "stop"):
        raise ValueError("on_failure must be 'raise' or 'stop'")
    raw = raw0.detach().clone().requires_grad_(True)
    if optim == "SGD":
        opt = torch.optim.SGD([raw], lr=lr)
    elif optim == "Adam":
        opt = torch.optim.Adam([raw], lr=lr, eps=eps)
    elif optim == "AdamW":
        opt = torch.optim.AdamW([raw], lr=lr, eps=eps)
    else:
        raise ValueError("optim must be 'SGD', 'Adam' or 'AdamW'")
    res = {"loss": [], "delta_loss": [], "raw": [raw.detach().clone().numpy()]}
    if on_failure == "stop":
        res["info"] = []
    for i in range(maxiter):
        opt.zero_grad()
        theta = constrain(raw, kinds, lb, ub)
        mll, info = _mll_from_theta(x, y, fixed_noise, theta, spec, jitter)
        if on_failure == "stop":
            res["info"].append(int(info))
        if int(info) < 0:
            if on_failure == "stop":
                res["loss"].append(np.array(float("nan")))
                break
            raise RuntimeError(f"Cholesky failed (info={int(info)}) at iteration {i}")
        loss = -mll
        loss.backward()
        opt.step()
        lv = loss.detach().numpy()
        if i > 0:
            res["delta_loss"].append(lv - res["loss"][-1])
        res["loss"].append(lv)
        res["raw"].append(raw.detach().clone().numpy())
        if stop and i > miniter:
            if np.std(res["loss"][-stopavg:]) < stop:
                break
    return res
