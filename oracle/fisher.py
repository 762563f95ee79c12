"""fp64 torch-CPU restatement of the expected (Fisher) information of the exact Gaussian
log-likelihood l(theta) = log p(y | theta) in the constrained packed parameters theta
(pgm_sm_fisher_f64, include/pgmuvi_b200.h):

    I_pq = 1/2 tr(K~^-1 dK~_p K~^-1 dK~_q),   I_00 = 1^T K~^-1 1,   I_0p = 0,

K~ = kernel_dense + noise_diag (+ the jitter rung the Cholesky needed), dK~ by autograd."""
from __future__ import annotations

import torch

from .sm_gp import (ModelSpec, default_jitter, jitter_rung, kernel_dense, noise_diag,
                    psd_safe_cholesky, unpack_params)


def covariance(x, fixed_noise, theta, spec: ModelSpec):
    """K~(theta) without jitter: x [n, d], theta [P] constrained."""
    n = x.shape[0]
    noise = unpack_params(theta, spec)[4]
    return kernel_dense(x, x, theta, spec) + torch.diag_embed(
        noise_diag(n, fixed_noise, noise, theta.dtype))


def fisher(x, fixed_noise, theta, spec: ModelSpec, jitter=None):
    """(I [P, P], info) of one light curve; I is NaN when the Cholesky fails (info < 0)."""
    theta = theta.detach().to(torch.float64)
    x = x.to(torch.float64)
    fixed_noise = None if fixed_noise is None else fixed_noise.to(torch.float64)
    n, P = x.shape[0], theta.shape[0]
    Kt = covariance(x, fixed_noise, theta, spec)
    L, info = psd_safe_cholesky(Kt, jitter=jitter)
    if int(info) < 0:
        return torch.full((P, P), float("nan"), dtype=torch.float64), int(info)
    dK = torch.autograd.functional.jacobian(lambda th: covariance(x, fixed_noise, th, spec), theta,
                                            vectorize=True, strategy="forward-mode")
    Kinv = torch.cholesky_inverse(L)
    A = torch.einsum("ij,jkp->ikp", Kinv, dK)
    F = 0.5 * torch.einsum("ijp,jiq->pq", A, A)
    F[0, 0] = Kinv.sum()
    return 0.5 * (F + F.T), int(info)


def gaussian_kl(m0, K0, m1, K1):
    """KL(N(m0, K0) || N(m1, K1)) in closed form."""
    n = K0.shape[0]
    L1 = torch.linalg.cholesky(K1)
    dm = (m1 - m0).unsqueeze(-1)
    z = torch.linalg.solve_triangular(L1, dm, upper=False)
    tr = torch.cholesky_solve(K0, L1).diagonal().sum()
    logdet1 = 2.0 * torch.log(torch.diagonal(L1)).sum()
    logdet0 = torch.linalg.slogdet(K0)[1]
    return 0.5 * (tr + (z * z).sum() - n + logdet1 - logdet0)


def fisher_from_kl(x, fixed_noise, theta0, spec: ModelSpec, jitter_add=0.0):
    """Independent route: the Hessian at theta0 of KL(N(c0 1, K~(theta0)) || N(c 1, K~(theta)))."""
    theta0 = theta0.detach().to(torch.float64)
    x = x.to(torch.float64)
    n = x.shape[0]
    eye = torch.eye(n, dtype=torch.float64)
    K0 = covariance(x, fixed_noise, theta0, spec) + jitter_add * eye
    m0 = theta0[0] * torch.ones(n, dtype=torch.float64)

    def kl(th):
        return gaussian_kl(m0, K0, th[0] * torch.ones(n, dtype=torch.float64),
                           covariance(x, fixed_noise, th, spec) + jitter_add * eye)

    return torch.autograd.functional.hessian(kl, theta0)


def jitter_of(info, dtype=torch.float64):
    """Diagonal jitter of Cholesky rung `info` (0 = none)."""
    return 0.0 if int(info) <= 0 else jitter_rung(info, default_jitter(dtype))
