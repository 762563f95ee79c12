"""Fisher information of the exact Gaussian log-likelihood (standard errors of fitted parameters),
without a GPU: the fp64 oracle against an independent route (the Hessian of the Gaussian KL
divergence), the host assembly of ``Lightcurve.parameter_uncertainties`` driven by oracle Fisher
matrices, and the argument checks of ``pgm_sm_fisher_f64``."""
import warnings

import numpy as np
import pytest
import torch

from oracle import ModelSpec, constrain
from oracle.fisher import fisher, fisher_from_kl
from oracle.sm_gp import stat_kind
from pgmuvi_b200 import _lib, mll, ops
from pgmuvi_b200.lightcurve import Lightcurve
from pgmuvi_b200.mll import UnsupportedModelError, pack_model


def _theta(spec, rng, zero_mu_last=False):
    th = [0.3]
    th += list(rng.uniform(0.5, 1.5, spec.Q))                       # weights
    mu = rng.uniform(0.05, 0.4, spec.Q * spec.ds)
    if zero_mu_last:
        mu[-spec.ds:] = 0.0
    th += list(mu)
    th += list(rng.uniform(0.02, 0.1, spec.Q * spec.ds))            # frequency scales
    if spec.learn_noise:
        th.append(0.05)
    th += list(rng.uniform(0.6, 2.0, spec.NL))
    return torch.tensor(th, dtype=torch.float64)


def _inputs(d, n, rng):
    t = np.sort(rng.uniform(0.0, 30.0, n))
    if d == 1:
        return torch.tensor(t).unsqueeze(-1)
    wl = rng.integers(0, 3, n) * 0.7 + 0.5
    return torch.tensor(np.stack([t, wl], 1))


CASES = {
    "sm1d": (ModelSpec(d=1, Q=3, kind=_lib.KIND_SM1D), False),
    "ard2d_prodsum": (ModelSpec(d=2, Q=2, kind=_lib.KIND_SM_ARD_PRODSUM), False),
    "ard2d_sumprod": (ModelSpec(d=2, Q=2, kind=_lib.KIND_SM_ARD_SUMPROD), False),
    "sep_rq": (ModelSpec(d=2, Q=2, kind=_lib.KIND_SEP_RQ), False),
    "quasi_periodic": (ModelSpec(d=1, Q=0, kind=stat_kind(2, 0)), False),
    "learned_noise": (ModelSpec(d=1, Q=2, kind=_lib.KIND_SM1D, learn_noise=True), False),
    "flicker": (ModelSpec(d=2, Q=3, kind=_lib.KIND_SEP_RBF), True),
}


@pytest.mark.parametrize("case", sorted(CASES))
def test_oracle_fisher_is_the_hessian_of_the_gaussian_kl(case):
    spec, zero_mu = CASES[case]
    rng = np.random.default_rng(7)
    x = _inputs(spec.d, 14, rng)
    fn = None if spec.learn_noise else torch.full((14,), 0.02, dtype=torch.float64)
    theta = _theta(spec, rng, zero_mu)
    F, info = fisher(x, fn, theta, spec)
    assert info == 0
    H = fisher_from_kl(x, fn, theta, spec)
    sd = F.diagonal().clamp_min(1e-300).sqrt()
    err = (F - H).abs() / (sd[:, None] * sd[None, :])
    nz = F.diagonal() > 0
    assert float(err[nz][:, nz].max()) <= 1e-10
    # slots without a derivative (the flicker term's zero mean frequency) are exactly 0
    assert torch.equal(F[~nz], torch.zeros_like(F[~nz]))
    assert float(F[0, 1:].abs().max()) == 0.0


def test_oracle_fisher_includes_the_jitter_rung_and_reports_failures():
    spec = ModelSpec(d=1, Q=1, kind=_lib.KIND_SM1D)
    x = torch.linspace(0, 1, 10, dtype=torch.float64).unsqueeze(-1)
    x[1] = x[0]                                   # duplicated input, no noise: singular K
    theta = torch.tensor([0.0, 1.0, 0.01, 0.01], dtype=torch.float64)
    F, info = fisher(x, None, theta, spec)
    assert info >= 1 and torch.isfinite(F).all()
    H = fisher_from_kl(x, None, theta, spec, jitter_add=1e-8 * 10 ** (info - 1))
    sd = F.diagonal().sqrt()
    # K~ + jitter has a condition number near 1e8 here: agreement to that conditioning
    assert float(((F - H).abs() / (sd[:, None] * sd[None, :])).max()) <= 1e-4
    x[3, 0] = float("nan")
    F, info = fisher(x, None, theta, spec)
    assert info == -1 and torch.isnan(F).all()


# ---- host assembly ----------------------------------------------------------------------------
def fake_sm_fisher(x, y, fixed_noise, raw, kinds, lb, ub, n_valid, kind, Q, learn_noise):
    """Oracle stand-in with pgm_sm_fisher_f64's contract."""
    B, P = raw.shape
    spec = ModelSpec(d=x.shape[-1], Q=Q, kind=kind, learn_noise=learn_noise)
    out = torch.empty(B, P, P, dtype=torch.float64)
    info = torch.zeros(B, dtype=torch.int32)
    for b in range(B):
        n = x.shape[1] if n_valid is None else int(n_valid[b])
        theta = constrain(raw[b], kinds, lb[b] if lb.dim() == 2 else lb, ub[b] if ub.dim() == 2 else ub)
        out[b], info[b] = fisher(x[b, :n], None if fixed_noise is None else fixed_noise[b, :n],
                                 theta, spec)
    return out, info


@pytest.fixture
def oracle_engine(monkeypatch):
    monkeypatch.setattr(ops, "sm_fisher", fake_sm_fisher)
    monkeypatch.setattr(mll, "engine_device", lambda t=None: torch.device("cpu"))


def _lc(n=40, seed=0, yerr=True, **kw):
    rng = np.random.default_rng(seed)
    t = np.sort(rng.uniform(2450000.0, 2450300.0, n))
    y = 3.0 + np.sin(2 * np.pi * t / 47.0) + 0.2 * rng.standard_normal(n)
    kw.setdefault("xtransform", "minmax")
    lc = Lightcurve(t, y, yerr=np.full(n, 0.2) if yerr else None, **kw).double()
    return lc


def _setup(lc, model="1D", likelihood=None, **kw):
    lc.set_model(model, likelihood, **kw)
    lc.set_default_constraints()
    lc.model.double()          # float64 parameters: finite differences below resolve 1e-6 steps
    return lc


def _fd_stderr(lc, res, h=1e-6):
    """stderr of every get_parameters() entry by central differences in the raw parameters."""
    pk = pack_model(lc.model, lc.likelihood)
    raw0 = pk.raw().detach().clone()
    th = lambda r: constrain(r, pk.kinds, pk.lb, pk.ub)
    base = lc.get_parameters()
    J = {k: torch.zeros(v.numel(), pk.P, dtype=torch.float64) for k, v in base.items()}
    for s in range(pk.P):
        if res["covariance"][s, s] == 0:
            continue
        vals = []
        for sgn in (1, -1):
            r = raw0.clone()
            r[s] += sgn * h
            pk.scatter_raw_(r)
            vals.append(lc.get_parameters())
        dth = float(th(raw0 + h * torch.eye(pk.P, dtype=torch.float64)[s])[s]
                    - th(raw0 - h * torch.eye(pk.P, dtype=torch.float64)[s])[s])
        for k in base:
            J[k][:, s] = (vals[0][k] - vals[1][k]).reshape(-1).double() / dth
    pk.scatter_raw_(raw0)
    C = res["covariance"]
    return {k: torch.einsum("ij,jk,ik->i", J[k], C, J[k]).sqrt().reshape(base[k].shape) for k in J}


@pytest.mark.parametrize("model,likelihood,ytr", [("1D", None, None), ("1D", "learn", "zscore"),
                                                  ("1DQuasiPeriodic", None, None)])
def test_host_assembly_matches_finite_differences_of_get_parameters(oracle_engine, model,
                                                                    likelihood, ytr):
    lc = _lc(ytransform=ytr)
    _setup(lc, model, likelihood, **({} if model.startswith("1DQ") else {"num_mixtures": 2}))
    res = lc.parameter_uncertainties()
    assert res["fisher_ok"] and res["info"] == 0
    pk = pack_model(lc.model, lc.likelihood)
    assert len(res["names"]) == pk.P
    # covariance = inverse Fisher over the free slots
    F = res["fisher"]
    free = res["covariance"].diagonal() != 0
    eye = res["covariance"][free][:, free] @ F[free][:, free]
    assert torch.allclose(eye, torch.eye(int(free.sum()), dtype=torch.float64), atol=1e-8)
    fd = _fd_stderr(lc, res)
    pars = lc.get_parameters()
    assert set(res["stderr"]) == set(pars)
    for k, v in pars.items():
        assert res["stderr"][k].shape == v.shape
        np.testing.assert_allclose(res["stderr"][k].numpy(), fd[k].numpy(), rtol=1e-5, atol=1e-12)
    if model == "1D":
        mu = pars["covar_module.mixture_means"].double()
        np.testing.assert_allclose(res["period_stderr"],
                                   (res["stderr"]["covar_module.mixture_means"][:, 0, 0]
                                    / mu[:, 0, 0] ** 2).numpy(), rtol=1e-12)
        assert (res["period_stderr"] > 0).all()
    else:
        assert res["period_stderr"] is None


def test_frozen_slots_get_zero(oracle_engine, monkeypatch):
    """The flicker term's mean frequency is an Interval(0, 0) slot that is not a Parameter.  A ridge
    keeps the Fisher matrix of the default-initialised model positive definite on the free slots."""
    def ridged(*a):
        F, info = fake_sm_fisher(*a)
        return F + torch.eye(F.shape[-1], dtype=F.dtype), info
    monkeypatch.setattr(ops, "sm_fisher", ridged)
    rng = np.random.default_rng(2)
    n = 36
    x = np.stack([np.sort(rng.uniform(0, 60, n)), rng.integers(0, 3, n) * 0.5 + 0.5], 1)
    y = np.sin(x[:, 0] / 5.0) + 0.1 * rng.standard_normal(n)
    lc = Lightcurve(x, y, yerr=np.full(n, 0.1), xtransform="minmax").double()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        _setup(lc, "2DWavelengthDependent", time_kernel_type="sm", num_mixtures=2,
               add_flicker=True, mean_module="constant")
    pk = pack_model(lc.model, lc.likelihood)
    frozen = [s for s in range(pk.P) if float(pk.lb[s]) == float(pk.ub[s]) and
              int(pk.kinds[s]) == _lib.CON_INTERVAL]
    assert frozen
    res = lc.parameter_uncertainties()
    assert res["fisher_ok"]
    C = res["covariance"]
    for s in frozen:
        assert float(C[s].abs().max()) == 0.0 and float(C[:, s].abs().max()) == 0.0
    assert all(torch.isfinite(v).all() for v in res["stderr"].values())


def test_singular_fisher_gives_nan_and_a_flag(oracle_engine, monkeypatch):
    def singular(*a):
        F, info = fake_sm_fisher(*a)
        F[:, 2, :] = F[:, 1, :]
        F[:, :, 2] = F[:, :, 1]
        return F, info
    monkeypatch.setattr(ops, "sm_fisher", singular)
    lc = _setup(_lc(), "1D", num_mixtures=2)
    res = lc.parameter_uncertainties()
    assert not res["fisher_ok"]
    assert all(torch.isnan(v).all() for k, v in res["stderr"].items() if "mixture" in k)
    assert np.isnan(res["period_stderr"]).all()


def test_batch_equals_one_by_one_and_chunks(oracle_engine):
    from pgmuvi_b200.batch import uncertainties_batch
    lcs = [_setup(_lc(n=n, seed=s), "1D", num_mixtures=2) for s, n in enumerate((30, 41, 25))]
    one = [lc.parameter_uncertainties() for lc in lcs]
    many = uncertainties_batch(lcs, budget_bytes=1)        # one light curve per chunk
    for a, b in zip(one, many):
        assert torch.equal(a["covariance"], b["covariance"])
        for k in a["stderr"]:
            assert torch.equal(a["stderr"][k], b["stderr"][k])


def test_non_constant_means_are_rejected(oracle_engine):
    lc = _setup(_lc(), "1DLinear", num_mixtures=2)
    with pytest.raises(UnsupportedModelError):
        lc.parameter_uncertainties()


# ---- C ABI -------------------------------------------------------------------------------------
def test_fisher_abi_checks_arguments_before_any_launch():
    lib = _lib.load()
    one = 8     # any non-null fake pointer: validation fails before it is dereferenced
    need = lib.pgm_fisher_workspace_bytes(512, 4, 1, 4, _lib.KIND_SM1D, 0)
    assert need > lib.pgm_staged_workspace_bytes(512, 4)
    # 12 carriers x (N^2 + ntri) tiles per light curve (N = 8)
    assert need >= 4 * 12 * (64 + 36) * 4096 * 8
    assert lib.pgm_fisher_workspace_bytes(512, 4, 1, 9, _lib.KIND_SM1D, 0) == 0
    args = lambda B, n, d, Q, ws: (one, None, one, None, one, one, one, one, B, n, d, Q,
                                   _lib.KIND_SM1D, 0, one, one, one, ws, None)
    assert lib.pgm_sm_fisher_f64(*args(4, 512, 1, 4, need - 1)) == -1
    assert b"workspace" in lib.pgm_last_error()
    assert lib.pgm_sm_fisher_f64(*args(4, 512, 2, 4, need)) == -1
    assert b"d == 1" in lib.pgm_last_error()
    assert lib.pgm_sm_fisher_f64(*args(4, 512, 1, 0, need)) == -1
    assert b"Q" in lib.pgm_last_error()
    assert lib.pgm_sm_fisher_f64(*args(70000, 64, 1, 4, 1 << 62)) == -1
    assert b"65535" in lib.pgm_last_error()
    a = list(args(4, 512, 1, 4, need))
    a[14] = None                                   # fisher output
    assert lib.pgm_sm_fisher_f64(*a) == -1 and b"null" in lib.pgm_last_error()
    assert lib.pgm_sm_fisher_f64(*args(0, 512, 1, 4, 0)) == 0


def test_sm_fisher_refuses_cpu_tensors():
    x = torch.zeros(1, 8, 1, dtype=torch.float64)
    y = torch.zeros(1, 8, dtype=torch.float64)
    raw = torch.zeros(1, 13, dtype=torch.float64)
    k = torch.ones(13, dtype=torch.int32)
    b = torch.zeros(13, dtype=torch.float64)
    with pytest.raises((RuntimeError, NotImplementedError)):
        ops.sm_fisher(x, y, None, raw, k, b, b, None, 0, 4, False)
