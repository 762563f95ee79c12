"""GPU parity tests: the CUDA path (through the C ABI) against the oracle's golden vectors,
against the oracle itself on seeded inputs, and - at BASELINE.json's full C2 size - through
size-independent properties.  Tolerances are the north star's: MLL and gradients within
1e-6 relative in fp64 (we assert 1e-9, leaving head-room for the 1e-6 bar)."""
import math

import numpy as np
import pytest
import torch

from conftest import golden_names, load_golden

pytestmark = pytest.mark.gpu

RTOL = 1e-9      # asserted; the contract is 1e-6 relative in fp64
K_ATOL = 1e-13   # kernel entries vs oracle (SURVEY.md section 7 acceptance)


def _dev(g, dev):
    t = lambda a, dt=torch.float64: None if a is None else torch.tensor(a, dtype=dt, device=dev)
    return dict(x=t(g["x"]), y=t(g["y"]), noise=t(g["noise"]), raw=t(g["raw"]),
                kinds=t(g["kinds"], torch.int32), lb=t(g["lb"]), ub=t(g["ub"]),
                n_valid=t(g["n_valid"], torch.int32))


def _eval(ops, g, d, want_grad=True, raw=None):
    return ops.sm_mll_grad(d["x"], d["y"], d["noise"], d["raw"] if raw is None else raw,
                           d["kinds"], d["lb"], d["ub"], d["n_valid"], g["kind"], g["Q"],
                           g["learn_noise"], want_grad)


@pytest.mark.parametrize("name", golden_names())
def test_mll_and_grad_match_goldens(name, cuda_device):
    from pgmuvi_b200 import ops
    g = load_golden(name)
    d = _dev(g, cuda_device)
    mll, grad, info = _eval(ops, g, d)
    mll, grad, info = mll.cpu().numpy(), grad.cpu().numpy(), info.cpu().numpy()
    assert np.array_equal(info, g["info"])
    assert np.abs(mll - g["mll"]).max() <= RTOL * np.abs(g["mll"]).max()
    for b in range(len(mll)):
        scale = np.abs(g["grad_autograd"][b]).max()
        assert np.abs(grad[b] - g["grad_autograd"][b]).max() <= RTOL * 100 * scale
    # MLL-only entry gives the same value
    mll2, _, _ = _eval(ops, g, d, want_grad=False)
    assert np.array_equal(mll2.cpu().numpy(), mll)


@pytest.mark.parametrize("name", golden_names())
def test_kernel_builder_matches_goldens(name, cuda_device):
    from pgmuvi_b200 import ops
    g = load_golden(name)
    d = _dev(g, cuda_device)
    K = ops.sm_kernel_dense(d["x"], d["noise"], d["raw"], d["kinds"], d["lb"], d["ub"],
                            d["n_valid"], g["kind"], g["Q"], g["learn_noise"]).cpu().numpy()
    n = g["x"].shape[1]
    for b in range(K.shape[0]):
        nb = n if g["n_valid"] is None else int(g["n_valid"][b])
        ii = np.minimum(g["k_index"], nb - 1)
        assert np.abs(K[b][np.ix_(ii, ii)] - g["k_sample"][b]).max() <= K_ATOL * max(
            1.0, np.abs(g["k_sample"][b]).max())
        assert np.array_equal(K[b][:nb, :nb], K[b][:nb, :nb].T)   # bitwise symmetric builder


@pytest.mark.parametrize("name", ["sm1d_n100_q2_learn", "sm1d_n200_q4", "sm2d_prodsum_4x48_q4",
                                  "sm1d_ragged_q4", "sm2d_prodsum_3x64_q8",
                                  "sm2d_sumprod_3x64_q6_learn"])
def test_fused_fit_kernel_matches_oracle_adamw_steps(name, cuda_device):
    """pgm_sm_fit (whole loop on device) vs trainers.train restated in the oracle: loss
    before each step and raw parameters after each step (AdamW, lr 0.1, torch defaults)."""
    from pgmuvi_b200 import ops, _lib
    g = load_golden(name)
    d = _dev(g, cuda_device)
    raw = d["raw"].clone()
    loss, raw_hist, n_iter, info = ops.sm_fit(
        d["x"], d["y"], d["noise"], raw, d["kinds"], d["lb"], d["ub"], d["n_valid"], g["kind"],
        g["Q"], g["learn_noise"], _lib.OPT_ADAMW, 0.1, 0.9, 0.999, 1e-8, 0.01, 3, 3, 0.0, 9, True)
    assert n_iter.cpu().tolist() == [3] * raw.shape[0]
    assert np.abs(loss.cpu().numpy().T - g["adamw_loss"]).max() <= 1e-9
    got = raw_hist.cpu().numpy().transpose(1, 0, 2)
    assert np.abs(got - g["adamw_raw"]).max() <= 1e-8
    assert np.array_equal(raw.cpu().numpy(), got[:, -1])


def test_optim_step_kernel_matches_torch_optim(cuda_device):
    from pgmuvi_b200 import ops, _lib
    gen = torch.Generator().manual_seed(3)
    for kind, mk in ((_lib.OPT_SGD, lambda p: torch.optim.SGD([p], lr=0.05)),
                     (_lib.OPT_ADAM, lambda p: torch.optim.Adam([p], lr=0.05, eps=1e-8)),
                     (_lib.OPT_ADAMW, lambda p: torch.optim.AdamW([p], lr=0.05, eps=1e-8))):
        p0 = torch.randn(5, 13, generator=gen, dtype=torch.float64)
        pref = p0.clone().requires_grad_(True)
        opt = mk(pref)
        raw = p0.to(cuda_device)
        m, v = torch.zeros_like(raw), torch.zeros_like(raw)
        wd = 0.01 if kind == _lib.OPT_ADAMW else 0.0
        for step in range(1, 6):
            grad_mll = torch.cos(pref.detach() * step)          # d mll / d raw
            pref.grad = -grad_mll.clone()                       # loss = -mll
            opt.step()
            ops.optim_step(raw, grad_mll.to(cuda_device), m, v, None, kind, 0.05, 0.9, 0.999,
                           1e-8, wd, step)
            assert np.abs(raw.cpu().numpy() - pref.detach().numpy()).max() <= 1e-13
        # masked light curves do not move
        active = torch.tensor([1, 0, 1, 0, 1], dtype=torch.int32, device=cuda_device)
        before = raw.clone()
        ops.optim_step(raw, torch.ones_like(raw), m, v, active, kind, 0.05, 0.9, 0.999, 1e-8,
                       wd, 6)
        assert torch.equal(raw[1], before[1]) and not torch.equal(raw[0], before[0])


def test_against_oracle_on_fresh_seeds(cuda_device):
    """Seeded inputs that are NOT in the golden set, evaluated by the oracle on the host."""
    from oracle import ModelSpec, mll_and_grad_analytic
    from pgmuvi_b200 import ops, synthetic as S
    torch.set_default_dtype(torch.float64)
    for (n, Q, ln) in ((89, 2, False), (225, 3, True), (400, 1, True)):
        bt = S.make_batch_1d(2, n, Q=Q, learn_noise=ln, seed0=777)
        g = dict(bt, kind=0, n_valid=None)
        d = _dev(g, cuda_device)
        mll, grad, info = _eval(ops, g, d)
        spec = ModelSpec(d=1, Q=Q, kind=0, learn_noise=ln)
        for b in range(2):
            c = lambda a: torch.tensor(a[b])
            mo, go, io = mll_and_grad_analytic(c(bt["x"]), c(bt["y"]), c(bt["noise"]),
                                               c(bt["raw"]), torch.tensor(bt["kinds"]),
                                               c(bt["lb"]), c(bt["ub"]), spec)
            assert abs(float(mll[b]) - float(mo)) <= RTOL * abs(float(mo))
            assert float((grad[b].cpu() - go).abs().max()) <= RTOL * 100 * float(go.abs().max())


def test_jitter_ladder_and_failure_codes(cuda_device):
    """info semantics (SURVEY.md A.5): duplicate time stamps with ~zero noise are singular ->
    jitter rescues them; a negative 'variance' is not PD even after 3 tries; NaN in the
    covariance -> -1 (NanError); NaN only in y leaves the factorisation fine (info 0) and
    gives a NaN loss, exactly as torch does."""
    from oracle import ModelSpec, mll_and_grad_analytic
    from pgmuvi_b200 import ops, synthetic as S
    bt = S.make_batch_1d(5, 96, Q=2, seed0=4242)
    bt["x"][1, 50, 0] = bt["x"][1, 49, 0]          # duplicated epoch ...
    bt["noise"][1, :] = 1e-17                       # ... with (almost) no noise: singular
    bt["noise"][2, 10] = -50.0                      # hopeless
    bt["x"][3, 5, 0] = float("nan")
    bt["y"][4, 5] = float("nan")
    g = dict(bt, kind=0, n_valid=None)
    d = _dev(g, cuda_device)
    mll, grad, info = _eval(ops, g, d)
    info = info.cpu().tolist()
    assert info[0] == 0 and info[2] == -2 and info[3] == -1 and info[4] == 0
    assert torch.isnan(mll[2]) and torch.isnan(mll[3]) and torch.isnan(grad[2]).all()
    assert torch.isnan(mll[4]) and torch.isfinite(mll[0])
    spec = ModelSpec(d=1, Q=2)
    c = lambda a: torch.tensor(a[1], dtype=torch.float64)
    mo, go, io = mll_and_grad_analytic(c(bt["x"]), c(bt["y"]), c(bt["noise"]), c(bt["raw"]),
                                       torch.tensor(bt["kinds"]), c(bt["lb"]), c(bt["ub"]), spec)
    assert int(io) >= 1 and info[1] >= 1       # both needed jitter
    if info[1] == int(io):                     # same rung -> same numbers (ill-conditioned: 1e-4)
        assert abs(float(mll[1]) - float(mo)) <= 1e-4 * abs(float(mo))


def test_empty_and_tiny_inputs(cuda_device):
    from pgmuvi_b200 import ops, synthetic as S
    bt = S.make_batch_1d(2, 8, Q=1, seed0=99)
    g = dict(bt, kind=0, n_valid=None)
    d = _dev(g, cuda_device)
    mll, grad, info = _eval(ops, g, d)
    assert torch.isfinite(mll).all() and torch.isfinite(grad).all()
    e = lambda *s: torch.zeros(*s, dtype=torch.float64, device=cuda_device)
    m0, g0, i0 = ops.sm_mll_grad(e(0, 8, 1), e(0, 8), None, e(0, 4), d["kinds"], e(4), e(4),
                                 None, 0, 1, False, True)
    assert m0.numel() == 0 and g0.shape == (0, 4)


# ---------------------------------------------------------------------------------------
# BASELINE.json C2 at full size (4096 x n=512, SM-4): size-independent properties
# ---------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def c2(cuda_device):
    from pgmuvi_b200 import synthetic as S
    bt = S.make_batch_1d(256, 512, Q=4)
    rep = 16                                        # 4096 = 16 x 256 distinct light curves
    g = {k: (np.concatenate([bt[k]] * rep, 0) if k in ("x", "y", "noise", "raw", "lb", "ub")
             else bt[k]) for k in bt}
    g.update(kind=0, n_valid=None)
    return g, _dev(g, cuda_device)


def test_c2_full_size_replicas_agree_bitwise(c2):
    from pgmuvi_b200 import ops
    g, d = c2
    mll, grad, info = _eval(ops, g, d)
    assert int((info != 0).sum()) == 0
    m = mll.view(16, 256)
    gr = grad.view(16, 256, -1)
    assert torch.equal(m, m[0:1].expand_as(m))      # every block computes the same bits
    assert torch.equal(gr, gr[0:1].expand_as(gr))


def test_c2_full_size_time_shift_and_permutation_invariance(c2, cuda_device):
    from pgmuvi_b200 import ops
    g, d = c2
    mll, grad, _ = _eval(ops, g, d)
    d2 = dict(d)
    d2["x"] = d["x"] + 0.375                         # stationary kernel: MLL unchanged
    mll_s, grad_s, _ = _eval(ops, g, d2)
    assert (mll_s - mll).abs().max() <= 1e-10 * mll.abs().max()
    assert (grad_s - grad).abs().max() <= 1e-8 * grad.abs().max()
    perm = torch.randperm(512, generator=torch.Generator().manual_seed(0)).to(cuda_device)
    d3 = dict(d, x=d["x"][:, perm].contiguous(), y=d["y"][:, perm].contiguous(),
              noise=d["noise"][:, perm].contiguous())
    mll_p, grad_p, _ = _eval(ops, g, d3)
    assert (mll_p - mll).abs().max() <= 1e-10 * mll.abs().max()
    assert (grad_p - grad).abs().max() <= 1e-8 * grad.abs().max()


def test_c2_full_size_gradient_is_the_derivative_of_the_mll(c2):
    """Central finite difference of the kernel's own MLL along a random direction."""
    from pgmuvi_b200 import ops
    g, d = c2
    _, grad, _ = _eval(ops, g, d)
    gen = torch.Generator().manual_seed(5)
    v = torch.randn(d["raw"].shape, generator=gen, dtype=torch.float64).to(d["raw"].device)
    h = 1e-5
    mp, _, _ = _eval(ops, g, d, want_grad=False, raw=d["raw"] + h * v)
    mm, _, _ = _eval(ops, g, d, want_grad=False, raw=d["raw"] - h * v)
    fd = (mp - mm) / (2 * h)
    an = (grad * v).sum(1)
    assert ((fd - an).abs() <= 1e-6 * an.abs().clamp_min(1e-3)).all()


def test_c2_full_size_quadratic_form_second_difference(c2):
    """F(y) = -2 n mll(y) = (y-m)^T K^-1 (y-m) + const, so its second difference along r,
    F(y+r) + F(y-r) - 2 F(y) = 2 r^T K^-1 r, is positive, independent of const and exactly
    quadratic in the step: the step 2r gives 4x the value."""
    from pgmuvi_b200 import ops
    g, d = c2
    n = 512
    gen = torch.Generator().manual_seed(9)
    r = torch.randn(d["y"].shape, generator=gen, dtype=torch.float64).to(d["y"].device)
    F = lambda y: -2 * n * _eval(ops, g, dict(d, y=y.contiguous()), want_grad=False)[0]
    f0 = F(d["y"])
    q1 = F(d["y"] + r) + F(d["y"] - r) - 2 * f0
    q2 = F(d["y"] + 2 * r) + F(d["y"] - 2 * r) - 2 * f0
    assert (q1 > 0).all()
    assert ((q2 - 4 * q1).abs() <= 1e-8 * q2.abs()).all()


# ---- fp32 entry points (the reference's default dtype, SURVEY F8) ---------------------------
F32_RTOL = 1e-4   # north star: MLL and gradients within 1e-4 relative in fp32


@pytest.mark.parametrize("name", ["sm1d_n100_q2_learn", "sm1d_n512_q4", "sm1d_ragged_q4",
                                  "sm2d_prodsum_4x48_q4", "sep_rq_4x48_q4", "sm2d_prodsum_3x64_q8",
                                  "sm1d_n130_q5_learn"])
def test_f32_entry_matches_f64_path_on_the_same_rounded_inputs(name, cuda_device):
    """pgm_sm_mll_grad_f32 = fp32 storage, fp64 arithmetic: on the fp32-rounded inputs it must
    equal the fp64 entry point rounded once to fp32, and stay within the fp32 bar of the
    oracle evaluated on those same inputs."""
    from pgmuvi_b200 import ops
    from oracle import ModelSpec, mll_and_grad_analytic
    g = load_golden(name)
    d = _dev(g, cuda_device)
    f32 = {k: (v.to(torch.float32) if v is not None and v.dtype == torch.float64 else v)
           for k, v in d.items()}
    mll32, grad32, info32 = _eval(ops, g, f32)
    assert mll32.dtype == torch.float32 and grad32.dtype == torch.float32
    up = {k: (v.to(torch.float64) if v is not None and v.dtype == torch.float32 else v)
          for k, v in f32.items()}
    mll64, grad64, info64 = _eval(ops, g, up)
    assert torch.equal(info32, info64)
    assert torch.equal(mll32, mll64.to(torch.float32))
    assert torch.equal(grad32, grad64.to(torch.float32))
    # oracle on the rounded inputs (first light curve)
    spec = ModelSpec(d=g["d"], Q=g["Q"], kind=g["kind"], learn_noise=g["learn_noise"])
    nb = g["x"].shape[1] if g["n_valid"] is None else int(g["n_valid"][0])
    c = lambda t: None if t is None else t[0].cpu()
    lb, ub = up["lb"].cpu(), up["ub"].cpu()
    if lb.dim() == 2:
        lb, ub = lb[0], ub[0]
    xo = c(up["x"])[:nb]
    mo, go, _ = mll_and_grad_analytic(xo, c(up["y"])[:nb],
                                      None if up["noise"] is None else c(up["noise"])[:nb],
                                      c(up["raw"]), d["kinds"].cpu(), lb, ub, spec)
    assert abs(float(mll32[0]) - float(mo)) <= F32_RTOL * abs(float(mo))
    assert float((grad32[0].cpu().double() - go).abs().max()) <= F32_RTOL * float(go.abs().max())


def test_f32_fit_entry_matches_f64_fit(cuda_device):
    from pgmuvi_b200 import ops, _lib
    g = load_golden("sm1d_n100_q2_learn")
    d = _dev(g, cuda_device)
    f32 = {k: (v.to(torch.float32) if v is not None and v.dtype == torch.float64 else v)
           for k, v in d.items()}
    args = (g["kind"], g["Q"], g["learn_noise"], _lib.OPT_ADAMW, 0.1, 0.9, 0.999, 1e-8, 0.01, 5,
            5, 0.0, 9, True)
    raw32 = f32["raw"].clone()
    loss32, hist32, it32, info32 = ops.sm_fit(f32["x"], f32["y"], f32["noise"], raw32,
                                              f32["kinds"], f32["lb"], f32["ub"], f32["n_valid"],
                                              *args)
    raw64 = f32["raw"].double().clone()
    loss64, hist64, it64, info64 = ops.sm_fit(f32["x"].double(), f32["y"].double(),
                                              f32["noise"].double(), raw64, f32["kinds"],
                                              f32["lb"].double(), f32["ub"].double(),
                                              f32["n_valid"], *args)
    assert loss32.dtype == torch.float32 and hist32.dtype == torch.float32
    assert torch.equal(it32, it64) and torch.equal(info32, info64)
    assert torch.equal(loss32, loss64.float())
    assert torch.equal(hist32, hist64.float())
    assert torch.equal(raw32, raw64.float())
