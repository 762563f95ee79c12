"""CPU tests of the oracle: golden vectors, internal cross-checks, and the reference-produced
known-answer test K3 (SURVEY.md Appendix C).  The oracle is the checker for the CUDA path."""
import math

import numpy as np
import pytest
import torch

from conftest import golden_names, load_golden
from oracle import (ModelSpec, adam_step, constrain, mll_and_grad_analytic,
                    mll_and_grad_autograd, psd_safe_cholesky, sm_kernel_dense, train_loop,
                    unconstrain, unpack_params)
from oracle.sm_gp import batched_mll_and_grad, noise_diag

torch.set_default_dtype(torch.float64)


def _case(g, b):
    n = g["x"].shape[1] if g["n_valid"] is None else int(g["n_valid"][b])
    t = lambda a: None if a is None else torch.tensor(a[b][:n])
    spec = ModelSpec(d=g["d"], Q=g["Q"], kind=g["kind"], learn_noise=g["learn_noise"])
    return (t(g["x"]), t(g["y"]), t(g["noise"]), torch.tensor(g["raw"][b]),
            torch.tensor(g["kinds"]), torch.tensor(g["lb"][b]), torch.tensor(g["ub"][b]), spec)


@pytest.mark.parametrize("name", golden_names())
def test_oracle_reproduces_goldens(name):
    g = load_golden(name)
    for b in range(g["x"].shape[0]):
        x, y, nz, raw, kinds, lb, ub, spec = _case(g, b)
        m, gr, info = mll_and_grad_analytic(x, y, nz, raw, kinds, lb, ub, spec)
        assert int(info) == int(g["info"][b])
        assert abs(float(m) - g["mll"][b]) <= 1e-11 * abs(g["mll"][b])
        scale = np.abs(g["grad_autograd"][b]).max()
        assert np.abs(gr.numpy() - g["grad_autograd"][b]).max() <= 1e-8 * scale
        assert np.abs(g["grad_analytic"][b] - g["grad_autograd"][b]).max() <= 1e-9 * scale


@pytest.mark.parametrize("name", ["sm1d_n100_q2_learn", "sm2d_prodsum_4x48_q4",
                                  "sm2d_sumprod_4x48_q4"])
def test_autograd_matches_closed_form(name):
    g = load_golden(name)
    x, y, nz, raw, kinds, lb, ub, spec = _case(g, 0)
    m1, g1, _ = mll_and_grad_autograd(x, y, nz, raw, kinds, lb, ub, spec)
    m2, g2, _ = mll_and_grad_analytic(x, y, nz, raw, kinds, lb, ub, spec)
    assert abs(float(m1) - float(m2)) <= 1e-12 * abs(float(m1))
    assert float((g1 - g2).abs().max()) <= 1e-10 * float(g1.abs().max())


def test_kernel_symmetry_stationarity_and_diag():
    g = load_golden("sm1d_n100_q2_learn")
    x, y, nz, raw, kinds, lb, ub, spec = _case(g, 0)
    mean, w, mu, sg, noise = unpack_params(constrain(raw, kinds, lb, ub), spec)
    K = sm_kernel_dense(x, x, w, mu, sg, spec.kind)
    assert torch.allclose(K, K.T, atol=1e-14)                       # tests/test_kernels.py:44-47
    assert torch.allclose(torch.diagonal(K), w.sum().expand(len(y)), atol=1e-14)
    Ks = sm_kernel_dense(x + 3.25, x + 3.25, w, mu, sg, spec.kind)  # stationary kernel
    assert torch.allclose(K, Ks, atol=1e-11)


def test_2d_variants_factorise():
    """prod-of-sums with Q=1 equals sum-of-products with Q=1 equals K_t o K_lambda
    (mirrors the ProductKernel identity of tests/test_kernels.py:130-139)."""
    g = load_golden("sm2d_prodsum_4x48_q2_learn")
    x = torch.tensor(g["x"][0])
    w = torch.tensor([0.7])
    mu = torch.tensor([[3.0, 0.4]])
    sg = torch.tensor([[1.1, 0.6]])
    K1 = sm_kernel_dense(x, x, w, mu, sg, 1)
    K2 = sm_kernel_dense(x, x, w, mu, sg, 2)
    Kt = sm_kernel_dense(x[:, :1], x[:, :1], torch.ones(1), mu[:, :1], sg[:, :1], 0)
    Kl = sm_kernel_dense(x[:, 1:], x[:, 1:], torch.ones(1), mu[:, 1:], sg[:, 1:], 0)
    assert torch.allclose(K2, 0.7 * Kt * Kl, atol=1e-13)
    assert torch.allclose(K1, 0.49 * Kt * Kl, atol=1e-13)   # weight enters once per dimension


def test_mll_is_per_datum_gaussian_logprob():
    g = load_golden("sm1d_n40_q4")
    x, y, nz, raw, kinds, lb, ub, spec = _case(g, 1)
    mean, w, mu, sg, noise = unpack_params(constrain(raw, kinds, lb, ub), spec)
    K = sm_kernel_dense(x, x, w, mu, sg, 0) + torch.diag_embed(noise_diag(len(y), nz, noise, y.dtype))
    mvn = torch.distributions.MultivariateNormal(mean.expand(len(y)), covariance_matrix=K)
    assert abs(float(mvn.log_prob(y)) / len(y) - g["mll"][1]) < 1e-10


def test_constraint_roundtrip():
    kinds = torch.tensor([0, 1, 1, 2])
    lb = torch.tensor([0.0, 0.0, 1.5, -2.0])
    ub = torch.tensor([0.0, 0.0, 0.0, 3.0])
    raw = torch.tensor([0.3, -2.0, 40.0, 0.7])
    v = constrain(raw, kinds, lb, ub)
    assert torch.allclose(unconstrain(v, kinds, lb, ub), raw, atol=1e-10)
    assert float(v[2]) == pytest.approx(41.5)
    assert -2.0 < float(v[3]) < 3.0


def test_jitter_ladder():
    A = torch.eye(4).repeat(3, 1, 1)
    A[1, 3, 3] = -1e-9          # rescued by the first jitter (1e-8)
    A[2, 3, 3] = -1.0           # not PD even with 1e-6
    L, info = psd_safe_cholesky(A)
    assert info.tolist() == [0, 1, -2]
    A[0, 0, 0] = float("nan")
    assert psd_safe_cholesky(A)[1].tolist()[0] == -1


def test_jitter_base_parameter():
    """jitter=None keeps the ladder by dtype (1e-8 float64, 1e-6 float32); jitter=1e-6 on float64
    input is the float32 ladder in float64 arithmetic: a member rescued at rung 3 of the float64
    ladder (t = 3e-7) is rescued at rung 1 there, factored as A + 1e-6 I."""
    A = torch.eye(4).repeat(4, 1, 1)
    A[1, 3, 3] = -3e-9
    A[2, 3, 3] = -3e-8
    A[3, 3, 3] = -3e-7
    L, info = psd_safe_cholesky(A)
    L8, info8 = psd_safe_cholesky(A, jitter=1e-8)
    assert info.tolist() == info8.tolist() == [0, 1, 2, 3] and torch.equal(L, L8)
    L6, info6 = psd_safe_cholesky(A, jitter=1e-6)
    assert info6.tolist() == [0, 1, 1, 1]
    assert torch.equal(L6[3], torch.linalg.cholesky(A[3] + 1e-6 * torch.eye(4)))
    assert psd_safe_cholesky(A.float())[1].tolist() == [0, 1, 1, 1]
    assert psd_safe_cholesky(A, jitter=1e-6)[1].tolist() == psd_safe_cholesky(A.float())[1].tolist()


@pytest.mark.parametrize("name", ["sm1d_n40_q4", "stat_matern_rbf_4x48"])
def test_jitter_base_through_mll_and_predict(name):
    """A light curve shifted to lambda_min(K~) = -3e-7: the default call is the float64 ladder's rung
    3 and equals jitter=1e-8; with jitter=1e-6 it is rung 1, and the closed form (the stationary
    kinds' _mll_and_grad_stat included), autograd, predict and train_loop all add 1e-6."""
    from oracle import predict
    from oracle.sm_gp import kernel_dense
    x, y, nz, raw, kinds, lb, ub, spec = _case(load_golden(name), 0)
    th = constrain(raw, kinds, lb, ub)
    Kt = kernel_dense(x, x, th, spec) + torch.diag_embed(
        noise_diag(len(y), nz, unpack_params(th, spec)[4], y.dtype))
    nz = nz - float(torch.linalg.eigvalsh(Kt)[0]) - 3e-7
    a = (x, y, nz, raw, kinds, lb, ub, spec)
    m0, g0, i0 = mll_and_grad_analytic(*a)
    m8, g8, i8 = mll_and_grad_analytic(*a, jitter=1e-8)
    assert int(i0) == int(i8) == 3 and float(m0) == float(m8) and torch.equal(g0, g8)
    m6, g6, i6 = mll_and_grad_analytic(*a, jitter=1e-6)
    ma, ga, ia = mll_and_grad_autograd(*a, jitter=1e-6)
    mj, gj, ij = mll_and_grad_analytic(x, y, nz + 1e-6, raw, kinds, lb, ub, spec)
    assert int(i6) == int(ia) == 1 and int(ij) == 0
    for m, gr in ((ma, ga), (mj, gj)):
        assert abs(float(m6) - float(m)) <= 1e-10 * abs(float(m))
        assert float((g6 - gr).abs().max()) <= 1e-8 * float(gr.abs().max())
    xs = x[:5] + 0.01
    p6 = predict(*a, xs, jitter=1e-6)
    pj = predict(x, y, nz + 1e-6, raw, kinds, lb, ub, spec, xs)
    assert int(p6[2]) == 1 and torch.allclose(p6[0], pj[0], rtol=1e-10)
    r6 = train_loop(*a, maxiter=1, lr=1e-3, jitter=1e-6, on_failure="stop")
    assert r6["info"] == [1] and len(r6["raw"]) == 2
    with pytest.raises(RuntimeError, match="info=-2"):
        train_loop(x, y, nz - 1.0, raw, kinds, lb, ub, spec, maxiter=2, jitter=1e-6)
    r = train_loop(x, y, nz - 1.0, raw, kinds, lb, ub, spec, maxiter=3, jitter=1e-6,
                   on_failure="stop")
    assert r["info"] == [-2] and np.isnan(r["loss"][0]) and len(r["raw"]) == 1


@pytest.mark.parametrize("decoupled,wd", [(False, 0.0), (True, 0.01)])
def test_adam_step_matches_torch(decoupled, wd):
    p0 = torch.randn(7, generator=torch.Generator().manual_seed(1))
    p = p0.clone().requires_grad_(True)
    opt = (torch.optim.AdamW([p], lr=0.1, eps=1e-8) if decoupled
           else torch.optim.Adam([p], lr=0.1, eps=1e-8))
    q, m, v = p0.numpy().copy(), np.zeros(7), np.zeros(7)
    for step in range(1, 5):
        gr = torch.sin(p.detach() * step)
        p.grad = gr.clone()
        opt.step()
        q, m, v = adam_step(q, gr.numpy(), m, v, step, 0.1, weight_decay=wd, decoupled=decoupled)
        assert np.allclose(q, p.detach().numpy(), rtol=0, atol=1e-14)


def test_train_loop_schema_and_goldens():
    g = load_golden("sm1d_n100_q2_learn")
    x, y, nz, raw, kinds, lb, ub, spec = _case(g, 0)
    res = train_loop(x, y, nz, raw, kinds, lb, ub, spec, maxiter=3, miniter=3, lr=0.1,
                     optim="AdamW")
    assert len(res["loss"]) == 3 and len(res["delta_loss"]) == 2 and len(res["raw"]) == 4
    assert np.allclose(np.stack(res["raw"]), g["adamw_raw"][0], atol=1e-12)
    assert np.allclose(np.array(res["loss"], dtype=float), g["adamw_loss"][0], atol=1e-12)


def test_batched_baseline_matches_single():
    g = load_golden("sm1d_n200_q4")
    t = torch.tensor
    spec = ModelSpec(d=1, Q=4)
    m, gr = batched_mll_and_grad(t(g["x"]), t(g["y"]), t(g["noise"]), t(g["raw"]), t(g["kinds"]),
                                 t(g["lb"]), t(g["ub"]), spec)
    assert np.allclose(m.numpy(), g["mll"], rtol=1e-11)
    assert np.allclose(gr.numpy(), g["grad_autograd"], rtol=1e-7, atol=1e-12)


def test_kat_k3_tutorial_fit():
    """The only reference-produced numbers for the path (executed notebook): fp32, AdamW,
    3000 iterations.  Published: loss -0.36470833, period 178.2802, weight 0.47454086."""
    from oracle.kats import K3_PUBLISHED, k3_problem, k3_run
    *_, meta = k3_problem()
    assert meta["P"] == pytest.approx(178.17964606037768)          # cell 6 printout
    assert meta["period_guess"] == pytest.approx(196.48998803679268)  # cell 21 printout
    assert meta["ystd"] == pytest.approx(0.7348, abs(1e-4))        # cell 10: weights = std(y)
    assert meta["ymid"] == pytest.approx(0.0200181, abs=1e-6)      # cell 10: constant
    out, _ = k3_run(torch.float32)
    assert out["loss"] == pytest.approx(K3_PUBLISHED["loss"], abs=1e-3)
    assert out["period"] == pytest.approx(K3_PUBLISHED["period"], rel=1e-3)
    assert out["weight"] == pytest.approx(K3_PUBLISHED["weight"], rel=5e-3)
    assert out["noise"] == pytest.approx(K3_PUBLISHED["noise"], rel=5e-3)


def test_kat_k1_comparison_notebook_1d_fit():
    """K1 (PGMUVI_comparison_with_other_codes.ipynb cells 7, 11): data from the reference's own
    generator (oracle/make_golden_kats.py), start state from the notebook printout, AdamW
    lr 0.05, 1000 iterations, float32 parameters on float64 data as the reference ran it.
    Published: loss -1.562, frequencies 0.00665436 / 0.0151593, no early stop; the printed
    start constant 0.028102993965148926 is reproduced to the last digit."""
    from oracle.kats import K1_PUBLISHED, k1_run
    out = k1_run(torch.float32)
    assert out["constant0"] == K1_PUBLISHED["constant0"]
    assert out["weight0"] == pytest.approx(K1_PUBLISHED["weight0"], abs=5e-5)
    assert out["n_iter"] == 1000                                   # no early stop
    assert out["loss"] == pytest.approx(K1_PUBLISHED["loss"], abs=4e-3)
    for f, fp in zip(out["freqs"], K1_PUBLISHED["freqs"]):
        assert f == pytest.approx(fp, rel=1.5e-3)


def test_kat_k2_comparison_notebook_2d_fit():
    """K2 (same notebook, cell 30): 2-D SM kernel (ard_num_dims = 2, product over dimensions of
    per-dimension mixture sums), all raw parameters 0, AdamW lr 0.05.  Published: start
    means 9.4067 / weights 0.6931, loss 0.904 at the early stop (iteration 348), both time
    frequencies 13.842627.  The trajectory has two basins (0.871 / 0.904) and which one is
    reached flips with the parameter dtype (SURVEY.md App. C); the float64-parameter run is the
    one that stays in the published basin."""
    from oracle.kats import K2_PUBLISHED, k2_run
    out = k2_run(torch.float64)
    assert out["means0"] == pytest.approx(K2_PUBLISHED["means0"], abs=5e-5)
    assert out["weight0"] == pytest.approx(K2_PUBLISHED["weight0"], abs=5e-5)
    assert out["constant0"] == pytest.approx(K2_PUBLISHED["constant0"], abs=1e-7)
    assert out["loss_hist"][K2_PUBLISHED["stop_iter"]] == pytest.approx(K2_PUBLISHED["loss"], abs=5e-4)
    assert out["loss"] == pytest.approx(K2_PUBLISHED["loss"], abs=5e-4)
    for f in out["time_freqs"]:
        assert f == pytest.approx(K2_PUBLISHED["time_freq"], rel=1e-4)


@pytest.mark.parametrize("name", ["sm1d_n512_q4_learn", "sm2d_prodsum_4x256_q4", "sep_rq_4x48_q4",
                                  "stat_qp_rbf_4x40", "sm1d_ragged_q4"])
def test_blocked_large_oracle_matches_goldens(name):
    """oracle/large.py (the generator of tests/golden_large: C3 / C4 / panel-schedule cases) is
    the same quantity as the per-light-curve oracle that produced tests/golden."""
    from oracle.large import mll_and_grad_blocked
    g = load_golden(name)
    for b in range(g["x"].shape[0]):
        x, y, nz, raw, kinds, lb, ub, spec = _case(g, b)
        m, gr, info = mll_and_grad_blocked(x, y, nz, raw, kinds, lb, ub, spec)
        assert int(info) == int(g["info"][b])
        assert abs(float(m) - g["mll"][b]) <= 1e-11 * abs(g["mll"][b])
        scale = np.abs(g["grad_autograd"][b]).max()
        assert np.abs(gr.numpy() - g["grad_autograd"][b]).max() <= 1e-9 * scale


def test_at_size_goldens_are_self_consistent():
    """tests/golden_large/*.npz: inputs regenerate from the committed generator's seeds and the
    stored gradient is finite with the packed layout's length."""
    import os
    from oracle.make_golden_large import CASES, OUT, case_inputs
    for name in CASES:
        z = np.load(os.path.join(OUT, name + ".npz"))
        bt, kind = case_inputs(name) if z["x"].shape[0] <= 16384 else (None, int(z["kind"]))
        if bt is not None:
            assert np.array_equal(bt["x"][0].astype(np.float32), z["x"])
            assert np.array_equal(bt["raw"][0], z["raw"])
        assert int(z["kind"]) == kind and int(z["info"]) == 0
        assert np.isfinite(z["grad"]).all() and z["grad"].shape == z["raw"].shape
