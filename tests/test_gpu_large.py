"""GPU tests of the single-large-GP path (pgm_sm_mll_grad_large_f64; BASELINE configs C3 / C4):
the whole device factors ONE K~.  Checked against the oracle's golden vectors (every kernel
kind, ragged last tile), against the fused one-block-per-light-curve kernel at n = 1500, and -
at n = 8000 (C3's size) - through size-independent properties (finite differences of the MLL
along the gradient; permutation invariance)."""
import os

import numpy as np
import pytest
import torch

from conftest import golden_names, load_golden

pytestmark = pytest.mark.gpu


def _t(a, dev, dt=torch.float64):
    return None if a is None else torch.tensor(np.asarray(a), dtype=dt, device=dev)


@pytest.mark.parametrize("name", golden_names())
def test_large_path_matches_goldens(name, cuda_device):
    from pgmuvi_b200 import ops
    g = load_golden(name)
    dev = cuda_device
    n = g["x"].shape[1]
    for b in range(g["x"].shape[0]):
        nb = n if g["n_valid"] is None else int(g["n_valid"][b])
        lb = g["lb"][b] if np.ndim(g["lb"]) == 2 else g["lb"]
        ub = g["ub"][b] if np.ndim(g["ub"]) == 2 else g["ub"]
        mll, grad, info = ops.sm_mll_grad_large(
            _t(g["x"][b][:nb], dev), _t(g["y"][b][:nb], dev),
            None if g["noise"] is None else _t(g["noise"][b][:nb], dev), _t(g["raw"][b], dev),
            _t(g["kinds"], dev, torch.int32), _t(lb, dev), _t(ub, dev), g["kind"], g["Q"],
            g["learn_noise"], True)
        assert info == int(g["info"][b])
        assert abs(float(mll) - g["mll"][b]) <= 1e-9 * abs(g["mll"][b])
        scale = np.abs(g["grad_autograd"][b]).max()
        assert np.abs(grad.cpu().numpy() - g["grad_autograd"][b]).max() <= 1e-7 * scale


def test_large_path_matches_fused_kernel_n1500(cuda_device):
    from pgmuvi_b200 import ops, synthetic as S
    bt = S.make_batch_1d(1, 1500, Q=4, learn_noise=True, seed0=4242)
    dev = cuda_device
    x, y, nz, raw = (_t(bt[k], dev) for k in ("x", "y", "noise", "raw"))
    kinds, lb, ub = _t(bt["kinds"], dev, torch.int32), _t(bt["lb"], dev), _t(bt["ub"], dev)
    m0, g0, i0 = ops.sm_mll_grad(x, y, nz, raw, kinds, lb, ub, None, 0, 4, True, True)
    m1, g1, i1 = ops.sm_mll_grad_large(x[0], y[0], nz[0], raw[0], kinds, lb[0], ub[0], 0, 4, True)
    assert i1 == int(i0[0]) == 0
    assert abs(float(m1) - float(m0[0])) <= 1e-10 * abs(float(m0[0]))
    assert float((g1 - g0[0]).abs().max()) <= 1e-8 * float(g0[0].abs().max())
    # MLL-only entry
    m2, _, _ = ops.sm_mll_grad_large(x[0], y[0], nz[0], raw[0], kinds, lb[0], ub[0], 0, 4, True,
                                     want_grad=False)
    assert float(m2) == float(m1)


def test_large_path_c3_size_properties(cuda_device):
    """C3: 8 bands x 1000 epochs (n = 8000), 2-D SM-4, FixedNoise, fp64.  The gradient agrees
    with a central finite difference of the MLL along a random direction, and the MLL does not
    depend on the order of the points."""
    from pgmuvi_b200 import ops, synthetic as S
    bt = S.make_batch_2d(1, 8, 1000, Q=4, learn_noise=False, seed0=31)
    dev = cuda_device
    x, y, nz, raw = (_t(bt[k][0], dev) for k in ("x", "y", "noise", "raw"))
    kinds, lb, ub = _t(bt["kinds"], dev, torch.int32), _t(bt["lb"][0], dev), _t(bt["ub"][0], dev)
    ev = lambda r, wg=False, xx=x, yy=y, nn=nz: ops.sm_mll_grad_large(
        xx, yy, nn, r, kinds, lb, ub, 1, 4, False, want_grad=wg)
    mll, grad, info = ev(raw, True)
    assert info == 0 and np.isfinite(float(mll)) and bool(torch.isfinite(grad).all())
    gen = torch.Generator().manual_seed(0)
    u = torch.randn(raw.shape, generator=gen, dtype=torch.float64).to(dev)
    u = u / u.norm()
    h = 1e-5
    fd = (float(ev(raw + h * u)[0]) - float(ev(raw - h * u)[0])) / (2 * h)
    an = float((grad * u).sum())
    assert abs(fd - an) <= 1e-5 * max(1.0, abs(an))
    perm = torch.randperm(x.shape[0], generator=gen).to(dev)
    mp = float(ev(raw, False, x[perm], y[perm], nz[perm])[0])
    assert abs(mp - float(mll)) <= 1e-9 * abs(float(mll))


LARGE_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden_large")
LARGE_CASES = sorted(f[:-4] for f in os.listdir(LARGE_DIR) if f.endswith(".npz")) \
    if os.path.isdir(LARGE_DIR) else []


@pytest.mark.parametrize("name", LARGE_CASES)
def test_large_path_matches_at_size_goldens(name, cuda_device):
    """PARITY AT SIZE (tests/golden_large, oracle/make_golden_large.py): C3 (n = 8000, 2-D SM-4),
    C4 (n = 32768, SM-8) and an n = 14000 case (N = 219 tile rows, ragged last tile, learned
    noise) that takes the staged engine's right-looking PANEL schedule (N > 200).  MLL, the full
    raw-parameter gradient and info against the blocked fp64 CPU oracle - LAPACK dpotrf / dpotri
    on the assembled K~, gradient by autograd through the restated kernel - i.e. the Cholesky
    branch of pgmuvi/trainers.py:179-181 (fast_computations off, lightcurve.py:5965-5968).
    Tolerance: 1e-6 relative (north star, fp64); measured agreement is ~1e-9."""
    from pgmuvi_b200 import ops
    z = np.load(os.path.join(LARGE_DIR, name + ".npz"))
    dev = cuda_device
    mll, grad, info = ops.sm_mll_grad_large(
        _t(z["x"], dev), _t(z["y"], dev), _t(z["noise"], dev), _t(z["raw"], dev),
        _t(z["kinds"], dev, torch.int32), _t(z["lb"], dev), _t(z["ub"], dev), int(z["kind"]),
        int(z["Q"]), bool(z["learn_noise"]), want_grad=True)
    assert info == int(z["info"])
    ref = float(z["mll"])
    err_m = abs(float(mll) - ref) / abs(ref)
    gref = z["grad"]
    err_g = float(np.abs(grad.cpu().numpy() - gref).max() / np.abs(gref).max())
    print(f"[at-size parity] {name}: n={z['x'].shape[0]} mll rel err {err_m:.2e}, "
          f"grad rel err {err_g:.2e}")
    assert err_m <= 1e-6 and err_g <= 1e-6
    # MLL-only entry: the same Cholesky phase, no inverse / gradient
    m2, _, i2 = ops.sm_mll_grad_large(
        _t(z["x"], dev), _t(z["y"], dev), _t(z["noise"], dev), _t(z["raw"], dev),
        _t(z["kinds"], dev, torch.int32), _t(z["lb"], dev), _t(z["ub"], dev), int(z["kind"]),
        int(z["Q"]), bool(z["learn_noise"]), want_grad=False)
    assert i2 == int(z["info"]) and abs(float(m2) - ref) <= 1e-6 * abs(ref)


def test_train_routes_long_light_curves_through_the_large_path(cuda_device):
    """trainers.train on n = 2600 > LARGE_N: host loop over the whole-device MLL+gradient and
    the optimiser kernel, against the oracle's restatement of pgmuvi/trainers.py:177-207; the
    torch-optimizer seam (loss.backward with a stock optimiser) follows the same trajectory."""
    from oracle import ModelSpec, train_loop
    from pgmuvi_b200.lightcurve import Lightcurve
    from pgmuvi_b200.mll import pack_model
    from pgmuvi_b200.trainers import LARGE_N, train
    n = 2600
    assert n > LARGE_N
    outs = []
    for use_instance in (False, True):
        rng = np.random.default_rng(11)
        t = np.sort(rng.uniform(0.0, 900.0, n))
        y = np.sin(2 * np.pi * t / 61.0) + 0.1 * rng.standard_normal(n)
        lc = Lightcurve(t, y, yerr=np.full(n, 0.1), max_samples=None,
                        xtransform="minmax").double()
        lc.set_model("1D", num_mixtures=2)
        lc.double()
        lc.set_default_constraints()
        lc.model.initialize(**{"covar_module.mixture_means": torch.tensor([14.5, 30.0]),
                               "covar_module.mixture_scales": torch.tensor([1.5, 1.0])})
        pk = pack_model(lc.model)
        if not use_instance:
            spec = ModelSpec(d=1, Q=2, kind=0, learn_noise=False)
            ref = train_loop(lc._xdata_transformed.double().unsqueeze(-1),
                             lc._ydata_transformed.double(), pk.fixed_noise.double(),
                             pk.raw().detach().double(), pk.kinds, pk.lb, pk.ub, spec, maxiter=3,
                             miniter=3, stop=None, lr=0.05, optim="Adam")
            res = train(lc, maxiter=3, miniter=3, stop=None, lr=0.05, optim="Adam")
            assert np.allclose(np.array(res["loss"], dtype=float),
                               np.array(ref["loss"], dtype=float), rtol=1e-9, atol=1e-12)
            assert np.allclose(pk.raw().detach().numpy(), ref["raw"][-1], rtol=1e-7, atol=1e-9)
        else:
            opt = torch.optim.Adam(lc.model.parameters(), lr=0.05)
            res = train(lc, maxiter=3, miniter=3, stop=None, optim=opt)
        outs.append(np.array(res["loss"], dtype=float))
        assert len(res["covar_module.mixture_means"]) == 4
    assert np.allclose(outs[0], outs[1], rtol=1e-9, atol=1e-12)


@pytest.mark.parametrize("name", golden_names())
def test_staged_batch_matches_goldens(name, cuda_device):
    """The whole golden batch in ONE staged call (ragged n_valid, per-light-curve bounds)."""
    from pgmuvi_b200 import ops
    g = load_golden(name)
    dev = cuda_device
    mll, grad, info = ops.sm_mll_grad_staged(
        _t(g["x"], dev), _t(g["y"], dev), _t(g["noise"], dev), _t(g["raw"], dev),
        _t(g["kinds"], dev, torch.int32), _t(g["lb"], dev), _t(g["ub"], dev),
        _t(g["n_valid"], dev, torch.int32), g["kind"], g["Q"], g["learn_noise"], True)
    assert np.array_equal(info.cpu().numpy(), g["info"])
    assert np.abs(mll.cpu().numpy() - g["mll"]).max() <= 1e-9 * np.abs(g["mll"]).max()
    for b in range(len(g["mll"])):
        scale = np.abs(g["grad_autograd"][b]).max()
        assert np.abs(grad[b].cpu().numpy() - g["grad_autograd"][b]).max() <= 1e-7 * scale


def test_staged_engine_jitter_ladder_and_bitwise_agreement_with_fused(cuda_device):
    """Per-light-curve jitter ladder in the staged engine: the same failure codes as the fused
    kernel (tests/test_gpu_parity.py::test_jitter_ladder_and_failure_codes) and - for healthy
    members - the same MLL to 1e-12."""
    from pgmuvi_b200 import ops, synthetic as S
    bt = S.make_batch_1d(5, 96, Q=2, seed0=4242)
    bt["x"][1, 50, 0] = bt["x"][1, 49, 0]
    bt["noise"][1, :] = 1e-17
    bt["noise"][2, 10] = -50.0
    bt["x"][3, 5, 0] = float("nan")
    dev = cuda_device
    args = (_t(bt["x"], dev), _t(bt["y"], dev), _t(bt["noise"], dev), _t(bt["raw"], dev),
            _t(bt["kinds"], dev, torch.int32), _t(bt["lb"], dev), _t(bt["ub"], dev), None, 0, 2,
            False, True)
    m0, g0, i0 = ops.sm_mll_grad(*args)
    m1, g1, i1 = ops.sm_mll_grad_staged(*args)
    assert i1.cpu().tolist() == i0.cpu().tolist()
    assert i1[2] == -2 and i1[3] == -1 and i1[1] >= 1
    for b in (0, 4):
        assert abs(float(m1[b]) - float(m0[b])) <= 1e-12 * abs(float(m0[b]))
        assert float((g1[b] - g0[b]).abs().max()) <= 1e-9 * float(g0[b].abs().max())
    assert torch.isnan(m1[2]) and torch.isnan(m1[3]) and torch.isnan(g1[2]).all()


# ---------------------------------------------------------------------------------------
# N1: posterior prediction (pgm_sm_predict_f64)
# ---------------------------------------------------------------------------------------
HERE = os.path.dirname(os.path.abspath(__file__))
PRED_FILES = {f[:-4]: os.path.join(dd, f)
              for dd in (os.path.join(HERE, "golden_predict"), os.path.join(HERE, "golden", "predict"))
              for f in os.listdir(dd) if f.endswith(".npz")}
PRED_CASES = sorted(PRED_FILES)


@pytest.mark.parametrize("name", PRED_CASES)
def test_prediction_matches_oracle_goldens(name, cuda_device):
    """mean* and the exact latent variance at 150 test points per light curve against the
    oracle's Cholesky-solve prediction (tests/golden_predict and tests/golden/predict,
    oracle/make_golden_predict.py).
    Tolerance 1e-9 of the prior variance scale (var* is a difference of O(1) quantities)."""
    from pgmuvi_b200 import ops
    g = load_golden(name)
    p = np.load(PRED_FILES[name])
    dev = cuda_device
    mean, var, info = ops.sm_predict(
        _t(g["x"], dev), _t(g["y"], dev), _t(g["noise"], dev), _t(g["raw"], dev),
        _t(g["kinds"], dev, torch.int32), _t(g["lb"], dev), _t(g["ub"], dev),
        _t(g["n_valid"], dev, torch.int32), _t(p["xstar"], dev), g["kind"], g["Q"],
        g["learn_noise"])
    assert info.cpu().tolist() == [0] * mean.shape[0]
    scale = max(1.0, float(np.abs(p["var"]).max()), float(np.abs(p["mean"]).max()))
    assert np.abs(mean.cpu().numpy() - p["mean"]).max() <= 1e-9 * scale
    assert np.abs(var.cpu().numpy() - p["var"]).max() <= 1e-9 * scale


def test_prediction_interpolates_and_reverts_to_the_prior(cuda_device):
    """Properties at C2's size (n = 512): at the training inputs the latent variance is below
    the noise level and the mean tracks y; far outside the data var* -> k(0) = sum w_q and
    mean* -> the constant mean.  Also 10000 test points per light curve (the reference's grid)."""
    from pgmuvi_b200 import ops, synthetic as S
    bt = S.make_batch_1d(3, 512, Q=4, seed0=909)
    dev = cuda_device
    x, y, nz, raw = (_t(bt[k], dev) for k in ("x", "y", "noise", "raw"))
    kinds, lb, ub = _t(bt["kinds"], dev, torch.int32), _t(bt["lb"], dev), _t(bt["ub"], dev)
    xs = torch.cat([x[:, :, 0], torch.full((3, 64), 50.0, dtype=torch.float64, device=dev)], 1)
    mean, var, info = ops.sm_predict(x, y, nz, raw, kinds, lb, ub, None, xs.unsqueeze(-1), 0, 4,
                                     False)
    assert info.cpu().tolist() == [0, 0, 0]
    assert bool((var[:, :512] < nz).all()) and bool((var[:, :512] > -1e-12).all())
    assert float((mean[:, :512] - y).abs().max()) < 0.5
    from oracle import CON_SOFTPLUS  # noqa: F401  (constraints follow the oracle's table)
    w = torch.nn.functional.softplus(raw[:, 1:5])
    assert torch.allclose(var[:, 512:], w.sum(1, keepdim=True).expand(-1, 64), rtol=1e-9)
    grid = torch.linspace(0, 1, 10000, dtype=torch.float64, device=dev).expand(3, -1).contiguous()
    m2, v2, _ = ops.sm_predict(x, y, nz, raw, kinds, lb, ub, None, grid.unsqueeze(-1), 0, 4, False)
    assert bool(torch.isfinite(m2).all()) and bool((v2 > -1e-10).all())
