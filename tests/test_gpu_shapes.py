"""GPU tests at the shapes where the kernels go wrong: ragged tile edges, scratch reused across light
curves of different length, the fused kernel at fit_batch's limit and the on-device early stop.

Every reference is the fp64 oracle evaluated on the host at test time.  Inputs beyond a light
curve's n_valid are NaN, so a kernel that reads them produces NaN.  Tolerances are the same as the
golden tests: MLL 1e-9 relative, gradient 1e-7 of max |grad|, dense K 1e-13 max(1, |K|),
alpha 1e-9 of max |alpha|."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

MLL_RTOL = 1e-9
GRAD_RTOL = 1e-7
K_RTOL = 1e-13
ALPHA_RTOL = 1e-9

# one point, and one below / at / above every multiple of the 64-point tile up to 6 tiles
EDGES = [1, 2, 3, 63, 64, 65, 127, 128, 129, 191, 192, 193, 255, 256, 257, 383, 384, 385]

# (kind, Q, learn_noise) -> instantiation (KIND, QT, D)
MODELS = {
    "sm1d_q4": (0, 4, False),     # (0, 4, 1): 1-D SM-4 (BASELINE C2)
    "sm1d_q5": (0, 5, True),      # (0, 8, 1): LEAN layout with three padded mixtures
    "ard_q8": (1, 8, False),      # (1, 8, 2): one block per SM, full shared-memory layout
    "matern_rbf": (14, 0, False),  # Matern-1.5 x RBF, the reference's default 2DSeparable
}


def _batch(kind, Q, learn_noise, n_valid, n_max, seed0):
    """Seeded batch of len(n_valid) light curves of n_max points, NaN beyond each n_valid.  2-D light
    curves have their rows shuffled so that short ones still see several wavelengths."""
    from pgmuvi_b200 import synthetic as S
    B = len(n_valid)
    if kind == 0:
        bt = S.make_batch_1d(B, n_max, Q=Q, learn_noise=learn_noise, seed0=seed0)
    else:
        bands = next(k for k in (8, 5, 4, 3) if n_max % k == 0)
        if kind >= 8:
            bt = S.make_batch_stat(B, kind, n_bands=bands, n_per_band=n_max // bands,
                                   learn_noise=learn_noise, seed0=seed0)
        else:
            bt = S.make_batch_2d(B, bands, n_max // bands, Q=Q, learn_noise=learn_noise,
                                 seed0=seed0)
        rng = np.random.default_rng(seed0)
        for b in range(B):
            p = rng.permutation(n_max)
            for k in ("x", "y", "noise"):
                bt[k][b] = bt[k][b][p]
    for b, m in enumerate(n_valid):
        for k in ("x", "y", "noise"):
            bt[k][b, m:] = np.nan
    bt.update(kind=kind, Q=Q, learn_noise=learn_noise, n_valid=np.asarray(n_valid, np.int32))
    return bt


def _dev(bt, dev, sl=slice(None)):
    """Arguments of the ops for the light curves bt[sl] (the whole n_max, NaN padding included)."""
    T = lambda a, dt=torch.float64: torch.tensor(np.ascontiguousarray(a), dtype=dt, device=dev)
    return (T(bt["x"][sl]), T(bt["y"][sl]), T(bt["noise"][sl]), T(bt["raw"][sl]),
            T(bt["kinds"], torch.int32), T(bt["lb"][sl]), T(bt["ub"][sl]),
            T(bt["n_valid"][sl], torch.int32), bt["kind"], bt["Q"], bt["learn_noise"])


def _oracle(bt, b, dense=False):
    """The oracle on light curve b: (mll, grad, info) and, with dense=True, K~ and alpha."""
    from oracle import ModelSpec, constrain, kernel_dense, mll_and_grad_analytic, unpack_params
    from oracle.sm_gp import noise_diag, psd_safe_cholesky
    m = int(bt["n_valid"][b])
    t = lambda a: torch.tensor(a[b][:m])
    x, y, nz = t(bt["x"]), t(bt["y"]), t(bt["noise"])
    raw, kinds = torch.tensor(bt["raw"][b]), torch.tensor(bt["kinds"])
    lb, ub = torch.tensor(bt["lb"][b]), torch.tensor(bt["ub"][b])
    spec = ModelSpec(d=x.shape[1], Q=bt["Q"], kind=bt["kind"], learn_noise=bt["learn_noise"])
    mll, grad, info = mll_and_grad_analytic(x, y, nz, raw, kinds, lb, ub, spec)
    out = dict(mll=float(mll), grad=grad.numpy(), info=int(info))
    if dense:
        th = constrain(raw, kinds, lb, ub)
        mean, _, _, _, noise = unpack_params(th, spec)
        Kt = kernel_dense(x, x, th, spec) + torch.diag_embed(noise_diag(m, nz, noise, y.dtype))
        L, _ = psd_safe_cholesky(Kt)
        out["K"] = Kt.numpy()
        out["alpha"] = torch.cholesky_solve((y - mean).unsqueeze(-1), L).squeeze(-1).numpy()
    return out


def _check(what, bt, b, ref, mll, grad, info):
    tag = f"{what}: light curve {b}, n_valid {int(bt['n_valid'][b])}"
    assert int(info) == ref["info"] == 0, tag
    assert abs(float(mll) - ref["mll"]) <= MLL_RTOL * abs(ref["mll"]), tag
    scale = np.abs(ref["grad"]).max()
    assert np.abs(np.asarray(grad) - ref["grad"]).max() <= GRAD_RTOL * scale, tag


def _same_bits(a, b):
    """Bitwise equality of two float64 tensors (NaN included)."""
    return a.shape == b.shape and torch.equal(a.contiguous().view(torch.int64),
                                              b.contiguous().view(torch.int64))


@pytest.mark.parametrize("model", list(MODELS))
def test_tile_edges_against_the_oracle(model, cuda_device):
    """n_valid on both sides of every tile boundary up to n_max = 385, NaN beyond it: MLL, gradient
    and info of the fused and staged engines, alpha of both, and the whole dense K~."""
    from pgmuvi_b200 import ops
    kind, Q, learn_noise = MODELS[model]
    bt = _batch(kind, Q, learn_noise, EDGES, 385, seed0=4100 + kind)
    args = _dev(bt, cuda_device)
    refs = [_oracle(bt, b, dense=True) for b in range(len(EDGES))]
    for what, fn in (("fused", ops.sm_mll_grad), ("staged", ops.sm_mll_grad_staged)):
        mll, grad, info = (t.cpu().numpy() for t in fn(*args, True))
        for b, ref in enumerate(refs):
            _check(what, bt, b, ref, mll[b], grad[b], info[b])
    for staged in (False, True):
        mll, grad, info, alpha = (t.cpu().numpy() for t in ops.sm_mll_grad_alpha(*args, staged))
        for b, ref in enumerate(refs):
            m = int(bt["n_valid"][b])
            _check(f"alpha entry, staged={staged}", bt, b, ref, mll[b], grad[b], info[b])
            scale = np.abs(ref["alpha"]).max()
            assert np.abs(alpha[b, :m] - ref["alpha"]).max() <= ALPHA_RTOL * scale, (staged, b)
            assert not alpha[b, m:].any(), (staged, b)
    x, y, nz, raw, kinds, lb, ub, nv, *spec = args
    K = ops.sm_kernel_dense(x, nz, raw, kinds, lb, ub, nv, *spec).cpu().numpy()
    for b, ref in enumerate(refs):
        m = int(bt["n_valid"][b])
        Kr = ref["K"]
        assert np.abs(K[b, :m, :m] - Kr).max() <= K_RTOL * max(1.0, np.abs(Kr).max()), b
        assert not K[b, m:].any() and not K[b, :, m:].any(), b


@pytest.mark.parametrize("kind,Q", [(0, 4), (1, 8)])
def test_scratch_reuse_and_neighbour_independence(kind, Q, cuda_device, monkeypatch):
    """More light curves than resident blocks; with the static stride every block first takes a
    long light curve (n_valid >= 1000), then short ones, so its scratch is reused under a smaller
    stride.  Each light curve's result is bit for bit what it gives alone (B = 1, same n_max and
    NaN padding), for evaluation and for a 3-step fit; the ticket scheduler gives the same bits;
    a seeded sample matches the oracle."""
    from pgmuvi_b200 import _lib, ops
    d = 1 if kind == 0 else 2
    grid = _lib.load().pgm_fused_grid(d, Q, kind)
    assert grid > 0
    B = 2 * grid + 37
    n_valid = [1000 + (7 * b) % 41 if b < grid else EDGES[(b - grid) % len(EDGES)]
               for b in range(B)]
    bt = _batch(kind, Q, False, n_valid, 1040, seed0=6100 + kind)
    args = _dev(bt, cuda_device)
    one = lambda b: _dev(bt, cuda_device, slice(b, b + 1))

    monkeypatch.setenv("PGM_STATIC_STRIDE", "1")
    mll, grad, info = ops.sm_mll_grad(*args, True)
    alone = [ops.sm_mll_grad(*one(b), True) for b in range(B)]
    for k, name in enumerate(("mll", "grad", "info")):
        got = torch.cat([a[k] for a in alone])
        want = (mll, grad, info)[k]
        assert _same_bits(got, want) if k < 2 else torch.equal(got, want), name
    assert int(info.abs().sum()) == 0

    fit = lambda a, raw: ops.sm_fit(*a[:3], raw, *a[4:], _lib.OPT_ADAMW, 0.1, 0.9, 0.999, 1e-8,
                                    0.01, 3, 3, 0.0, 9, True)
    raw_b = args[3].clone()
    loss_b, hist_b, it_b, info_b = fit(args, raw_b)
    for b in range(B):
        a = one(b)
        raw1 = a[3].clone()
        loss1, hist1, it1, info1 = fit(a, raw1)
        assert _same_bits(loss1[:, 0], loss_b[:, b]), b
        assert _same_bits(hist1[:, 0], hist_b[:, b]), b
        assert _same_bits(raw1[0], raw_b[b]), b
        assert int(it1[0]) == int(it_b[b]) == 3 and int(info1[0]) == int(info_b[b]), b
    monkeypatch.delenv("PGM_STATIC_STRIDE")

    mll_t, grad_t, info_t = ops.sm_mll_grad(*args, True)          # ticket scheduler where it runs
    assert _same_bits(mll_t, mll) and _same_bits(grad_t, grad) and torch.equal(info_t, info)

    mll, grad, info = mll.cpu().numpy(), grad.cpu().numpy(), info.cpu().numpy()
    for b in np.random.default_rng(12).choice(B, 12, replace=False):
        _check("batch", bt, b, _oracle(bt, b), mll[b], grad[b], info[b])


@pytest.mark.parametrize("kind,Q", [(0, 4), (1, 8)])
def test_fused_kernel_at_the_fit_batch_limit(kind, Q, cuda_device):
    """n_max = 2048, the longest light curve fit_batch hands to the fused kernel, full and ragged."""
    from pgmuvi_b200 import ops
    bt = _batch(kind, Q, False, [2048, 1985], 2048, seed0=8100 + kind)
    mll, grad, info = (t.cpu().numpy() for t in ops.sm_mll_grad(*_dev(bt, cuda_device), True))
    for b in range(2):
        _check("fused n = 2048", bt, b, _oracle(bt, b), mll[b], grad[b], info[b])


def test_device_early_stop_matches_the_oracle_loop(cuda_device):
    """sm_fit's on-device rule (stop after iteration i > miniter once np.std of the last stopavg
    losses is below stop) against oracle.train_loop: members stop at different iterations, the
    first ones while the window is still shorter than stopavg."""
    from oracle import ModelSpec, train_loop
    from pgmuvi_b200 import _lib, ops, synthetic as S
    B, maxiter, miniter, stopavg, stop, lr = 6, 40, 1, 9, 0.0225, 0.1
    bt = S.make_batch_1d(B, 60, Q=2, seed0=31)
    spec = ModelSpec(d=1, Q=2)
    refs = []
    for b in range(B):
        c = lambda a: torch.tensor(a[b])
        refs.append(train_loop(c(bt["x"]), c(bt["y"]), c(bt["noise"]), c(bt["raw"]),
                               torch.tensor(bt["kinds"]), c(bt["lb"]), c(bt["ub"]), spec,
                               maxiter=maxiter, miniter=miniter, stop=stop, lr=lr, optim="AdamW",
                               stopavg=stopavg))
    # preconditions: distinct stopping iterations, and no window within rounding of the threshold
    n_ref = [len(r["loss"]) for r in refs]
    assert len(set(n_ref)) >= 2 and min(n_ref) < stopavg
    for r in refs:
        loss = np.array(r["loss"], dtype=float)
        for i in range(miniter + 1, len(loss)):
            assert abs(np.std(loss[:i + 1][-stopavg:]) - stop) > 1e-6 * stop
    T = lambda a, dt=torch.float64: torch.tensor(np.asarray(a), dtype=dt, device=cuda_device)
    raw = T(bt["raw"])
    loss, hist, n_iter, info = ops.sm_fit(
        T(bt["x"]), T(bt["y"]), T(bt["noise"]), raw, T(bt["kinds"], torch.int32), T(bt["lb"]),
        T(bt["ub"]), None, 0, 2, False, _lib.OPT_ADAMW, lr, 0.9, 0.999, 1e-8, 0.01, maxiter, miniter,
        stop, stopavg, True)
    assert n_iter.cpu().tolist() == n_ref and info.cpu().tolist() == [0] * B
    loss, hist, raw = loss.cpu().numpy(), hist.cpu().numpy(), raw.cpu().numpy()
    for b, (r, n) in enumerate(zip(refs, n_ref)):
        want = np.array(r["loss"], dtype=float)
        assert np.abs(loss[:n, b] - want).max() <= 1e-9 * np.abs(want).max(), b
        assert np.isnan(loss[n:, b]).all(), b
        assert np.abs(hist[:n + 1, b] - np.stack(r["raw"])).max() <= 1e-8, b
        assert np.abs(raw[b] - r["raw"][-1]).max() <= 1e-8, b
