"""The jitter ladder and the Cholesky failure codes on every engine route, against the fp64 oracle.

Every engine restates GPyTorch's psd_safe_cholesky: when the Cholesky fails, retry with jit(1),
jit(2), jit(3) = 1e-8, 1e-7, 1e-6 on the diagonal (1e-6, 1e-5, 1e-4 for float32 models,
PGM_FLAG_JITTER_F32).  info is the rung that succeeded, -1 for a NaN in K~ and -2 for not positive
definite.  An exactly singular K~ passes or fails on rounding, so the members here choose their rung
through the smallest eigenvalue instead: with the healthy K~ built by the oracle, every valid point's
fixed noise is shifted by -lambda_min - t, which moves lambda_min to -t.  Rung r needs
jit(r-1) < t < jit(r) (jit(0) = 0); t is the geometric mean of the two (0.3 jit(1) for rung 1, 3 jit(3)
for -2).

The values of a jittered member can only be compared where they are well conditioned, so every
member is scaled first (output scale and noise by s, y - c by sqrt(s)) to ||K~||_2 / jit(1) = 1e4.  At
1.5e6 the oracle's permutation spread of the shortest rung-1 member of the 1-D batch is 1.1e-2 of
the MLL bar, and at 1.5e5 that of a Matern x RBF member is 5.6e-2 of it; at 1e4 the largest over
every member below is 1e-3 of the bar.
Two preconditions guard each designed member, and a case that fails them is mis-designed, not a
kernel finding: the oracle's own spread under a permutation of the points is at most 1/100 of the
bar, and the rung margin min(t - jit(r-1), jit(r) - t) is at least 1e6 n u ||K~||_2.

Tolerances are test_gpu_shapes.py's: MLL 1e-9 max(1, |MLL|), gradient 1e-7 of max |grad|, alpha
1e-9 of max |alpha|."""
import math
from functools import lru_cache

import numpy as np
import pytest
import torch

from test_gpu_schedules import C_TC, U, _map
from test_gpu_shapes import MODELS, _batch, _dev, _same_bits

TS = 64
N_MAX = 385                     # 7 tile rows
U64 = 2.0 ** -53
MLL_RTOL, GRAD_RTOL, ALPHA_RTOL = 1e-9, 1e-7, 1e-9
LADDERS = {"f64": 1e-8, "f32": 1e-6}        # jit(1) of each ladder
KT_OVER_JIT = 1e4           # ||K~||_2 / jit(1) of every designed member (see the module docstring)

# (label, n_valid, design): n_valid on both sides of the tile edges.  An int design is the rung the
# member is built for; the strings break the member in one way each (see _break).
MEMBERS = [
    ("rung0", 385, 0), ("rung1", 384, 1), ("rung2", 257, 2), ("rung3", 193, 3), ("not_pd", 129, -2),
    ("rung0_b", 64, 0), ("rung1_b", 65, 1), ("rung2_b", 128, 2), ("rung3_b", 383, 3),
    ("not_pd_b", 256, -2),
    ("neg_first", 255, "neg_first"),     # -50 noise in tile 0: fails in the first panel
    ("neg_mid", 321, "neg_mid"),         # ... in tile 3 of 6: a middle panel
    ("neg_last", 385, "neg_last"),       # ... at point 384, alone in the last tile (tile 6)
    ("nan_x", 192, "nan_x"), ("nan_wl", 191, "nan_wl"), ("nan_noise", 127, "nan_noise"),
    ("nan_raw", 63, "nan_raw"),
    ("nan_behind", 320, "nan_behind"),   # -50 noise in tile 0 and a NaN x in the last tile
    ("nan_y", 193, "nan_y"),             # NaN only in y: K~ is healthy, info 0 and a NaN MLL
]
EXPECT = {"neg_first": -2, "neg_mid": -2, "neg_last": -2, "nan_x": -1, "nan_wl": -1,
          "nan_noise": -1, "nan_raw": -1, "nan_behind": -1, "nan_y": 0}


def _members(model):
    d2 = MODELS[model][0] != 0
    return [m for m in MEMBERS if d2 or m[2] != "nan_wl"]


def _rung_t(r, j1):
    """t = -lambda_min that lands on rung r of the ladder with first rung j1."""
    jit = [0.0, j1, 10 * j1, 100 * j1]
    if r == 0:
        return None
    if r == 1:
        return 0.3 * j1
    if r == -2:
        return 3 * jit[3]
    return math.sqrt(jit[r - 1] * jit[r])


def rung_margin(r, t, j1):
    """How far t = -lambda_min is inside the interval of rung r (negative: outside)."""
    th = [0.0, j1, 10 * j1, 100 * j1]
    if r == 0:
        return th[0] - t
    if r == -2:
        return t - th[3]
    return min(t - th[r - 1], th[r] - t)


# ---------------------------------------------------------------------------------------------
# the member's inputs through the oracle
# ---------------------------------------------------------------------------------------------
def _spec(bt):
    from oracle import ModelSpec
    return ModelSpec(d=bt["x"].shape[2], Q=bt["Q"], kind=bt["kind"], learn_noise=bt["learn_noise"])


def _host(bt, b, perm=None):
    """Light curve b's valid points (optionally permuted) and parameters as CPU tensors."""
    m = int(bt["n_valid"][b])
    p = np.arange(m) if perm is None else perm
    t = lambda a: torch.tensor(a[b][:m][p])
    return (t(bt["x"]), t(bt["y"]), t(bt["noise"]), torch.tensor(bt["raw"][b]),
            torch.tensor(bt["kinds"]), torch.tensor(bt["lb"][b]), torch.tensor(bt["ub"][b]))


def _ktilde(bt, b):
    from oracle import constrain, kernel_dense, unpack_params
    from oracle.sm_gp import noise_diag
    x, y, nz, raw, kinds, lb, ub = _host(bt, b)
    th = constrain(raw, kinds, lb, ub)
    noise = unpack_params(th, _spec(bt))[4]
    K = kernel_dense(x, x, th, _spec(bt))
    return K, K + torch.diag_embed(noise_diag(len(y), nz, noise, y.dtype))


def _scale_slot(bt, b, slot, f):
    """Multiply the constrained value of raw slot `slot` of member b by f (bounds per member)."""
    from oracle.sm_gp import CON_INTERVAL, CON_NONE, CON_SOFTPLUS
    from pgmuvi_b200.synthetic import inv_softplus
    k = int(bt["kinds"][slot])
    if k == CON_SOFTPLUS:
        v = float(torch.nn.functional.softplus(torch.tensor(bt["raw"][b, slot])))
        bt["raw"][b, slot] = inv_softplus(np.array(f * v))
        bt["lb"][b, slot] *= f
    elif k == CON_INTERVAL:
        bt["lb"][b, slot] *= f
        bt["ub"][b, slot] *= f
    else:
        assert k == CON_NONE
        bt["raw"][b, slot] *= f


def _scale(bt, b, s):
    """K -> s K, noise -> s noise, y - c -> sqrt(s) (y - c) for member b."""
    from oracle import constrain
    spec = _spec(bt)
    K0 = _ktilde(bt, b)[0]
    if bt["kind"] >= 8:            # stationary kinds: the time kernel's output scale
        slots, f = [spec.o_lam], s
    else:                          # spectral mixture: the weights (K = prod over ds of sums over q)
        slots, f = range(spec.o_w, spec.o_w + spec.Q), s ** (1.0 / spec.ds)
    for p in slots:
        _scale_slot(bt, b, p, f)
    if bt["learn_noise"]:
        _scale_slot(bt, b, spec.o_noise, s)
    bt["noise"][b] *= s
    c = float(constrain(torch.tensor(bt["raw"][b]), torch.tensor(bt["kinds"]),
                        torch.tensor(bt["lb"][b]), torch.tensor(bt["ub"][b]))[0])
    bt["y"][b] = c + math.sqrt(s) * (bt["y"][b] - c)
    K1 = _ktilde(bt, b)[0]
    assert float((K1 - s * K0).abs().max()) <= 1e-12 * s * float(K0.abs().max()), "K is not s K"


def _design(bt, b, r, j1):
    """Shift member b's fixed noise so that lambda_min(K~) = -t of rung r."""
    if r == 0:
        return
    lam = float(np.linalg.eigvalsh(_ktilde(bt, b)[1].numpy())[0])
    m = int(bt["n_valid"][b])
    bt["noise"][b, :m] -= lam + _rung_t(r, j1)


def _break(bt, b, how):
    m = int(bt["n_valid"][b])
    nan = float("nan")
    if how.startswith("neg"):
        p = {"neg_first": 10, "neg_mid": 3 * TS + 17, "neg_last": m - 1}[how]
        bt["noise"][b, p] = -50.0
    elif how == "nan_x":
        bt["x"][b, 2 * TS + 5, 0] = nan
    elif how == "nan_wl":
        bt["x"][b, TS + 9, 1] = nan
    elif how == "nan_noise":
        bt["noise"][b, 70] = nan
    elif how == "nan_raw":
        bt["raw"][b, 1] = nan
    elif how == "nan_behind":
        bt["noise"][b, 10] = -50.0
        bt["x"][b, m - 2, 0] = nan
    else:
        assert how == "nan_y"
        bt["y"][b, 40] = nan


@lru_cache(maxsize=None)
def designed(model, ladder):
    """(batch, members) for `model` on `ladder` ("f64" or "f32": the inputs are then float32 values).
    Each designed member is a distinct light curve; the broken ones are rung-0 members broken after
    scaling."""
    kind, Q, learn_noise = MODELS[model]
    mem = _members(model)
    bt = _batch(kind, Q, learn_noise, [m[1] for m in mem], N_MAX, seed0=31000 + 100 * kind)
    bt = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in bt.items()}
    bt["lb"], bt["ub"] = bt["lb"].astype(np.float64), bt["ub"].astype(np.float64)
    j1 = LADDERS[ladder]
    for b, (_, _, how) in enumerate(mem):
        norm = float(np.linalg.eigvalsh(_ktilde(bt, b)[1].numpy())[-1])
        _scale(bt, b, KT_OVER_JIT * j1 / norm)
        if isinstance(how, int):
            _design(bt, b, how, j1)
    if ladder == "f32":
        for k in ("x", "y", "noise", "raw", "lb", "ub"):
            bt[k] = bt[k].astype(np.float32).astype(np.float64)
    for b, (_, _, how) in enumerate(mem):
        if isinstance(how, str):
            _break(bt, b, how)
    return bt, mem


def expected_info(how):
    return how if isinstance(how, int) else EXPECT[how]


def _oracle_at(bt, b, j1, perm=None):
    """(mll, grad, info, alpha) of the oracle on member b with first rung j1."""
    from oracle import mll_and_grad_analytic
    from oracle.sm_gp import psd_safe_cholesky
    x, y, nz, raw, kinds, lb, ub = _host(bt, b, perm)
    mll, grad, info = mll_and_grad_analytic(x, y, nz, raw, kinds, lb, ub, _spec(bt), jitter=j1)
    alpha = None
    if int(info) >= 0:
        from oracle import constrain
        L, _ = psd_safe_cholesky(_ktilde_perm(bt, b, perm), jitter=j1)
        c = constrain(raw, kinds, lb, ub)[0]
        alpha = torch.cholesky_solve((y - c).unsqueeze(-1), L).squeeze(-1).numpy()
    return float(mll), grad.numpy(), int(info), alpha


def _ktilde_perm(bt, b, perm):
    Kt = _ktilde(bt, b)[1]
    return Kt if perm is None else Kt[perm][:, perm]


@lru_cache(maxsize=None)
def references(model, ladder):
    """Oracle results of every member, with both preconditions checked on the designed ones."""
    bt, mem = designed(model, ladder)
    j1 = LADDERS[ladder]

    def one(b):
        how = mem[b][2]
        mll, grad, info, alpha = _oracle_at(bt, b, j1)
        assert info == expected_info(how), (model, ladder, mem[b][0], info)
        if isinstance(how, int) and how >= 0:
            m = int(bt["n_valid"][b])
            Kt = _ktilde(bt, b)[1].numpy()
            ev = np.linalg.eigvalsh(Kt)
            norm = float(ev[-1])
            margin = rung_margin(how, -float(ev[0]), j1)
            assert margin >= 1e6 * m * U64 * norm, (mem[b][0], margin, norm)
            perm = np.random.default_rng(b).permutation(m)
            mp, gp, ip, _ = _oracle_at(bt, b, j1, perm)
            assert ip == info
            assert abs(mp - mll) <= 0.01 * MLL_RTOL * max(1.0, abs(mll)), mem[b][0]
            assert np.abs(gp - grad).max() <= 0.01 * GRAD_RTOL * np.abs(grad).max(), mem[b][0]
        return dict(mll=mll, grad=grad, info=info, alpha=alpha)
    return _map(one, range(len(mem)))


def _check(what, bt, mem, refs, mll, grad, info, alpha=None):
    """info equals the designed code; failed members are NaN; the others match the oracle."""
    for b, ((label, m, how), ref) in enumerate(zip(mem, refs)):
        tag = f"{what}: {label} (n_valid {m})"
        assert int(info[b]) == ref["info"], (tag, int(info[b]), ref["info"])
        if ref["info"] < 0:
            assert np.isnan(mll[b]) and np.isnan(grad[b]).all(), tag
            if alpha is not None:
                assert np.isnan(alpha[b, :m]).all() and not alpha[b, m:].any(), tag
            continue
        if how == "nan_y":
            assert np.isnan(mll[b]), tag
            continue
        assert abs(float(mll[b]) - ref["mll"]) <= MLL_RTOL * max(1.0, abs(ref["mll"])), tag
        scale = np.abs(ref["grad"]).max()
        assert np.abs(np.asarray(grad[b]) - ref["grad"]).max() <= GRAD_RTOL * scale, tag
        if alpha is not None:
            scale = np.abs(ref["alpha"]).max()
            assert np.abs(alpha[b, :m] - ref["alpha"]).max() <= ALPHA_RTOL * scale, tag
            assert not alpha[b, m:].any(), tag


def _np(ts):
    return [t.cpu().numpy() for t in ts]


def _staged(args, monkeypatch, nb=None, **kw):
    from pgmuvi_b200 import ops
    with monkeypatch.context() as mp:
        if nb is not None:
            mp.setenv("PGM_STAGED_NB", str(nb))
            mp.setenv("PGM_STAGED_CHOL_ALL_N", "0")
        return _np(ops.sm_mll_grad_staged(*args, True, **kw))


# ---------------------------------------------------------------------------------------------
# without a GPU: the design itself
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("ladder", list(LADDERS))
def test_designed_members_land_on_their_rung_in_the_oracle(ladder):
    """Every member of the 1-D SM-4 batch gets its designed info from the oracle on its ladder (with
    both preconditions), and the rung-2 and rung-3 members designed for one ladder do not land on the same
    rung on the other: the base of the ladder decides."""
    refs = references("sm1d_q4", ladder)
    bt, mem = designed("sm1d_q4", ladder)
    assert [r["info"] for r in refs] == [expected_info(h) for _, _, h in mem]
    other = LADDERS["f32" if ladder == "f64" else "f64"]
    for b, (label, _, how) in enumerate(mem):
        if how in (2, 3):
            assert _oracle_at(bt, b, other)[2] != how, label


# ---------------------------------------------------------------------------------------------
# routes
# ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("model", list(MODELS))
def test_fused_engine_ladder(model, cuda_device):
    """ops.sm_mll_grad with and without the gradient and sm_mll_grad_alpha(staged=False): info is the
    designed code, NaN MLL / gradient / alpha for info < 0 (a NaN behind a failed pivot is -1), and
    every other member equals the oracle at its rung, alpha against (K~ + jit I)^-1 (y - c)."""
    from pgmuvi_b200 import ops
    bt, mem = designed(model, "f64")
    refs = references(model, "f64")
    args = _dev(bt, cuda_device)
    mll, grad, info = _np(ops.sm_mll_grad(*args, True))
    _check("fused", bt, mem, refs, mll, grad, info)
    m0, _, i0 = _np(ops.sm_mll_grad(*args, False))
    assert i0.tolist() == info.tolist()
    assert _same_bits(torch.tensor(m0), torch.tensor(mll))
    mll, grad, info, alpha = _np(ops.sm_mll_grad_alpha(*args, False))
    _check("fused, alpha", bt, mem, refs, mll, grad, info, alpha)


@pytest.mark.gpu
@pytest.mark.parametrize("model", list(MODELS))
def test_staged_engine_ladder_one_launch_and_nosync(model, cuda_device, monkeypatch):
    """The staged engine on the same batch (B * N < 1024: lg_chol_all and lg_inv_all), through
    sm_mll_grad_staged and sm_mll_grad_alpha(staged=True); with nosync=True, where all four ladder
    passes are enqueued without a host round trip, mll, grad and info are bitwise the synced call's.
    A batch that needs the panel schedule is refused under nosync."""
    from pgmuvi_b200 import _lib, ops
    bt, mem = designed(model, "f64")
    refs = references(model, "f64")
    args = _dev(bt, cuda_device)
    assert len(mem) * -(-N_MAX // TS) < 1024
    mll, grad, info = _staged(args, monkeypatch)
    _check("staged", bt, mem, refs, mll, grad, info)
    ms, gs, is_ = _np(ops.sm_mll_grad_staged(*args, True, nosync=True))
    torch.cuda.synchronize()
    assert is_.tolist() == info.tolist()
    assert _same_bits(torch.tensor(ms), torch.tensor(mll))
    assert _same_bits(torch.tensor(gs), torch.tensor(grad))
    mll, grad, info, alpha = _np(ops.sm_mll_grad_alpha(*args, True))
    _check("staged, alpha", bt, mem, refs, mll, grad, info, alpha)
    big = _dev(_tiled(bt, 160), cuda_device)
    with pytest.raises(_lib.EngineError, match="NOSYNC needs the one-launch schedule"):
        ops.sm_mll_grad_staged(*big, True, nosync=True)


def _tiled(bt, B):
    """B members cycling through bt's (B * 7 tile rows >= 1024 for B >= 147: the panel schedule)."""
    idx = np.arange(B) % len(bt["n_valid"])
    out = dict(bt)
    for k in ("x", "y", "noise", "raw", "lb", "ub", "n_valid"):
        out[k] = bt[k][idx]
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("model", list(MODELS))
def test_staged_engine_ladder_panel_schedules(model, cuda_device, monkeypatch):
    """The panel Cholesky: the batch repeated to B = 152 (B * N >= 1024, one panel), and the batch
    itself with the one-launch schedule turned off at panel widths 1, 2 and 3 (trailing updates
    between the failing pivots of neg_first, neg_mid and neg_last)."""
    bt, mem = designed(model, "f64")
    refs = references(model, "f64")
    k = len(mem)
    big = _tiled(bt, 152)
    mll, grad, info = _staged(_dev(big, cuda_device), monkeypatch)
    for c in range(0, 152, k):
        sl = slice(c, min(c + k, 152))
        n = sl.stop - sl.start
        _check(f"panel B=152, copy {c // k}", bt, mem[:n], refs[:n], mll[sl], grad[sl], info[sl])
    args = _dev(bt, cuda_device)
    for nb in (1, 2, 3):
        mll, grad, info = _staged(args, monkeypatch, nb=nb)
        _check(f"panel NB={nb}", bt, mem, refs, mll, grad, info)


def _tc_scale(bt, b, j1, info):
    """S_p = 1/(2n) sum_ij (|X|^T |X|)_ij |dK~_ij / draw_p| at the member's rung (X = L^-1)."""
    from oracle import constrain, kernel_dense, unpack_params
    from oracle.sm_gp import noise_diag
    x, y, nz, raw, kinds, lb, ub = _host(bt, b)
    spec, m = _spec(bt), len(y)
    jit = j1 * 10 ** (info - 1) if info > 0 else 0.0

    def K(r):
        th = constrain(r, kinds, lb, ub)
        noise = unpack_params(th, spec)[4]
        return kernel_dense(x, x, th, spec) + torch.diag_embed(noise_diag(m, nz, noise, x.dtype))
    L = torch.linalg.cholesky(K(raw) + jit * torch.eye(m, dtype=raw.dtype))
    X = torch.linalg.solve_triangular(L, torch.eye(m, dtype=L.dtype), upper=False)
    A = X.abs().T @ X.abs()
    return np.array([float((A * torch.func.jvp(K, (raw,), (e,))[1].abs()).sum()) / (2 * m)
                     for e in torch.eye(len(raw), dtype=raw.dtype)])


@pytest.mark.gpu
@pytest.mark.parametrize("model", list(MODELS))
def test_tcgen05_gradient_ladder(model, cuda_device, monkeypatch):
    """tf32x3=True: the same info codes and NaN members as the FP64 staged call, the MLL bitwise
    equal to it, and each jittered or healthy member's gradient within C_TC u S_p of it
    (test_gpu_schedules.py's bound, S_p at the member's rung)."""
    bt, mem = designed(model, "f64")
    refs = references(model, "f64")
    args = _dev(bt, cuda_device)
    m0, g0, i0 = _staged(args, monkeypatch)
    mll, grad, info = _staged(args, monkeypatch, tf32x3=True)
    assert info.tolist() == i0.tolist() == [r["info"] for r in refs]
    assert mll.view(np.int64).tolist() == m0.view(np.int64).tolist()
    for b, (label, _, how) in enumerate(mem):
        if info[b] < 0 or how == "nan_y":
            assert np.isnan(grad[b]).all(), label
            continue
        S = _tc_scale(bt, b, LADDERS["f64"], int(info[b]))
        dg = np.abs(grad[b] - g0[b])
        assert np.all(dg[S == 0] == 0), label
        assert np.all(dg[S > 0] <= C_TC * U * S[S > 0]), (label, (dg[S > 0] / (U * S[S > 0])).max())


@pytest.mark.gpu
@pytest.mark.parametrize("model", list(MODELS))
def test_prediction_ladder(model, cuda_device):
    """ops.sm_predict: mean and latent variance of every member with info >= 0 against oracle.predict
    at its rung; the failed members are NaN throughout.  The posterior part of the mean, K*^T alpha,
    is held to 1e-9 of its own largest value, and the variance k** - |L^-1 k*|^2 to 1e-9 of the prior
    variance k**: the members are scaled to ||K~|| = 1e4 jit(1), so a floor of 1 would be no bar, and
    the posterior variance itself (down to ~1e-9 at rung 1) is a difference of two terms of size
    k** whose rounding is set by k**."""
    from oracle import constrain
    from oracle.sm_gp import predict
    from pgmuvi_b200 import ops
    bt, mem = designed(model, "f64")
    refs = references(model, "f64")
    B, d, ms = len(mem), bt["x"].shape[2], 70
    rng = np.random.default_rng(3)
    xs = np.empty((B, ms, d))
    for b in range(B):
        xv = bt["x"][b, :int(bt["n_valid"][b])]
        lo, hi = np.nanmin(xv, 0), np.nanmax(xv, 0)
        xs[b] = lo + (hi - lo) * rng.uniform(0, 1, (ms, d))
    x, y, nz, raw, kinds, lb, ub, nv, *rest = _dev(bt, cuda_device)
    mean, var, info = _np(ops.sm_predict(x, y, nz, raw, kinds, lb, ub, nv,
                                         torch.tensor(xs, device=cuda_device), *rest))
    assert info.tolist() == [r["info"] for r in refs]
    for b, (label, _, how) in enumerate(mem):
        if info[b] < 0:
            assert np.isnan(mean[b]).all() and np.isnan(var[b]).all(), label
            continue
        if how == "nan_y":
            continue
        xh, yh, nzh, rawh, kh, lbh, ubh = _host(bt, b)
        rm, rv, ri = predict(xh, yh, nzh, rawh, kh, lbh, ubh, _spec(bt), torch.tensor(xs[b]),
                             jitter=LADDERS["f64"])
        assert int(ri) == info[b], label
        c = float(constrain(rawh, kh, lbh, ubh)[0])
        post = rm.numpy() - c
        assert np.abs((mean[b] - c) - post).max() <= 1e-9 * np.abs(post).max(), label
        kss = float(_ktilde(bt, b)[0].diagonal().max())         # stationary: k** = K_ii
        assert np.abs(var[b] - rv.numpy()).max() <= 1e-9 * kss, label


@pytest.mark.gpu
@pytest.mark.parametrize("model", list(MODELS))
def test_float32_entries_use_the_float32_ladder(model, cuda_device, monkeypatch):
    """The float32 entry points (PGM_FLAG_JITTER_F32) on the batch designed for the float32 ladder:
    info is the designed code for ops.sm_mll_grad and for sm_mll_grad_staged(tf32x3=True) (one-launch
    schedule); the fused values are the oracle's on the widened inputs to float32 rounding,
    |v32 - v| <= 2^-24 |v| + 1e-9 max(1, |v|) (gradient: of max |grad|)."""
    from pgmuvi_b200 import ops
    bt, mem = designed(model, "f32")
    refs = references(model, "f32")
    x, y, nz, raw, kinds, lb, ub, nv, *rest = _dev(bt, cuda_device)
    f = lambda t: t.float()
    args32 = (f(x), f(y), f(nz), f(raw), kinds, f(lb), f(ub), nv, *rest)
    mll, grad, info = _np(ops.sm_mll_grad(*args32, True))
    assert info.tolist() == [r["info"] for r in refs]
    for b, ((label, _, how), ref) in enumerate(zip(mem, refs)):
        if ref["info"] < 0 or how == "nan_y":
            assert np.isnan(mll[b]), label
            if ref["info"] < 0:
                assert np.isnan(grad[b]).all(), label
            continue
        v = ref["mll"]
        assert abs(float(mll[b]) - v) <= 2.0 ** -24 * abs(v) + 1e-9 * max(1.0, abs(v)), label
        gs = np.abs(ref["grad"]).max()
        assert np.abs(grad[b] - ref["grad"]).max() <= (2.0 ** -24 + GRAD_RTOL) * gs, label
    m2, g2, i2 = _staged(args32, monkeypatch, tf32x3=True)
    assert i2.tolist() == [r["info"] for r in refs]
    for b, ref in enumerate(refs):
        assert np.isnan(m2[b]) == np.isnan(mll[b]), mem[b][0]


@pytest.mark.gpu
@pytest.mark.parametrize("model", list(MODELS))
def test_float32_tcgen05_trailing_updates_ladder(model, cuda_device, monkeypatch):
    """The float32 batch through sm_mll_grad_staged(tf32x3=True, tf32x3_chol=True) with the panel
    schedule forced at NB = 2: the trailing updates at J1 = 2, 4, 6 run on tcgen05 (lg_update_tc),
    which builds K~ + jit of the trailing tiles on the float32 ladder.  info is the designed code on
    every member whose rung margin is at least 100 * 2^-21 ||K~||_2 (3xTF32 products are accurate to
    a few units of 2^-21 of ||K~||), and on every broken member; failed members are NaN."""
    from test_gpu_schedules import schedule
    bt, mem = designed(model, "f32")
    refs = references(model, "f32")
    j1 = LADDERS["f32"]
    assert schedule(len(mem), N_MAX, nb=2, chol_all_n=0, tf32x3=True, tf32x3_chol=True)[3] == (
        (2, "lg_update_tc"), (4, "lg_update_tc"), (6, "lg_update_tc"))
    checked = []
    for b, (label, _, how) in enumerate(mem):
        if isinstance(how, str) and how != "nan_y":
            checked.append(b)
            continue
        ev = np.linalg.eigvalsh(_ktilde(bt, b)[1].numpy())
        if rung_margin(refs[b]["info"], -ev[0], j1) >= 100 * 2.0 ** -21 * ev[-1]:
            checked.append(b)
    assert {2, 3, -2} <= {refs[b]["info"] for b in checked}
    x, y, nz, raw, kinds, lb, ub, nv, *rest = _dev(bt, cuda_device)
    f = lambda t: t.float()
    args32 = (f(x), f(y), f(nz), f(raw), kinds, f(lb), f(ub), nv, *rest)
    mll, grad, info = _staged(args32, monkeypatch, nb=2, tf32x3=True, tf32x3_chol=True)
    for b in checked:
        assert int(info[b]) == refs[b]["info"], (mem[b][0], int(info[b]), refs[b]["info"])
        if refs[b]["info"] < 0:
            assert np.isnan(mll[b]) and np.isnan(grad[b]).all(), mem[b][0]


@pytest.mark.gpu
@pytest.mark.parametrize("model", list(MODELS))
def test_failed_members_do_not_touch_their_neighbours(model, cuda_device, monkeypatch):
    """Each broken member swapped for a copy of the rung-0 member (same B, so the same schedule):
    every other member's mll, grad and info stay bitwise identical, fused and staged."""
    from pgmuvi_b200 import ops
    bt, mem = designed(model, "f64")
    swap = [b for b, (_, _, how) in enumerate(mem) if not isinstance(how, int) or how < 0]
    good = dict(bt)
    for k in ("x", "y", "noise", "raw", "lb", "ub", "n_valid"):
        good[k] = bt[k].copy()
        good[k][swap] = bt[k][0]
    keep = [b for b in range(len(mem)) if b not in swap]
    for fn in (lambda a: _np(ops.sm_mll_grad(*a, True)), lambda a: _staged(a, monkeypatch)):
        r1 = fn(_dev(bt, cuda_device))
        r2 = fn(_dev(good, cuda_device))
        for a1, a2 in zip(r1, r2):
            assert a1[keep].tobytes() == a2[keep].tobytes()


# ---------------------------------------------------------------------------------------------
# sm_fit through the ladder into a failure
# ---------------------------------------------------------------------------------------------
FIT_STEPS = 80
FIT_SCALE = {"f64": 1e-4, "f32": 1e-3}      # ||K~||_2 / jit(1) ~ 1.5e5 and 1.5e4


@lru_cache(maxsize=None)
def fit_case(ladder):
    """SM-5 with learned noise (no constraint), y = the mean so that alpha = 0 and d loss / d noise =
    tr K~^-1 / 2n > 0: Adam walks the noise down from rung 1 through rung 3 into -2 (lr = 10 jit(1):
    smaller steps shrink to a crawl once the first steps' large gradients are in Adam's second
    moment).
    Returns (batch, lr, oracle replay)."""
    from oracle import train_loop
    from oracle.sm_gp import CON_NONE
    kind, Q, _ = MODELS["sm1d_q5"]
    j1 = LADDERS[ladder]
    bt = _batch(kind, Q, True, [N_MAX - 2], N_MAX, seed0=41000)
    bt = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in bt.items()}
    spec = _spec(bt)
    bt["kinds"] = bt["kinds"].copy()
    bt["kinds"][spec.o_noise] = CON_NONE
    bt["raw"][0, spec.o_noise] = 0.0
    _scale(bt, 0, FIT_SCALE[ladder])
    lam = float(np.linalg.eigvalsh(_ktilde(bt, 0)[1].numpy())[0])
    lr = 10.0 * j1
    bt["raw"][0, spec.o_noise] = -lam - 0.5 * j1         # rung 1 at the start
    m = int(bt["n_valid"][0])
    bt["y"][0, :m] = float(bt["lb"][0, 0] + (bt["ub"][0, 0] - bt["lb"][0, 0]) / 2)   # raw mean 0
    if ladder == "f32":
        for k in ("x", "y", "noise", "raw", "lb", "ub"):
            bt[k] = bt[k].astype(np.float32).astype(np.float64)
    x, y, nz, raw, kinds, lb, ub = _host(bt, 0)
    ref = train_loop(x, y, nz, raw, kinds, lb, ub, spec, maxiter=FIT_STEPS, lr=lr, optim="Adam",
                     jitter=j1, on_failure="stop")
    # preconditions: two jittered rungs are passed, it ends in -2, and no iterate is within rounding
    # of a rung
    assert ref["info"][-1] == -2 and {1, 3} <= set(ref["info"]), ref["info"]
    for it, inf in enumerate(ref["info"]):
        b2 = dict(bt)
        b2["raw"] = ref["raw"][it][None]
        ev = np.linalg.eigvalsh(_ktilde(b2, 0)[1].numpy())
        assert rung_margin(inf, -ev[0], j1) >= 1e6 * m * U64 * ev[-1], (it, inf)
    return bt, lr, ref


@pytest.mark.gpu
@pytest.mark.parametrize("ladder", list(LADDERS))
def test_fit_stops_at_the_failing_evaluation(ladder, cuda_device):
    """ops.sm_fit (f64 on the f64 ladder, the f32 entry on the float32 ladder) against the oracle's
    replay that stops at the failed evaluation: loss and raw histories agree, n_iter is the failing
    iteration + 1, info is -2, the loss is NaN from the failing iteration on and raw is the iterate
    that failed."""
    from pgmuvi_b200 import _lib, ops
    bt, lr, ref = fit_case(ladder)
    x, y, nz, raw, kinds, lb, ub, nv, kind, Q, ln = _dev(bt, cuda_device)
    if ladder == "f32":
        x, y, nz, raw, lb, ub = (t.float() for t in (x, y, nz, raw, lb, ub))
    loss, hist, n_iter, info = ops.sm_fit(x, y, nz, raw, kinds, lb, ub, nv, kind, Q, ln,
                                          _lib.OPT_ADAM, lr, 0.9, 0.999, 1e-8, 0.0, FIT_STEPS, 0, 0.0,
                                          9, True)
    torch.cuda.synchronize()
    k = len(ref["loss"])                      # failing iteration + 1
    assert int(n_iter[0]) == k and int(info[0]) == -2
    loss, hist, raw = (t.double().cpu().numpy() for t in (loss, hist, raw))
    want = np.array(ref["loss"], dtype=float)
    assert np.isnan(loss[k - 1:, 0]).all()
    tol = (2.0 ** -24 if ladder == "f32" else 0.0) + 1e-9
    assert np.abs(loss[:k - 1, 0] - want[:-1]).max() <= tol * np.abs(want[:-1]).max()
    rh = np.stack(ref["raw"])
    rtol = 2.0 ** -24 if ladder == "f32" else 1e-12
    scale = np.maximum(np.abs(rh), 1.0)
    assert np.all(np.abs(hist[:k, 0] - rh) <= rtol * scale + 1e-3 * lr)
    assert np.all(np.abs(raw[0] - rh[-1]) <= rtol * scale[-1] + 1e-3 * lr)
