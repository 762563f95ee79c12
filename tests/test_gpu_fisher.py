"""GPU: the Fisher information of pgm_sm_fisher_f64 against the fp64 oracle (oracle/fisher.py) on
every golden (which together reach every compiled instantiation), ragged tile edges, chunked and
mixed batches (a jittered and a failing light curve), one n ~ 2000 single GP, and opcheck."""
import numpy as np
import pytest
import torch

from conftest import golden_names, load_golden
from oracle import ModelSpec, constrain
from oracle.fisher import fisher as oracle_fisher

pytestmark = pytest.mark.gpu

TOL = 1e-10


def _dev(g, dev):
    t = lambda a, dt=torch.float64: None if a is None else torch.tensor(a, dtype=dt, device=dev)
    return dict(x=t(g["x"]), y=t(g["y"]), noise=t(g["noise"]), raw=t(g["raw"]),
                kinds=t(g["kinds"], torch.int32), lb=t(g["lb"]), ub=t(g["ub"]),
                n_valid=t(g["n_valid"], torch.int32))


def _oracle(g, b):
    spec = ModelSpec(d=int(g["d"]), Q=int(g["Q"]), kind=int(g["kind"]),
                     learn_noise=bool(g["learn_noise"]))
    n = g["x"].shape[1] if g["n_valid"] is None else int(g["n_valid"][b])
    lb = g["lb"][b] if np.ndim(g["lb"]) == 2 else g["lb"]
    ub = g["ub"][b] if np.ndim(g["ub"]) == 2 else g["ub"]
    theta = constrain(torch.tensor(g["raw"][b]), torch.tensor(g["kinds"]), torch.tensor(lb),
                      torch.tensor(ub))
    fn = None if g["noise"] is None else torch.tensor(g["noise"][b, :n])
    return oracle_fisher(torch.tensor(g["x"][b, :n]), fn, theta, spec)


def _compare(F, R, tol=TOL):
    """Correlation form: diagonal relative error and off-diagonal error scaled by sqrt(F_pp F_qq)."""
    dg = np.abs(np.diag(R))
    nz = dg > 0
    rel = np.abs(np.diag(F) - np.diag(R))[nz] / dg[nz]
    assert rel.max() <= tol, rel.max()
    sc = np.sqrt(np.outer(dg, dg))
    m = np.outer(nz, nz)
    assert (np.abs(F - R)[m] / sc[m]).max() <= tol
    assert np.abs(F[~m] - R[~m]).max(initial=0.0) <= tol * max(dg.max(), 1.0)


def _run(ops, g, d):
    F, info = ops.sm_fisher(d["x"], d["y"], d["noise"], d["raw"], d["kinds"], d["lb"], d["ub"],
                            d["n_valid"], int(g["kind"]), int(g["Q"]), bool(g["learn_noise"]))
    return F.cpu().numpy(), info.cpu().numpy()


@pytest.mark.parametrize("name", golden_names())
def test_fisher_matches_the_oracle_on_goldens(name, cuda_device):
    from pgmuvi_b200 import ops
    g = load_golden(name)
    F, info = _run(ops, g, _dev(g, cuda_device))
    assert np.array_equal(info, g["info"])
    for b in range(F.shape[0]):
        R, ri = _oracle(g, b)
        assert ri == info[b]
        if ri < 0:
            assert np.isnan(F[b]).all()
        else:
            _compare(F[b], R.numpy())


def _synthetic(B, ns, Q=2, seed=0, learn_noise=False):
    rng = np.random.default_rng(seed)
    n_max = max(ns)
    x = np.zeros((B, n_max, 1))
    y = np.zeros((B, n_max))
    noise = np.ones((B, n_max))
    for b, n in enumerate(ns):
        x[b, :n, 0] = np.sort(rng.uniform(0.0, 1.0, n))
        y[b, :n] = np.sin(2 * np.pi * 7 * x[b, :n, 0]) + 0.1 * rng.standard_normal(n)
        noise[b, :n] = 0.01
    P = 1 + 3 * Q + (1 if learn_noise else 0)
    kinds = np.array([0] + [1] * (P - 1), dtype=np.int32)
    raw = np.zeros((B, P))
    raw[:, 0] = 0.1
    raw[:, 1:1 + Q] = rng.uniform(-1.0, 0.0, (B, Q))
    raw[:, 1 + Q:1 + 2 * Q] = np.log(np.expm1(rng.uniform(3.0, 9.0, (B, Q))))
    raw[:, 1 + 2 * Q:1 + 3 * Q] = np.log(np.expm1(rng.uniform(0.5, 2.0, (B, Q))))
    if learn_noise:
        raw[:, -1] = -4.0
    return dict(x=x, y=y, noise=None if learn_noise else noise, raw=raw, kinds=kinds,
                lb=np.zeros(P), ub=np.zeros(P), n_valid=np.array(ns, dtype=np.int32),
                kind=0, Q=Q, d=1, learn_noise=learn_noise)


@pytest.mark.parametrize("n", [1, 63, 64, 65, 128, 129])
def test_tile_edges_and_ragged_batches(n, cuda_device):
    from pgmuvi_b200 import ops
    ns = [n, max(1, n - 1), n + 1 if n < 129 else 70]
    g = _synthetic(3, ns, seed=n, learn_noise=(n % 2 == 1))
    F, info = _run(ops, g, _dev(g, cuda_device))
    for b in range(3):
        R, ri = _oracle(g, b)
        assert ri == info[b]
        _compare(F[b], R.numpy())


def test_chunked_batch_with_jittered_and_failing_members(cuda_device):
    """uncertainties-style chunking through the op: a forced small budget gives several launches;
    member 1 needs a jitter rung (duplicated input, no noise) and member 2 has a NaN input."""
    from pgmuvi_b200 import ops
    g = _synthetic(7, [90, 75, 60, 90, 33, 80, 64], seed=3)
    g["noise"][1, :] = 0.0
    g["x"][1, 1, 0] = g["x"][1, 0, 0]
    g["x"][2, 5, 0] = np.nan
    d = _dev(g, cuda_device)
    whole, info = _run(ops, g, d)
    assert info[1] >= 1 and info[2] == -1
    assert np.isnan(whole[2]).all()
    for b in range(7):
        R, ri = _oracle(g, b)
        assert ri == info[b]
        if ri >= 0:
            _compare(whole[b], R.numpy(), 1e-4 if ri > 0 else TOL)   # rung 1: cond(K~) ~ 1e10
    # chunks of 3 light curves give the same bytes as the whole batch
    for a in range(0, 7, 3):
        sl = {k: (v[a:a + 3] if (v is not None and k not in ("kinds", "lb", "ub")) else v)
              for k, v in d.items()}
        F, i = ops.sm_fisher(sl["x"], sl["y"], sl["noise"], sl["raw"], sl["kinds"], sl["lb"],
                             sl["ub"], sl["n_valid"], 0, 2, False)
        assert np.array_equal(i.cpu().numpy(), info[a:a + 3])
        np.testing.assert_array_equal(F.cpu().numpy(), whole[a:a + 3])


def test_single_gp_n2000(cuda_device):
    from pgmuvi_b200 import ops
    g = _synthetic(1, [2000], Q=4, seed=11)
    F, info = _run(ops, g, _dev(g, cuda_device))
    R, ri = _oracle(g, 0)
    assert ri == info[0] == 0
    _compare(F[0], R.numpy(), 1e-9)


def test_opcheck(cuda_device):
    from pgmuvi_b200 import ops
    g = _synthetic(2, [40, 33], seed=5)
    d = _dev(g, cuda_device)
    torch.library.opcheck(torch.ops.pgmuvi_b200.sm_fisher.default,
                          (d["x"], d["y"], d["noise"], d["raw"], d["kinds"], d["lb"], d["ub"],
                           d["n_valid"], 0, 2, False))
