"""Generate tests/golden/*.npz from the oracle (run from the repo root:
``python -m oracle.make_golden``).

TEST INFRASTRUCTURE.  The reference holds no golden vectors for this path (SURVEY.md F5) and
GPyTorch is not installable here (F3), so these vectors are produced by the restated oracle
itself - they guard the oracle against drift and are what the CUDA path is compared with on
the GPU box (where /root/reference and the oracle's CPU time budget do not exist).  Each
file stores inputs, packed raw parameters, constraint table, and the oracle's outputs:
MLL, gradient by autograd AND by the closed form, K samples, three optimiser steps.
"""
from __future__ import annotations

import os

import numpy as np
import torch

from pgmuvi_b200 import synthetic as S

from .sm_gp import (ModelSpec, constrain, kernel_dense, mll_and_grad_analytic,
                    mll_and_grad_autograd, noise_diag, train_loop, unpack_params)

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests", "golden")

# name, generator kwargs
CASES = [
    ("sm1d_n40_q4", dict(dim=1, B=3, n=40, Q=4, learn_noise=False)),
    ("sm1d_n64_q4_learn", dict(dim=1, B=3, n=64, Q=4, learn_noise=True)),
    ("sm1d_n100_q1", dict(dim=1, B=3, n=100, Q=1, learn_noise=False)),
    ("sm1d_n100_q2_learn", dict(dim=1, B=3, n=100, Q=2, learn_noise=True)),
    ("sm1d_n100_q3_gauss", dict(dim=1, B=3, n=100, Q=3, learn_noise=True, fixed_noise=False)),
    ("sm1d_n100_q8", dict(dim=1, B=2, n=100, Q=8, learn_noise=False)),
    ("sm1d_n200_q4", dict(dim=1, B=3, n=200, Q=4, learn_noise=False)),
    ("sm1d_n512_q4", dict(dim=1, B=4, n=512, Q=4, learn_noise=False)),       # C2 shape
    ("sm1d_n512_q4_learn", dict(dim=1, B=2, n=512, Q=4, learn_noise=True)),
    ("sm2d_prodsum_4x48_q2_learn", dict(dim=2, kind=1, B=2, bands=4, per=48, Q=2, learn_noise=True)),
    ("sm2d_prodsum_4x48_q4", dict(dim=2, kind=1, B=2, bands=4, per=48, Q=4, learn_noise=False)),
    ("sm2d_sumprod_4x48_q4", dict(dim=2, kind=2, B=2, bands=4, per=48, Q=4, learn_noise=False)),
    ("sm2d_prodsum_4x256_q4", dict(dim=2, kind=1, B=1, bands=4, per=256, Q=4, learn_noise=False)),  # C5 shape
    ("sm1d_ragged_q4", dict(dim=1, B=4, n=200, Q=4, learn_noise=False, n_valid=[200, 130, 64, 77])),
    # separable SM(time) x wavelength kernel (gps.py:1274-1342), kinds 3..6
    ("sep_rbf_4x48_q4", dict(dim=2, kind=3, B=2, bands=4, per=48, Q=4, learn_noise=False)),
    ("sep_matern_4x48_q2_learn", dict(dim=2, kind=4, B=2, bands=4, per=48, Q=2, learn_noise=True)),
    ("sep_rq_4x48_q4", dict(dim=2, kind=5, B=2, bands=4, per=48, Q=4, learn_noise=False)),
    ("sep_const_3x40_q3_learn", dict(dim=2, kind=6, B=2, bands=3, per=40, Q=3, learn_noise=True)),
    ("sep_rbf_4x128_q8", dict(dim=2, kind=3, B=1, bands=4, per=128, Q=8, learn_noise=False)),
    # N3: stationary time kernels, kind = 8 + 5 * TK + WK (Q = 0)
    ("stat_rbf_1d_n100_learn", dict(dim=1, kind=8, B=2, n=100, Q=0, learn_noise=True)),
    ("stat_matern_1d_n150", dict(dim=1, kind=13, B=2, n=150, Q=0, learn_noise=False)),
    ("stat_matern_rbf_4x48", dict(dim=2, kind=14, B=2, bands=4, per=48, Q=0, learn_noise=False)),  # reference default 2DSeparable
    ("stat_rbf_rq_3x40_learn", dict(dim=2, kind=11, B=2, bands=3, per=40, Q=0, learn_noise=True)),
    ("stat_matern_const_4x32", dict(dim=2, kind=17, B=2, bands=4, per=32, Q=0, learn_noise=False)),
    ("stat_matern_matern_4x40", dict(dim=2, kind=15, B=1, bands=4, per=40, Q=0, learn_noise=False)),
    ("stat_qp_1d_n120_learn", dict(dim=1, kind=18, B=2, n=120, Q=0, learn_noise=True)),   # 1DQuasiPeriodic
    ("stat_qp_rbf_4x40", dict(dim=2, kind=19, B=2, bands=4, per=40, Q=0, learn_noise=False)),
    ("stat_qp_const_3x48_learn", dict(dim=2, kind=22, B=1, bands=3, per=48, Q=0, learn_noise=True)),
    ("stat_qp_plus_rbf_1d_n130", dict(dim=1, kind=23, B=2, n=130, Q=0, learn_noise=False)),  # 1DPeriodicStochastic
    ("stat_matern12_1d_n110_learn", dict(dim=1, kind=28, B=2, n=110, Q=0, learn_noise=True)),
    ("stat_matern25_1d_n140", dict(dim=1, kind=33, B=2, n=140, Q=0, learn_noise=False)),
    # ARD 2-D with one mixture (QT = 1) and sum-of-products with two (QT = 2)
    ("sm2d_prodsum_4x48_q1", dict(dim=2, kind=1, B=2, bands=4, per=48, Q=1, learn_noise=False)),
    ("sm2d_sumprod_4x48_q1", dict(dim=2, kind=2, B=2, bands=4, per=48, Q=1, learn_noise=False)),
    ("sm2d_sumprod_4x48_q2_learn", dict(dim=2, kind=2, B=2, bands=4, per=48, Q=2, learn_noise=True)),
    # ARD 2-D with QT = 8: one block per SM, full shared-memory layout; ragged down to n = 1
    ("sm2d_prodsum_3x64_q8", dict(dim=2, kind=1, B=2, bands=3, per=64, Q=8, learn_noise=False)),
    ("sm2d_sumprod_3x64_q6_learn", dict(dim=2, kind=2, B=3, bands=3, per=64, Q=6, learn_noise=True,
                                        n_valid=[192, 65, 1])),
    # padded mixtures inside QT = 8 (Q = 5 is the flicker term packed behind num_mixtures = 4)
    ("sm1d_n130_q5_learn", dict(dim=1, B=2, n=130, Q=5, learn_noise=True)),
    ("sep_rbf_3x40_q6_learn", dict(dim=2, kind=3, B=2, bands=3, per=40, Q=6, learn_noise=True)),
    ("sep_matern_4x48_q5", dict(dim=2, kind=4, B=2, bands=4, per=48, Q=5, learn_noise=False)),
    ("sep_rq_3x50_q8_learn", dict(dim=2, kind=5, B=2, bands=3, per=50, Q=8, learn_noise=True)),
    ("sep_rq_3x50_q7", dict(dim=2, kind=5, B=1, bands=3, per=50, Q=7, learn_noise=False)),
    ("sep_const_3x50_q7", dict(dim=2, kind=6, B=2, bands=3, per=50, Q=7, learn_noise=False)),
    # stationary time kernel x wavelength kernel: RBF x {RBF, Matern-1.5, Constant},
    # Matern-1.5 x RQ, quasi-periodic x {Matern-1.5, RQ}
    ("stat_rbf_rbf_3x40_learn", dict(dim=2, kind=9, B=2, bands=3, per=40, Q=0, learn_noise=True)),
    ("stat_rbf_matern_4x32", dict(dim=2, kind=10, B=2, bands=4, per=32, Q=0, learn_noise=False)),
    ("stat_rbf_const_3x48_learn", dict(dim=2, kind=12, B=2, bands=3, per=48, Q=0, learn_noise=True)),
    ("stat_matern_rq_4x40", dict(dim=2, kind=16, B=2, bands=4, per=40, Q=0, learn_noise=False)),
    ("stat_qp_matern_3x40_learn", dict(dim=2, kind=20, B=2, bands=3, per=40, Q=0, learn_noise=True)),
    ("stat_qp_rq_4x32", dict(dim=2, kind=21, B=2, bands=4, per=32, Q=0, learn_noise=False)),
]


def make_case(name, kw):
    kw = dict(kw)
    dim = kw.pop("dim")
    kind = kw.pop("kind", 0)
    n_valid = kw.pop("n_valid", None)
    if kind >= 8:
        bt = S.make_batch_stat(kw["B"], kind, n=kw.get("n"), n_bands=kw.get("bands"),
                               n_per_band=kw.get("per"), learn_noise=kw["learn_noise"])
    elif dim == 1:
        bt = S.make_batch_1d(kw["B"], kw["n"], Q=kw["Q"], learn_noise=kw["learn_noise"],
                             fixed_noise=kw.get("fixed_noise", True))
    elif kind >= 3:
        bt = S.make_batch_sep(kw["B"], kw["bands"], kw["per"], Q=kw["Q"], kind=kind,
                              learn_noise=kw["learn_noise"])
    else:
        bt = S.make_batch_2d(kw["B"], kw["bands"], kw["per"], Q=kw["Q"],
                             learn_noise=kw["learn_noise"])
    spec = ModelSpec(d=bt["d"], Q=bt["Q"], kind=kind, learn_noise=bt["learn_noise"])
    B = bt["x"].shape[0]
    n = bt["x"].shape[1]
    mll = np.zeros(B)
    g_auto = np.zeros((B, spec.P))
    g_ana = np.zeros((B, spec.P))
    info = np.zeros(B, dtype=np.int32)
    steps = np.zeros((B, 4, spec.P))
    losses = np.zeros((B, 3))
    kidx = np.stack([np.arange(0, n, max(1, n // 16))[:16]] * 2)  # sampled K rows/cols
    ksamp = np.zeros((B, kidx.shape[1], kidx.shape[1]))
    kinds = torch.tensor(bt["kinds"])
    for b in range(B):
        nb = n if n_valid is None else n_valid[b]
        x = torch.tensor(bt["x"][b][:nb])
        y = torch.tensor(bt["y"][b][:nb])
        nz = None if bt["noise"] is None else torch.tensor(bt["noise"][b][:nb])
        raw = torch.tensor(bt["raw"][b])
        lb, ub = torch.tensor(bt["lb"][b]), torch.tensor(bt["ub"][b])
        m1, g1, i1 = mll_and_grad_autograd(x, y, nz, raw, kinds, lb, ub, spec)
        m2, g2, i2 = mll_and_grad_analytic(x, y, nz, raw, kinds, lb, ub, spec)
        assert abs(float(m1) - float(m2)) <= 1e-12 * abs(float(m1)), name
        assert float((g1 - g2).abs().max()) <= 1e-9 * float(g1.abs().max()), name
        mll[b], g_auto[b], g_ana[b], info[b] = float(m1), g1.numpy(), g2.numpy(), int(i1)
        th = constrain(raw, kinds, lb, ub)
        mean, w, mu, sg, noise = unpack_params(th, spec)
        K = kernel_dense(x, x, th, spec) + torch.diag_embed(
            noise_diag(nb, nz, noise, y.dtype))
        ii = np.minimum(kidx[0], nb - 1)
        ksamp[b] = K[ii][:, ii].numpy()
        res = train_loop(x, y, nz, raw, kinds, lb, ub, spec, maxiter=3, miniter=3, stop=None,
                         lr=0.1, optim="AdamW")
        steps[b] = np.stack(res["raw"])
        losses[b] = np.array(res["loss"], dtype=float)
    out = dict(x=bt["x"], y=bt["y"], raw=bt["raw"], kinds=bt["kinds"], lb=bt["lb"], ub=bt["ub"],
               Q=bt["Q"], d=bt["d"], kind=kind, learn_noise=bt["learn_noise"], mll=mll,
               grad_autograd=g_auto, grad_analytic=g_ana, info=info, k_index=kidx[0],
               k_sample=ksamp, adamw_raw=steps, adamw_loss=losses)
    if bt["noise"] is not None:
        out["noise"] = bt["noise"]
    if n_valid is not None:
        out["n_valid"] = np.array(n_valid, dtype=np.int32)
    return out


def main():
    import sys
    os.makedirs(OUT, exist_ok=True)
    torch.set_default_dtype(torch.float64)
    only = sys.argv[1:]          # optional name prefixes: regenerate a subset
    for name, kw in CASES:
        if only and not any(name.startswith(o) for o in only):
            continue
        out = make_case(name, kw)
        # x / y / noise hold float32-representable values: store them as float32 to keep the
        # fixtures small (exactly recoverable); everything else float64.
        for k in ("x", "y", "noise"):
            if k in out:
                assert np.array_equal(out[k].astype(np.float32).astype(np.float64), out[k])
                out[k] = out[k].astype(np.float32)
        path = os.path.join(OUT, name + ".npz")
        np.savez_compressed(path, **out)
        print(f"{name}: mll={out['mll']}  {os.path.getsize(path) / 1024:.1f} KiB")


if __name__ == "__main__":
    main()
