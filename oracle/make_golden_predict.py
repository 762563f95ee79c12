"""Generate posterior predictions of the oracle (N1) for a few of the golden cases
(``python -m oracle.make_golden_predict [name ...]``; names regenerate a subset, as for
``oracle.make_golden``): name.npz in tests/golden_predict/ for the first six cases, in
tests/golden/predict/ for the later ones.  TEST INFRASTRUCTURE."""
from __future__ import annotations

import os

import numpy as np
import torch

from .sm_gp import ModelSpec, predict

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(HERE, "..", "tests", "golden")
OUT = os.path.join(GOLD, "predict")
OUT_FIRST = os.path.join(HERE, "..", "tests", "golden_predict")
CASES_FIRST = ["sm1d_n100_q2_learn", "sm1d_n200_q4", "sm1d_ragged_q4", "sm2d_prodsum_4x48_q4",
               "sep_rq_4x48_q4", "sep_const_3x40_q3_learn"]
CASES = CASES_FIRST + ["sm2d_prodsum_3x64_q8", "sep_matern_4x48_q5", "sm1d_n130_q5_learn",
                       "stat_qp_rq_4x32"]
M = 150   # test points per light curve (not a multiple of 64: ragged last test tile)


def main():
    import sys
    torch.set_default_dtype(torch.float64)
    os.makedirs(OUT, exist_ok=True)
    os.makedirs(OUT_FIRST, exist_ok=True)
    only = sys.argv[1:]          # optional name prefixes: regenerate a subset
    for name in CASES:
        if only and not any(name.startswith(o) for o in only):
            continue
        g = np.load(os.path.join(GOLD, name + ".npz"))
        B, n, d = g["x"].shape
        spec = ModelSpec(d=int(g["d"]), Q=int(g["Q"]), kind=int(g["kind"]),
                         learn_noise=bool(g["learn_noise"]))
        rng = np.random.default_rng(123)
        xs = np.zeros((B, M, d))
        mean = np.zeros((B, M))
        var = np.zeros((B, M))
        for b in range(B):
            nb = int(g["n_valid"][b]) if "n_valid" in g.files else n
            x = torch.tensor(g["x"][b][:nb].astype(np.float64))
            # test grid: slightly beyond the training span; 2-D: random training wavelengths
            xs[b, :, 0] = np.linspace(-0.05, 1.05, M)
            if d == 2:
                xs[b, :, 1] = rng.choice(np.unique(g["x"][b][:nb, 1]), M)
            lb = g["lb"][b] if g["lb"].ndim == 2 else g["lb"]
            ub = g["ub"][b] if g["ub"].ndim == 2 else g["ub"]
            mu, vv, info = predict(x, torch.tensor(g["y"][b][:nb].astype(np.float64)),
                                   torch.tensor(g["noise"][b][:nb].astype(np.float64)) if "noise" in g.files else None,
                                   torch.tensor(g["raw"][b]), torch.tensor(g["kinds"]),
                                   torch.tensor(lb), torch.tensor(ub), spec, torch.tensor(xs[b]))
            assert int(info) == 0
            mean[b], var[b] = mu.numpy(), vv.numpy()
        out = OUT_FIRST if name in CASES_FIRST else OUT
        np.savez_compressed(os.path.join(out, name + ".npz"), xstar=xs, mean=mean, var=var)
        print(name, mean[0, :3], var[0, :3])


if __name__ == "__main__":
    main()
