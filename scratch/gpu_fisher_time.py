"""Fisher information (pgm_sm_fisher_f64) times with CUDA events: C1 (AlfOri, n = 1000 SM-4, learned
noise), a 4096 x n = 512 SM-4 batch (two launches of 2048 light curves) and C3 (n = 8000, 2-D SM-4).
Prints the card and its power limit, and the achieved rate of the Fisher products (the tile products
of fs_xc + fs_xcx, 2 * 64^3 flops each) over the WHOLE call (P and T phases included), against the
self-measured DMMA peak."""
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from pgmuvi_b200 import ops  # noqa: E402

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
dev = torch.device("cuda:0")
print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                     capture_output=True, text=True).stdout.strip(), flush=True)
peak = ops.peak_probe(0)
print(f"DMMA peak (self-measured): {peak:.1f} TFLOP/s", flush=True)


def product_flops(n, nc):
    N = (n + 63) // 64
    tiles = sum((i + 1) + (j + 1) for i in range(N) for j in range(i + 1))
    return nc * tiles * 2.0 * 64 ** 3


def timed(args, chunks=1, reps=3):
    t = lambda a, dt=torch.float64: None if a is None else torch.as_tensor(a, dtype=dt).to(dev)
    x, y, noise, raw, kinds, lb, ub, kind, Q, learn = args
    B = x.shape[0]
    parts = [(a, min(B, a + (B + chunks - 1) // chunks)) for a in range(0, B, (B + chunks - 1) // chunks)]
    dx = [tuple(t(v[a:z]) if v is not None else None for v in (x, y, noise, raw)) for a, z in parts]
    best = 1e30
    for rep in range(reps + 1):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for (xx, yy, nn, rr) in dx:
            F, info = ops.sm_fisher(xx, yy, nn, rr, t(kinds, torch.int32), t(lb), t(ub), None, kind, Q,
                                    learn)
            del F
        e1.record()
        torch.cuda.synchronize()
        if rep > 0:
            best = min(best, e0.elapsed_time(e1) / 1e3)
    return best, info


# C1
z = np.load(os.path.join(ROOT, "tests", "golden_c1", "alfori_adam300.npz"))
c1 = (z["x"][None], z["y"][None], None, z["raw_final"][None], z["kinds"], z["lb"], z["ub"], 0, 4, True)
s, info = timed(c1)
fl = product_flops(1000, 13)
print(f"C1 n=1000 SM-4: {s * 1e3:.2f} ms  {fl / s / 1e12:.2f} TFLOP/s ({fl / s / 1e12 / peak:.3f} of peak)"
      f"  info {info.tolist()}", flush=True)

# 4096 x n = 512 SM-4 (fixed noise)
rng = np.random.default_rng(0)
B, n = 4096, 512
x = np.sort(rng.uniform(0, 1, (B, n)), 1)[..., None]
y = np.sin(2 * np.pi * 9 * x[..., 0]) + 0.1 * rng.standard_normal((B, n))
raw = np.zeros((B, 13))
raw[:, 1:5] = rng.uniform(-1, 0, (B, 4))
raw[:, 5:9] = np.log(np.expm1(rng.uniform(2, 20, (B, 4))))
raw[:, 9:13] = np.log(np.expm1(rng.uniform(0.3, 2, (B, 4))))
kinds = np.array([0] + [1] * 12, dtype=np.int32)
bat = (x, y, np.full((B, n), 0.01), raw, kinds, np.zeros(13), np.zeros(13), 0, 4, False)
s, info = timed(bat, chunks=2, reps=2)
fl = B * product_flops(n, 12)
print(f"4096 x n=512 SM-4 (2 launches of 2048): {s:.3f} s  {fl / s / 1e12:.2f} TFLOP/s "
      f"({fl / s / 1e12 / peak:.3f} of peak)", flush=True)

# C3
z = np.load(os.path.join(ROOT, "tests", "golden_large", "c3_2d_8x1000_q4.npz"))
c3 = (z["x"][None], z["y"][None], z["noise"][None], z["raw"][None], z["kinds"], z["lb"], z["ub"],
      int(z["kind"]), int(z["Q"]), bool(z["learn_noise"]))
s, info = timed(c3, reps=2)
fl = product_flops(8000, 20)
print(f"C3 n=8000 2-D SM-4: {s:.3f} s  {fl / s / 1e12:.2f} TFLOP/s ({fl / s / 1e12 / peak:.3f} of peak)"
      f"  info {info.tolist()}", flush=True)
