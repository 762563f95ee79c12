"""Seeded synthetic light curves for the benchmark configs (numpy only).

Mimics the reference's generators (pgmuvi/synthetic.py: irregular sampling
``sort(U(0, t_span))`` :160-161, default span factor 2.3 :76, multi-sinusoid signal
:385-500, Gaussian noise ``_apply_noise`` :236-300) without importing pgmuvi (whose import
needs gpytorch/matplotlib).  Shapes follow BASELINE.json configs C2..C5 / SURVEY.md 8(d).

Everything here is host-side data preparation; the default constraints restate
``Lightcurve.set_default_constraints`` (pgmuvi/lightcurve.py:3817-3932).
"""
from __future__ import annotations

import math

import numpy as np

from ._lib import KIND_STAT_BASE, NUM_LAM, param_count, stat_num_lam

# constraint kinds - must match include/pgmuvi_b200.h
CON_NONE, CON_SOFTPLUS, CON_INTERVAL = 0, 1, 2


def inv_softplus(v):
    v = np.asarray(v, dtype=np.float64)
    return np.where(v > 30, v, v + np.log(-np.expm1(-np.maximum(v, 1e-300))))


def logit(u):
    u = np.asarray(u, dtype=np.float64)
    return np.log(u) - np.log1p(-u)


def fixed_noise_variance(yerr):
    """yerr -> variance as the reference forms it: float32 ``yerr ** 2``
    (lightcurve.py:2780-2784), clamped to GPyTorch's fp64 ``min_fixed_noise`` 1e-6."""
    v = (np.asarray(yerr, dtype=np.float32) ** 2).astype(np.float64)
    return np.maximum(v, 1e-6)


def default_constraints(x, y, yerr, Q, d, learn_noise):
    """kinds [P], lb [P], ub [P] as `fit()` would register them.

    mean: Interval(min y, max y) (:3830-3838); weights/scales: Positive (SMK defaults);
    means: 1D GreaterThan(1/span) (:3920-3932), 2D Interval(1/span_t, 1/(2 min dt))
    (:3883-3906); learned noise: Interval(noise_min, std y) (:3817-3829).
    """
    P = param_count(Q, d, learn_noise)
    kinds = np.full(P, CON_SOFTPLUS, dtype=np.int32)
    lb = np.zeros(P)
    ub = np.zeros(P)
    kinds[0] = CON_INTERVAL
    lb[0], ub[0] = float(y.min()), float(y.max())
    o_mu = 1 + Q
    t = x[:, 0] if x.ndim == 2 else x
    span = float(t.max() - t.min())
    if d == 1:
        lb[o_mu:o_mu + Q] = 1.0 / span
    else:
        ts = np.sort(t)
        dt = np.diff(ts)
        dt = dt[dt > 0]
        kinds[o_mu:o_mu + Q * d] = CON_INTERVAL
        lb[o_mu:o_mu + Q * d] = 1.0 / span
        ub[o_mu:o_mu + Q * d] = 1.0 / (2.0 * float(dt.min()))
    if learn_noise:
        kinds[P - 1] = CON_INTERVAL
        ystd = float(np.std(y, ddof=1))  # torch.std default is unbiased
        if yerr is not None:
            lb[P - 1] = min(1e-4, float(yerr.min()) / 10.0)
        else:
            lb[P - 1] = 1e-4 * ystd
        ub[P - 1] = ystd
    return kinds, lb, ub


def make_lightcurve_1d(seed, n, noise_sigma=0.1):
    """One irregularly sampled two-sinusoid light curve, min-max scaled to [0, 1].

    Returns t01 [n], y [n], yerr [n], (P_true, span) - float64 holding float32-rounded
    values (the reference stores float32, lightcurve.py:2434-2446; fp64 runs upcast them).
    """
    rng = np.random.default_rng(seed)
    period = rng.uniform(30.0, 300.0)
    k = rng.uniform(1.3, 4.0)
    t = np.sort(rng.uniform(0.0, 2.3 * period * k, n))
    y = np.sin(2 * np.pi * t / period) + 0.5 * np.sin(2 * np.pi * t / (0.44 * period) + 1.3)
    y = y + noise_sigma * rng.standard_normal(n)
    span = t.max() - t.min()
    t01 = (t - t.min()) / span
    t01 = t01.astype(np.float32).astype(np.float64)
    y = y.astype(np.float32).astype(np.float64)
    yerr = np.full(n, noise_sigma, dtype=np.float32).astype(np.float64)
    return t01, y, yerr, (period, span)


def make_batch_1d(B, n, Q=4, learn_noise=False, fixed_noise=True, seed0=1000):
    """BASELINE config C2: B independent 1-D light curves of n points, SM-Q.

    Returns a dict of float64 numpy arrays: x [B,n,1], y [B,n], noise [B,n] (variance;
    None if not fixed_noise), raw [B,P], kinds [P], lb [B,P], ub [B,P], and 'periods' [B].
    Initial hyper-parameters (fixed across reference/oracle/engine): weights std(y)/Q;
    means near the true frequencies and a harmonic/sub-harmonic (as an LS init would give,
    lightcurve.py:5475-5653); scales U(0.5, 5) in 1/[0,1] units; mean raw 0; noise raw 0.
    """
    d = 1
    P = param_count(Q, d, learn_noise)
    x = np.zeros((B, n, 1))
    y = np.zeros((B, n))
    noise = np.zeros((B, n)) if fixed_noise else None
    raw = np.zeros((B, P))
    lb = np.zeros((B, P))
    ub = np.zeros((B, P))
    periods = np.zeros(B)
    kinds = None
    for b in range(B):
        t01, yy, yerr, (period, span) = make_lightcurve_1d(seed0 + b, n)
        rng = np.random.default_rng(10_000_000 + seed0 + b)
        x[b, :, 0] = t01
        y[b] = yy
        if fixed_noise:
            noise[b] = fixed_noise_variance(yerr)
        kinds, lbb, ubb = default_constraints(t01, yy, yerr if fixed_noise else None, Q, d,
                                              learn_noise)
        lb[b], ub[b] = lbb, ubb
        periods[b] = period
        f1 = span / period
        f2 = span / (0.44 * period)
        base = np.array([f1, f2, 2.0 * f1, 0.5 * f1, 3.0 * f1, 0.5 * f2, 2.0 * f2, 1.5 * f1])
        mu = base[np.arange(Q) % len(base)] * (1.0 + 0.05 * rng.standard_normal(Q))
        mu = np.maximum(mu, lbb[1 + Q] + 0.05)
        sig = rng.uniform(0.5, 5.0, Q)
        wv = np.full(Q, np.std(yy, ddof=1) / Q)
        raw[b, 0] = 0.0
        raw[b, 1:1 + Q] = inv_softplus(wv)
        raw[b, 1 + Q:1 + 2 * Q] = inv_softplus(mu - lbb[1 + Q:1 + 2 * Q])
        raw[b, 1 + 2 * Q:1 + 3 * Q] = inv_softplus(sig)
        if learn_noise:
            raw[b, P - 1] = 0.0
    return dict(x=x, y=y, noise=noise, raw=raw, kinds=kinds, lb=lb, ub=ub, periods=periods,
                Q=Q, d=d, learn_noise=learn_noise)


def make_lightcurve_2d(seed, n_bands, n_per_band, noise_sigma=0.05):
    """Chromatic sinusoid on (time, wavelength), rows concatenated band by band as the
    reference does (synthetic.py:656-683); both columns min-max scaled."""
    rng = np.random.default_rng(seed)
    period = rng.uniform(100.0, 600.0)
    t_span = 2.3 * period * rng.uniform(1.0, 2.0)
    wl = np.linspace(0.45, 2.2, n_bands)
    xs, ys = [], []
    for b in range(n_bands):
        t = np.sort(rng.uniform(0.0, t_span, n_per_band))
        amp = 1.0 * math.exp(-0.6 * wl[b] ** -1.0) + 0.3
        ph = 0.1 * wl[b]
        f = amp * np.sin(2 * np.pi * t / period + ph) + noise_sigma * rng.standard_normal(n_per_band)
        xs.append(np.stack([t, np.full(n_per_band, wl[b])], 1))
        ys.append(f)
    x = np.concatenate(xs, 0)
    y = np.concatenate(ys, 0)
    mn, rg = x.min(0), x.max(0) - x.min(0)
    x01 = ((x - mn) / rg).astype(np.float32).astype(np.float64)
    y = y.astype(np.float32).astype(np.float64)
    yerr = np.full(len(y), noise_sigma, dtype=np.float32).astype(np.float64)
    return x01, y, yerr, (period, rg[0])


def make_batch_2d(B, n_bands, n_per_band, Q=4, learn_noise=False, seed0=5000):
    """BASELINE configs C3 / C5: 2-D (time, wavelength) SM-Q light curves, FixedNoise."""
    d = 2
    n = n_bands * n_per_band
    P = param_count(Q, d, learn_noise)
    x = np.zeros((B, n, 2))
    y = np.zeros((B, n))
    noise = np.zeros((B, n))
    raw = np.zeros((B, P))
    lb = np.zeros((B, P))
    ub = np.zeros((B, P))
    periods = np.zeros(B)
    kinds = None
    for b in range(B):
        x01, yy, yerr, (period, span) = make_lightcurve_2d(seed0 + b, n_bands, n_per_band)
        rng = np.random.default_rng(20_000_000 + seed0 + b)
        x[b], y[b] = x01, yy
        noise[b] = fixed_noise_variance(yerr)
        kinds, lbb, ubb = default_constraints(x01, yy, yerr, Q, d, learn_noise)
        lb[b], ub[b] = lbb, ubb
        periods[b] = period
        f1 = span / period
        o_mu, o_sg = 1 + Q, 1 + Q + Q * d
        mu = np.zeros((Q, d))
        mu[:, 0] = f1 * np.array([1.0, 2.0, 0.5, 3.0, 1.5, 4.0, 0.75, 2.5])[np.arange(Q) % 8] \
            * (1.0 + 0.05 * rng.standard_normal(Q))
        mu[:, 1] = lbb[o_mu] + rng.uniform(0.05, 0.5, Q)
        mu = np.clip(mu, lbb[o_mu] * 1.0001 + 1e-6, ubb[o_mu] * 0.9999)
        sig = rng.uniform(0.3, 2.0, (Q, d))
        wv = np.full(Q, math.sqrt(np.std(yy, ddof=1) / Q))
        raw[b, 1:1 + Q] = inv_softplus(wv)
        raw[b, o_mu:o_mu + Q * d] = logit((mu.ravel() - lbb[o_mu:o_mu + Q * d])
                                          / (ubb[o_mu:o_mu + Q * d] - lbb[o_mu:o_mu + Q * d]))
        raw[b, o_sg:o_sg + Q * d] = inv_softplus(sig.ravel())
    return dict(x=x, y=y, noise=noise, raw=raw, kinds=kinds, lb=lb, ub=ub, periods=periods,
                Q=Q, d=d, learn_noise=learn_noise)


def make_batch_sep(B, n_bands, n_per_band, Q=4, kind=3, learn_noise=False, seed0=7000):
    """Separable models (pgmuvi/gps.py:1274-1342): SM-Q in time x {RBF, Matern-1.5, RQ,
    Constant} in wavelength on the 2-D synthetic light curves of :func:`make_batch_2d`.
    Constraints: mean Interval(min y, max y); SM means GreaterThan(1/span) as for the 1-D
    model; everything else GPyTorch's default Positive; learned noise Interval."""
    n = n_bands * n_per_band
    P = param_count(Q, 2, learn_noise, kind)
    NL = NUM_LAM[kind]
    o_mu, o_sg, o_noise = 1 + Q, 1 + 2 * Q, 1 + 3 * Q
    o_lam = o_noise + (1 if learn_noise else 0)
    x = np.zeros((B, n, 2))
    y = np.zeros((B, n))
    noise = np.zeros((B, n))
    raw = np.zeros((B, P))
    lb = np.zeros((B, P))
    ub = np.zeros((B, P))
    kinds = np.full(P, CON_SOFTPLUS, dtype=np.int32)
    kinds[0] = CON_INTERVAL
    if learn_noise:
        kinds[o_noise] = CON_INTERVAL
    for b in range(B):
        x01, yy, yerr, (period, span) = make_lightcurve_2d(seed0 + b, n_bands, n_per_band)
        rng = np.random.default_rng(30_000_000 + seed0 + b)
        x[b], y[b] = x01, yy
        noise[b] = fixed_noise_variance(yerr)
        lb[b, 0], ub[b, 0] = float(yy.min()), float(yy.max())
        tspan = float(x01[:, 0].max() - x01[:, 0].min())
        lb[b, o_mu:o_mu + Q] = 1.0 / tspan
        f1 = span / period
        mu = f1 * np.array([1.0, 2.0, 0.5, 3.0, 1.5, 4.0, 0.75, 2.5])[np.arange(Q) % 8] \
            * (1.0 + 0.05 * rng.standard_normal(Q))
        mu = np.maximum(mu, lb[b, o_mu] * 1.01 + 1e-3)
        sig = rng.uniform(0.3, 2.0, Q)
        wv = np.full(Q, np.std(yy, ddof=1) / Q)
        raw[b, 1:1 + Q] = inv_softplus(wv)
        raw[b, o_mu:o_mu + Q] = inv_softplus(mu - lb[b, o_mu])
        raw[b, o_sg:o_sg + Q] = inv_softplus(sig)
        if learn_noise:
            ystd = float(np.std(yy, ddof=1))
            lb[b, o_noise], ub[b, o_noise] = min(1e-4, float(yerr.min()) / 10.0), ystd
        lamv = [rng.uniform(0.6, 1.5)]                       # outputscale / constant
        if NL >= 2:
            lamv.append(rng.uniform(0.3, 1.2))               # lengthscale (x in [0, 1])
        if NL >= 3:
            lamv.append(rng.uniform(0.5, 3.0))               # RQ alpha
        raw[b, o_lam:o_lam + NL] = inv_softplus(np.array(lamv))
    return dict(x=x, y=y, noise=noise, raw=raw, kinds=kinds, lb=lb, ub=ub, Q=Q, d=2,
                kind=kind, learn_noise=learn_noise)


def make_batch_stat(B, kind, n=None, n_bands=None, n_per_band=None, learn_noise=False, seed0=9000):
    """N3: stationary time kernels (ScaleKernel(RBF | Matern-1.5) in time, optionally x a
    wavelength kernel; pgmuvi/gps.py:985-990, 1131-1184, 1316-1319) on the 1-D / 2-D synthetic
    light curves.  kind = 8 + 5 * TK + WK, Q = 0; packed [mean | (noise) | os_t, l_t | wavelength
    parameters]; GPyTorch's default Positive constraints, mean / learned noise Interval."""
    tk, wk = divmod(kind - KIND_STAT_BASE, 5)
    d = 1 if wk == 0 else 2
    NL = stat_num_lam(kind)
    P = param_count(0, d, learn_noise, kind)
    o_noise = 1
    o_lam = 1 + (1 if learn_noise else 0)
    npts = n if d == 1 else n_bands * n_per_band
    x = np.zeros((B, npts, d))
    y = np.zeros((B, npts))
    noise = np.zeros((B, npts))
    raw = np.zeros((B, P))
    lb = np.zeros((B, P))
    ub = np.zeros((B, P))
    kinds = np.full(P, CON_SOFTPLUS, dtype=np.int32)
    kinds[0] = CON_INTERVAL
    if learn_noise:
        kinds[o_noise] = CON_INTERVAL
    for b in range(B):
        rng = np.random.default_rng(40_000_000 + seed0 + b)
        if d == 1:
            bt = make_batch_1d(1, npts, Q=1, seed0=seed0 + b)
            x[b], yy, noise[b] = bt["x"][0], bt["y"][0], bt["noise"][0]
            yerr = np.sqrt(bt["noise"][0])
        else:
            x01, yy, yerr, _ = make_lightcurve_2d(seed0 + b, n_bands, n_per_band)
            x[b] = x01
            noise[b] = fixed_noise_variance(yerr)
        y[b] = yy
        lb[b, 0], ub[b, 0] = float(yy.min()), float(yy.max())
        if learn_noise:
            lb[b, o_noise], ub[b, o_noise] = min(1e-4, float(yerr.min()) / 10.0), float(np.std(yy, ddof=1))
        if tk in (2, 3):    # quasi-periodic: os, lambda (periodic lengthscale), period, l_rbf
            lamv = [rng.uniform(0.5, 1.5), rng.uniform(0.5, 2.0), rng.uniform(0.08, 0.3),
                    rng.uniform(0.3, 1.0)]
            if tk == 3:                                              # + os_2, l_2 (stochastic RBF)
                lamv += [rng.uniform(0.1, 0.6), rng.uniform(0.02, 0.1)]
        else:
            lamv = [rng.uniform(0.5, 1.5), rng.uniform(0.03, 0.2)]   # os_t, l_t (x in [0, 1])
        if wk in (1, 2, 3):
            lamv += [rng.uniform(0.6, 1.5), rng.uniform(0.3, 1.2)]   # os_w, l_w
        if wk == 3:
            lamv.append(rng.uniform(0.5, 3.0))                       # RQ alpha
        if wk == 4:
            lamv.append(rng.uniform(0.6, 1.5))                       # constant
        raw[b, o_lam:o_lam + NL] = inv_softplus(np.array(lamv))
    return dict(x=x, y=y, noise=noise, raw=raw, kinds=kinds, lb=lb, ub=ub, Q=0, d=d,
                kind=kind, learn_noise=learn_noise)


def alfori_csv(path):
    """Write the AlfOri V-band light curve of BASELINE config C1 (tests/data/alfori_vband.npz:
    the 1564 (JD, Magnitude) rows of the reference's bundled pgmuvi/AlfOriAAVSO_Vband.csv) as a
    CSV with the reference's column names, for ``Lightcurve.from_csv``.  Returns ``path``."""
    import os
    here = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    z = np.load(os.path.join(here, "tests", "data", "alfori_vband.npz"))
    with open(path, "w") as f:
        f.write("JD,Magnitude\n")
        for jd, mag in zip(z["JD"], z["Magnitude"]):
            f.write(f"{float(jd)!r},{float(mag)!r}\n")
    return path
