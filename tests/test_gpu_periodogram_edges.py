"""N2 / N4 kernels at their edges.

* ``ls_power_kernel`` (the Lomb-Scargle periodogram) past one 512-point shared-memory chunk, at
  1024-frequency block boundaries, for every residue of nf mod 4, with Julian-date times and with
  NaN beyond each row's length, against the extended-precision ``oracle.lombscargle.power_exact``;
* ``ls_peaks_kernel`` (``find_peaks(distance=...)`` highest first) on plateaus, clipped distance
  windows, ties and -1 / NaN padding, against ``scipy.signal.find_peaks``;
* ``sm_psd_peak_kernel`` (dominant peak of the spectral-mixture PSD) for Q = 1..8 and grids at the
  256-thread stride edges, against ``oracle.period_summary``;
* the multiband periodogram of a band longer than one chunk and its Monte-Carlo null maxima.
"""
import numpy as np
import pytest
from scipy.signal import find_peaks

from oracle import lombscargle as ols

L = np.longdouble
TOL = 1e-12             # absolute, on the power (which lies in [0, 1])
JD = 2450000.0
N_VALID = (511, 512, 513, 1000, 1024, 1025, 1537, 4099)
FIT_MEAN, CENTER_DATA = 1, 2


# ---------------------------------------------------------------- helpers
def _light_curve(n, offset, rng):
    """irregular sampling over ~3000 d, a 217 d sinusoid on a constant, heteroscedastic errors"""
    t = np.sort(rng.uniform(0.0, 3000.0, n)) + offset
    y = 1.3 * np.sin(2 * np.pi * t / 217.0) + 0.5 + rng.normal(0.0, 0.3, n)
    dy = rng.uniform(0.05, 0.3, n)
    return t, y, dy


def _exact_freq(f0, df, k):
    """f0 + k df without rounding to fp64: the frequencies the kernel is asked for"""
    return L(f0) + np.asarray(k).astype(L) * L(df)


def _sample_idx(nf, power, rng, n_random=150):
    """every index within 8 of a multiple of 1024, the first and last 8, seeded random ones and
    the 5 highest values (the peaks)"""
    m = np.arange(1024, nf + 8, 1024)
    idx = np.r_[np.arange(8), nf - 8 + np.arange(8), (m[:, None] + np.arange(-8, 9)).ravel(),
                rng.integers(0, nf, n_random), np.argsort(power[:nf])[-5:]]
    return np.unique(idx[(idx >= 0) & (idx < nf)])


def _padded(rows, n_max, fill=np.nan):
    out = np.full((len(rows), n_max), fill)
    for b, r in enumerate(rows):
        out[b, :len(r)] = r
    return out


def _tensor(a, dev, dtype=None):
    import torch
    if a is None:
        return None
    return torch.tensor(np.asarray(a), dtype=dtype or torch.float64, device=dev)


def _ls_abi(dev, t, y, dy, nv, f0, df, nf, nf_max, flags=FIT_MEAN | CENTER_DATA):
    """pgm_lombscargle_f64 with an explicit grid (f0, df, nf per row) into a NaN-filled
    [B, nf_max] power array; nf[b] <= nf_max and every pointer valid (the ABI checks neither)"""
    import torch
    from pgmuvi_b200 import _lib
    from pgmuvi_b200._lib import check, ptr
    assert max(nf) <= nf_max
    T = lambda a, dt=None: _tensor(a, dev, dt)
    B, n_max = t.shape
    args = (T(t), T(nv, torch.int32), T(y), T(dy), T(f0), T(df), T(nf, torch.int32))
    power = torch.full((B, nf_max), float("nan"), dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        check(_lib.load().pgm_lombscargle_f64(
            ptr(args[0]), ptr(args[1]), ptr(args[2]), ptr(args[3]), B, n_max, ptr(args[4]),
            ptr(args[5]), ptr(args[6]), nf_max, flags, ptr(power),
            torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize(dev)
    return power.cpu().numpy()


def _lombscargle(dev, t, y, dy, nv=None, **kw):
    """pgmuvi_b200.lombscargle on host arrays: (f0, df, nf, power) as numpy"""
    import torch
    from pgmuvi_b200 import lombscargle as ls
    T = lambda a, dt=None: _tensor(a, dev, dt)
    f0, df, nf, p = ls.lombscargle(T(t), T(y), T(dy), T(nv, torch.int32) if nv is not None else None,
                                   **kw)
    return f0.cpu().numpy(), df.cpu().numpy(), nf.cpu().numpy(), p.cpu().numpy()


# ---------------------------------------------------------------- CPU: the extended-precision oracle
def _golden_cases():
    from conftest import ROOT
    import os
    z = np.load(os.path.join(ROOT, "tests", "golden_ls", "ls_cases.npz"))
    for name in z["names"]:
        dy = z[name + "_dy"]
        yield (str(name), z[name + "_t"], z[name + "_y"], None if dy.size == 0 else dy,
               z[name + "_grid"], z[name + "_power"])


def test_longdouble_is_wider_than_double():
    """power_exact is only exact where long double has a 64-bit mantissa (x86 extended)"""
    assert np.finfo(np.longdouble).eps < 1e-18


def test_power_exact_matches_the_fp64_goldens():
    """1e-13 on the goldens whose times start near 0; the Julian-date golden is fp64 power_slow
    evaluating sin(2 pi f t) at t ~ 2.45e6 and carries ~8e-11 of its own error"""
    for name, t, y, dy, grid, power in _golden_cases():
        freq = grid[0] + grid[1] * np.arange(int(grid[2]))
        err = np.abs(ols.power_exact(t, y, dy, freq) - power).max()
        assert err <= (2e-10 if name.endswith("_jd") else 1e-13), (name, err)


def test_power_exact_flags_and_time_origin():
    """fit_mean / center_data as power_slow does them, and no dependence on the time origin"""
    rng = np.random.default_rng(4)
    t, y, dy = _light_curve(90, 0.0, rng)
    f0, df, nf = ols.autofrequency(t)
    freq = f0 + df * np.arange(0, nf, 7)
    for fm, cd in ((True, True), (True, False), (False, True), (False, False)):
        ref = ols.power_slow(t, y, dy, freq, fit_mean=fm, center_data=cd)
        assert np.abs(ols.power_exact(t, y, dy, freq, fm, cd) - ref).max() <= 1e-13
    perm = rng.permutation(90)                   # t[0] is not the minimum any more
    assert np.abs(ols.power_exact(t[perm], y[perm], dy[perm], freq)
                  - ols.power_exact(t, y, dy, freq)).max() <= 1e-15


# ---------------------------------------------------------------- GPU: ls_power_kernel
@pytest.fixture(scope="module")
def ragged(cuda_device):
    """one ragged batch per dy setting: every n_valid at t0 = 0 and at t0 = 2.45e6 (JD), NaN in
    t, y and dy beyond n_valid; each member also evaluated alone"""
    rng = np.random.default_rng(2024)
    members = [(n, off) + _light_curve(n, off, rng) for n in N_VALID for off in (0.0, JD)]
    n_max = max(N_VALID) + 5
    out = {}
    for use_dy in (True, False):
        t = _padded([m[2] for m in members], n_max)
        y = _padded([m[3] for m in members], n_max)
        dy = _padded([m[4] for m in members], n_max) if use_dy else None
        nv = np.array([m[0] for m in members], np.int32)
        batch = _lombscargle(cuda_device, t, y, dy, nv)
        alone = [_lombscargle(cuda_device, m[2][None], m[3][None], m[4][None] if use_dy else None)
                 for m in members]
        out[use_dy] = (members, (t, y, dy, nv), batch, alone)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("use_dy", [True, False], ids=["dy", "nody"])
def test_gpu_periodogram_ragged_batch_past_one_chunk(ragged, use_dy):
    members, _, (f0, df, nf, p), alone = ragged[use_dy]
    rng = np.random.default_rng(7)
    assert p.shape[1] == int(nf.max())
    for b, (n, off, t, y, dy) in enumerate(members):
        g = ols.autofrequency(t)
        assert (f0[b], df[b], int(nf[b])) == g, (n, off)
        k = int(nf[b])
        assert np.isfinite(p[b, :k]).all() and np.isnan(p[b, k:]).all(), (n, off)
        # bitwise the light curve evaluated on its own
        a_f0, a_df, a_nf, a_p = alone[b]
        assert (a_f0[0], a_df[0], int(a_nf[0])) == (f0[b], df[b], k)
        assert np.array_equal(a_p[0], p[b, :k]), (n, off)
        idx = _sample_idx(k, p[b], rng)
        ref = ols.power_exact(t, y, dy if use_dy else None, _exact_freq(f0[b], df[b], idx))
        err = np.abs(p[b, idx] - ref)
        assert err.max() <= TOL, (n, off, idx[err.argmax()], err.max())
        assert ref.max() > 0.5     # the 217 d signal's peak is among the sampled indices


@pytest.mark.gpu
def test_gpu_periodogram_jd_golden_against_the_exact_power(cuda_device):
    """the n = 200 Julian-date golden light curve, whole grid, at the 1e-12 bar"""
    name, t, y, dy, grid, _ = next(c for c in _golden_cases() if c[0] == "n200_dy_jd")
    f0, df, nf, p = _lombscargle(cuda_device, t[None], y[None], dy[None])
    ref = ols.power_exact(t, y, dy, _exact_freq(f0[0], df[0], np.arange(int(nf[0]))))
    assert np.abs(p[0] - ref).max() <= TOL


@pytest.mark.gpu
def test_gpu_periodogram_per_row_nf_writes_exactly_its_row(cuda_device):
    """nf per row covering all four residues mod 4 and the 1024-frequency block edges: every
    k < nf[b] written (bitwise the full row's value: a frequency's power does not depend on how
    many follow it), every k >= nf[b] left at the NaN sentinel"""
    rng = np.random.default_rng(11)
    t, y, dy = _light_curve(700, JD, rng)
    f0, df, _ = ols.autofrequency(t)
    nfs = [1, 4, 1023, 1024, 1025, 2048, 2050, 2053]
    nf_max = 2053
    B = len(nfs)
    rep = lambda a: np.repeat(a[None], B, 0)
    p = _ls_abi(cuda_device, rep(t), rep(y), rep(dy), None, [f0] * B, [df] * B, nfs, nf_max)
    full = p[-1]
    for b, k in enumerate(nfs):
        assert np.isfinite(p[b, :k]).all() and np.isnan(p[b, k:]).all(), k
        assert np.array_equal(p[b, :k], full[:k]), k
    ref = ols.power_exact(t, y, dy, _exact_freq(f0, df, np.arange(nf_max)))
    assert np.abs(full - ref).max() <= TOL


@pytest.mark.gpu
def test_gpu_periodogram_empty_row_is_left_alone(cuda_device):
    """n_valid = 0 between two light curves (explicit grid through the C ABI): the empty row stays
    NaN and its neighbours are bitwise what they are on their own"""
    rng = np.random.default_rng(12)
    a, c = _light_curve(600, 0.0, rng), _light_curve(530, JD, rng)
    n_max = 610
    t = _padded([a[0], [], c[0]], n_max)
    y = _padded([a[1], [], c[1]], n_max)
    dy = _padded([a[2], [], c[2]], n_max)
    f0, df, nf = 1e-4, 2e-4, 3000
    p = _ls_abi(cuda_device, t, y, dy, [600, 0, 530], [f0] * 3, [df] * 3, [nf] * 3, nf)
    assert np.isnan(p[1]).all()
    for row, lc in ((0, a), (2, c)):
        one = _ls_abi(cuda_device, lc[0][None], lc[1][None], lc[2][None], None, [f0], [df], [nf], nf)
        assert np.isfinite(p[row]).all() and np.array_equal(p[row], one[0])


@pytest.mark.gpu
@pytest.mark.parametrize("fit_mean,center_data", [(True, True), (True, False), (False, True),
                                                  (False, False)])
def test_gpu_periodogram_flags_past_one_chunk(cuda_device, fit_mean, center_data):
    rng = np.random.default_rng(13)
    t, y, dy = _light_curve(1000, JD, rng)
    f0, df, nf, p = _lombscargle(cuda_device, t[None], y[None], dy[None], fit_mean=fit_mean,
                                 center_data=center_data)
    idx = _sample_idx(int(nf[0]), p[0], rng)
    ref = ols.power_exact(t, y, dy, _exact_freq(f0[0], df[0], idx), fit_mean, center_data)
    assert np.abs(p[0, idx] - ref).max() <= TOL


@pytest.mark.gpu
def test_gpu_periodogram_does_not_depend_on_point_order(cuda_device):
    """the kernel measures phases from t[0]: with the points permuted t[0] is not the minimum"""
    rng = np.random.default_rng(14)
    t, y, dy = _light_curve(1000, JD, rng)
    perm = rng.permutation(len(t))
    assert t[perm][0] != t.min()
    _, _, nf, p = _lombscargle(cuda_device, t[None], y[None], dy[None])
    _, _, nf2, p2 = _lombscargle(cuda_device, t[perm][None], y[perm][None], dy[perm][None])
    assert nf2[0] == nf[0] and np.abs(p2 - p).max() <= TOL


# ---------------------------------------------------------------- GPU: ls_peaks_kernel
def _plateau_row(nf, rng, distinct=True, levels=24):
    """quantised heights in runs of width 1..9; the first and last run and a run across every
    multiple of 256 sit at the top level (edge plateaus, which are not peaks, and plateau peaks
    that straddle a 256-thread stride).  ``distinct``: every run gets its own height (integer
    level * 8192 + a distinct run number), so distinct peaks never tie."""
    lev = np.empty(nf, np.int64)
    pos = 0
    while pos < nf:
        w = int(rng.integers(1, 10))
        lev[pos:pos + w] = rng.integers(0, levels)
        pos += w
    lev[:int(rng.integers(1, 10))] = levels
    lev[nf - int(rng.integers(1, 10)):] = levels
    for m in range(256, nf - 16, 256):          # clear of the last run
        lev[max(m - int(rng.integers(1, 5)), 0):m + int(rng.integers(1, 5))] = levels
    if not distinct:
        return lev.astype(np.float64)
    run = np.r_[0, np.cumsum(lev[1:] != lev[:-1])] if nf else lev
    return (lev * 8192 + rng.permutation(int(run.max()) + 1 if nf else 0)[run]).astype(np.float64)


def _greedy_stable(p, distance):
    """scipy's distance filter restated with a stable sort of the heights: among equal heights
    the larger index is kept first.  Returns the kept peaks highest first."""
    peaks, _ = find_peaks(p)
    order = np.argsort(p[peaks], kind="stable")[::-1]
    keep = np.ones(len(peaks), bool)
    out = []
    for j in order:
        if keep[j]:
            out.append(peaks[j])
            keep[np.abs(peaks - peaks[j]) < distance] = False
    return np.array(out, np.int64)


def _scipy_top(p, distance):
    pk, _ = find_peaks(p, distance=distance)
    assert len(np.unique(p[pk])) == len(pk)    # distinct heights: the order is defined
    return pk[np.argsort(p[pk])[::-1]]


@pytest.mark.gpu
@pytest.mark.parametrize("distance", [1, 2, 5, 7, 12504 + 3], ids=["d1", "d2", "d5", "d7", "dnf+3"])
def test_gpu_peaks_plateaus_ties_and_padding_match_find_peaks(cuda_device, distance):
    """one batch: distinct-height rows at nf in {1, 2, 3, 255, 256, 257, 2049, 12501}, tied-height
    rows, an all-NaN row (a constant light curve's power); NaN, +inf and 1e300 beyond each row's
    nf.  num_peaks below, at and above every row's number of surviving peaks."""
    import torch
    from pgmuvi_b200 import lombscargle as ls
    rng = np.random.default_rng(100 + distance)
    spec = [(nf, True) for nf in (1, 2, 3, 255, 256, 257, 2049, 12501)]
    spec += [(nf, False) for nf in (257, 2049, 12501)] + [(600, None)]
    nf_max = 12501 + 3
    pads = (np.nan, np.inf, 1e300)
    rows, want, nfs = np.empty((len(spec), nf_max)), [], []
    d = distance                                  # the last case exceeds every row's nf
    for b, (nf, distinct) in enumerate(spec):
        rows[b] = pads[b % 3]
        if distinct is None:                      # all-NaN row: no peaks
            rows[b, :nf] = np.nan
            want.append(np.zeros(0, np.int64))
        else:
            p = _plateau_row(nf, rng, distinct, levels=24 if distinct else 3)
            rows[b, :nf] = p
            w = _greedy_stable(p, d)
            if distinct:
                assert np.array_equal(w, _scipy_top(p, d))
            want.append(w)
        nfs.append(nf)
        if distinct and nf > 256 + 16:            # the construction does what it says
            _, pr = find_peaks(rows[b, :nf], plateau_size=1)
            m = np.arange(256, nf, 256)
            assert ((pr["left_edges"][:, None] < m) & (pr["right_edges"][:, None] >= m)).any()
    counts = sorted({len(w) for w in want})
    power = _tensor(rows, cuda_device)
    nf_t = _tensor(nfs, cuda_device, torch.int32)
    for K in sorted({1, 2, 3, max(counts) + 3} | {c for c in counts if c > 0}):
        idx, val = ls.top_peaks(power, nf_t, distance=distance, num_peaks=K)
        idx, val = idx.cpu().numpy(), val.cpu().numpy()
        for b, w in enumerate(want):
            k = min(K, len(w))
            assert np.array_equal(idx[b, :k], w[:k]), (spec[b], K)
            assert np.array_equal(val[b, :k], rows[b, w[:k]])
            assert (idx[b, k:] == -1).all() and np.isnan(val[b, k:]).all(), (spec[b], K)


@pytest.mark.gpu
def test_gpu_fit_ls_batch_matches_the_oracle_route_past_one_chunk(cuda_device, ragged):
    """fit_LS on the members with n_valid <= 1025 (with dy, t0 = 0 and JD) as one NaN-padded
    batch: every surviving peak is searched (num_peaks = nf / 5 + 2, ~2500 rounds of the peak
    kernel at n = 1000) and the frequencies and significance mask are the oracle route's
    (fp64 power_slow on t - t[0] over the whole grid, scipy peaks, Davies FAP, BH over all peaks)"""
    import torch
    from pgmuvi_b200 import lombscargle as ls
    members = [m for m in ragged[True][0] if m[0] <= 1025]
    n_max = 1025 + 3
    T = lambda a, dt=None: _tensor(a, cuda_device, dt)
    nv = np.array([m[0] for m in members], np.int32)
    freqs, sig = ls.fit_ls_batch(T(_padded([m[2] for m in members], n_max)),
                                 T(_padded([m[3] for m in members], n_max)),
                                 T(_padded([m[4] for m in members], n_max)),
                                 T(nv, torch.int32), num_peaks=3)
    for b, (n, off, t, y, dy) in enumerate(members):
        f0, df, nf = ols.autofrequency(t)
        freq = f0 + df * np.arange(nf)
        p = ols.power_slow(t - t[0], y, dy, freq)
        pk = ols.top_peaks(p, 5, 10**6)
        assert np.allclose(freqs[b], freq[pk[:3]], rtol=1e-12), (n, off)
        if ols.fap_davies(p.max(), freq[-1], t, dy) > 0.05:
            want = np.zeros(3, dtype=bool)
        else:
            m = ols.fdr_bh(ols.fap_single(p[pk], n), 0.05)
            m[0] = True
            want = m[:3]
        assert np.array_equal(sig[b], want), (n, off)
        assert sig[b, 0]                  # the 217 d signal is significant


# ---------------------------------------------------------------- GPU: sm_psd_peak_kernel
def _psd_rows(Q, rng, n_random=4):
    """[B, Q] mixtures and [B] limits: random mixtures inside the grid with some zero weights, one
    PSD that rises over the whole grid (components far above it, broad) and one that is all
    zeros (components far above it, narrow: every exp underflows)"""
    B = n_random + 2
    fmin = 10.0 ** rng.uniform(-4, -2, B)
    fmax = fmin * 10.0 ** rng.uniform(1, 3, B)
    mu = np.exp(rng.uniform(np.log(fmin), np.log(fmax), (Q, B))).T
    sg = mu * rng.uniform(0.02, 0.3, (B, Q))
    w = rng.uniform(0.05, 1.0, (B, Q))
    w[:n_random][rng.random((n_random, Q)) < 0.3] = 0.0
    r, z = n_random, n_random + 1
    mu[r], sg[r] = fmax[r] * rng.uniform(8, 12, Q), 3.0 * fmax[r]
    mu[z], sg[z] = 1e6 * fmax[z], 1e-3 * fmax[z]
    return mu, sg, w, fmin, fmax


@pytest.mark.gpu
@pytest.mark.parametrize("Q", range(1, 9))
def test_gpu_psd_peak_every_mixture_count_and_stride_edge(cuda_device, Q):
    """PSD at the existing tolerance, peak index and number of local maxima exactly, for grids of
    3, 4, 255, 256, 257 and 5000 points.  Known difference, left untested: the kernel takes strict
    local maxima, scipy the midpoint of a flat top; an exact plateau at a maximum of a sum of
    Gaussians does not occur on these grids."""
    from oracle import period_summary as ops_
    from pgmuvi_b200.period_summary import period_summary_batch
    rng = np.random.default_rng(300 + Q)
    mu, sg, w, fmin, fmax = _psd_rows(Q, rng)
    rising, zero = len(fmin) - 2, len(fmin) - 1
    for n_grid in (3, 4, 255, 256, 257, 5000):
        out = period_summary_batch(_tensor(mu, cuda_device), sg, w, fmin=fmin, fmax=fmax,
                                   n_grid=n_grid, return_psd=True)
        for b in range(len(fmin)):
            ref = ops_.dominant_peak(mu[b], sg[b], w[b], fmin[b], fmax[b], n_grid)
            key = (Q, n_grid, b)
            assert np.allclose(out["freq_grid"][b], ref["grid"], rtol=1e-13), key
            assert np.allclose(out["psd"][b], ref["psd"], rtol=1e-10, atol=1e-13), key
            assert int(out["peak_index"][b]) == ref["index"], key
            assert int(out["n_peaks"][b]) == ref["n_peaks"], key
            assert np.isclose(out["dominant_frequency"][b], ref["frequency"], rtol=1e-13), key
            assert np.isclose(out["peak_height"][b], ref["height"], rtol=1e-10, atol=1e-300), key
        # the arg-max fall-back at the pinned last grid point, and at index 0 of an all-zero PSD
        assert out["peak_index"][rising] == n_grid - 1 and out["n_peaks"][rising] == 0
        assert out["dominant_frequency"][rising] == out["freq_grid"][rising, -1]
        assert (out["psd"][zero] == 0).all()
        assert out["peak_index"][zero] == 0 and out["n_peaks"][zero] == 0
        assert out["peak_height"][zero] == 0.0


# ---------------------------------------------------------------- GPU: multiband
def _multiband_long(rng):
    """three bands of 600, 260 and 140 points (the first longer than one 512-point chunk)"""
    t, y, b, dy = [], [], [], []
    for k, n in enumerate((600, 260, 140)):
        tk = np.sort(rng.uniform(0, 2000, n))
        t.append(tk)
        y.append((1 + 0.3 * k) * np.sin(2 * np.pi * tk / 37.0 + 0.4 * k) + 0.2 * k
                 + 0.4 * rng.standard_normal(n))
        b.append(np.full(n, k))
        dy.append(rng.uniform(0.2, 0.5, n))
    return tuple(np.concatenate(a) for a in (t, y, b, dy))


@pytest.mark.gpu
def test_gpu_multiband_power_past_one_chunk_against_the_exact_power(cuda_device):
    from pgmuvi_b200.lombscargle import MultibandLS
    rng = np.random.default_rng(21)
    t, y, b, dy = _multiband_long(rng)
    LS = MultibandLS(t, y, b, dy, device=cuda_device)
    freq = LS.autofrequency()
    got = LS.power(freq)
    f0, df, nf = MultibandLS._regular(freq)       # the grid the kernel is given
    idx = _sample_idx(nf, got, rng)
    ref = ols.multiband_power(t, y, b, dy, _exact_freq(f0, df, idx), exact=True)
    assert np.abs(got[idx] - ref).max() <= TOL


@pytest.mark.gpu
def test_gpu_multiband_null_maxima_replay_on_the_host(cuda_device):
    """65 bootstrap samples (two launches of 64 and 1): each null maximum is the maximum of the
    multiband power of the same seeded permutation evaluated on its own.  Not bitwise: torch may
    sum the chi2 weights in another order for another number of rows."""
    from pgmuvi_b200.lombscargle import MultibandLS
    t, y, b, dy = _multiband_long(np.random.default_rng(22))
    LS = MultibandLS(t, y, b, dy, device=cuda_device)
    freq = LS.autofrequency(nyquist_factor=2)
    null = LS.null_max_powers(freq, "bootstrap", 65, generator=np.random.default_rng(5))
    rng = np.random.default_rng(5)
    want = []
    for _ in range(65):
        ys = y.copy()
        for v in np.unique(b):
            m = b == v
            ys[m] = y[m][rng.permutation(int(m.sum()))]
        want.append(MultibandLS(t, ys, b, dy, device=cuda_device).power(freq).max())
    assert null.shape == (65,)
    assert np.allclose(null, want, rtol=1e-14, atol=0)
