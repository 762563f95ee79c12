"""CPU oracle for N2, the Lomb-Scargle initialisation in front of the path.
TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

pgmuvi's ``Lightcurve.fit_LS`` (pgmuvi/lightcurve.py:4214-4611) calls the third-party
``astropy.timeseries.LombScargle`` (un-pinned, ``pyproject.toml``; ABSENT from this image) and
``scipy.signal.find_peaks`` (present).  PARITY UNPINNED at the astropy boundary: this module
restates astropy's published algorithms -

* ``autofrequency``  - LombScargle.autofrequency(samples_per_peak=5, nyquist_factor):
  df = 1 / (samples_per_peak * baseline), f_min = df / 2, f_max = nyquist_factor * n / (2 baseline),
  Nf = 1 + round((f_max - f_min) / df);
* ``power_slow``     - the floating-mean generalised periodogram of the "slow" implementation
  (Zechmeister & Kuerster 2009; fit_mean=True, center_data=True, normalization='standard'),
  with an explicit time shift tau and explicitly recomputed shifted sums - i.e. NOT the
  angle-difference shortcut the CUDA kernel uses, so the two are independent routes;
* ``fap_davies`` / ``fap_single`` - Baluev's analytic false-alarm bounds used for the
  significance mask (lightcurve.py:4566-4590).

Caveat kept from the reference: for more than 200 frequencies with
``assume_regular_frequency=True`` astropy's ``method='auto'`` picks its FFT-based *approximation*
("fast"); the exact periodogram restated here is what that approximates (peak positions agree,
powers to ~1e-3).  ``find_peaks`` is scipy's own (the reference's call, lightcurve.py:4531)."""
import numpy as np
from scipy.signal import find_peaks
from scipy.special import gammaln


def autofrequency(t, samples_per_peak=5, nyquist_factor=5):
    t = np.asarray(t, dtype=np.float64)
    baseline = t.max() - t.min()
    n = t.size
    df = 1.0 / baseline / samples_per_peak
    fmin = 0.5 * df
    fmax = nyquist_factor * (0.5 * n / baseline)
    nf = 1 + int(np.round((fmax - fmin) / df))
    return fmin, df, nf


def power_slow(t, y, dy, freq, fit_mean=True, center_data=True):
    t, y = np.asarray(t, np.float64), np.asarray(y, np.float64)
    dy = np.ones_like(y) if dy is None else np.asarray(dy, np.float64)
    w = dy ** -2.0
    w = w / w.sum()
    if fit_mean or center_data:
        y = y - np.dot(w, y)
    out = np.empty(len(freq))
    for k, f in enumerate(np.asarray(freq, np.float64)):
        om = 2 * np.pi * f
        s, c = np.sin(om * t), np.cos(om * t)
        S2 = 2 * np.dot(w, s * c)
        C2 = 2 * np.dot(w, 0.5 - s * s)
        if fit_mean:
            S, C = np.dot(w, s), np.dot(w, c)
            S2 -= 2 * S * C
            C2 -= C * C - S * S
        arg = om * t - 0.5 * np.arctan2(S2, C2)
        st, ct = np.sin(arg), np.cos(arg)
        Y = np.dot(w, y)
        YC, YS = np.dot(w * y, ct), np.dot(w * y, st)
        CC, SS = np.dot(w, ct * ct), np.dot(w, st * st)
        if fit_mean:
            Ct, St = np.dot(w, ct), np.dot(w, st)
            YC -= Y * Ct
            YS -= Y * St
            CC -= Ct * Ct
            SS -= St * St
        out[k] = (YC * YC / CC + YS * YS / SS) / np.dot(w, y * y)
    return out


def power_exact(t, y, dy, freq, fit_mean=True, center_data=True, chunk=256):
    """``power_slow`` restated in extended precision (``np.longdouble``, 64-bit mantissa on x86)
    on ``t - t[0]``, vectorised over chunks of ``chunk`` frequencies.  The periodogram does not
    depend on the time origin; shifting it in extended precision keeps the phases 2 pi f t exact
    to ~1e-19 relative even for Julian dates (t ~ 2.45e6 d), where the fp64 ``power_slow`` loses
    ~1e-10 in the power.  ``freq`` may itself be a longdouble array (e.g. ``f0 + k * df`` formed
    without rounding to fp64).  About 0.7 us per (frequency, point) on one x86 core: sample the
    grid rather than evaluating all of it for long light curves."""
    L = np.longdouble
    t = np.asarray(t, np.float64)
    t = t.astype(L) - L(t[0])
    y = np.asarray(y, np.float64).astype(L)
    w = np.ones_like(y) if dy is None else np.asarray(dy, np.float64).astype(L) ** -2
    w = w / w.sum()
    if fit_mean or center_data:
        y = y - np.dot(w, y)
    wy, Y, YY = w * y, np.dot(w, y), np.dot(w, y * y)
    two_pi = 2 * L("3.14159265358979323846264338327950288")
    freq = np.asarray(freq).astype(L)
    out = np.empty(freq.size, np.float64)
    for s in range(0, freq.size, chunk):
        ph = two_pi * freq[s:s + chunk, None] * t[None, :]
        sn, cs = np.sin(ph), np.cos(ph)
        S2 = 2 * ((sn * cs) @ w)
        C2 = (cs * cs - sn * sn) @ w
        if fit_mean:
            S, C = sn @ w, cs @ w
            S2 -= 2 * S * C
            C2 -= C * C - S * S
        arg = ph - 0.5 * np.arctan2(S2, C2)[:, None]
        st, ct = np.sin(arg), np.cos(arg)
        YC, YS = ct @ wy, st @ wy
        CC, SS = (ct * ct) @ w, (st * st) @ w
        if fit_mean:
            Ct, St = ct @ w, st @ w
            YC -= Y * Ct
            YS -= Y * St
            CC -= Ct * Ct
            SS -= St * St
        out[s:s + chunk] = ((YC * YC / CC + YS * YS / SS) / YY).astype(np.float64)
    return out


def top_peaks(power, distance, num_peaks):
    """find_peaks(power, distance=distance), sorted by height, first num_peaks
    (lightcurve.py:4531-4532, 4555)."""
    peaks, _ = find_peaks(power, distance=distance)
    peaks = peaks[np.argsort(power[peaks])][::-1]
    return peaks[:num_peaks]


def fap_single(z, n):
    return (1.0 - z) ** (0.5 * (n - 3))


def fap_davies(z, fmax, t, dy=None):
    """Davies upper bound of the false-alarm probability of the highest peak ('standard'
    normalisation): fap_single + tau_davies (Baluev 2008)."""
    t = np.asarray(t, np.float64)
    n = t.size
    w = np.ones_like(t) if dy is None else np.asarray(dy, np.float64) ** -2.0
    tm = np.dot(w, t) / w.sum()
    dt = np.dot(w, (t - tm) ** 2) / w.sum()
    teff = np.sqrt(4 * np.pi * dt)
    nh, nk = n - 1, n - 3
    gam = np.sqrt(2.0 / nh) * np.exp(gammaln(0.5 * nh) - gammaln(0.5 * (nh - 1)))
    tau = gam * fmax * teff * (1 - z) ** (0.5 * (nk - 1)) * np.sqrt(0.5 * nh * z)
    return fap_single(z, n) + tau


def fdr_bh(fap_values, alpha=0.05):
    """Benjamini-Hochberg mask (lightcurve.py:4342-4382)."""
    fap_values = np.asarray(fap_values, np.float64)
    order = np.argsort(fap_values)
    ok = fap_values[order] <= np.arange(1, len(order) + 1) / len(order) * alpha
    res = np.zeros(len(order), dtype=bool)
    if ok.any():
        res[order[: np.where(ok)[0].max() + 1]] = True
    return res


def multiband_power(t, y, bands, dy, freq, exact=False):
    """astropy ``LombScargleMultiband(t, y, bands, dy).power(freq, method='fast')`` restated
    (astropy/timeseries/periodograms/lombscargle_multiband/implementations/mbfast_impl.py, the
    ``ls_method`` default of pgmuvi/multiband_ls_significance.py:136): a floating-mean single-band
    periodogram per band, combined with the bands' reference chi-squares chi2_0b = sum w (y - ybar_w)^2
    as weights.  astropy is absent from the image: parity with it is unpinned.  ``exact``: each
    band's power from ``power_exact`` (extended precision) instead of ``power_slow``."""
    band_power = power_exact if exact else power_slow
    t, y, bands = (np.asarray(a) for a in (t, y, bands))
    dy = np.ones_like(t, dtype=np.float64) if dy is None else np.asarray(dy, np.float64)
    ub = np.unique(bands)
    powers, chi2 = [], []
    for b in ub:
        m = bands == b
        powers.append(band_power(t[m], y[m], dy[m], freq))
        w = dy[m] ** -2.0
        ybar = np.dot(w, y[m]) / w.sum()
        chi2.append(np.dot(w, (y[m] - ybar) ** 2))
    chi2 = np.asarray(chi2)
    return np.dot(chi2 / chi2.sum(), np.asarray(powers))


def multiband_fap_analytical(power_values, n_freq):
    """pgmuvi/multiband_ls_significance.py:408-467"""
    return np.clip(1.0 - (1.0 - np.exp(-np.asarray(power_values, np.float64))) ** (n_freq / 5.0), 0.0, 1.0)
