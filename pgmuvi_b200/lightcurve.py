"""Host-side mirror of the slice of ``pgmuvi.lightcurve.Lightcurve`` that CALLS the hot path
(seam #0, SURVEY section 8b): data container + transforms, likelihood / model / default
constraint / hyper-parameter setup and ``fit(model='1D'|'2D')``.

The real class (pgmuvi/lightcurve.py:1677-10793) cannot be imported in this image
(``import gpytorch`` / ``matplotlib`` at lightcurve.py:7,31), so this restates exactly the parts
that fix the parameterisation the engine sees, each method citing what it follows.  Everything
outside the path (ingest, Lomb-Scargle init, period summaries, plotting) is out of scope; with
the real pgmuvi installed one uses its ``Lightcurve`` and only swaps ``train`` (INTEGRATION.md).
Nothing here computes the GP on the CPU.
"""
from __future__ import annotations

import warnings

import numpy as np
import torch

from . import gp
from .constraints import GreaterThan, Interval
from .trainers import train

# lightcurve.py:2901-2930 - the spectral-mixture exact models; the separable ones are built
# with the spectral-mixture time kernel (SURVEY.md section 8a row a4)
_SM_MODELS = {"1D": gp.SpectralMixtureGPModel, "2D": gp.TwoDSpectralMixtureGPModel,
              "1DLinear": gp.SpectralMixtureLinearMeanGPModel,
              "2DLinear": gp.TwoDSpectralMixtureLinearMeanGPModel,
              "2DPowerLaw": gp.TwoDSpectralMixturePowerLawMeanGPModel,
              "2DDust": gp.TwoDSpectralMixtureDustMeanGPModel,
              "2DSeparable": gp.SeparableGPModel, "2DAchromatic": gp.AchromaticGPModel,
              "2DWavelengthDependent": gp.WavelengthDependentGPModel,
              "2DDustMean": gp.DustMeanGPModel, "2DPowerLawMean": gp.PowerLawMeanGPModel,
              "1DMatern": gp.MaternGPModel, "1DQuasiPeriodic": gp.QuasiPeriodicGPModel,
              "1DLinearQuasiPeriodic": gp.LinearMeanQuasiPeriodicGPModel,
              "1DPeriodicStochastic": gp.PeriodicPlusStochasticGPModel}
_NO_MIXTURE_MODELS = ("1DMatern", "1DQuasiPeriodic", "1DLinearQuasiPeriodic",
                      "1DPeriodicStochastic")
CONSTRAINT_SETS = {"LPV": {"period": {"lower": (20.0, True), "upper": (None, False)}}}


class Transformer(torch.nn.Module):
    """pgmuvi/lightcurve.py:157-194."""

    def transform(self, data, **kwargs):
        raise NotImplementedError

    def inverse(self, data, shift=True, **kwargs):
        raise NotImplementedError


class MinMax(Transformer):
    """pgmuvi/lightcurve.py:196-243: rescale every column to [0, 1]."""

    def transform(self, data, dim=0, apply_to=None, recalc=False, shift=True, **kwargs):
        if recalc or not hasattr(self, "min"):
            self.register_buffer("min", torch.min(data, dim=dim, keepdim=True)[0])
            self.register_buffer("range", torch.max(data, dim=dim, keepdim=True)[0] - self.min)
            shift = True
        if apply_to is not None:
            return (data - (shift * self.min[apply_to])) / self.range[apply_to]
        return (data - (shift * self.min)) / self.range

    def inverse(self, data, shift=True, **kwargs):
        return (data * self.range) + (shift * self.min)


class ZScore(Transformer):
    """pgmuvi/lightcurve.py:245-288."""

    def transform(self, data, dim=0, apply_to=None, recalc=False, shift=True, **kwargs):
        if recalc or not hasattr(self, "mean"):
            self.register_buffer("mean", torch.mean(data, dim=dim, keepdim=True))
            self.register_buffer("sd", torch.std(data, dim=dim, keepdim=True))
            shift = True
        if apply_to is not None:
            return (data - (shift * self.mean[apply_to])) / self.sd[apply_to]
        return (data - shift * self.mean) / self.sd

    def inverse(self, data, shift=True, **kwargs):
        return (data * self.sd) + (self.mean * shift)


def _make_transform(t):
    if t is None or isinstance(t, Transformer):
        return t
    if t == "minmax":
        return MinMax()
    if t == "zscore":
        return ZScore()
    raise ValueError(f"unknown transform {t!r}")


class Lightcurve(torch.nn.Module):
    """``Lightcurve(xdata, ydata, yerr=None, xtransform=None, ytransform=None, ...)`` with the
    reference's signature and defaults (pgmuvi/lightcurve.py:1724-1742).  Data are stored float32
    like the reference (``_ensure_tensor``, :2434-2446); ``.double()`` opts into float64.  The
    pre-processing gates (``check_sampling``, ``check_variability``, per-band sub-sampling) sit
    outside the path: the flags are accepted, the gates are not run."""

    def __init__(self, xdata, ydata, yerr=None, xtransform=None, ytransform=None, name=None,
                 time_units=None, max_samples=1000, max_samples_per_band=None,
                 subsample_seed=None, check_sampling=False, sampling_kwargs=None,
                 check_variability=False, variability_kwargs=None, band=None, **kwargs):
        super().__init__()
        self.name = name
        self.time_units = time_units
        self.xtransform = _make_transform(xtransform)
        self.ytransform = _make_transform(ytransform)
        x = self._ensure_tensor(xdata)
        y = self._ensure_tensor(ydata)
        if x.dim() == 2 and x.shape[1] == 1:
            x = x[:, 0]
        if torch.isnan(x).any() or torch.isnan(y).any():
            raise ValueError("The x / y values contain NaNs.")
        # 1-D light curves longer than max_samples are sub-sampled before anything else
        # (lightcurve.py:1733, 2150-2181; random unless subsample_seed is given)
        if max_samples is not None and x.dim() == 1 and x.shape[0] > max_samples:
            from .preprocess import subsample_lightcurve
            n_total = x.shape[0]
            idx = subsample_lightcurve(
                x.numpy(), max_samples=max_samples, random_seed=subsample_seed,
                max_gap_fraction=(sampling_kwargs or {}).get("max_gap_fraction", 0.3))
            warnings.warn(
                f"Lightcurve has {n_total} points, which exceeds max_samples={max_samples}. "
                f"Retaining a random subsample of {len(idx)} points. "
                "Set max_samples=None to disable subsampling.", UserWarning, stacklevel=2)
            idx_t = torch.as_tensor(idx, dtype=torch.long)
            x, y = x[idx_t], y[idx_t]
            if yerr is not None:
                yerr = self._ensure_tensor(yerr)[idx_t]
        self.register_buffer("_xdata_raw", x)
        self.register_buffer("_xdata_transformed",
                             x if self.xtransform is None else self.xtransform.transform(x))
        self.register_buffer("_ydata_raw", y)
        self.register_buffer("_ydata_transformed",
                             y if self.ytransform is None else self.ytransform.transform(y))
        if yerr is not None:
            e = self._ensure_tensor(yerr)
            self.register_buffer("_yerr_raw", e)
            # the same transform object is applied to the errors (lightcurve.py:2421-2432)
            self.register_buffer("_yerr_transformed",
                                 e if self.ytransform is None else self.ytransform.transform(e))
        self._constraints_set = False
        self._fitted = False

    @classmethod
    def from_csv(cls, path, xcol=None, ycol=None, yerrcol=None, **kwargs):
        """1-D subset of ``Lightcurve.from_csv`` (lightcurve.py:510-760): a headed CSV with a
        time column, a value column and an optional uncertainty column; rows with NaNs are
        dropped with a warning, data are cast to float32 like the reference (:742-745)."""
        data = np.genfromtxt(path, delimiter=",", names=True, dtype=None, encoding="utf-8")
        cols = list(data.dtype.names)
        xcol = xcol or cols[0]
        ycol = ycol or cols[1]
        for c in (xcol, ycol) + ((yerrcol,) if yerrcol else ()):
            if c not in cols:
                raise ValueError(f"Column '{c}' not found in CSV. Available columns: {cols}")
        use = [xcol, ycol] + ([yerrcol] if yerrcol else [])
        arr = np.stack([np.asarray(data[c], dtype=np.float64) for c in use], 1)
        good = ~np.isnan(arr).any(1)
        if (~good).any():
            warnings.warn(f"Dropped {int((~good).sum())} row(s) containing NaN values.",
                          stacklevel=2)
        if not good.any():
            raise ValueError("No valid data rows remain after dropping NaN-containing rows.")
        arr = arr[good]
        return cls(arr[:, 0], arr[:, 1], yerr=arr[:, 2] if yerrcol else None, **kwargs)

    @staticmethod
    def _ensure_tensor(values):
        return torch.as_tensor(np.asarray(values) if not torch.is_tensor(values) else values
                               ).to(torch.float32)

    @property
    def ndim(self):
        return 1 if self._xdata_raw.dim() == 1 else self._xdata_raw.shape[-1]

    xdata = property(lambda self: self._xdata_raw)
    ydata = property(lambda self: self._ydata_raw)
    yerr = property(lambda self: self._yerr_raw)

    # ---- likelihood (lightcurve.py:2718-2823) ------------------------------------------
    def set_likelihood(self, likelihood=None, variance=False, **kwargs):
        has_noise = hasattr(self, "_yerr_transformed")
        if has_noise:
            noise = self._yerr_transformed if variance else self._yerr_transformed ** 2
        if has_noise and likelihood is None:
            self.likelihood = gp.FixedNoiseGaussianLikelihood(noise)
        elif has_noise and likelihood == "learn":
            self.likelihood = gp.FixedNoiseGaussianLikelihood(noise, learn_additional_noise=True)
        elif likelihood == "learn":
            self.likelihood = gp.GaussianLikelihood(learn_additional_noise=True)
        elif "Interval" in [t.__name__ for t in type(likelihood).__mro__]:
            self.likelihood = gp.GaussianLikelihood(noise_constraint=likelihood)
        elif likelihood is None:
            self.likelihood = gp.GaussianLikelihood()
        elif isinstance(likelihood, (gp.GaussianLikelihood, gp.FixedNoiseGaussianLikelihood)):
            self.likelihood = likelihood
        else:
            raise ValueError(f"Expected a string, a constraint or a Likelihood instance, but got "
                             f"{type(likelihood)}.")

    # ---- model (lightcurve.py:2825-2974; only the SM exact models are on the path) -------
    def set_model(self, model=None, likelihood=None, num_mixtures=None, variance=False, **kwargs):
        if not hasattr(self, "likelihood") or likelihood is not None and not isinstance(
                likelihood, torch.nn.Module):
            self.set_likelihood(likelihood, variance=variance)
        elif isinstance(likelihood, torch.nn.Module):
            self.likelihood = likelihood
        if isinstance(model, torch.nn.Module):
            self.model = model
        elif model in _SM_MODELS:
            if model.startswith("1D") and self.ndim > 1:
                raise ValueError("You have selected a 1D model but your data has more than one "
                                 "input dimension; use model='2D'.")   # tests/test_2d_integration.py:167-186
            if model.startswith("2D") and self.ndim != 2:
                raise ValueError(f"model={model!r} needs xdata of shape [n, 2] (time, wavelength)")
            mk = {} if model in _NO_MIXTURE_MODELS else {"num_mixtures": num_mixtures or 4}
            self.model = _SM_MODELS[model](self._xdata_transformed, self._ydata_transformed,
                                           self.likelihood, **mk, **kwargs)
        else:
            raise UnsupportedModel(
                f"model {model!r} is outside the accelerated path (SURVEY section 8a): "
                "only '1D' / '2D' spectral-mixture exact GPs and the separable '2DSeparable' / "
                "'2DAchromatic' / '2DWavelengthDependent' models with a spectral-mixture time "
                "kernel")
        self._make_parameter_dict()
        self._constraints_set = False

    def _make_parameter_dict(self):
        """name -> owning module, with the aliases of lightcurve.py:2976-3043."""
        self._model_pars = {}
        for name, p in self.model.named_parameters():
            base, _, leaf = name.rpartition(".")
            mod = self.model.get_submodule(base) if base else self.model
            key = ".".join(c.lstrip("raw_") for c in name.split("."))
            self._model_pars[key] = {"module": mod, "raw_name": leaf, "param": p}
            for alias in ("noise", "mixture_means", "mixture_scales", "mixture_weights"):
                if key.endswith(alias):
                    self._model_pars[alias] = self._model_pars[key]

    # ---- default constraints (lightcurve.py:3777-4011) -----------------------------------
    def set_default_constraints(self, constraint_set=None, **kwargs):
        y = self._ydata_transformed
        if "noise" in self._model_pars:
            if hasattr(self, "_yerr_transformed"):
                noise_min = float(np.minimum(1e-4, float(self._yerr_transformed.min()) / 10))
            else:
                noise_min = 1e-4 * float(y.std())
            self._model_pars["noise"]["module"].register_constraint(
                "raw_noise", Interval(noise_min, float(y.std())))
        for key, ent in self._model_pars.items():
            if "mean_module.constant" in key:
                ent["module"].register_constraint("raw_constant",
                                                  Interval(float(y.min()), float(y.max())))
        if "mixture_means" in self._model_pars:
            xt = self._xdata_transformed
            t = xt[:, 0] if self.ndim > 1 else xt
            span = float(t.max() - t.min())
            if span <= 0.0:
                raise ValueError("set_default_constraints requires a dataset whose timestamps "
                                 "span a positive time range")
            if self.ndim > 1:
                ts = t.sort().values
                diffs = ts[1:] - ts[:-1]
                con = Interval(1.0 / span, float(1 / (2 * diffs[diffs > 0].min())))
            else:
                con = GreaterThan(1.0 / span)
            if constraint_set is not None:
                cs = CONSTRAINT_SETS[constraint_set]
                lower_val, lower_active = cs["period"]["lower"]
                xr = self._xdata_raw[:, 0] if self.ndim > 1 else self._xdata_raw
                freq_scale = float(xr.max() - xr.min()) / span
                if lower_active and lower_val is not None:
                    fmax = freq_scale / lower_val
                    lo = float(con.lower_bound)
                    if fmax > lo:
                        hi = float(con.upper_bound)
                        con = Interval(lo, min(hi, fmax))
            self._model_pars["mixture_means"]["module"].register_constraint(
                "raw_mixture_means", con)
        self._constraints_set = True

    # ---- hyper-parameters (lightcurve.py:4061-4156) --------------------------------------
    def set_hypers(self, hypers=None, **kwargs):
        if hypers is None:
            return
        hypers = {k: torch.as_tensor(v, dtype=self._ydata_transformed.dtype)
                  for k, v in hypers.items()}
        for key in hypers:
            if any(p in key for p in ("mixture_means", "mixture_scales")):
                if self.xtransform is not None:
                    if hypers[key].dim() == 2:
                        out = torch.zeros_like(hypers[key])
                        for dim in range(hypers[key].shape[1]):
                            out[:, dim] = 1 / ((1 / hypers[key][:, dim])
                                               / self.xtransform.range[0, dim])
                        hypers[key] = out
                    else:
                        hypers[key] = 1 / self.xtransform.transform(1 / hypers[key], shift=False)
            elif any(p in key for p in ("noise", "mean_module")):
                if self.ytransform is not None:
                    hypers[key] = self.ytransform.transform(hypers[key])
        for key, val in hypers.items():
            par = self._lookup(key)
            if par is not None and val.numel() == par.numel():
                val = val.reshape(par.shape)
            self.model.initialize(**{key: val})

    def _lookup(self, key):
        mod = self.model
        parts = key.split(".")
        for p in parts[:-1]:
            mod = getattr(mod, p, None)
            if mod is None:
                return None
        return mod._parameters.get("raw_" + parts[-1], mod._parameters.get(parts[-1]))

    # ---- reporting (lightcurve.py:8999-9077, 6279-6343) ------------------------------------
    def get_parameters(self, raw=False, transform=True):
        pars = {}
        for name, param in self.model.named_parameters():
            if not raw and "raw" in name:
                key = ".".join(c.lstrip("raw_") for c in name.split("."))
                ent = self._model_pars[key]
                con = ent["module"]._modules.get(ent["raw_name"] + "_constraint")
                val = (con.transform(param) if con is not None else param).data
            else:
                key, val = name, param.data
            pars[key] = self._report(key, val) if transform else val
        return pars

    def _report(self, key, val):
        """The x / y transforms ``get_parameters`` applies to the constrained value of ``key``."""
        if self.xtransform is not None and any(p in key for p in ("mixture_means", "mixture_scales")):
            return 1 / self.xtransform.inverse(1 / val, shift=False)
        if self.ytransform is not None and any(p in key for p in ("noise", "mean_module")):
            return self.ytransform.inverse(val)
        return val

    def parameter_uncertainties(self, device=None):
        """Standard errors of the fitted hyper-parameters from the exact Fisher information of the
        Gaussian log-likelihood (``pgm_sm_fisher_f64``, evaluated at the current parameters).

        Returns ``{"names", "covariance", "stderr", "period_stderr", "fisher_ok", "fisher",
        "info"}``: ``names`` / ``covariance`` / ``fisher`` per packed slot (constrained values, the
        inverse Fisher matrix over the free slots, 0 for frozen ones); ``stderr`` keyed and shaped
        like ``get_parameters()`` and in its units (delta method through the same transforms);
        ``period_stderr = stderr(mu) / mu^2`` per spectral-mixture component (time dimension, raw
        units) or None.  Frozen slots (an ``Interval(lb, lb)``, values that are not Parameters)
        get 0.  If the Fisher matrix of the free slots is not positive definite, ``stderr`` is
        NaN and ``fisher_ok`` False.  Models with a non-constant mean raise
        ``UnsupportedModelError``."""
        from .batch import uncertainties_batch
        return uncertainties_batch([self], device=device)[0]

    def get_periods(self):
        """Periods ``1/mu`` (time dimension), mixture weights and scales ``1/(2 pi sigma)`` in the
        units of the raw x data (lightcurve.py:6279-6343)."""
        pars = self.get_parameters()
        pick = lambda leaf: next(v for k, v in pars.items() if k.endswith(leaf)).detach().cpu()
        mu, sg, w = pick("mixture_means"), pick("mixture_scales"), pick("mixture_weights")
        periods = (1 / mu[:, 0, 0]).numpy()
        scales = (1 / (2 * np.pi * sg[:, 0, 0])).numpy()
        return periods, w.numpy(), scales

    def get_period_summary(self, n_grid=5000, min_freq=None, max_freq=None, peak_threshold_rel=0.2,
                           uncertainty="peak_mass", n_peaks=None, mass_level=0.68,
                           classify_lsp=False):
        """``get_period_summary`` of a fitted spectral-mixture model (lightcurve.py:7860-8130,
        8134-8305): the summed PSD on the log-spaced grid and its dominant peak on the GPU
        (``pgm_sm_psd_peak_f64``, re-evaluated while the half-maximum of the dominant peak is not
        contained), then per-peak basins, peak-centred ``mass_level`` intervals, physical ranking
        and optional LSP flags.  Returns a :class:`pgmuvi_b200.period_summary.PeriodSummary` (a
        dict with the reference's keys plus ``peaks``; ``write_text`` / ``write_json``)."""
        if uncertainty != "peak_mass":
            raise NotImplementedError(f"uncertainty='{uncertainty}' is not yet implemented. "
                                      "Supported values: ['peak_mass'].")
        if getattr(self, "model", None) is None:
            raise RuntimeError("Model not initialised.  Call set_model() first.")
        from .period_summary import sm_components, summarise_batch
        mu, sg, w = sm_components(self)
        xr = self._xdata_raw[:, 0] if self.ndim > 1 else self._xdata_raw
        span = np.array([float(xr.max() - xr.min())])
        f = lambda v: None if v is None else np.array([float(v)])
        if n_peaks is None:
            n_peaks = getattr(self, "_fit_num_mixtures_effective", None)
        return summarise_batch(mu[None], sg[None], w[None], span, fmin=f(min_freq), fmax=f(max_freq),
                               n_grid=n_grid, peak_threshold_rel=peak_threshold_rel, n_peaks=n_peaks,
                               mass_level=mass_level, classify_lsp=classify_lsp)[0]

    def write_period_summary_outputs(self, text_file=None, png_file=None, json_file=None, summary=None,
                                     include_components=True, include_peaks=True,
                                     include_psd_info=False, include_psd_in_json=False,
                                     summary_kwargs=None, **kwargs):
        """lightcurve.py:8862-8990: the text report and / or the JSON export of the period summary
        (figures are outside the path: ``png_file`` raises)."""
        if png_file is not None:
            raise UnsupportedModel("write_period_summary_outputs: plotting is outside the B200 path")
        if summary is None:
            summary = self.get_period_summary(**(summary_kwargs or {}))
        elif summary_kwargs:
            warnings.warn("summary_kwargs are ignored because a pre-computed summary was supplied "
                          "via the summary= argument.", UserWarning, stacklevel=2)
        if text_file is not None:
            summary.write_text(text_file, include_components=include_components,
                               include_peaks=include_peaks, include_psd_info=include_psd_info)
        if json_file is not None:
            summary.write_json(json_file, include_psd=include_psd_in_json)
        return summary

    # ---- posterior prediction (lightcurve.py:9607-9640, 9849-9880: the body of plot()) -----
    def predict(self, x_fine_raw=None, n_points=10000):
        """``observed_pred = self.likelihood(self.model(x_fine_transformed))`` on the GPU (N1).

        ``x_fine_raw``: raw-unit test inputs ([m] for 1-D data, [m, 2] for 2-D); default: the
        reference's 10000-point grid across the time range (lightcurve.py:9624).  Returns
        ``{"x", "mean", "variance", "lower", "upper"}`` (numpy; transformed-y units like
        GPyTorch's ``observed_pred``): ``variance`` is the exact latent variance plus the learned
        homoskedastic noise (a FixedNoise likelihood adds nothing at new inputs, as GPyTorch
        warns), ``lower/upper = mean -/+ 2 stddev`` (``confidence_region``)."""
        from . import ops
        from .mll import engine_device, pack_model
        if x_fine_raw is None:
            if self.ndim != 1:
                raise ValueError("pass x_fine_raw [m, 2] (time, wavelength) for 2-D data")
            xr = self._xdata_raw
            x_fine_raw = torch.linspace(float(xr.min()), float(xr.max()), n_points)
        xf = torch.as_tensor(np.asarray(x_fine_raw) if not torch.is_tensor(x_fine_raw)
                             else x_fine_raw).to(self._xdata_raw.dtype)
        xt = xf if self.xtransform is None else self.xtransform.transform(xf)
        pk = pack_model(self.model, self.likelihood)
        dev = engine_device(pk.params[0])
        f64 = lambda t: t.detach().to(device=dev, dtype=torch.float64)
        x = self._xdata_transformed
        x = x if x.dim() > 1 else x.unsqueeze(-1)
        xs = xt if xt.dim() > 1 else xt.unsqueeze(-1)
        y_fit = self._ydata_transformed
        m_star = None
        if pk.external_mean:      # non-constant mean: condition on y - m(x), add m(x*) back
            with torch.no_grad():
                pdt = next(self.model.mean_module.parameters()).dtype
                y_fit = y_fit - self.model.mean_module(x.to(pdt)).to(y_fit.dtype)
                m_star = self.model.mean_module(xs.to(pdt)).to(torch.float64).cpu()
        mean, var, info = ops.sm_predict(
            f64(x).unsqueeze(0).contiguous(), f64(y_fit).unsqueeze(0).contiguous(),
            None if pk.fixed_noise is None else f64(pk.fixed_noise).unsqueeze(0).contiguous(),
            f64(pk.raw()).unsqueeze(0).contiguous(), pk.kinds.to(dev), pk.lb.to(dev),
            pk.ub.to(dev), None, f64(xs).unsqueeze(0).contiguous(), pk.kind, pk.Q, pk.learn_noise)
        code = int(info.item())
        if code < 0:
            from .gp import NanError, NotPSDError
            raise (NanError if code == -1 else NotPSDError)(
                "the covariance of the fitted model could not be factorised")
        mean, var = mean[0].cpu(), var[0].cpu()
        if m_star is not None:
            mean = mean + m_star
        if pk.learn_noise:
            # the learned-noise Parameter: its position differs between the spectral-mixture
            # layout [mean, w, mu, sigma, noise, ...] and the stationary one [mean, noise, ...]
            noise_par = pk.params[pk.noise_index]
            noise_con = getattr(self._owner_of(noise_par), "raw_noise_constraint", None)
            nv = noise_con.transform(noise_par) if noise_con is not None else noise_par
            var = var + float(nv.detach().reshape(-1)[0])
        std = var.clamp_min(1e-9).sqrt()      # MultivariateNormal.stddev clamps the variance
        return {"x": xf.cpu().numpy(), "mean": mean.numpy(), "variance": var.numpy(),
                "lower": (mean - 2 * std).numpy(), "upper": (mean + 2 * std).numpy()}

    def _owner_of(self, param):
        for mod in list(self.model.modules()) + list(self.likelihood.modules()):
            for p in mod._parameters.values():
                if p is param:
                    return mod
        return None

    # ---- Lomb-Scargle initialisation (lightcurve.py:4214-4611), on the GPU (N2) -----------
    def fit_LS(self, freq_only=False, num_peaks=1, single_threshold=0.05, Nyquist_factor=5,
               return_full=False, device=None, fap_method=None, use_best_band_init=True,
               n_samples=100, **kwargs):
        """``fit_LS`` (pgmuvi/lightcurve.py:4214-4611): the periodogram on astropy's
        ``autofrequency`` grid, the ``num_peaks`` highest peaks ``Nyquist_factor`` samples apart
        and their significance mask (Benjamini-Hochberg over the per-peak false-alarm
        probabilities, after a gate on the highest peak).  Computed by ``pgm_lombscargle_f64`` /
        ``pgm_ls_peaks_f64`` (exact floating-mean periodogram; the reference's astropy call uses
        its FFT approximation beyond 200 frequencies).
        1-D: 'davies' bound on the maximum, single-frequency FAPs per peak.
        2-D (multiband, ``:4372-4497``): ``use_best_band_init`` (default) takes grid and
        periodogram from the most-sampled band, else the chi2-weighted multiband periodogram;
        FAP method default 'phase_scramble' (``n_samples`` null periodograms in one launch;
        also 'bootstrap', 'analytical', 'calibrated') - :mod:`pgmuvi_b200.lombscargle`."""
        from . import lombscargle as ls
        dev = torch.device(device) if device is not None else torch.device("cuda:0")
        if self.ndim > 1:
            xr = self._xdata_raw
            has_err = getattr(self, "_yerr_transformed", None) is not None
            pf, sm, freq, power = ls.fit_ls_multiband(
                xr[:, 0].cpu().numpy(), self._ydata_raw.cpu().numpy(), xr[:, 1].cpu().numpy(),
                self._yerr_raw.cpu().numpy() if has_err else None, num_peaks=num_peaks,
                single_threshold=single_threshold, nyquist_factor=Nyquist_factor,
                fap_method=fap_method, use_best_band_init=use_best_band_init,
                n_samples=n_samples, device=dev)
            o = lambda a, dt=None: torch.as_tensor(np.asarray(a), dtype=dt or self.xdata.dtype,
                                                   device=self.xdata.device)
            if freq_only:
                return o(freq), o(power)
            if return_full:
                return o(pf), o(sm, torch.bool), o(freq), o(power)
            return o(pf), o(sm, torch.bool)
        t = self._xdata_raw.to(dev, torch.float64).unsqueeze(0)
        y = self._ydata_raw.to(dev, torch.float64).unsqueeze(0)
        has_err = getattr(self, "_yerr_transformed", None) is not None
        dy = self._yerr_raw.to(dev, torch.float64).unsqueeze(0) if has_err else None
        out_t = lambda a, dt=None: torch.as_tensor(a, dtype=dt or self.xdata.dtype,
                                                   device=self.xdata.device)
        f0, df, nf, power = ls.lombscargle(t, y, dy, nyquist_factor=Nyquist_factor)
        if freq_only or return_full:
            freq = (f0[0] + df[0] * torch.arange(int(nf[0]), device=dev, dtype=torch.float64))
            freq_t, power_t = out_t(freq.cpu()), out_t(power[0].cpu())
            if freq_only:
                return freq_t, power_t
        freqs, sig = ls.fit_ls_batch(t, y, dy, num_peaks=num_peaks,
                                     single_threshold=single_threshold,
                                     nyquist_factor=Nyquist_factor)
        keep = ~np.isnan(freqs[0])
        pf, sm = out_t(freqs[0][keep]), out_t(sig[0][keep], torch.bool)
        return (pf, sm, freq_t, power_t) if return_full else (pf, sm)

    def _mls_initial_frequencies(self, num_mixtures, constraint_set, peaks=None, f_cap=None):
        """Choice of seed frequencies from the periodogram peaks (lightcurve.py:5475-5660,
        1-D branch): peaks outside [1/span, constraint-set limit] are dropped; significant peaks
        first, then the others, then evenly spaced padding.  ``peaks`` = precomputed
        ``(peak_freqs, significance_mask)`` (``fit_batch`` runs one periodogram launch for all
        its light curves)."""
        t = self._xdata_raw[:, 0] if self.ndim > 1 else self._xdata_raw
        span = float(t.max() - t.min())
        f_lo = 1.0 / span if span > 0 else 0.0
        d = torch.diff(torch.sort(t).values)
        d = d[d > 0]
        f_hi = 1.0 / (2.0 * float(d.min())) if len(d) else float("inf")
        cs_lo, cs_hi = f_lo, float("inf")
        if constraint_set is not None and constraint_set in CONSTRAINT_SETS:
            pb = CONSTRAINT_SETS[constraint_set].get("period")
            if pb is not None:
                (pl, pl_on), (pu, pu_on) = pb["lower"], pb["upper"]
                if pl_on and pl is not None:
                    cs_hi = min(cs_hi, 1.0 / pl)
                if pu_on and pu is not None:
                    cs_lo = max(cs_lo, 1.0 / pu)
        if f_cap is not None:      # best-band Nyquist (lightcurve.py:5533-5552)
            cs_hi = min(cs_hi, f_cap)
            f_hi = cs_hi
        freqs, sig = peaks if peaks is not None else self.fit_LS(
            num_peaks=max(num_mixtures or 1, 10))
        if len(freqs) and cs_lo > 0:
            ok = (freqs >= cs_lo) & (freqs <= cs_hi)
            if not bool(ok.all()):
                warnings.warn(f"{int((~ok).sum())} MLS peak(s) fell outside the allowed frequency "
                              f"range [{cs_lo:.4g}, {cs_hi:.4g}] and were excluded from the "
                              "initialisation.", RuntimeWarning, stacklevel=3)
                freqs, sig = freqs[ok], sig[ok]
        if len(freqs) == 0:
            warnings.warn("MLS periodogram returned no peaks; falling back to "
                          f"num_mixtures={num_mixtures or 4} with default initialisation.",
                          RuntimeWarning, stacklevel=3)
            return None, num_mixtures or 4
        sig_f, insig_f = freqs[sig], freqs[~sig]
        if num_mixtures is None:
            init = sig_f if len(sig_f) else freqs[:1]
            return init, len(init)
        if num_mixtures <= len(sig_f):
            return sig_f[:num_mixtures], num_mixtures
        init = torch.cat([sig_f, insig_f[:num_mixtures - len(sig_f)]])
        n_pad = num_mixtures - len(init)
        if n_pad > 0:
            lo, hi = f_lo, f_hi
            if cs_lo > 0:
                lo, hi = max(lo, cs_lo), min(hi, cs_hi)
            if hi > lo:
                warnings.warn(f"Only {len(init)} MLS peak(s) found but {num_mixtures} were "
                              f"requested. Padding with {n_pad} evenly-spaced frequencies in "
                              f"[{lo:.4g}, {hi:.4g}].", RuntimeWarning, stacklevel=3)
                pad = torch.linspace(lo, hi, n_pad + 2, dtype=init.dtype)[1:-1]
            else:
                pad = init.new_full((n_pad,), float(init[-1]))
            init = torch.cat([init, pad])
        return init, num_mixtures

    # ---- fit (lightcurve.py:5211-5882) -------------------------------------------------
    def _get_best_sampled_band_lc(self):
        """1-D light curve of the band with the most points (lightcurve.py:5512-5520 uses it for
        ``use_best_band_init``): same transforms off, no sub-sampling."""
        wl = self._xdata_raw[:, 1]
        vals, counts = torch.unique(wl, return_counts=True)
        m = wl == vals[int(torch.argmax(counts))]
        err = self._yerr_raw[m] if hasattr(self, "_yerr_raw") else None
        return Lightcurve(self._xdata_raw[m, 0], self._ydata_raw[m], yerr=err, max_samples=None)

    def fit(self, model=None, likelihood=None, num_mixtures=None, guess=None, periods=None,
            use_mls_init=True, use_best_band_init=False, constraint_set=None, grid_size=2000,
            cuda=False, training_iter=300, max_cg_iterations=None, optim="AdamW", miniter=None,
            stop=1e-5, lr=0.1, stopavg=30, variance=False, **kwargs):
        """The reference's signature and defaults (lightcurve.py:5211-5232): AdamW, lr 0.1, 300
        iterations, stop 1e-5, stopavg 30, ``miniter=None -> training_iter`` (so the early stop
        never fires, SURVEY F10), ``use_mls_init=True``.

        MLS initialisation (lightcurve.py:5475-5688): 1-D spectral-mixture models are seeded from
        the GPU Lomb-Scargle periodogram; 2-D ones from the best-sampled band's 1-D periodogram
        when ``use_best_band_init`` is set (:5512-5532, 5777-5839).  As in the reference, ANY
        failure of that step (here: no CUDA device, or the multiband periodogram, which is
        outside the path) degrades to a ``RuntimeWarning`` and the default initialisation with
        ``num_mixtures`` (4 if not given) - :5668-5688.  ``periods`` / ``guess`` take precedence.
        ``grid_size`` only concerns the KISS-GP models (outside the path);
        ``max_cg_iterations`` is GPyTorch's CG budget (:5852-5870) and has no effect on the
        exact-Cholesky path.  ``cuda`` is accepted: the engine always runs on the GPU."""
        if num_mixtures is not None:
            if isinstance(num_mixtures, bool) or not isinstance(num_mixtures, int):
                raise TypeError("`num_mixtures` must be a positive integer or None, "
                                f"got {num_mixtures!r} of type {type(num_mixtures)!r}.")
            if num_mixtures < 1:
                raise ValueError("`num_mixtures` must be a positive integer or None, "
                                 f"got {num_mixtures}.")
        if likelihood is not None or not hasattr(self, "likelihood"):
            self.set_likelihood(likelihood, variance=variance)
        init_freqs = None
        if periods is not None:
            pt = torch.as_tensor(np.asarray(periods, dtype=np.float64)).flatten()
            if pt.numel() == 0:
                raise ValueError("When providing explicit `periods`, the sequence must be "
                                 "non-empty.")
            if not torch.isfinite(pt).all():
                raise ValueError("All values in `periods` must be finite (no NaN or inf).")
            if not (pt > 0).all():
                raise ValueError("All values in `periods` must be strictly positive.")
            init_freqs = 1.0 / pt
            num_mixtures = len(pt)
        elif use_mls_init and isinstance(model, str) and model in _SM_MODELS \
                and model not in _NO_MIXTURE_MODELS:
            try:
                if self.ndim > 1 and use_best_band_init:
                    bb = self._get_best_sampled_band_lc()
                    peaks = bb.fit_LS(num_peaks=max(num_mixtures or 1, 10))
                    tb = bb._xdata_raw.sort().values
                    db = tb[1:] - tb[:-1]
                    db = db[db > 0]
                    nyq = float(1.0 / (2.0 * db.min())) if len(db) else float("inf")
                    init_freqs, num_mixtures = self._mls_initial_frequencies(
                        num_mixtures, constraint_set, peaks, f_cap=nyq)
                else:
                    init_freqs, num_mixtures = self._mls_initial_frequencies(
                        num_mixtures, constraint_set)
            except Exception as exc:      # lightcurve.py:5668-5688
                if num_mixtures is None:
                    num_mixtures = 4
                init_freqs = None
                warnings.warn("MLS-based initialisation failed; falling back to "
                              f"num_mixtures={num_mixtures}. Original error was: {exc}",
                              RuntimeWarning, stacklevel=2)
        if num_mixtures is None:
            num_mixtures = 4
        if model is not None or not hasattr(self, "model"):
            if model is None:
                raise ValueError("""You must provide a model""")
            self.set_model(model, self.likelihood, num_mixtures=num_mixtures, **kwargs)
        if not self._constraints_set:
            self.set_default_constraints(constraint_set=constraint_set)
        hypers = {}
        sm = getattr(self.model, "covar_module", None)
        ard = getattr(sm, "ard_num_dims", None) if hasattr(sm, "raw_mixture_means") else None
        if init_freqs is not None and ard == 1 and self.ndim == 1:
            hypers["covar_module.mixture_means"] = init_freqs
        elif init_freqs is not None and use_best_band_init and self.ndim > 1 and ard == 2:
            # time frequencies from the best band, 1 / wavelength span as the wavelength
            # placeholder (lightcurve.py:5777-5839)
            wl = self._xdata_raw[:, 1]
            wspan = float(wl.max() - wl.min())
            f2 = torch.stack([init_freqs, init_freqs.new_full((len(init_freqs),),
                                                              1.0 / wspan if wspan > 0 else 1e-6)], 1)
            if self.xtransform is None:
                con = getattr(sm, "raw_mixture_means_constraint", None)
                if con is not None and hasattr(con, "lower_bound"):
                    hi = float(con.upper_bound) if hasattr(con, "upper_bound") else float("inf")
                    f2 = f2.clamp(min=float(con.lower_bound), max=hi)
            hypers["covar_module.mixture_means"] = f2
        if guess is not None:
            hypers.update(guess)
        if hypers:
            self.set_hypers(hypers)
        if miniter is None:
            miniter = training_iter
        self.model.train()
        self.likelihood.train()
        self.results = train(self, maxiter=training_iter, miniter=miniter, stop=stop, lr=lr,
                             optim=optim, stopavg=stopavg)
        self._fitted = True
        return self.results


class UnsupportedModel(NotImplementedError):
    pass
