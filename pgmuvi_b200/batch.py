"""Batched engine: many independent light curves on one GPU (or sharded over ranks).

pgmuvi has no batch API (one ``Lightcurve`` = one source, SURVEY.md F11); surveys loop over
``Lightcurve.fit``.  ``BatchEngine`` is the B200-native replacement of that loop for the
hot path: ``evaluate`` = one ``model(train_x) -> -mll -> backward`` pass for every light
curve (pgmuvi/trainers.py:179-181), ``fit`` = the whole ``trainers.train`` loop
(trainers.py:177-207) on device.  Host buffers in, host buffers out; device staging buffers
are owned by the engine and reused.

Multi-GPU: light curves are independent, so ranks take contiguous shards and nothing is
exchanged inside the loop; ``gather_results`` does the single end-of-job all-gather.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional

import numpy as np
import torch

from . import _lib, ops
from ._lib import (KIND_SM1D, OPT_ADAM, OPT_ADAMW, OPT_SGD)

OPTIM_KINDS = {"SGD": OPT_SGD, "Adam": OPT_ADAM, "AdamW": OPT_ADAMW}


def shard_range(total: int, rank: int, world: int):
    """Contiguous, balanced split of ``total`` light curves: returns (start, stop)."""
    base, rem = divmod(total, world)
    start = rank * base + min(rank, rem)
    return start, start + base + (1 if rank < rem else 0)


def optimizer_defaults(optim: str, eps: float = 1e-8):
    """torch.optim defaults as trainers.py:141-147 constructs them."""
    if optim not in OPTIM_KINDS:
        raise ValueError("optim must be either 'SGD', 'Adam', 'AdamW'")
    return dict(optim_kind=OPTIM_KINDS[optim], beta1=0.9, beta2=0.999, eps=eps,
                weight_decay=0.01 if optim == "AdamW" else 0.0)


@dataclass
class HostBatch:
    """Host-side (preferably pinned) inputs of a batch, float64 / int32, C-contiguous."""
    x: torch.Tensor                      # [B, n, d]
    y: torch.Tensor                      # [B, n]
    noise: Optional[torch.Tensor]        # [B, n] variance or None
    raw: torch.Tensor                    # [B, P]
    kinds: torch.Tensor                  # [P] int32
    lb: torch.Tensor                     # [B, P] or [P]
    ub: torch.Tensor
    n_valid: Optional[torch.Tensor] = None  # [B] int32

    @staticmethod
    def from_numpy(d, pin=True):
        def t(a, dt=torch.float64):
            if a is None:
                return None
            out = torch.as_tensor(np.ascontiguousarray(a), dtype=dt)
            return out.pin_memory() if pin and torch.cuda.is_available() else out
        return HostBatch(t(d["x"]), t(d["y"]), t(d.get("noise")), t(d["raw"]),
                         t(d["kinds"], torch.int32), t(d["lb"]), t(d["ub"]),
                         t(d.get("n_valid"), torch.int32))

    def slice(self, start, stop):
        s = lambda a: None if a is None else a[start:stop]
        per_lc = self.lb.dim() == 2
        return HostBatch(s(self.x), s(self.y), s(self.noise), s(self.raw), self.kinds,
                         s(self.lb) if per_lc else self.lb, s(self.ub) if per_lc else self.ub,
                         s(self.n_valid))

    def h2d_bytes(self):
        return sum(t.numel() * t.element_size() for t in
                   (self.x, self.y, self.noise, self.raw, self.kinds, self.lb, self.ub,
                    self.n_valid) if t is not None)


class BatchEngine:
    """Owns the device buffers for batches of one model family on one GPU."""

    def __init__(self, kind=KIND_SM1D, Q=4, learn_noise=False, device=None):
        if not torch.cuda.is_available():
            raise RuntimeError("pgmuvi_b200.BatchEngine needs a CUDA device (no CPU fallback)")
        self.kind, self.Q, self.learn_noise = kind, Q, learn_noise
        self.device = torch.device(device if device is not None
                                   else f"cuda:{torch.cuda.current_device()}")
        self._dev = {}
        self._out = {}

    # -- staging -------------------------------------------------------------------------
    def _stage(self, name, host):
        if host is None:
            return None
        buf = self._dev.get(name)
        if buf is None or buf.shape != host.shape or buf.dtype != host.dtype:
            buf = torch.empty(host.shape, dtype=host.dtype, device=self.device)
            self._dev[name] = buf
        buf.copy_(host, non_blocking=True)
        return buf

    def upload(self, hb: HostBatch):
        """Host -> device copy of one batch (async on the current stream)."""
        return dict(x=self._stage("x", hb.x), y=self._stage("y", hb.y),
                    noise=self._stage("noise", hb.noise), raw=self._stage("raw", hb.raw),
                    kinds=self._stage("kinds", hb.kinds), lb=self._stage("lb", hb.lb),
                    ub=self._stage("ub", hb.ub), n_valid=self._stage("n_valid", hb.n_valid))

    def _host_out(self, name, dev):
        buf = self._out.get(name)
        if buf is None or buf.shape != dev.shape or buf.dtype != dev.dtype:
            buf = torch.empty(dev.shape, dtype=dev.dtype).pin_memory()
            self._out[name] = buf
        buf.copy_(dev, non_blocking=True)
        return buf

    # -- device-resident calls -------------------------------------------------------------
    def tail_split(self, B, d_in):
        """How many light curves of a batch of B go to the staged engine so that the LAST WAVE of
        the fused kernel's persistent grid stays balanced.  The fused kernel holds `grid` = SMs x 2
        blocks, one light curve per block at a time; with r = B mod grid light curves in the last
        wave and r > SMs, r - SMs SMs run two blocks while the others run one and then idle
        (B = 512 on 148 SMs: 4.52 ms, the time of 592).  Handing those r - SMs light curves to the
        staged engine on a second stream - whose tile-sized blocks fill the slots that free up on
        EVERY SM when the blocks with no further light curve exit - finishes the shard in about the
        time of B - (r - SMs) (measured: profiles/r02m_tail_balance.log).  0 = no split."""
        import os
        if os.environ.get("PGM_TAIL_BALANCE", "1") == "0" or B <= 0:
            return 0
        grid = _lib.load().pgm_fused_grid(int(d_in), self.Q, self.kind)
        sms = torch.cuda.get_device_properties(self.device).multi_processor_count
        # worth it while the last wave is a noticeable share of the batch (B = 4096: 0.6 %)
        if grid != 2 * sms or B <= grid or B > 8 * grid:
            return 0
        r = B % grid
        return r - sms if r > sms else 0

    def evaluate_device(self, d, want_grad=True):
        B = d["y"].shape[0]
        k = self.tail_split(B, d["x"].shape[2] if d["x"].dim() == 3 else 1)
        args = (self.kind, self.Q, self.learn_noise, want_grad)
        if k == 0:
            return ops.sm_mll_grad(d["x"], d["y"], d["noise"], d["raw"], d["kinds"], d["lb"],
                                   d["ub"], d["n_valid"], *args)
        cut = lambda t, a, z: None if t is None else (t[a:z] if t.dim() and t.shape[0] == B else t)
        part = lambda a, z: (cut(d["x"], a, z), cut(d["y"], a, z), cut(d["noise"], a, z),
                             cut(d["raw"], a, z), d["kinds"],
                             d["lb"][a:z] if d["lb"].dim() == 2 else d["lb"],
                             d["ub"][a:z] if d["ub"].dim() == 2 else d["ub"], cut(d["n_valid"], a, z))
        cur = torch.cuda.current_stream(self.device)
        if getattr(self, "_side", None) is None:
            self._side = torch.cuda.Stream(self.device)
        self._side.wait_stream(cur)
        m0, g0, i0 = ops.sm_mll_grad(*part(0, B - k), *args)          # asynchronous
        with torch.cuda.stream(self._side):                           # blocks on its own stream only
            m1, g1, i1 = ops.sm_mll_grad_staged(*part(B - k, B), *args)
        cur.wait_stream(self._side)
        for t in (m1, g1, i1):          # allocated on the side stream, consumed on the current one
            t.record_stream(cur)
        return torch.cat([m0, m1]), torch.cat([g0, g1]), torch.cat([i0, i1])

    def fit_device(self, d, maxiter=300, miniter=None, stop=1e-5, lr=0.1, optim="AdamW",
                   eps=1e-8, stopavg=30, keep_history=True):
        """trainers.train for every light curve; ``d['raw']`` is updated in place.
        Defaults are ``Lightcurve.fit``'s (lightcurve.py:5223-5229: AdamW, lr 0.1, 300
        iterations, stop 1e-5, stopavg 30, miniter=None -> training_iter)."""
        od = optimizer_defaults(optim, eps)
        miniter = maxiter if miniter is None else miniter
        return ops.sm_fit(d["x"], d["y"], d["noise"], d["raw"], d["kinds"], d["lb"], d["ub"],
                          d["n_valid"], self.kind, self.Q, self.learn_noise, od["optim_kind"],
                          float(lr), od["beta1"], od["beta2"], od["eps"], od["weight_decay"],
                          int(maxiter), int(miniter), float(stop or 0.0), int(stopavg),
                          bool(keep_history))

    # -- host in / host out (the call a user makes) ---------------------------------------
    def evaluate(self, hb: HostBatch, want_grad=True):
        """MLL (+ gradient w.r.t. raw parameters) of every light curve in the batch.
        Returns pinned host tensors (mll [B], grad [B,P], info [B]); synchronises."""
        d = self.upload(hb)
        mll, grad, info = self.evaluate_device(d, want_grad)
        out = (self._host_out("mll", mll), self._host_out("grad", grad),
               self._host_out("info", info))
        torch.cuda.current_stream().synchronize()
        return out

    def fit(self, hb: HostBatch, **kw):
        """Fit every light curve; returns dict(loss [iters,B], raw [B,P], raw_hist, n_iter,
        info) on the host."""
        d = self.upload(hb)
        loss, raw_hist, n_iter, info = self.fit_device(d, **kw)
        out = dict(loss=loss.cpu(), raw=d["raw"].cpu(), raw_hist=raw_hist.cpu(),
                   n_iter=n_iter.cpu(), info=info.cpu())
        return out


def gather_results(local: torch.Tensor, counts=None):
    """All-gather per-light-curve results [B_local, ...] over the ranks of the default
    process group (NCCL on GPUs, gloo on CPU); shards may be uneven (``counts`` = list of
    per-rank sizes, needed only then).  No-op without torch.distributed."""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return local
    world = dist.get_world_size()
    if counts is None or len(set(counts)) == 1:
        out = [torch.empty_like(local) for _ in range(world)]
        dist.all_gather(out, local.contiguous())
        return torch.cat(out, 0)
    mx = max(counts)
    pad = torch.zeros((mx,) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
    pad[: local.shape[0]] = local
    out = [torch.empty_like(pad) for _ in range(world)]
    dist.all_gather(out, pad)
    return torch.cat([o[:c] for o, c in zip(out, counts)], 0)


def _pack_batch(lcs, packs, who):
    """Pad and pack set-up light curves of one model family into host float64 buffers
    ``(x [B, n_max, d], y [B, n_max], noise [B, n_max] or None, raw, lb, ub [B, P], n_valid [B])``
    (padding beyond ``n_valid``: zeros, unit noise)."""
    pk0 = packs[0]
    for pk in packs[1:]:
        if (pk.kind, pk.Q, pk.d, pk.learn_noise, pk.P) != (pk0.kind, pk0.Q, pk0.d, pk0.learn_noise,
                                                        pk0.P) or not torch.equal(pk.kinds,
                                                                                  pk0.kinds):
            raise ValueError(f"{who}: all light curves must share one model family, number "
                             "of mixtures and likelihood type")
    B = len(lcs)
    n_each = [int(lc._ydata_transformed.shape[0]) for lc in lcs]
    n_max = max(n_each)
    d, P = pk0.d, pk0.P
    x = torch.zeros(B, n_max, d, dtype=torch.float64)
    y = torch.zeros(B, n_max, dtype=torch.float64)
    has_fixed = pk0.fixed_noise is not None
    noise = torch.ones(B, n_max, dtype=torch.float64) if has_fixed else None
    raw = torch.zeros(B, P, dtype=torch.float64)
    lb = torch.zeros(B, P, dtype=torch.float64)
    ub = torch.zeros(B, P, dtype=torch.float64)
    for b, (lc, pk) in enumerate(zip(lcs, packs)):
        n = n_each[b]
        xt = lc._xdata_transformed.detach().to(torch.float64)
        x[b, :n] = xt if xt.dim() > 1 else xt.unsqueeze(-1)
        y[b, :n] = lc._ydata_transformed.detach().to(torch.float64)
        if has_fixed:
            noise[b, :n] = pk.fixed_noise.detach().to(torch.float64)
        raw[b] = pk.raw().detach().to(torch.float64)
        lb[b], ub[b] = pk.lb, pk.ub
    return x, y, noise, raw, lb, ub, torch.tensor(n_each, dtype=torch.int32)


def fit_batch(lightcurves, model="1D", likelihood=None, num_mixtures=None, periods=None,
              use_mls_init=False, constraint_set=None, training_iter=300, optim="AdamW",
              miniter=None, stop=1e-5, lr=0.1, stopavg=30, variance=False, keep_history=True,
              device=None, **kwargs):
    """``[lc.fit(model=..., ...) for lc in lightcurves]`` as ONE launch of the fused training
    kernel per rank (the survey-scale loop pgmuvi users write today, SURVEY F11).

    Every ``Lightcurve`` is set up exactly as ``Lightcurve.fit`` would (likelihood, model,
    default constraints, Lomb-Scargle or explicit period seeds: the same host code, so the
    packed parameters are the single-source ones), the ragged batch is padded and packed once,
    ``pgm_sm_fit`` runs the whole optimisation for all of them, and each object gets its fitted
    parameters and its ``results`` dict back.  Under ``torch.distributed`` (one process per
    GPU) each rank fits ``shard_range(B, rank, world)`` and the fitted raw parameters, losses
    and iteration counts are all-gathered once at the end (no collective inside the loop).

    ``periods``: None, one sequence for all light curves, or one sequence per light curve.
    ``use_mls_init``: seed 1-D models from the batched GPU periodogram (one launch for all).
    Returns ``dict(loss [iters, B], raw [B, P], n_iter [B], info [B])`` plus, for spectral-
    mixture models, ``periods`` / ``weights`` [B, Q] (component values, ``get_periods``) and
    ``dominant_period`` [B] (highest peak of the summed PSD, ``get_period_summary``'s first
    stage, one launch for the batch) - host tensors / arrays, all B light curves on every rank."""
    import torch.distributed as dist
    from .mll import UnsupportedModelError, engine_device, pack_model
    from .trainers import history_from_raw

    lcs = list(lightcurves)
    B = len(lcs)
    if B == 0:
        raise ValueError("fit_batch needs at least one light curve")
    per_lc_periods = (periods is not None and len(periods) == B
                      and np.ndim(periods[0]) >= 1)
    # ---- host set-up, identical to Lightcurve.fit (lightcurve.py:5211-5850) -----------------
    seeds = [None] * B
    nmix = [num_mixtures] * B
    if periods is not None:
        for b in range(B):
            p = np.asarray(periods[b] if per_lc_periods else periods, dtype=np.float64).ravel()
            if p.size == 0 or not np.isfinite(p).all() or not (p > 0).all():
                raise ValueError("`periods` must be non-empty, finite and strictly positive")
            seeds[b] = torch.as_tensor(1.0 / p)
            if nmix[b] is None:
                nmix[b] = p.size
    elif use_mls_init and all(lc.ndim == 1 for lc in lcs):
        # one periodogram + peak-search launch for all light curves (lightcurve.py:4214-4611),
        # then the reference's per-source peak selection (lightcurve.py:5475-5660)
        from . import lombscargle as ls
        ldev = torch.device(device) if device is not None else torch.device("cuda:0")
        ns = [int(lc._xdata_raw.shape[0]) for lc in lcs]
        tt = torch.zeros(B, max(ns), dtype=torch.float64)
        yy = torch.zeros(B, max(ns), dtype=torch.float64)
        have_err = all(getattr(lc, "_yerr_transformed", None) is not None for lc in lcs)
        ee = torch.ones(B, max(ns), dtype=torch.float64) if have_err else None
        for b, lc in enumerate(lcs):
            tt[b, :ns[b]] = lc._xdata_raw.to(torch.float64)
            yy[b, :ns[b]] = lc._ydata_raw.to(torch.float64)
            if have_err:
                ee[b, :ns[b]] = lc._yerr_raw.to(torch.float64)
        k = max(num_mixtures or 1, 10)
        freqs, sig = ls.fit_ls_batch(tt.to(ldev), yy.to(ldev), None if ee is None else ee.to(ldev),
                                     torch.tensor(ns, dtype=torch.int32, device=ldev), num_peaks=k)
        for b, lc in enumerate(lcs):
            keep = ~np.isnan(freqs[b])
            pf = torch.as_tensor(freqs[b][keep], dtype=lc.xdata.dtype)
            sm = torch.as_tensor(sig[b][keep], dtype=torch.bool)
            seeds[b], nmix[b] = lc._mls_initial_frequencies(num_mixtures, constraint_set, (pf, sm))
    packs = []
    for b, lc in enumerate(lcs):
        if likelihood is not None or not hasattr(lc, "likelihood"):
            lc.set_likelihood(likelihood, variance=variance)
        lc.set_model(model, lc.likelihood, num_mixtures=nmix[b], **kwargs)
        lc.set_default_constraints(constraint_set=constraint_set)
        if seeds[b] is not None and lc.ndim == 1:
            lc.set_hypers({"covar_module.mixture_means": seeds[b]})
        lc.model.train()
        lc.likelihood.train()
        packs.append(pack_model(lc.model, lc.likelihood))
    pk0 = packs[0]
    if any(pk.external_mean for pk in packs):
        # non-constant mean modules keep their parameters on the host (autograd through
        # y - m(x), pgm_sm_mll_grad_alpha_f64): the one-launch batch loop cannot train them
        raise UnsupportedModelError(
            f"fit_batch: model {model!r} has a non-constant mean function, whose parameters are "
            "optimised on the host; fit these light curves one by one with Lightcurve.fit")
    # ---- pack the (ragged) batch ----------------------------------------------------------
    x, y, noise, raw, lb, ub, n_valid = _pack_batch(lcs, packs, "fit_batch")
    if x.shape[1] > 2048:
        raise ValueError("fit_batch: light curves longer than 2048 points go through "
                         "Lightcurve.fit (staged whole-device engine)")
    P = pk0.P
    # ---- shard, fit, gather ----------------------------------------------------------------
    distributed = dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
    world = dist.get_world_size() if distributed else 1
    rank = dist.get_rank() if distributed else 0
    a, z = shard_range(B, rank, world)
    dev = torch.device(device) if device is not None else engine_device(pk0.params[0])
    od = optimizer_defaults(optim, 1e-8)
    miniter = training_iter if miniter is None else miniter
    to = lambda t: None if t is None else t[a:z].contiguous().to(dev)
    raw_dev = to(raw)
    if z > a:
        loss, raw_hist, n_iter, info = ops.sm_fit(
            to(x), to(y), to(noise), raw_dev, pk0.kinds.to(dev), to(lb), to(ub), to(n_valid),
            pk0.kind, pk0.Q, pk0.learn_noise, od["optim_kind"], float(lr), od["beta1"],
            od["beta2"], od["eps"], od["weight_decay"], int(training_iter), int(miniter),
            float(stop or 0.0), int(stopavg), bool(keep_history))
    else:   # more ranks than light curves
        loss = torch.zeros(training_iter, 0, dtype=torch.float64, device=dev)
        raw_hist = torch.zeros(training_iter + 1, 0, P, dtype=torch.float64, device=dev)
        n_iter = torch.zeros(0, dtype=torch.int32, device=dev)
        info = torch.zeros(0, dtype=torch.int32, device=dev)
    # local light curves get their history; everyone gets the fitted parameters
    if keep_history:
        rh = raw_hist.cpu()
        lh = loss.cpu()
        for b in range(a, z):
            k = int(n_iter[b - a])
            lc, pk = lcs[b], packs[b]
            pdt = pk.params[0].dtype
            ls_ = lh[:k, b - a].to(pdt).numpy()
            res = {"loss": [ls_[i] for i in range(k)],
                   "delta_loss": [ls_[i] - ls_[i - 1] for i in range(1, k)]}
            res.update(history_from_raw(rh[:k + 1, b - a], pk, lc.model, lc))
            lc.results = res
    counts = [shard_range(B, r, world)[1] - shard_range(B, r, world)[0] for r in range(world)]
    g = lambda t: gather_results(t.contiguous(), counts) if distributed else t
    raw_all = g(raw_dev).cpu()
    loss_all = g(loss.t().contiguous()).t().cpu()          # gather along the light-curve axis
    n_iter_all, info_all = g(n_iter).cpu(), g(info).cpu()
    for b, (lc, pk) in enumerate(zip(lcs, packs)):
        pk.scatter_raw_(raw_all[b])
        lc._fitted = True
    out = dict(loss=loss_all, raw=raw_all, n_iter=n_iter_all, info=info_all)
    if packs[0].Q > 0:      # spectral-mixture models: component periods + the PSD period summary
        from .period_summary import period_summary_batch, sm_components
        out["periods"] = np.stack([lc.get_periods()[0] for lc in lcs])
        out["weights"] = np.stack([lc.get_periods()[1] for lc in lcs])
        comps = [sm_components(lc) for lc in lcs]
        spans = []
        for lc in lcs:
            xr = lc._xdata_raw[:, 0] if lc.ndim > 1 else lc._xdata_raw
            spans.append(float(xr.max() - xr.min()))
        summ = period_summary_batch(torch.stack([c[0] for c in comps]),
                                    torch.stack([c[1] for c in comps]),
                                    torch.stack([c[2] for c in comps]),
                                    t_span=torch.tensor(spans, dtype=torch.float64)) \
            if dev.type == "cuda" else None
        if summ is not None:
            out["dominant_period"] = summ["dominant_period"]
    return out


def uncertainties_batch(lightcurves, device=None, budget_bytes=None):
    """:meth:`Lightcurve.parameter_uncertainties` for many set-up (usually fitted) light curves of
    one model family: the ragged batch is packed as ``fit_batch`` packs it and the Fisher matrices
    come from ``pgm_sm_fisher_f64`` in chunks whose workspace (``pgm_fisher_workspace_bytes``)
    stays within ``budget_bytes`` (default: 80 % of the free device memory).  Returns one dict per
    light curve, in order."""
    from . import mll
    from .mll import UnsupportedModelError, pack_model

    lcs = list(lightcurves)
    if not lcs:
        raise ValueError("uncertainties_batch needs at least one light curve")
    packs = [pack_model(lc.model, lc.likelihood) for lc in lcs]
    if any(pk.external_mean for pk in packs):
        raise UnsupportedModelError("parameter uncertainties: models with a non-constant mean "
                                    "function are not supported")
    x, y, noise, raw, lb, ub, n_valid = _pack_batch(lcs, packs, "uncertainties_batch")
    pk0 = packs[0]
    B, n_max = y.shape
    dev = torch.device(device) if device is not None else mll.engine_device(pk0.params[0])
    if budget_bytes is None:
        budget_bytes = int(0.8 * torch.cuda.mem_get_info(dev)[0]) if dev.type == "cuda" else 1 << 62
    per_lc = ops.fisher_workspace_bytes(n_max, 2, pk0.d, pk0.Q, pk0.kind, pk0.learn_noise) - \
        ops.fisher_workspace_bytes(n_max, 1, pk0.d, pk0.Q, pk0.kind, pk0.learn_noise)
    chunk = int(max(1, min(65535, budget_bytes // max(per_lc, 1))))
    fisher = torch.empty(B, pk0.P, pk0.P, dtype=torch.float64)
    info = torch.empty(B, dtype=torch.int32)
    to = lambda t, a, z: None if t is None else t[a:z].contiguous().to(dev)
    for a in range(0, B, chunk):
        z = min(B, a + chunk)
        f, i = ops.sm_fisher(to(x, a, z), to(y, a, z), to(noise, a, z), to(raw, a, z),
                             pk0.kinds.to(dev), to(lb, a, z), to(ub, a, z), to(n_valid, a, z),
                             pk0.kind, pk0.Q, pk0.learn_noise)
        fisher[a:z], info[a:z] = f.cpu(), i.cpu()
    return [_uncertainties(lc, pk, fisher[b], int(info[b])) for b, (lc, pk) in
            enumerate(zip(lcs, packs))]


def _uncertainties(lc, pk, fisher, info):
    """Host assembly of one light curve: free-slot inverse of the Fisher matrix, then the delta
    method through ``Lightcurve._report`` (autograd) for every ``get_parameters`` entry."""
    from ._lib import CON_INTERVAL
    P = pk.P
    names, owner = [], []
    for i, (p, nm) in enumerate(zip(pk.params, pk.names)):
        k = p.numel()
        names += [nm if k == 1 else f"{nm}[{j}]" for j in range(k)]
        owner += [i] * k
    frozen = torch.tensor([pk.names[owner[s]] == "?" or (int(pk.kinds[s]) == CON_INTERVAL and
                                                         float(pk.lb[s]) == float(pk.ub[s]))
                           for s in range(P)])
    free = ~frozen
    Ff = fisher[free][:, free]
    dg = Ff.diagonal()
    ok = bool(torch.isfinite(Ff).all()) and bool((dg > 0).all())
    cov = torch.zeros(P, P, dtype=torch.float64)
    if ok:
        sc = dg.rsqrt()
        L, inf = torch.linalg.cholesky_ex(Ff * sc[:, None] * sc[None, :])
        ok = int(inf) == 0
        if ok:
            cf = torch.cholesky_inverse(L) * sc[:, None] * sc[None, :]
    idx = torch.nonzero(free).flatten()
    cov[idx[:, None], idx[None, :]] = cf if ok else float("nan")
    stderr, o = {}, {}
    pos = 0
    for i, p in enumerate(pk.params):
        o[id(p)] = (pos, p.numel())
        pos += p.numel()
    for name, param in lc.model.named_parameters():
        key = ".".join(c.lstrip("raw_") for c in name.split(".")) if "raw" in name else name
        ent = lc._model_pars.get(key)
        con = ent["module"]._modules.get(ent["raw_name"] + "_constraint") if ent else None
        theta = (con.transform(param) if con is not None else param).detach().to(torch.float64)
        shape = lc._report(key, theta).shape       # get_parameters' shape (transforms broadcast)
        if id(param) not in o:
            stderr[key] = torch.zeros(shape, dtype=torch.float64)
            continue
        a, k = o[id(param)]
        J = torch.autograd.functional.jacobian(
            lambda th: lc._report(key, th.reshape(param.shape)).reshape(-1).to(torch.float64),
            theta.reshape(-1))
        var = torch.einsum("ij,jk,ik->i", J, cov[a:a + k, a:a + k], J)
        stderr[key] = var.clamp_min(0).sqrt().reshape(shape) if ok else \
            torch.full(shape, float("nan"), dtype=torch.float64)
    period_stderr = None
    mk = next((k for k in stderr if k.endswith("mixture_means")), None)
    if mk is not None:
        mu = lc.get_parameters()[mk].detach().to(torch.float64)
        period_stderr = (stderr[mk][:, 0, 0] / mu[:, 0, 0] ** 2).numpy()
    return {"names": names, "covariance": cov, "stderr": stderr, "period_stderr": period_stderr,
            "fisher_ok": ok, "fisher": fisher, "info": info}
