"""Base Gibbs loop (mirror of GibbsSampler.py:8-192).  State (alms, maps, D_l) stays in HBM across
iterations; only the binned D_l history, accept flags and timings come back to the host."""
import time

import numpy as np
import torch

from . import _dev, utils
from ._dev import f64


class SigmaRecorder():
    """Empirical spectra sigma^i of the sky samples of a run (the input of BlackwellRao): one (n_iter, lmax + 1) device buffer
    per spectrum, filled by device-to-device copies as the chain runs (no synchronisation) and copied to the host once."""

    def __init__(self, keys, n_iter, lmax):
        self.buf = {k: torch.empty((n_iter, lmax + 1), dtype=torch.float64, device=_dev.device()) for k in keys}

    def record(self, i, sigma):
        for k, b in self.buf.items():
            b[i].copy_(sigma[k])

    def result(self):
        return {k: b.cpu().numpy() for k, b in self.buf.items()}


class GibbsSampler():
    keep_sigma = False   # CenteredGibbs(keep_sigma=True): run() leaves the empirical spectra of its sky samples in sigma_history

    def __init__(self, pix_map, noise, beam_fwhm_deg, nside, lmax, polarization=False, bins=None, n_iter=10000,
                 gibbs_cr=False, rj_step=False, ula=False, *, verbose=False):
        self.noise = noise
        self.beam = beam_fwhm_deg
        self.nside = nside
        self.lmax = lmax
        self.polarization = polarization
        self.bins = bins
        self.pix_map = pix_map
        self.Npix = 12 * nside ** 2
        self.bl_map = self.compute_bl_map(beam_fwhm_deg)
        self.constrained_sampler = None
        self.cls_sampler = None
        self.n_iter = n_iter
        self.gibbs_cr = gibbs_cr
        self.rj_step = rj_step
        self.ula = True  # the reference ignores its `ula` argument (GibbsSampler.py:41, SURVEY appendix A.1)
        self.verbose = verbose
        if bins is None:
            if not polarization:
                self.bins = np.array([l for l in range(lmax + 2)])
            else:
                bins = np.array([l for l in range(2, lmax + 1)])
                self.bins = {"TT": bins, "EE": bins, "TE": bins, "BB": bins}
        else:
            self.bins = bins
        self.dls_to_cls_array = np.array([2 * np.pi / (l * (l + 1)) if l != 0 else 0 for l in range(lmax + 1)])

    def dls_to_cls(self, dls_):
        return dls_[:] * self.dls_to_cls_array

    def compute_bl_map(self, beam_fwhm_deg):
        """b_l expanded over the real alm layout (GibbsSampler.py:64-74); kept as a CUDA tensor."""
        fwhm_radians = (np.pi / 180) * beam_fwhm_deg
        bl_gauss = _dev.gauss_beam(fwhm_radians, self.lmax)
        return utils.expand_per_l(f64(bl_gauss), 0)

    def _unfold(self, binned, pol):
        return utils.unfold_bins(f64(binned[pol]), self.bins[pol])

    def run_polarization(self, dls_init):
        """Mirror of GibbsSampler.run_polarization (GibbsSampler.py:118-180); same return tuple."""
        h_accept_cr = []
        h_duration_cr = []
        h_duration_cls_sampling = []
        h_dls = {"EE": [], "BB": []}
        binned_dls = {k: f64(v) for k, v in dls_init.items()}
        dls_unbinned = {"EE": self._unfold(binned_dls, "EE"), "BB": self._unfold(binned_dls, "BB")}
        if self.rj_step == True or self.gibbs_cr == True or self.ula == True:
            skymap, accept = self.constrained_sampler.sample(dls_unbinned)
        h_dls["EE"].append(_dev.to_host(binned_dls["EE"]))
        h_dls["BB"].append(_dev.to_host(binned_dls["BB"]))
        rec = SigmaRecorder(("EE", "BB"), self.n_iter, self.lmax) if self.keep_sigma else None
        for i in range(self.n_iter):
            if self.verbose and i % 100 == 0:
                print("Default Gibbs" if not self.ula else "ULA")
                print(i)
            start_time = time.perf_counter()  # time.clock was removed in Python 3.8
            if self.rj_step is False and self.gibbs_cr is False and self.ula is False:
                skymap, _ = self.constrained_sampler.sample(dict(dls_unbinned))
            else:
                skymap, accept = self.constrained_sampler.sample(dict(dls_unbinned), skymap)
                h_accept_cr.append(accept)
            torch.cuda.synchronize()
            h_duration_cr.append(time.perf_counter() - start_time)

            start_time = time.perf_counter()
            binned_dls = self.cls_sampler.sample(dict(skymap))
            if rec is not None:
                rec.record(i, self.cls_sampler.last_sigma)
            dls_unbinned = {"EE": self._unfold(binned_dls, "EE"), "BB": self._unfold(binned_dls, "BB")}
            torch.cuda.synchronize()
            h_duration_cls_sampling.append(time.perf_counter() - start_time)
            h_dls["EE"].append(_dev.to_host(binned_dls["EE"]))
            h_dls["BB"].append(_dev.to_host(binned_dls["BB"]))
        if self.verbose and (self.rj_step == True or self.ula == True):
            print("Acception rate constrained realization:", np.mean(h_accept_cr))
        if rec is not None:
            self.sigma_history = rec.result()
        h_dls["EE"] = np.array(h_dls["EE"])
        h_dls["BB"] = np.array(h_dls["BB"])
        return h_dls, np.array(h_accept_cr), np.array(h_duration_cr), np.array(h_duration_cls_sampling)

    def _tt_state(self, binned_dls):
        """binned D_l -> (C_l, expanded variances) as GibbsSampler.py:88-90."""
        dls = utils.unfold_bins(f64(binned_dls), self.bins)
        return dls * f64(self.dls_to_cls_array), utils.generate_var_cl(dls)

    def run_temperature(self, dls_init):
        """Mirror of GibbsSampler.run_temperature (GibbsSampler.py:76-116); same return tuple."""
        h_accept_cr, h_dls, h_time_seconds = [], [], []
        binned_dls = f64(dls_init)
        cls, var_cls_full = self._tt_state(binned_dls)
        skymap, accept = self.constrained_sampler.sample(cls, var_cls_full, None, metropolis_step=False)
        h_dls.append(_dev.to_host(binned_dls))
        rec = SigmaRecorder(("TT",), self.n_iter, self.lmax) if self.keep_sigma else None
        for i in range(self.n_iter):
            if self.verbose:
                print("Default Gibbs")
                print(i)
            start_time = time.perf_counter()
            skymap, accept = self.constrained_sampler.sample(cls, var_cls_full, skymap, metropolis_step=False, use_gibbs=False)
            binned_dls = self.cls_sampler.sample(skymap)
            if rec is not None:
                rec.record(i, self.cls_sampler.last_sigma)
            cls, var_cls_full = self._tt_state(binned_dls)
            torch.cuda.synchronize()
            h_accept_cr.append(accept)
            h_dls.append(_dev.to_host(binned_dls))
            h_time_seconds.append(time.perf_counter() - start_time)
        if rec is not None:
            self.sigma_history = rec.result()
        return np.array(h_dls), np.array(h_accept_cr), h_time_seconds

    def run(self, dls_init):
        if not self.polarization:
            return self.run_temperature(dls_init)
        return self.run_polarization(dls_init)
