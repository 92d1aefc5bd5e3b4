"""Base classes of the power-spectrum conditional samplers (mirror of ClsSampler.py:8-125)."""
import numpy as np
import torch

from . import _dev, _lib
from ._dev import f64, ptr, stream
from ._lib import check, GS_ALM_REAL
from .sht import Plan


class ClsSampler():
    def __init__(self, pix_map, lmax, nside, bins, bl_map, noise, mask_path=None, *, mask=None, rng="philox",
                 seed=None, plan=None):
        """Same arguments as ClsSampler.__init__ (ClsSampler.py:9); mask/rng as in ConstrainedRealization."""
        self.lmax = int(lmax)
        self.bins = bins
        self.nside = int(nside)
        self.pix_map = pix_map
        self.bl_map = bl_map
        self.noise = noise
        self.dev = _dev.device()
        self._mask_arr = _dev.load_mask(mask_path, self.nside, mask)
        self.mask_path = mask_path
        n = f64(noise)
        self.inv_noise = 1.0 / n
        if self._mask_arr is not None:
            self.inv_noise = self.inv_noise * f64(self._mask_arr)  # ClsSampler.py:28-33
        self.rng = rng if isinstance(rng, _dev.Rng) else _dev.Rng(rng, seed)
        self._call = 0
        self.plan = plan  # a ShardedPlan: alms are local m shards, alm2cl all-reduces (gs_shard_alm2cl)

    def sample(self, alm_map):
        return None

    # ---- shared device helpers -------------------------------------------------------------
    def _alm2cl_real(self, alms_real_d):
        if self.plan is not None:
            return self.plan.alm2cl(alms_real_d)
        cl = torch.empty(self.lmax + 1, dtype=torch.float64, device=self.dev)
        check(_lib.lib().gs_alm2cl(ptr(alms_real_d), GS_ALM_REAL, self.lmax, ptr(cl), stream()))
        return cl

    def _invgamma_draw(self, alms_real_d, bins):
        """One inverse-gamma draw of the binned D_l given real-layout alms (CenteredGibbs.py:54-79)."""
        edges = np.asarray(bins, dtype=np.int64)
        nb = len(edges) - 1
        cl = self._alm2cl_real(alms_real_d)
        self._last_cl = cl       # the empirical spectrum of this draw (GibbsSampler's keep_sigma records it)
        out = torch.empty(nb, dtype=torch.float64, device=self.dev)
        inject = None
        if self.rng.mode == "numpy":
            # the reference's own draw: invgamma.rvs(a=alphas) = 1 / standard_gamma(alphas) (CenteredGibbs.py:77)
            from scipy.stats import invgamma
            exponent = np.array([(2 * l + 1) / 2 for l in range(self.lmax + 1)])
            alphas = np.array([np.sum(exponent[edges[i]:edges[i + 1]]) - 1 for i in range(nb)])
            alphas[0] = 1
            inject = f64(1.0 / invgamma.rvs(a=alphas))
        # the call index comes from the SHARED generator's counter: samplers that share an Rng (EE / BB, several chains built with
        # one seed) never repeat a gamma stream, and the gamma domain (tag in the top byte, sampler.cu) is disjoint from the normals
        self.rng.counter += 1
        self._call = self.rng.counter
        check(_lib.lib().gs_cls_invgamma(ptr(cl), ptr(_dev.i32(edges)), nb, ptr(inject), self.rng.seed,
                                         self._call, ptr(out), None, None, stream()))
        return out


class MHClsSampler(ClsSampler):
    def __init__(self, pix_map, lmax, nside, bins, bl_map, noise, metropolis_blocks, proposal_variances, n_iter=1,
                 mask_path=None, polarization=False, *, mask=None, rng="philox", seed=None):
        """Mirror of MHClsSampler.__init__ (ClsSampler.py:46-73)."""
        super().__init__(pix_map, lmax, nside, bins, bl_map, noise, mask_path, mask=mask, rng=rng, seed=seed)
        if metropolis_blocks is None:
            self.metropolis_blocks = list(range(2, len(self.bins)))
        else:
            self.metropolis_blocks = metropolis_blocks
        self.n_iter = n_iter
        self.proposal_variances = proposal_variances
        self.polarization = polarization
        self.dls_to_cls_array = np.array([2 * np.pi / (l * (l + 1)) if l != 0 else 0 for l in range(lmax + 1)])

    def dls_to_cls(self, dls_):
        return dls_ * self.dls_to_cls_array

    # device versions of propose_dl / compute_log_proposal for one spectrum (ClsSampler.py:79-92)
    def _propose(self, dls_old_d, prop_var_d):
        nb = dls_old_d.numel()
        out = torch.empty_like(dls_old_d)
        if self.rng.mode == "numpy":
            from scipy.stats import truncnorm
            old = dls_old_d.cpu().numpy()
            sc = np.sqrt(prop_var_d.cpu().numpy())
            clip_low = -old[2:] / sc
            new = np.concatenate([np.zeros(2), truncnorm.rvs(a=clip_low, b=np.inf, loc=old[2:], scale=sc)])
            return f64(new)
        u = self.rng.uniform(nb - 2)
        check(_lib.lib().gs_truncnorm_propose(ptr(dls_old_d), ptr(prop_var_d), nb, ptr(u), ptr(out), stream()))
        return out

    def _log_proposal(self, x_d, from_d, prop_var_d):
        out = torch.empty_like(x_d)
        check(_lib.lib().gs_truncnorm_logpdf(ptr(x_d), ptr(from_d), ptr(prop_var_d), x_d.numel(), ptr(out), stream()))
        return out
