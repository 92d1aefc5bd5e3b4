"""Temperature-only (TT) samplers: mirrors of CenteredConstrainedRealization (CenteredGibbs.py:95-235),
NonCenteredConstrainedRealization (NonCenteredGibbs.py:17-101), NonCenteredClsSampler (NonCenteredGibbs.py:205-248)
and the recovered TT PNCP classes (SURVEY.md 2.3), on the spin-0 kernels of libgibbs_b200.so.

The TT code of the reference does not run at HEAD (it needs the removed config.mask_inversion / config.w /
config.bins and a forked qcinv; SURVEY.md 0), so behaviour follows the source text.  One inconsistency of that
text is resolved deliberately: CenteredConstrainedRealization.sample_mask returns the solver output as the map s
(CenteredGibbs.py:159-164) while NonCenteredConstrainedRealization.sample_mask treats the same output as C^-1 s
(NonCenteredGibbs.py:73-77).  Here the solver returns s (as the polarised twin does, CenteredGibbs.py:486-489), the
centred class returns it unchanged and the non-centred class returns C^-1/2 s.

Argument conventions are the reference's: `cls_` = C_l (L+1), `var_cls` = diagonal of C over the real alm layout
((L+1)^2, utils.generate_var_cl), `old_s` / returned maps = real-layout alms."""
import ctypes as C

import numpy as np
import torch

from . import _dev, _lib, utils
from ._dev import f64, ptr, stream
from ._lib import check, GS_ALM_REAL, GS_E_NOTCONVERGED
from .ClsSampler import MHClsSampler
from .ConstrainedRealization import ConstrainedRealization


class _TemperatureCR(ConstrainedRealization):
    """Shared setup of the TT constrained-realization classes."""

    def __init__(self, pix_map, noise, bl_map, fwhm_deg, lmax, Npix, mask_path=None, isotropic=True, *, mask=None,
                 rng="philox", seed=None, plan=None):
        super().__init__(pix_map, noise, bl_map, fwhm_deg, lmax, Npix, mask_path=mask_path, isotropic=isotropic, mask=mask,
                         rng=rng, seed=seed, plan=plan)
        self.d = self.plan.local_map(f64(pix_map))
        self.sqrt_inv_noise = torch.sqrt(self.inv_noise)
        self.ninv_sum_over_4pi = self.plan.allreduce_sum(_dev.dsum(self.inv_noise)) / (4 * np.pi)
        self.noise0 = float(f64(noise).reshape(-1)[0].item())
        self.inv_noise0 = 1.0 / self.noise0
        self.pcg_check_every = 8
        self.fluct_iter = 3   # utils.adjoint_synthesis_hp uses map2alm(iter=3) (utils.py:104)
        ell = torch.arange(self.lmax + 1, dtype=torch.float64, device=self.dev)
        self._c2d = torch.where(ell > 0, ell * (ell + 1) / (2 * np.pi), torch.ones_like(ell))
        # B A^T N^-1 d: what qcinv's chain.sample adds to the right-hand side (iter = 0 transpose)
        self.bdata = self.plan.map2alm(self.d, adjoint=True, pixw=self.inv_noise, fl=self.bl_gauss_d, real_layout=True)
        self._b_weiner = None

    # ---- helpers -------------------------------------------------------------------------------------
    def _dl(self, var_cls):
        """unbinned D_l (what the C ABI takes) from the expanded variances: entries 0..L are C_l (m = 0 block)."""
        v = f64(var_cls)
        assert v.numel() == (self.lmax + 1) ** 2, "var_cls must be the (L+1)^2 expansion of utils.generate_var_cl"
        return (v[: self.lmax + 1] * self._c2d).contiguous()

    def _draws(self, xi):
        """(xi_alm, xi_pix) in the reference's order: the alm draw is evaluated first (CenteredGibbs.py:145-147)."""
        if xi is not None:
            return self.plan.local_alm(f64(xi[0])), self.plan.local_map(f64(xi[1]))
        return self.rng.normal(self.dimension_alm), self.rng.normal(self.npix_local)

    def _rhs(self, dl, bdata, xi):
        xa, xp = self._draws(xi)
        rhs = torch.empty(self.dimension_alm, dtype=torch.float64, device=self.dev)
        check(_lib.lib().gs_cr_rhs_tt(self.plan._h, ptr(dl), ptr(self.bl_gauss_d), ptr(self.inv_noise), ptr(self.sqrt_inv_noise),
                                      ptr(bdata), None, ptr(xa), ptr(xp), self.fluct_iter, ptr(rhs), stream()))
        return rhs

    def _solve(self, dl, rhs, x0=None):
        x = torch.empty(self.dimension_alm, dtype=torch.float64, device=self.dev) if x0 is None else f64(x0).clone()
        nit, res = C.c_int(0), C.c_double(0.0)
        rc = _lib.lib().gs_cr_pcg_tt(self.plan._h, ptr(dl), ptr(self.bl_gauss_d), ptr(self.inv_noise), self.ninv_sum_over_4pi,
                                     ptr(rhs), ptr(x), 0 if x0 is None else 1, self.pcg_accuracy, self.pcg_itermax,
                                     self.pcg_check_every, C.byref(nit), C.byref(res), stream())
        self.last_pcg_iterations, self.last_pcg_residual = nit.value, res.value
        if rc not in (0, GS_E_NOTCONVERGED):
            check(rc)
        return x

    def apply_Q(self, dl, x):
        y = torch.empty_like(x)
        check(_lib.lib().gs_cr_apply_q_tt(self.plan._h, ptr(dl), ptr(self.bl_gauss_d), ptr(self.inv_noise), ptr(x), ptr(y), stream()))
        return y

    def _ret(self, t, like):
        return t if isinstance(like, torch.Tensor) else t.cpu().numpy()

    def _direct(self, dl, xi, l_cut, zero_low):
        """Diagonal draw for full sky + isotropic noise (gs_cr_direct_pix): l < l_cut centred, l >= l_cut non-centred."""
        resc = self.Npix / (4 * np.pi)
        if self._b_weiner is None:  # bl * adjoint_synthesis_hp(inv_noise * d), iter = 3 (CenteredGibbs.py:112)
            self._b_weiner = self.plan.map2alm(self.d, iter=3, pixw=self.inv_noise, fl=self.bl_gauss_d, real_layout=True) * resc
        xa, xp = self._draws(xi)
        bsum = self.plan.map2alm(xp, iter=3, pixw=self.sqrt_inv_noise, fl=self.bl_gauss_d, real_layout=True)
        bsum = torch.add(self._b_weiner, bsum, alpha=resc)
        out = torch.empty(self.dimension_alm, dtype=torch.float64, device=self.dev)
        check(_lib.lib().gs_cr_direct_pix(ptr(dl), ptr(self.bl_gauss_d), ptr(bsum), ptr(xa), self.inv_noise0 * resc, self.lmax,
                                          int(l_cut), int(zero_low), ptr(out), stream()))
        return out

    def _masked_solve(self, var_cls, s_old, metropolis_step, xi, u):
        """PCG draw (RJPO when metropolis_step): CenteredGibbs.py:130-189 / NonCenteredGibbs.py:43-92.  -> (s, accept, dl)."""
        dl = self._dl(var_cls)
        rhs = self._rhs(dl, self.bdata, xi)
        self.last_rhs = rhs
        if not metropolis_step:
            return self._solve(dl, rhs), 1, dl
        so = f64(s_old)
        x = self._solve(dl, rhs, x0=-so)
        r = rhs - self.apply_Q(dl, x)
        log_proba = min(0.0, -float(torch.dot(r, so - x).item()))
        if u is None:
            u = float(self.rng.uniform(2)[0].item()) if self.rng.mode == "philox" else np.random.uniform()
        if np.log(u) < log_proba:
            return x, 1, dl
        return so, 0, dl


class CenteredConstrainedRealization(_TemperatureCR):
    """TT constrained realization, centred parametrisation (CenteredGibbs.py:95-235)."""

    def sample_no_mask(self, var_cls, xi=None):
        """Full sky, isotropic noise: diagonal solve (CenteredGibbs.py:100-127)."""
        return self._ret(self._direct(self._dl(var_cls), xi, self.lmax + 1, 0), var_cls), 1

    def sample_mask(self, cls_, var_cls, s_old, metropolis_step=False, xi=None, u=None):
        x, acc, _ = self._masked_solve(var_cls, s_old, metropolis_step, xi, u)
        return self._ret(x, var_cls), acc

    def sample_gibbs_change_variable(self, var_cls, old_s, xi=None):
        """Auxiliary-variable step (CenteredGibbs.py:191-212): v | s in pixel space, then s | v diagonal in harmonic space."""
        L = _lib.lib()
        dl = self._dl(var_cls)
        s = f64(old_s).clone()
        m = self.plan.alm2map(s, fl=self.bl_gauss_d)
        xv = f64(xi[0]) if xi is not None else self.rng.normal(self.npix_local)
        v = torch.zeros(self.npix_local, dtype=torch.float64, device=self.dev)
        out = torch.empty_like(m)
        check(L.gs_aux_v_update(ptr(m), ptr(self.inv_noise), ptr(self.d), ptr(xv), self.mu, 0.0, ptr(v), ptr(out), self.npix_local, stream()))
        badj = self.plan.map2alm(out, adjoint=True, fl=self.bl_gauss_d, real_layout=True)
        xs = f64(xi[1]) if xi is not None else self.rng.normal(self.dimension_alm)
        w = 4 * np.pi / self.Npix
        check(L.gs_aux_s_update(ptr(badj), ptr(dl), ptr(self.bl_gauss_d), ptr(xs), self.mu / w, 0.0, self.lmax, ptr(s), stream()))
        return self._ret(s, var_cls), 1

    def sample(self, cls_, var_cls, old_s, metropolis_step=False, use_gibbs=False):
        """Dispatcher of the reference (CenteredGibbs.py:215-233)."""
        if use_gibbs:
            return self.sample_gibbs_change_variable(var_cls, old_s)
        if self.masked or self.mask_path is not None:
            return self.sample_mask(cls_, var_cls, old_s, metropolis_step)
        return self.sample_no_mask(var_cls)


class NonCenteredConstrainedRealization(_TemperatureCR):
    """TT constrained realization of the non-centred variable s_nc = C^-1/2 s (NonCenteredGibbs.py:17-101)."""

    def sample_no_mask(self, cls_, var_cls, xi=None):
        """NonCenteredGibbs.py:22-41: Sigma = 1/(1 + C w b^2), s_nc = Sigma (sqrt(C) b A^T N^-1 d + xi + sqrt(C) b A^T N^-1/2 xi')."""
        return self._ret(self._direct(self._dl(var_cls), xi, 0, 0), var_cls), 1

    def sample_mask(self, cls_, var_cls, s_old, metropolis_step=False, xi=None, u=None):
        x, acc, dl = self._masked_solve(var_cls, None if s_old is None else f64(s_old), metropolis_step, xi, u)
        if acc == 0:
            return self._ret(x, var_cls), 0
        s_nc = x * self.plan.expand_per_l(dl, 4)                 # C^-1/2 s; monopole and dipole are zeroed with it
        return self._ret(s_nc, var_cls), 1

    def sample(self, cls_, var_cls, old_s, metropolis_step=False):
        if self.masked or self.mask_path is not None:
            return self.sample_mask(cls_, var_cls, old_s, metropolis_step)
        return self.sample_no_mask(cls_, var_cls)


class NonCenteredClsSampler(MHClsSampler):
    """Blocked Metropolis-within-Gibbs on the binned D_l given the non-centred map, TT (NonCenteredGibbs.py:205-248;
    likelihood ClsSampler.py:94-108).  The sweep runs on the device; accept flags are read back at the end."""

    def __init__(self, pix_map, lmax, nside, bins, bl_map, noise, metropolis_blocks, proposal_variances, n_iter=1,
                 mask_path=None, polarization=False, *, mask=None, rng="philox", seed=None):
        super().__init__(pix_map, lmax, nside, bins, bl_map, noise, metropolis_blocks, proposal_variances, n_iter=n_iter,
                         mask_path=mask_path, polarization=polarization, mask=mask, rng=rng, seed=seed)
        from .sht import Plan
        self.plan = Plan.get(self.nside, self.lmax)
        self.Npix = 12 * self.nside ** 2
        inv = self.inv_noise
        if inv.numel() == 1:
            inv = inv.expand(self.Npix)
        self.inv_noise_d = inv.contiguous()
        self.d = f64(pix_map)
        self.bl_gauss_d = f64(bl_map)[: self.lmax + 1].contiguous()
        self.bins_d = _dev.i32(np.asarray(self.bins))
        self.nb = len(self.bins) - 1
        self.pv_d = f64(self.proposal_variances)
        self._m = torch.empty(self.Npix, dtype=torch.float64, device=self.dev)
        self._fl = torch.empty(self.lmax + 1, dtype=torch.float64, device=self.dev)
        self._fl2 = torch.empty_like(self._fl)
        self._scratch = torch.empty(592, dtype=torch.float64, device=self.dev)
        self._ones = torch.ones(self.nb, dtype=torch.float64, device=self.dev)

    def compute_log_proposal(self, dl_old, dl_new):
        """log q(dl_new | dl_old) per bin (NonCenteredGibbs.py:206-210)."""
        return self._log_proposal(f64(dl_new), f64(dl_old), self.pv_d)

    def _loglik_device(self, cur, prop, b0, b1, s_nc, out):
        L = _lib.lib()
        # per-l filter b_l sqrt(C_l) of (cur with bins [b0, b1) replaced by prop); the B spectrum slot is a dummy
        check(L.gs_mwg_filters(ptr(cur), ptr(self._ones), ptr(prop), ptr(prop), ptr(self.bins_d), self.nb, ptr(self.bins_d), self.nb,
                               0 if prop is not None else -1, b0, b1, ptr(self.bl_gauss_d), self.lmax, 0, ptr(self._fl), ptr(self._fl2),
                               stream()))
        check(L.gs_alm2map_spin0(self.plan._h, ptr(s_nc), GS_ALM_REAL, ptr(self._fl), ptr(self._m), stream()))
        check(L.gs_loglik_pix(ptr(self.d), None, ptr(self._m), None, ptr(self.inv_noise_d), self.Npix, ptr(self._scratch), ptr(out),
                              stream()))

    def compute_log_likelihood(self, var_cls, s_nonCentered):
        """ClsSampler.py:94-108 -> python float; var_cls = expanded variances."""
        v = f64(var_cls)
        fl = (self.bl_gauss_d * torch.sqrt(v[: self.lmax + 1])).contiguous()
        out = torch.empty(1, dtype=torch.float64, device=self.dev)
        s = f64(s_nonCentered)
        L = _lib.lib()
        check(L.gs_alm2map_spin0(self.plan._h, ptr(s), GS_ALM_REAL, ptr(fl), ptr(self._m), stream()))
        check(L.gs_loglik_pix(ptr(self.d), None, ptr(self._m), None, ptr(self.inv_noise_d), self.Npix, ptr(self._scratch), ptr(out),
                              stream()))
        return float(out.item())

    def sample(self, s_nonCentered, binned_dls_old, var_cls_old=None):
        """-> (binned_dls, var_cls, accept) as NonCenteredGibbs.py:212-248."""
        host = not isinstance(binned_dls_old, torch.Tensor)
        L = _lib.lib()
        s = f64(s_nonCentered)
        cur = f64(binned_dls_old).clone()
        prop = self._propose(cur, self.pv_d)
        logr = (self._log_proposal(prop, cur, self.pv_d) - self._log_proposal(cur, prop, self.pv_d)).contiguous()
        old_lik = torch.empty(1, dtype=torch.float64, device=self.dev)
        new_lik = torch.empty(1, dtype=torch.float64, device=self.dev)
        self._loglik_device(cur, None, 0, 0, s, old_lik)
        blocks = [int(b) for b in self.metropolis_blocks]
        ntot = (len(blocks) - 1) * self.n_iter
        if self.rng.mode == "numpy":
            u = f64(np.array([np.random.uniform() for _ in range(ntot)]))
        else:
            u = self.rng.uniform(max(ntot, 2))
        acc = torch.zeros(max(ntot, 1), dtype=torch.int32, device=self.dev)
        k = 0
        for i in range(len(blocks) - 1):
            for _ in range(self.n_iter):
                self._loglik_device(cur, prop, blocks[i], blocks[i + 1], s, new_lik)
                check(L.gs_mwg_accept(ptr(cur), ptr(prop), ptr(logr), blocks[i], blocks[i + 1], ptr(new_lik), ptr(old_lik),
                                      ptr(u[k:]), ptr(acc[k:]), stream()))
                k += 1
        accept = [int(x) for x in acc.cpu().numpy()[:ntot]]
        var_cls = utils.generate_var_cl(utils.unfold_bins(cur, self.bins))
        if host:
            return cur.cpu().numpy(), var_cls.cpu().numpy(), accept
        return cur, var_cls, accept


# ---------------------------------------------------------------------------- TT PNCP (recovered from PNCP.cpython-38.pyc)
class PNCPConstrainedRealizationTT(_TemperatureCR):
    """PNCPConstrainedRealization of the reference bytecode (SURVEY.md 2.3): full sky, isotropic noise, TT.
    Multipoles below l_cut are drawn centred, l >= l_cut non-centred; monopole / dipole entries are zeroed."""

    def __init__(self, *args, l_cut=5, **kw):
        super().__init__(*args, **kw)
        self.l_cut = int(l_cut)

    def sample(self, var_cls, xi=None):
        """-> (map, time, 0) as the recovered PNCPConstrainedRealization.sample(var_cls)."""
        import time
        t0 = time.perf_counter()
        out = self._direct(self._dl(var_cls), xi, self.l_cut, 1)
        return self._ret(out, var_cls), time.perf_counter() - t0, 0


class PNCPClsSamplerTT(NonCenteredClsSampler):
    """Recovered PNCPClsSampler: sample_low_l = inverse-gamma with alpha = (2l-1)/2, beta = (2l+1) l (l+1) Chat_l / 4pi for
    l < l_cut; sample_high_l = blocked MwG on the bins >= l_cut with the synthesised field b_l (s_l | sqrt(C_l) s_nc,l)."""

    def __init__(self, pix_map, lmax, nside, bins, bl_map, noise, metropolis_blocks, proposal_variances, l_cut, n_iter=1,
                 mask_path=None, *, mask=None, rng="philox", seed=None):
        if int(np.asarray(bins)[int(metropolis_blocks[0])]) < l_cut:
            raise ValueError("metropolis_blocks starts below l_cut")
        super().__init__(pix_map, lmax, nside, bins, bl_map, noise, metropolis_blocks, proposal_variances, n_iter=n_iter,
                         mask_path=mask_path, mask=mask, rng=rng, seed=seed)
        self.l_cut = int(l_cut)
        self.low_bins = int(np.searchsorted(np.asarray(bins), l_cut, side="left"))

    def _loglik_device(self, cur, prop, b0, b1, s_nc, out):
        L = _lib.lib()
        check(L.gs_mwg_filters(ptr(cur), ptr(self._ones), ptr(prop), ptr(prop), ptr(self.bins_d), self.nb, ptr(self.bins_d), self.nb,
                               0 if prop is not None else -1, b0, b1, ptr(self.bl_gauss_d), self.lmax, self.l_cut, ptr(self._fl),
                               ptr(self._fl2), stream()))
        check(L.gs_alm2map_spin0(self.plan._h, ptr(s_nc), GS_ALM_REAL, ptr(self._fl), ptr(self._m), stream()))
        check(L.gs_loglik_pix(ptr(self.d), None, ptr(self._m), None, ptr(self.inv_noise_d), self.Npix, ptr(self._scratch), ptr(out),
                              stream()))

    def sample_low_l(self, mixed, binned_dls):
        """Centred inverse-gamma draw of the bins below l_cut (their alms are the centred ones in the mixed map)."""
        draw = self._invgamma_draw(f64(mixed), self.bins)
        o = f64(binned_dls).clone()
        o[: self.low_bins] = draw[: self.low_bins]
        return o

    def sample_high_l(self, mixed, binned_dls):
        cur, _, acc = self.sample(mixed, binned_dls)
        return cur, acc
