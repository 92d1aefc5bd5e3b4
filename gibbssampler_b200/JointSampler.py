"""Joint TT/TE/EE/BB Gibbs sampling with per-multipole 3x3 covariances (SURVEY.md 8a row A9, 8f row 4).

The reference never finished this path: the per-l 3x3 helpers survive only as bytecode / object files
(utils.compute_inverse_and_cholesky, utils.matrix_product, linear_algebra.pyx) and a buggy Cython expansion
(variance_expension.pyx:36-61); the intended C_l conditional is the inverse-Wishart of
.ipynb_checkpoints/main-checkpoint.py:39-44,333-346.  Built here for the case those helpers were written for
-- full sky, isotropic noise, data in harmonic space -- where the constrained realization is a per-coefficient
3x3 solve:
    Sigma_l = (C_l^-1 + diag(b_l^2 w_X))^-1,  s = Sigma_l (b_l w_X d_X)_X + chol(Sigma_l) xi,  w_X = Npix / (4 pi sigma^2_X)
and  (C^TT, C^TE, C^EE)_l | s ~ IW(2l - 2, (2l+1) Chat_l),  C^BB_l | s ~ inverse-gamma as in CenteredGibbs.py:54-79.
With bins (D constant on each bin, as the reference bins EE/BB) the TT/TE/EE block of bin b is
    D_b | s ~ IW(nu_b, Psi_b),  nu_b = sum_{l in b} (2l+1) - 3,  Psi_b = sum_{l in b} (2l+1) l(l+1)/(2 pi) Chat_l
and BB takes the reference's binned inverse-gamma.
Every step is a batched one-thread-per-l (or per-coefficient) kernel of libgibbs_b200.so.

On a cut sky (pixel data, one mask for T and another for P, per-pixel noise) the constrained realization is the joint T/E/B
system Q x = b of qcinv's joint T+P filter, solved by the TE-coupled PCG of gs_cr_pcg_teb (include/gibbs_b200.h)."""
import ctypes as C
import math

import numpy as np
import torch

from . import _dev, _lib
from ._dev import f64, ptr, stream
from ._lib import check, GS_ALM_REAL


class JointConstrainedRealization():
    def __init__(self, pix_map, noise_temp, noise_pol, bl_gauss, lmax, Npix, *, mask=None, mask_pol=None, rng="philox", seed=None,
                 plan=None):
        """pix_map: either {"TT","EE","BB"} data alms in the real layout (full sky, isotropic noise: closed-form draw; noise_*
        are scalar per-pixel variances), or {"I","Q","U"} RING maps (masked sky: PCG on the joint T/E/B system).  With maps,
        noise_* are scalars or per-pixel variance maps, `mask` (RING array) multiplies N_T^-1 and `mask_pol` (default: `mask`)
        multiplies N_P^-1: N_T^-1 = mask / noise_temp, N_P^-1 = mask_pol / noise_pol.  `plan`: a single-GPU sht.Plan (default:
        the cached plan of (nside, lmax)); the joint solve does not run on m-sharded plans."""
        self.lmax, self.Npix = int(lmax), int(Npix)
        self.dev = _dev.device()
        self.n = (self.lmax + 1) ** 2
        self.bl = f64(bl_gauss)
        self.rng = rng if isinstance(rng, _dev.Rng) else _dev.Rng(rng, seed)
        self.pixel = "I" in pix_map
        if self.pixel:
            self._init_masked(pix_map, noise_temp, noise_pol, mask, mask_pol, plan)
            return
        self.w = torch.tensor([self.Npix / (4 * np.pi * float(noise_temp)), self.Npix / (4 * np.pi * float(noise_pol)),
                               self.Npix / (4 * np.pi * float(noise_pol))], dtype=torch.float64, device=self.dev)
        d = torch.stack([f64(pix_map["TT"]), f64(pix_map["EE"]), f64(pix_map["BB"])], dim=1).contiguous()   # (n, 3)
        from . import utils
        blx = utils.expand_per_l(self.bl, 0)
        self.b_w_d = (d * blx[:, None] * self.w[None, :]).contiguous()               # B N^-1 d per coefficient
        self.pix_part = (self.bl[:, None] ** 2 * self.w[None, :]).contiguous()      # (L+1, 3): b_l^2 w_X

    def covariances(self, all_dls):
        """D_l dict {"TT","EE","BB","TE"} (unbinned, L+1) -> per-l C_l matrices (L+1,3,3)."""
        ell = torch.arange(self.lmax + 1, dtype=torch.float64, device=self.dev)
        f = torch.where(ell > 0, 2 * np.pi / (ell * (ell + 1)).clamp(min=1), torch.ones_like(ell))
        c = torch.zeros(self.lmax + 1, 3, 3, dtype=torch.float64, device=self.dev)
        c[:, 0, 0] = f64(all_dls["TT"]) * f
        c[:, 1, 1] = f64(all_dls["EE"]) * f
        c[:, 2, 2] = f64(all_dls["BB"]) * f
        c[:, 0, 1] = c[:, 1, 0] = f64(all_dls["TE"]) * f
        return c.contiguous()

    # ------------------------------------------------------------------ masked sky: joint PCG
    def _init_masked(self, pix_map, noise_temp, noise_pol, mask, mask_pol, plan):
        from .sht import Plan
        self.nside = int(round(math.sqrt(self.Npix / 12)))
        if 12 * self.nside ** 2 != self.Npix:
            raise ValueError("Npix = %d is not 12 nside^2" % self.Npix)
        self.plan = plan if plan is not None else Plan.get(self.nside, self.lmax)
        if self.plan.world > 1:
            raise _lib.GibbsB200Error("the joint T/E/B constrained realization needs a single-GPU plan (this one is m-sharded over "
                                      "%d ranks)" % self.plan.world)
        mT = _dev.load_mask(None, self.nside, mask)
        mP = _dev.load_mask(None, self.nside, mask_pol) if mask_pol is not None else mT
        self.inv_noise_T = self._inv_noise(noise_temp, mT)
        same = mask_pol is None and np.array_equal(np.asarray(_dev.to_host(noise_pol)), np.asarray(_dev.to_host(noise_temp)))
        # one array for both when they are equal: the library then builds its ring flags once per call
        self.inv_noise_P = self.inv_noise_T if same else self._inv_noise(noise_pol, mP)
        self.sqrt_inv_noise_T = torch.sqrt(self.inv_noise_T)
        self.sqrt_inv_noise_P = self.sqrt_inv_noise_T if same else torch.sqrt(self.inv_noise_P)
        self.ninvT_sum_over_4pi = _dev.dsum(self.inv_noise_T) / (4 * np.pi)
        self.ninvP_sum_over_4pi = _dev.dsum(self.inv_noise_P) / (4 * np.pi)
        d_I, d_Q, d_U = f64(pix_map["I"]), f64(pix_map["Q"]), f64(pix_map["U"])
        # constant data terms B A^T N^-1 d of every right-hand side
        self.bdata_T = self.plan.map2alm(d_I, adjoint=True, pixw=self.inv_noise_T, fl=self.bl, real_layout=True)
        self.bdata_E, self.bdata_B = self.plan.map2alm_spin2(d_Q, d_U, adjoint=True, pixw=self.inv_noise_P, fl=self.bl,
                                                             real_layout=True)
        self.pcg_accuracy = 1.0e-6      # qcinv chain settings of the TT sampler (ConstrainedRealization.py:41)
        self.pcg_itermax = 4000
        self.pcg_check_every = 8
        self.fluct_iter = 3             # utils.adjoint_synthesis_hp uses iter=3 (utils.py:89)
        self.last_pcg_iterations, self.last_pcg_residual = 0, 0.0
        self.last_rhs = None

    def _inv_noise(self, noise, mask):
        n = f64(noise).reshape(-1)
        if n.numel() == 1:
            n = n.expand(self.Npix)
        if n.numel() != self.Npix:
            raise ValueError("noise must be a scalar or a map of %d pixels" % self.Npix)
        inv = (1.0 / n).contiguous()
        if mask is not None:
            inv.mul_(f64(mask))
        return inv

    def _dls(self, all_dls):
        out = tuple(f64(all_dls[k]).reshape(-1) for k in ("TT", "TE", "EE", "BB"))
        assert all(x.numel() == self.lmax + 1 for x in out), "need unbinned D_l of length lmax+1"
        return out

    def _masked_only(self, what):
        if not self.pixel:
            raise _lib.GibbsB200Error("%s needs pixel data (pix_map with 'I', 'Q', 'U')" % what)

    def build_rhs(self, all_dls, xi=None):
        """b of Q x = b.  xi = (xi_I, xi_Q, xi_U, xi_T, xi_E, xi_B) may be injected; drawn in that order otherwise."""
        self._masked_only("build_rhs")
        tt, te, ee, bb = self._dls(all_dls)
        if xi is None:
            xi = tuple(self.rng.normal(self.Npix) for _ in range(3)) + tuple(self.rng.normal(self.n) for _ in range(3))
        xi = [f64(x).reshape(-1) for x in xi]
        rhs = tuple(torch.empty(self.n, dtype=torch.float64, device=self.dev) for _ in range(3))
        check(_lib.lib().gs_cr_rhs_teb(self.plan._h, ptr(tt), ptr(te), ptr(ee), ptr(bb), ptr(self.bl), ptr(self.inv_noise_T),
                                       ptr(self.sqrt_inv_noise_T), ptr(self.inv_noise_P), ptr(self.sqrt_inv_noise_P),
                                       ptr(self.bdata_T), ptr(self.bdata_E), ptr(self.bdata_B), None, None, None,
                                       *[ptr(x) for x in xi], self.fluct_iter, *[ptr(r) for r in rhs], stream()))
        return rhs

    def solve(self, all_dls, rhs_t, rhs_e, rhs_b, x0=None):
        """PCG solve of the joint system; x0 = {"TT","EE","BB"} warm start.  -> (x_T, x_E, x_B)"""
        self._masked_only("solve")
        tt, te, ee, bb = self._dls(all_dls)
        if x0 is None:
            x = tuple(torch.empty(self.n, dtype=torch.float64, device=self.dev) for _ in range(3))
        else:
            x = tuple(f64(x0[k]).clone() for k in ("TT", "EE", "BB"))
        rhs = tuple(f64(r) for r in (rhs_t, rhs_e, rhs_b))
        nit, res = C.c_int(0), C.c_double(0.0)
        rc = _lib.lib().gs_cr_pcg_teb(self.plan._h, ptr(tt), ptr(te), ptr(ee), ptr(bb), ptr(self.bl), ptr(self.inv_noise_T),
                                      ptr(self.inv_noise_P), self.ninvT_sum_over_4pi, self.ninvP_sum_over_4pi,
                                      *[ptr(r) for r in rhs], *[ptr(v) for v in x], 0 if x0 is None else 1, self.pcg_accuracy,
                                      self.pcg_itermax, self.pcg_check_every, C.byref(nit), C.byref(res), stream())
        self.last_pcg_iterations, self.last_pcg_residual = nit.value, res.value
        if rc not in (0, -3):  # GS_E_NOTCONVERGED (-3) is reported through last_pcg_residual, as in the E/B sampler
            check(rc)
        return x

    def apply_Q(self, all_dls, x):
        """y = Q x for x = {"TT","EE","BB"} (real layout)."""
        self._masked_only("apply_Q")
        tt, te, ee, bb = self._dls(all_dls)
        xs = [f64(x[k]) for k in ("TT", "EE", "BB")]
        ys = [torch.empty_like(v) for v in xs]
        check(_lib.lib().gs_cr_apply_q_teb(self.plan._h, ptr(tt), ptr(te), ptr(ee), ptr(bb), ptr(self.bl), ptr(self.inv_noise_T),
                                           ptr(self.inv_noise_P), *[ptr(v) for v in xs], *[ptr(v) for v in ys], stream()))
        return {"TT": ys[0], "EE": ys[1], "BB": ys[2]}

    def sample(self, all_dls, xi=None):
        """-> ({"TT","EE","BB"} real-layout alms, 1).  Pixel data: RHS + joint PCG (xi: the six arrays of build_rhs);
        harmonic data: the closed-form per-coefficient draw (xi: (n, 3) normals)."""
        if self.pixel:
            rhs = self.build_rhs(all_dls, xi)
            self.last_rhs = rhs
            x = self.solve(all_dls, *rhs)
            return {"TT": x[0], "EE": x[1], "BB": x[2]}, 1
        L = _lib.lib()
        cl = self.covariances(all_dls)
        sig = torch.empty_like(cl)
        cho = torch.empty_like(cl)
        check(L.gs_inv_chol_3x3(ptr(cl), ptr(self.pix_part), self.lmax, ptr(sig), ptr(cho), stream()))
        if xi is None:
            xi = self.rng.normal(3 * self.n)
        xi = f64(xi).reshape(self.n, 3).contiguous()
        out = torch.empty(self.n, 3, dtype=torch.float64, device=self.dev)
        check(L.gs_matvec_3x3(ptr(sig), ptr(self.b_w_d), None, self.lmax, ptr(out), stream()))     # mean
        check(L.gs_matvec_3x3(ptr(cho), ptr(xi), ptr(out), self.lmax, ptr(out), stream()))          # + fluctuation
        return {"TT": out[:, 0].contiguous(), "EE": out[:, 1].contiguous(), "BB": out[:, 2].contiguous()}, 1


def _joint_bins(bins, lmax):
    """Validated bin edges {"TT": edges, "BB": edges} of the joint C_l step (int64 numpy arrays, host)."""
    if "TT" not in bins or "BB" not in bins:
        raise ValueError("bins needs 'TT' (shared by TE and EE) and 'BB' edges")
    out = {}
    for key in ("TT", "BB"):
        e = np.asarray(bins[key])
        if e.ndim != 1 or e.size < 3 or not np.issubdtype(e.dtype, np.integer):
            raise ValueError("bins[%r] must be a 1-d integer array of at least 3 edges" % key)
        e = e.astype(np.int64)
        if list(e[:3]) != [0, 1, 2]:
            raise ValueError("bins[%r] must start with the edges 0, 1, 2 (l = 0 and l = 1 are bins of their own)" % key)
        if e[-1] != lmax + 1:
            raise ValueError("bins[%r] must end at lmax + 1 = %d, not %d" % (key, lmax + 1, e[-1]))
        if np.any(np.diff(e) <= 0):
            raise ValueError("bins[%r] must be strictly ascending" % key)
        out[key] = e
    for key in ("TE", "EE"):   # one 2x2 matrix per bin: TT, TE and EE share the binning
        if key in bins and not np.array_equal(np.asarray(bins[key]), out["TT"]):
            raise ValueError("bins[%r] must equal bins['TT']" % key)
    return out


class JointClsSampler():
    def __init__(self, lmax, *, bins=None, rng="philox", seed=None):
        """bins: None (one draw per multipole) or {"TT": edges, "BB": edges} with int edges that start 0, 1, 2 and end at
        lmax + 1 ("TE" / "EE" may be given and must equal "TT"): then sample() draws D constant on each bin, TT/TE/EE by the
        binned inverse-Wishart of gs_cls_invwishart_binned and BB by the binned inverse-gamma of CenteredGibbs.py:54-79."""
        self.lmax = int(lmax)
        self.bins = None if bins is None else _joint_bins(bins, self.lmax)
        self.dev = _dev.device()
        self.rng = rng if isinstance(rng, _dev.Rng) else _dev.Rng(rng, seed)
        self._call = 0
        self.bins1 = _dev.i32(np.arange(self.lmax + 2))
        if self.bins is not None:
            self._bins_dev = {k: _dev.i32(v) for k, v in self.bins.items()}

    def empirical(self, alms):
        L = _lib.lib()
        out = {}
        dev_alms = {k: f64(alms[k]) for k in ("TT", "EE", "BB")}   # held until the launches below are queued
        for key, (a, b) in {"TT": ("TT", "TT"), "EE": ("EE", "EE"), "BB": ("BB", "BB"), "TE": ("TT", "EE")}.items():
            cl = torch.empty(self.lmax + 1, dtype=torch.float64, device=self.dev)
            check(L.gs_alm2cl_cross(ptr(dev_alms[a]), ptr(dev_alms[b]), self.lmax, ptr(cl), stream()))
            out[key] = cl
        return out

    def sample(self, alms, inject=None, gamma_inject=None):
        """-> D dict {"TT","EE","BB","TE"}: unbinned D_l (L+1) without bins, binned D (nbins_TT for TT/TE/EE, nbins_BB for BB)
        with bins.  inject: (L+1,3) or (nbins_TT,3) (chi2_df, chi2_{df-1}, normal) and gamma_inject (L+1) or (nbins_BB) Gamma
        variates for parity runs; default Philox."""
        if self.bins is not None:
            return self._sample_binned(alms, inject, gamma_inject)
        L = _lib.lib()
        ch = self.empirical(alms)
        self.rng.counter += 2          # shared generator counter (see ClsSampler._invgamma_draw): one index per draw kernel
        self._call = self.rng.counter - 1
        tt, te, ee = (torch.empty(self.lmax + 1, dtype=torch.float64, device=self.dev) for _ in range(3))
        inj = f64(inject).contiguous() if inject is not None else None
        check(L.gs_cls_invwishart(ptr(ch["TT"]), ptr(ch["TE"]), ptr(ch["EE"]), self.lmax, ptr(inj), self.rng.seed, self._call,
                                  ptr(tt), ptr(te), ptr(ee), stream()))
        ell = torch.arange(self.lmax + 1, dtype=torch.float64, device=self.dev)
        c2d = ell * (ell + 1) / (2 * np.pi)
        bb = torch.empty(self.lmax + 1, dtype=torch.float64, device=self.dev)
        gi = f64(gamma_inject).contiguous() if gamma_inject is not None else None
        check(L.gs_cls_invgamma(ptr(ch["BB"]), ptr(self.bins1), self.lmax + 1, ptr(gi), self.rng.seed, self._call + 1,
                                ptr(bb), None, None, stream()))
        return {"TT": tt * c2d, "TE": te * c2d, "EE": ee * c2d, "BB": bb}

    def _sample_binned(self, alms, inject, gamma_inject):
        L = _lib.lib()
        nt, nb = len(self.bins["TT"]) - 1, len(self.bins["BB"]) - 1
        inj = f64(inject).contiguous() if inject is not None else None
        gi = f64(gamma_inject).contiguous() if gamma_inject is not None else None
        if inj is not None and tuple(inj.shape) != (nt, 3):
            raise ValueError("inject must have shape (%d, 3), got %s" % (nt, tuple(inj.shape)))
        if gi is not None and gi.numel() != nb:
            raise ValueError("gamma_inject must have %d entries, got %d" % (nb, gi.numel()))
        ch = self.empirical(alms)
        self.rng.counter += 2          # the same two call indices as the per-l draw
        self._call = self.rng.counter - 1
        tt, te, ee = (torch.empty(nt, dtype=torch.float64, device=self.dev) for _ in range(3))
        check(L.gs_cls_invwishart_binned(ptr(ch["TT"]), ptr(ch["TE"]), ptr(ch["EE"]), self.lmax, ptr(self._bins_dev["TT"]), nt,
                                         ptr(inj), self.rng.seed, self._call, ptr(tt), ptr(te), ptr(ee), stream()))
        bb = torch.empty(nb, dtype=torch.float64, device=self.dev)
        check(L.gs_cls_invgamma(ptr(ch["BB"]), ptr(self._bins_dev["BB"]), nb, ptr(gi), self.rng.seed, self._call + 1, ptr(bb), None,
                                None, stream()))
        return {"TT": tt, "TE": te, "EE": ee, "BB": bb}


class JointGibbs():
    """CR <-> C_l Gibbs loop for (T, E, B) with TE correlation: full sky with isotropic noise and harmonic data
    ({"TT","EE","BB"}), or a cut sky with pixel data ({"I","Q","U"}, masks `mask` for T and `mask_pol` for P).
    bins (see JointClsSampler): D is sampled per bin; run() then takes binned initial D and returns binned histories, and each
    constrained realization sees D unfolded to L+1 multipoles (utils.unfold_bins)."""

    def __init__(self, pix_map, noise_temp, noise_pol, beam_fwhm_deg, nside, lmax, n_iter=1000, *, mask=None, mask_pol=None,
                 bins=None, rng="philox", seed=None):
        self.lmax, self.nside, self.n_iter = int(lmax), int(nside), int(n_iter)
        bl = _dev.gauss_beam(np.radians(beam_fwhm_deg), self.lmax)
        shared = _dev.Rng(rng, seed)
        self.cls_sampler = JointClsSampler(lmax, bins=bins, rng=shared)     # first: bad bins fail before the plan is built
        self.bins = self.cls_sampler.bins
        self.constrained_sampler = JointConstrainedRealization(pix_map, noise_temp, noise_pol, bl, lmax, 12 * nside ** 2, mask=mask,
                                                               mask_pol=mask_pol, rng=shared)

    def _unfold(self, dls):
        if self.bins is None:
            return dls
        from . import utils
        return {k: utils.unfold_bins(v, self.bins["BB" if k == "BB" else "TT"]) for k, v in dls.items()}

    def run(self, dls_init):
        keys = ("TT", "EE", "BB", "TE")
        dls = {k: f64(dls_init[k]) for k in keys}
        if self.bins is not None:
            for k in keys:
                want = len(self.bins["BB" if k == "BB" else "TT"]) - 1
                if dls[k].numel() != want:
                    raise ValueError("dls_init[%r] must hold %d binned values, got %d" % (k, want, dls[k].numel()))
        h = {k: [_dev.to_host(dls[k])] for k in keys}
        for _ in range(self.n_iter):
            sky, _ = self.constrained_sampler.sample(self._unfold(dls))
            dls = self.cls_sampler.sample(sky)
            for k in keys:
                h[k].append(_dev.to_host(dls[k]))
        return {k: np.array(v) for k, v in h.items()}
