"""Centred parametrisation (mirror of CenteredGibbs.py): inverse-gamma C_l draws and the
constrained-realization samplers (direct solve for full sky + isotropic noise, PCG for masked sky)."""
import ctypes as C

import numpy as np
import torch

from . import _dev, _lib, utils
from ._dev import f64, ptr, stream
from ._lib import check, GS_E_NOTCONVERGED
from .ClsSampler import ClsSampler
from .ConstrainedRealization import ConstrainedRealization
from .GibbsSampler import GibbsSampler


class CenteredClsSampler(ClsSampler):
    """TT: inverse-gamma draw of the binned D_l (CenteredGibbs.py:21-48)."""

    def sample(self, alms):
        out = self._invgamma_draw(f64(alms), self.bins)
        self.last_sigma = {"TT": self._last_cl}
        return out if isinstance(alms, torch.Tensor) else out.cpu().numpy()


class PolarizedCenteredClsSampler(ClsSampler):
    """EE then BB (CenteredGibbs.py:51-93).  The reference converts to complex alms first and calls
    hp.alm2cl; here alm2cl runs directly on the real layout."""

    def sample_one_pol(self, alms_real, pol="EE"):
        return self._invgamma_draw(f64(alms_real), self.bins[pol])

    def sample(self, alms):
        host = not isinstance(alms["EE"], torch.Tensor)
        ee = self.sample_one_pol(alms["EE"], "EE")
        cl_ee = self._last_cl
        bb = self.sample_one_pol(alms["BB"], "BB")
        self.last_sigma = {"EE": cl_ee, "BB": self._last_cl}
        if host:
            return {"EE": ee.cpu().numpy(), "BB": bb.cpu().numpy()}
        return {"EE": ee, "BB": bb}


class PolarizedCenteredConstrainedRealization(ConstrainedRealization):
    """CR step for EE/BB (CenteredGibbs.py:239-850)."""

    def __init__(self, pix_map, noise_temp, noise_pol, bl_map, lmax, Npix, bl_fwhm, mask_path=None,
                 gibbs_cr=False, n_gibbs=1, alpha=-0.995, overrelaxation=False, ula=True, *, mask=None,
                 rng="philox", seed=None, direct_when_isotropic=True, plan=None):
        super().__init__(pix_map, noise_temp, bl_map, bl_fwhm, lmax, Npix, mask_path=mask_path, mask=mask, rng=rng,
                         seed=seed, plan=plan)
        self.noise_temp = noise_temp
        self.noise_pol = noise_pol
        self.n_gibbs = n_gibbs
        self.ula = ula
        self.inv_noise_pol = self._inv_noise_from(noise_pol)          # mask / noise_pol (CenteredGibbs.py:261-274)
        self.sqrt_inv_noise_pol = torch.sqrt(self.inv_noise_pol)
        self.inv_noise = [self.inv_noise_pol]
        self.mu = float(self.inv_noise_pol.max().item()) + 1e-14       # CenteredGibbs.py:276 (local max on sharded plans)
        self.gibbs_cr = gibbs_cr
        self.overrelaxation = overrelaxation
        self.pcg_accuracy = 1.0e-5                                      # CenteredGibbs.py:280
        self.pcg_itermax = 4000
        self.pcg_check_every = 8
        self.fluct_iter = 3                                            # utils.adjoint_synthesis_hp uses iter=3 (utils.py:89)
        self.dls_to_cls_array = np.array([2 * np.pi / (l * (l + 1)) if l != 0 else 0 for l in range(lmax + 1)])
        self.alpha = alpha
        self.bl_fwhm = bl_fwhm
        self.tau = 0.02
        self.direct_when_isotropic = direct_when_isotropic
        self.ninv_sum_over_4pi = self.plan.allreduce_sum(_dev.dsum(self.inv_noise_pol)) / (4 * np.pi)
        self.noise_pol0 = float(f64(noise_pol).reshape(-1)[0].item())
        self.d_Q = self.plan.local_map(f64(pix_map["Q"])) if "Q" in pix_map else None
        self.d_U = self.plan.local_map(f64(pix_map["U"])) if "U" in pix_map else None
        self.d_E = self.plan.local_alm(f64(pix_map["EE"])) if "EE" in pix_map else None
        self.d_B = self.plan.local_alm(f64(pix_map["BB"])) if "BB" in pix_map else None
        # second_part_grad = b (Npix/4pi) map2alm_iter0(N^-1 d) = B A^T N^-1 d (CenteredGibbs.py:298-308):
        # constant data term of every right-hand side
        if self.d_Q is not None:
            e, b = self.plan.map2alm_spin2(self.d_Q, self.d_U, adjoint=True, pixw=self.inv_noise_pol,
                                           fl=self.bl_gauss_d, real_layout=True)
            self.second_part_grad_E, self.second_part_grad_B = e, b
        self.last_rhs = None

    # ------------------------------------------------------------------ helpers
    def _dls(self, all_dls):
        e, b = f64(all_dls["EE"]), f64(all_dls["BB"])
        assert e.numel() == self.lmax + 1 and b.numel() == self.lmax + 1, "need unbinned D_l of length lmax+1"
        return e, b

    def _ret(self, sol, like):
        if isinstance(like, torch.Tensor):
            return sol
        return {k: v.cpu().numpy() for k, v in sol.items()}

    # ------------------------------------------------------------------ full sky, isotropic noise
    def sample_no_mask(self, all_dls):
        """Diagonal solve (CenteredGibbs.py:317-353); needs the data in harmonic space (pix_map["EE"/"BB"])."""
        if self.d_E is None:
            raise _lib.GibbsB200Error("sample_no_mask needs pix_map['EE'] and pix_map['BB'] (main_polarization.py:44)")
        dle, dlb = self._dls(all_dls)
        w = self.Npix / (self.noise_pol0 * 4 * np.pi)
        n = self.dimension_alm
        xe, xb = self.rng.normal(n), self.rng.normal(n)
        oe, ob = torch.empty_like(xe), torch.empty_like(xb)
        L = _lib.lib()
        check(L.gs_cr_direct(ptr(dle), ptr(self.bl_gauss_d), ptr(self.d_E), ptr(xe), w, self.lmax, 0, ptr(oe), stream()))
        check(L.gs_cr_direct(ptr(dlb), ptr(self.bl_gauss_d), ptr(self.d_B), ptr(xb), w, self.lmax, 0, ptr(ob), stream()))
        return self._ret({"EE": oe, "BB": ob}, all_dls["EE"]), 1

    # ------------------------------------------------------------------ masked sky: PCG
    def build_rhs(self, all_dls, xi=None):
        """b of Q x = b (CenteredGibbs.py:469-483).  xi = (xi_Q, xi_U, xi_E, xi_B) may be injected."""
        dle, dlb = self._dls(all_dls)
        if xi is None:
            if self.plan.world > 1 and self.rng.mode == "numpy":
                # reference order on the full arrays (every rank draws the same stream), then cut to the shard
                xi = (self.rng.normal(self.plan.npix_global), self.rng.normal(self.plan.npix_global),
                      self.rng.normal(self.plan.nreal_global), self.rng.normal(self.plan.nreal_global))
            else:
                xi = (self.rng.normal(self.npix_local), self.rng.normal(self.npix_local),
                      self.rng.normal(self.dimension_alm), self.rng.normal(self.dimension_alm))
        xq, xu, xe, xb = [f64(x) for x in xi]
        xq, xu, xe, xb = self.plan.local_map(xq), self.plan.local_map(xu), self.plan.local_alm(xe), self.plan.local_alm(xb)
        rhs_e = torch.empty(self.dimension_alm, dtype=torch.float64, device=self.dev)
        rhs_b = torch.empty_like(rhs_e)
        check(_lib.lib().gs_cr_rhs_pol(self.plan._h, ptr(dle), ptr(dlb), ptr(self.bl_gauss_d), ptr(self.inv_noise_pol),
                                       ptr(self.sqrt_inv_noise_pol), ptr(self.second_part_grad_E),
                                       ptr(self.second_part_grad_B), None, None, ptr(xq), ptr(xu), ptr(xe), ptr(xb),
                                       self.fluct_iter, ptr(rhs_e), ptr(rhs_b), stream()))
        return rhs_e, rhs_b

    def solve(self, all_dls, rhs_e, rhs_b, x0=None):
        """PCG solve of Q x = b (qcinv chain, CenteredGibbs.py:467,486-488)."""
        dle, dlb = self._dls(all_dls)
        if x0 is None:
            xe = torch.empty(self.dimension_alm, dtype=torch.float64, device=self.dev)
            xb = torch.empty_like(xe)
        else:
            xe, xb = f64(x0["EE"]).clone(), f64(x0["BB"]).clone()
        nit, res = C.c_int(0), C.c_double(0.0)
        rc = _lib.lib().gs_cr_pcg_pol(self.plan._h, ptr(dle), ptr(dlb), ptr(self.bl_gauss_d), ptr(self.inv_noise_pol),
                                      self.ninv_sum_over_4pi, ptr(rhs_e), ptr(rhs_b), ptr(xe), ptr(xb),
                                      0 if x0 is None else 1, self.pcg_accuracy, self.pcg_itermax,
                                      self.pcg_check_every, C.byref(nit), C.byref(res), stream())
        self.last_pcg_iterations, self.last_pcg_residual = nit.value, res.value
        if rc not in (0, GS_E_NOTCONVERGED):  # GS_E_NOTCONVERGED is reported through last_pcg_residual: qcinv also just stops at iter_max
            check(rc)
        return xe, xb

    def apply_Q(self, all_dls, x):
        dle, dlb = self._dls(all_dls)
        xe, xb = f64(x["EE"]), f64(x["BB"])
        ye, yb = torch.empty_like(xe), torch.empty_like(xb)
        check(_lib.lib().gs_cr_apply_q_pol(self.plan._h, ptr(dle), ptr(dlb), ptr(self.bl_gauss_d), ptr(self.inv_noise_pol),
                                           ptr(xe), ptr(xb), ptr(ye), ptr(yb), stream()))
        return {"EE": ye, "BB": yb}

    def sample_mask(self, all_dls, xi=None):
        """CR step with a PCG solver (CenteredGibbs.py:448-491)."""
        rhs_e, rhs_b = self.build_rhs(all_dls, xi)
        self.last_rhs = (rhs_e, rhs_b)
        xe, xb = self.solve(all_dls, rhs_e, rhs_b)
        return self._ret({"EE": xe, "BB": xb}, all_dls["EE"]), 1

    def _single_gpu_only(self, what):
        """The Metropolis-adjusted / auxiliary-variable CR kernels reduce over whole vectors and draw full-size fields; on an
        m-sharded plan every rank would see partial sums and its own random numbers and the ranks' accept decisions would
        diverge.  They are not shard-aware: refuse instead of corrupting the chain."""
        if self.plan.world > 1:
            raise _lib.GibbsB200Error("%s is not available on an m-sharded plan (world = %d): use the PCG sampler "
                                      "(sample_mask) for sharded chains" % (what, self.plan.world))

    # ---- the alternative CR kernels of the reference class (CenteredGibbs.py:494-825) live in cr_extra; bound here as
    # ---- methods so that cr.sample_mala(...) etc. work as on the reference object
    def compute_gradient_mala(self, all_dls, s_old):
        """CenteredGibbs.py:494-520 -> (grad_E, grad_B, s_Q_pix, s_U_pix)."""
        from . import cr_extra
        return cr_extra.compute_gradient_mala(self, all_dls, s_old)

    def compute_log_density(self, all_dls, s, s_E_pix=None, s_B_pix=None):
        """CenteredGibbs.py:534-558 (the pixel-space maps are recomputed when not supplied)."""
        from . import cr_extra
        return cr_extra.compute_log_density(self, all_dls, s, s_E_pix, s_B_pix)

    def sample_mala(self, all_dls, s_old, grad_E_old=None, grad_B_old=None):
        """CenteredGibbs.py:560-603."""
        from . import cr_extra
        return cr_extra.sample_mala(self, all_dls, s_old)

    def sample_gibbs_change_variable(self, all_dls, old_s):
        """CenteredGibbs.py:676-729."""
        from . import cr_extra
        return cr_extra.sample_gibbs_change_variable(self, all_dls, old_s)

    def overrelaxation_sampler(self, all_dls, old_s):
        """CenteredGibbs.py:733-825."""
        from . import cr_extra
        return cr_extra.overrelaxation_sampler(self, all_dls, old_s)

    def ULA_no_mask(self, all_dls, s_old):
        """Preconditioned MALA step for full sky + isotropic noise, all in harmonic space (CenteredGibbs.py:417-446 with
        :355-414); RNG order: EE normals, BB normals, one uniform.  Returns (s, accept)."""
        self._single_gpu_only("ULA_no_mask")
        if self.d_E is None:
            raise _lib.GibbsB200Error("ULA_no_mask needs pix_map['EE'] and pix_map['BB'] (CenteredGibbs.py:364-365)")
        dle, dlb = self._dls(all_dls)
        w = self.Npix / (self.noise_pol0 * 4 * np.pi)
        L = _lib.lib()
        scratch = torch.empty(592, dtype=torch.float64, device=self.dev)
        lr = torch.empty(2, dtype=torch.float64, device=self.dev)
        new = {}
        for k, (pol, dl, d) in enumerate((("EE", dle, self.d_E), ("BB", dlb, self.d_B))):
            so = f64(s_old[pol])
            xi = self.rng.normal(self.dimension_alm)
            out = torch.empty_like(so)
            check(L.gs_ula_nomask(ptr(dl), ptr(self.bl_gauss_d), ptr(d), ptr(so), ptr(xi), w, self.tau, self.lmax, ptr(out),
                                  ptr(scratch), ptr(lr[k:]), stream()))
            new[pol] = out
        log_ratio = float(lr.sum().item())
        u = float(self.rng.uniform(2)[0].item()) if self.rng.mode == "philox" else np.random.uniform()
        if np.log(u) < log_ratio:
            return self._ret(new, s_old["EE"]), 1
        return s_old, 0

    def sample_mask_rj(self, all_dls, s_old, xi=None, u=None):
        """RJPO (CenteredGibbs.py:606-674): PCG started at -s_old, accept with min(1, exp(-r^T (s_old - s)))."""
        self._single_gpu_only("sample_mask_rj")
        rhs_e, rhs_b = self.build_rhs(all_dls, xi)
        so = {"EE": f64(s_old["EE"]), "BB": f64(s_old["BB"])}
        xe, xb = self.solve(all_dls, rhs_e, rhs_b, x0={"EE": -so["EE"], "BB": -so["BB"]})
        q = self.apply_Q(all_dls, {"EE": xe, "BB": xb})
        r_e, r_b = rhs_e - q["EE"], rhs_b - q["BB"]
        log_proba = -float((torch.dot(r_e, so["EE"] - xe) + torch.dot(r_b, so["BB"] - xb)).item())
        if u is None:
            u = float(self.rng.uniform(2)[0].item()) if self.rng.mode == "philox" else np.random.uniform()
        if np.log(u) < log_proba:
            return self._ret({"EE": xe, "BB": xb}, all_dls["EE"]), 1
        return s_old, 0

    def sample(self, all_dls, s_old=None):
        """Dispatcher of the reference (CenteredGibbs.py:828-850).  The auxiliary-variable, over-relaxation
        and MALA branches live in gibbssampler_b200.cr_extra."""
        masked = self.masked or self.mask_path is not None
        if self.gibbs_cr == True and s_old is not None and masked:
            from . import cr_extra
            if self.overrelaxation == True:
                return cr_extra.overrelaxation_sampler(self, all_dls, s_old)
            if self.ula == False:
                return cr_extra.sample_gibbs_change_variable(self, all_dls, s_old)
            s_int, _ = cr_extra.sample_gibbs_change_variable(self, all_dls, s_old)
            return cr_extra.sample_mala(self, all_dls, s_int)
        if masked and s_old is not None and self.ula == True:
            from . import cr_extra
            return cr_extra.sample_mala(self, all_dls, s_old)
        if (not masked) and self.direct_when_isotropic and self.d_E is not None:
            # the reference disables this branch with `and False` (CenteredGibbs.py:845) and runs the PCG with
            # an all-ones mask; the direct solve samples the same distribution exactly (SURVEY.md 3.2)
            return self.sample_no_mask(all_dls)
        return self.sample_mask(all_dls)


class CenteredGibbs(GibbsSampler):
    def __init__(self, pix_map, noise_temp, noise_pol, beam, nside, lmax, Npix, mask_path=None,
                 polarization=False, bins=None, n_iter=100000, rj_step=False, all_sph=False, gibbs_cr=False,
                 overrelaxation=False, ula=False, *, mask=None, rng="philox", seed=None, verbose=False, plan=None, keep_sigma=False):
        """`plan` = a gibbssampler_b200.sharded.ShardedPlan runs this single chain m-sharded over the GPUs of the
        plan's process group (BASELINE config #4); inputs are full-sky arrays as usual, sky maps returned by the
        constrained sampler are local alm shards (plan.gather_alm reassembles them).
        keep_sigma=True: run() also leaves sigma_history = {"TT"} or {"EE", "BB"}: (n_iter, lmax + 1) numpy arrays whose row i is
        the empirical spectrum of the sky drawn in iteration i (the sky row i + 1 of the D history was drawn from), the input of
        BlackwellRao.  Not available with a sharded plan (any world size), in run_fused or in multichain.run_chains."""
        if keep_sigma and plan is not None:
            raise _lib.GibbsB200Error("keep_sigma is not available with a sharded plan: the chain's spectra are not recorded there")
        self.keep_sigma = bool(keep_sigma)
        super().__init__(pix_map, noise_temp, beam, nside, lmax, polarization=polarization, bins=bins, n_iter=n_iter,
                         rj_step=rj_step, gibbs_cr=gibbs_cr, verbose=verbose)
        shared = _dev.Rng(rng, seed)
        # the C_l draw must be identical on every rank of a sharded chain (same seed); the pixel / alm draws of
        # the constrained realization are per shard and must differ between ranks
        cr_rng = shared
        if plan is not None and plan.world > 1 and shared.mode == "philox":
            cr_rng = _dev.Rng(rng, shared.seed + 7919 * (plan.rank + 1))
        if not polarization:  # CenteredGibbs.py:867-870
            from .Temperature import CenteredConstrainedRealization
            self.constrained_sampler = CenteredConstrainedRealization(pix_map, noise_temp, self.bl_map, beam, lmax, Npix, mask_path,
                                                                      isotropic=True, mask=mask, rng=cr_rng, plan=plan)
            self.cls_sampler = CenteredClsSampler(pix_map, lmax, nside, self.bins, self.bl_map, noise_temp, rng=shared, plan=plan)
            return
        self.cls_sampler = PolarizedCenteredClsSampler(pix_map, lmax, nside, self.bins, self.bl_map, noise_temp,
                                                       mask_path=mask_path, mask=mask, rng=shared, plan=plan)
        self.constrained_sampler = PolarizedCenteredConstrainedRealization(
            pix_map, noise_temp, noise_pol, self.bl_map, lmax, Npix, beam, mask_path=mask_path, gibbs_cr=gibbs_cr,
            overrelaxation=overrelaxation, ula=ula, mask=mask, rng=cr_rng, plan=plan)

    def run_fused(self, dls_init, use_graph=True):
        """run() for the full-sky isotropic-noise polarised chain (BASELINE config #1) in ONE C call: the whole loop of
        GibbsSampler.run_polarization (GibbsSampler.py:118-180) stays on the device (gs_gibbs_run_centered_fullsky: three kernels
        per iteration, captured once in a CUDA graph and replayed).  Same return tuple as run(); the per-iteration timing lists
        hold the mean.  Philox draws only (numpy-stream parity is what run() is for)."""
        import time
        cr = self.constrained_sampler
        if self.keep_sigma:
            raise _lib.GibbsB200Error("run_fused does not record the sky spectra: use run() for a chain built with keep_sigma=True")
        if not self.polarization or cr.masked or cr.d_E is None or cr.plan.world > 1 or cr.rng.mode != "philox":
            raise _lib.GibbsB200Error("run_fused: polarised full-sky chain with harmonic data (pix_map['EE'/'BB']) and Philox draws only")
        bins = {k: torch.as_tensor(np.asarray(self.bins[k]), dtype=torch.int32, device=cr.dev) for k in ("EE", "BB")}
        nb = {k: bins[k].numel() - 1 for k in bins}
        init = {k: f64(dls_init[k]).contiguous() for k in ("EE", "BB")}
        hist = {k: torch.empty((self.n_iter + 1, nb[k]), dtype=torch.float64, device=cr.dev) for k in bins}
        cr.rng.counter += 1
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        check(_lib.lib().gs_gibbs_run_centered_fullsky(self.lmax, cr.Npix, cr.noise_pol0, ptr(cr.bl_gauss_d), ptr(cr.d_E), ptr(cr.d_B),
                                                       ptr(bins["EE"]), nb["EE"], ptr(bins["BB"]), nb["BB"], ptr(init["EE"]), ptr(init["BB"]),
                                                       int(self.n_iter), ((cr.rng.seed << 8) + cr.rng.counter) & 0xFFFFFFFFFFFFFFFF, ptr(hist["EE"]), ptr(hist["BB"]),
                                                       None, None, 1 if use_graph else 0, stream()))
        dt = (time.perf_counter() - t0) / max(1, self.n_iter)
        h = {k: hist[k].cpu().numpy() for k in hist}
        return h, np.ones(self.n_iter), np.full(self.n_iter, 0.5 * dt), np.full(self.n_iter, 0.5 * dt)


def sample_mask_batch(crs, dls_list, xis=None):
    """sample_mask (CenteredGibbs.py:448-491) of TWO independent chains on the same data in one batched solve: every chain
    draws its own right-hand side from its own random stream (as two processes of the reference would), the two PCG solves run
    side by side with chain-batched mat-vecs that share the Legendre recurrences (gs_cr_pcg_pol_batch).  `crs`: the chains'
    PolarizedCenteredConstrainedRealization objects (same plan, data, mask and noise); returns [(alms dict, 1), ...]."""
    assert len(crs) == len(dls_list) and len(crs) in (1, 2)
    if len(crs) == 1:
        return [crs[0].sample_mask(dls_list[0], None if xis is None else xis[0])]
    a, b = crs
    if a.plan is not b.plan or a.plan.world > 1:
        raise _lib.GibbsB200Error("sample_mask_batch needs two chains on the same unsharded plan")
    if a.inv_noise_pol.data_ptr() != b.inv_noise_pol.data_ptr():
        if not torch.equal(a.inv_noise_pol, b.inv_noise_pol):
            raise _lib.GibbsB200Error("sample_mask_batch: the chains of a batch share the noise / mask (N^-1)")
        b.inv_noise_pol = a.inv_noise_pol   # checked once: later calls compare pointers only
    n, lmax = a.dimension_alm, a.lmax
    rhs = torch.empty((2, 2, n), dtype=torch.float64, device=a.dev)      # [chain][E, B][n]
    dl = torch.empty((2, 2, lmax + 1), dtype=torch.float64, device=a.dev)  # [E, B][chain][L + 1]
    for k, (cr, dls) in enumerate(zip(crs, dls_list)):
        re_, rb_ = cr.build_rhs(dls, None if xis is None else xis[k])
        cr.last_rhs = (re_, rb_)
        rhs[k, 0].copy_(re_)
        rhs[k, 1].copy_(rb_)
        dle, dlb = cr._dls(dls)
        dl[0, k].copy_(dle)
        dl[1, k].copy_(dlb)
    x = torch.empty_like(rhs)
    nit, res = (C.c_int * 2)(), (C.c_double * 2)()
    rc = _lib.lib().gs_cr_pcg_pol_batch(a.plan._h, 2, ptr(dl[0]), ptr(dl[1]), ptr(a.bl_gauss_d), ptr(a.inv_noise_pol),
                                        a.ninv_sum_over_4pi, ptr(rhs[0, 0]), ptr(rhs[0, 1]), ptr(x[0, 0]), ptr(x[0, 1]), 2 * n,
                                        a.pcg_accuracy, a.pcg_itermax, a.pcg_check_every, nit, res, stream())
    if rc not in (0, GS_E_NOTCONVERGED):
        check(rc)
    out = []
    for k, (cr, dls) in enumerate(zip(crs, dls_list)):
        cr.last_pcg_iterations, cr.last_pcg_residual = nit[k], res[k]
        out.append((cr._ret({"EE": x[k, 0], "BB": x[k, 1]}, dls["EE"]), 1))
    return out
