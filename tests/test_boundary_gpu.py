"""Reference-interface gaps closed in round 2 (VERDICT r1 "Boundary gaps", ADVICE r1): the alternative CR kernels are
METHODS of PolarizedCenteredConstrainedRealization (CenteredGibbs.py:494-825), ULA_no_mask (:355-446),
utils.remove_monopole_dipole_contributions (variance_expension.pyx:103-111), the pixel-domain branch of the
non-centred no-mask draw (NonCenteredGibbs.py:155-160), plan create / solve / destroy cycles, and the refusal of
non-shard-aware samplers on sharded plans."""
import ctypes as C
import os
import sys

import numpy as np
import pytest
import torch

from oracle import reference_logic as R
from oracle import sht as O

pytestmark = pytest.mark.gpu
G = dict(np.load(os.path.join(os.path.dirname(__file__), "golden", "reference_nside4.npz")))   # materialised: NpzFile is lazy and not thread-safe
NSIDE, LMAX = 4, 8
NPIX, NRE = 12 * NSIDE ** 2, (LMAX + 1) ** 2


def close(a, b, tol=1e-10):
    a, b = np.asarray(a), np.asarray(b)
    return np.abs(a - b).max() <= tol * max(np.abs(b).max(), 1e-300)


def make_cr(**kw):
    from gibbssampler_b200.CenteredGibbs import PolarizedCenteredConstrainedRealization
    pix_map = {"Q": G["dQ"], "U": G["dU"], "EE": G["dE"], "BB": G["dB"]}
    return PolarizedCenteredConstrainedRealization(pix_map, np.full(NPIX, 1600.0), G["noise_pol"], G["bl_map"], LMAX, NPIX, float(G["fwhm"]),
                                                   rng="numpy", **kw)


def test_alternative_cr_kernels_are_methods_and_match_reference_golden():
    cr = make_cr(mask=G["mask"], n_gibbs=2)
    dls = {"EE": G["dls_EE"], "BB": G["dls_BB"]}
    s_old = {"EE": G["sample_mask_E"].copy(), "BB": G["sample_mask_B"].copy()}
    np.random.seed(int(G["aux_seed"]))
    sol, _ = cr.sample_gibbs_change_variable(dls, s_old)
    assert close(sol["EE"], G["aux_E"]) and close(sol["BB"], G["aux_B"])
    np.random.seed(int(G["overrelax_seed"]))
    sol, _ = cr.overrelaxation_sampler(dls, s_old)
    assert close(sol["EE"], G["overrelax_E"], 1e-8)
    np.random.seed(112)
    sol, acc = cr.sample_mala(dls, s_old)
    assert acc == int(G["mala_acc_112"]) and close(sol["EE"], G["mala_E_112"])
    # compute_gradient_mala / compute_log_density against the restated formulas (CenteredGibbs.py:494-558)
    gE, gB, mq, mu = cr.compute_gradient_mala(dls, s_old)
    prob = R.PolProblem(NSIDE, LMAX, G["dQ"], G["dU"], G["mask"] / G["noise_pol"], float(G["fwhm"]))
    qE, qB = prob.apply_Q(dls["EE"], dls["BB"], s_old["EE"], s_old["BB"])
    assert close(gE, prob.bdata_E - qE, 1e-9) and close(gB, prob.bdata_B - qB, 1e-9)
    rq, ru = R.synth_pol(s_old["EE"] * prob.bl_map, s_old["BB"] * prob.bl_map, NSIDE, LMAX)
    assert close(mq, rq) and close(mu, ru)
    want = 0.0
    for pol, bd in (("EE", prob.bdata_E), ("BB", prob.bdata_B)):
        iv = R.safe_inv(R.generate_var_cl(dls[pol]))
        want += -0.5 * np.sum(s_old[pol] ** 2 * iv) + np.sum(s_old[pol] * bd)
    want += -0.5 * np.sum(rq ** 2 * prob.inv_noise) - 0.5 * np.sum(ru ** 2 * prob.inv_noise)
    assert abs(cr.compute_log_density(dls, s_old) - want) <= 1e-9 * abs(want)
    assert abs(cr.compute_log_density(dls, s_old, mq, mu) - want) <= 1e-9 * abs(want)


def test_ula_no_mask_matches_restatement():
    cr = make_cr()
    dls = {"EE": G["dls_EE"], "BB": G["dls_BB"]}
    rng = np.random.default_rng(3)
    s_old = {"EE": rng.standard_normal(NRE), "BB": rng.standard_normal(NRE)}
    n_acc = 0
    for seed in (5, 6, 7, 8):
        np.random.seed(seed)
        xiE, xiB = np.random.normal(size=NRE), np.random.normal(size=NRE)
        u = np.random.uniform()
        want, log_ratio = R.ula_no_mask(dls["EE"], dls["BB"], G["bl_map"], G["dE"], G["dB"], s_old, NPIX, G["noise_pol"][0], cr.tau, xiE, xiB)
        np.random.seed(seed)
        got, acc = cr.ULA_no_mask(dls, s_old)
        assert acc == int(np.log(u) < log_ratio)
        if acc:
            assert close(got["EE"], want["EE"], 1e-12) and close(got["BB"], want["BB"], 1e-12)
            s_old = want
        else:
            assert got is s_old
        n_acc += acc
    assert n_acc >= 1


def test_noncentred_no_mask_draw_from_pixel_maps():
    """NonCenteredGibbs(mask_path=None, all_sph=False) with only Q/U data (NonCenteredGibbs.py:155-160)."""
    from gibbssampler_b200.NonCenteredGibbs import PolarizedNonCenteredConstrainedRealization
    dls = {"EE": G["dls_EE"], "BB": G["dls_BB"]}
    nc = PolarizedNonCenteredConstrainedRealization({"Q": G["dQ"], "U": G["dU"]}, np.full(NPIX, 1600.0), G["noise_pol"], G["bl_map"], LMAX, NPIX,
                                                    float(G["fwhm"]), all_sph=False, rng="numpy")
    np.random.seed(42)
    xiE, xiB = np.random.normal(size=NRE), np.random.normal(size=NRE)
    wE, wB = R.sample_no_mask_nc_pix(dls["EE"], dls["BB"], G["bl_map"], G["dQ"], G["dU"], 1.0 / G["noise_pol"], xiE, xiB, NSIDE, LMAX)
    np.random.seed(42)
    sol, acc = nc.sample(dls)
    assert acc == 0 and close(sol["EE"], wE) and close(sol["BB"], wB)


def test_remove_monopole_dipole_contributions():
    from gibbssampler_b200 import utils
    rng = np.random.default_rng(0)
    for L in (2, 5, 16):
        a = rng.standard_normal((L + 1) ** 2)
        want = a.copy()
        want[[0, 1, L + 1, L + 2]] = 0
        try:
            sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "_ref"))
            import variance_expension as ref   # the reference's own compiled Cython, when built
            assert np.array_equal(np.asarray(ref.remove_monopole_dipole_contributions(a.copy())), want)
        except ImportError:
            pass
        d = torch.as_tensor(a.copy(), device="cuda")
        out = utils.remove_monopole_dipole_contributions(d)
        assert out is d and np.array_equal(d.cpu().numpy(), want)
        h = a.copy()
        assert utils.remove_monopole_dipole_contributions(h) is h and np.array_equal(h, want)


def test_plan_create_solve_destroy_cycles():
    """ADVICE r1: the PCG workspaces live in the plan and die with it (no pointer-keyed cache): create, solve (E/B, a two-chain
    E/B batch, joint T/E/B), destroy, create at the same or another size, solve again."""
    from gibbssampler_b200 import _lib, _dev
    L = _lib.lib()
    th, _ = O.pix_angles(NSIDE)
    rng = np.random.default_rng(1)
    sols = []
    for cycle, (nside, lmax) in enumerate([(4, 8), (8, 16), (4, 8), (4, 8)]):
        h = C.c_void_p()
        _lib.check(L.gs_plan_create(C.byref(h), nside, lmax, -1))
        npix, nre = 12 * nside ** 2, (lmax + 1) ** 2
        g = np.random.default_rng(7)
        ell = np.arange(lmax + 1)
        dl_np = np.where(ell >= 2, 1.0 + 0.1 * ell, 0.0)
        dl, dl_te = _dev.f64(dl_np), _dev.f64(0.3 * dl_np)
        dl2 = _dev.f64(np.stack([dl_np, 0.5 * dl_np]))   # [chain][l]
        bl = _dev.f64(O.gauss_beam(np.radians(8.0), lmax))
        invn = _dev.f64(np.full(npix, 20.0))
        ninv = float(invn.sum().item()) / (4 * np.pi)
        rhs = _dev.f64(g.standard_normal((3, nre)))   # E, B, T
        rhs[:, [0, 1, lmax + 1, lmax + 2]] = 0
        rhs_e, rhs_b, rhs_t = rhs
        xe, xb = torch.empty_like(rhs_e), torch.empty_like(rhs_b)
        nit, res = C.c_int(0), C.c_double(0)
        rc = L.gs_cr_pcg_pol(h, _dev.ptr(dl), _dev.ptr(dl), _dev.ptr(bl), _dev.ptr(invn), ninv,
                             _dev.ptr(rhs_e), _dev.ptr(rhs_b), _dev.ptr(xe), _dev.ptr(xb), 0, 1e-10, 500, 8, C.byref(nit), C.byref(res),
                             _dev.stream())
        assert rc == 0 and res.value <= 1e-10
        rhs2 = torch.stack([rhs[[0, 1]], rhs[[1, 0]]])   # [chain][E, B][nre]
        x2 = torch.empty_like(rhs2)
        nit2, res2 = (C.c_int * 2)(), (C.c_double * 2)()
        rc = L.gs_cr_pcg_pol_batch(h, 2, _dev.ptr(dl2), _dev.ptr(dl2), _dev.ptr(bl), _dev.ptr(invn), ninv, _dev.ptr(rhs2[0, 0]),
                                   _dev.ptr(rhs2[0, 1]), _dev.ptr(x2[0, 0]), _dev.ptr(x2[0, 1]), 2 * nre, 1e-10, 500, 8, nit2, res2,
                                   _dev.stream())
        assert rc == 0 and max(res2) <= 1e-10
        x3 = torch.empty_like(rhs)   # T, E, B
        rc = L.gs_cr_pcg_teb(h, _dev.ptr(dl), _dev.ptr(dl_te), _dev.ptr(dl), _dev.ptr(dl), _dev.ptr(bl), _dev.ptr(invn), _dev.ptr(invn),
                             ninv, ninv, *[_dev.ptr(r) for r in (rhs_t, rhs_e, rhs_b)], *[_dev.ptr(v) for v in x3], 0, 1e-10, 500, 8,
                             C.byref(nit), C.byref(res), _dev.stream())
        assert rc == 0 and res.value <= 1e-10
        torch.cuda.synchronize()
        sols.append([a.cpu().numpy().copy() for a in (xe, x2, x3)])
        _lib.check(L.gs_plan_destroy(h))
    for k in range(3):
        assert np.array_equal(sols[0][k], sols[2][k]) and np.array_equal(sols[2][k], sols[3][k])


def test_non_shard_aware_samplers_refuse_sharded_plans():
    from gibbssampler_b200 import _lib
    from gibbssampler_b200.CenteredGibbs import PolarizedCenteredConstrainedRealization
    from gibbssampler_b200.sharded import ShardedPlan, run_local_group
    plans = ShardedPlan.local_group(NSIDE, LMAX, 2)
    dls = {"EE": G["dls_EE"], "BB": G["dls_BB"]}

    def work(p):
        cr = PolarizedCenteredConstrainedRealization({"Q": G["dQ"], "U": G["dU"]}, np.full(NPIX, 1600.0), G["noise_pol"], G["bl_map"], LMAX,
                                                     NPIX, float(G["fwhm"]), mask=G["mask"], plan=p, seed=3)
        s_old = {"EE": torch.zeros(p.nreal, dtype=torch.float64, device="cuda"), "BB": torch.zeros(p.nreal, dtype=torch.float64, device="cuda")}
        errs = 0
        for fn in (cr.sample_mala, cr.sample_gibbs_change_variable, cr.overrelaxation_sampler, cr.sample_mask_rj):
            try:
                fn(dls, s_old)
            except _lib.GibbsB200Error:
                errs += 1
        return errs

    assert run_local_group(plans, work) == [4, 4]
