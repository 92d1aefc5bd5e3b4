"""Joint T/E/B constrained realization on a cut sky (gs_cr_rhs_teb / gs_cr_pcg_teb / gs_cr_apply_q_teb and
JointSampler.JointConstrainedRealization with pixel data) against the oracle (tests.teb_oracle.TPProblem), against the
separate TT and E/B solves when C^TE = 0, and in distribution.  T and P masks differ and cut different rings; noise is per pixel."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import reference_logic as R
from tests import teb_problem as T
from tests.teb_oracle import te_blocks

pytestmark = pytest.mark.gpu

PAIRS = [("galplane", "band"), ("holes", "galplane"), ("band", "holes")]


def dev(x):
    return torch.as_tensor(np.ascontiguousarray(x, dtype=np.float64), device="cuda")


def host(x):
    return x.cpu().numpy() if isinstance(x, torch.Tensor) else np.asarray(x)


def rel(a, b):
    a, b = np.concatenate([host(v) for v in a]), np.concatenate([np.asarray(v) for v in b])
    return float(np.abs(a - b).max() / np.abs(b).max())


def sampler(P, nside, lmax, **kw):
    from gibbssampler_b200 import _dev
    from gibbssampler_b200.JointSampler import JointConstrainedRealization
    bl = _dev.gauss_beam(np.radians(P["fwhm"]), lmax)
    return JointConstrainedRealization(P["d"], P["noise_T"], P["noise_P"], bl, lmax, 12 * nside ** 2, mask=P["mask_T"],
                                       mask_pol=P["mask_P"], **kw)


def as_dict(x):
    return {"TT": dev(x[0]), "EE": dev(x[1]), "BB": dev(x[2])}


@pytest.mark.parametrize("kinds", PAIRS)
def test_apply_q_matches_oracle_and_ignores_ring_shortcuts(kinds):
    from gibbssampler_b200 import _lib
    nside, lmax = 8, 16
    P = T.problem(nside, lmax, *kinds, seed=11)
    dls = T.spectra(lmax)
    cr = sampler(P, nside, lmax, seed=1)
    n = (lmax + 1) ** 2
    rng = np.random.default_rng(5)
    x = tuple(rng.standard_normal(n) for _ in range(3))
    ref = P["prob"].apply_Q(dls, x)
    y = cr.apply_Q(dls, as_dict(x))
    got = (y["TT"], y["EE"], y["BB"])
    assert rel(got, ref) < 1e-10
    # the operator does not depend on which rings are skipped or taken without transforms: this fails if the spin-0 half
    # reads the ring flags (or the constant ring weights) built from N_P^-1
    L = _lib.lib()
    for setter in (L.gs_set_ring_skip, L.gs_set_ring_const):
        old = setter(0)
        try:
            y2 = cr.apply_Q(dls, as_dict(x))
        finally:
            setter(old)
        assert rel((y2["TT"], y2["EE"], y2["BB"]), [host(v) for v in got]) < 1e-12


def test_masks_of_the_tests_cut_different_rings():
    import bench
    nside = 8
    z = bench.pixel_z(nside)
    rings = np.unique(z)
    for a, b in PAIRS:
        ma, mb = T.make_mask(nside, a), T.make_mask(nside, b)
        ca = [np.ptp(ma[z == r]) > 0 for r in rings]
        cb = [np.ptp(mb[z == r]) > 0 for r in rings]
        assert ca != cb, (a, b)


def test_uncoupled_system_equals_the_separate_tt_and_pol_calls():
    from gibbssampler_b200 import _lib
    from gibbssampler_b200._dev import ptr, stream
    nside, lmax = 8, 16
    P = T.problem(nside, lmax, "galplane", "band", seed=12)
    dls = T.spectra(lmax, te_frac=0.0)
    cr = sampler(P, nside, lmax, seed=2)
    L = _lib.lib()
    n = (lmax + 1) ** 2
    rng = np.random.default_rng(6)
    x = tuple(dev(rng.standard_normal(n)) for _ in range(3))
    d = {k: dev(v) for k, v in dls.items()}
    y = cr.apply_Q(dls, {"TT": x[0], "EE": x[1], "BB": x[2]})
    yt, ye, yb = (torch.empty(n, dtype=torch.float64, device="cuda") for _ in range(3))
    _lib.check(L.gs_cr_apply_q_tt(cr.plan._h, ptr(d["TT"]), ptr(cr.bl), ptr(cr.inv_noise_T), ptr(x[0]), ptr(yt), stream()))
    _lib.check(L.gs_cr_apply_q_pol(cr.plan._h, ptr(d["EE"]), ptr(d["BB"]), ptr(cr.bl), ptr(cr.inv_noise_P), ptr(x[1]), ptr(x[2]),
                                   ptr(ye), ptr(yb), stream()))
    assert rel((y["TT"], y["EE"], y["BB"]), [host(v) for v in (yt, ye, yb)]) < 1e-12
    # solutions to 1e-11
    cr.pcg_accuracy = 1e-11
    rhs = cr.build_rhs(dls)
    xs = cr.solve(dls, *rhs)
    st, se, sb = (torch.empty(n, dtype=torch.float64, device="cuda") for _ in range(3))
    it = C.c_int(0)
    _lib.check(L.gs_cr_pcg_tt(cr.plan._h, ptr(d["TT"]), ptr(cr.bl), ptr(cr.inv_noise_T), cr.ninvT_sum_over_4pi, ptr(rhs[0]), ptr(st),
                              0, 1e-11, 4000, 8, C.byref(it), None, stream()))
    _lib.check(L.gs_cr_pcg_pol(cr.plan._h, ptr(d["EE"]), ptr(d["BB"]), ptr(cr.bl), ptr(cr.inv_noise_P), cr.ninvP_sum_over_4pi,
                               ptr(rhs[1]), ptr(rhs[2]), ptr(se), ptr(sb), 0, 1e-11, 4000, 8, C.byref(it), None, stream()))
    for a, b in zip(xs, (st, se, sb)):
        assert np.abs(host(a) - host(b)).max() <= 1e-8 * np.abs(host(b)).max()


@pytest.mark.parametrize("kinds", PAIRS[:2])
def test_rhs_with_injected_draws_matches_oracle(kinds):
    from gibbssampler_b200 import _lib
    from gibbssampler_b200._dev import ptr, stream
    nside, lmax = 8, 16
    P = T.problem(nside, lmax, *kinds, seed=13)
    dls = T.spectra(lmax)
    cr = sampler(P, nside, lmax, seed=3)
    npix, n = 12 * nside ** 2, (lmax + 1) ** 2
    rng = np.random.default_rng(7)
    xi = [rng.standard_normal(npix) for _ in range(3)] + [rng.standard_normal(n) for _ in range(3)]
    ref = P["prob"].rhs(dls, *xi, fluct_iter=3)
    got = cr.build_rhs(dls, xi=xi)
    assert rel(got, ref) < 1e-10
    # the data terms computed from the maps instead of passed precomputed
    L = _lib.lib()
    d = {k: dev(v) for k, v in dls.items()}
    maps = [dev(P["d"][k]) for k in ("I", "Q", "U")]
    xd = [dev(v) for v in xi]
    out = [torch.empty(n, dtype=torch.float64, device="cuda") for _ in range(3)]
    _lib.check(L.gs_cr_rhs_teb(cr.plan._h, ptr(d["TT"]), ptr(d["TE"]), ptr(d["EE"]), ptr(d["BB"]), ptr(cr.bl), ptr(cr.inv_noise_T),
                               ptr(cr.sqrt_inv_noise_T), ptr(cr.inv_noise_P), ptr(cr.sqrt_inv_noise_P), None, None, None,
                               *[ptr(m) for m in maps], *[ptr(v) for v in xd], 3, *[ptr(o) for o in out], stream()))
    assert rel(out, ref) < 1e-10


def test_pcg_reaches_the_dense_solve():
    nside, lmax = 4, 8
    P = T.problem(nside, lmax, "holes", "galplane", seed=14)
    dls = T.spectra(lmax)
    cr = sampler(P, nside, lmax, seed=4)
    cr.pcg_accuracy = 1e-12
    npix, n = 12 * nside ** 2, (lmax + 1) ** 2
    rng = np.random.default_rng(8)
    xi = [rng.standard_normal(npix) for _ in range(3)] + [rng.standard_normal(n) for _ in range(3)]
    s, acc = cr.sample(dls, xi=xi)
    assert acc == 1 and 0 < cr.last_pcg_iterations < 4000 and cr.last_pcg_residual <= 1e-12
    b = np.concatenate(P["prob"].rhs(dls, *xi))
    act = T.active(lmax)
    Q = P["prob"].dense_Q(dls)
    ref = np.zeros(3 * n)
    ref[act] = np.linalg.solve(Q[np.ix_(act, act)], b[act])
    got = np.concatenate([host(s[k]) for k in ("TT", "EE", "BB")])
    assert np.abs(got - ref).max() <= 1e-8 * np.abs(ref).max()
    # the oracle's PCG takes about as many iterations
    _, it = P["prob"].pcg(dls, P["prob"].rhs(dls, *xi), eps=1e-12)
    assert abs(it - cr.last_pcg_iterations) <= 3
    # warm start (r0 = b - Q x0) from a perturbed solution reaches the same solution
    live = {k: dev(a) for k, a in zip(("TT", "EE", "BB"), np.split(act.astype(np.float64), 3))}   # Q is zero off these entries
    x0 = {k: s[k] + dev(0.1 * rng.standard_normal(n)) * live[k] * s[k].abs().max() for k in ("TT", "EE", "BB")}
    x = cr.solve(dls, *cr.last_rhs, x0=x0)
    assert cr.last_pcg_iterations > 0 and cr.last_pcg_residual <= 1e-12
    assert np.abs(np.concatenate([host(v) for v in x]) - ref).max() <= 1e-8 * np.abs(ref).max()


def test_device_draws_have_mean_and_covariance_of_the_conditional():
    """fluct_iter = 0: x = Q^-1 b with b ~ N(B A^T N^-1 d, Q), so x ~ N(Q^-1 B A^T N^-1 d, Q^-1) exactly.  4000 draws at NSIDE 4;
    on 24 fixed projections u (12 random, 12 on single T / E / B coefficients and T-E pairs of one (l, m)):
    |mean - u.mu| / sqrt(u Q^-1 u / N) < 4.5 and the sample variance within 5 standard errors ((2 / (N - 1))^1/2 relative) of
    u Q^-1 u; plus the T-E cross covariance of 4 coefficients within 5 standard errors."""
    nside, lmax, N = 4, 8, 4000
    P = T.problem(nside, lmax, "galplane", "band", seed=15, noise_T=3000.0, noise_P=80.0)   # noise per a_lm ~ C_l at l ~ 5
    dls = T.spectra(lmax, te_frac=0.8)
    cr = sampler(P, nside, lmax, seed=1234)
    cr.fluct_iter = 0
    cr.pcg_accuracy = 1e-10
    n = (lmax + 1) ** 2
    act = T.active(lmax)
    prob = P["prob"]
    Q = prob.dense_Q(dls)[np.ix_(act, act)]
    cov = np.linalg.inv(Q)
    mu = np.zeros(3 * n)
    mu[act] = np.linalg.solve(Q, np.concatenate(prob.bdata)[act])
    X = np.empty((N, 3 * n))
    for k in range(N):
        s, _ = cr.sample(dls)
        X[k] = np.concatenate([host(s[f]) for f in ("TT", "EE", "BB")])
    assert np.abs(X[:, ~act]).max() <= 1e-12 * np.abs(X).max()
    Xa, mua = X[:, act], mu[act]
    na = int(act.sum())
    rng = np.random.default_rng(0)
    U = [rng.standard_normal(na) for _ in range(12)]
    ell = R.l_of_real_layout(lmax)
    idx = np.nonzero(act)[0]
    pos = {int(g): i for i, g in enumerate(idx)}
    pairs = []
    for j in (ell.tolist().index(2), ell.tolist().index(5), lmax + 1 + 2 * 4, (lmax + 1) ** 2 - 1):
        t, e, b = pos[j], pos[n + j], pos[2 * n + j]
        pairs.append((t, e))
        for coef in ((t,), (e,), (b,)):
            u = np.zeros(na)
            u[list(coef)] = 1.0
            U.append(u)
    for k, u in enumerate(U):
        proj = Xa @ u
        var = u @ cov @ u
        zm = abs(proj.mean() - u @ mua) / np.sqrt(var / N)
        zv = abs(proj.var(ddof=1) / var - 1) / np.sqrt(2.0 / (N - 1))
        assert zm < 4.5 and zv < 5, (k, zm, zv, proj.var(ddof=1), var)
    C_s = np.cov(Xa.T)
    for t, e in pairs:
        se = np.sqrt((cov[t, t] * cov[e, e] + cov[t, e] ** 2) / (N - 1))
        assert abs(C_s[t, e] - cov[t, e]) < 5 * se, (t, e, C_s[t, e], cov[t, e], se)
    # the coupling is really there: posterior T-E correlation of about 0.3 at l = 2 and 5 for these inputs
    t, e = pairs[0]
    assert abs(cov[t, e]) > 0.2 * np.sqrt(cov[t, t] * cov[e, e]) and abs(C_s[t, e] - cov[t, e]) < 0.2 * abs(cov[t, e])


def test_masked_joint_gibbs_chain_tracks_the_realised_spectra():
    """Short TT/TE/EE/BB chain on a high-S/N masked simulation (T: galplane, P: band): the C_l step samples C | s, whose mean
    for the TT/TE/EE block is (2l+1) Chat_l / (2l - 5); with low noise s follows the input sky on the observed part, so the
    chain's posterior means of TT, EE and TE stay within 35 % of that value for the realised spectra at l = 10, 20 (the bound
    also covers the 20 % of the sky that the masks fill from the prior)."""
    from gibbssampler_b200 import _dev
    from gibbssampler_b200.JointSampler import JointGibbs
    from gibbssampler_b200.sht import Plan
    nside, lmax = 16, 32
    npix = 12 * nside ** 2
    rng = np.random.default_rng(9)
    dls = T.spectra(lmax, te_frac=0.7)
    a, b, d, e = te_blocks(dls, lmax)
    lof = R.l_of_real_layout(lmax)
    chol = np.zeros((lmax + 1, 2, 2))
    for l in range(2, lmax + 1):
        chol[l] = np.linalg.cholesky([[a[l], b[l]], [b[l], d[l]]])
    z = rng.standard_normal(((lmax + 1) ** 2, 3))
    sT = chol[lof, 0, 0] * z[:, 0]
    sE = chol[lof, 1, 0] * z[:, 0] + chol[lof, 1, 1] * z[:, 1]
    sB = np.sqrt(e[lof]) * z[:, 2]
    fwhm = 1.0
    bl = _dev.gauss_beam(np.radians(fwhm), lmax)
    plan = Plan.get(nside, lmax)
    mI = host(plan.alm2map(dev(sT * bl[lof])))
    mQ, mU = (host(v) for v in plan.alm2map_spin2(dev(sE * bl[lof]), dev(sB * bl[lof])))
    nT, nP = 24.0, 0.5    # noise per a_lm about 1 % of C^TT_l and C^EE_l at l = 20
    data = {"I": mI + rng.standard_normal(npix) * np.sqrt(nT), "Q": mQ + rng.standard_normal(npix) * np.sqrt(nP),
            "U": mU + rng.standard_normal(npix) * np.sqrt(nP)}
    mask_T, mask_P = T.make_mask(nside, "galplane"), T.make_mask(nside, "band")
    init = {k: v.copy() for k, v in dls.items()}
    gs = JointGibbs(data, nT, nP, fwhm, nside, lmax, n_iter=150, mask=mask_T, mask_pol=mask_P, seed=3)
    gs.constrained_sampler.pcg_accuracy = 1e-6
    h = gs.run(init)
    for k in ("TT", "TE", "EE", "BB"):
        assert np.all(np.isfinite(h[k]))
    ell = np.arange(lmax + 1)
    c2d = ell * (ell + 1) / (2 * np.pi)
    for key, s in (("TT", sT), ("EE", sE)):
        chat = np.bincount(lof, weights=s ** 2, minlength=lmax + 1) / (2 * ell + 1) * c2d
        for l in (10, 20):
            expect = (2 * l + 1) * chat[l] / (2 * l - 5)
            got = h[key][30:, l].mean()
            assert abs(got - expect) < 0.35 * expect, (key, l, got, expect)
    chat_te = np.bincount(lof, weights=sT * sE, minlength=lmax + 1) / (2 * ell + 1) * c2d
    chat_tt = np.bincount(lof, weights=sT * sT, minlength=lmax + 1) / (2 * ell + 1) * c2d
    chat_ee = np.bincount(lof, weights=sE * sE, minlength=lmax + 1) / (2 * ell + 1) * c2d
    for l in (10, 20):
        scale = np.sqrt(chat_tt[l] * chat_ee[l])
        assert abs(h["TE"][30:, l].mean() - (2 * l + 1) * chat_te[l] / (2 * l - 5)) < 0.35 * scale, l


def test_bad_arguments_and_sharded_plans_are_refused():
    from gibbssampler_b200 import _lib
    from gibbssampler_b200._dev import ptr, stream
    from gibbssampler_b200.JointSampler import JointConstrainedRealization
    from gibbssampler_b200.sharded import ShardedPlan, run_local_group
    nside, lmax = 8, 16
    P = T.problem(nside, lmax, "galplane", "band", seed=16)
    dls = T.spectra(lmax)
    cr = sampler(P, nside, lmax, seed=5)
    L = _lib.lib()
    n = (lmax + 1) ** 2
    d = {k: dev(v) for k, v in dls.items()}
    v = [torch.zeros(n, dtype=torch.float64, device="cuda") for _ in range(6)]
    args = [ptr(d["TT"]), ptr(d["TE"]), ptr(d["EE"]), ptr(d["BB"]), ptr(cr.bl), ptr(cr.inv_noise_T), ptr(cr.inv_noise_P)]
    assert L.gs_cr_apply_q_teb(None, *args, *[ptr(x) for x in v], stream()) == -1
    assert b"null plan" in L.gs_last_error_string()
    bad = list(args)
    bad[1] = None
    assert L.gs_cr_apply_q_teb(cr.plan._h, *bad, *[ptr(x) for x in v], stream()) == -1
    nit, res = C.c_int(0), C.c_double(0.0)
    assert L.gs_cr_pcg_teb(cr.plan._h, *args, 1.0, 1.0, *[ptr(x) for x in v], 0, 0.0, 10, 8, C.byref(nit), C.byref(res),
                           stream()) == -1   # eps <= 0
    assert L.gs_cr_rhs_teb(cr.plan._h, *args[:6], ptr(cr.sqrt_inv_noise_T), ptr(cr.inv_noise_P), ptr(cr.sqrt_inv_noise_P),
                           None, None, None, None, None, None, *[ptr(x) for x in v], 3, *[ptr(x) for x in v[:3]], stream()) == -1
    assert b"data" in L.gs_last_error_string()
    plans = ShardedPlan.local_group(nside, lmax, 2)

    def work(p):
        codes = [L.gs_cr_apply_q_teb(p._h, *args, *[ptr(x) for x in v], stream()),
                 L.gs_cr_pcg_teb(p._h, *args, 1.0, 1.0, *[ptr(x) for x in v], 0, 1e-6, 10, 8, None, None, stream())]
        msg = L.gs_last_error_string()
        try:
            JointConstrainedRealization(P["d"], P["noise_T"], P["noise_P"], np.ones(lmax + 1), lmax, 12 * nside ** 2,
                                        mask=P["mask_T"], plan=p)
            codes.append(0)
        except _lib.GibbsB200Error:
            codes.append(-1)
        return codes, b"unsharded" in msg

    assert run_local_group(plans, work) == [([-1, -1, -1], True)] * 2
