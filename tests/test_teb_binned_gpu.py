"""Binned TT/TE/EE/BB spectra in the joint sampler: gs_cls_invwishart_binned against the per-l gs_cls_invwishart it reduces to,
against the oracle (tests.teb_binned_oracle) and in distribution; JointClsSampler(bins=) and JointGibbs(bins=) on a cut sky and on
the full sky."""
import numpy as np
import pytest
import torch

from oracle import reference_logic as R
from tests import teb_binned_oracle as B
from tests import teb_problem as T
from tests.teb_oracle import te_blocks

pytestmark = pytest.mark.gpu


def dev(x):
    return torch.as_tensor(np.ascontiguousarray(x, dtype=np.float64), device="cuda")


def host(x):
    return x.cpu().numpy() if isinstance(x, torch.Tensor) else np.asarray(x)


def spectra(lmax, seed=0):
    """per-l C_l (TT, TE, EE) with a TE correlation that changes sign"""
    rng = np.random.default_rng(seed)
    ell = np.arange(lmax + 1)
    tt = 2.0 / (ell + 10.0) ** 2 * (1 + 0.1 * rng.random(lmax + 1))
    ee = 0.5 / (ell + 10.0) ** 2 * (1 + 0.1 * rng.random(lmax + 1))
    te = 0.6 * np.sqrt(tt * ee) * np.cos(ell / 7.0)
    return tt, te, ee


def draw_binned(cl, edges, inject=None, seed=1, call=1):
    from gibbssampler_b200 import _lib
    from gibbssampler_b200._dev import i32, ptr, stream
    nb = len(edges) - 1
    lmax = len(cl[0]) - 1
    out = [torch.empty(nb, dtype=torch.float64, device="cuda") for _ in range(3)]
    cl_d, e_d = [dev(x) for x in cl], i32(edges)
    inj = dev(inject) if inject is not None else None
    _lib.check(_lib.lib().gs_cls_invwishart_binned(*[ptr(x) for x in cl_d], lmax, ptr(e_d), nb, ptr(inj), seed, call,
                                                   *[ptr(o) for o in out], stream()))
    return [host(o) for o in out]


def draw_per_l(cl, inject=None, seed=1, call=1):
    from gibbssampler_b200 import _lib
    from gibbssampler_b200._dev import ptr, stream
    lmax = len(cl[0]) - 1
    out = [torch.empty(lmax + 1, dtype=torch.float64, device="cuda") for _ in range(3)]
    cl_d = [dev(x) for x in cl]
    inj = dev(inject) if inject is not None else None
    _lib.check(_lib.lib().gs_cls_invwishart(*[ptr(x) for x in cl_d], lmax, ptr(inj), seed, call, *[ptr(o) for o in out], stream()))
    return [host(o) for o in out]


def assert_blocks_close(got, ref, rtol, first=2):
    """per bin, (TT, TE, EE) relative to the scale of the block"""
    for b in range(first, len(ref[0])):
        scale = max(abs(ref[0][b]), abs(ref[2][b]))
        for g, r in zip(got, ref):
            assert abs(g[b] - r[b]) <= rtol * scale, (b, g[b], r[b])


def test_one_l_bins_reduce_to_the_per_l_draw():
    lmax = 300
    cl = spectra(lmax)
    ell = np.arange(lmax + 1)
    c2d = ell * (ell + 1) / (2 * np.pi)
    edges = np.arange(lmax + 2)
    nu, _ = B.nu_psi(*cl, edges)
    inject = B.bartlett_draws(nu, np.random.default_rng(2), 1)[0]
    for kw in ({"inject": inject}, {"seed": 77, "call": 5}):
        per_l = [x * c2d for x in draw_per_l(cl, **kw)]
        binned = draw_binned(cl, edges, **kw)
        assert_blocks_close(binned, per_l, 1e-12)
        assert all(np.all(x[:2] == 0) for x in binned)


def test_injected_draws_on_uneven_bins_match_the_oracle():
    lmax = 1024
    cl = spectra(lmax, 3)
    edges = np.array([0, 1, 2, 3, 5, 9, 17, 30, 31, 60, 100, 250, 251, 400, 700, 825, lmax + 1])   # last bin: 200 multipoles
    nu, _ = B.nu_psi(*cl, edges)
    inject = B.bartlett_draws(nu, np.random.default_rng(4), 1)[0]
    got = draw_binned(cl, edges, inject=inject)
    ref = B.invwishart_bartlett_binned(*cl, edges, inject)
    assert_blocks_close(got, (ref[:, 0, 0], ref[:, 0, 1], ref[:, 1, 1]), 1e-11)
    assert all(np.all(x[:2] == 0) for x in got)


def test_bins_that_break_the_edge_conditions_come_out_nan():
    """The C ABI cannot check device edges on the host: the kernel marks every bin whose edges break the conditions with NaN and
    draws the others as usual."""
    lmax = 40
    cl = spectra(lmax, 7)
    good = np.array([0, 1, 2, 6, 15, lmax + 1])
    ref = draw_binned(cl, good, seed=3, call=9)
    cases = [
        (np.array([0, 2, 6, 15, lmax + 1]), [0, 1]),              # no l = 1 bin: bins 0 and 1 are not [0,1) and [1,2)
        (np.array([0, 1, 2, 6, 6, 15, lmax + 1]), [3]),           # an empty bin
        (np.array([0, 1, 2, 6, 15, lmax]), [4]),                  # last edge short of lmax + 1
        (np.array([0, 1, 2, 6, 15, lmax + 5]), [4]),              # last edge past lmax + 1
    ]
    for edges, bad in cases:
        got = draw_binned(cl, edges, seed=3, call=9)
        for b in range(len(edges) - 1):
            isnan = [bool(np.isnan(x[b])) for x in got]
            assert isnan == [b in bad] * 3, (edges, b, isnan)
    assert all(np.all(np.isfinite(x)) for x in ref) and all(np.all(x[:2] == 0) for x in ref)
    got = draw_binned(cl, np.array([0, 1, 2, 6, 6, 15, lmax + 1]), seed=3, call=9)   # bin 2 = [2, 6) is still draw 2
    assert all(g[2] == r[2] for g, r in zip(got, ref))


def test_philox_draws_have_the_inverse_wishart_moments():
    """4000 device draws (call = 1..4000) for fixed Chat on bins with nu from 12 to 2.4e5 (Marsaglia-Tsang up to shape 1.2e5): mean
    and variance of TT, TE and EE per bin within 5 standard errors (the sample variance's error from the fourth central moment)."""
    from gibbssampler_b200 import _lib
    from gibbssampler_b200._dev import i32, ptr, stream
    lmax, n = 520, 4000
    edges = np.array([0, 1, 2, 7, 8, 20, 25, 100, 110, 500, 510, lmax + 1])
    cl = spectra(lmax, 5)
    nu, psi = B.nu_psi(*cl, edges)
    nb = len(edges) - 1
    L = _lib.lib()
    cl_d, e_d = [dev(x) for x in cl], i32(edges)
    out = torch.empty(n, 3, nb, dtype=torch.float64, device="cuda")
    for k in range(n):
        _lib.check(L.gs_cls_invwishart_binned(*[ptr(x) for x in cl_d], lmax, ptr(e_d), nb, None, 2024, k + 1,
                                              *[ptr(out[k, i]) for i in range(3)], stream()))
    X = host(out)
    assert np.all(X[:, :, :2] == 0)
    X = np.moveaxis(X[:, :, 2:], 1, 2)      # (n, bin, entry)
    mean, var = B.iw_moments(nu[2:], psi[2:])
    m, v = X.mean(0), X.var(0, ddof=1)
    m4 = ((X - m) ** 4).mean(0)
    zm = np.abs(m - mean) / np.sqrt(var / n)
    zv = np.abs(v - var) / np.sqrt((m4 - v ** 2) / n)
    assert zm.max() < 5 and zv.max() < 5, (zm.max(), zv.max())


def test_binned_cls_sampler_draws_and_refusals():
    from gibbssampler_b200 import _lib
    from gibbssampler_b200._dev import i32, ptr, stream
    from gibbssampler_b200.JointSampler import JointClsSampler
    lmax = 64
    n = (lmax + 1) ** 2
    rng = np.random.default_rng(6)
    alms = {k: rng.standard_normal(n) for k in ("TT", "EE", "BB")}
    alms["EE"] = 0.5 * alms["TT"] + alms["EE"]
    alms_d = {k: dev(v) for k, v in alms.items()}
    tt_edges = np.concatenate([np.arange(0, 11), np.arange(15, lmax, 7), [lmax + 1]])
    bins = {"TT": tt_edges, "TE": tt_edges, "EE": tt_edges, "BB": np.array([0, 1, 2, 10, 30, lmax + 1])}
    nt, nb = len(bins["TT"]) - 1, len(bins["BB"]) - 1
    s = JointClsSampler(lmax, bins=bins, seed=5)
    out = s.sample(alms_d)
    assert [out[k].shape for k in ("TT", "TE", "EE", "BB")] == [(nt,)] * 3 + [(nb,)]
    # Philox: the sampler's two draws are the kernels' draws for its call indices
    ch = s.empirical(alms_d)
    L = _lib.lib()
    ref = [torch.empty(nt, dtype=torch.float64, device="cuda") for _ in range(3)]
    e_tt, e_bb = i32(bins["TT"]), i32(bins["BB"])
    _lib.check(L.gs_cls_invwishart_binned(ptr(ch["TT"]), ptr(ch["TE"]), ptr(ch["EE"]), lmax, ptr(e_tt), nt, None, 5, s._call,
                                          *[ptr(r) for r in ref], stream()))
    bb = torch.empty(nb, dtype=torch.float64, device="cuda")
    _lib.check(L.gs_cls_invgamma(ptr(ch["BB"]), ptr(e_bb), nb, None, 5, s._call + 1, ptr(bb), None, None, stream()))
    for k, r in zip(("TT", "TE", "EE", "BB"), ref + [bb]):
        assert np.array_equal(host(out[k]), host(r)), k
    # injected: TT/TE/EE against the oracle, BB against the reference's binned inverse-gamma (CenteredGibbs.py:54-79)
    nu, _ = B.nu_psi(*[host(ch[k]) for k in ("TT", "TE", "EE")], bins["TT"])
    inject = B.bartlett_draws(nu, rng, 1)[0]
    alpha, beta = R.cls_alpha_beta(alms["BB"], bins["BB"], lmax)
    gam = rng.gamma(alpha)
    out = s.sample(alms_d, inject=inject, gamma_inject=gam)
    iw = B.invwishart_bartlett_binned(*[host(ch[k]) for k in ("TT", "TE", "EE")], bins["TT"], inject)
    assert_blocks_close([host(out[k]) for k in ("TT", "TE", "EE")], (iw[:, 0, 0], iw[:, 0, 1], iw[:, 1, 1]), 1e-11)
    want = beta / gam
    want[:2] = 0
    assert np.allclose(host(out["BB"]), want, rtol=1e-12, atol=0)
    with pytest.raises(ValueError):
        s.sample(alms_d, inject=inject[:-1])
    with pytest.raises(ValueError):
        s.sample(alms_d, gamma_inject=gam[:-1])
    with pytest.raises(ValueError):
        JointClsSampler(lmax, bins={"TT": bins["TT"], "BB": bins["BB"][1:]})
    # the library refuses what it can check: null pointers and more bins than multipoles
    o = [torch.empty(lmax + 2, dtype=torch.float64, device="cuda") for _ in range(3)]
    e = i32(np.arange(lmax + 3))
    assert L.gs_cls_invwishart_binned(ptr(ch["TT"]), None, ptr(ch["EE"]), lmax, ptr(e), nt, None, 5, 1, *[ptr(x) for x in o],
                                      stream()) == -1
    assert L.gs_cls_invwishart_binned(ptr(ch["TT"]), ptr(ch["TE"]), ptr(ch["EE"]), lmax, ptr(e), lmax + 2, None, 5, 1,
                                      *[ptr(x) for x in o], stream()) == -1


def masked_sky(nside, lmax, seed):
    """high-S/N masked simulation (T: galplane, P: band) as in test_teb_masked_gpu: -> (data maps, noise, masks, sT, sE, init D_l)"""
    from gibbssampler_b200 import _dev
    from gibbssampler_b200.sht import Plan
    rng = np.random.default_rng(seed)
    npix = 12 * nside ** 2
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
    bl = _dev.gauss_beam(np.radians(1.0), lmax)
    plan = Plan.get(nside, lmax)
    mI = host(plan.alm2map(dev(sT * bl[lof])))
    mQ, mU = (host(v) for v in plan.alm2map_spin2(dev(sE * bl[lof]), dev(sB * bl[lof])))
    nT, nP = 24.0, 0.5
    data = {"I": mI + rng.standard_normal(npix) * np.sqrt(nT), "Q": mQ + rng.standard_normal(npix) * np.sqrt(nP),
            "U": mU + rng.standard_normal(npix) * np.sqrt(nP)}
    return data, (nT, nP), (T.make_mask(nside, "galplane"), T.make_mask(nside, "band")), sT, sE, dls


def test_masked_chain_with_one_l_bins_reproduces_the_per_l_chain():
    from gibbssampler_b200.JointSampler import JointGibbs
    nside, lmax = 16, 32
    data, (nT, nP), (mT, mP), _, _, dls = masked_sky(nside, lmax, 9)
    one = np.arange(lmax + 2)
    runs = []
    for bins in (None, {"TT": one, "BB": one}):
        gs = JointGibbs(data, nT, nP, 1.0, nside, lmax, n_iter=5, mask=mT, mask_pol=mP, bins=bins, seed=3)
        gs.constrained_sampler.pcg_accuracy = 1e-9
        cr, its = gs.constrained_sampler, []

        def counted(all_dls, xi=None, cr=cr, sample=cr.sample, its=its):   # records the PCG iterations of every CR step
            r = sample(all_dls, xi)
            its.append(cr.last_pcg_iterations)
            return r

        cr.sample = counted
        runs.append((gs.run({k: v.copy() for k, v in dls.items()}), its))
    (h0, it0), (h1, it1) = runs
    for k in ("TT", "TE", "EE", "BB"):
        assert h1[k].shape == h0[k].shape == (6, lmax + 1)
        assert np.abs(h1[k] - h0[k]).max() <= 1e-8 * np.abs(h0[k]).max(), k
    assert len(it0) == len(it1) == 5 and all(abs(x - y) <= 2 for x, y in zip(it0, it1)), (it0, it1)


def test_masked_chain_with_wide_bins_tracks_the_realised_binned_spectra():
    """150 iterations, TT/TE/EE bins of 4 multipoles and wide BB bins: with low noise s follows the input sky on the observed part,
    so the posterior mean of D_b stays within 35 % of Psi_b / (nu_b - 3) of the input sky (TE: of the TT/EE geometric mean)."""
    from gibbssampler_b200.JointSampler import JointGibbs
    nside, lmax = 16, 32
    data, (nT, nP), (mT, mP), sT, sE, dls = masked_sky(nside, lmax, 9)
    bins = {"TT": np.array([0, 1, 2, 4, 8, 12, 16, 20, 24, 28, lmax + 1]), "BB": np.array([0, 1, 2, 12, 22, lmax + 1])}
    init = {k: dls[k][bins["BB" if k == "BB" else "TT"][:-1]] for k in dls}
    gs = JointGibbs(data, nT, nP, 1.0, nside, lmax, n_iter=150, mask=mT, mask_pol=mP, bins=bins, seed=3)
    h = gs.run(init)
    assert [h[k].shape for k in ("TT", "TE", "EE", "BB")] == [(151, 10)] * 3 + [(151, 5)]
    for k in ("TT", "TE", "EE", "BB"):
        assert np.all(np.isfinite(h[k])) and np.all(h[k][1:, :2] == 0)
    assert np.all(h["BB"][1:, 2:] > 0)
    lof = R.l_of_real_layout(lmax)
    ell = np.arange(lmax + 1)
    chat = {k: np.bincount(lof, weights=x * y, minlength=lmax + 1) / (2 * ell + 1)
            for k, (x, y) in {"TT": (sT, sT), "TE": (sT, sE), "EE": (sE, sE)}.items()}
    nu, psi = B.nu_psi(chat["TT"], chat["TE"], chat["EE"], bins["TT"])
    for b in (4, 5, 6, 7):        # l = 8-11, 12-15, 16-19, 20-23
        expect = psi[b] / (nu[b] - 3)
        for key, (i, j) in (("TT", (0, 0)), ("EE", (1, 1))):
            got = h[key][30:, b].mean()
            assert abs(got - expect[i, j]) < 0.35 * expect[i, j], (key, b, got, expect[i, j])
        got = h["TE"][30:, b].mean()
        assert abs(got - expect[0, 1]) < 0.35 * np.sqrt(expect[0, 0] * expect[1, 1]), (b, got, expect[0, 1])


def test_full_sky_chain_with_bins_returns_binned_histories():
    """Harmonic data on the full sky: binned histories of the right shapes, and one-l bins reproduce the per-l chain."""
    from gibbssampler_b200 import _dev
    from gibbssampler_b200.JointSampler import JointGibbs
    lmax, nside = 32, 16
    npix = 12 * nside ** 2
    rng = np.random.default_rng(8)
    dls = T.spectra(lmax)
    a, b, d, e = te_blocks(dls, lmax)
    lof = R.l_of_real_layout(lmax)
    sd = np.sqrt(np.stack([a, d, e], 1))[lof]
    s_true = rng.standard_normal(((lmax + 1) ** 2, 3)) * sd
    bl = _dev.gauss_beam(np.radians(1.0), lmax)
    nt, npol = 1e-6, 1e-8
    nl = np.array([nt, npol, npol]) * 4 * np.pi / npix
    dat = s_true * bl[lof][:, None] + rng.standard_normal(s_true.shape) * np.sqrt(nl)[None, :]
    data = {"TT": dat[:, 0], "EE": dat[:, 1], "BB": dat[:, 2]}
    bins = {"TT": np.array([0, 1, 2, 5, 10, 20, lmax + 1]), "BB": np.array([0, 1, 2, 16, lmax + 1])}
    init = {k: dls[k][bins["BB" if k == "BB" else "TT"][:-1]] for k in dls}
    h = JointGibbs(data, nt, npol, 1.0, nside, lmax, n_iter=40, bins=bins, seed=2).run(init)
    assert [h[k].shape for k in ("TT", "TE", "EE", "BB")] == [(41, 6)] * 3 + [(41, 4)]
    assert all(np.all(np.isfinite(h[k])) for k in h) and np.all(h["TT"][1:, 2:] > 0) and np.all(h["BB"][1:, 2:] > 0)
    with pytest.raises(ValueError):
        JointGibbs(data, nt, npol, 1.0, nside, lmax, n_iter=1, bins=bins, seed=2).run(dls)     # unbinned start
    one = np.arange(lmax + 2)
    h0 = JointGibbs(data, nt, npol, 1.0, nside, lmax, n_iter=10, seed=4).run(dls)
    h1 = JointGibbs(data, nt, npol, 1.0, nside, lmax, n_iter=10, bins={"TT": one, "BB": one}, seed=4).run(dls)
    for k in ("TT", "TE", "EE", "BB"):
        assert np.abs(h1[k] - h0[k]).max() <= 1e-10 * np.abs(h0[k]).max(), k
