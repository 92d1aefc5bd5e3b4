"""GPU: the Blackwell-Rao estimator (csrc/blackwell_rao.cu, gibbssampler_b200.BlackwellRao) against the numpy oracle
(tests/br_oracle.py), keep_sigma recording in CenteredGibbs / JointGibbs, and known answers on the full sky."""
import numpy as np
import pytest
import torch

from oracle import reference_logic as R
from tests import br_oracle as O
from tests.test_br_oracle import _joint_models, _joint_sigma

pytestmark = pytest.mark.gpu


def _lib():
    from gibbssampler_b200 import _lib
    return _lib


def test_sample_features_match_the_cl_kernels():
    """beta rows equal gs_cls_invgamma's beta_out bit for bit, alpha log beta uses its alpha_out; Psi equals the oracle."""
    from gibbssampler_b200 import _dev
    from gibbssampler_b200._dev import f64, i32, ptr, stream
    L = _lib().lib()
    rng = np.random.default_rng(4)
    lmax, n = 40, 37
    sig = _joint_sigma(rng, n, lmax)
    edges = np.array([0, 1, 2, 3, 7, 12, 20, 33, lmax + 1])
    nb = len(edges) - 1
    e_dev = i32(edges[2:])
    s = f64(sig["BB"])
    S = torch.empty((nb - 2, n), dtype=torch.float64, device="cuda")
    c = torch.empty(n, dtype=torch.float64, device="cuda")
    scr = torch.empty((nb - 2) * n, dtype=torch.float64, device="cuda")
    _lib().check(L.gs_br_sample_features(0, ptr(s), None, None, n, lmax + 1, ptr(e_dev), nb - 2, ptr(S), ptr(c), 0, ptr(scr), stream()))
    alpha = torch.empty(nb, dtype=torch.float64, device="cuda")
    beta = torch.empty(nb, dtype=torch.float64, device="cuda")
    out = torch.empty(nb, dtype=torch.float64, device="cuda")
    for i in range(n):
        _lib().check(L.gs_cls_invgamma(ptr(s[i]), ptr(i32(edges)), nb, None, 1, 1, ptr(out), ptr(alpha), ptr(beta), stream()))
        assert torch.equal(S[:, i], beta[2:])
        want = float((alpha[2:] * torch.log(beta[2:])).sum())
        assert abs(float(c[i]) - want) <= 1e-14 * abs(want)
    # inverse-Wishart rows against the oracle
    tt, te, ee = (f64(sig[k]) for k in ("TT", "TE", "EE"))
    S3 = torch.empty((3 * (nb - 2), n), dtype=torch.float64, device="cuda")
    _lib().check(L.gs_br_sample_features(1, ptr(tt), ptr(te), ptr(ee), n, lmax + 1, ptr(e_dev), nb - 2, ptr(S3), ptr(c), 0, ptr(scr), stream()))
    nu, psi = O.iw_nu_psi(sig["TT"], sig["TE"], sig["EE"], edges[2:])
    got = S3.cpu().numpy().T.reshape(n, nb - 2, 3)
    assert np.abs(got - psi).max() <= 1e-14 * np.abs(psi).max()
    want_c = (0.5 * nu * np.log(psi[..., 0] * psi[..., 2] - psi[..., 1] ** 2)).sum(1)
    assert np.allclose(c.cpu().numpy(), want_c, rtol=1e-13, atol=0)
    # a broken bin (empty) comes out NaN, its neighbours do not
    bad = i32(np.array([2, 5, 5, 9]))
    _lib().check(L.gs_br_sample_features(0, ptr(s), None, None, n, lmax + 1, ptr(bad), 3, ptr(S), ptr(c), 0, ptr(scr), stream()))
    Sh = S.cpu().numpy()
    assert np.all(np.isnan(Sh[1])) and np.all(np.isfinite(Sh[0])) and np.all(np.isfinite(Sh[2])) and np.all(np.isnan(c.cpu().numpy()))
    # ... and a NaN log-density reaches the estimate as NaN (not -inf), for the narrow and the wide tile
    for m in (1, 100):
        W = torch.zeros((3, m), dtype=torch.float64, device="cuda")
        e = torch.zeros(m, dtype=torch.float64, device="cuda")
        scr2 = torch.empty(int(L.gs_br_logmeanexp_scratch(n, m)), dtype=torch.float64, device="cuda")
        logl, neff = (torch.empty(m, dtype=torch.float64, device="cuda") for _ in range(2))
        _lib().check(L.gs_br_logmeanexp(ptr(S), ptr(c), n, ptr(W), ptr(e), m, 3, ptr(scr2), ptr(logl), ptr(neff), stream()))
        assert torch.isnan(logl).all() and torch.isnan(neff).all(), m


def _oracle_edges(br):
    return {k: br.edges[k][2:] for k in br.keys}


def _near_models(br, sig, m, rng):
    """m models scattered by 5 % around the sample-mean conditional mode of every bin (columns 0 and 1: 1, not evaluated), so
    that log L stays within the range a user evaluates and every model is valid"""
    out = {}
    for kind, keys in br.groups:
        e = br.edges[keys[0]][2:]
        if kind == 0:
            a, be = O.ig_alpha_beta(sig[keys[0]], e)
            base = {keys[0]: be.mean(0) / (a + 1)}
        else:
            nu, psi = O.iw_nu_psi(sig["TT"], sig["TE"], sig["EE"], e)
            mode = psi.mean(0) / (nu + 3)[:, None]
            base = {"TT": mode[:, 0], "TE": 0.8 * mode[:, 1], "EE": mode[:, 2]}
        for k, v in base.items():
            out[k] = np.concatenate([np.ones((m, 2)), v[None, :] * (1 + 0.05 * rng.standard_normal((m, len(v))))], axis=1)
    return out


def _tolerance(sig, edges, dls):
    """1e-9 absolute, or 2e-14 of the largest term of the decomposition c + S^T W + e where those terms reach beyond 5e4: the sum of
    FP64 terms of magnitude T carries rounding of order eps T whatever the order of summation"""
    S, c, groups = O.features(sig, edges)
    W, e = O.model_features(dls, groups)
    return max(1e-9, 2e-14 * (np.abs(c).max() + np.abs(e[np.isfinite(e)]).max(initial=0.0)))


@pytest.mark.parametrize("n", [1, 999, 4097])
@pytest.mark.parametrize("m", [1, 17, 257, 1000])
@pytest.mark.parametrize("layout", ["tt_one_bin", "ee_bb", "joint_planck"])
def test_logpdf_matches_the_oracle(n, m, layout):
    from gibbssampler_b200.BlackwellRao import BlackwellRao
    rng = np.random.default_rng(n + 7 * m)
    if layout == "tt_one_bin":
        lmax = 12
        sig = {"TT": _joint_sigma(rng, n, lmax)["TT"]}
        bins = np.array([0, 1, 2, lmax + 1])
    elif layout == "ee_bb":
        lmax = 60
        s = _joint_sigma(rng, n, lmax)
        sig = {"EE": s["EE"], "BB": s["BB"]}
        bins = {"EE": np.arange(lmax + 2), "BB": np.array([0, 1, 2, 5, 11, 30, 44, lmax + 1])}
    else:
        lmax = 300 if n > 1000 else 1024 if n == 1 else 500
        sig = _joint_sigma(rng, n, lmax)
        tt = np.concatenate([np.arange(0, 31), np.arange(31, lmax + 1, 10)[1:], [lmax + 1]])
        import bench
        bins = {"TT": np.unique(tt), "BB": bench.bins_for(lmax)["BB"]}
    br = BlackwellRao(sig, bins)
    dls = _near_models(br, sig, m, rng)
    if m > 2:
        for k in dls:
            dls[k][1, -1] = -1.0 if k != "TE" else dls[k][1, -1]      # invalid model: D <= 0
    got, neff = br.logpdf(dls, n_eff=True)
    want, wneff = O.logpdf(sig, _oracle_edges(br), {k: v[:, 2:] for k, v in dls.items()})
    fin = np.isfinite(want)
    assert fin.sum() == m - (m > 2)
    assert np.array_equal(np.isfinite(got), fin) and np.all(got[~fin] == -np.inf) and np.all(neff[~fin] == 0)
    tol = _tolerance(sig, _oracle_edges(br), {k: v[:, 2:] for k, v in dls.items()})
    assert np.abs(got[fin] - want[fin]).max() <= tol, (np.abs(got[fin] - want[fin]).max(), tol, np.abs(want[fin]).max())
    assert np.allclose(neff[fin], wneff[fin], rtol=1e-6, atol=0)
    again, neff2 = br.logpdf(dls, n_eff=True)
    assert np.array_equal(got, again) and np.array_equal(neff, neff2)        # bitwise repeatable
    t = br.logpdf({k: torch.as_tensor(v, device="cuda") for k, v in dls.items()})
    assert isinstance(t, torch.Tensor) and t.is_cuda and np.array_equal(t.cpu().numpy(), got)
    one = br.logpdf({k: v[0] for k, v in dls.items()})
    assert np.ndim(one) == 0 and abs(one - got[0]) <= tol


def test_lrange_and_marginal():
    from gibbssampler_b200.BlackwellRao import BlackwellRao
    rng = np.random.default_rng(5)
    lmax, n = 40, 3000
    sig = _joint_sigma(rng, n, lmax)
    bins = {"TT": np.concatenate([np.arange(0, 11), np.arange(12, lmax + 1, 4), [lmax + 1]]),
            "BB": np.array([0, 1, 2, 10, 20, 30, lmax + 1])}
    br = BlackwellRao(sig, bins, burn_in=0)
    dls = _joint_models(rng, 9, len(bins["TT"]) - 1, len(bins["BB"]) - 1)
    got = br.logpdf(dls, lrange=(2, 19))     # TT bins 2..9 (l 2..9) + [10, 11] + [12, 15] + [16, 19]; BB bin [2, 9] + [10, 19]
    e = {"TT": np.array([2, 3, 4, 5, 6, 7, 8, 9, 10, 12, 16, 20]), "BB": np.array([2, 10, 20])}
    sub = {k: dls[k][:, 2:13] if k != "BB" else dls[k][:, 2:4] for k in dls}
    want, _ = O.logpdf(sig, e, sub)
    assert np.abs(got - want).max() <= _tolerance(sig, e, sub)
    with pytest.raises(ValueError, match="cuts bin"):
        br.logpdf(dls, lrange=(2, 14))
    with pytest.raises(ValueError):
        br.logpdf({k: v[:, :-1] for k, v in dls.items()})
    with pytest.raises(ValueError):
        br.marginal("TE", np.linspace(1, 2, 5))
    # marginals: BB (inverse-gamma) and EE (diagonal of the inverse-Wishart), per-bin grids
    nbb, nt = len(bins["BB"]) - 1, len(bins["TT"]) - 1
    grid = np.linspace(0.05, 3.0, 300)[None, :] * np.ones((nbb, 1))
    mb = br.marginal("BB", grid)
    assert mb.shape == (nbb, 300) and np.all(np.isnan(mb[:2]))
    a, be = O.ig_alpha_beta(sig["BB"], bins["BB"][2:])
    for b in range(2, nbb):
        assert np.allclose(mb[b], O.marginal_ig(a[b - 2], be[:, b - 2], grid[b]), rtol=0, atol=1e-10)
    g = np.linspace(0.5, 20.0, 257)
    me = br.marginal("EE", torch.as_tensor(g, device="cuda"))
    assert isinstance(me, torch.Tensor) and me.shape == (nt, 257)
    nu, psi = O.iw_nu_psi(sig["TT"], sig["TE"], sig["EE"], bins["TT"][2:])
    for b in range(2, nt):
        want = O.marginal_ig(0.5 * (nu[b - 2] - 1), 0.5 * psi[:, b - 2, 2], g)
        assert np.allclose(me[b].cpu().numpy(), want, rtol=0, atol=1e-10)


# ---------------------------------------------------------------------------------------------------------- recording
def _pol_masked(seed=0):
    nside, lmax = 8, 16
    npix = 12 * nside ** 2
    rng = np.random.default_rng(seed)
    import bench
    mask = bench.make_mask(nside, 0.8, "band")
    noise = np.full(npix, 0.05)
    d = {"Q": rng.standard_normal(npix) * mask, "U": rng.standard_normal(npix) * mask}
    return nside, lmax, npix, mask, noise, d


def test_centered_pol_recording_is_the_sky_behind_the_next_row():
    from gibbssampler_b200 import _dev
    from gibbssampler_b200.CenteredGibbs import CenteredGibbs
    nside, lmax, npix, mask, noise, d = _pol_masked()
    bins = {"EE": np.arange(lmax + 2), "BB": np.array([0, 1, 2, 6, 11, lmax + 1])}
    init = {"EE": np.where(np.arange(lmax + 1) >= 2, 1.0, 0.0), "BB": np.array([0, 0, 0.3, 0.3, 0.3])}
    mk = lambda ks: CenteredGibbs(d, 1.0, noise, 5.0, nside, lmax, npix, mask=mask, polarization=True, bins=bins, n_iter=6, seed=21,
                                  keep_sigma=ks)
    h0 = mk(False).run(init)[0]
    g = mk(True)
    h1 = g.run(init)[0]
    assert all(np.array_equal(h0[k], h1[k]) for k in ("EE", "BB"))
    assert set(g.sigma_history) == {"EE", "BB"} and g.sigma_history["EE"].shape == (6, lmax + 1)
    # the same chain by hand
    g2 = mk(False)
    cs, cl = g2.constrained_sampler, g2.cls_sampler
    binned = {k: _dev.f64(v) for k, v in init.items()}
    un = {k: g2._unfold(binned, k) for k in ("EE", "BB")}
    sky, _ = cs.sample(un)
    for i in range(6):
        sky, _ = cs.sample(dict(un), sky)
        for k in ("EE", "BB"):
            assert np.array_equal(cl._alm2cl_real(_dev.f64(sky[k])).cpu().numpy(), g.sigma_history[k][i]), (i, k)
        binned = cl.sample(dict(sky))
        un = {k: g2._unfold(binned, k) for k in ("EE", "BB")}
        for k in ("EE", "BB"):
            assert np.array_equal(binned[k].cpu().numpy(), h1[k][i + 1]), (i, k)
    from gibbssampler_b200.BlackwellRao import BlackwellRao
    br = BlackwellRao.from_sampler(g, burn_in=1)
    assert br.n == 5 and br.keys == ("EE", "BB")


def test_centered_tt_recording_is_the_sky_behind_the_next_row():
    from gibbssampler_b200 import _dev
    from gibbssampler_b200.CenteredGibbs import CenteredGibbs
    nside, lmax, npix, mask, noise, d = _pol_masked(1)
    mk = lambda ks: CenteredGibbs(d["Q"], np.full(npix, 0.05), None, 5.0, nside, lmax, npix, mask=mask, n_iter=5, seed=8, keep_sigma=ks)
    init = np.where(np.arange(lmax + 1) >= 2, 1.0, 0.0)
    h0 = mk(False).run(init)[0]
    g = mk(True)
    h1 = g.run(init)[0]
    assert np.array_equal(h0, h1) and g.sigma_history["TT"].shape == (5, lmax + 1)
    g2 = mk(False)
    cs, cl = g2.constrained_sampler, g2.cls_sampler
    binned = _dev.f64(init)
    cls, var = g2._tt_state(binned)
    sky, _ = cs.sample(cls, var, None, metropolis_step=False)
    for i in range(5):
        sky, _ = cs.sample(cls, var, sky, metropolis_step=False, use_gibbs=False)
        assert np.array_equal(cl._alm2cl_real(_dev.f64(sky)).cpu().numpy(), g.sigma_history["TT"][i]), i
        binned = cl.sample(sky)
        cls, var = g2._tt_state(binned)
        assert np.array_equal(_dev.to_host(binned), h1[i + 1]), i


@pytest.mark.parametrize("sky", ["full", "cut"])
@pytest.mark.parametrize("binned", [False, True])
def test_joint_recording_is_the_sky_behind_the_next_row(sky, binned):
    from gibbssampler_b200.JointSampler import JointGibbs
    lmax, nside = 16, 8
    if sky == "cut":
        from tests.test_teb_binned_gpu import masked_sky
        data, (nT, nP), (mT, mP), _, _, dls = masked_sky(nside, lmax, 9)
        kw = dict(mask=mT, mask_pol=mP)
    else:
        from tests import teb_problem as T
        rng = np.random.default_rng(3)
        dls = T.spectra(lmax)
        n = (lmax + 1) ** 2
        data = {k: rng.standard_normal(n) for k in ("TT", "EE", "BB")}
        nT, nP, kw = 1e-3, 1e-4, {}
    bins = {"TT": np.array([0, 1, 2, 4, 9, lmax + 1]), "BB": np.array([0, 1, 2, 8, lmax + 1])} if binned else None
    init = {k: dls[k][bins["BB" if k == "BB" else "TT"][:-1]] for k in dls} if binned else dls
    mk = lambda ks: JointGibbs(data, nT, nP, 1.0, nside, lmax, n_iter=4, bins=bins, seed=6, keep_sigma=ks, **kw)
    h0 = mk(False).run({k: v.copy() for k, v in init.items()})
    g = mk(True)
    h1 = g.run({k: v.copy() for k, v in init.items()})
    assert all(np.array_equal(h0[k], h1[k]) for k in h0)
    assert set(g.sigma_history) == {"TT", "TE", "EE", "BB"}
    g2 = mk(False)
    from gibbssampler_b200._dev import f64
    cur = {k: f64(v) for k, v in init.items()}
    for i in range(4):
        s, _ = g2.constrained_sampler.sample(g2._unfold(cur))
        emp = g2.cls_sampler.empirical(s)
        for k in ("TT", "TE", "EE", "BB"):
            assert np.array_equal(emp[k].cpu().numpy(), g.sigma_history[k][i]), (i, k)
        cur = g2.cls_sampler.sample(s)
        for k in cur:
            assert np.array_equal(cur[k].cpu().numpy(), h1[k][i + 1]), (i, k)


def test_keep_sigma_refusals():
    from gibbssampler_b200 import GibbsB200Error
    from gibbssampler_b200.BlackwellRao import BlackwellRao
    from gibbssampler_b200.CenteredGibbs import CenteredGibbs
    nside, lmax, npix, mask, noise, d = _pol_masked()
    g = CenteredGibbs(d, 1.0, noise, 5.0, nside, lmax, npix, polarization=True, n_iter=2, seed=1, keep_sigma=True)
    with pytest.raises(GibbsB200Error, match="keep_sigma"):
        g.run_fused({"EE": np.ones(lmax - 1), "BB": np.ones(lmax - 1)})
    with pytest.raises(ValueError, match="keep_sigma"):
        BlackwellRao.from_sampler(CenteredGibbs(d, 1.0, noise, 5.0, nside, lmax, npix, polarization=True, n_iter=2, seed=1))


# ---------------------------------------------------------------------------------------------------------- known answers
def _harmonic_data(rng, lmax, nside, fwhm, cov, noise):
    """full-sky harmonic data d = b s + n in the real layout; cov (L+1, p, p) per-l signal covariance (C units), noise (p,) per-pixel
    variances -> (d (n, p), N_l (p,) = 4 pi noise / Npix)"""
    npix = 12 * nside ** 2
    lof = R.l_of_real_layout(lmax)
    p = cov.shape[1]
    chol = np.zeros_like(cov)
    for l in range(2, lmax + 1):
        chol[l] = np.linalg.cholesky(cov[l])
    z = rng.standard_normal(((lmax + 1) ** 2, p))
    s = np.einsum("nij,nj->ni", chol[lof], z)
    bl = np.exp(-0.5 * np.arange(lmax + 1) * (np.arange(lmax + 1) + 1) * (np.radians(fwhm) / np.sqrt(8 * np.log(2))) ** 2)
    nl = 4 * np.pi * np.asarray(noise) / npix
    d = s * bl[lof][:, None] + rng.standard_normal(s.shape) * np.sqrt(nl)[None, :]
    d[lof < 2] = 0.0
    return d, nl, bl


@pytest.mark.slow
def test_ee_marginal_matches_the_exact_posterior():
    """Full sky, isotropic noise, harmonic data: the exact posterior of D_l with a flat prior is
        p(D) ~ exp(-(2l+1)/2 [Chat_d / (b^2 C + N) + log(b^2 C + N)]),  C = 2 pi D / (l (l+1)).
    High S/N (N << b^2 C) makes the centred chain mix in a few iterations.  Both densities are compared on the same finite grid
    (30 times the fiducial D; the l = 2 posterior has no second moment).  Monte-Carlo error: batch means over 20 batches of the
    chain, which accounts for its autocorrelation; 4 standard errors.  CDF: the BR marginal averages the per-sample
    inverse-gamma CDFs; 0.02 is several times the batch-mean spread of that average at 3000 samples."""
    from gibbssampler_b200.BlackwellRao import BlackwellRao
    from gibbssampler_b200.CenteredGibbs import CenteredGibbs
    nside, lmax, fwhm, noise0 = 8, 16, 5.0, 1e-4
    npix = 12 * nside ** 2
    rng = np.random.default_rng(17)
    ell = np.arange(lmax + 1)
    dl_true = np.where(ell >= 2, 1.0, 0.0)
    cl_true = np.where(ell >= 2, 2 * np.pi / np.maximum(ell * (ell + 1), 1), 0.0)
    d, nl, bl = _harmonic_data(rng, lmax, nside, fwhm, cl_true[:, None, None] * np.ones((1, 2, 2)) * np.eye(2), [noise0, noise0])
    pix_map = {"EE": d[:, 0], "BB": d[:, 1], "Q": np.zeros(npix), "U": np.zeros(npix)}
    bins = {"EE": np.arange(lmax + 2), "BB": np.arange(lmax + 2)}
    n_iter = 3000
    g = CenteredGibbs(pix_map, np.full(npix, 1.0), np.full(npix, noise0), fwhm, nside, lmax, npix, polarization=True, bins=bins,
                      n_iter=n_iter, seed=5, keep_sigma=True)
    g.run({"EE": dl_true.copy(), "BB": dl_true.copy()})
    burn = 100
    br = BlackwellRao.from_sampler(g, burn_in=burn)
    lof = R.l_of_real_layout(lmax)
    chat = np.bincount(lof, weights=d[:, 0] ** 2, minlength=lmax + 1) / (2 * ell + 1)
    sig = g.sigma_history["EE"][burn:]
    for l in (2, 5, 10):
        grid = np.linspace(1e-4, 30.0, 6000)
        dx = grid[1] - grid[0]
        lm = br.marginal("EE", grid)[l]
        p_br = np.exp(lm)
        v = bl[l] ** 2 * grid * 2 * np.pi / (l * (l + 1)) + nl[0]
        le = -(2 * l + 1) / 2 * (chat[l] / v + np.log(v))
        p_ex = np.exp(le - le.max())
        p_ex /= p_ex.sum() * dx

        def moments(p):
            w = p / p.sum()
            mu = (w * grid).sum()
            return mu, np.sqrt((w * (grid - mu) ** 2).sum()), np.cumsum(w)
        mb, sb, cb = moments(p_br)
        me, se, ce = moments(p_ex)
        # batch means of the BR marginal's moments
        a, be = O.ig_alpha_beta(sig, np.array([l, l + 1]))
        bm, bs = [], []
        for part in np.array_split(np.arange(len(sig)), 20):
            pb = np.exp(O.marginal_ig(a[0], be[part, 0], grid))
            m_, s_, _ = moments(pb)
            bm.append(m_)
            bs.append(s_)
        em, es = np.std(bm) / np.sqrt(20), np.std(bs) / np.sqrt(20)
        assert abs(mb - me) < 4 * em, (l, mb, me, em)
        assert abs(sb - se) < 4 * es, (l, sb, se, es)
        assert np.abs(cb - ce).max() < 0.02, (l, np.abs(cb - ce).max())


@pytest.mark.slow
def test_joint_likelihood_differences_match_the_exact_likelihood():
    """Full sky, isotropic noise, harmonic data, per-l JointGibbs to lmax = 6: the exact log-likelihood is
        sum_l -(2l+1)/2 [tr(Chat_d M_l^-1) + log|M_l|],  M_l = b_l^2 C_l + N,  N = diag(4 pi n_X / Npix),
    with the 3x3 (TT, TE, EE; BB) C_l.  Flat priors on D: log L_BR(theta_k) - log L_BR(theta_0) estimates the exact difference.
    20 models within Delta log L > -10 of the peak; high S/N keeps the chain mixing fast and the BR sum well sampled at l <= 6
    (n_eff in the hundreds at 4000 samples), so its Monte-Carlo error is a few hundredths; tolerance 0.1."""
    from gibbssampler_b200.BlackwellRao import BlackwellRao
    from gibbssampler_b200.JointSampler import JointGibbs
    from tests import teb_problem as T
    nside, lmax, fwhm = 4, 6, 10.0
    npix = 12 * nside ** 2
    rng = np.random.default_rng(23)
    dls = T.spectra(lmax, te_frac=0.6)
    ell = np.arange(lmax + 1)
    f = np.where(ell >= 2, 2 * np.pi / np.maximum(ell * (ell + 1), 1), 0.0)
    cov = np.zeros((lmax + 1, 3, 3))
    cov[:, 0, 0], cov[:, 1, 1], cov[:, 2, 2] = dls["TT"] * f, dls["EE"] * f, dls["BB"] * f
    cov[:, 0, 1] = cov[:, 1, 0] = dls["TE"] * f
    cov[:2] = np.eye(3)
    nT, nP = 1e-3, 1e-4
    d, nl, bl = _harmonic_data(rng, lmax, nside, fwhm, cov, [nT, nP, nP])
    data = {"TT": d[:, 0], "EE": d[:, 1], "BB": d[:, 2]}
    g = JointGibbs(data, nT, nP, fwhm, nside, lmax, n_iter=4000, seed=9, keep_sigma=True)
    g.run(dls)
    br = BlackwellRao.from_sampler(g, burn_in=100)
    lof = R.l_of_real_layout(lmax)
    chat = np.zeros((lmax + 1, 3, 3))
    for i in range(3):
        for j in range(3):
            chat[:, i, j] = np.bincount(lof, weights=d[:, i] * d[:, j], minlength=lmax + 1) / (2 * ell + 1)

    def exact(th):
        out = 0.0
        for l in range(2, lmax + 1):
            C = np.zeros((3, 3))
            C[0, 0], C[1, 1], C[2, 2] = th["TT"][l] * f[l], th["EE"][l] * f[l], th["BB"][l] * f[l]
            C[0, 1] = C[1, 0] = th["TE"][l] * f[l]
            M = bl[l] ** 2 * C + np.diag(nl)
            out += -(2 * l + 1) / 2 * (np.trace(chat[l] @ np.linalg.inv(M)) + np.linalg.slogdet(M)[1])
        return out
    # theta_0: the deconvolved data spectra (near the peak)
    th0 = {"TT": (chat[:, 0, 0] - nl[0]) / bl ** 2 / np.maximum(f, 1e-300), "EE": (chat[:, 1, 1] - nl[1]) / bl ** 2 / np.maximum(f, 1e-300),
           "BB": (chat[:, 2, 2] - nl[2]) / bl ** 2 / np.maximum(f, 1e-300), "TE": chat[:, 0, 1] / bl ** 2 / np.maximum(f, 1e-300)}
    for k in th0:
        th0[k][:2] = 0.0
    models, deltas = [th0], []
    e0 = exact(th0)
    while len(models) < 21:
        th = {k: v * (1 + 0.08 * rng.standard_normal(lmax + 1)) for k, v in th0.items()}
        pd = all(th["TT"][l] * th["EE"][l] > th["TE"][l] ** 2 and th["TT"][l] > 0 and th["BB"][l] > 0 for l in range(2, lmax + 1))
        dlt = exact(th) - e0 if pd else -np.inf
        if dlt > -10:
            models.append(th)
            deltas.append(dlt)
    M = {k: np.stack([m[k] for m in models]) for k in th0}
    got = br.logpdf(M, lrange=(2, lmax))
    assert np.all(np.isfinite(got))
    diff = got[1:] - got[0]
    assert np.abs(diff - np.array(deltas)).max() < 0.1, np.c_[diff, deltas]
