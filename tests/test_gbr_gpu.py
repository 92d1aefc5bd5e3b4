"""GPU: the Gaussianized Blackwell-Rao transform (gs_gbr_transform, csrc/blackwell_rao.cu) and GaussianizedBlackwellRao against
the numpy / scipy oracle (tests/gbr_oracle.py) and high-precision references, chain plumbing, and a known answer on the full sky."""
import numpy as np
import pytest
import torch
from scipy.special import gammaln, ndtr, ndtri
from scipy.stats import norm

from oracle import reference_logic as R
from tests import br_oracle as O
from tests import gbr_oracle as G
from tests.test_br_oracle import _joint_sigma
from tests.test_br_gpu import _harmonic_data

pytestmark = pytest.mark.gpu


def _transform(kind, S, ncl, edges, comp, dl):
    """one gs_gbr_transform call: S (rows, N), edges (nbins + 1,), dl (M, nbins) -> host (x, logm)"""
    from gibbssampler_b200 import _lib
    from gibbssampler_b200._dev import f64, i32, ptr, stream
    L = _lib.lib()
    S, dl, e = f64(S), f64(dl), i32(edges)
    n, (m, nb) = S.shape[1], dl.shape
    x, lm = (torch.empty((m, nb), dtype=torch.float64, device="cuda") for _ in range(2))
    scr = torch.empty(int(L.gs_gbr_transform_scratch(n, m, nb)), dtype=torch.float64, device="cuda")
    _lib.check(L.gs_gbr_transform(kind, ptr(S), n, ncl, ptr(e), nb, comp, ptr(dl), m, ptr(x), ptr(lm), ptr(scr), stream()))
    return x.cpu().numpy(), lm.cpu().numpy()


def test_incomplete_gamma_sweep():
    """One sample (beta = 1) of one-multipole bins l = alpha + 1/2 for alpha from 1.5 to 49999.5 and t / alpha from 0.02 to 50.
    The reference is mpmath at 30 digits: scipy's gammaincc itself is off by up to 1e-11 relative near alpha = 5000, t / alpha = 1.5.
    Wherever the smaller tail is >= 1e-300 it must match to 1e-12 relative.  x is compared through that tail: an error dx moves
    Phi(-|x|) by a factor exp(h dx), h = phi(x) / Phi(-|x|), so |dx| h <= 1e-12 plus eight ulps of x for the rounding of Phi^-1
    itself.  logm (the IG log-density) to 1e-13 of max(1, |logm|): the large-alpha form has no cancellation."""
    import mpmath as mp
    mp.mp.dps = 50
    r = np.unique(np.concatenate([np.geomspace(0.02, 50, 97), np.linspace(0.8, 1.25, 64)]))
    for a in (1.5, 2.5, 7.5, 49.5, 499.5, 4999.5, 49999.5):
        l = int(a + 0.5)
        t = a * r
        x, lm = _transform(0, np.ones((1, 1)), l + 1, [l, l + 1], 0, (1.0 / t)[:, None])
        x, lm = x[:, 0], lm[:, 0]
        lp = np.array([float(a * mp.log(ti) - ti - mp.loggamma(a) + mp.log(ti)) for ti in t])
        out = np.isinf(x)                # F or 1 - F is 0 in FP64: the model lies beyond what the transform represents
        assert np.all(lm[out] == -np.inf) and np.all(lp[out] < -700), a
        assert np.all(np.abs(lm - lp)[~out] <= 1e-13 * np.maximum(1.0, np.abs(lp[~out]))), (a, np.abs(lm - lp)[~out].max())
        checked = 0
        for i in range(len(t)):
            if lp[i] < -700:            # tail < 1e-300: only its sign and the order of magnitude matter
                assert np.isinf(x[i]) or abs(x[i]) > 35, (a, r[i], x[i])
                continue
            q = mp.gammainc(a, t[i], mp.inf, regularized=True)
            small = q if q <= 0.5 else mp.gammainc(a, 0, t[i], regularized=True)      # never 1 - q: it loses the digits
            if small < mp.mpf("1e-300"):
                continue
            xr = mp.mpf(float(ndtri(float(small))))           # Phi^-1(small) by Newton steps in 50 digits
            for _ in range(4):
                xr -= (mp.ncdf(xr) - small) / mp.npdf(xr)
            xr = float(xr) if q <= 0.5 else -float(xr)
            h = norm.pdf(xr) / ndtr(-abs(xr))
            assert abs(x[i] - xr) * h <= 1e-12 + 8 * 2.2e-16 * abs(xr) * h, (a, r[i], x[i], xr, float(small))
            checked += 1
        assert checked > 25, a


@pytest.mark.parametrize("n", [1, 300, 4097])
@pytest.mark.parametrize("m", [1, 33, 700])
@pytest.mark.parametrize("kind_comp", [(0, 0), (1, 0), (1, 2)])
def test_transform_matches_the_oracle(n, m, kind_comp):
    kind, comp = kind_comp
    rng = np.random.default_rng(n + 11 * m + 101 * kind + comp)
    lmax = 40
    sig = _joint_sigma(rng, n, lmax)
    edges = np.array([2, 3, 5, 9, 16, 28, lmax + 1])
    nb = len(edges) - 1
    if kind == 0:
        a, be = O.ig_alpha_beta(sig["BB"], edges)
        S, pars = be.T, [(a[b], be[:, b]) for b in range(nb)]
    else:
        nu, psi = O.iw_nu_psi(sig["TT"], sig["TE"], sig["EE"], edges)
        S = psi.transpose(1, 2, 0).reshape(3 * nb, n)
        pars = [(0.5 * (nu[b] - 1), 0.5 * psi[:, b, comp]) for b in range(nb)]
    mode = np.array([be_.mean() / (a_ + 1) for a_, be_ in pars])
    dl = mode[None, :] * np.exp(0.6 * rng.standard_normal((m, nb)))
    x, lm = _transform(kind, S, lmax + 1, edges, comp, dl)
    for b, (a_, be_) in enumerate(pars):
        xr, lr = G.transform(a_, be_, dl[:, b])
        sp, sq = G.tails(a_, be_, dl[:, b])
        acc = np.minimum(sp, sq) / n >= 1e-300        # the accuracy region; beyond it the tail is too small to resolve
        assert np.allclose(x[acc, b], xr[acc], rtol=1e-10, atol=1e-10), (b, np.abs(x[acc, b] - xr[acc]).max())
        assert np.all(np.abs(x[~acc, b]) > 37) and np.all(np.sign(x[~acc, b]) == np.sign(xr[~acc]))
        fin = np.isfinite(x[:, b])       # where F or 1 - F is 0 in FP64, logm is -inf by definition
        assert np.all(lm[~fin, b] == -np.inf)
        assert np.allclose(lm[fin, b], lr[fin], rtol=1e-12, atol=1e-12), (b, np.abs(lm[fin, b] - lr[fin]).max())


def test_consistency_determinism_and_special_values():
    from gibbssampler_b200.BlackwellRao import BlackwellRao
    rng = np.random.default_rng(7)
    lmax, n = 40, 2000
    sig = _joint_sigma(rng, n, lmax)
    bins = {"TT": np.concatenate([np.arange(0, 11), np.arange(12, lmax + 1, 4), [lmax + 1]]),
            "BB": np.array([0, 1, 2, 10, 20, 30, lmax + 1])}
    br = BlackwellRao(sig, bins)
    for key in ("TT", "EE", "BB"):
        nb = br.nbins[key]
        grid = np.geomspace(0.02, 50, 200)[None, :] * (np.array([1.0, 1.0] + [1.0] * (nb - 2)))[:, None]
        scale = {"TT": 200.0, "EE": 6.0, "BB": 0.5}[key]
        grid = grid * scale
        lm_br = br.marginal(key, grid)
        x, lm = br._transform(key, torch.as_tensor(grid[2:].T.copy(), device="cuda"))
        lm = lm.cpu().numpy().T
        fin = np.isfinite(x.cpu().numpy().T)        # F or 1 - F is 0 in FP64 beyond: x = +-inf and logm = -inf there
        assert np.all(lm[~fin] == -np.inf) and fin.sum() > 0.5 * fin.size and np.all(np.isfinite(lm_br[2:][fin]))
        # 1e-13 relative, or where larger the rounding of the direct form alpha log beta - beta / D - lgamma(alpha) - (alpha + 1) log D
        # that br_marginal_kernel evaluates (a few ulps of its largest term)
        pars = G.bin_params(sig, br.edges[key][2:], key)
        big = np.array([[a_ * np.abs(np.log(be_)).max() + gammaln(a_) + a_ * abs(np.log(g_)) + be_.max() / g_ for g_ in grid[2 + b]]
                        for b, (a_, be_) in enumerate(pars)])
        tol = np.maximum(1e-13 * np.abs(lm_br[2:]), 8 * 2.2e-16 * big)
        assert np.all(np.abs(lm - lm_br[2:])[fin] <= tol[fin]), (key, (np.abs(lm - lm_br[2:])[fin] / tol[fin]).max())
        cdf = br.cdf(key, grid)
        assert np.all(np.isnan(cdf[:2])) and np.all((cdf[2:] >= 0) & (cdf[2:] <= 1)) and np.all(np.diff(cdf[2:], axis=1) >= 0), key
        again = br.cdf(key, torch.as_tensor(grid, device="cuda"))
        assert isinstance(again, torch.Tensor) and np.array_equal(again.cpu().numpy(), cdf, equal_nan=True)
        x2, lm2 = br._transform(key, torch.as_tensor(grid[2:].T.copy(), device="cuda"))
        assert torch.equal(x, x2) and torch.equal(torch.as_tensor(lm.T.copy(), device="cuda"), lm2)       # bitwise repeatable
    # D <= 0: -inf; a model beyond every sample: x = +-inf, logm = -inf; a broken edge: NaN, its neighbours finite
    a, be = O.ig_alpha_beta(sig["BB"], np.array([2, 10, 20]))
    dl = np.array([[-1.0, 0.5], [0.0, 0.5], [1e-300, 0.5], [1e300, 0.5]])
    x, lm = _transform(0, be.T, lmax + 1, [2, 10, 20], 0, dl)
    assert np.all(x[:2, 0] == -np.inf) and np.all(lm[:2, 0] == -np.inf)
    assert x[2, 0] == -np.inf and x[3, 0] == np.inf and np.all(lm[2:, 0] == -np.inf)     # F = 0 below every sample, 1 above
    assert np.all(np.isfinite(x[:, 1])) and np.all(np.isfinite(lm[:, 1]))
    x, lm = _transform(0, np.vstack([be.T, be.T[:1]]), lmax + 1, [2, 10, 10, 20], 0, np.full((3, 3), 0.5))
    assert np.all(np.isnan(x[:, 1])) and np.all(np.isnan(lm[:, 1])) and np.all(np.isfinite(x[:, [0, 2]]))


def _batch_se(v, nbatch=20):
    """standard error of the mean of the rows of v (n, p) from batch means (the chain's autocorrelation included)"""
    parts = np.array_split(np.arange(len(v)), nbatch)
    bm = np.stack([v[p].mean(0) for p in parts])
    return bm.std(0, ddof=1) / np.sqrt(nbatch)


def _check_standard_normal(g, hist, keys, burn):
    x = np.concatenate([g.gaussianize(k, np.asarray(hist[k])[burn + 1:])[:, 2:] for k in keys], axis=1)
    mu, cov = g.mean.cpu().numpy(), g.cov.cpu().numpy()
    assert np.allclose(mu, x.mean(0), rtol=0, atol=1e-12)
    se_mu, se_var = _batch_se(x), _batch_se(x * x)
    assert np.all(np.abs(mu) <= 5 * se_mu + 1e-3), np.c_[mu, se_mu]
    assert np.all(np.abs(np.diag(cov) - 1) <= 5 * se_var + 0.02), np.c_[np.diag(cov), se_var]


def test_chain_plumbing_centered_tt_and_joint():
    """D rows are draws from the BR marginal of the same chain, so x = Phi^-1(F(D)) is N(0, 1) by construction: mu ~ 0 and
    diag Sigma ~ 1 within batch-means errors.  A wrong alpha, comp or row pairing breaks this."""
    from gibbssampler_b200.BlackwellRao import GaussianizedBlackwellRao
    from gibbssampler_b200.CenteredGibbs import CenteredGibbs
    from gibbssampler_b200.JointSampler import JointGibbs
    from tests.test_br_gpu import _pol_masked
    from tests.test_teb_binned_gpu import masked_sky
    nside, lmax, npix, mask, noise, d = _pol_masked(1)
    bins = np.array([0, 1, 2, 4, 7, 11, lmax + 1])
    g = CenteredGibbs(d["Q"], np.full(npix, 0.05), None, 5.0, nside, lmax, npix, mask=mask, bins=bins, n_iter=1200, seed=8,
                      keep_sigma=True)
    init = np.array([0, 0, 1.0, 1.0, 1.0, 1.0])
    h = g.run(init)
    gbr = GaussianizedBlackwellRao.from_sampler(g, h, burn_in=50)
    assert gbr.br.n == 1150 and gbr.keys == ("TT",)
    _check_standard_normal(gbr, {"TT": h[0]}, ("TT",), 50)
    data, (nT, nP), (mT, mP), _, _, dls = masked_sky(nside, lmax, 9)
    jb = {"TT": np.array([0, 1, 2, 4, 9, lmax + 1]), "BB": np.array([0, 1, 2, 8, lmax + 1])}
    jg = JointGibbs(data, nT, nP, 1.0, nside, lmax, n_iter=1200, bins=jb, seed=6, keep_sigma=True, mask=mT, mask_pol=mP)
    jh = jg.run({k: dls[k][jb["BB" if k == "BB" else "TT"][:-1]] for k in dls})
    jgbr = GaussianizedBlackwellRao.from_sampler(jg, jh, burn_in=50)
    assert jgbr.keys == ("TT", "EE", "BB") and jgbr.nbins == 3 + 3 + 2
    _check_standard_normal(jgbr, jh, ("TT", "EE", "BB"), 50)
    models = {k: np.asarray(jh[k])[-5:] for k in ("TT", "EE", "BB")}
    assert np.all(np.isfinite(jgbr.logpdf(models)))
    with pytest.raises(ValueError, match="TE is marginalised"):
        jgbr.logpdf(dict(models, TE=np.asarray(jh["TE"])[-5:]))
    # the oracle on the same chain: mu, Sigma and log L
    sig = {k: jg.sigma_history[k][50:] for k in ("TT", "TE", "EE", "BB")}
    e = {"TT": jb["TT"][2:], "EE": jb["TT"][2:], "BB": jb["BB"][2:]}
    rows = {k: np.asarray(jh[k])[51:, 2:] for k in ("TT", "EE", "BB")}
    want = G.logpdf(sig, e, rows, {k: v[:, 2:] for k, v in models.items()}, ("TT", "EE", "BB"))
    assert np.allclose(jgbr.logpdf(models), want, rtol=1e-9, atol=1e-8)


@pytest.mark.slow
def test_known_answer_full_sky_ee_bb():
    """Full sky, isotropic noise, harmonic data, per-l EE / BB CenteredGibbs to lmax = 20: the exact log-likelihood is
        sum_l sum_{EE,BB} -(2l+1)/2 [Chat_d / (b^2 C + N) + log(b^2 C + N)],  C = 2 pi D / (l (l+1)),
    which factorizes over l, so the GBR copula is the identity in the limit and GBR Delta log L estimates the exact one.  The
    noise makes S/N of a few at l = 20, where the 38-bin BR sum rests on a handful of samples (its n_eff is in the message).
    Tolerance: 5 batch-mean standard errors of the GBR Delta (10 batches, each its own GBR fit) plus 0.05."""
    from gibbssampler_b200.BlackwellRao import BlackwellRao, GaussianizedBlackwellRao
    from gibbssampler_b200.CenteredGibbs import CenteredGibbs
    nside, lmax, fwhm, noise0 = 8, 20, 5.0, 0.1
    npix = 12 * nside ** 2
    rng = np.random.default_rng(31)
    ell = np.arange(lmax + 1)
    f = np.where(ell >= 2, 2 * np.pi / np.maximum(ell * (ell + 1), 1), 0.0)
    dl_true = {"EE": np.where(ell >= 2, 1.0, 0.0), "BB": np.where(ell >= 2, 0.5, 0.0)}
    cov = np.zeros((lmax + 1, 2, 2))
    cov[:, 0, 0], cov[:, 1, 1] = dl_true["EE"] * f, dl_true["BB"] * f
    cov[:2] = np.eye(2)
    d, nl, bl = _harmonic_data(rng, lmax, nside, fwhm, cov, [noise0, noise0])
    pix_map = {"EE": d[:, 0], "BB": d[:, 1], "Q": np.zeros(npix), "U": np.zeros(npix)}
    bins = {"EE": np.arange(lmax + 2), "BB": np.arange(lmax + 2)}
    n_iter, burn = 4000, 100
    g = CenteredGibbs(pix_map, np.full(npix, 1.0), np.full(npix, noise0), fwhm, nside, lmax, npix, polarization=True, bins=bins,
                      n_iter=n_iter, seed=5, keep_sigma=True)
    h = g.run({k: v.copy() for k, v in dl_true.items()})[0]
    gbr = GaussianizedBlackwellRao.from_sampler(g, h, burn_in=burn)
    lof = R.l_of_real_layout(lmax)
    chat = {k: np.bincount(lof, weights=d[:, i] ** 2, minlength=lmax + 1) / (2 * ell + 1) for i, k in enumerate(("EE", "BB"))}

    def exact(th):
        out = 0.0
        for k in ("EE", "BB"):
            v = bl[2:] ** 2 * th[k][2:] * f[2:] + nl[0]
            out = out + (-(2 * ell[2:] + 1) / 2 * (chat[k][2:] / v + np.log(v))).sum(-1)
        return out
    th0 = {k: np.maximum((chat[k] - nl[0]) / bl ** 2 / np.maximum(f, 1e-300), 0.05) for k in chat}
    for k in th0:
        th0[k][:2] = 1.0
    models, deltas = [th0], []
    e0 = exact(th0)
    while len(models) < 16:
        th = {k: v * np.exp(0.1 * rng.standard_normal(lmax + 1)) for k, v in th0.items()}
        dlt = exact(th) - e0
        if dlt > -10:
            models.append(th)
            deltas.append(dlt)
    M = {k: np.stack([m[k] for m in models]) for k in th0}
    got = gbr.logpdf(M)
    diff = got[1:] - got[0]
    # batch means: one GBR per tenth of the chain
    sig = g.sigma_history
    parts = np.array_split(np.arange(burn, n_iter), 10)
    bd = []
    for p in parts:
        gb = GaussianizedBlackwellRao({k: sig[k][p] for k in ("EE", "BB")}, {k: h[k][np.r_[p[0], p + 1]] for k in ("EE", "BB")}, bins)
        v = gb.logpdf(M)
        bd.append(v[1:] - v[0])
    se = np.std(bd, axis=0, ddof=1) / np.sqrt(len(parts))
    _, neff = BlackwellRao.from_sampler(g, burn_in=burn).logpdf(M, n_eff=True)
    assert np.all(np.abs(diff - np.array(deltas)) <= 5 * se + 0.05), (np.c_[diff, deltas, se], "BR n_eff %s" % np.round(neff, 1))
