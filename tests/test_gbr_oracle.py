"""CPU: the Gaussianized Blackwell-Rao oracle (tests/gbr_oracle.py) against scipy, the host argument checks of
GaussianizedBlackwellRao, and the argument checks of the gs_gbr_transform entry points."""
import ctypes as C

import numpy as np
import pytest
from scipy import integrate
from scipy.special import ndtr
from scipy.stats import invgamma, norm

from tests import br_oracle as B
from tests import gbr_oracle as G
from tests.test_br_oracle import _joint_sigma


def test_one_sample_cdf_is_the_inverse_gamma_cdf():
    for a, beta in ((1.5, 0.7), (7.5, 30.0), (499.5, 2e3)):
        D = np.geomspace(beta / a / 30, beta / a * 30, 41)
        sp, sq = G.tails(a, np.array([beta]), D)
        assert np.allclose(sq, invgamma.cdf(D, a, scale=beta), rtol=1e-12, atol=0)
        assert np.allclose(sp, invgamma.sf(D, a, scale=beta), rtol=1e-12, atol=0)
        x, lm = G.transform(a, np.array([beta]), D)
        assert np.allclose(lm, invgamma.logpdf(D, a, scale=beta), rtol=1e-12, atol=1e-12)
        assert np.allclose(ndtr(x), invgamma.cdf(D, a, scale=beta), rtol=1e-11, atol=0)


def _mixture(rng, n=40, lmax=12):
    sig = _joint_sigma(rng, n, lmax)
    a, be = B.ig_alpha_beta(sig["BB"], np.array([4, 7]))
    return a[0], be[:, 0]


def test_jacobian_is_marginal_over_phi():
    a, be = _mixture(np.random.default_rng(1))
    D = np.geomspace(be.mean() / a / 3, be.mean() / a * 3, 15)
    h = 1e-6 * D
    xp, _ = G.transform(a, be, D + h)
    xm, _ = G.transform(a, be, D - h)
    x, lm = G.transform(a, be, D)
    assert np.allclose((xp - xm) / (2 * h), np.exp(lm) / norm.pdf(x), rtol=1e-6, atol=0)


def test_one_bin_density_integrates_to_one():
    a, be = _mixture(np.random.default_rng(2))
    mu, var = np.array([0.3]), np.array([[1.7]])

    def p(D):
        x, lm = G.transform(a, be, np.array([D]))
        return float(np.exp(G.logpdf_x(x[:, None], lm[:, None], mu, var))[0]) if np.isfinite(x[0]) else 0.0
    s = be.mean() / a
    val, _ = integrate.quad(p, 1e-3 * s, 200 * s, points=[0.3 * s, s, 3 * s], limit=400, epsabs=0, epsrel=1e-10)
    assert val == pytest.approx(1.0, abs=1e-7)


def test_identity_copula_is_the_product_of_marginals():
    rng = np.random.default_rng(3)
    sig = _joint_sigma(rng, 30, 10)
    edges = {"TT": np.array([2, 4, 7, 11]), "EE": np.array([2, 4, 7, 11]), "BB": np.array([2, 6, 11])}
    dls = {"TT": rng.uniform(150, 250, (5, 3)), "EE": rng.uniform(4, 8, (5, 3)), "BB": rng.uniform(0.3, 0.8, (5, 2))}
    x, lm = G.gaussianize(sig, edges, dls, ("TT", "EE", "BB"))
    got = G.logpdf_x(x, lm, np.zeros(8), np.eye(8))
    assert np.allclose(got, lm.sum(1), rtol=0, atol=1e-10)
    # the marginal is the BR marginal of br_oracle (IW diagonal for TT / EE of a joint sigma)
    nu, psi = B.iw_nu_psi(sig["TT"], sig["TE"], sig["EE"], edges["TT"])
    want = B.marginal_ig(0.5 * (nu[1] - 1), 0.5 * psi[:, 1, 2], dls["EE"][:, 1])
    assert np.allclose(lm[:, 4], want, rtol=0, atol=1e-12)


def test_gaussianized_br_argument_checks():
    """Every check below fails on the host before any device work, so it runs with or without a GPU."""
    from gibbssampler_b200.BlackwellRao import BlackwellRao, GaussianizedBlackwellRao
    sig = {"TT": np.ones((6, 5))}
    hist = np.ones((7, 5))
    bad = [
        (sig, np.ones((6, 5)), "expected \\(7, 5\\)"),                        # D history one row short
        ([sig, sig], [hist], "1 chains, sigma 2"),
        (sig, {"EE": hist}, "no history"),
        ({"EE": np.ones((6, 5)), "BB": np.ones((6, 5))}, np.ones((7, 5)), "dict of D histories"),
        ({"TT": np.ones((2, 5))}, np.ones((3, 5)), "at least 4"),            # 3 bins, 2 samples
    ]
    for s, h, msg in bad:
        with pytest.raises(ValueError, match=msg):
            GaussianizedBlackwellRao(s, h, None)
    with pytest.raises(ValueError, match="burn_in"):
        GaussianizedBlackwellRao(sig, hist, None, burn_in=6)
    # model checks, on an object whose host state alone is set up
    joint = {k: np.ones((40, 21)) for k in ("TT", "TE", "EE", "BB")}
    bins = {"TT": np.concatenate([np.arange(0, 11), np.arange(12, 21, 4), [21]]), "BB": np.array([0, 1, 2, 10, 21])}
    g = GaussianizedBlackwellRao.__new__(GaussianizedBlackwellRao)
    g.br = BlackwellRao.__new__(BlackwellRao)
    g.br._validate(joint, bins, 0)
    g.keys = ("TT", "EE", "BB")
    models = {k: np.ones(len(bins["BB" if k == "BB" else "TT"]) - 1) for k in ("TT", "TE", "EE", "BB")}
    with pytest.raises(ValueError, match="TE is marginalised"):
        g.logpdf(models)
    with pytest.raises(ValueError, match="cuts bin"):
        g.logpdf({k: v for k, v in models.items() if k != "TE"}, lrange=(2, 14))


def test_gbr_entry_points_reject_bad_arguments():
    from gibbssampler_b200 import _lib
    L = _lib.lib()
    x = C.c_void_p(16)     # never dereferenced: every call below fails its argument check first
    assert L.gs_gbr_transform(0, None, 10, 5, x, 2, 0, x, 3, x, x, x, None) == -1
    assert b"null" in L.gs_last_error_string()
    assert L.gs_gbr_transform(0, x, 10, 5, x, 2, 0, x, 3, None, x, x, None) == -1
    assert L.gs_gbr_transform(0, x, 10, 5, x, 2, 0, x, 3, x, x, None, None) == -1
    assert L.gs_gbr_transform(2, x, 10, 5, x, 2, 0, x, 3, x, x, x, None) == -1           # bad kind
    assert L.gs_gbr_transform(1, x, 10, 5, x, 2, 1, x, 3, x, x, x, None) == -1           # TE comp
    assert L.gs_gbr_transform(0, x, 10, 5, x, 2, 2, x, 3, x, x, x, None) == -1           # comp of an IG group
    assert L.gs_gbr_transform(0, x, 0, 5, x, 2, 0, x, 3, x, x, x, None) == -1            # no sample
    assert L.gs_gbr_transform(0, x, 10, 5, x, 2, 0, x, 0, x, x, x, None) == -1           # no model
    assert L.gs_gbr_transform(0, x, 10, 5, x, 6, 0, x, 3, x, x, x, None) == -1           # nbins > ncl
    assert L.gs_gbr_transform(0, x, 10, 5, x, 0, 0, x, 3, x, x, x, None) == -1           # nbins < 1
    assert L.gs_gbr_transform(0, x, 10, 70000, x, 65536, 0, x, 3, x, x, x, None) == -1   # nbins > 65535
    assert L.gs_gbr_transform_scratch(0, 3, 2) == -1 and L.gs_gbr_transform_scratch(10, 0, 2) == -1
    assert L.gs_gbr_transform_scratch(10, 3, 0) == -1
    assert L.gs_gbr_transform_scratch(65536, 1, 28) > 0
