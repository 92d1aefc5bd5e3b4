"""CPU: the Blackwell-Rao oracle (tests/br_oracle.py) against scipy, the argument checks of BlackwellRao and of the
keep_sigma option, and the null-pointer checks of the gs_br_* entry points."""
import ctypes as C

import numpy as np
import pytest
from scipy import integrate
from scipy.stats import invgamma, invwishart

from tests import br_oracle as O


def _joint_sigma(rng, n, lmax):
    ell = np.arange(lmax + 1)
    tt = rng.uniform(0.5, 2.0, (n, lmax + 1)) * 1e3 / np.maximum(ell * (ell + 1), 1)
    ee = rng.uniform(0.5, 2.0, (n, lmax + 1)) * 30.0 / np.maximum(ell * (ell + 1), 1)
    te = 0.4 * np.sqrt(tt * ee) * rng.uniform(-1, 1, (n, lmax + 1))
    bb = rng.uniform(0.5, 2.0, (n, lmax + 1)) * 3.0 / np.maximum(ell * (ell + 1), 1)
    return {"TT": tt, "TE": te, "EE": ee, "BB": bb}


def _joint_models(rng, m, nt, nb):
    tt = rng.uniform(150, 250, (m, nt))
    ee = rng.uniform(4, 8, (m, nt))
    te = 0.3 * np.sqrt(tt * ee) * rng.uniform(-1, 1, (m, nt))
    return {"TT": tt, "TE": te, "EE": ee, "BB": rng.uniform(0.3, 0.8, (m, nb))}


def test_gemm_decomposition_equals_direct_scipy_sum():
    rng = np.random.default_rng(1)
    lmax = 9
    sigma = _joint_sigma(rng, 7, lmax)
    edges = {"TT": np.array([2, 3, 5, 10]), "BB": np.array([2, 4, 7, 10])}
    dls = _joint_models(rng, 5, 3, 3)
    dls["TT"][4, 1] = -1.0      # an invalid model
    got, neff = O.logpdf(sigma, edges, dls)
    want = O.logpdf_direct(sigma, edges, {k: v[:4] for k, v in dls.items()})
    assert got[4] == -np.inf and neff[4] == 0
    assert np.allclose(got[:4], want, rtol=0, atol=1e-9)
    # independent inverse-gamma spectra
    ig = {"EE": sigma["EE"], "BB": sigma["BB"]}
    e2 = {"EE": np.array([2, 6, 10]), "BB": np.array([2, 4, 7, 10])}
    d2 = {"EE": rng.uniform(4, 8, (3, 2)), "BB": rng.uniform(0.3, 0.8, (3, 3))}
    assert np.allclose(O.logpdf(ig, e2, d2)[0], O.logpdf_direct(ig, e2, d2), rtol=0, atol=1e-9)


def test_one_sample_estimator_is_the_conditional():
    rng = np.random.default_rng(2)
    sigma = _joint_sigma(rng, 1, 6)
    edges = {"TT": np.array([2, 4, 7]), "BB": np.array([2, 3, 7])}
    dls = _joint_models(rng, 3, 2, 2)
    got, neff = O.logpdf(sigma, edges, dls)
    nu, psi = O.iw_nu_psi(sigma["TT"], sigma["TE"], sigma["EE"], edges["TT"])
    a, be = O.ig_alpha_beta(sigma["BB"], edges["BB"])
    for m in range(3):
        want = sum(invgamma.logpdf(dls["BB"][m, b], a[b], scale=be[0, b]) for b in range(2))
        for b in range(2):
            P = [[psi[0, b, 0], psi[0, b, 1]], [psi[0, b, 1], psi[0, b, 2]]]
            D = [[dls["TT"][m, b], dls["TE"][m, b]], [dls["TE"][m, b], dls["EE"][m, b]]]
            want += invwishart.logpdf(D, df=nu[b], scale=P)
        assert got[m] == pytest.approx(want, abs=1e-10)
    assert np.all(neff == 1.0)


def test_iw_diagonal_marginal_matches_integration():
    rng = np.random.default_rng(3)
    sigma = _joint_sigma(rng, 1, 5)
    nu, psi = O.iw_nu_psi(sigma["TT"], sigma["TE"], sigma["EE"], np.array([2, 4]))
    P = np.array([[psi[0, 0, 0], psi[0, 0, 1]], [psi[0, 0, 1], psi[0, 0, 2]]])
    for j in (0, 1):
        x = P[j, j] / (nu[0] - 1)          # near the mode of the marginal
        other = 1 - j

        def f(t, y):                         # joint density at D_jj = x, D_oo = t, D_jo = y
            D = np.zeros((2, 2))
            D[j, j], D[other, other], D[0, 1] = x, t, y
            D[1, 0] = y
            if t <= 0 or x * t - y * y <= 0:
                return 0.0
            return np.exp(invwishart.logpdf(D, df=nu[0], scale=P))
        s = np.sqrt(P[other, other] / nu[0])
        to = P[other, other] / (nu[0] + 3)
        val, _ = integrate.dblquad(lambda y, t: f(t, y), 1e-6 * to, 20 * to,
                                   lambda t: -np.sqrt(x * t), lambda t: np.sqrt(x * t), epsabs=0, epsrel=1e-8)
        want = O.marginal_ig(0.5 * (nu[0] - 1), np.array([0.5 * P[j, j]]), np.array([x]))[0]
        assert np.log(val) == pytest.approx(want, abs=2e-3), (j, s)


def test_blackwellrao_argument_checks():
    """Every check below fails before any device work, so it runs with or without a GPU."""
    from gibbssampler_b200.BlackwellRao import BlackwellRao
    sig = {"TT": np.ones((4, 5))}
    joint = {k: np.ones((4, 5)) for k in ("TT", "TE", "EE", "BB")}
    bad = [
        ({"TT": np.ones((4, 5)), "TE": np.ones((4, 5))}, None, "exactly the keys"),
        ({"XX": np.ones((4, 5))}, None, "keys must be among"),
        ({"TT": np.ones(5)}, None, "2-d"),
        ({"EE": np.ones((4, 5)), "BB": np.ones((3, 5))}, None, "shape"),
        ([sig, {"EE": np.ones((4, 5))}], None, "same spectra"),
        (sig, np.array([0, 1, 1, 3]), "ascending"),
        (sig, np.array([0, 1, 2, 6]), "lie in"),
        (sig, np.array([0.0, 1.0, 2.0, 3.0]), "integer"),
        (sig, np.array([0, 1, 2]), "at least 4"),
        (joint, {"TT": np.arange(6)}, "'BB'"),
        (joint, {"TT": np.array([0, 1, 2, 4]), "BB": np.arange(6)}, "end at lmax"),
        (joint, {"TT": np.arange(6), "EE": np.array([0, 1, 2, 5]), "BB": np.arange(6)}, "must equal"),
    ]
    for s, bins, msg in bad:
        with pytest.raises(ValueError, match=msg):
            BlackwellRao(s, bins)
    with pytest.raises(ValueError, match="burn_in"):
        BlackwellRao(sig, None, burn_in=4)
    with pytest.raises(ValueError, match="burn_in"):
        BlackwellRao(sig, None, burn_in=-1)


def test_keep_sigma_only_where_it_is_built():
    from gibbssampler_b200.ASIS import ASIS
    from gibbssampler_b200.NonCenteredGibbs import NonCenteredGibbs
    from gibbssampler_b200.PNCP import PNCPGibbs
    for cls in (NonCenteredGibbs, ASIS, PNCPGibbs):
        with pytest.raises(TypeError, match="keep_sigma"):
            cls(None, None, None, 1.0, 4, 8, 192, None, keep_sigma=True)
    from gibbssampler_b200 import GibbsB200Error, multichain
    from gibbssampler_b200.CenteredGibbs import CenteredGibbs
    with pytest.raises(GibbsB200Error, match="sharded plan"):     # refused before the plan or the data are looked at
        CenteredGibbs(None, None, None, 1.0, 4, 8, 192, polarization=True, plan=object(), keep_sigma=True)

    class G:
        keep_sigma, n_iter, polarization = True, 1, True
    with pytest.raises(ValueError, match="keep_sigma"):
        multichain.run_chains([G()], [{}])


def test_br_entry_points_reject_null_pointers():
    from gibbssampler_b200 import _lib
    L = _lib.lib()
    x = C.c_void_p(16)     # never dereferenced: every call below fails its argument check first
    assert L.gs_br_sample_features(0, None, None, None, 10, 5, x, 2, x, x, 0, x, None) == -1
    assert b"null" in L.gs_last_error_string()
    assert L.gs_br_sample_features(1, x, None, x, 10, 5, x, 2, x, x, 0, x, None) == -1
    assert L.gs_br_sample_features(2, x, x, x, 10, 5, x, 2, x, x, 0, x, None) == -1        # bad kind
    assert L.gs_br_sample_features(0, x, None, None, 10, 5, x, 6, x, x, 0, x, None) == -1  # nbins > ncl
    assert L.gs_br_model_features(0, None, None, None, 10, 5, x, 2, x, x, 0, x, None) == -1
    assert L.gs_br_model_features(0, x, None, None, 0, 5, x, 2, x, x, 0, x, None) == -1    # no model
    assert L.gs_br_logmeanexp(x, None, 10, x, x, 3, 4, x, x, None, None) == -1
    assert L.gs_br_logmeanexp(x, x, 10, x, x, 3, 0, x, x, None, None) == -1                # K = 0
    assert L.gs_br_marginal(0, None, 10, 5, x, 2, 0, x, 0, 8, x, None) == -1
    assert L.gs_br_marginal(1, x, 10, 5, x, 2, 1, x, 0, 8, x, None) == -1                  # TE marginal
