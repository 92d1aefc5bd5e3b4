"""CPU: the oracle of the binned TT/TE/EE conditional (tests.teb_binned_oracle) against the per-l oracle it generalises and
against the analytic inverse-Wishart moments; host-side validation of the joint sampler's bins; the C ABI of
gs_cls_invwishart_binned (declaration and argument checks, which run before anything touches a GPU)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from oracle import reference_logic as R
from tests import teb_binned_oracle as B

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def spectra(lmax, seed=0):
    rng = np.random.default_rng(seed)
    ell = np.arange(lmax + 1)
    tt = np.where(ell >= 2, 2.0 / (ell + 10.0) ** 2 * (1 + 0.1 * rng.random(lmax + 1)), 0.0)
    ee = np.where(ell >= 2, 0.5 / (ell + 10.0) ** 2 * (1 + 0.1 * rng.random(lmax + 1)), 0.0)
    te = 0.6 * np.sqrt(tt * ee) * np.cos(ell / 7.0)
    return tt, te, ee


def test_one_l_bins_reduce_to_the_per_l_draw():
    lmax = 60
    tt, te, ee = spectra(lmax)
    rng = np.random.default_rng(1)
    df = 2 * np.arange(lmax + 1) - 2.0
    draws = np.zeros((lmax + 1, 3))
    draws[2:, 0] = rng.chisquare(df[2:])
    draws[2:, 1] = rng.chisquare(df[2:] - 1)
    draws[2:, 2] = rng.standard_normal(lmax - 1)
    got = B.invwishart_bartlett_binned(tt, te, ee, np.arange(lmax + 2), draws)
    ell = np.arange(lmax + 1)
    ref = R.invwishart_bartlett(tt, te, ee, draws) * (ell * (ell + 1) / (2 * np.pi))[:, None, None]
    for l in range(2, lmax + 1):
        assert np.abs(got[l] - ref[l]).max() <= 1e-13 * np.abs(ref[l]).max(), l
    assert np.all(got[:2] == 0)
    nu, _ = B.nu_psi(tt, te, ee, np.arange(lmax + 2))
    assert np.array_equal(nu[2:], df[2:])


def test_numpy_stream_draws_have_the_inverse_wishart_moments():
    """4000 draws per bin, nu from 12 to 2.4e5: mean Psi / (nu - 3) and the p = 2 entry variances within 5 standard errors (the
    error of the sample variance from the sample's fourth central moment)."""
    lmax, n = 520, 4000
    edges = np.array([0, 1, 2, 7, 8, 20, 25, 100, 110, 500, 510, lmax + 1])
    tt, te, ee = spectra(lmax, 2)
    nu, psi = B.nu_psi(tt, te, ee, edges)
    assert nu[3] == 12 and nu[-1] > 1e4
    draws = B.bartlett_draws(nu, np.random.default_rng(3), n)
    X = np.array([B.invwishart_bartlett_binned(tt, te, ee, edges, d) for d in draws])
    X = np.stack([X[:, :, 0, 0], X[:, :, 0, 1], X[:, :, 1, 1]], axis=-1)[:, 2:]
    mean, var = B.iw_moments(nu[2:], psi[2:])
    m, v = X.mean(0), X.var(0, ddof=1)
    m4 = ((X - m) ** 4).mean(0)
    zm = np.abs(m - mean) / np.sqrt(var / n)
    zv = np.abs(v - var) / np.sqrt((m4 - v ** 2) / n)
    assert zm.max() < 5 and zv.max() < 5, (zm.max(), zv.max())


@pytest.mark.parametrize("bins, what", [
    ({"TT": [0, 2, 5, 11], "BB": [0, 1, 2, 11]}, "start"),
    ({"TT": [1, 2, 5, 11], "BB": [0, 1, 2, 11]}, "start"),
    ({"TT": [0, 1, 2, 5, 11], "BB": [0, 1, 2, 10]}, "end"),
    ({"TT": [0, 1, 2, 5, 12], "BB": [0, 1, 2, 11]}, "end"),
    ({"TT": [0, 1, 2, 5, 5, 11], "BB": [0, 1, 2, 11]}, "ascending"),
    ({"TT": [0, 1, 2, 7, 5, 11], "BB": [0, 1, 2, 11]}, "ascending"),
    ({"TT": [0, 1, 2, 5, 11], "BB": [0, 1, 2, 11], "TE": [0, 1, 2, 6, 11]}, "equal"),
    ({"TT": [0, 1, 2, 5, 11], "BB": [0, 1, 2, 11], "EE": [0, 1, 2, 11]}, "equal"),
    ({"TT": [0, 1, 2, 5, 11]}, "'BB'"),
    ({"TT": [0.0, 1.0, 2.0, 11.0], "BB": [0, 1, 2, 11]}, "integer"),
])
def test_bad_bins_are_refused_on_the_host(bins, what):
    from gibbssampler_b200.JointSampler import JointClsSampler
    with pytest.raises(ValueError, match=what):
        JointClsSampler(10, bins={k: np.array(v) for k, v in bins.items()})


def test_header_declares_the_binned_entry_point_and_the_library_checks_its_arguments():
    hdr = open(os.path.join(ROOT, "include", "gibbs_b200.h")).read()
    code = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    assert re.search(r"\bint\s+gs_cls_invwishart_binned\s*\(", code)
    from gibbssampler_b200 import _lib
    assert len(_lib.SIGNATURES["gs_cls_invwishart_binned"][1]) == 13
    L = _lib.lib()
    p = C.c_void_p(8)   # never dereferenced: every call below is refused before a launch

    def call(lmax, nbins, null=None):
        args = [p] * 3 + [lmax, p, nbins, None, 1, 1] + [p] * 3 + [None]
        if null is not None:
            args[null] = None
        return L.gs_cls_invwishart_binned(*args)

    for k in (0, 1, 2, 4, 9, 10, 11):
        assert call(16, 5, null=k) == -1, k
    assert b"null" in L.gs_last_error_string()
    assert call(-1, 1) == -1
    assert call(16, 0) == -1
    assert call(16, 18) == -1      # more bins than multipoles
    assert b"nbins" in L.gs_last_error_string()
