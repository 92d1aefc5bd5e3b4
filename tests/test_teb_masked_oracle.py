"""CPU: the oracle of the joint T/E/B masked-sky system (tests.teb_oracle.TPProblem) against the TT and E/B restatements
it is built from, its dense operator, its PCG, and the C ABI declaring the three joint entry points."""
import os
import re

import numpy as np

from oracle import reference_logic as R
from tests import teb_problem as T
from tests.teb_oracle import TPProblem

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_uncoupled_operator_is_tt_plus_pol():
    nside, lmax = 4, 8
    P = T.problem(nside, lmax, "galplane", "band", seed=1)
    dls = T.spectra(lmax, te_frac=0.0)
    rng = np.random.default_rng(2)
    n = (lmax + 1) ** 2
    x = tuple(rng.standard_normal(n) for _ in range(3))
    y = P["prob"].apply_Q(dls, x)
    tt = R.TTProblem(nside, lmax, P["d"]["I"], P["inv_T"], P["fwhm"])
    pol = R.PolProblem(nside, lmax, P["d"]["Q"], P["d"]["U"], P["inv_P"], P["fwhm"])
    yT = tt.apply_Q(R.generate_var_cl(dls["TT"]), x[0])
    yE, yB = pol.apply_Q(dls["EE"], dls["BB"], x[1], x[2])
    for a, b in zip(y, (yT, yE, yB)):
        assert np.abs(a - b).max() <= 1e-13 * np.abs(b).max()


def test_coupled_dense_operator_is_symmetric_positive_definite():
    nside, lmax = 4, 8
    P = T.problem(nside, lmax, "holes", "galplane", seed=3)
    dls = T.spectra(lmax)
    Q = P["prob"].dense_Q(dls)
    act = T.active(lmax)
    assert np.all(Q[~act] == 0) and np.all(Q[:, ~act] == 0)
    Qa = Q[np.ix_(act, act)]
    assert np.abs(Qa - Qa.T).max() <= 1e-12 * np.abs(Qa).max()
    w = np.linalg.eigvalsh(0.5 * (Qa + Qa.T))
    assert w.min() > 0
    # the TE coupling is really there: T rows see E columns
    n = (lmax + 1) ** 2
    assert np.abs(Q[:n, n:2 * n]).max() > 1e-3 * np.abs(Q[:n, :n]).max()


def test_oracle_pcg_reaches_the_dense_solve():
    nside, lmax = 4, 8
    P = T.problem(nside, lmax, "galplane", "band", seed=4)
    prob, rng = P["prob"], P["rng"]
    dls = T.spectra(lmax)
    npix, n = 12 * nside * nside, (lmax + 1) ** 2
    xi = [rng.standard_normal(npix) for _ in range(3)] + [rng.standard_normal(n) for _ in range(3)]
    b = prob.rhs(dls, *xi)
    x, it = prob.pcg(dls, b, eps=1e-12)
    act = T.active(lmax)
    Q = prob.dense_Q(dls)
    ref = np.zeros(3 * n)
    ref[act] = np.linalg.solve(Q[np.ix_(act, act)], np.concatenate(b)[act])
    got = np.concatenate(x)
    assert 0 < it < 4000
    assert np.abs(got - ref).max() <= 1e-8 * np.abs(ref).max()


def test_prior_factor_squares_to_the_inverse_covariance():
    lmax = 12
    dls = T.spectra(lmax)
    prob = TPProblem.__new__(TPProblem)
    prob.lmax = lmax
    fTT, fTE, fEE, fBB = prob.factor(dls)
    iTT, iTE, iEE, iBB = prob.inv_cov(dls)
    for l in range(lmax + 1):
        F = np.array([[fTT[l], fTE[l]], [0.0, fEE[l]]])
        FF = F @ F.T
        assert np.allclose(FF, [[iTT[l], iTE[l]], [iTE[l], iEE[l]]], rtol=1e-12, atol=0)
        assert np.isclose(fBB[l] ** 2, iBB[l], rtol=1e-14, atol=0)


def test_header_declares_the_joint_entry_points():
    hdr = open(os.path.join(ROOT, "include", "gibbs_b200.h")).read()
    code = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    for name in ("gs_cr_rhs_teb", "gs_cr_pcg_teb", "gs_cr_apply_q_teb"):
        assert re.search(r"\bint\s+" + name + r"\s*\(", code), name
    from gibbssampler_b200 import _lib
    assert len(_lib.SIGNATURES["gs_cr_rhs_teb"][1]) == 27
    assert len(_lib.SIGNATURES["gs_cr_pcg_teb"][1]) == 23
    assert len(_lib.SIGNATURES["gs_cr_apply_q_teb"][1]) == 15
