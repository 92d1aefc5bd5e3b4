"""Inputs of the joint T/E/B masked-sky tests: spectra with a strong TE correlation, three kinds of mask (the two synthetic
masks of bench.py and one with holes) and per-pixel noise."""
import numpy as np

import bench

MASKS = ("band", "galplane", "holes")


def spectra(lmax, te_frac=0.6):
    """D_l (unbinned) with |TE| = te_frac sqrt(TT EE) and a sign that changes with l; D_0 = D_1 = 0."""
    ell = np.arange(lmax + 1, dtype=np.float64)
    on = ell >= 2
    tt = np.where(on, 2000.0 / (1.0 + ell / 10.0), 0.0)
    ee = np.where(on, 40.0 * (1.0 + ell / 20.0) ** -1.5, 0.0)
    bb = np.where(on, 2.0 / (1.0 + ell / 30.0), 0.0)
    te = te_frac * np.sqrt(tt * ee) * np.cos(ell / 5.0)
    return {"TT": tt, "TE": te, "EE": ee, "BB": bb}


def make_mask(nside, kind):
    if kind in ("band", "galplane"):
        return bench.make_mask(nside, 0.8, kind)
    z, phi = bench.pixel_z(nside), bench.pixel_phi(nside)
    m = np.ones(12 * nside * nside)
    th = np.arccos(z)
    for th0, ph0, rad in ((0.6, 1.0, 0.45), (1.9, 3.5, 0.5), (2.6, 5.2, 0.35), (1.3, 0.2, 0.3)):
        cosd = np.cos(th) * np.cos(th0) + np.sin(th) * np.sin(th0) * np.cos(phi - ph0)
        m[cosd > np.cos(rad)] = 0.0
    return m


def noise_map(nside, level, seed, rough):
    """per-pixel noise variance: level times a pattern in latitude, times a random factor on the pixels of one hemisphere
    (rough = "north" or "south").  The rings of the other hemisphere keep one weight each (where the mask does not cut them), so
    T (rough north) and P (rough south) have constant-weight rings in different places: a spin-0 half that took the constant
    ring weights of N_P^-1 would give a wrong T operator."""
    rng = np.random.default_rng(seed)
    z = bench.pixel_z(nside)
    f = rng.uniform(0.7, 1.3, 12 * nside * nside)
    side = z > 0 if rough == "north" else z < 0
    return level * (1.0 + 0.5 * z ** 2) * np.where(side, f, 1.0)


def problem(nside, lmax, kind_T, kind_P, seed=0, fwhm=3.0, noise_T=30.0, noise_P=5.0):
    """-> dict with masks, noise maps, N^-1, data maps and the oracle TPProblem"""
    from tests.teb_oracle import TPProblem
    rng = np.random.default_rng(seed)
    npix = 12 * nside * nside
    mT, mP = make_mask(nside, kind_T), make_mask(nside, kind_P)
    nT, nP = noise_map(nside, noise_T, seed + 1, "north"), noise_map(nside, noise_P, seed + 2, "south")
    ivT, ivP = mT / nT, mP / nP
    d = {k: rng.standard_normal(npix) * s for k, s in (("I", 40.0), ("Q", 5.0), ("U", 5.0))}
    prob = TPProblem(nside, lmax, d["I"], d["Q"], d["U"], ivT, ivP, fwhm)
    return dict(mask_T=mT, mask_P=mP, noise_T=nT, noise_P=nP, inv_T=ivT, inv_P=ivP, d=d, prob=prob, fwhm=fwhm, rng=rng)


def active(lmax):
    """entries of the concatenated (T, E, B) vector that Q acts on: E and B have no l < 2 harmonics (spin 2), and there the
    prior is zero too (D_0 = D_1 = 0), so those rows and columns of Q vanish identically"""
    from oracle import reference_logic as R
    ell = R.l_of_real_layout(lmax)
    return np.concatenate([np.ones(ell.size, bool), ell >= 2, ell >= 2])
