"""Test oracle of the binned TT/TE/EE conditional of the joint sampler (gs_cls_invwishart_binned), a restatement of the
formula next to the per-l oracle.invwishart_bartlett it reduces to, plus the analytic moments of a 2x2 inverse-Wishart:
    D_b | s ~ IW(nu_b, Psi_b),  nu_b = sum_{l in b} (2l+1) - 3,  Psi_b = sum_{l in b} (2l+1) l(l+1)/(2 pi) Chat_l."""
import numpy as np


def nu_psi(cl_tt, cl_te, cl_ee, bins):
    """-> (nu, Psi) per bin: (nbins,), (nbins, 2, 2); bins 0 and 1 are left at 0"""
    nb = len(bins) - 1
    nu, psi = np.zeros(nb), np.zeros((nb, 2, 2))
    for b in range(2, nb):
        ls = np.arange(bins[b], bins[b + 1])
        w = (2 * ls + 1) * ls * (ls + 1) / (2 * np.pi)
        nu[b] = np.sum(2 * ls + 1) - 3
        psi[b] = [[w @ cl_tt[ls], w @ cl_te[ls]], [w @ cl_te[ls], w @ cl_ee[ls]]]
    return nu, psi


def invwishart_bartlett_binned(cl_tt, cl_te, cl_ee, bins, draws):
    """Binned D_b (nbins, 2, 2) from supplied (chi2_nu, chi2_{nu-1}, N(0,1)) per bin: X^-1 = (G A)(G A)^T with
    Psi_b^-1 = G G^T and A = [[sqrt(chi2_nu), 0], [N(0,1), sqrt(chi2_{nu-1})]]; bins 0 and 1 (l = 0 and l = 1) -> 0."""
    _, psi = nu_psi(cl_tt, cl_te, cl_ee, bins)
    out = np.zeros_like(psi)
    for b in range(2, len(psi)):
        g = np.linalg.cholesky(np.linalg.inv(psi[b]))
        a = np.array([[np.sqrt(draws[b, 0]), 0.0], [draws[b, 2], np.sqrt(draws[b, 1])]])
        h = g @ a
        out[b] = np.linalg.inv(h @ h.T)
    return out


def iw_moments(nu, psi):
    """Mean Psi / (nu - 3) and entry variances ((nu-1) psi_ij^2 + (nu-3) psi_ii psi_jj) / ((nu-2) (nu-3)^2 (nu-5)) of IW(nu, Psi),
    p = 2, for the entries (TT, TE, EE) = (00, 01, 11): two arrays (..., 3)."""
    nu = np.asarray(nu, dtype=np.float64)[..., None]
    p00, p01, p11 = psi[..., 0, 0], psi[..., 0, 1], psi[..., 1, 1]
    ent = np.stack([p00, p01, p11], axis=-1)
    diag = np.stack([p00 * p00, p00 * p11, p11 * p11], axis=-1)
    mean = ent / (nu - 3)
    var = ((nu - 1) * ent ** 2 + (nu - 3) * diag) / ((nu - 2) * (nu - 3) ** 2 * (nu - 5))
    return mean, var


def bartlett_draws(nu, rng, n):
    """(n, nbins, 3) numpy-stream variates (chi2_nu, chi2_{nu-1}, N(0,1)) per bin; bins with nu <= 1 get ones and zeros"""
    nu = np.asarray(nu, dtype=np.float64)
    on = nu > 1
    d = np.zeros((n, nu.size, 3))
    d[:, :, :2] = 1.0
    d[:, on, 0] = rng.chisquare(nu[on], size=(n, int(on.sum())))
    d[:, on, 1] = rng.chisquare(nu[on] - 1, size=(n, int(on.sum())))
    d[:, on, 2] = rng.standard_normal((n, int(on.sum())))
    return d
