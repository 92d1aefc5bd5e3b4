"""numpy / scipy oracle of the Blackwell-Rao estimator (gibbssampler_b200.BlackwellRao, csrc/blackwell_rao.cu).

sigma: dict of (N, lmax + 1) empirical C_l per sample; edges of the evaluated bins only (the chains' bins 0 and 1 are
dropped by the caller).  Without "TE" every key is an inverse-gamma spectrum; with "TE" the TT edges carry the
(TT, TE; TE, EE) inverse-Wishart and the BB edges an inverse-gamma BB."""
import numpy as np
from scipy.special import gammaln, logsumexp


def ig_alpha_beta(sig, edges):
    """alpha (nb,), beta (N, nb) of cls_invgamma_kernel on the bins [edges[b], edges[b+1])."""
    ell = np.arange(sig.shape[1], dtype=np.float64)
    w = (2 * ell + 1) * ell * (ell + 1) / (4 * np.pi)
    alpha = np.array([np.sum((2 * ell[a:b] + 1) / 2) - 1 for a, b in zip(edges[:-1], edges[1:])])
    beta = np.stack([(sig[:, a:b] * w[a:b]).sum(1) for a, b in zip(edges[:-1], edges[1:])], axis=1)
    return alpha, beta


def iw_nu_psi(tt, te, ee, edges):
    """nu (nb,), Psi (N, nb, 3) = (Psi00, Psi01, Psi11) of invwishart_binned_kernel."""
    ell = np.arange(tt.shape[1], dtype=np.float64)
    w = (2 * ell + 1) * ell * (ell + 1) / (2 * np.pi)
    nu = np.array([np.sum(2 * ell[a:b] + 1) - 3 for a, b in zip(edges[:-1], edges[1:])])
    psi = np.stack([np.stack([(x[:, a:b] * w[a:b]).sum(1) for x in (tt, te, ee)], axis=1)
                    for a, b in zip(edges[:-1], edges[1:])], axis=1)
    return nu, psi


def features(sigma, edges):
    """-> (S (N, K), c (N,), groups) with the row layout of BlackwellRao: joint: IW rows (3 per TT bin), then BB rows;
    otherwise one row per bin of each key in dict order."""
    S, c, groups = [], 0.0, []
    if "TE" in sigma:
        nu, psi = iw_nu_psi(sigma["TT"], sigma["TE"], sigma["EE"], edges["TT"])
        S.append(psi.reshape(psi.shape[0], -1))
        c = c + (0.5 * nu * np.log(psi[..., 0] * psi[..., 2] - psi[..., 1] ** 2)).sum(1)
        groups.append(("IW", ("TT", "TE", "EE"), nu))
        keys = ("BB",)
    else:
        keys = tuple(sigma)
    for k in keys:
        a, be = ig_alpha_beta(sigma[k], edges[k])
        S.append(be)
        c = c + (a * np.log(be)).sum(1)
        groups.append(("IG", (k,), a))
    return np.concatenate(S, axis=1), c, groups


def model_features(dls, groups):
    """dls: dict of (M, nb) binned D of the evaluated bins -> (W (K, M), e (M,)); invalid models: W = 0, e = -inf."""
    W, e = [], 0.0
    for kind, keys, par in groups:
        if kind == "IG":
            D = dls[keys[0]]
            ok = D > 0
            Ds = np.where(ok, D, 1.0)
            W.append(np.where(ok, -1.0 / Ds, 0.0).T)
            e = e + np.where(ok, -gammaln(par) - (par + 1) * np.log(Ds), -np.inf).sum(1)
        else:
            tt, te, ee = (dls[k] for k in keys)
            det = tt * ee - te * te
            ok = (tt > 0) & (det > 0)
            ds = np.where(ok, det, 1.0)
            w = np.stack([np.where(ok, -0.5 * ee / ds, 0), np.where(ok, te / ds, 0), np.where(ok, -0.5 * tt / ds, 0)], axis=2)
            W.append(w.reshape(w.shape[0], -1).T)
            lg2 = 0.5 * np.log(np.pi) + gammaln(par / 2) + gammaln(par / 2 - 0.5)
            e = e + np.where(ok, -par * np.log(2) - lg2 - 0.5 * (par + 3) * np.log(ds), -np.inf).sum(1)
    return np.concatenate(W, axis=0), e


def logmeanexp(S, c, W, e):
    """GEMM decomposition, evaluated in extended precision: -> (log L (M,), n_eff (M,))."""
    x = (c.astype(np.longdouble)[:, None] + S.astype(np.longdouble) @ W.astype(np.longdouble)
         + e.astype(np.longdouble)[None, :])
    out, neff = np.full(x.shape[1], -np.inf), np.zeros(x.shape[1])
    for k in range(x.shape[1]):
        if not np.isfinite(e[k]):
            continue
        m = x[:, k].max()
        w = np.exp(x[:, k] - m)
        out[k] = float(m + np.log(w.sum()) - np.log(x.shape[0]))
        neff[k] = float(w.sum() ** 2 / (w * w).sum())
    return out, neff


def logpdf(sigma, edges, dls):
    S, c, groups = features(sigma, edges)
    W, e = model_features(dls, groups)
    return logmeanexp(S, c, W, e)


def logpdf_direct(sigma, edges, dls):
    """The same estimator as a direct sum of scipy log-densities and scipy's logsumexp (no GEMM)."""
    from scipy.stats import invgamma, invwishart
    N = next(iter(sigma.values())).shape[0]
    M = next(iter(dls.values())).shape[0]
    x = np.zeros((N, M))
    ig_keys = ("BB",) if "TE" in sigma else tuple(sigma)
    for k in ig_keys:
        a, be = ig_alpha_beta(sigma[k], edges[k])
        for i in range(N):
            for m in range(M):
                x[i, m] += invgamma.logpdf(dls[k][m], a, scale=be[i]).sum()
    if "TE" in sigma:
        nu, psi = iw_nu_psi(sigma["TT"], sigma["TE"], sigma["EE"], edges["TT"])
        for i in range(N):
            for m in range(M):
                for b in range(len(nu)):
                    P = np.array([[psi[i, b, 0], psi[i, b, 1]], [psi[i, b, 1], psi[i, b, 2]]])
                    D = np.array([[dls["TT"][m, b], dls["TE"][m, b]], [dls["TE"][m, b], dls["EE"][m, b]]])
                    x[i, m] += invwishart.logpdf(D, df=nu[b], scale=P)
    return logsumexp(x, axis=0) - np.log(N)


def marginal_ig(alpha, beta, grid):
    """log mean_i IG(grid | alpha, beta_i) for one bin: beta (N,), grid (G,)."""
    g = grid[None, :]
    lp = alpha * np.log(beta[:, None]) - gammaln(alpha) - (alpha + 1) * np.log(g) - beta[:, None] / g
    return logsumexp(lp, axis=0) - np.log(len(beta))
