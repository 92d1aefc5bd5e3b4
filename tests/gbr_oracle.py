"""numpy / scipy oracle of the Gaussianized Blackwell-Rao likelihood (gibbssampler_b200.BlackwellRao.GaussianizedBlackwellRao,
gs_gbr_transform in csrc/blackwell_rao.cu), built on tests/br_oracle.py.

One bin's BR marginal is the mixture (1/N) sum_i IG(alpha, beta_i).  With t_i = beta_i / D ~ Gamma(alpha, 1), its CDF is
F = (1/N) sum_i Q(alpha, t_i) and 1 - F = (1/N) sum_i P(alpha, t_i); x = Phi^-1(F) is taken from the smaller of the two sums."""
import numpy as np
from scipy.special import gammainc, gammaincc, gammaln, logsumexp, ndtri

from tests import br_oracle as B


def tails(alpha, beta, D):
    """(sum_i P(alpha, beta_i / D), sum_i Q(alpha, beta_i / D)) for beta (N,) and D (G,): each sample's smaller tail is the direct
    one (P below t = alpha + 1, Q above, as the kernel chooses), the other 1 - small."""
    t = beta[:, None] / D[None, :]
    lower = t < alpha + 1.0
    P = np.where(lower, gammainc(alpha, t), 1.0 - gammaincc(alpha, t))
    Q = np.where(lower, 1.0 - gammainc(alpha, t), gammaincc(alpha, t))
    return P.sum(0), Q.sum(0)


def transform(alpha, beta, D):
    """-> (x (G,), logm (G,)) of one bin at the points D > 0"""
    D = np.asarray(D, dtype=np.float64)
    sp, sq = tails(alpha, beta, D)
    n = len(beta)
    F, G = sq / n, sp / n
    x = np.where(F <= 0.5, ndtri(F), -ndtri(G))
    lp = alpha * np.log(beta[:, None] / D[None, :]) - beta[:, None] / D[None, :] - gammaln(alpha) - np.log(D)[None, :]
    logm = logsumexp(lp, axis=0) - np.log(n)
    return x, logm


def bin_params(sigma, edges, key):
    """[(alpha, beta (N,)) per bin] of the BR marginal of `key`: its inverse gamma, or for TT / EE of a joint sigma (with "TE")
    the inverse-Wishart diagonal IG((nu - 1)/2, Psi_jj / 2)"""
    if "TE" in sigma and key in ("TT", "EE"):
        nu, psi = B.iw_nu_psi(sigma["TT"], sigma["TE"], sigma["EE"], edges)
        j = 0 if key == "TT" else 2
        return [(0.5 * (nu[b] - 1), 0.5 * psi[:, b, j]) for b in range(len(nu))]
    a, be = B.ig_alpha_beta(sigma[key], edges)
    return [(a[b], be[:, b]) for b in range(len(a))]


def gaussianize(sigma, edges, dls, keys):
    """dls: {key: (M, nb_key)} of the evaluated bins -> (x (M, B), logm (M, B)), keys concatenated in order"""
    xs, ls = [], []
    for k in keys:
        for b, (a, be) in enumerate(bin_params(sigma, edges[k], k)):
            x, lm = transform(a, be, dls[k][:, b])
            xs.append(x)
            ls.append(lm)
    return np.stack(xs, 1), np.stack(ls, 1)


def fit(x):
    """mu, Sigma of the Gaussianized chain rows x (n, B)"""
    return x.mean(0), np.cov(x, rowvar=False, ddof=1).reshape(x.shape[1], x.shape[1])


def logpdf_x(x, logm, mu, cov):
    """log N(x; mu, Sigma) + sum_b (logm_b - log phi(x_b))"""
    r = x - mu
    Bn = x.shape[1]
    sign, ld = np.linalg.slogdet(cov)
    q = np.einsum("mi,ij,mj->m", r, np.linalg.inv(cov), r)
    lnorm = -0.5 * (q + ld + Bn * np.log(2 * np.pi))
    lphi = -0.5 * x * x - 0.5 * np.log(2 * np.pi)
    return lnorm + (logm - lphi).sum(1)


def logpdf(sigma, edges, chain_dls, dls, keys):
    """Gaussianized BR log L of the models dls fitted on the chain rows chain_dls (both {key: (rows, nb_key)} of the evaluated
    bins; chain row i pairs with sigma row i)"""
    xc, _ = gaussianize(sigma, edges, chain_dls, keys)
    mu, cov = fit(xc)
    x, lm = gaussianize(sigma, edges, dls, keys)
    return logpdf_x(x, lm, mu, cov)
