"""Blackwell-Rao estimator of the power-spectrum posterior from Gibbs chains (Wandelt, Larson & Lakshminarayanan 2004;
Chu et al. 2005).  The reference has no BR code.

    p(D | d) ~ (1/N) sum_i p(D | sigma^i)

sigma^i is the empirical spectrum of the i-th sky sample of a chain (`keep_sigma=True` on CenteredGibbs / JointGibbs records
it) and p(D | sigma) the C_l conditional the chain draws from, in D units: the binned inverse-gamma of gs_cls_invgamma for
TT, EE and BB, and the (TT, TE; TE, EE) inverse-Wishart of gs_cls_invwishart_binned plus the inverse-gamma BB of the joint
sampler.  Every conditional corresponds to a flat prior on D_b, so the estimate is the normalised posterior density and
equals the likelihood up to a constant.  The sum over samples runs on the device as one fused FP64 GEMM + log-mean-exp
(gs_br_logmeanexp, include/gibbs_b200.h): the N x M matrix of log-densities is never formed.

GaussianizedBlackwellRao (Rudjord et al. 2009) joins the one-dimensional BR marginals, which converge where the multivariate sum
does not, by a Gaussian copula fitted to the chain; its mixture-CDF transform is gs_gbr_transform."""
import numpy as np
import torch

from . import _dev, _lib
from ._dev import f64, ptr, stream
from ._lib import check, GS_BR_IG, GS_BR_IW


def _edges(e, ncl, key):
    """Host validation of one set of bin edges of a chain with ncl = lmax + 1 multipoles."""
    e = np.asarray(e)
    if e.ndim != 1 or e.size < 4 or not np.issubdtype(e.dtype, np.integer):
        raise ValueError("bins[%r] must be a 1-d integer array of at least 4 edges (bins 0 and 1 are not evaluated)" % key)
    e = e.astype(np.int64)
    if np.any(np.diff(e) <= 0):
        raise ValueError("bins[%r] must be strictly ascending" % key)
    if e[0] < 0 or e[-1] > ncl:
        raise ValueError("bins[%r] must lie in [0, %d] (sigma holds l = 0 .. %d)" % (key, ncl, ncl - 1))
    return e


def _is_host(x):
    return not isinstance(x, torch.Tensor)


class BlackwellRao:
    """BlackwellRao(sigma, bins, *, burn_in=0).

    sigma: a dict of (n_iter, lmax + 1) empirical spectra per sample (a chain's `sigma_history`), or a list of such dicts
    (several chains: each loses its first `burn_in` rows, then they are concatenated).  Keys: "TT" and / or "EE", "BB" for
    independent inverse-gamma spectra; "TT", "TE", "EE", "BB" (the joint sampler) for the inverse-Wishart TT/TE/EE block on the
    TT edges plus an inverse-gamma BB on the BB edges.
    bins: the chain's edges: None (one multipole per bin, edges 0 .. lmax + 1), one edge array for every key, or a dict of
    edges per key (joint: "TT" and "BB", as JointGibbs).  The chains' bins 0 and 1 are fixed at D = 0 and are not evaluated.
    Inputs may be numpy arrays or CUDA tensors; results come back as numpy arrays or CUDA tensors like the input of each call."""

    def __init__(self, sigma, bins, *, burn_in=0):
        chains, burn_in = self._validate(sigma, bins, burn_in)
        self.sigma = {k: torch.cat([f64(c[k])[burn_in:] for c in chains]).contiguous() for k in self.keys}
        self._feat = {}
        self._features(None)     # the full set of bins, built once

    def _validate(self, sigma, bins, burn_in):
        """host checks of sigma, bins and burn_in; sets keys, edges, groups, nbins, ncl, lmax and n -> (chains, burn_in)"""
        chains = [sigma] if isinstance(sigma, dict) else list(sigma)
        if not chains or not all(isinstance(c, dict) and c for c in chains):
            raise ValueError("sigma must be a non-empty dict of spectra or a list of such dicts")
        keys = tuple(chains[0])
        if any(set(c) != set(keys) for c in chains):
            raise ValueError("every chain must hold the same spectra, got %s" % [sorted(c) for c in chains])
        self.joint = "TE" in keys
        if self.joint and set(keys) != {"TT", "TE", "EE", "BB"}:
            raise ValueError("a joint sigma (with 'TE') needs exactly the keys TT, TE, EE, BB, got %s" % sorted(keys))
        if not self.joint and not set(keys) <= {"TT", "EE", "BB"}:
            raise ValueError("sigma keys must be among TT, EE, BB (or TT, TE, EE, BB for the joint sampler), got %s" % sorted(keys))
        burn_in = int(burn_in)
        if burn_in < 0:
            raise ValueError("burn_in must be >= 0")
        self.keys = ("TT", "TE", "EE", "BB") if self.joint else keys
        ncl = None
        for c in chains:
            n_iter = None
            for k in self.keys:
                s = c[k] if isinstance(c[k], torch.Tensor) else np.asarray(c[k])
                if len(s.shape) != 2:
                    raise ValueError("sigma[%r] must be a 2-d (n_iter, lmax + 1) array" % k)
                shape = tuple(s.shape)
                ncl = shape[1] if ncl is None else ncl
                n_iter = shape[0] if n_iter is None else n_iter
                if shape != (n_iter, ncl):
                    raise ValueError("sigma[%r] has shape %s, expected (%d, %d)" % (k, shape, n_iter, ncl))
            if n_iter <= burn_in:
                raise ValueError("burn_in = %d leaves no sample of a chain of %d iterations" % (burn_in, n_iter))
        self.ncl, self.lmax = int(ncl), int(ncl) - 1
        if self.joint:
            from .JointSampler import _joint_bins
            jb = _joint_bins({"TT": np.arange(ncl + 1), "BB": np.arange(ncl + 1)} if bins is None else bins, self.lmax)
            self.edges = {"TT": jb["TT"], "TE": jb["TT"], "EE": jb["TT"], "BB": jb["BB"]}
            self.groups = [(GS_BR_IW, ("TT", "TE", "EE")), (GS_BR_IG, ("BB",))]
        else:
            if bins is None:
                bins = np.arange(ncl + 1)
            self.edges = {k: _edges(bins[k] if isinstance(bins, dict) else bins, ncl, k) for k in self.keys}
            self.groups = [(GS_BR_IG, (k,)) for k in self.keys]
        self.nbins = {k: len(e) - 1 for k, e in self.edges.items()}
        self.n = sum(int(c[self.keys[0]].shape[0]) - burn_in for c in chains)
        return chains, burn_in

    @classmethod
    def from_sampler(cls, gibbs, burn_in=0):
        """The estimator of a chain run with keep_sigma=True (CenteredGibbs or JointGibbs)."""
        sig = getattr(gibbs, "sigma_history", None)
        if sig is None:
            raise ValueError("the sampler has no sigma_history: construct it with keep_sigma=True and call run()")
        bins = gibbs.bins
        if isinstance(bins, dict) and "TE" not in sig:
            bins = {k: bins[k] for k in sig}
        return cls(sig, bins, burn_in=burn_in)

    # ------------------------------------------------------------------ bin selection and sample features
    def _selection(self, lrange):
        """-> tuple of (first bin, end bin) per group (bins >= 2 that lie inside lrange = (lmin, lmax), inclusive)."""
        sel = []
        for _, keys in self.groups:
            e = self.edges[keys[0]]
            if lrange is None:
                sel.append((2, len(e) - 1))
                continue
            lo, hi = int(lrange[0]), int(lrange[1])
            inside = [b for b in range(2, len(e) - 1) if e[b] >= lo and e[b + 1] - 1 <= hi]
            for b in range(2, len(e) - 1):
                if b not in inside and e[b] <= hi and e[b + 1] - 1 >= lo:
                    raise ValueError("lrange %s cuts bin %d = [%d, %d] of %s: lrange must select whole bins"
                                     % ((lo, hi), b, e[b], e[b + 1] - 1, "/".join(keys)))
            sel.append((inside[0], inside[-1] + 1) if inside else (0, 0))
        if all(b1 == b0 for b0, b1 in sel):
            raise ValueError("lrange %s selects no bin" % (lrange,))
        return tuple(sel)

    def _features(self, lrange):
        sel = self._selection(lrange)
        if sel in self._feat:
            return self._feat[sel]
        rows = [(3 if kind == GS_BR_IW else 1) * (b1 - b0) for (kind, _), (b0, b1) in zip(self.groups, sel)]
        K = sum(rows)
        dev = self.sigma[self.keys[0]].device
        S = torch.empty((K, self.n), dtype=torch.float64, device=dev)
        c = torch.empty(self.n, dtype=torch.float64, device=dev)
        scratch = torch.empty(max(b1 - b0 for b0, b1 in sel) * self.n, dtype=torch.float64, device=dev)
        L, r0, first = _lib.lib(), 0, True
        edges_dev = []
        for (kind, keys), (b0, b1), nr in zip(self.groups, sel, rows):
            if b1 == b0:
                edges_dev.append(None)
                continue
            e = _dev.i32(self.edges[keys[0]][b0:b1 + 1])
            edges_dev.append(e)
            s = [self.sigma[k] for k in keys] + [None] * (3 - len(keys))
            check(L.gs_br_sample_features(kind, ptr(s[0]), ptr(s[1]), ptr(s[2]), self.n, self.ncl, ptr(e), b1 - b0, ptr(S[r0]), ptr(c),
                                          0 if first else 1, ptr(scratch), stream()))
            r0 += nr
            first = False
        f = {"sel": sel, "S": S, "c": c, "K": K, "edges": edges_dev, "rows": rows}
        # the features of all bins are kept; of the lrange selections only the latest, so that a scan over many ranges does not
        # pile up K x N matrices on the device
        full = self._selection(None)
        self._feat = {k: v for k, v in self._feat.items() if k == full}
        self._feat[sel] = f
        return f

    # ------------------------------------------------------------------ estimator
    def _dls(self, dls, keys=None):
        keys = self.keys if keys is None else keys
        if set(dls) != set(keys):
            raise ValueError("dls must hold the keys %s, got %s" % (sorted(keys), sorted(dls)))
        out, m, one = {}, None, None
        for k in keys:
            d = f64(dls[k])
            if d.dim() not in (1, 2) or d.shape[-1] != self.nbins[k]:
                raise ValueError("dls[%r] must have shape (%d,) or (M, %d), got %s" % (k, self.nbins[k], self.nbins[k], tuple(d.shape)))
            one = d.dim() == 1 if one is None else one
            if (d.dim() == 1) != one:
                raise ValueError("dls entries must all be 1-d or all 2-d")
            d = d.reshape(-1, self.nbins[k])
            m = d.shape[0] if m is None else m
            if d.shape[0] != m or m < 1:
                raise ValueError("dls entries must hold the same number M >= 1 of models")
            out[k] = d
        return out, m, one

    def logpdf(self, dls, *, lrange=None, n_eff=False):
        """log of the BR estimate at the binned D of each model: dls = {key: (nbins,) or (M, nbins)} in the chain's bins (all of
        them, bins 0 and 1 included and ignored).  lrange = (lmin, lmax) evaluates only the bins that lie inside it (a bin it cuts
        raises ValueError).  A model with some D_b <= 0, or an IW block that is not positive definite, gets -inf.  n_eff=True
        also returns the effective sample size (sum w)^2 / sum w^2 of each model, w_i = the sample's share of the estimate."""
        host = _is_host(next(iter(dls.values())))
        d, M, one = self._dls(dls)
        f = self._features(lrange)
        dev, K = f["S"].device, f["K"]
        W = torch.empty((K, M), dtype=torch.float64, device=dev)
        e = torch.empty(M, dtype=torch.float64, device=dev)
        nbmax = max(b1 - b0 for b0, b1 in f["sel"])
        scratch = torch.empty(max(nbmax * M, self._lme_scratch(M)), dtype=torch.float64, device=dev)
        L, r0, first, cols = _lib.lib(), 0, True, []
        for (kind, keys), (b0, b1), nr, ed in zip(self.groups, f["sel"], f["rows"], f["edges"]):
            if b1 == b0:
                continue
            x = [d[k][:, b0:b1].contiguous() for k in keys] + [None] * (3 - len(keys))
            cols.append(x)
            check(L.gs_br_model_features(kind, ptr(x[0]), ptr(x[1]), ptr(x[2]), M, self.ncl, ptr(ed), b1 - b0, ptr(W[r0]), ptr(e),
                                         0 if first else 1, ptr(scratch), stream()))
            r0 += nr
            first = False
        logl = torch.empty(M, dtype=torch.float64, device=dev)
        neff = torch.empty(M, dtype=torch.float64, device=dev) if n_eff else None
        check(L.gs_br_logmeanexp(ptr(f["S"]), ptr(f["c"]), self.n, ptr(W), ptr(e), M, K, ptr(scratch), ptr(logl), ptr(neff), stream()))
        res = [logl] + ([neff] if n_eff else [])
        if one:
            res = [r[0] for r in res]
        if host:
            res = [r.cpu().numpy() for r in res]
        return tuple(res) if n_eff else res[0]

    def _lme_scratch(self, M):
        """doubles of scratch gs_br_logmeanexp needs (the library owns the split of the sample axis)"""
        return int(_lib.lib().gs_br_logmeanexp_scratch(self.n, M))

    def _group_of(self, key):
        """-> (group index, kind, comp) of a TT, EE or BB key; TE has no marginal"""
        if key not in self.keys:
            raise ValueError("no spectrum %r (have %s)" % (key, sorted(self.keys)))
        if key == "TE":
            raise ValueError("the TE marginal is not available (only TT, EE and BB)")
        gi = next(i for i, (_, keys) in enumerate(self.groups) if key in keys)
        kind, keys = self.groups[gi]
        return gi, kind, 0 if kind == GS_BR_IG else keys.index(key)

    def _transform(self, key, d, lrange=None):
        """gs_gbr_transform of the (M, nbins of the selection) D of one key on the bins lrange selects -> (x, logm), CUDA tensors"""
        gi, kind, comp = self._group_of(key)
        f = self._features(lrange)
        b0, b1 = f["sel"][gi]
        M, nb = d.shape[0], b1 - b0
        x = torch.empty((M, nb), dtype=torch.float64, device=d.device)
        logm = torch.empty_like(x)
        L = _lib.lib()
        scratch = torch.empty(int(L.gs_gbr_transform_scratch(self.n, M, nb)), dtype=torch.float64, device=d.device)
        check(L.gs_gbr_transform(kind, ptr(f["S"][sum(f["rows"][:gi])]), self.n, self.ncl, ptr(f["edges"][gi]), nb, comp,
                                 ptr(d.contiguous()), M, ptr(x), ptr(logm), ptr(scratch), stream()))
        return x, logm

    def cdf(self, key, grid):
        """Per-bin BR marginal CDF P(D_b <= g | d) = (1/N) sum_i Q(alpha, beta_i / g) on a grid laid out as for marginal(): grid (G,)
        or (nbins, G) -> (nbins, G), rows of the bins 0 and 1 NaN.  Computed by gs_gbr_transform as Phi(x), so both tails keep
        their relative accuracy."""
        self._group_of(key)
        host = _is_host(grid)
        g = f64(grid)
        nb = self.nbins[key]
        if g.dim() == 1:
            d = g[:, None].expand(g.shape[0], nb - 2)
        elif g.dim() == 2 and g.shape[0] == nb:
            d = g[2:].T
        else:
            raise ValueError("grid must have shape (G,) or (%d, G), got %s" % (nb, tuple(g.shape)))
        if d.shape[0] < 1:
            raise ValueError("grid is empty")
        x, _ = self._transform(key, d.contiguous())
        out = torch.full((nb, d.shape[0]), float("nan"), dtype=torch.float64, device=g.device)
        out[2:] = torch.special.ndtr(x).T
        return out.cpu().numpy() if host else out

    def marginal(self, key, grid):
        """Per-bin BR marginal log p(D_b = g | d) on a grid: grid (G,) for every bin or (nbins, G) per bin; -> (nbins, G), rows of
        the bins 0 and 1 NaN.  IG spectra use their inverse-gamma; TT and EE of the joint block the marginal of a diagonal entry of
        the inverse-Wishart, IG((nu - 1)/2, Psi_jj / 2).  The TE marginal is not built."""
        if key not in self.keys:
            raise ValueError("no spectrum %r (have %s)" % (key, sorted(self.keys)))
        if key == "TE":
            raise ValueError("the TE marginal is not available (only TT, EE and BB)")
        host = _is_host(grid)
        g = f64(grid)
        nb = self.nbins[key]
        if g.dim() == 1:
            ld, G = 0, g.shape[0]
        elif g.dim() == 2 and g.shape[0] == nb:
            ld, G = g.shape[1], g.shape[1]
            g = g[2:].contiguous()
        else:
            raise ValueError("grid must have shape (G,) or (%d, G), got %s" % (nb, tuple(g.shape)))
        if G < 1:
            raise ValueError("grid is empty")
        f = self._features(None)
        gi = next(i for i, (_, keys) in enumerate(self.groups) if key in keys)
        kind, keys = self.groups[gi]
        r0 = sum(f["rows"][:gi])
        comp = 0 if kind == GS_BR_IG else keys.index(key)
        out = torch.full((nb, G), float("nan"), dtype=torch.float64, device=g.device)
        check(_lib.lib().gs_br_marginal(kind, ptr(f["S"][r0]), self.n, self.ncl, ptr(f["edges"][gi]), nb - 2, comp, ptr(g), ld, G,
                                        ptr(out[2]), stream()))
        return out.cpu().numpy() if host else out


def _history_rows(h, keys, chain):
    """the (n_iter + 1, nbins) D history of each key of one chain: a dict (polarised and joint samplers) or an array (TT)"""
    if isinstance(h, tuple):                  # CenteredGibbs.run() returns (history, ...)
        h = h[0]
    if not isinstance(h, dict):
        if keys != ("TT",):
            raise ValueError("dls of chain %d must be a dict of D histories with the keys %s" % (chain, sorted(keys)))
        h = {"TT": h}
    missing = [k for k in keys if k not in h]
    if missing:
        raise ValueError("dls of chain %d has no history for %s" % (chain, missing))
    return {k: h[k] for k in keys}


class GaussianizedBlackwellRao:
    """GaussianizedBlackwellRao(sigma, dls, bins, *, burn_in=0): the Gaussianized Blackwell-Rao likelihood of Rudjord et al. (2009).

    Each bin b is mapped through its own BR marginal, x_b = Phi^-1(F_b(D_b)) with F_b(D) = (1/N) sum_i F_IG(D; alpha_b, beta_b^i), and
    the bins are joined by a Gaussian copula fitted to the chain's own D samples:
        log L(D) = log N(x; mu, Sigma) + sum_b [log p_b(D_b) - log phi(x_b)],
    p_b the BR marginal density (so dx_b / dD_b = p_b / phi(x_b)).  Unlike BlackwellRao.logpdf it needs only the one-dimensional
    marginals to converge, so it stays usable when the multivariate BR sum rests on a handful of samples (many bins).

    sigma, bins, burn_in: as BlackwellRao (its validation, bins and sample features are used as they are).  dls: the D histories
    run() returned, in the same layout as sigma (a dict, a list of dicts, or a TT array per chain); a history has n_iter + 1 rows.
    Row alignment: sigma row i is the sky that D row i + 1 was drawn from, so after burn_in, mu and Sigma come from the D rows
    burn_in + 1 ... n_iter of every chain.  Spectra: TT, EE, BB of CenteredGibbs; TT, EE, BB of JointGibbs, TT and EE through the
    inverse-Wishart diagonal marginal, so TE is marginalised (a "TE" model entry raises ValueError).  The transform runs on the
    device (gs_gbr_transform); mu and Sigma are FP64, and the Cholesky factor of every lrange selection's sub-matrix is kept."""

    def __init__(self, sigma, dls, bins, *, burn_in=0):
        # every check runs on the host before anything reaches the device
        br = self.br = BlackwellRao.__new__(BlackwellRao)
        chains, burn_in = br._validate(sigma, bins, burn_in)
        self.keys = ("TT", "EE", "BB") if br.joint else br.keys
        hists = [dls] if isinstance(dls, (dict, tuple, np.ndarray, torch.Tensor)) else list(dls)
        if len(hists) != len(chains):
            raise ValueError("dls holds %d chains, sigma %d" % (len(hists), len(chains)))
        hists = [_history_rows(h, self.keys, i) for i, h in enumerate(hists)]
        for i, (s, h) in enumerate(zip(chains, hists)):
            n_iter = int(s[br.keys[0]].shape[0])
            for k in self.keys:
                shape = tuple(np.shape(h[k]))
                if shape != (n_iter + 1, br.nbins[k]):
                    raise ValueError("dls[%r] of chain %d has shape %s, expected (%d, %d): the D history of a chain of %d iterations"
                                     % (k, i, shape, n_iter + 1, br.nbins[k], n_iter))
        # the Gaussianized chain, bins 2 .. nbins - 1 of every key in key order
        self._cols, c0 = {}, 0
        for k in self.keys:
            self._cols[k] = c0
            c0 += br.nbins[k] - 2
        B, n = c0, br.n
        if n < B + 1:
            raise ValueError("%d samples after burn_in for %d bins: the copula covariance needs at least %d" % (n, B, B + 1))
        br.sigma = {k: torch.cat([f64(c[k])[burn_in:] for c in chains]).contiguous() for k in br.keys}
        br._feat = {}
        X = torch.empty((n, B), dtype=torch.float64, device=br.sigma[br.keys[0]].device)
        for k in self.keys:
            d = torch.cat([f64(h[k])[burn_in + 1:] for h in hists])[:, 2:].contiguous()
            X[:, self._cols[k]:self._cols[k] + d.shape[1]] = self.br._transform(k, d)[0]
        bad = int((~torch.isfinite(X)).sum())
        if bad:
            raise ValueError("%d of the chain's %d Gaussianized values are not finite" % (bad, X.numel()))
        self.mean = X.mean(0)
        Xc = X - self.mean
        self.cov = (Xc.T @ Xc) / (n - 1)
        self.nbins = B
        self._chol = {}
        self._factor(None)

    @classmethod
    def from_sampler(cls, gibbs, history, burn_in=0):
        """The likelihood of a chain run with keep_sigma=True (CenteredGibbs or JointGibbs); history = what its run() returned."""
        sig = getattr(gibbs, "sigma_history", None)
        if sig is None:
            raise ValueError("the sampler has no sigma_history: construct it with keep_sigma=True and call run()")
        bins = gibbs.bins
        if isinstance(bins, dict) and "TE" not in sig:
            bins = {k: bins[k] for k in sig}
        return cls(sig, history, bins, burn_in=burn_in)

    def _factor(self, lrange):
        """-> (selection, column index, Cholesky factor of the sub-matrix of Sigma) of the bins lrange selects"""
        sel = self.br._selection(lrange)
        if sel in self._chol:
            return self._chol[sel]
        idx = []
        for k in self.keys:
            gi = self.br._group_of(k)[0]
            b0, b1 = sel[gi]
            idx += [self._cols[k] + b - 2 for b in range(b0, b1)]
        idx = torch.as_tensor(idx, dtype=torch.long, device=self.cov.device)
        L, info = torch.linalg.cholesky_ex(self.cov[idx][:, idx])
        if int(info):
            raise ValueError("the copula covariance of %d bins is not positive definite (leading minor %d)" % (len(idx), int(info)))
        self._chol[sel] = (sel, idx, L)
        return self._chol[sel]

    def gaussianize(self, key, dls):
        """x = Phi^-1(F_b(D_b)) of one spectrum: dls (nbins,) or (M, nbins) -> the same shape, columns of the bins 0 and 1 NaN"""
        if key not in self.keys:
            raise ValueError("no spectrum %r (have %s)" % (key, sorted(self.keys)))
        host = _is_host(dls)
        d = f64(dls)
        nb = self.br.nbins[key]
        if d.dim() not in (1, 2) or d.shape[-1] != nb or d.numel() == 0:
            raise ValueError("dls must have shape (%d,) or (M, %d), got %s" % (nb, nb, tuple(d.shape)))
        d2 = d.reshape(-1, nb)
        out = torch.full(d2.shape, float("nan"), dtype=torch.float64, device=d.device)
        out[:, 2:] = self.br._transform(key, d2[:, 2:].contiguous())[0]
        out = out.reshape(d.shape)
        return out.cpu().numpy() if host else out

    def logpdf(self, dls, *, lrange=None):
        """Gaussianized BR log-likelihood of each model, in the layout of BlackwellRao.logpdf (keys TT / EE / BB, (nbins,) or
        (M, nbins), bins 0 and 1 ignored, lrange selecting whole bins).  A model with some D_b <= 0, or one so far out that F_b or
        1 - F_b is 0 in FP64, gets -inf; broken input (NaN) gives NaN."""
        if "TE" in dls and self.br.joint:
            raise ValueError("TE is marginalised in the Gaussianized BR likelihood: pass TT, EE and BB only")
        self.br._selection(lrange)          # a cut bin raises before any device work
        host = _is_host(next(iter(dls.values())))
        d, M, one = self.br._dls(dls, self.keys)
        sel, idx, L = self._factor(lrange)
        xs, lms = [], []
        for k in self.keys:
            b0, b1 = sel[self.br._group_of(k)[0]]
            if b1 == b0:
                continue
            x, lm = self.br._transform(k, d[k][:, b0:b1], lrange)
            xs.append(x)
            lms.append(lm)
        x, lm = torch.cat(xs, 1), torch.cat(lms, 1)
        z = torch.linalg.solve_triangular(L, (x - self.mean[idx]).T, upper=False)
        out = -0.5 * (z * z).sum(0) - torch.log(torch.diagonal(L)).sum() + (lm + 0.5 * x * x).sum(1)
        finite = torch.isfinite(x).all(1) & torch.isfinite(lm).all(1)
        nan = torch.isnan(x).any(1) | torch.isnan(lm).any(1)
        out = torch.where(finite, out, torch.full_like(out, -float("inf")))
        out = torch.where(nan, torch.full_like(out, float("nan")), out)
        if one:
            out = out[0]
        return out.cpu().numpy() if host else out
