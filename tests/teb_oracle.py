"""numpy restatement of the joint T/E/B masked-sky constrained realization (TEST INFRASTRUCTURE ONLY): qcinv's joint T+P
filter (opfilt_tp upstream, not vendored), built from the TT and E/B restatements of oracle.reference_logic (TTProblem,
PolProblem, on the long-double transforms of oracle.sht) plus the 2x2 TE block of the prior.  The library's twin is
gs_cr_rhs_teb / gs_cr_pcg_teb / gs_cr_apply_q_teb (include/gibbs_b200.h)."""
import numpy as np

from oracle.reference_logic import PolProblem, TTProblem, adjoint_pol, l_of_real_layout, safe_inv


# ---------------------------------------------------------------- joint T/E/B on a cut sky (gs_cr_*_teb)
def te_blocks(dls, lmax):
    """per-l C_l of the (T, E) block and of B, D_l -> C_l with l = 0 copied unscaled (generate_var_cl)"""
    f = np.array([2 * np.pi / (l * (l + 1)) if l else 1.0 for l in range(lmax + 1)])
    return tuple(np.asarray(dls[k], dtype=np.float64) * f for k in ("TT", "TE", "EE", "BB"))


def inv_2x2_safe(a, b, d):
    """inverse of [[a, b], [b, d]] per l; C^TE = 0 -> field by field with safe_inv; zero determinant -> zeros"""
    i11, i12, i22 = safe_inv(a), np.zeros(len(a)), safe_inv(d)
    c = b != 0
    det = a[c] * d[c] - b[c] ** 2
    idet = safe_inv(det)
    i11[c], i12[c], i22[c] = d[c] * idet, -b[c] * idet, a[c] * idet
    return i11, i12, i22


class TPProblem:
    """Inputs of the joint T/E/B masked-sky CR step: qcinv's joint T+P filter (opfilt_tp upstream, not vendored), restated
    from the TT (TTProblem) and E/B (PolProblem) systems plus the 2x2 TE block of the prior:
        Q = C^-1 + B A^T N^-1 A B,  N^-1 = diag(N_T^-1, N_P^-1, N_P^-1) on (I, Q, U),
        b = B A^T N^-1 d + B (Npix/4pi) map2alm_iter(N^-1/2 xi_pix) + F xi_alm,  F = L^-T (C^TE block = L L^T), 1/sqrt(C^BB).
    Vectors are (T, E, B) tuples in the real layout; dls = {"TT", "TE", "EE", "BB"} unbinned D_l."""

    def __init__(self, nside, lmax, d_I, d_Q, d_U, inv_noise_T, inv_noise_P, fwhm_deg, kind="ld"):
        self.nside, self.lmax = nside, lmax
        self.n = (lmax + 1) ** 2
        self.tt = TTProblem(nside, lmax, d_I, inv_noise_T, fwhm_deg, kind)
        self.pol = PolProblem(nside, lmax, d_Q, d_U, inv_noise_P, fwhm_deg, kind)
        self.inv_noise_T, self.inv_noise_P = inv_noise_T, inv_noise_P
        self.bl_gauss, self.bl_map = self.tt.bl_gauss, self.tt.bl_map
        self.ell = l_of_real_layout(lmax)
        self.bdata = (self.tt.bdata, self.pol.bdata_E, self.pol.bdata_B)

    def inv_cov(self, dls):
        """per-l (ic_TT, ic_TE, ic_EE, ic_BB)"""
        a, b, d, e = te_blocks(dls, self.lmax)
        return inv_2x2_safe(a, b, d) + (safe_inv(e),)

    def factor(self, dls):
        """per-l (f_TT, f_TE, f_EE, f_BB) of F = L^-T: T gets f_TT xi_T + f_TE xi_E, E gets f_EE xi_E, B gets f_BB xi_B"""
        a, b, d, e = te_blocks(dls, self.lmax)
        fTT, fTE, fEE = np.sqrt(safe_inv(a)), np.zeros(len(a)), np.sqrt(safe_inv(d))
        c = b != 0
        for l in np.nonzero(c)[0]:
            L = np.linalg.cholesky(np.array([[a[l], b[l]], [b[l], d[l]]]))
            F = np.linalg.inv(L).T
            fTT[l], fTE[l], fEE[l] = F[0, 0], F[0, 1], F[1, 1]
        return fTT, fTE, fEE, np.sqrt(safe_inv(e))

    def block_mul(self, blk, x):
        i11, i12, i22, ibb = (np.asarray(v)[self.ell] for v in blk)
        xT, xE, xB = x
        return i11 * xT + i12 * xE, i12 * xT + i22 * xE, ibb * xB

    def noise_op(self, x):
        """B A^T N^-1 A B x: the spin-0 operator on N_T^-1 and the spin-2 operator on N_P^-1"""
        xT, xE, xB = x
        z = np.zeros(self.n)
        yT = self.tt.apply_Q(z, xT)                                     # safe_inv(0) = 0: noise part only
        yE, yB = self.pol.apply_Q(None, None, xE, xB, inv_var=(z, z))
        return yT, yE, yB

    def apply_Q(self, dls, x, ic=None):
        ic = self.inv_cov(dls) if ic is None else ic
        return tuple(u + v for u, v in zip(self.noise_op(x), self.block_mul(ic, x)))

    def rhs(self, dls, xi_I, xi_Q, xi_U, xi_T, xi_E, xi_B, fluct_iter=3):
        fT = self.bl_map * self.tt.adjoint(xi_I * np.sqrt(self.inv_noise_T), fluct_iter)
        sP = np.sqrt(self.inv_noise_P)
        fE, fB = adjoint_pol(xi_Q * sP, xi_U * sP, self.nside, self.lmax, fluct_iter, self.pol.kind)
        f = [np.asarray(v)[self.ell] for v in self.factor(dls)]
        return (fT + f[0] * xi_T + f[1] * xi_E + self.bdata[0],
                fE * self.bl_map + f[2] * xi_E + self.bdata[1],
                fB * self.bl_map + f[3] * xi_B + self.bdata[2])

    def precond(self, dls):
        """per-l diag_cl block M_l = (C_l^-1 + diag(b^2 nT, b^2 nP, b^2 nP))^-1, nX = sum(N_X^-1) / (4 pi)"""
        i11, i12, i22, ibb = self.inv_cov(dls)
        b2 = self.bl_gauss ** 2
        nT, nP = np.sum(self.inv_noise_T) / (4 * np.pi), np.sum(self.inv_noise_P) / (4 * np.pi)
        return inv_2x2_safe(i11 + b2 * nT, i12, i22 + b2 * nP) + (safe_inv(ibb + b2 * nP),)

    def pcg(self, dls, b, eps=1e-6, itermax=4000, x0=None):
        """PCG with monitor_basic on the joint vector: stop when <r,r> <= eps^2 <r0,r0> (sums over T, E and B)"""
        M, ic = self.precond(dls), self.inv_cov(dls)
        cat = np.concatenate

        def split(v):
            return v[:self.n], v[self.n:2 * self.n], v[2 * self.n:]
        bv = cat(b)
        x = np.zeros(3 * self.n) if x0 is None else cat(x0)
        r = bv - cat(self.apply_Q(dls, split(x), ic)) if x0 is not None else bv.copy()
        d0 = r @ r
        z = cat(self.block_mul(M, split(r)))
        p = z.copy()
        delta = r @ z
        it = 0
        while it < itermax and r @ r > eps ** 2 * d0:
            q = cat(self.apply_Q(dls, split(p), ic))
            alpha = delta / (p @ q)
            x += alpha * p
            r -= alpha * q
            z = cat(self.block_mul(M, split(r)))
            dn = r @ z
            p = z + (dn / delta) * p
            delta = dn
            it += 1
        return split(x), it

    def dense_Q(self, dls):
        n3 = 3 * self.n
        Q = np.zeros((n3, n3))
        ic = self.inv_cov(dls)
        for i in range(n3):
            v = np.zeros(n3)
            v[i] = 1
            Q[:, i] = np.concatenate(self.apply_Q(dls, (v[:self.n], v[self.n:2 * self.n], v[2 * self.n:]), ic))
        return Q
