// Per-multipole 3x3 TT/TE/EE/BB machinery (SURVEY.md 8a row A9, 8f row 4; BASELINE north_star (c)).
//
// Replaces variance_expension.generate_polarization_var_cl_cython (variance_expension.pyx:36-61), the
// recovered utils.compute_inverse_and_cholesky / utils.matrix_product and the deleted native module
// linear_algebra.pyx (LAPACK dgesv/dpotrf/dpotri per l; SURVEY.md 2.3) by closed-form 3x3 algebra with one
// thread per multipole (or per coefficient), and adds the inverse-Wishart draw the reference intended for
// the TT/TE/EE block (.ipynb_checkpoints/main-checkpoint.py:39-44, 333-346: df = 2l - 2, scale = (2l+1) Chat_l), per multipole
// or, with D_l constant on each bin as in the reference's binned EE/BB (CenteredGibbs.py:54-79), per bin.
// All arrays are row-major: per-l matrices (L+1,3,3), per-coefficient matrices ((L+1)^2,3,3), vectors
// ((L+1)^2,3) with component order (T, E, B).
#include <algorithm>

#include "gs_internal.h"
#include "rng.cuh"
#include "spectra.cuh"

#define TB_NT 256
static inline int tb_blocks(int64_t n) { return (int)std::max<int64_t>(1, std::min<int64_t>((n + TB_NT - 1) / TB_NT, 148 * 16)); }

// ---- variance_expension.pyx:36-61: (L+1,3,3) D_l -> ((L+1)^2,3,3) C_l over the real alm layout.
// The reference indexes cls_[idx] instead of cls_[l] at :51 and raises IndexError (SURVEY.md 8c); the
// intended per-l lookup is implemented.  l = 0 is copied unscaled, as in the scalar twin (:23-27).
__global__ void expand_var_cl_3x3_kernel(const double* __restrict__ dls, int L, double* __restrict__ out)
{
    const int64_t n = (int64_t)(L + 1) * (L + 1) * 9;
    for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < n; t += (int64_t)gridDim.x * blockDim.x) {
        const int64_t i = t / 9;
        const int e = (int)(t - i * 9);
        const int l = l_of_real(i, L);
        out[t] = dl_to_cl(dls[l * 9 + e], l);
    }
}

// ---- utils.compute_inverse_and_cholesky (recovered): for l >= 2
//   M = blockdiag(inv(C[:2,:2]), 1/C[2,2]) + diag(pix_part),  Sigma = inv(M),  Lc = chol(Sigma) (lower);  l < 2: zeros.
__device__ __forceinline__ void inv_sym3(const double* a, double* o)
{  // inverse of a symmetric 3x3 (row-major) by cofactors
    const double c00 = a[4] * a[8] - a[5] * a[7], c01 = a[5] * a[6] - a[3] * a[8], c02 = a[3] * a[7] - a[4] * a[6];
    const double det = a[0] * c00 + a[1] * c01 + a[2] * c02, id = 1.0 / det;
    o[0] = c00 * id; o[1] = (a[2] * a[7] - a[1] * a[8]) * id; o[2] = (a[1] * a[5] - a[2] * a[4]) * id;
    o[3] = c01 * id; o[4] = (a[0] * a[8] - a[2] * a[6]) * id; o[5] = (a[2] * a[3] - a[0] * a[5]) * id;
    o[6] = c02 * id; o[7] = (a[1] * a[6] - a[0] * a[7]) * id; o[8] = (a[0] * a[4] - a[1] * a[3]) * id;
}

__device__ __forceinline__ void chol3(const double* a, double* l)
{  // lower Cholesky factor of a symmetric positive-definite 3x3
    const double l00 = sqrt(a[0]), l10 = a[3] / l00, l20 = a[6] / l00;
    const double l11 = sqrt(a[4] - l10 * l10), l21 = (a[7] - l20 * l10) / l11;
    const double l22 = sqrt(a[8] - l20 * l20 - l21 * l21);
    l[0] = l00; l[1] = 0.0; l[2] = 0.0; l[3] = l10; l[4] = l11; l[5] = 0.0; l[6] = l20; l[7] = l21; l[8] = l22;
}

__global__ void inv_chol_3x3_kernel(const double* __restrict__ cls, const double* __restrict__ pix_part, int L,
                                    double* __restrict__ sigma, double* __restrict__ chol)
{
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l > L) return;
    double S[9], C[9];
#pragma unroll
    for (int e = 0; e < 9; ++e) { S[e] = 0.0; C[e] = 0.0; }
    if (l >= 2) {
        const double* c = cls + (int64_t)l * 9;
        const double tt = c[0], te = c[1], ee = c[4], bb = c[8];
        const double d2 = tt * ee - te * te, id2 = 1.0 / d2;
        double M[9] = {ee * id2 + pix_part[l * 3], -te * id2, 0.0, -te * id2, tt * id2 + pix_part[l * 3 + 1], 0.0, 0.0, 0.0,
                       1.0 / bb + pix_part[l * 3 + 2]};
        inv_sym3(M, S);
        // symmetrise the rounding of the off-diagonal pair before factorising
        S[3] = S[1] = 0.5 * (S[1] + S[3]); S[6] = S[2] = 0.5 * (S[2] + S[6]); S[7] = S[5] = 0.5 * (S[5] + S[7]);
        chol3(S, C);
    }
#pragma unroll
    for (int e = 0; e < 9; ++e) { sigma[(int64_t)l * 9 + e] = S[e]; if (chol) chol[(int64_t)l * 9 + e] = C[e]; }
}

// ---- utils.matrix_product (recovered): out[i] = mats[l(i)] @ v[i] + (add ? add[i] : 0) for every real coefficient i
__global__ void matvec_3x3_kernel(const double* __restrict__ mats, const double* __restrict__ v, const double* __restrict__ add, int L,
                                  double* __restrict__ out)
{
    const int64_t n = (int64_t)(L + 1) * (L + 1);
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const double* m = mats + (int64_t)l_of_real(i, L) * 9;
        const double x = v[3 * i], y = v[3 * i + 1], z = v[3 * i + 2];
        double o0 = m[0] * x + m[1] * y + m[2] * z, o1 = m[3] * x + m[4] * y + m[5] * z, o2 = m[6] * x + m[7] * y + m[8] * z;
        if (add) { o0 += add[3 * i]; o1 += add[3 * i + 1]; o2 += add[3 * i + 2]; }
        out[3 * i] = o0; out[3 * i + 1] = o1; out[3 * i + 2] = o2;
    }
}

// ---- cross spectrum in the real layout: cl[l] = sum_entries x y / (2l+1) (= hp.alm2cl(alm1, alm2)); one warp per l
__global__ void alm2cl_cross_kernel(const double* __restrict__ x, const double* __restrict__ y, int L, double* __restrict__ cl)
{
    const int l = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (l > L) return;
    const double s = warp_sum(alm2cl_cross_real_lane(x, y, l, L, lane));
    if (lane == 0) cl[l] = s / (2.0 * l + 1.0);
}

// ---- inverse-Wishart draw of a (TT, TE; TE, EE) block, Bartlett decomposition:
//   X ~ IW(nu, Psi)   <=>   X^-1 ~ Wishart(nu, Psi^-1)
//   Psi^-1 = G G^T,  A = [[sqrt(chi2_nu), 0], [N(0,1), sqrt(chi2_{nu-1})]],  X^-1 = (G A)(G A)^T.
// Draw k (a multipole or a bin) takes row k of inject ((chi2_nu, chi2_{nu-1}, normal) supplied by the caller, parity with a numpy
// stream) or, without inject, Philox / Marsaglia-Tsang on the streams base, base + 1, base + 2 with
// base = RNG_WISHART | ((call << 22) + 4 k) (rng.cuh).
__device__ __forceinline__ void invwishart_2x2_draw(double p00, double p01, double p11, double nu, const double* __restrict__ inject, int k,
                                                    uint64_t seed, uint64_t call, double& x00, double& x01, double& x11)
{
    const double det = p00 * p11 - p01 * p01;
    const double q00 = p11 / det, q01 = -p01 / det, q11 = p00 / det;  // Psi^-1
    const double g00 = sqrt(q00), g10 = q01 / g00, g11 = sqrt(q11 - g10 * g10);  // lower Cholesky of Psi^-1
    double c1, c2, z;
    if (inject) { c1 = inject[3 * k]; c2 = inject[3 * k + 1]; z = inject[3 * k + 2]; }
    else {
        const Philox ph(seed);
        const uint64_t base = RNG_WISHART | (((call << 22) + 4ull * (uint64_t)k) & RNG_ID_MASK);
        c1 = 2.0 * gamma_mt(0.5 * nu, ph, base);
        c2 = 2.0 * gamma_mt(0.5 * (nu - 1.0), ph, base + 1);
        double z2;
        box_muller(ph(0, base + 2), z, z2);
    }
    const double a00 = sqrt(c1), a10 = z, a11 = sqrt(c2);
    // H = G A (lower triangular), W = H H^T, X = W^-1
    const double h00 = g00 * a00, h10 = g10 * a00 + g11 * a10, h11 = g11 * a11;
    const double w00 = h00 * h00, w01 = h00 * h10, w11 = h10 * h10 + h11 * h11;
    const double dw = w00 * w11 - w01 * w01;
    x00 = w11 / dw; x01 = -w01 / dw; x11 = w00 / dw;
}

// Per multipole (.ipynb_checkpoints/main-checkpoint.py:39-44, 333-346): C_l ~ IW(2l - 2, (2l+1) Chat_l), draw k = l.
// inject (nullable): (L+1, 3).  l < 2 -> 0.  Output in C_l units.
__global__ void invwishart_2x2_kernel(const double* __restrict__ tt, const double* __restrict__ te, const double* __restrict__ ee, int L,
                                      const double* __restrict__ inject, uint64_t seed, uint64_t call, double* __restrict__ o_tt,
                                      double* __restrict__ o_te, double* __restrict__ o_ee)
{
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l > L) return;
    if (l < 2) { o_tt[l] = 0.0; o_te[l] = 0.0; o_ee[l] = 0.0; return; }
    const double f = 2.0 * l + 1.0, nu = 2.0 * l - 2.0;
    double x00, x01, x11;
    invwishart_2x2_draw(f * tt[l], f * te[l], f * ee[l], nu, inject, l, seed, call, x00, x01, x11);
    o_tt[l] = x00; o_te[l] = x01; o_ee[l] = x11;
}

// Per bin, with D_l = D_b constant on bin b (the binned model of CenteredGibbs.py:54-79, utils.unfold_bins):
//   D_b | s ~ IW(nu_b, Psi_b),  nu_b = sum_{l in b} (2l+1) - 3,  Psi_b = sum_{l in b} (2l+1) l(l+1)/(2 pi) Chat_l,
// the product over l in b of the per-l likelihoods |C_l|^{-(2l+1)/2} exp(-(2l+1)/2 tr(C_l^-1 Chat_l)) times the flat prior of the
// per-l draw (for p = 1 the inverse-gamma alpha = sum (2l+1)/2 - 1 of cls_invgamma_kernel).  With one-l bins this is the per-l
// draw scaled by l(l+1)/(2 pi), on the same variates (draw k = b).  Psi_b is summed in ascending l (deterministic); bins 0 and 1
// are l = 0 and l = 1 (edges start 0, 1, 2) and are 0.  inject (nullable): (nbins, 3).  Output in D units.
// The edges live on the device, so the host cannot check them without a copy and a synchronisation: each thread checks its own
// bin instead and writes NaN where the edges break the conditions (bin 0 / 1 not [0, 1) / [1, 2), a bin empty, below l = 2 or
// past L, a last edge other than L + 1), so such a binning shows up in the output instead of being zeroed or read out of range.
__global__ void invwishart_binned_kernel(const double* __restrict__ tt, const double* __restrict__ te, const double* __restrict__ ee, int L,
                                         const int* __restrict__ bins, int nbins, const double* __restrict__ inject, uint64_t seed,
                                         uint64_t call, double* __restrict__ o_tt, double* __restrict__ o_te, double* __restrict__ o_ee)
{
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nbins) return;
    const int l0 = bins[b], l1 = bins[b + 1];
    const bool ok = b < 2 ? (l0 == b && l1 == b + 1) : (l0 >= 2 && l1 > l0 && l1 <= L + 1 && (b < nbins - 1 || l1 == L + 1));
    if (b < 2 || !ok) {
        const double v = ok ? 0.0 : __longlong_as_double(0x7ff8000000000000ll);   // 0 for l = 0, 1; NaN for a bad bin
        o_tt[b] = v; o_te[b] = v; o_ee[b] = v;
        return;
    }
    double psi[3], nu = iw_bin_stats(tt, te, ee, l0, l1, psi);
    double x00, x01, x11;
    invwishart_2x2_draw(psi[0], psi[1], psi[2], nu, inject, b, seed, call, x00, x01, x11);
    o_tt[b] = x00; o_te[b] = x01; o_ee[b] = x11;
}

// ---- C ABI
extern "C" int gs_expand_var_cl_3x3(const double* dls, int lmax, double* out, void* stream)
{
    GS_REQUIRE(dls && out && lmax >= 0, "bad arguments");
    expand_var_cl_3x3_kernel<<<tb_blocks((int64_t)(lmax + 1) * (lmax + 1) * 9), TB_NT, 0, STREAM(stream)>>>(dls, lmax, out);
    GS_CHECK_LAUNCH();
    return GS_OK;
}

extern "C" int gs_inv_chol_3x3(const double* all_cls, const double* pix_part, int lmax, double* sigma, double* chol, void* stream)
{
    GS_REQUIRE(all_cls && pix_part && sigma && lmax >= 0, "bad arguments");
    inv_chol_3x3_kernel<<<(lmax + TB_NT) / TB_NT, TB_NT, 0, STREAM(stream)>>>(all_cls, pix_part, lmax, sigma, chol);
    GS_CHECK_LAUNCH();
    return GS_OK;
}

extern "C" int gs_matvec_3x3(const double* mats, const double* v, const double* add, int lmax, double* out, void* stream)
{
    GS_REQUIRE(mats && v && out && lmax >= 0, "bad arguments");
    matvec_3x3_kernel<<<tb_blocks((int64_t)(lmax + 1) * (lmax + 1)), TB_NT, 0, STREAM(stream)>>>(mats, v, add, lmax, out);
    GS_CHECK_LAUNCH();
    return GS_OK;
}

extern "C" int gs_alm2cl_cross(const double* alm_x, const double* alm_y, int lmax, double* cl, void* stream)
{
    GS_REQUIRE(alm_x && alm_y && cl && lmax >= 0, "bad arguments");
    alm2cl_cross_kernel<<<(lmax + 8) / 8, 256, 0, STREAM(stream)>>>(alm_x, alm_y, lmax, cl);
    GS_CHECK_LAUNCH();
    return GS_OK;
}

extern "C" int gs_cls_invwishart(const double* cl_tt, const double* cl_te, const double* cl_ee, int lmax, const double* inject,
                                 uint64_t seed, uint64_t call, double* out_tt, double* out_te, double* out_ee, void* stream)
{
    GS_REQUIRE(cl_tt && cl_te && cl_ee && out_tt && out_te && out_ee && lmax >= 0, "bad arguments");
    invwishart_2x2_kernel<<<(lmax + TB_NT) / TB_NT, TB_NT, 0, STREAM(stream)>>>(cl_tt, cl_te, cl_ee, lmax, inject, seed, call, out_tt, out_te,
                                                                               out_ee);
    GS_CHECK_LAUNCH();
    return GS_OK;
}

extern "C" int gs_cls_invwishart_binned(const double* cl_tt, const double* cl_te, const double* cl_ee, int lmax, const int* bins, int nbins,
                                        const double* inject, uint64_t seed, uint64_t call, double* dl_tt, double* dl_te, double* dl_ee,
                                        void* stream)
{
    GS_REQUIRE(cl_tt && cl_te && cl_ee && bins && dl_tt && dl_te && dl_ee, "null pointer");
    GS_REQUIRE(lmax >= 0 && nbins >= 1 && nbins <= lmax + 1, "need lmax >= 0 and 1 <= nbins <= lmax + 1");
    invwishart_binned_kernel<<<(nbins + TB_NT - 1) / TB_NT, TB_NT, 0, STREAM(stream)>>>(cl_tt, cl_te, cl_ee, lmax, bins, nbins, inject, seed,
                                                                                       call, dl_tt, dl_te, dl_ee);
    GS_CHECK_LAUNCH();
    return GS_OK;
}
