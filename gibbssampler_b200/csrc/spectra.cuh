// Per-multipole spectrum formulas of the sampler kernels, one definition each: alm index maps, D_l -> C_l, gs_expand_per_l values,
// the real-layout alm2cl walk, the bin of a multipole and the binned inverse-gamma / inverse-Wishart statistics.  The Blackwell-Rao
// estimator (blackwell_rao.cu) evaluates exactly the conditionals the chains draw from because both call the statistics below.
#pragma once
#include <math.h>
#include <stdint.h>

#define GS_PI 3.14159265358979323846

// ---------------------------------------------------------------- index maps
// (l, m) of healpy index id for lmax L:  id = m(2L+1-m)/2 + l,  m <= l <= L.
__device__ __forceinline__ void lm_of_index(int64_t id, int L, int& l, int& m)
{
    // largest m with m(2L+1-m)/2 + m <= id  <=>  first element of column m is (m,m)
    const double b = 2.0 * L + 3.0;
    int mm = (int)floor((b - sqrt(b * b - 8.0 * (double)id)) * 0.5);
    if (mm < 0) mm = 0;
    if (mm > L) mm = L;
    while (mm > 0 && (int64_t)mm * (2 * L + 1 - mm) / 2 + mm > id) --mm;
    while (mm < L && (int64_t)(mm + 1) * (2 * L + 1 - (mm + 1)) / 2 + (mm + 1) <= id) ++mm;
    m = mm;
    l = (int)(id - (int64_t)mm * (2 * L + 1 - mm) / 2);
}

// l of entry i of the real layout ((L+1)^2 doubles: the L+1 entries of m = 0, then (Re, Im) of every m > 0 coefficient)
__device__ __forceinline__ int l_of_real(int64_t i, int L)
{
    if (i <= L) return (int)i;
    int l, m;
    lm_of_index((i + L + 1) >> 1, L, l, m);
    return l;
}

// ---------------------------------------------------------------- per-l values
// C_l = D_l 2 pi / (l(l+1)); l = 0 is passed through (utils.generate_var_cl, variance_expension.pyx:23-27)
__device__ __forceinline__ double dl_to_cl(double d, int l) { return l ? d * 2.0 * GS_PI / ((double)l * (double)(l + 1)) : d; }

// 1/v, and 0 where v = 0 (an unconstrained or switched-off multipole)
__device__ __forceinline__ double safe_rcp(double v) { return v != 0.0 ? 1.0 / v : 0.0; }

// per-l array -> value at multipole l.  mode 0: copy x_l (GibbsSampler.compute_bl_map, GibbsSampler.py:64-74,
// config.generate_var_cl config.py:75-84); mode 1: C_l = dl_to_cl(x_l) (utils.generate_var_cl_cython utils.py:114-137,
// variance_expension.pyx:8-33); mode 2: safe_rcp(C_l); mode 3: sqrt(C_l); mode 4: sqrt(safe_rcp(C_l)).
__device__ __forceinline__ double per_l_value(const double* x, int l, int mode)
{
    double v = x[l];
    if (mode == 0) return v;
    v = dl_to_cl(v, l);
    if (mode == 1) return v;
    if (mode == 3) return sqrt(v);
    const double inv = safe_rcp(v);
    return mode == 2 ? inv : sqrt(inv);
}

// ---------------------------------------------------------------- hp.alm2cl on the real layout
// One warp per multipole l: lane k sums the entries of m = k, k + 32, ... <= l (m = 0: entry l; m > 0: the (Re, Im) pair at
// 2 idx(l, m) - (L+1)); warp_sum then adds the 32 lane sums in a fixed shuffle tree and C_l = sum / (2l+1).  The auto spectrum
// loads each coefficient once.
__device__ __forceinline__ double warp_sum(double s)
{
    for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    return s;
}

__device__ __forceinline__ double alm2cl_real_lane(const double* a, int l, int L, int lane)
{
    double s = 0.0;
    for (int m = lane; m <= l; m += 32) {
        if (m == 0) { const double v = a[l]; s += v * v; }
        else {
            const int64_t id = (int64_t)m * (2 * L + 1 - m) / 2 + l, o = 2 * id - (L + 1);
            const double x = a[o], y = a[o + 1];
            s += x * x + y * y;
        }
    }
    return s;
}

// cross spectrum of x and y (= hp.alm2cl(alm1, alm2))
__device__ __forceinline__ double alm2cl_cross_real_lane(const double* x, const double* y, int l, int L, int lane)
{
    double s = 0.0;
    for (int m = lane; m <= l; m += 32) {
        const int64_t id = (int64_t)m * (2 * L + 1 - m) / 2 + l;
        if (m == 0) s += x[l] * y[l];
        else { const int64_t o = 2 * id - (L + 1); s += x[o] * y[o] + x[o + 1] * y[o + 1]; }
    }
    return s;
}

// ---------------------------------------------------------------- binning
// index of the last bin whose lower edge bins[b] <= l (binary search over bins[0..nbins-1]; 0 when l < bins[1]).  What a
// multipole outside [bins[0], bins[nbins]) maps to is the caller's rule.
__device__ __forceinline__ int bin_of(const int* bins, int nbins, int l)
{
    int lo = 0, hi = nbins - 1;
    while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (bins[mid] <= l) lo = mid; else hi = mid - 1; }
    return lo;
}

// ---------------------------------------------------------------- binned C_l conditionals
// Both are summed over l = l0 .. l1-1 in ascending order, so every caller gets the same numbers bit for bit.
//
// Inverse gamma (CenteredGibbs.py:24-79), D_b | s ~ IG(alpha_b, beta_b) from the empirical spectrum cl:
//   alpha_b = sum (2l+1)/2 - 1,   beta_b = sum (2l+1) l(l+1) cl_l / (4 pi).
template <bool BETA>
__device__ __forceinline__ double ig_bin_sums(const double* cl, int l0, int l1, double* beta)
{
    double bt = 0.0, ex = 0.0;
    for (int l = l0; l < l1; ++l) {
        if constexpr (BETA) bt += (2.0 * l + 1.0) * (double)l * (double)(l + 1) * (cl[l] / (4.0 * GS_PI));
        ex += (2.0 * l + 1.0) / 2.0;
    }
    if constexpr (BETA) *beta = bt;
    return ex - 1.0;
}

// alpha_b and beta_b (returns alpha_b), or alpha_b alone
__device__ __forceinline__ double ig_bin_stats(const double* cl, int l0, int l1, double& beta) { return ig_bin_sums<true>(cl, l0, l1, &beta); }
__device__ __forceinline__ double ig_bin_alpha(int l0, int l1) { return ig_bin_sums<false>(nullptr, l0, l1, nullptr); }

// Inverse Wishart of a (TT, TE; TE, EE) block (teb.cu, invwishart_binned_kernel), D_b | s ~ IW(nu_b, Psi_b) from the empirical
// spectra tt, te, ee:  nu_b = sum (2l+1) - 3,   Psi_b = sum (2l+1) l(l+1)/(2 pi) (tt_l, te_l, ee_l).
template <bool PSI>
__device__ __forceinline__ double iw_bin_sums(const double* tt, const double* te, const double* ee, int l0, int l1, double* psi)
{
    double p00 = 0.0, p01 = 0.0, p11 = 0.0, nu = -3.0;
    for (int l = l0; l < l1; ++l) {
        const double f = 2.0 * l + 1.0;
        const double w = f * ((double)l * (double)(l + 1) / (2.0 * GS_PI));
        if constexpr (PSI) { p00 += w * tt[l]; p01 += w * te[l]; p11 += w * ee[l]; }
        nu += f;
    }
    if constexpr (PSI) { psi[0] = p00; psi[1] = p01; psi[2] = p11; }
    return nu;
}

// nu_b and psi = (Psi00, Psi01, Psi11) (returns nu_b), or nu_b alone
__device__ __forceinline__ double iw_bin_stats(const double* tt, const double* te, const double* ee, int l0, int l1, double (&psi)[3])
{
    return iw_bin_sums<true>(tt, te, ee, l0, l1, psi);
}
__device__ __forceinline__ double iw_bin_nu(int l0, int l1) { return iw_bin_sums<false>(nullptr, nullptr, nullptr, l0, l1, nullptr); }
