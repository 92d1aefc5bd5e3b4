// Blackwell–Rao estimator of the power-spectrum posterior from a Gibbs chain (Wandelt, Larson & Lakshminarayanan 2004;
// Chu et al. 2005):  p̂(D | d) = (1/N) Σ_i p(D | σ^i),  σ^i = empirical spectrum of the i-th sky sample, p(D | σ) = the C_ℓ
// conditional the chain draws from (binned inverse-gamma of cls_invgamma_kernel, 2×2 inverse-Wishart of invwishart_binned_kernel).
// Written x_ik = Σ_b log p(D_b^k | σ^i) = c_i + Σ_j S_ij W_jk + e_k, the estimator is an FP64 GEMM (samples × features ×
// models) followed by a log-mean-exp over the sample axis; the br_logmeanexp kernels fuse the two and never writes the N × M matrix.
// Every reduction runs in a fixed order that depends on (N, M) only, so results are bit-identical from run to run.
#include <math.h>

#include <algorithm>

#include "gs_internal.h"
#include "spectra.cuh"

#define BR_NT 256
#define BR_BK 8                   // features per shared-memory stage of the GEMM
#define BR_SPLIT_UNIT 256         // the sample axis is split over CTAs in multiples of this many samples
#define BR_TARGET_CTAS (148 * 16) // CTAs the split aims at: 16 waves of one CTA per SM keep the last-wave tail small
#define BR_SMALL_M 32             // up to this many models the narrow 8-model tile runs (one parameter-MCMC call is M = 1)

__device__ __forceinline__ bool br_bin(const int* __restrict__ bins, int b, int ncl, int& l0, int& l1)
{
    l0 = bins[b];
    l1 = bins[b + 1];
    return l0 >= 0 && l1 > l0 && l1 <= ncl;
}

__device__ __forceinline__ double br_nan() { return __longlong_as_double(0x7ff8000000000000ll); }

// ------------------------------------------------------------------ features
// Thread (sample i, bin b).  IG: S row b = beta_b^i (ig_bin_stats, as cls_invgamma_kernel, so it equals its beta_out bit for bit),
// t[b][i] = alpha_b log beta_b^i.  IW: S rows 3b..3b+2 = (Psi00, Psi01, Psi11) (iw_bin_stats, as invwishart_binned_kernel),
// t[b][i] = (nu_b / 2) log|Psi_b^i|.  A bin whose device edges are broken (empty, negative, past ncl) comes out NaN.
__global__ void br_sample_features_kernel(int kind, const double* __restrict__ sig, const double* __restrict__ sig_te,
                                          const double* __restrict__ sig_ee, int64_t n, int ncl, const int* __restrict__ bins,
                                          double* __restrict__ S, double* __restrict__ t)
{
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const int b = blockIdx.y;
    if (i >= n) return;
    int l0, l1;
    const bool ok = br_bin(bins, b, ncl, l0, l1);
    if (kind == GS_BR_IG) {
        if (!ok) { S[b * n + i] = br_nan(); t[b * n + i] = br_nan(); return; }
        double beta, alpha = ig_bin_stats(sig + i * ncl, l0, l1, beta);
        S[b * n + i] = beta;
        t[b * n + i] = alpha * log(beta);
        return;
    }
    double* s = S + (int64_t)3 * b * n + i;
    if (!ok) { s[0] = br_nan(); s[n] = br_nan(); s[2 * n] = br_nan(); t[b * n + i] = br_nan(); return; }
    double psi[3], nu = iw_bin_stats(sig + i * ncl, sig_te + i * ncl, sig_ee + i * ncl, l0, l1, psi);
    s[0] = psi[0]; s[n] = psi[1]; s[2 * n] = psi[2];
    t[b * n + i] = 0.5 * nu * log(psi[0] * psi[2] - psi[1] * psi[1]);
}

// Thread (model k, bin b).  IG: W row b = -1/D_b, t = -lgamma(alpha) - (alpha+1) log D_b.  IW: W rows = (-(D^-1)00 / 2, -(D^-1)01,
// -(D^-1)11 / 2), t = -nu log 2 - log Gamma_2(nu/2) - (nu+3)/2 log|D|.  D_b <= 0 (or NaN), or an IW block that is not positive
// definite: W = 0 and t = -inf, so the model's x_ik is exactly -inf.  Broken edges: NaN.
__global__ void br_model_features_kernel(int kind, const double* __restrict__ d, const double* __restrict__ d_te,
                                         const double* __restrict__ d_ee, int64_t m, int ncl, const int* __restrict__ bins, int nbins,
                                         double* __restrict__ W, double* __restrict__ t)
{
    const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const int b = blockIdx.y;
    if (k >= m) return;
    int l0, l1;
    const bool ok = br_bin(bins, b, ncl, l0, l1);
    const int64_t j = k * nbins + b;
    if (kind == GS_BR_IG) {
        const double D = d[j], alpha = ok ? ig_bin_alpha(l0, l1) : 0.0;
        const bool valid = D > 0.0;
        W[b * m + k] = !ok ? br_nan() : valid ? -1.0 / D : 0.0;
        t[b * m + k] = !ok ? br_nan() : valid ? -lgamma(alpha) - (alpha + 1.0) * log(D) : -INFINITY;
        return;
    }
    double* w = W + (int64_t)3 * b * m + k;
    if (!ok) { w[0] = br_nan(); w[m] = br_nan(); w[2 * m] = br_nan(); t[b * m + k] = br_nan(); return; }
    const double tt = d[j], te = d_te[j], ee = d_ee[j], det = tt * ee - te * te, nu = iw_bin_nu(l0, l1);
    if (!(tt > 0.0 && det > 0.0)) { w[0] = 0.0; w[m] = 0.0; w[2 * m] = 0.0; t[b * m + k] = -INFINITY; return; }
    w[0] = -0.5 * (ee / det);
    w[m] = te / det;
    w[2 * m] = -0.5 * (tt / det);
    const double lg2 = 0.5 * log(GS_PI) + lgamma(0.5 * nu) + lgamma(0.5 * nu - 0.5);
    t[b * m + k] = -nu * log(2.0) - lg2 - 0.5 * (nu + 3.0) * log(det);
}

// out[i] = (accumulate ? out[i] : 0) + sum_{r < nrows} t[r][i], r ascending
__global__ void br_rowsum_kernel(const double* __restrict__ t, int64_t n, int nrows, int accumulate, double* __restrict__ out)
{
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    double s = accumulate ? out[i] : 0.0;
    for (int r = 0; r < nrows; ++r) s += t[r * n + i];
    out[i] = s;
}

// ------------------------------------------------------------------ fused GEMM + log-mean-exp
// running (max, sum exp(x - max), sum exp(2 (x - max))) of one model; merge() is commutative bit for bit
struct BrAcc {
    double m, s1, s2;
};

__device__ __forceinline__ BrAcc br_merge(BrAcc a, BrAcc b)
{
    const double m = fmax(a.m, b.m);
    if (m == -INFINITY) return {m, a.s1 + b.s1, a.s2 + b.s2};   // both empty: zeros, or NaN from a poisoned part
    const double fa = exp(a.m - m), fb = exp(b.m - m);
    return {m, a.s1 * fa + b.s1 * fb, a.s2 * (fa * fa) + b.s2 * (fb * fb)};
}

// fold R log-densities x of one model into its running state; a NaN among them (a broken bin passed through the C ABI) makes
// s1 NaN, which every later merge keeps, so the model's estimate comes out NaN rather than dropping the sample
template <int R>
__device__ __forceinline__ void br_fold(BrAcc& r, const double (&x)[R])
{
    double xm = -INFINITY;
    bool bad = false;
#pragma unroll
    for (int j = 0; j < R; ++j) {
        xm = fmax(xm, x[j]);
        bad |= isnan(x[j]);
    }
    if (bad) r.s1 = br_nan();
    if (xm > r.m) {
        const double f = exp(r.m - xm);
        r.s1 *= f;
        r.s2 *= f * f;
        r.m = xm;
    }
    if (r.m != -INFINITY) {
#pragma unroll
        for (int j = 0; j < R; ++j) {
            const double w = exp(x[j] - r.m);
            r.s1 += w;
            r.s2 = fma(w, w, r.s2);
        }
    }
}

// Narrow tile (M <= 32, e.g. one parameter-MCMC call): CTA = 8 models x 256 samples of one split; thread ty owns sample n0 + ty of
// each tile and all 8 models.  Every sample is used by one thread only, so S streams from global memory straight into registers
// (8 independent loads in flight per thread) and W, the same address for every thread, is a broadcast load.  The 32 lanes of a warp
// then merge by shuffles and the 8 warps through shared memory, in a fixed order; the CTA writes one partial per (split, model).
__global__ void __launch_bounds__(BR_NT) br_logmeanexp_narrow_kernel(const double* __restrict__ S, const double* __restrict__ c,
                                                                     int64_t n, const double* __restrict__ W, const double* __restrict__ e,
                                                                     int64_t m, int K, int64_t chunk, double* __restrict__ part)
{
    constexpr int RM = 8;
    const int64_t m0 = blockIdx.x * (int64_t)RM;
    const int64_t nbeg = blockIdx.y * chunk, nend = min(n, nbeg + chunk);
    double ev[RM];
    BrAcc acc_run[RM];
#pragma unroll
    for (int i = 0; i < RM; ++i) {
        ev[i] = m0 + i < m ? e[m0 + i] : -INFINITY;
        acc_run[i] = {-INFINITY, 0.0, 0.0};
    }
    for (int64_t n0 = nbeg; n0 < nend; n0 += BR_NT) {
        const int64_t col = n0 + threadIdx.x;
        const bool in = col < nend;
        double acc[RM];
#pragma unroll
        for (int i = 0; i < RM; ++i) acc[i] = 0.0;
#pragma unroll 8
        for (int k = 0; k < K; ++k) {
            const double sv = in ? __ldg(S + (int64_t)k * n + col) : 0.0;
#pragma unroll
            for (int i = 0; i < RM; ++i) {
                const double wv = m0 + i < m ? __ldg(W + (int64_t)k * m + m0 + i) : 0.0;
                acc[i] = fma(wv, sv, acc[i]);
            }
        }
        const double cj = in ? c[col] : -INFINITY;
#pragma unroll
        for (int i = 0; i < RM; ++i) {
            const double x[1] = {(cj + acc[i]) + ev[i]};
            br_fold(acc_run[i], x);
        }
    }
#pragma unroll
    for (int i = 0; i < RM; ++i) {
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            BrAcc other;
            other.m = __shfl_xor_sync(0xffffffffu, acc_run[i].m, o);
            other.s1 = __shfl_xor_sync(0xffffffffu, acc_run[i].s1, o);
            other.s2 = __shfl_xor_sync(0xffffffffu, acc_run[i].s2, o);
            acc_run[i] = br_merge(acc_run[i], other);
        }
    }
    constexpr int NW = BR_NT / 32;
    __shared__ BrAcc red[NW][RM];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) {
#pragma unroll
        for (int i = 0; i < RM; ++i) red[warp][i] = acc_run[i];
    }
    __syncthreads();
    if (threadIdx.x < RM && m0 + threadIdx.x < m) {
        BrAcc r = red[0][threadIdx.x];
        for (int w = 1; w < NW; ++w) r = br_merge(r, red[w][threadIdx.x]);
        double* o = part + ((int64_t)blockIdx.y * m + m0 + threadIdx.x) * 3;
        o[0] = r.m; o[1] = r.s1; o[2] = r.s2;
    }
}

// Wide tile (M > 32): CTA = 64 models x 128 samples of one split on the FP64 tensor instruction (mma.sync.m8n8k4.f64, SASS
// DMMA.8x8x4), which measured 1.4-1.5x faster than the same tile on DFMA (DESIGN.md, "Blackwell-Rao estimator"): warp (wm, wn) of
// the 2 x 4 warp grid owns a 32 x 32 block as 4 x 4 tiles of 8 x 8.  A = W^T (models x features) and B = S (features x samples) are
// read as fragments from the same double-buffered shared-memory stages (rows padded by 8 doubles: the four k rows of a fragment
// fall on alternate bank halves); lane (g, t) = (lane / 4, lane % 4) holds models mw + 8 i + g and samples nw + 8 j + 2 t + {0, 1}.
#define BR_PAD 8
__device__ __forceinline__ void br_dmma(double& d0, double& d1, double a, double b)
{
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};" : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
}

__global__ void __launch_bounds__(BR_NT) br_logmeanexp_dmma_kernel(const double* __restrict__ S, const double* __restrict__ c, int64_t n,
                                                                   const double* __restrict__ W, const double* __restrict__ e, int64_t m,
                                                                   int K, int64_t chunk, double* __restrict__ part)
{
    constexpr int BM = 64, BN = 128, LS = BR_BK * BN / BR_NT, LW = BR_BK * BM / BR_NT;
    __shared__ double sS[2][BR_BK][BN + BR_PAD];
    __shared__ double sW[2][BR_BK][BM + BR_PAD];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, g = lane >> 2, t = lane & 3;
    const int mw = 32 * (warp >> 2), nw = 32 * (warp & 3);
    const int64_t m0 = blockIdx.x * (int64_t)BM;
    const int64_t nbeg = blockIdx.y * chunk, nend = min(n, nbeg + chunk);
    const int nkt = (K + BR_BK - 1) / BR_BK;
    double ev[4];
    BrAcc acc_run[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int64_t k = m0 + mw + 8 * i + g;
        ev[i] = k < m ? e[k] : -INFINITY;
        acc_run[i] = {-INFINITY, 0.0, 0.0};
    }
    for (int64_t n0 = nbeg; n0 < nend; n0 += BN) {
        double pS[LS], pW[LW];
        auto gload = [&](int k0) {
#pragma unroll
            for (int r = 0; r < LS; ++r) {
                const int q = threadIdx.x + r * BR_NT, kk = q / BN;
                const int64_t col = n0 + q % BN;
                pS[r] = (k0 + kk < K && col < nend) ? S[(int64_t)(k0 + kk) * n + col] : 0.0;
            }
#pragma unroll
            for (int r = 0; r < LW; ++r) {
                const int q = threadIdx.x + r * BR_NT, kk = q / BM;
                const int64_t col = m0 + q % BM;
                pW[r] = (k0 + kk < K && col < m) ? W[(int64_t)(k0 + kk) * m + col] : 0.0;
            }
        };
        auto sstore = [&](int buf) {
#pragma unroll
            for (int r = 0; r < LS; ++r) {
                const int q = threadIdx.x + r * BR_NT;
                sS[buf][q / BN][q % BN] = pS[r];
            }
#pragma unroll
            for (int r = 0; r < LW; ++r) {
                const int q = threadIdx.x + r * BR_NT;
                sW[buf][q / BM][q % BM] = pW[r];
            }
        };
        double acc[4][4][2];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
        gload(0);
        sstore(0);
        __syncthreads();
        for (int kt = 0; kt < nkt; ++kt) {
            const int cur = kt & 1;
            if (kt + 1 < nkt) gload((kt + 1) * BR_BK);
#pragma unroll
            for (int kk = 0; kk < BR_BK; kk += 4) {
                double a[4], b[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) a[i] = sW[cur][kk + t][mw + 8 * i + g];
#pragma unroll
                for (int j = 0; j < 4; ++j) b[j] = sS[cur][kk + t][nw + 8 * j + g];
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) br_dmma(acc[i][j][0], acc[i][j][1], a[i], b[j]);
            }
            if (kt + 1 < nkt) sstore(cur ^ 1);
            __syncthreads();
        }
        double cj[8];
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                const int64_t col = n0 + nw + 8 * j + 2 * t + q;
                cj[2 * j + q] = col < nend ? c[col] : -INFINITY;
            }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            double x[8];
#pragma unroll
            for (int j = 0; j < 4; ++j)
#pragma unroll
                for (int q = 0; q < 2; ++q) x[2 * j + q] = (cj[2 * j + q] + acc[i][j][q]) + ev[i];
            br_fold(acc_run[i], x);
        }
    }
    // the four lanes of a group g hold the same models: merge over t, then over the four warps of a model half
#pragma unroll
    for (int i = 0; i < 4; ++i) {
#pragma unroll
        for (int o = 1; o < 4; o <<= 1) {
            BrAcc other;
            other.m = __shfl_xor_sync(0xffffffffu, acc_run[i].m, o);
            other.s1 = __shfl_xor_sync(0xffffffffu, acc_run[i].s1, o);
            other.s2 = __shfl_xor_sync(0xffffffffu, acc_run[i].s2, o);
            acc_run[i] = br_merge(acc_run[i], other);
        }
    }
    __shared__ BrAcc red[4][BM];
    if (t == 0) {
#pragma unroll
        for (int i = 0; i < 4; ++i) red[warp & 3][mw + 8 * i + g] = acc_run[i];
    }
    __syncthreads();
    if (threadIdx.x < BM && m0 + threadIdx.x < m) {
        BrAcc r = red[0][threadIdx.x];
        for (int w = 1; w < 4; ++w) r = br_merge(r, red[w][threadIdx.x]);
        double* o = part + ((int64_t)blockIdx.y * m + m0 + threadIdx.x) * 3;
        o[0] = r.m; o[1] = r.s1; o[2] = r.s2;
    }
}

// CTA per model: thread t merges the split partials t, t + 128, ... in ascending order, then a fixed shared-memory tree merges the
// 128 results (the same order on every run); log L = max + log(s1 / N), n_eff = s1^2 / s2
#define BR_FIN_NT 128
__global__ void __launch_bounds__(BR_FIN_NT) br_finish_kernel(const double* __restrict__ part, const double* __restrict__ e, int64_t n,
                                                              int64_t m, int P, double* __restrict__ logl, double* __restrict__ neff)
{
    __shared__ BrAcc red[BR_FIN_NT];
    const int64_t k = blockIdx.x;
    BrAcc r = {-INFINITY, 0.0, 0.0};
    for (int p = threadIdx.x; p < P; p += BR_FIN_NT) {
        const double* q = part + ((int64_t)p * m + k) * 3;
        r = br_merge(r, BrAcc{q[0], q[1], q[2]});
    }
    red[threadIdx.x] = r;
    __syncthreads();
    for (int s = BR_FIN_NT / 2; s > 0; s >>= 1) {
        if (threadIdx.x < s) red[threadIdx.x] = br_merge(red[threadIdx.x], red[threadIdx.x + s]);
        __syncthreads();
    }
    if (threadIdx.x) return;
    r = red[0];
    double ll, ne;
    if (isnan(e[k]) || isnan(r.s1)) { ll = br_nan(); ne = br_nan(); }
    else if (e[k] == -INFINITY || r.m == -INFINITY) { ll = -INFINITY; ne = 0.0; }
    else { ll = r.m + log(r.s1) - log((double)n); ne = r.s1 * r.s1 / r.s2; }
    logl[k] = ll;
    if (neff) neff[k] = ne;
}

// ------------------------------------------------------------------ per-bin marginals
// CTA (grid chunk, bin b): log mean_i p(g | sigma_b^i) for 256 grid points g, p = IG(alpha, beta_i).  IG spectra: alpha_b, beta = S row b;
// diagonal entry comp (0 = TT, 2 = EE) of an IW bin: IG((nu_b - 1)/2, Psi_jj / 2).  beta_i and alpha log beta_i are staged in shared
// memory once per 256-sample tile for all grid points; each thread keeps an online log-sum-exp over the samples.
__global__ void __launch_bounds__(BR_NT) br_marginal_kernel(int kind, const double* __restrict__ S, int64_t n, int ncl,
                                                            const int* __restrict__ bins, int comp, const double* __restrict__ grid,
                                                            int64_t grid_ld, int ng, double* __restrict__ out)
{
    __shared__ double sb[BR_NT], slb[BR_NT];
    const int b = blockIdx.y, g = blockIdx.x * BR_NT + threadIdx.x;
    int l0, l1;
    const bool ok = br_bin(bins, b, ncl, l0, l1);
    double alpha = 0.0, scale = 1.0;
    const double* row = S + (int64_t)b * n;
    if (ok) {
        if (kind == GS_BR_IG) {
            alpha = ig_bin_alpha(l0, l1);
        } else {
            alpha = 0.5 * (iw_bin_nu(l0, l1) - 1.0);
            scale = 0.5;
            row = S + ((int64_t)3 * b + comp) * n;
        }
    }
    const double x = g < ng ? grid[b * grid_ld + g] : 1.0, ix = 1.0 / x;
    double mx = -INFINITY, s = 0.0;
    for (int64_t i0 = 0; ok && i0 < n; i0 += BR_NT) {
        __syncthreads();
        if (i0 + threadIdx.x < n) {
            const double beta = scale * row[i0 + threadIdx.x];
            sb[threadIdx.x] = beta;
            slb[threadIdx.x] = alpha * log(beta);
        }
        __syncthreads();
        const int cnt = (int)(n - i0 < BR_NT ? n - i0 : BR_NT);
        double tm = -INFINITY;
        for (int j = 0; j < cnt; ++j) tm = fmax(tm, fma(-sb[j], ix, slb[j]));
        if (tm > mx) { s *= exp(mx - tm); mx = tm; }
        if (mx != -INFINITY)
            for (int j = 0; j < cnt; ++j) s += exp(fma(-sb[j], ix, slb[j]) - mx);
    }
    if (g >= ng) return;
    double v;
    if (!ok) v = br_nan();
    else if (!(x > 0.0) || mx == -INFINITY) v = -INFINITY;
    else v = mx + log(s) - log((double)n) - lgamma(alpha) - (alpha + 1.0) * log(x);
    out[(int64_t)b * ng + g] = v;
}

// ------------------------------------------------------------------ Gaussianized Blackwell-Rao transform (Rudjord et al. 2009)
// Per bin, the BR marginal is the mixture (1/N) sum_i IG(alpha, beta_i).  With t = beta_i / D ~ Gamma(alpha, 1) its CDF is
// F(D) = (1/N) sum_i Q(alpha, t_i) and 1 - F = (1/N) sum_i P(alpha, t_i) (regularized incomplete gammas).  Each sample computes its
// smaller tail directly and the other as 1 - small; both sums are kept, so x = Phi^-1(F) never forms 1 - (something near 1).
// The prefactor t^alpha e^-t / Gamma(alpha) of P and Q is also the IG density times D, so log p_i(D) costs nothing extra.
#define GBR_NT 256
#define GBR_TEMME_ALPHA 20.0   // Temme's uniform expansion for alpha >= this and |t / alpha - 1| < GBR_TEMME_DEV
#define GBR_TEMME_DEV 0.3
#define GBR_TEMME_NK 10        // terms c_k(eta) a^-k, k < 10: the first omitted one is below 1e-16 of the sum for alpha >= 20
#define GBR_TEMME_NC 18        // Taylor terms of each c_k(eta); |eta| < 0.34 in the Temme region, radius of convergence 2 sqrt(pi)
#define GBR_SERIES_MAX 4096    // iteration caps of the series and the continued fraction (never reached in their regions)

// Taylor coefficients of Temme's c_k(eta) (DLMF 8.12.8-9: c_0 = 1/(lambda - 1) - 1/eta, c_k = c_{k-1}'(eta) / eta
// + (-1)^k g_k / (lambda - 1), g_k Stirling's coefficients), derived in exact rational arithmetic and rounded to double
__constant__ double gbr_temme_c[GBR_TEMME_NK][GBR_TEMME_NC] = {
    {-0.33333333333333331, 0.083333333333333329, -0.014814814814814815, 0.0011574074074074073, 0.00035273368606701942, -0.0001787551440329218, 3.9192631785224377e-05, -2.185448510679992e-06, -1.85406221071516e-06, 8.2967113409530865e-07, -1.7665952736826078e-07, 6.7078535434014984e-09, 1.0261809784240309e-08, -4.3820360184533529e-09, 9.1476995822367902e-10, -2.5514193994946248e-11, -5.8307721325504256e-11, 2.4361948020667415e-11},
    {-0.0018518518518518519, -0.003472222222222222, 0.0026455026455026454, -0.00099022633744855963, 0.00020576131687242798, -4.018775720164609e-07, -1.8098550334489977e-05, 7.6491609160811098e-06, -1.6120900894563446e-06, 4.647127802807434e-09, 1.3786334469157209e-07, -5.7525456035177047e-08, 1.1951628599778148e-08, -1.7543241719747647e-11, -1.0091543710600413e-09, 4.1627929918425828e-10, -8.5639070264929801e-11, 6.0672151016047582e-14},
    {0.0041335978835978834, -0.0026813271604938273, 0.0007716049382716049, 2.0093878600823047e-06, -0.0001073665322636516, 5.2923448829120125e-05, -1.2760635188618728e-05, 3.4235787340961378e-08, 1.3721957309062934e-06, -6.2989921383800548e-07, 1.4280614206064242e-07, -2.0477098421990866e-10, -1.409252991086752e-08, 6.2289740849220218e-09, -1.3670488396617114e-09, 9.428356159014678e-13, 1.2872252400089318e-10, -5.5645956134363323e-11},
    {0.00064943415637860077, 0.00022947209362139917, -0.0004691894943952557, 0.00026772063206283885, -7.5618016718839766e-05, -2.3965051138672968e-07, 1.1082654115347302e-05, -5.6749528269915965e-06, 1.4230900732435883e-06, -2.7861080291528143e-11, -1.6958404091930278e-07, 8.0994649053880827e-08, -1.9111168485973655e-08, 2.3928620439808118e-12, 2.0620131815488797e-09, -9.460496661855133e-10, 2.1541049775774907e-10, -1.388823336813903e-14},
    {-0.00086188829091671173, 0.00078403922172006662, -0.00029907248030319018, -1.4638452578843418e-06, 6.6414982154651219e-05, -3.9683650471794347e-05, 1.1375726970678419e-05, 2.5074972262375329e-10, -1.6954149536558305e-06, 8.9075075322053094e-07, -2.2929348340008049e-07, 2.9567941375440492e-11, 2.8865829742708783e-08, -1.4189739437803219e-08, 3.4463580499464896e-09, -2.3024517174528067e-13, -3.9409233028046403e-10, 1.8602338968504501e-10},
    {-0.00033679855336635813, -6.9728137583658571e-05, 0.00027727532449593918, -0.00019932570516188847, 6.797780477937208e-05, 1.4190629206439671e-07, -1.3594048189768693e-05, 8.018470256334202e-06, -2.2914811765080952e-06, -3.2524735512984538e-10, 3.4652846491085265e-07, -1.8447187191171344e-07, 4.8240967037894184e-08, -1.7989466721743514e-14, -6.3061945000135231e-09, 3.1624176287745678e-09, 0, 0},
    {0.00053130793646399225, -0.00059216643735369393, 0.0002708782096718045, 7.9023532326603281e-07, -8.1539693675619691e-05, 5.6116827531062497e-05, -1.8329116582843375e-05, -3.0796134506033047e-09, 3.4651553688036091e-06, -2.0291327396058603e-06, 5.7887928631490039e-07, 2.3386306738266568e-13, -8.828600746330484e-08, 4.7435958880408125e-08, 0, 0, 0, 0},
    {0.00034436760689237765, 5.1717909082605919e-05, -0.00033493161081142234, 0.00028126951547632369, -0.00010976582244684731, -1.2741009095484485e-07, 2.7744451511563645e-05, -1.8263488805711332e-05, 5.7876949497350525e-06, 4.9387589339362701e-10, -1.0595367014026043e-06, 6.1667143761104078e-07, 0, 0, 0, 0, 0, 0},
    {-0.00065262391859530937, 0.00083949872067208726, -0.00043829709854172099, -6.9690914584205523e-07, 0.00016644846642067547, -0.00012783517679769218, 4.6299532636913042e-05, 4.557909867922708e-09, -1.0595271125805195e-05, 6.7833429048651668e-06, 0, 0, 0, 0, 0, 0, 0, 0},
    {-0.00059676129019274626, -7.2048954160200109e-05, 0.0006782308837667328, -0.0006401475260262758, 0.00027750107634328704, 1.8197008380465151e-07, -8.4795071170685031e-05, 6.1051920825015314e-05, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0}
};

// d - log(1 + d) >= 0 for d > -1.  Near 0 it is ~ d^2 / 2 and the direct difference loses digits: with r = d / (2 + d),
// log(1 + d) = 2 atanh(r), so d - log(1 + d) = r d - 2 r (r^2/3 + r^4/5 + ...), |r| <= 1/3 for |d| <= 0.5 (20 terms: r^40 < 1e-19)
__device__ __forceinline__ double gbr_log1pmx(double d)
{
    if (fabs(d) > 0.5) return d - log1p(d);
    const double r = d / (2.0 + d), r2 = r * r;
    double s = 1.0 / 41.0;
#pragma unroll
    for (int k = 19; k >= 1; --k) s = fma(s, r2, 1.0 / (2 * k + 1));
    return r * d - 2.0 * r * (r2 * s);
}

// lgamma(a) - [(a - 1/2) log a - a + log(2 pi) / 2]: Stirling's series for a >= 10 (7 terms, the next is < 1e-16 of the sum)
__device__ __forceinline__ double gbr_stirling_rem(double a)
{
    if (a < 10.0) return lgamma(a) - ((a - 0.5) * log(a) - a + 0.5 * log(2.0 * GS_PI));
    const double r = 1.0 / a, r2 = r * r;
    return r * (1.0 / 12 + r2 * (-1.0 / 360 + r2 * (1.0 / 1260 + r2 * (-1.0 / 1680 + r2 * (1.0 / 1188 + r2 * (-691.0 / 360360 + r2 / 156))))));
}

// smaller tail of Gamma(a, 1) at t; upper = true when it is Q(a, t) = P(T > t), false for P(a, t).  lp = log(t^a e^-t / Gamma(a)),
// pm = u - 1 - log u with u = t / a.  Temme (|u - 1| < 0.3, a >= 20): Q = erfc(eta sqrt(a/2)) / 2 + R, P = erfc(-eta sqrt(a/2)) / 2 - R,
// eta = sign(u - 1) sqrt(2 pm), R = e^{-a pm} / sqrt(2 pi a) sum_k c_k(eta) a^-k.  Otherwise the series of P for t < a + 1 and the
// continued fraction of Q (modified Lentz) beyond.
__device__ __forceinline__ double gbr_gamma_tail(double a, double t, double u, double lp, double pm, bool& upper)
{
    if (a >= GBR_TEMME_ALPHA && fabs(u - 1.0) < GBR_TEMME_DEV) {
        const double eta = copysign(sqrt(2.0 * pm), u - 1.0), ia = 1.0 / a;
        double sum = 0.0;
        for (int k = GBR_TEMME_NK - 1; k >= 0; --k) {
            double ck = gbr_temme_c[k][GBR_TEMME_NC - 1];
            for (int j = GBR_TEMME_NC - 2; j >= 0; --j) ck = fma(ck, eta, gbr_temme_c[k][j]);
            sum = fma(sum, ia, ck);
        }
        const double R = exp(-a * pm) * rsqrt(2.0 * GS_PI * a) * sum, z = eta * sqrt(0.5 * a);
        upper = eta >= 0.0;
        return upper ? 0.5 * erfc(z) + R : 0.5 * erfc(-z) - R;
    }
    if (t < a + 1.0) {
        double ap = a, term = 1.0, sum = 1.0;
        for (int n = 0; n < GBR_SERIES_MAX; ++n) {
            ap += 1.0;
            term *= t / ap;
            sum += term;
            if (term <= sum * 0x1p-54) break;
        }
        upper = false;
        return exp(lp) * sum / a;
    }
    const double tiny = 1e-300;
    double b = t + 1.0 - a, c = 1.0 / tiny, d = 1.0 / b, h = d;
    for (int i = 1; i < GBR_SERIES_MAX; ++i) {
        const double an = -i * (i - a);
        b += 2.0;
        d = fma(an, d, b);
        if (fabs(d) < tiny) d = tiny;
        c = b + an / c;
        if (fabs(c) < tiny) c = tiny;
        d = 1.0 / d;
        const double del = d * c;
        h *= del;
        if (fabs(del - 1.0) <= 0x1p-54) break;
    }
    upper = true;
    return exp(lp) * h;
}

// running sums of one (model, bin) over samples: P and Q tails, and (max, sum exp(lp - max)) of the log prefactors
struct GbrAcc {
    double p, q, m, s;
};

__device__ __forceinline__ GbrAcc gbr_merge(GbrAcc a, GbrAcc b)
{
    const double m = fmax(a.m, b.m);
    const double s = m == -INFINITY ? a.s + b.s : a.s * exp(a.m - m) + b.s * exp(b.m - m);
    return {a.p + b.p, a.q + b.q, m, s};
}

// one sample of IG(alpha, beta) at D > 0.  lc = log(alpha / 2 pi) / 2 - stirling_rem(alpha), so that
// lp = alpha log t - t - lgamma(alpha) = -alpha (u - 1 - log u) + lc without the cancellation of the direct form (alpha up to ~5e4)
__device__ __forceinline__ void gbr_fold(GbrAcc& r, double alpha, double lc, double beta, double D)
{
    const double t = beta / D, u = t / alpha;
    double tail, lp;
    bool upper;
    if (u == INFINITY || u == 0.0) {              // t overflows (Q = 0) or beta = 0 (P = 0): density 0; a NaN beta runs on as NaN
        lp = -INFINITY;
        upper = u != 0.0;
        tail = 0.0;
    } else {
        const double pm = gbr_log1pmx(u - 1.0);
        lp = fma(-alpha, pm, lc);
        tail = gbr_gamma_tail(alpha, t, u, lp, pm, upper);
    }
    r.q += upper ? tail : 1.0 - tail;
    r.p += upper ? 1.0 - tail : tail;
    if (lp > r.m) {
        r.s = fma(r.s, exp(r.m - lp), 1.0);
        r.m = lp;
    } else if (lp != -INFINITY) {
        r.s += exp(lp - r.m);
    }
}

// CTA = (tile of TM = 2^tm_log2 models, bin b, split z); thread (mi, si) = (tid % TM, tid / TM) folds samples si, si + TS, ... of each
// 256-sample tile (TS = 256 / TM), beta staged in shared memory as br_marginal_kernel does; the TS lanes of a model then merge in a
// fixed shared-memory tree and lane 0 writes the partial (p, q, m, s) of (z, model, bin).  Same bin conventions as br_marginal_kernel.
__global__ void __launch_bounds__(GBR_NT) gbr_transform_kernel(int kind, const double* __restrict__ S, int64_t n, int ncl,
                                                               const int* __restrict__ bins, int nbins, int comp,
                                                               const double* __restrict__ dl, int64_t m, int tm_log2, int64_t chunk,
                                                               double* __restrict__ part)
{
    __shared__ double sb[GBR_NT];
    __shared__ GbrAcc red[GBR_NT];
    const int b = blockIdx.y, TM = 1 << tm_log2, TS = GBR_NT >> tm_log2;
    const int mi = threadIdx.x & (TM - 1), si = threadIdx.x >> tm_log2;
    const int64_t k = blockIdx.x * (int64_t)TM + mi;
    const int64_t nbeg = blockIdx.z * chunk, nend = min(n, nbeg + chunk);
    int l0, l1;
    const bool ok = br_bin(bins, b, ncl, l0, l1);
    double alpha = 1.0, scale = 1.0;
    const double* row = S + (int64_t)b * n;
    if (ok) {
        if (kind == GS_BR_IG) {
            alpha = ig_bin_alpha(l0, l1);
        } else {
            alpha = 0.5 * (iw_bin_nu(l0, l1) - 1.0);
            scale = 0.5;
            row = S + ((int64_t)3 * b + comp) * n;
        }
    }
    const double lc = 0.5 * log(alpha / (2.0 * GS_PI)) - gbr_stirling_rem(alpha);
    const double D = k < m ? dl[k * nbins + b] : 0.0;
    const bool live = ok && D > 0.0;
    GbrAcc acc = {0.0, 0.0, -INFINITY, 0.0};
    for (int64_t i0 = nbeg; ok && i0 < nend; i0 += GBR_NT) {
        __syncthreads();
        if (i0 + threadIdx.x < nend) sb[threadIdx.x] = scale * row[i0 + threadIdx.x];
        __syncthreads();
        const int cnt = (int)(nend - i0 < GBR_NT ? nend - i0 : GBR_NT);
        if (live)
            for (int j = si; j < cnt; j += TS) gbr_fold(acc, alpha, lc, sb[j], D);
    }
    red[threadIdx.x] = acc;
    __syncthreads();
    for (int s = TS >> 1; s > 0; s >>= 1) {
        if (si < s) red[threadIdx.x] = gbr_merge(red[threadIdx.x], red[threadIdx.x + (s << tm_log2)]);
        __syncthreads();
    }
    if (si == 0 && k < m) {
        const GbrAcc r = red[threadIdx.x];
        double* o = part + (((int64_t)blockIdx.z * m + k) * nbins + b) * 4;
        o[0] = r.p; o[1] = r.q; o[2] = r.m; o[3] = r.s;
    }
}

// thread per (model, bin): merge the P partials in ascending split order, then x = Phi^-1(F) from the smaller of F = sum Q / N and
// 1 - F = sum P / N, logm = max + log(s / N) - log D.  Broken edges: NaN; D <= 0 (or NaN), or F or 1 - F = 0 in FP64: x = -inf / +inf
// and logm = -inf.
__global__ void __launch_bounds__(GBR_NT) gbr_finish_kernel(const double* __restrict__ part, int64_t n, int ncl, const int* __restrict__ bins,
                                                            int nbins, const double* __restrict__ dl, int64_t m, int P,
                                                            double* __restrict__ x_out, double* __restrict__ logm_out)
{
    const int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x, mb = m * nbins;
    if (j >= mb) return;
    int l0, l1;
    if (!br_bin(bins, (int)(j % nbins), ncl, l0, l1)) { x_out[j] = br_nan(); logm_out[j] = br_nan(); return; }
    const double D = dl[j];
    if (!(D > 0.0)) { x_out[j] = -INFINITY; logm_out[j] = -INFINITY; return; }
    GbrAcc r = {0.0, 0.0, -INFINITY, 0.0};
    for (int p = 0; p < P; ++p) {
        const double* q = part + ((int64_t)p * mb + j) * 4;
        r = gbr_merge(r, GbrAcc{q[0], q[1], q[2], q[3]});
    }
    const double inv_n = 1.0 / (double)n, F = r.q * inv_n, G = r.p * inv_n;
    double x, lm;
    if (isnan(F) || isnan(G) || isnan(r.s)) { x = br_nan(); lm = br_nan(); }
    else {
        x = F <= 0.5 ? normcdfinv(F) : -normcdfinv(G);
        lm = (F == 0.0 || G == 0.0 || r.m == -INFINITY) ? -INFINITY : r.m + log(r.s) - log((double)n) - log(D);
    }
    x_out[j] = x;
    logm_out[j] = lm;
}

// ------------------------------------------------------------------ C ABI
extern "C" int gs_br_sample_features(int kind, const double* sigma, const double* sigma_te, const double* sigma_ee, int64_t nsamp,
                                     int ncl, const int* bins, int nbins, double* S, double* c, int accumulate, double* scratch,
                                     void* stream)
{
    GS_REQUIRE(kind == GS_BR_IG || kind == GS_BR_IW, "kind must be GS_BR_IG or GS_BR_IW");
    GS_REQUIRE(sigma && bins && S && c && scratch && (kind == GS_BR_IG || (sigma_te && sigma_ee)), "null pointer");
    GS_REQUIRE(nsamp >= 1 && ncl >= 1 && nbins >= 1 && nbins <= ncl && nbins <= 65535, "need nsamp >= 1 and 1 <= nbins <= min(ncl, 65535)");
    const dim3 grid((unsigned)((nsamp + BR_NT - 1) / BR_NT), (unsigned)nbins);
    br_sample_features_kernel<<<grid, BR_NT, 0, STREAM(stream)>>>(kind, sigma, sigma_te, sigma_ee, nsamp, ncl, bins, S, scratch);
    br_rowsum_kernel<<<(unsigned)((nsamp + BR_NT - 1) / BR_NT), BR_NT, 0, STREAM(stream)>>>(scratch, nsamp, nbins, accumulate, c);
    GS_CHECK_LAUNCH();
    return GS_OK;
}

extern "C" int gs_br_model_features(int kind, const double* dl, const double* dl_te, const double* dl_ee, int64_t nmod, int ncl,
                                    const int* bins, int nbins, double* W, double* e, int accumulate, double* scratch, void* stream)
{
    GS_REQUIRE(kind == GS_BR_IG || kind == GS_BR_IW, "kind must be GS_BR_IG or GS_BR_IW");
    GS_REQUIRE(dl && bins && W && e && scratch && (kind == GS_BR_IG || (dl_te && dl_ee)), "null pointer");
    GS_REQUIRE(nmod >= 1 && ncl >= 1 && nbins >= 1 && nbins <= ncl && nbins <= 65535, "need nmod >= 1 and 1 <= nbins <= min(ncl, 65535)");
    const dim3 grid((unsigned)((nmod + BR_NT - 1) / BR_NT), (unsigned)nbins);
    br_model_features_kernel<<<grid, BR_NT, 0, STREAM(stream)>>>(kind, dl, dl_te, dl_ee, nmod, ncl, bins, nbins, W, scratch);
    br_rowsum_kernel<<<(unsigned)((nmod + BR_NT - 1) / BR_NT), BR_NT, 0, STREAM(stream)>>>(scratch, nmod, nbins, accumulate, e);
    GS_CHECK_LAUNCH();
    return GS_OK;
}

// split of the sample axis: P = min(ceil(N / 256), ceil(2368 / ceil(M / 64))) parts of `chunk` samples (a multiple of 256); the
// last part may be shorter and P is lowered so that none is empty.  A function of (N, M) only.
static void br_split(int64_t n, int64_t m, int64_t& chunk, int& P)
{
    const int64_t units = (n + BR_SPLIT_UNIT - 1) / BR_SPLIT_UNIT, tiles = (m + 63) / 64;
    const int64_t p = std::max<int64_t>(1, std::min<int64_t>(units, (BR_TARGET_CTAS + tiles - 1) / tiles));
    chunk = BR_SPLIT_UNIT * ((units + p - 1) / p);
    P = (int)((n + chunk - 1) / chunk);
}

extern "C" int64_t gs_br_logmeanexp_scratch(int64_t nsamp, int64_t nmod)
{
    if (nsamp < 1 || nmod < 1) { gs_set_error("gs_br_logmeanexp_scratch: need nsamp, nmod >= 1"); return -1; }
    int64_t chunk;
    int P;
    br_split(nsamp, nmod, chunk, P);
    return 3 * nmod * (int64_t)P;
}

extern "C" int gs_br_logmeanexp(const double* S, const double* c, int64_t nsamp, const double* W, const double* e, int64_t nmod, int K,
                                double* scratch, double* logl_out, double* neff_out, void* stream)
{
    GS_REQUIRE(S && c && W && e && scratch && logl_out, "null pointer");
    GS_REQUIRE(nsamp >= 1 && nmod >= 1 && K >= 1, "need nsamp, nmod, K >= 1");
    int64_t chunk;
    int P;
    br_split(nsamp, nmod, chunk, P);
    cudaStream_t st = STREAM(stream);
    if (nmod <= BR_SMALL_M) {
        const dim3 grid((unsigned)((nmod + 7) / 8), (unsigned)P);
        br_logmeanexp_narrow_kernel<<<grid, BR_NT, 0, st>>>(S, c, nsamp, W, e, nmod, K, chunk, scratch);
    } else {
        const dim3 grid((unsigned)((nmod + 63) / 64), (unsigned)P);
        br_logmeanexp_dmma_kernel<<<grid, BR_NT, 0, st>>>(S, c, nsamp, W, e, nmod, K, chunk, scratch);
    }
    br_finish_kernel<<<(unsigned)nmod, BR_FIN_NT, 0, st>>>(scratch, e, nsamp, nmod, P, logl_out, neff_out);
    GS_CHECK_LAUNCH();
    return GS_OK;
}

extern "C" int gs_br_marginal(int kind, const double* S, int64_t nsamp, int ncl, const int* bins, int nbins, int comp, const double* grid,
                              int64_t grid_ld, int ngrid, double* out, void* stream)
{
    GS_REQUIRE(kind == GS_BR_IG || kind == GS_BR_IW, "kind must be GS_BR_IG or GS_BR_IW");
    GS_REQUIRE(S && bins && grid && out, "null pointer");
    GS_REQUIRE(nsamp >= 1 && ncl >= 1 && nbins >= 1 && nbins <= ncl && nbins <= 65535 && ngrid >= 1 && grid_ld >= 0,
               "need nsamp, ngrid >= 1, 1 <= nbins <= min(ncl, 65535), grid_ld >= 0");
    GS_REQUIRE(kind == GS_BR_IG ? comp == 0 : (comp == 0 || comp == 2), "comp: 0 for IG; 0 (TT) or 2 (EE) for IW");
    const dim3 g((unsigned)((ngrid + BR_NT - 1) / BR_NT), (unsigned)nbins);
    br_marginal_kernel<<<g, BR_NT, 0, STREAM(stream)>>>(kind, S, nsamp, ncl, bins, comp, grid, grid_ld, ngrid, out);
    GS_CHECK_LAUNCH();
    return GS_OK;
}

// split of the transform's sample axis: tiles = ceil(nmod / TM) nbins CTAs per split, TM = the power of two >= nmod up to 256;
// P = min(ceil(N / 256), ceil(2368 / tiles)) parts of `chunk` samples (a multiple of 256), P lowered so that none is empty.
// A function of (nsamp, nmod, nbins) only.
static void gbr_split(int64_t n, int64_t m, int nbins, int& tm_log2, int64_t& chunk, int& P)
{
    tm_log2 = 0;
    while (tm_log2 < 8 && ((int64_t)1 << tm_log2) < m) ++tm_log2;
    const int64_t units = (n + BR_SPLIT_UNIT - 1) / BR_SPLIT_UNIT, tiles = ((m + (1 << tm_log2) - 1) >> tm_log2) * nbins;
    const int64_t p = std::max<int64_t>(1, std::min<int64_t>(units, (BR_TARGET_CTAS + tiles - 1) / tiles));
    chunk = BR_SPLIT_UNIT * ((units + p - 1) / p);
    P = (int)((n + chunk - 1) / chunk);
}

extern "C" int64_t gs_gbr_transform_scratch(int64_t nsamp, int64_t nmod, int nbins)
{
    if (nsamp < 1 || nmod < 1 || nbins < 1 || nbins > 65535) {
        gs_set_error("gs_gbr_transform_scratch: need nsamp, nmod >= 1 and 1 <= nbins <= 65535");
        return -1;
    }
    int tm_log2, P;
    int64_t chunk;
    gbr_split(nsamp, nmod, nbins, tm_log2, chunk, P);
    return 4 * nmod * (int64_t)nbins * P;
}

extern "C" int gs_gbr_transform(int kind, const double* S, int64_t nsamp, int ncl, const int* bins, int nbins, int comp, const double* dl,
                                int64_t nmod, double* x_out, double* logm_out, double* scratch, void* stream)
{
    GS_REQUIRE(kind == GS_BR_IG || kind == GS_BR_IW, "kind must be GS_BR_IG or GS_BR_IW");
    GS_REQUIRE(S && bins && dl && x_out && logm_out && scratch, "null pointer");
    GS_REQUIRE(nsamp >= 1 && nmod >= 1 && ncl >= 1 && nbins >= 1 && nbins <= ncl && nbins <= 65535,
               "need nsamp, nmod >= 1 and 1 <= nbins <= min(ncl, 65535)");
    GS_REQUIRE(kind == GS_BR_IG ? comp == 0 : (comp == 0 || comp == 2), "comp: 0 for IG; 0 (TT) or 2 (EE) for IW");
    int tm_log2, P;
    int64_t chunk;
    gbr_split(nsamp, nmod, nbins, tm_log2, chunk, P);
    cudaStream_t st = STREAM(stream);
    const dim3 grid((unsigned)((nmod + (1 << tm_log2) - 1) >> tm_log2), (unsigned)nbins, (unsigned)P);
    gbr_transform_kernel<<<grid, GBR_NT, 0, st>>>(kind, S, nsamp, ncl, bins, nbins, comp, dl, nmod, tm_log2, chunk, scratch);
    gbr_finish_kernel<<<(unsigned)((nmod * nbins + GBR_NT - 1) / GBR_NT), GBR_NT, 0, st>>>(scratch, nsamp, ncl, bins, nbins, dl, nmod, P,
                                                                                          x_out, logm_out);
    GS_CHECK_LAUNCH();
    return GS_OK;
}
