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
