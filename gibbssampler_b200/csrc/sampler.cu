// Random draws, diagonal (full-sky isotropic) constrained realizations and the C_l conditional
// samplers (SURVEY.md 8a rows A10, A11, A12, A14).  All HBM-bound single-pass kernels; every
// reduction uses a fixed summation order.
#include <math.h>

#include <algorithm>

#include "gs_internal.h"
#include "rng.cuh"

#define SM_NT 256
#define SM_GRID (148 * 4)

__global__ void randn_kernel(double* __restrict__ out, int64_t n, uint64_t seed, uint64_t stream)
{
    const Philox ph(seed);
    const int64_t npair = (n + 1) >> 1;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < npair; i += (int64_t)gridDim.x * blockDim.x) {
        double a, b;
        box_muller(ph((uint64_t)i, stream), a, b);
        out[2 * i] = a;
        if (2 * i + 1 < n) out[2 * i + 1] = b;
    }
}

__global__ void randu_kernel(double* __restrict__ out, int64_t n, uint64_t seed, uint64_t stream)
{
    const Philox ph(seed);
    const int64_t npair = (n + 1) >> 1;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < npair; i += (int64_t)gridDim.x * blockDim.x) {
        const uint4 r = ph((uint64_t)i, stream);
        out[2 * i] = u01(r.x, r.y);
        if (2 * i + 1 < n) out[2 * i + 1] = u01(r.z, r.w);
    }
}

// ------------------------------------------------------------------ deterministic reductions
// out[k] = sum_i f_k(i), NR values, two launches (partials, then a single block)
template <int NR>
__device__ __forceinline__ void block_sum(double (&v)[NR], double* dst)
{
    __shared__ double sm[NR][SM_NT / 32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < NR; ++k) {
        double s = v[k];
        for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) sm[k][w] = s;
    }
    __syncthreads();
    if (threadIdx.x < NR) {
        double s = 0.0;
        for (int i = 0; i < SM_NT / 32; ++i) s += sm[threadIdx.x][i];
        dst[threadIdx.x] = s;
    }
}

__global__ void __launch_bounds__(SM_NT) sum_partial_kernel(const double* __restrict__ a, int64_t n, double* __restrict__ partials)
{
    double v[1] = {0.0};
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) v[0] += a[i];
    block_sum<1>(v, partials + blockIdx.x);
}

// -1/2 sum_p N^-1_p [ (dQ - mQ)^2 + (dU - mU)^2 ]   (NonCenteredGibbs.py:353-355); mU/dU nullable (TT: ClsSampler.py:107-108)
__global__ void __launch_bounds__(SM_NT)
chi2_partial_kernel(const double* __restrict__ dQ, const double* __restrict__ dU, const double* __restrict__ mQ,
                    const double* __restrict__ mU, const double* __restrict__ invn, int64_t n, double* __restrict__ partials)
{
    double v[1] = {0.0};
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const double a = dQ[i] - mQ[i];
        double s = a * a;
        if (dU) { const double b = dU[i] - mU[i]; s = fma(b, b, s); }
        v[0] = fma(s, invn[i], v[0]);
    }
    block_sum<1>(v, partials + blockIdx.x);
}

__global__ void __launch_bounds__(SM_NT) final_sum_kernel(const double* __restrict__ partials, int np, double scale, double* __restrict__ out)
{
    double v[1] = {0.0};
    for (int i = threadIdx.x; i < np; i += blockDim.x) v[0] += partials[i];
    __shared__ double res[1];
    block_sum<1>(v, res);
    __syncthreads();
    if (threadIdx.x == 0) out[0] = scale * res[0];
}

// ------------------------------------------------------------------ diagonal constrained realizations
// mode 0: PolarizedCenteredConstrainedRealization.sample_no_mask (CenteredGibbs.py:317-353)
//         sigma = 1/(Npix/(noise 4pi) b^2 + 1/C); s = sigma b (Npix/(noise 4pi)) d + xi sqrt(sigma)
// mode 1: PolarizedNonCenteredConstrainedRealization.sample_no_mask, all_sph (NonCenteredGibbs.py:138-176)
//         sigma = 1/(1 + b^2 C Npix/(noise 4pi)); s = sigma sqrt(C) b (Npix/(noise 4pi)) d + xi sqrt(sigma)
__global__ void cr_direct_kernel(const double* __restrict__ dl, const double* __restrict__ bl, const double* __restrict__ d_alm,
                                 const double* __restrict__ xi, double w, int L, int mode, double* __restrict__ out)
{
    const int64_t n = (int64_t)(L + 1) * (L + 1);
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int l = l_of_real(i, L);
        double c = dl[l];
        if (l) c = c * 2.0 * 3.14159265358979323846 / ((double)l * (double)(l + 1));
        const double b = bl[l];
        if (mode == 0) {
            const double ic = c != 0.0 ? 1.0 / c : 0.0;
            const double sigma = 1.0 / (w * b * b + ic);
            out[i] = sigma * (b * (w * d_alm[i])) + xi[i] * sqrt(sigma);
        } else {
            const double sigma = 1.0 / (1.0 + b * b * c * w);
            out[i] = sigma * (sqrt(c) * b * (w * d_alm[i])) + xi[i] * sqrt(sigma);
        }
    }
}

// Diagonal TT draw with the data and the noise fluctuation given as pixel-space adjoints (full sky, isotropic noise):
//   bsum = b_l (Npix/4pi) map2alm_iter3(N^-1 d) + b_l (Npix/4pi) map2alm_iter3(N^-1/2 xi_pix)   (real layout)
//   l <  l_cut (centred,     CenteredGibbs.py:100-127):  Sigma = 1/(1/C + w b^2),  s    = Sigma (bsum + xi sqrt(1/C))
//   l >= l_cut (non-centred, NonCenteredGibbs.py:22-41): Sigma = 1/(1 + C w b^2),  s_nc = Sigma (sqrt(C) bsum + xi)
// l_cut = L+1: centred sampler; 0: non-centred sampler; in between: the recovered TT PNCPConstrainedRealization.sample
// (SURVEY.md 2.3), which also zeroes the monopole / dipole entries (zero_low).
__global__ void cr_direct_pix_kernel(const double* __restrict__ dl, const double* __restrict__ bl, const double* __restrict__ bsum,
                                     const double* __restrict__ xi, double w, int L, int l_cut, int zero_low, double* __restrict__ out)
{
    const int64_t n = (int64_t)(L + 1) * (L + 1);
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int l = l_of_real(i, L);
        double c = dl[l];
        if (l) c = c * 2.0 * 3.14159265358979323846 / ((double)l * (double)(l + 1));
        const double b = bl[l];
        double v;
        if (l < l_cut) {
            const double ic = c != 0.0 ? 1.0 / c : 0.0;
            v = (bsum[i] + xi[i] * sqrt(ic)) / (ic + w * b * b);
        } else {
            v = (sqrt(c) * bsum[i] + xi[i]) / (1.0 + c * w * b * b);
        }
        if (zero_low && l < 2) v = 0.0;
        out[i] = v;
    }
}

// ------------------------------------------------------------------ inverse-gamma C_l draw
// PolarizedCenteredClsSampler.sample_one_pol / CenteredClsSampler.sample (CenteredGibbs.py:24-79):
//   beta_l = (2l+1) l (l+1) Chat_l / (4 pi); per bin: beta = sum beta_l, alpha = sum (2l+1)/2 - 1;
//   alpha[0] := 1; D_bin = beta / Gamma(alpha, 1); D[:2] := 0.
// gamma_inject (nullable): Gamma(alpha,1) variates drawn by the caller (parity with numpy's stream).
__global__ void cls_invgamma_kernel(const double* __restrict__ cl_hat, const int* __restrict__ bins, int nbins,
                                    const double* __restrict__ gamma_inject, uint64_t seed, uint64_t call,
                                    double* __restrict__ out, double* __restrict__ alpha_out, double* __restrict__ beta_out)
{
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nbins) return;
    double beta = 0.0, ex = 0.0;
    for (int l = bins[b]; l < bins[b + 1]; ++l) {
        beta += (2.0 * l + 1.0) * (double)l * (double)(l + 1) * (cl_hat[l] / (4.0 * 3.14159265358979323846));
        ex += (2.0 * l + 1.0) / 2.0;
    }
    double alpha = ex - 1.0;
    if (b == 0) alpha = 1.0;
    if (alpha_out) alpha_out[b] = alpha;
    if (beta_out) beta_out[b] = beta;
    double g;
    if (gamma_inject) g = gamma_inject[b];
    // Philox stream ids carry the consumer in the top byte: the running counters of gs_randn / gs_randu stay below 2^56, "G"amma
    // draws sit at 0x47 << 56, the inverse-Wishart draws of teb.cu at 0x57 << 56, the fused chain of gibbs_step.cu at 0x43 / 0x47 with
    // its own seed word: no consumer can walk into another one's streams however long the chain runs
    else g = alpha > 0.0 ? gamma_mt(alpha, Philox(seed), (0x47ull << 56) | (((call << 20) + (uint64_t)b) & 0x00ffffffffffffffull)) : 1.0;
    out[b] = (b < 2) ? 0.0 : beta / g;
}

// ------------------------------------------------------------------ truncated-normal proposals
// scipy.stats.truncnorm(a = -loc/scale, b = inf, loc, scale) on [0, inf): rvs by inverse CDF of a
// uniform, and logpdf (ClsSampler.py:79-92, NonCenteredGibbs.py:292-330).  Entry j <-> bin j + 2.
__global__ void truncnorm_propose_kernel(const double* __restrict__ dl_old, const double* __restrict__ prop_var, int nbins,
                                         const double* __restrict__ u, double* __restrict__ dl_new)
{
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nbins) return;
    if (b < 2) { dl_new[b] = 0.0; return; }
    const double loc = dl_old[b], sc = sqrt(prop_var[b - 2]), a = -loc / sc, q = u[b - 2];
    double t;
    if (a < 0.0) { const double pa = normcdf(a); t = normcdfinv(fma(q, 1.0 - pa, pa)); }
    else { const double sa = normcdf(-a); t = -normcdfinv((1.0 - q) * sa); }
    dl_new[b] = fmax(loc + sc * t, 0.0);
}

// logpdf(x; loc = from, scale) - used as log q(from -> x); out[0], out[1] = 0
__global__ void truncnorm_logpdf_kernel(const double* __restrict__ x, const double* __restrict__ from,
                                        const double* __restrict__ prop_var, int nbins, double* __restrict__ out)
{
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nbins) return;
    if (b < 2) { out[b] = 0.0; return; }
    const double loc = from[b], sc = sqrt(prop_var[b - 2]), a = -loc / sc, t = (x[b] - loc) / sc;
    const double logz = log(normcdf(-a));  // log(1 - Phi(a))
    out[b] = (x[b] < 0.0) ? -INFINITY : -0.5 * t * t - 0.91893853320467274178 - log(sc) - logz;
}

// ------------------------------------------------------------------ C ABI
#define STREAM(s) ((cudaStream_t)(s))
static inline int nblk(int64_t n) { return (int)std::min<int64_t>((n + SM_NT - 1) / SM_NT, SM_GRID); }

extern "C" int gs_randn(double* out, int64_t n, uint64_t seed, uint64_t stream_id, void* stream)
{
    GS_REQUIRE(out && n >= 0, "bad arguments");
    if (n == 0) return GS_OK;
    randn_kernel<<<nblk((n + 1) / 2), SM_NT, 0, STREAM(stream)>>>(out, n, seed, stream_id);
    GS_CHECK_LAUNCH();
    return GS_OK;
}

extern "C" int gs_randu(double* out, int64_t n, uint64_t seed, uint64_t stream_id, void* stream)
{
    GS_REQUIRE(out && n >= 0, "bad arguments");
    if (n == 0) return GS_OK;
    randu_kernel<<<nblk((n + 1) / 2), SM_NT, 0, STREAM(stream)>>>(out, n, seed, stream_id);
    GS_CHECK_LAUNCH();
    return GS_OK;
}

extern "C" int gs_sum(const double* a, int64_t n, double* scratch, double* out, void* stream)
{
    GS_REQUIRE(a && scratch && out && n >= 0, "bad arguments (scratch needs 592 doubles)");
    sum_partial_kernel<<<SM_GRID, SM_NT, 0, STREAM(stream)>>>(a, n, scratch);
    final_sum_kernel<<<1, SM_NT, 0, STREAM(stream)>>>(scratch, SM_GRID, 1.0, out);
    GS_CHECK_LAUNCH();
    return GS_OK;
}

extern "C" int gs_loglik_pix(const double* d_Q, const double* d_U, const double* m_Q, const double* m_U,
                             const double* inv_noise, int64_t npix, double* scratch, double* out, void* stream)
{
    GS_REQUIRE(d_Q && m_Q && inv_noise && scratch && out && npix > 0 && ((d_U == nullptr) == (m_U == nullptr)), "bad arguments");
    chi2_partial_kernel<<<SM_GRID, SM_NT, 0, STREAM(stream)>>>(d_Q, d_U, m_Q, m_U, inv_noise, npix, scratch);
    final_sum_kernel<<<1, SM_NT, 0, STREAM(stream)>>>(scratch, SM_GRID, -0.5, out);
    GS_CHECK_LAUNCH();
    return GS_OK;
}

// compute_log_likelihood_all_sph (NonCenteredGibbs.py:357-377): full sky, isotropic noise, everything in harmonic space:
//   -1/2 w sum_i [(dE_i - flE_l(i) sE_i)^2 + (dB_i - flB_l(i) sB_i)^2],  i over the real alm layout, fl = b_l sqrt(C_l),
//   w = N^-1 Npix / 4 pi.  Thread per complex coefficient c = idx(l, m): real-layout entry l (m = 0) or 2 c - (L+1) + {0,1}.
__global__ void __launch_bounds__(SM_NT)
loglik_alm_partial_kernel(const double* __restrict__ dE, const double* __restrict__ dB, const double* __restrict__ sE,
                          const double* __restrict__ sB, const double* __restrict__ flE, const double* __restrict__ flB, int L,
                          double* __restrict__ partials)
{
    double v[1] = {0.0};
    const int64_t nm = L + 1, total = nm * (nm + 1) / 2;   // complex coefficients, m-major
    for (int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; c < total; c += (int64_t)gridDim.x * blockDim.x) {
        // c = idx(l, m) = m (2L + 1 - m) / 2 + l, l = m..L: column m starts at s_m = m (2L + 3 - m) / 2 <= c
        const double t = 2.0 * L + 3.0;
        int m = (int)((t - sqrt(fmax(t * t - 8.0 * (double)c, 0.0))) * 0.5);
        m = max(0, min(m, L));
        while (m > 0 && (int64_t)m * (2 * L + 3 - m) / 2 > c) --m;
        while (m < L && (int64_t)(m + 1) * (2 * L + 3 - (m + 1)) / 2 <= c) ++m;
        const int l = (int)(c - (int64_t)m * (2 * L + 1 - m) / 2);
        const double fe = flE[l], fb = flB[l];
        if (m == 0) {
            const double a = dE[l] - fe * sE[l], b = dB[l] - fb * sB[l];
            v[0] += a * a + b * b;
        } else {
            const int64_t off = 2 * c - nm;
            const double a0 = dE[off] - fe * sE[off], a1 = dE[off + 1] - fe * sE[off + 1];
            const double b0 = dB[off] - fb * sB[off], b1 = dB[off + 1] - fb * sB[off + 1];
            v[0] += a0 * a0 + a1 * a1 + b0 * b0 + b1 * b1;
        }
    }
    block_sum<1>(v, partials + blockIdx.x);
}

extern "C" int gs_loglik_alm(const double* d_E, const double* d_B, const double* s_E, const double* s_B, const double* fl_E,
                             const double* fl_B, int lmax, double weight, double* scratch, double* out, void* stream)
{
    GS_REQUIRE(d_E && d_B && s_E && s_B && fl_E && fl_B && scratch && out && lmax >= 0, "bad arguments (scratch needs 592 doubles)");
    loglik_alm_partial_kernel<<<SM_GRID, SM_NT, 0, STREAM(stream)>>>(d_E, d_B, s_E, s_B, fl_E, fl_B, lmax, scratch);
    final_sum_kernel<<<1, SM_NT, 0, STREAM(stream)>>>(scratch, SM_GRID, -0.5 * weight, out);
    GS_CHECK_LAUNCH();
    return GS_OK;
}

extern "C" int gs_cr_direct(const double* dl, const double* bl, const double* d_alm, const double* xi, double npix_over_noise_4pi,
                            int lmax, int mode, double* out, void* stream)
{
    GS_REQUIRE(dl && bl && d_alm && xi && out && lmax >= 0 && (mode == 0 || mode == 1), "bad arguments");
    cr_direct_kernel<<<nblk((int64_t)(lmax + 1) * (lmax + 1)), SM_NT, 0, STREAM(stream)>>>(dl, bl, d_alm, xi, npix_over_noise_4pi, lmax, mode, out);
    GS_CHECK_LAUNCH();
    return GS_OK;
}

extern "C" int gs_cr_direct_pix(const double* dl, const double* bl, const double* bsum, const double* xi, double npix_over_noise_4pi,
                                int lmax, int l_cut, int zero_low, double* out, void* stream)
{
    GS_REQUIRE(dl && bl && bsum && xi && out && lmax >= 0 && l_cut >= 0, "bad arguments");
    cr_direct_pix_kernel<<<nblk((int64_t)(lmax + 1) * (lmax + 1)), SM_NT, 0, STREAM(stream)>>>(dl, bl, bsum, xi, npix_over_noise_4pi, lmax,
                                                                                                l_cut, zero_low, out);
    GS_CHECK_LAUNCH();
    return GS_OK;
}

extern "C" int gs_cls_invgamma(const double* cl_hat, const int* bins, int nbins, const double* gamma_inject,
                               uint64_t seed, uint64_t call, double* dl_binned, double* alpha_out, double* beta_out,
                               void* stream)
{
    GS_REQUIRE(cl_hat && bins && dl_binned && nbins >= 1, "bad arguments");
    cls_invgamma_kernel<<<(nbins + 127) / 128, 128, 0, STREAM(stream)>>>(cl_hat, bins, nbins, gamma_inject, seed, call, dl_binned, alpha_out, beta_out);
    GS_CHECK_LAUNCH();
    return GS_OK;
}

extern "C" int gs_truncnorm_propose(const double* dl_old, const double* prop_var, int nbins, const double* u,
                                    double* dl_new, void* stream)
{
    GS_REQUIRE(dl_old && prop_var && u && dl_new && nbins >= 2, "bad arguments");
    truncnorm_propose_kernel<<<(nbins + 127) / 128, 128, 0, STREAM(stream)>>>(dl_old, prop_var, nbins, u, dl_new);
    GS_CHECK_LAUNCH();
    return GS_OK;
}

extern "C" int gs_truncnorm_logpdf(const double* x, const double* from, const double* prop_var, int nbins, double* out,
                                   void* stream)
{
    GS_REQUIRE(x && from && prop_var && out && nbins >= 2, "bad arguments");
    truncnorm_logpdf_kernel<<<(nbins + 127) / 128, 128, 0, STREAM(stream)>>>(x, from, prop_var, nbins, out);
    GS_CHECK_LAUNCH();
    return GS_OK;
}

// ------------------------------------------------------------------ Metropolis-within-Gibbs on binned D_l
// (PolarizationNonCenteredClsSampler.sample, NonCenteredGibbs.py:401-445; blocks index the BINNED arrays)
__device__ __forceinline__ double binned_value(const double* cur, const double* prop, const int* bins, int nbins,
                                               int l, bool use_prop, int b0, int b1)
{
    if (l < bins[0] || l >= bins[nbins]) return 0.0;
    int lo = 0, hi = nbins - 1;
    while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (bins[mid] <= l) lo = mid; else hi = mid - 1; }
    return (use_prop && lo >= b0 && lo < b1) ? prop[lo] : cur[lo];
}

// Per-l synthesis filters of the candidate state: cand = cur with bins [b0,b1) of spectrum `pol` (0 = EE,
// 1 = BB, -1 = none) replaced by the proposal.  fl_X[l] = b_l sqrt(C^X_l), C_l = D_l 2pi/(l(l+1)); for
// l < l_cut (partially non-centred parametrisation) fl_X[l] = b_l.
__global__ void mwg_filters_kernel(const double* cur_E, const double* cur_B, const double* prop_E, const double* prop_B,
                                   const int* bins_E, int nb_E, const int* bins_B, int nb_B, int pol, int b0, int b1,
                                   const double* bl, int L, int l_cut, double* flE, double* flB)
{
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l > L) return;
    double dE = binned_value(cur_E, prop_E, bins_E, nb_E, l, pol == 0, b0, b1);
    double dB = binned_value(cur_B, prop_B, bins_B, nb_B, l, pol == 1, b0, b1);
    const double f = l ? 2.0 * 3.14159265358979323846 / ((double)l * (double)(l + 1)) : 1.0;
    flE[l] = bl[l] * (l < l_cut ? 1.0 : sqrt(dE * f));
    flB[l] = bl[l] * (l < l_cut ? 1.0 : sqrt(dB * f));
}

// One Metropolis accept/reject of block [b0,b1) of spectrum pol, entirely on the device:
//   log r = sum_{b in block} logr[b] + new_lik - old_lik ; accept iff log(u) < log r
__global__ void mwg_accept_kernel(double* cur, const double* prop, const double* logr, int b0, int b1,
                                  const double* new_lik, double* old_lik, const double* u, int* accept_out)
{
    if (blockIdx.x || threadIdx.x) return;
    double s = 0.0;
    for (int b = b0; b < b1; ++b) s += logr[b];
    const double log_r = s + (new_lik[0] - old_lik[0]);
    const bool acc = log(u[0]) < log_r;
    if (acc) {
        for (int b = b0; b < b1; ++b) cur[b] = prop[b];
        old_lik[0] = new_lik[0];
    }
    accept_out[0] = acc ? 1 : 0;
}

__global__ void mul_kernel(const double* a, const double* b, double* out, int64_t n)
{
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) out[i] = a[i] * b[i];
}

extern "C" int gs_mwg_filters(const double* cur_E, const double* cur_B, const double* prop_E, const double* prop_B,
                              const int* bins_E, int nbins_E, const int* bins_B, int nbins_B, int pol, int b_start,
                              int b_end, const double* bl, int lmax, int l_cut, double* flE, double* flB, void* stream)
{
    GS_REQUIRE(cur_E && cur_B && bins_E && bins_B && bl && flE && flB && nbins_E >= 1 && nbins_B >= 1 && lmax >= 0, "bad arguments");
    GS_REQUIRE(pol == -1 || ((pol == 0 || pol == 1) && prop_E && prop_B && b_start >= 0 && b_end >= b_start), "bad block");
    mwg_filters_kernel<<<(lmax + 128) / 128, 128, 0, STREAM(stream)>>>(cur_E, cur_B, prop_E, prop_B, bins_E, nbins_E, bins_B, nbins_B,
                                                                       pol, b_start, b_end, bl, lmax, l_cut, flE, flB);
    GS_CHECK_LAUNCH();
    return GS_OK;
}

extern "C" int gs_mwg_accept(double* cur, const double* prop, const double* logr, int b_start, int b_end,
                             const double* new_lik, double* old_lik, const double* u, int* accept_out, void* stream)
{
    GS_REQUIRE(cur && prop && logr && new_lik && old_lik && u && accept_out && b_start >= 0 && b_end >= b_start, "bad arguments");
    mwg_accept_kernel<<<1, 32, 0, STREAM(stream)>>>(cur, prop, logr, b_start, b_end, new_lik, old_lik, u, accept_out);
    GS_CHECK_LAUNCH();
    return GS_OK;
}

extern "C" int gs_mul(const double* a, const double* b, double* out, int64_t n, void* stream)
{
    GS_REQUIRE(a && b && out && n >= 0, "bad arguments");
    if (n == 0) return GS_OK;
    mul_kernel<<<nblk(n), SM_NT, 0, STREAM(stream)>>>(a, b, out, n);
    GS_CHECK_LAUNCH();
    return GS_OK;
}

// ------------------------------------------------------------------ block-batched Metropolis-within-Gibbs sweep
// SURVEY.md 8f row 1.  The likelihood is -1/2 sum_p N^-1_p |d_p - M_p|^2 with M = A (fl (.) s_nc) linear in the per-l
// filter fl, and every Metropolis block touches its own multipoles only.  So with r = d - M(current state) and
//   dM_k = A (dfl_k (.) s_nc),  dfl_k[l] = b_l (sqrt(C'_l) - sqrt(C_l)) on block k, 0 elsewhere,
// the candidate likelihood of block k is -1/2 sum N^-1 (r - dM_k)^2 and an acceptance is r -= dM_k.  All dM_k of a
// group of blocks come out of ONE Legendre pass (leg_synth_blocks_kernel) and one batched ring-FFT launch; each
// Metropolis test is then one launch (mwg_step_kernel), nothing leaves the device.
__global__ void mwg_dfl_kernel(const double* cur_E, const double* cur_B, const double* prop_E, const double* prop_B,
                               const int* bins_E, int nb_E, const int* bins_B, int nb_B, int eb0, int eb1, int bb0, int bb1,
                               const double* bl, int L, int l_cut, double* flE, double* flB, double* dflE, double* dflB)
{
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l > L) return;
    const double f = l ? 2.0 * 3.14159265358979323846 / ((double)l * (double)(l + 1)) : 1.0;
    const double cE = binned_value(cur_E, prop_E, bins_E, nb_E, l, false, 0, 0);
    const double cB = binned_value(cur_B, prop_B, bins_B, nb_B, l, false, 0, 0);
    const double pE = binned_value(cur_E, prop_E, bins_E, nb_E, l, true, eb0, eb1);
    const double pB = binned_value(cur_B, prop_B, bins_B, nb_B, l, true, bb0, bb1);
    const bool nc = l >= l_cut;
    flE[l] = bl[l] * (nc ? sqrt(cE * f) : 1.0);
    flB[l] = bl[l] * (nc ? sqrt(cB * f) : 1.0);
    dflE[l] = nc ? bl[l] * (sqrt(pE * f) - sqrt(cE * f)) : 0.0;
    dflB[l] = nc ? bl[l] * (sqrt(pB * f) - sqrt(cB * f)) : 0.0;
}

// r = d - m (in place over m) and the chi^2 partials of the current state
__global__ void __launch_bounds__(SM_NT)
mwg_resid_kernel(const double* __restrict__ dQ, const double* __restrict__ dU, double* __restrict__ mQ, double* __restrict__ mU,
                 const double* __restrict__ invn, int64_t n, double* __restrict__ partials)
{
    double v[1] = {0.0};
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const double a = dQ[i] - mQ[i], b = dU[i] - mU[i];
        mQ[i] = a; mU[i] = b;
        v[0] = fma(fma(b, b, a * a), invn[i], v[0]);
    }
    block_sum<1>(v, partials + blockIdx.x);
}

// r -= (gQ, gU) when the last test accepted (*do_apply != 0): the pending update of mwg_step_kernel, applied on its own
// before the block maps it reads are overwritten
__global__ void __launch_bounds__(SM_NT)
mwg_apply_kernel(double* __restrict__ rQ, double* __restrict__ rU, const double* __restrict__ gQ, const double* __restrict__ gU,
                 int64_t n, const int* __restrict__ do_apply)
{
    if (*do_apply == 0) return;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        rQ[i] -= gQ[i];
        rU[i] -= gU[i];
    }
}

// One Metropolis test in one launch: the r update of the PREVIOUS test (pend_flag, maps pQ / pU) is applied as r is read, the
// chi^2 partials of the candidate r - dM_k follow (the block's change is already in r when *applied != 0), and the block that
// finishes last sums them in a fixed order and takes the decision: lik[0] = old, lik[1] = new likelihood.  pend_flag may alias
// do_apply_out and `applied` is written by the deciding block only: every block reads both before its loop, and the decision
// comes after all loops (counter).
__global__ void __launch_bounds__(SM_NT)
mwg_step_kernel(double* __restrict__ rQ, double* __restrict__ rU, const double* __restrict__ pQ, const double* __restrict__ pU,
                const int* pend_flag, const double* __restrict__ gQ, const double* __restrict__ gU,
                const double* __restrict__ invn, int64_t n, double* partials, unsigned* counter, double* cur,
                const double* prop, const double* logr, int b0, int b1, double* lik, const double* u, int* applied, int* do_apply_out,
                int* accept_out)
{
    const bool pend = pQ != nullptr && *pend_flag != 0;
    const bool sub = *applied == 0;
    double v[1] = {0.0};
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        double a = rQ[i], b = rU[i];
        if (pend) { a -= pQ[i]; b -= pU[i]; rQ[i] = a; rU[i] = b; }
        if (sub) { a -= gQ[i]; b -= gU[i]; }
        v[0] = fma(fma(b, b, a * a), invn[i], v[0]);
    }
    block_sum<1>(v, partials + blockIdx.x);
    __shared__ int last;
    if (threadIdx.x == 0) {
        __threadfence();
        last = atomicAdd(counter, 1u) == gridDim.x - 1 ? 1 : 0;
    }
    __syncthreads();
    if (!last) return;
    __threadfence();
    double s[1] = {0.0};
    for (int i = threadIdx.x; i < (int)gridDim.x; i += blockDim.x) s[0] += __ldcg(partials + i);
    __shared__ double res[1];
    block_sum<1>(s, res);
    __syncthreads();
    if (threadIdx.x) return;
    *counter = 0u;
    const double new_lik = -0.5 * res[0];
    double t = 0.0;
    for (int b = b0; b < b1; ++b) t += logr[b];
    const bool acc = log(u[0]) < t + (new_lik - lik[0]);
    int apply = 0;
    if (acc) {
        lik[0] = new_lik;
        if (*applied == 0) {
            for (int b = b0; b < b1; ++b) cur[b] = prop[b];
            *applied = 1;
            apply = 1;
        }
    }
    lik[1] = new_lik;
    *do_apply_out = apply;
    accept_out[0] = acc ? 1 : 0;
}

__global__ void mwg_first_lik_kernel(const double* partials, int np, double* lik)
{
    double v[1] = {0.0};
    for (int i = threadIdx.x; i < np; i += blockDim.x) v[0] += partials[i];
    __shared__ double res[1];
    block_sum<1>(v, res);
    __syncthreads();
    if (threadIdx.x == 0) lik[0] = lik[1] = -0.5 * res[0];
}

extern "C" int gs_mwg_sweep_blocks(gs_plan* p, const double* snc_E, const double* snc_B, double* cur_E, double* cur_B,
                                   const double* prop_E, const double* prop_B, const double* logr_E, const double* logr_B,
                                   const int* bins_E_host, int nbins_E, const int* bins_B_host, int nbins_B,
                                   const int* blocks_E_host, int nblk_E, const int* blocks_B_host, int nblk_B, int n_iter,
                                   const double* bl, int l_cut, const double* d_Q, const double* d_U, const double* inv_noise,
                                   const double* u, int* accept_out, double* loglik_out, int64_t workspace_bytes, void* stream)
{
    if (!p) { gs_set_error("null plan"); return GS_E_BADARG; }
    GS_CHECK_CUDA(cudaSetDevice(p->device));
    GS_REQUIRE(snc_E && snc_B && cur_E && cur_B && prop_E && prop_B && logr_E && logr_B && bins_E_host && bins_B_host && bl && d_Q &&
                   d_U && inv_noise && u && accept_out && nbins_E >= 1 && nbins_B >= 1 && nblk_E >= 0 && nblk_B >= 0 && n_iter >= 1 &&
                   l_cut >= 0,
               "bad arguments");
    GS_REQUIRE((nblk_E == 0 || blocks_E_host) && (nblk_B == 0 || blocks_B_host), "null block list");
    GS_REQUIRE(p->world == 1 && p->nsjobs2 == 0, "needs an unsharded plan without split rings (NSIDE <= 1024)");
    const int L = p->d.lmax, nring = p->d.nring;
    const int64_t npix = p->d.npix;
    cudaStream_t st = STREAM(stream);
    // ---- block boundaries in l; blocks index the binned arrays (NonCenteredGibbs.py:421-426)
    std::vector<int> meta;  // [bins_E | bins_B | lbE | lbB | mmax per block (E blocks then B blocks)]
    auto check_blocks = [&](const int* blocks, int nblk, const int* bins, int nbins) {
        for (int i = 0; i <= nblk && nblk > 0; ++i)
            if (blocks[i] < 0 || blocks[i] > nbins || (i && blocks[i] <= blocks[i - 1])) return false;
        return true;
    };
    GS_REQUIRE(check_blocks(blocks_E_host, nblk_E, bins_E_host, nbins_E) && check_blocks(blocks_B_host, nblk_B, bins_B_host, nbins_B),
               "block boundaries must be increasing bin indices");
    meta.insert(meta.end(), bins_E_host, bins_E_host + nbins_E + 1);
    meta.insert(meta.end(), bins_B_host, bins_B_host + nbins_B + 1);
    const int off_lbE = (int)meta.size();
    for (int i = 0; i <= nblk_E && nblk_E > 0; ++i) meta.push_back(std::min(bins_E_host[blocks_E_host[i]], L + 1));
    if (nblk_E == 0) meta.push_back(0);
    const int off_lbB = (int)meta.size();
    for (int i = 0; i <= nblk_B && nblk_B > 0; ++i) meta.push_back(std::min(bins_B_host[blocks_B_host[i]], L + 1));
    if (nblk_B == 0) meta.push_back(0);
    const int off_mmax = (int)meta.size();
    // a block that ends at l <= 2 has no spin-2 multipole: mmax = -1 makes its (never written) spectra slot read as zero
    for (int i = 0; i < nblk_E; ++i) meta.push_back(meta[off_lbE + i + 1] <= 2 ? -1 : meta[off_lbE + i + 1] - 1);
    for (int i = 0; i < nblk_B; ++i) meta.push_back(meta[off_lbB + i + 1] <= 2 ? -1 : meta[off_lbB + i + 1] - 1);
    const int ntot = nblk_E + nblk_B;
    // ---- workspace (plan-owned, grown on demand): group of G blocks
    const int64_t slotF = 2LL * nring * (L + 1);  // double2 per block
    const int64_t per_block = slotF * 16 + 2 * npix * 8;
    if (workspace_bytes <= 0) workspace_bytes = 8LL << 30;
    int G = (int)std::max<int64_t>(1, std::min<int64_t>(std::max(ntot, 1), workspace_bytes / per_block));
    if (G > p->mwg_group) {
        if (p->mwg_F) { cudaFree(p->mwg_F); cudaFree(p->mwg_maps); p->mwg_F = nullptr; p->mwg_maps = nullptr; p->mwg_group = 0; }
        GS_CHECK_CUDA(cudaMalloc(&p->mwg_F, (size_t)G * slotF * 16));
        GS_CHECK_CUDA(cudaMalloc(&p->mwg_maps, (size_t)G * 2 * npix * 8));
        // rings without pixel weight are not synthesised below: their (never written) pixels meet N^-1 = 0 and must be finite
        GS_CHECK_CUDA(cudaMemsetAsync(p->mwg_maps, 0, (size_t)G * 2 * npix * 8, st));
        p->mwg_group = G;
    }
    G = p->mwg_group;
    if (!p->mwg_small) {
        GS_CHECK_CUDA(cudaMalloc(&p->mwg_small, (SM_GRID + 8 + 4 * (size_t)(L + 1)) * sizeof(double)));
    }
    if (meta != p->mwg_meta_host) {
        GS_CHECK_CUDA(cudaStreamSynchronize(st));
        if (p->mwg_meta) cudaFree(p->mwg_meta);
        p->mwg_meta = nullptr;
        GS_CHECK_CUDA(cudaMalloc(&p->mwg_meta, (meta.size() + ntot + 4) * sizeof(int)));
        GS_CHECK_CUDA(cudaMemcpy(p->mwg_meta, meta.data(), meta.size() * sizeof(int), cudaMemcpyHostToDevice));
        p->mwg_meta_host = meta;
    }
    const int* bins_E = p->mwg_meta;
    const int* bins_B = p->mwg_meta + nbins_E + 1;
    const int* lbE = p->mwg_meta + off_lbE;
    const int* lbB = p->mwg_meta + off_lbB;
    const int* mmax = p->mwg_meta + off_mmax;
    int* flags = p->mwg_meta + meta.size();  // [ntot] applied, then do_apply, then the ticket counter of mwg_step_kernel
    int* do_apply = flags + ntot;
    unsigned* ticket = reinterpret_cast<unsigned*>(flags + ntot + 1);
    double* partials = p->mwg_small;
    double* lik = partials + SM_GRID;
    double* flE = lik + 8;
    double* flB = flE + (L + 1);
    double* dflE = flB + (L + 1);
    double* dflB = dflE + (L + 1);
    double* rQ = p->mapQ_tmp;
    double* rU = p->mapU_tmp;

    GS_CHECK_CUDA(cudaMemsetAsync(flags, 0, (ntot + 2) * sizeof(int), st));
    // block maps are only ever weighted by N^-1: the rings on which it vanishes identically need no ring FFT
    // Rings on which N^-1 is one number w (isotropic noise, not cut by the mask edge; gs_set_ring_const): every quantity of the sweep
    // on such a ring is w sum_j |z_j - z'_j|^2 with z = Q + i U, which the unitary DFT along the ring leaves unchanged.  Data, current
    // model and all block maps of these rings are therefore kept as sqrt(n) times the alias-folded ring spectrum (what the ring FFT
    // would start from) and their FFTs are never run; the Metropolis test kernels see ordinary arrays.
    const unsigned char* ract = nullptr;
    const double* wconst = nullptr;
    if (g_gs_ring_skip) {
        int rc0 = gs_active_rings_build(p, inv_noise, st);
        if (rc0) return rc0;
        ract = p->act_ring;
        if (g_gs_ring_const && p->ring_wconst) wconst = p->ring_wconst;
    }
    const double* dTQ = d_Q;
    const double* dTU = d_U;
    if (wconst) {
        if (!p->mwg_data) GS_CHECK_CUDA(cudaMalloc(&p->mwg_data, (size_t)2 * npix * sizeof(double)));
        int rc0 = gs_ring_mwg_data(p, d_Q, d_U, p->mwg_data, p->mwg_data + npix, wconst, st);
        if (rc0) return rc0;
        dTQ = p->mwg_data;
        dTU = p->mwg_data + npix;
    }
    const int eb0 = nblk_E ? blocks_E_host[0] : 0, eb1 = nblk_E ? blocks_E_host[nblk_E] : 0;
    const int bb0 = nblk_B ? blocks_B_host[0] : 0, bb1 = nblk_B ? blocks_B_host[nblk_B] : 0;
    mwg_dfl_kernel<<<(L + 128) / 128, 128, 0, st>>>(cur_E, cur_B, prop_E, prop_B, bins_E, nbins_E, bins_B, nbins_B, eb0, eb1, bb0, bb1,
                                                    bl, L, l_cut, flE, flB, dflE, dflB);
    GS_CHECK_LAUNCH();
    int rc;
    if ((rc = gs_leg_synth(p, 2, snc_E, snc_B, GS_ALM_REAL, flE, st, nullptr, flB))) return rc;
    if ((rc = gs_ring_synth(p, 2, rQ, rU, st, nullptr, 1, 0, wconst))) return rc;
    mwg_resid_kernel<<<SM_GRID, SM_NT, 0, st>>>(dTQ, dTU, rQ, rU, inv_noise, npix, partials);
    mwg_first_lik_kernel<<<1, SM_NT, 0, st>>>(partials, SM_GRID, lik);
    GS_CHECK_LAUNCH();
    g_gs_launches += 4;

    const double* pQ = nullptr;   // maps of the previous test: mwg_step_kernel applies its r update as the next test reads r
    const double* pU = nullptr;
    for (int g0 = 0; g0 < ntot; g0 += G) {
        const int g1 = std::min(ntot, g0 + G), ng = g1 - g0;
        if (pQ) {   // the block maps are about to be overwritten: apply the pending update now
            mwg_apply_kernel<<<SM_GRID, SM_NT, 0, st>>>(rQ, rU, pQ, pU, npix, do_apply);
            pQ = pU = nullptr;
            g_gs_launches += 1;
        }
        const int e0 = std::min(g0, nblk_E), e1 = std::min(g1, nblk_E);
        const int b0 = std::max(g0 - nblk_E, 0), b1 = std::max(g1 - nblk_E, 0);
        int lend = 0;
        if (e1 > e0) lend = std::max(lend, meta[off_lbE + e1]);
        if (b1 > b0) lend = std::max(lend, meta[off_lbB + b1]);
        lend = std::min(lend, L + 1);
        if ((rc = gs_leg_synth_blocks(p, snc_E, snc_B, dflE, dflB, lbE, e0, e1, lbB, b0, b1, lend, p->mwg_F, st))) return rc;
        if ((rc = gs_ring_synth_batch(p, p->mwg_F, slotF, mmax + g0, p->mwg_maps, p->mwg_maps + (int64_t)G * npix, npix, ng, st, ract, wconst)))
            return rc;
        for (int k = g0; k < g1; ++k) {
            const bool isE = k < nblk_E;
            const int* blocks = isE ? blocks_E_host : blocks_B_host;
            const int i = isE ? k : k - nblk_E;
            const double* gQ = p->mwg_maps + (int64_t)(k - g0) * npix;
            const double* gU = p->mwg_maps + (int64_t)(G + k - g0) * npix;
            for (int it = 0; it < n_iter; ++it) {
                const int64_t idx = (int64_t)k * n_iter + it;
                mwg_step_kernel<<<SM_GRID, SM_NT, 0, st>>>(rQ, rU, pQ, pU, do_apply, gQ, gU, inv_noise, npix, partials, ticket,
                                                           isE ? cur_E : cur_B, isE ? prop_E : prop_B, isE ? logr_E : logr_B, blocks[i],
                                                           blocks[i + 1], lik, u + idx, flags + k, do_apply, accept_out + idx);
                pQ = gQ; pU = gU;
                g_gs_launches += 1;
            }
        }
        GS_CHECK_LAUNCH();
    }
    if (loglik_out) GS_CHECK_CUDA(cudaMemcpyAsync(loglik_out, lik, sizeof(double), cudaMemcpyDeviceToDevice, st));
    return GS_OK;
}

// ------------------------------------------------------------------ auxiliary-variable CR sampler (pixel / alm updates)
// sample_gibbs_change_variable / overrelaxation_sampler (CenteredGibbs.py:676-825):
//   v | s : v = mean_v + [alpha (v_old - mean_v)] + sqrt(1 - alpha^2) sqrt(gamma) xi,  gamma = mu - N^-1, mean_v = gamma (A B s)
//   out   = v + N^-1 d  (the map handed to map2alm for the s | v step); v itself is kept in v_io
__global__ void aux_v_kernel(const double* __restrict__ map, const double* __restrict__ inv_noise, const double* __restrict__ d,
                             const double* __restrict__ xi, double mu, double alpha, double* v_io, double* __restrict__ out, int64_t n)
{
    const double sq = sqrt(1.0 - alpha * alpha);
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const double g = mu - inv_noise[i];
        const double mean = g * map[i];
        double v = mean + sq * xi[i] * sqrt(g);
        if (alpha != 0.0) v += alpha * (v_io[i] - mean);
        v_io[i] = v;
        out[i] = v + inv_noise[i] * d[i];
    }
}

//   s | v : var_s = 1 / ((mu/w) b_l^2 + 1/C_l), mean_s = var_s * badj  (badj = b_l A^T (v + N^-1 d), real layout)
//           s = mean_s + alpha (s_old - mean_s) + sqrt(1 - alpha^2) sqrt(var_s) xi
__global__ void aux_s_kernel(const double* __restrict__ badj, const double* __restrict__ dl, const double* __restrict__ bl,
                             const double* __restrict__ xi, double mu_over_w, double alpha, int L, double* s_io)
{
    const int64_t n = (int64_t)(L + 1) * (L + 1);
    const double sq = sqrt(1.0 - alpha * alpha);
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int l = l_of_real(i, L);
        double c = dl[l];
        if (l) c = c * 2.0 * 3.14159265358979323846 / ((double)l * (double)(l + 1));
        const double ic = c != 0.0 ? 1.0 / c : 0.0;
        const double var = 1.0 / (mu_over_w * bl[l] * bl[l] + ic);
        const double mean = var * badj[i];
        double s = mean + sq * xi[i] * sqrt(var);
        if (alpha != 0.0) s += alpha * (s_io[i] - mean);
        s_io[i] = s;
    }
}

// per-l factor of the partially non-centred parametrisation: f_l = 1 for l < l_cut, sqrt(1/C_l) (mode 0) or
// sqrt(C_l) (mode 1) for l >= l_cut (0 where C_l = 0)
__global__ void pncp_factor_kernel(const double* __restrict__ dl, int L, int l_cut, int mode, double* __restrict__ out)
{
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l > L) return;
    double c = dl[l];
    if (l) c = c * 2.0 * 3.14159265358979323846 / ((double)l * (double)(l + 1));
    double f = 1.0;
    if (l >= l_cut) f = mode ? sqrt(c) : (c != 0.0 ? sqrt(1.0 / c) : 0.0);
    out[l] = f;
}

extern "C" int gs_aux_v_update(const double* map, const double* inv_noise, const double* d, const double* xi, double mu,
                               double alpha, double* v_io, double* out, int64_t npix, void* stream)
{
    GS_REQUIRE(map && inv_noise && d && xi && v_io && out && npix > 0 && alpha > -1.0 && alpha < 1.0, "bad arguments");
    aux_v_kernel<<<nblk(npix), SM_NT, 0, STREAM(stream)>>>(map, inv_noise, d, xi, mu, alpha, v_io, out, npix);
    GS_CHECK_LAUNCH();
    return GS_OK;
}

extern "C" int gs_aux_s_update(const double* badj, const double* dl, const double* bl, const double* xi, double mu_over_w,
                               double alpha, int lmax, double* s_io, void* stream)
{
    GS_REQUIRE(badj && dl && bl && xi && s_io && lmax >= 0 && alpha > -1.0 && alpha < 1.0, "bad arguments");
    aux_s_kernel<<<nblk((int64_t)(lmax + 1) * (lmax + 1)), SM_NT, 0, STREAM(stream)>>>(badj, dl, bl, xi, mu_over_w, alpha, lmax, s_io);
    GS_CHECK_LAUNCH();
    return GS_OK;
}

extern "C" int gs_pncp_factor(const double* dl, int lmax, int l_cut, int mode, double* out, void* stream)
{
    GS_REQUIRE(dl && out && lmax >= 0 && l_cut >= 0 && (mode == 0 || mode == 1), "bad arguments");
    pncp_factor_kernel<<<(lmax + 128) / 128, 128, 0, STREAM(stream)>>>(dl, lmax, l_cut, mode, out);
    GS_CHECK_LAUNCH();
    return GS_OK;
}

// ------------------------------------------------------------------ MALA pieces (CenteredGibbs.py:494-603)
// sigma = 1 / (w b_l^2 + 1/C_l) per coefficient (the diagonal preconditioner of the Langevin proposal)
__global__ void mala_sigma_kernel(const double* __restrict__ dl, const double* __restrict__ bl, double w, int L, double* __restrict__ out)
{
    const int64_t n = (int64_t)(L + 1) * (L + 1);
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int l = l_of_real(i, L);
        double c = dl[l];
        if (l) c = c * 2.0 * 3.14159265358979323846 / ((double)l * (double)(l + 1));
        const double ic = c != 0.0 ? 1.0 / c : 0.0;
        out[i] = 1.0 / (w * bl[l] * bl[l] + ic);
    }
}

// grad = bdata - C^-1 s - y   (y = B A^T N^-1 A B s);  invc = 1/C expanded
__global__ void mala_grad_kernel(const double* __restrict__ bdata, const double* __restrict__ invc, const double* __restrict__ s,
                                 const double* __restrict__ y, double* __restrict__ g, int64_t n)
{
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        g[i] = bdata[i] - invc[i] * s[i] - y[i];
}

// s_new = s + tau sigma g + sqrt(2 tau sigma) xi   (CenteredGibbs.py:523-527)
__global__ void mala_propose_kernel(const double* __restrict__ s, const double* __restrict__ g, const double* __restrict__ sigma,
                                    const double* __restrict__ xi, double tau, double* __restrict__ out, int64_t n)
{
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        out[i] = s[i] + tau * sigma[i] * g[i] + sqrt(2.0 * tau * sigma[i]) * xi[i];
}

// partial sums of (to - from - tau sigma g)^2 / (2 tau sigma)   (compute_log_proposal, CenteredGibbs.py:530-532)
__global__ void __launch_bounds__(SM_NT)
mala_logq_partial_kernel(const double* __restrict__ to, const double* __restrict__ from, const double* __restrict__ g,
                         const double* __restrict__ sigma, double tau, int64_t n, double* __restrict__ partials)
{
    double v[1] = {0.0};
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const double r = to[i] - from[i] - tau * sigma[i] * g[i];
        v[0] += r * r / (2.0 * tau * sigma[i]);
    }
    block_sum<1>(v, partials + blockIdx.x);
}

// partial sums of a * b * c (c nullable)
__global__ void __launch_bounds__(SM_NT)
dot3_partial_kernel(const double* __restrict__ a, const double* __restrict__ b, const double* __restrict__ c, int64_t n,
                    double* __restrict__ partials)
{
    double v[1] = {0.0};
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        v[0] = fma(a[i] * b[i], c ? c[i] : 1.0, v[0]);
    block_sum<1>(v, partials + blockIdx.x);
}

extern "C" int gs_mala_sigma(const double* dl, const double* bl, double npix_over_noise_4pi, int lmax, double* out, void* stream)
{
    GS_REQUIRE(dl && bl && out && lmax >= 0, "bad arguments");
    mala_sigma_kernel<<<nblk((int64_t)(lmax + 1) * (lmax + 1)), SM_NT, 0, STREAM(stream)>>>(dl, bl, npix_over_noise_4pi, lmax, out);
    GS_CHECK_LAUNCH();
    return GS_OK;
}

extern "C" int gs_mala_grad(const double* bdata, const double* invc, const double* s, const double* y, double* g, int64_t n,
                            void* stream)
{
    GS_REQUIRE(bdata && invc && s && y && g && n > 0, "bad arguments");
    mala_grad_kernel<<<nblk(n), SM_NT, 0, STREAM(stream)>>>(bdata, invc, s, y, g, n);
    GS_CHECK_LAUNCH();
    return GS_OK;
}

extern "C" int gs_mala_propose(const double* s, const double* g, const double* sigma, const double* xi, double tau, double* out,
                               int64_t n, void* stream)
{
    GS_REQUIRE(s && g && sigma && xi && out && n > 0 && tau > 0.0, "bad arguments");
    mala_propose_kernel<<<nblk(n), SM_NT, 0, STREAM(stream)>>>(s, g, sigma, xi, tau, out, n);
    GS_CHECK_LAUNCH();
    return GS_OK;
}

extern "C" int gs_mala_logq(const double* to, const double* from, const double* g_from, const double* sigma, double tau, int64_t n,
                            double* scratch, double* out, void* stream)
{
    GS_REQUIRE(to && from && g_from && sigma && scratch && out && n > 0 && tau > 0.0, "bad arguments");
    mala_logq_partial_kernel<<<SM_GRID, SM_NT, 0, STREAM(stream)>>>(to, from, g_from, sigma, tau, n, scratch);
    final_sum_kernel<<<1, SM_NT, 0, STREAM(stream)>>>(scratch, SM_GRID, -0.5, out);
    GS_CHECK_LAUNCH();
    return GS_OK;
}

// ULA_no_mask (CenteredGibbs.py:355-446) for one spectrum, full sky + isotropic noise, everything diagonal in the real layout:
//   sigma = 1/(w b^2 + 1/C), mean = sigma b w d, grad(s) = -(s - mean)/sigma,
//   s_new = s_old + tau sigma grad(s_old) + sqrt(2 tau sigma) xi,
//   log density(s) = -1/2 (s - mean)^2 / sigma,  log q(to | from) = -1/2 (to - from - tau sigma grad(from))^2 / (2 tau sigma);
// partial sums of  [log dens(new) + log q(old | new)] - [log dens(old) + log q(new | old)].
__global__ void __launch_bounds__(SM_NT)
ula_nomask_kernel(const double* __restrict__ dl, const double* __restrict__ bl, const double* __restrict__ d_alm,
                  const double* __restrict__ s_old, const double* __restrict__ xi, double w, double tau, int L,
                  double* __restrict__ s_new, double* __restrict__ partials)
{
    double v[1] = {0.0};
    const int64_t n = (int64_t)(L + 1) * (L + 1);
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int l = l_of_real(i, L);
        double c = dl[l];
        if (l) c = c * 2.0 * 3.14159265358979323846 / ((double)l * (double)(l + 1));
        const double b = bl[l];
        const double ic = c != 0.0 ? 1.0 / c : 0.0;
        const double sigma = 1.0 / (w * b * b + ic);
        const double mean = sigma * (b * (w * d_alm[i]));
        const double so = s_old[i];
        const double g_old = -(1.0 / sigma) * (so - mean);
        const double sn = so + tau * sigma * g_old + sqrt(2.0 * tau * sigma) * xi[i];
        const double g_new = -(1.0 / sigma) * (sn - mean);
        s_new[i] = sn;
        const double den = 2.0 * tau * sigma;
        const double a_new = sn - mean, a_old = so - mean;
        const double q_on = so - sn - tau * sigma * g_new;   // old | new
        const double q_no = sn - so - tau * sigma * g_old;   // new | old
        v[0] += -0.5 * (a_new * a_new / sigma) - 0.5 * (q_on * q_on / den) + 0.5 * (a_old * a_old / sigma) + 0.5 * (q_no * q_no / den);
    }
    block_sum<1>(v, partials + blockIdx.x);
}

extern "C" int gs_ula_nomask(const double* dl, const double* bl, const double* d_alm, const double* s_old, const double* xi,
                             double npix_over_noise_4pi, double tau, int lmax, double* s_new, double* scratch, double* log_ratio_out,
                             void* stream)
{
    GS_REQUIRE(dl && bl && d_alm && s_old && xi && s_new && scratch && log_ratio_out && lmax >= 0 && tau > 0.0, "bad arguments");
    ula_nomask_kernel<<<SM_GRID, SM_NT, 0, STREAM(stream)>>>(dl, bl, d_alm, s_old, xi, npix_over_noise_4pi, tau, lmax, s_new, scratch);
    final_sum_kernel<<<1, SM_NT, 0, STREAM(stream)>>>(scratch, SM_GRID, 1.0, log_ratio_out);
    GS_CHECK_LAUNCH();
    return GS_OK;
}

// remove_monopole_dipole_contributions (variance_expension.pyx:103-111): entries 0, 1, L+1, L+2 of the real layout := 0
__global__ void zero_mono_dipole_kernel(double* a, int L)
{
    if (blockIdx.x == 0 && threadIdx.x < 4) {
        const int idx[4] = {0, 1, L + 1, L + 2};
        a[idx[threadIdx.x]] = 0.0;
    }
}

extern "C" int gs_remove_monopole_dipole(double* alm_real, int lmax, void* stream)
{
    GS_REQUIRE(alm_real && lmax >= 1, "bad arguments");
    zero_mono_dipole_kernel<<<1, 32, 0, STREAM(stream)>>>(alm_real, lmax);
    GS_CHECK_LAUNCH();
    return GS_OK;
}

extern "C" int gs_dot3(const double* a, const double* b, const double* c, int64_t n, double* scratch, double* out, void* stream)
{
    GS_REQUIRE(a && b && scratch && out && n > 0, "bad arguments");
    dot3_partial_kernel<<<SM_GRID, SM_NT, 0, STREAM(stream)>>>(a, b, c, n, scratch);
    final_sum_kernel<<<1, SM_NT, 0, STREAM(stream)>>>(scratch, SM_GRID, 1.0, out);
    GS_CHECK_LAUNCH();
    return GS_OK;
}
