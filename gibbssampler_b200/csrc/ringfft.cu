// Ring (azimuthal) stage of the spherical-harmonic transforms: per HEALPix ring, the sum over m
// of F_m(theta) exp(i m phi) on the ring's n equidistant pixels (synthesis) and its transpose
// (analysis).  Replaces the per-ring FFTs of libsharp behind hp.alm2map / hp.map2alm.
//
// One CTA per job; a job is ONE complex DFT of length n that carries TWO real ring sequences
// (spin 2: Q and U of a ring; spin 0: a north ring and its southern mirror), so no real-FFT
// post-processing pass is needed.  m > n/2 is alias-folded in shared memory, the phase
// exp(i m phi_0) of the ring's first pixel is applied on load.  The DFT itself runs in shared
// memory in FP64: power-of-two rings (the 2 nside + 1 equatorial-belt rings when nside is a power
// of two) use an in-place radix-4 decimation-in-time transform on bit-reversed input; every other
// length (polar-cap rings have 4 i pixels, i < nside) uses Bluestein's chirp-z algorithm on top of
// the same kernel: DIF forward -> pointwise product with a precomputed table stored in DIF
// (bit-reversed) order -> DIT inverse, so no permutation pass is ever executed.
#include <math.h>
#include <stdlib.h>

#include <algorithm>
#include <map>

#include "gs_internal.h"

#define RF_NT 256   // threads per CTA of the ring kernels

__device__ __forceinline__ double2 cmul(double2 a, double2 b) { return make_double2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x); }
__device__ __forceinline__ double2 cmulc(double2 a, double2 b) { return make_double2(a.x * b.x + a.y * b.y, a.y * b.x - a.x * b.y); }  // a conj(b)
__device__ __forceinline__ double2 cadd(double2 a, double2 b) { return make_double2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ double2 csub(double2 a, double2 b) { return make_double2(a.x - b.x, a.y - b.y); }

// ---- shared-memory FFT core -------------------------------------------------------------------
// Layout: element i of the transform lives at buf[PADI(i)], PADI(i) = i + (i >> 4) + (i >> 8): one 16-byte pad per
// 16 elements makes the stride-16 accesses of the final radix-16 pass bank-conflict free and leaves the
// unit-stride passes (consecutive lanes -> consecutive elements) conflict free as well; the pad per 256 elements (r02)
// does the same for the BIT-REVERSED accesses of the power-of-two rings (alias fold stores and spectrum unpack loads of
// consecutive k touch elements n/8 apart: 8-way conflicts on every belt ring with the first pad alone).
// Passes: a radix-16 butterfly (= two radix-4 levels) is done entirely in registers, so a 4096-point
// transform makes 3 trips through shared memory (6 with radix-4); leftover stages (log2 M mod 4) are a
// radix-2 and/or radix-4 pass at the top (DIF) / bottom (DIT).
// Twiddles: quarter table twq[k] = exp(-2 pi i k / twn), k <= twn/4, in shared memory;
// W^(k + twn/4) = -i W^k covers the second quadrant (indices stay below twn/2).
#define PADI(i) ((i) + ((i) >> 4) + ((i) >> 8))
#define PADLEN(M) ((M) + ((M) >> 4) + ((M) >> 8) + 2)   // shared-memory slots of a padded M-point buffer

__device__ __forceinline__ double2 tw_get(const double2* twq, int idx, int quarter)
{
    if (idx < quarter) return twq[idx];
    const double2 w = twq[idx - quarter];
    return make_double2(w.y, -w.x);  // -i w
}

// radix-4 DIF butterfly in registers: twiddles w1 = W^x, w2 = W^2x (forward kernel exp(-2 pi i ..))
__device__ __forceinline__ void bf4_dif(double2& a0, double2& a1, double2& a2, double2& a3, double2 w1, double2 w2)
{
    const double2 b0 = cadd(a0, a2), b2 = cmul(csub(a0, a2), w1), b1 = cadd(a1, a3);
    const double2 d13 = csub(a1, a3);
    const double2 b3 = cmul(make_double2(d13.y, -d13.x), w1);  // (a1 - a3) (-i) W^x
    a0 = cadd(b0, b1); a1 = cmul(csub(b0, b1), w2); a2 = cadd(b2, b3); a3 = cmul(csub(b2, b3), w2);
}
// its transpose-conjugate (inverse DIT butterfly, kernel exp(+2 pi i ..))
__device__ __forceinline__ void bf4_dit(double2& c0, double2& c1, double2& c2, double2& c3, double2 w1, double2 w2)
{
    const double2 t1 = cmulc(c1, w2), t3 = cmulc(c3, w2);
    const double2 b0 = cadd(c0, t1), b1 = csub(c0, t1), b2 = cadd(c2, t3), b3 = csub(c2, t3);
    const double2 t2 = cmulc(b2, w1), v3 = cmulc(b3, w1);
    const double2 u3 = make_double2(-v3.y, v3.x);  // (+i) conj(W)^x b3
    c0 = cadd(b0, t2); c2 = csub(b0, t2); c1 = cadd(b1, u3); c3 = csub(b1, u3);
}

// exp(-2 pi i a / 16) and exp(-2 pi i a / 8), a = 0..3
__device__ __forceinline__ double2 w16c(int a)
{
    const double c1 = 0.92387953251128675613, s1 = 0.38268343236508977173, h = 0.70710678118654752440;
    return a == 0 ? make_double2(1.0, 0.0) : a == 1 ? make_double2(c1, -s1) : a == 2 ? make_double2(h, -h) : make_double2(s1, -c1);
}
__device__ __forceinline__ double2 w8c(int a)
{
    const double h = 0.70710678118654752440;
    return a == 0 ? make_double2(1.0, 0.0) : a == 1 ? make_double2(h, -h) : a == 2 ? make_double2(0.0, -1.0) : make_double2(-h, -h);
}

struct NoPre { __device__ __forceinline__ double2 operator()(int, double2 v) const { return v; } };   // identity load hook of the passes

// radix-16 pass over sub-transforms of size N (N >= 16).  INV = false: DIF (forward), true: DIT (inverse).
// POST (DIF only): outputs are multiplied by post[position].
template <bool INV, bool POST, class PRE = NoPre>
__device__ __forceinline__ void pass16(double2* buf, int M, int N, const double2* twq, int twn, const double2* __restrict__ post,
                                       int tid, int nt, PRE pre = PRE())
{
    const int s = N >> 4, ls = 31 - __clz(s), ts = twn / N, quarter = twn >> 2, ng = M >> 4;
    for (int t = tid; t < ng; t += nt) {
        const int g = t >> ls, j = t & (s - 1), i0 = g * N + j;
        double2 x[16];
#pragma unroll
        for (int k = 0; k < 16; ++k) x[k] = pre(i0 + k * s, buf[PADI(i0 + k * s)]);
        double2 wj = make_double2(1.0, 0.0), w2j = wj, w4j = wj, w8j = wj;
        if (s > 1) {
            wj = twq[j * ts];
            w2j = tw_get(twq, 2 * j * ts, quarter);
            w4j = tw_get(twq, 4 * j * ts, quarter);
            w8j = tw_get(twq, 8 * j * ts, quarter);
        }
        if (!INV) {
#pragma unroll
            for (int a = 0; a < 4; ++a) bf4_dif(x[a], x[a + 4], x[a + 8], x[a + 12], cmul(wj, w16c(a)), cmul(w2j, w8c(a)));
#pragma unroll
            for (int c = 0; c < 4; ++c) bf4_dif(x[4 * c], x[4 * c + 1], x[4 * c + 2], x[4 * c + 3], w4j, w8j);
        } else {
#pragma unroll
            for (int c = 0; c < 4; ++c) bf4_dit(x[4 * c], x[4 * c + 1], x[4 * c + 2], x[4 * c + 3], w4j, w8j);
#pragma unroll
            for (int a = 0; a < 4; ++a) bf4_dit(x[a], x[a + 4], x[a + 8], x[a + 12], cmul(wj, w16c(a)), cmul(w2j, w8c(a)));
        }
#pragma unroll
        for (int k = 0; k < 16; ++k) {
            double2 v = x[k];
            if (POST) v = cmul(v, __ldg(&post[i0 + k * s]));
            buf[PADI(i0 + k * s)] = v;
        }
    }
    __syncthreads();
}

// radix-4 pass over sub-transforms of size N (N >= 4)
template <bool INV, class PRE = NoPre>
__device__ __forceinline__ void pass4(double2* buf, int M, int N, const double2* twq, int twn, int tid, int nt, PRE pre = PRE())
{
    const int q = N >> 2, lq = 31 - __clz(q), ts = twn / N, quarter = twn >> 2, nq = M >> 2;
    for (int t = tid; t < nq; t += nt) {
        const int g = t >> lq, j = t & (q - 1), i0 = g * N + j;
        double2 a0 = pre(i0, buf[PADI(i0)]), a1 = pre(i0 + q, buf[PADI(i0 + q)]), a2 = pre(i0 + 2 * q, buf[PADI(i0 + 2 * q)]),
                a3 = pre(i0 + 3 * q, buf[PADI(i0 + 3 * q)]);
        const double2 w1 = twq[j * ts], w2 = tw_get(twq, 2 * j * ts, quarter);
        if (!INV) bf4_dif(a0, a1, a2, a3, w1, w2); else bf4_dit(a0, a1, a2, a3, w1, w2);
        buf[PADI(i0)] = a0; buf[PADI(i0 + q)] = a1; buf[PADI(i0 + 2 * q)] = a2; buf[PADI(i0 + 3 * q)] = a3;
    }
    __syncthreads();
}

// radix-8 pass over sub-transforms of size N (N >= 8) = one radix-2 level + one radix-4 level in registers.  Transform lengths
// 2^(4k+3) (2048: the belt rings of nside 512 and the Bluestein length of the cap rings with 516..1024 pixels) used to take a
// radix-2 AND a radix-4 trip through shared memory at the top (DIF) / bottom (DIT) of the transform; this is one trip.
// PRE (DIF only): the loaded element idx is replaced by pre(idx, value) (fused pointwise products, see ring_apply_kernel).
template <bool INV, class PRE = NoPre>
__device__ __forceinline__ void pass8(double2* buf, int M, int N, const double2* twq, int twn, int tid, int nt, PRE pre = PRE())
{
    const int s = N >> 3, ls = 31 - __clz(s), ts = twn / N, quarter = twn >> 2, ng = M >> 3;
    for (int t = tid; t < ng; t += nt) {
        const int g = t >> ls, j = t & (s - 1), i0 = g * N + j;
        double2 x[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) x[k] = pre(i0 + k * s, buf[PADI(i0 + k * s)]);
        double2 wj = make_double2(1.0, 0.0), w2j = wj, w4j = wj;
        if (s > 1) {
            wj = twq[j * ts];
            w2j = tw_get(twq, 2 * j * ts, quarter);
            w4j = tw_get(twq, 4 * j * ts, quarter);
        }
        if (!INV) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const double2 u = cadd(x[k], x[k + 4]), v = cmul(csub(x[k], x[k + 4]), cmul(wj, w8c(k)));
                x[k] = u; x[k + 4] = v;
            }
            bf4_dif(x[0], x[1], x[2], x[3], w2j, w4j);
            bf4_dif(x[4], x[5], x[6], x[7], w2j, w4j);
        } else {
            bf4_dit(x[0], x[1], x[2], x[3], w2j, w4j);
            bf4_dit(x[4], x[5], x[6], x[7], w2j, w4j);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const double2 tb = cmulc(x[k + 4], cmul(wj, w8c(k)));
                const double2 a = x[k];
                x[k] = cadd(a, tb); x[k + 4] = csub(a, tb);
            }
        }
#pragma unroll
        for (int k = 0; k < 8; ++k) buf[PADI(i0 + k * s)] = x[k];
    }
    __syncthreads();
}

// radix-2 pass over sub-transforms of size N (N >= 2)
template <bool INV, class PRE = NoPre>
__device__ __forceinline__ void pass2(double2* buf, int M, int N, const double2* twq, int twn, int tid, int nt, PRE pre = PRE())
{
    const int h = N >> 1, lh = 31 - __clz(h), ts = twn / N;
    for (int t = tid; t < (M >> 1); t += nt) {
        const int g = t >> lh, j = t & (h - 1), i0 = g * N + j;
        const double2 a = pre(i0, buf[PADI(i0)]), b = pre(i0 + h, buf[PADI(i0 + h)]);
        const double2 w = tw_get(twq, j * ts, twn >> 2);
        if (!INV) { buf[PADI(i0)] = cadd(a, b); buf[PADI(i0 + h)] = cmul(csub(a, b), w); }
        else { const double2 tb = cmulc(b, w); buf[PADI(i0)] = cadd(a, tb); buf[PADI(i0 + h)] = csub(a, tb); }
    }
    __syncthreads();
}

// In-place forward DIF FFT (kernel exp(-2 pi i jk/M)), natural order in, bit-reversed order out;
// POST: the bit-reversed-order output is multiplied by post[] inside the last pass (needs M >= 16).
// (tid, nt): index and number of the threads working on THIS transform (a CTA may run several transforms of
// equal length side by side, see RingGroup); every barrier is CTA-wide.
// PRE: pre(idx, value) replaces every element as the FIRST pass loads it (M >= 2): pointwise products in front of a transform
// (pixel weights, Bluestein chirps, zero padding) cost no trip through shared memory of their own.
template <bool POST, class PRE = NoPre>
__device__ void fft_dif(double2* buf, int M, const double2* twq, int twn, const double2* __restrict__ post, int tid = threadIdx.x,
                        int nt = RF_NT, PRE pre = PRE())
{
    const int lg = 31 - __clz(M), r = lg & 3;
    int N = M;
    bool first = true;
    if (r == 3) { pass8<false, PRE>(buf, M, N, twq, twn, tid, nt, pre); N >>= 3; first = false; }
    else {
        if (r & 1) { pass2<false, PRE>(buf, M, N, twq, twn, tid, nt, pre); N >>= 1; first = false; }
        if (r & 2) {
            if (first) pass4<false, PRE>(buf, M, N, twq, twn, tid, nt, pre); else pass4<false>(buf, M, N, twq, twn, tid, nt);
            N >>= 2; first = false;
        }
    }
    while (N >= 16) {
        if (first) {
            if (POST && N == 16) pass16<false, true, PRE>(buf, M, N, twq, twn, post, tid, nt, pre);
            else pass16<false, false, PRE>(buf, M, N, twq, twn, post, tid, nt, pre);
        } else if (POST && N == 16) pass16<false, true>(buf, M, N, twq, twn, post, tid, nt);
        else pass16<false, false>(buf, M, N, twq, twn, post, tid, nt);
        first = false;
        N >>= 4;
    }
}

// In-place inverse DIT FFT (kernel exp(+2 pi i jk/M), unnormalised), bit-reversed in, natural out.
__device__ void fft_dit_inv(double2* buf, int M, const double2* twq, int twn, int tid = threadIdx.x, int nt = RF_NT)
{
    const int lg = 31 - __clz(M), r = lg & 3;
    const int Ntop = M >> r;  // largest radix-16 sub-transform size
    for (int N = 16; N <= Ntop; N <<= 4) pass16<true, false>(buf, M, N, twq, twn, nullptr, tid, nt);
    int N = Ntop;
    if (r == 3) { N <<= 3; pass8<true>(buf, M, N, twq, twn, tid, nt); return; }
    if (r & 2) { N <<= 2; pass4<true>(buf, M, N, twq, twn, tid, nt); }
    if (r & 1) { N <<= 1; pass2<true>(buf, M, N, twq, twn, tid, nt); }
}

__device__ __forceinline__ void load_twq(const PlanDev& P, double2* twq)
{
    const int nq = (P.tw_n >> 2) + 1;
    for (int k = threadIdx.x; k < nq; k += RF_NT) twq[k] = __ldg(&P.tw[k]);
}

__device__ __forceinline__ double2 chirp_val(int t, int n)
{  // exp(i pi t^2 / n)
    const int r = (int)(((long long)t * t) % (2 * n));
    double s, c;
    sincospi((double)r / (double)n, &s, &c);
    return make_double2(c, s);
}

// z_j = sum_{k<n} Z_k exp(+2 pi i jk / n), in place in buf[0..n).
// Power-of-two n (bsi < 0): the caller stored Z_k at the bit-reversed position of k.
// Otherwise (Bluestein): the caller stored Z_k * chirp[k] at k < n and zeros at n <= k < M; the result
// still has to be multiplied by chirp[j] by the caller (fused into its output pass).
// All threads of the CTA must call; begins and ends with a barrier.
__device__ void ring_idft(const PlanDev& P, double2* buf, const double2* twq, int n, int bsi, int tid = threadIdx.x, int nt = RF_NT)
{
    __syncthreads();
    if (bsi < 0) { fft_dit_inv(buf, n, twq, P.tw_n, tid, nt); return; }
    const BluesteinDesc d = P.bs[bsi];
    fft_dif<true>(buf, d.M, twq, P.tw_n, P.bs_tab + d.bhat_off, tid, nt);
    fft_dit_inv(buf, d.M, twq, P.tw_n, tid, nt);
}

__global__ void __launch_bounds__(RF_NT) bluestein_setup_kernel(PlanDev P, double2* tab, int nbs)
{
    extern __shared__ double2 smem_all[];
    double2* twq = smem_all;
    double2* buf = smem_all + (P.tw_n >> 2) + 1;
    load_twq(P, twq);
    const BluesteinDesc d = P.bs[blockIdx.x];
    double2* chirp = tab + d.chirp_off;
    double2* bhat = tab + d.bhat_off;
    for (int k = threadIdx.x; k < d.M; k += blockDim.x) buf[PADI(k)] = make_double2(0.0, 0.0);
    __syncthreads();
    for (int t = threadIdx.x; t < d.n; t += blockDim.x) {
        const double2 c = chirp_val(t, d.n);
        chirp[t] = c;
        const double2 cc = make_double2(c.x, -c.y);
        buf[PADI(t)] = cc;
        if (t > 0) buf[PADI(d.M - t)] = cc;
    }
    __syncthreads();
    fft_dif<false>(buf, d.M, twq, P.tw_n, nullptr);
    const double inv = 1.0 / (double)d.M;
    for (int k = threadIdx.x; k < d.M; k += blockDim.x) { const double2 v = buf[PADI(k)]; bhat[k] = make_double2(v.x * inv, v.y * inv); }
    (void)nbs;
}

__device__ __forceinline__ double2 ring_phase(const PlanDev& P, int ring, int m)
{  // exp(i m phi0), phi0 = pi q / den
    const int q = P.ring_phq[ring], den = P.ring_phden[ring];
    const unsigned r = ((unsigned)m * (unsigned)q) % (2u * (unsigned)den);  // m q < 2^31 for every supported size
    double s, c;
    sincospi((double)r / (double)den, &s, &c);
    return make_double2(c, s);
}

// Position of F_m(ring) in the ring-spectra buffer as seen from the ring-sharded side (see ShardDev).
template <bool SH>
__device__ __forceinline__ int64_t fm_ring_index(const PlanDev& P, int comp, int ring, int m)
{
    if (SH) return P.sh.m_base[m] + ((int64_t)comp * P.sh.RL + P.sh.ring_loc[ring]) * P.sh.MLb;   // see ShardDev
    return ((int64_t)comp * P.nring + ring) * (P.lmax + 1) + m;
}
template <bool SH>
__device__ __forceinline__ int64_t ring_first_pixel(const PlanDev& P, int ring)
{
    return SH ? P.sh.ring_start_loc[ring] : P.ring_start[ring];
}

// Highest m that carries signal on a ring: the Legendre kernels neither write (synthesis) nor read (analysis) the spectrum
// of a ring above the m_lim of its ring pair, so the ring stage must treat those entries as zero / may skip them.
__device__ __forceinline__ int ring_mtop(const PlanDev& P, int ring, int spin2)
{
    const int p = ring < P.npair ? ring : P.nring - 1 - ring;
    return spin2 ? P.mlim2[p] : P.mlim0[p];
}

// Rings without pixel weight (gs_active_rings_build; flags are per ring PAIR): nobody reads what the ring stage would
// produce for them.  ract == nullptr: every ring is processed.
__device__ __forceinline__ bool group_idle(const unsigned char* __restrict__ ract, const RingJob* __restrict__ jobs, const int2* __restrict__ groups)
{
    if (!ract) return false;
    const int2 g = groups[blockIdx.x];
    bool any = false;
    for (int s = 0; s < g.y; ++s) {
        const RingJob jb = jobs[g.x + s];
        any = any || ract[jb.ringA] || (jb.ringB >= 0 && ract[jb.ringB]);
    }
    return !any;
}
// Every ring of the CTA's group has one pixel weight for all its pixels (wconst from gs_active_rings_build, NaN = weights differ)
__device__ __forceinline__ bool group_const(const double* __restrict__ wconst, const RingJob* __restrict__ jobs, const int2* __restrict__ groups)
{
    if (!wconst) return false;
    const int2 g = groups[blockIdx.x];
    bool all = true;
    for (int s = 0; s < g.y; ++s) {
        const RingJob jb = jobs[g.x + s];
        const double a = wconst[jb.ringA], b = jb.ringB >= 0 ? wconst[jb.ringB] : 0.0;
        all = all && a == a && b == b;
    }
    return all;
}
// groups_out = groups, stably partitioned into (needs transforms | constant weights only | idle): one block
__global__ void __launch_bounds__(1024) ring_order_kernel(const RingJob* __restrict__ jobs, const int2* __restrict__ groups, int ngroups,
                                                          const unsigned char* __restrict__ ract, const double* __restrict__ wconst,
                                                          int2* __restrict__ groups_out)
{
    __shared__ int wcount[32][3];
    __shared__ int base[3], total[3];
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    auto cls_of = [&](int gi) {
        if (gi >= ngroups) return 3;
        const int2 g = groups[gi];
        bool any = false, allc = true;
        for (int s = 0; s < g.y; ++s) {
            const RingJob jb = jobs[g.x + s];
            any = any || ract[jb.ringA] || (jb.ringB >= 0 && ract[jb.ringB]);
            const double a = wconst[jb.ringA], b = jb.ringB >= 0 ? wconst[jb.ringB] : 0.0;
            allc = allc && a == a && b == b;
        }
        return !any ? 2 : allc ? 1 : 0;
    };
    for (int pass = 0; pass < 2; ++pass) {
        if (tid < 3) { if (pass == 0) total[tid] = 0; else base[tid] = tid == 0 ? 0 : tid == 1 ? total[0] : total[0] + total[1]; }
        __syncthreads();
        for (int g0 = 0; g0 < ngroups; g0 += 1024) {
            const int gi = g0 + tid, c = cls_of(gi);
            unsigned bal[3];
#pragma unroll
            for (int k = 0; k < 3; ++k) { bal[k] = __ballot_sync(0xffffffffu, c == k); if (lane == 0) wcount[w][k] = __popc(bal[k]); }
            __syncthreads();
            if (pass == 1 && c < 3) {
                int off = base[c];
                for (int i = 0; i < w; ++i) off += wcount[i][c];
                groups_out[off + __popc(bal[c] & ((1u << lane) - 1u))] = groups[gi];
            }
            __syncthreads();
            if (tid < 3) {
                int t = 0;
                for (int i = 0; i < 32; ++i) t += wcount[i][tid];
                if (pass == 0) total[tid] += t; else base[tid] += t;
            }
            __syncthreads();
        }
    }
}

__device__ __forceinline__ bool split_idle(const unsigned char* __restrict__ ract, const SplitJob& jb)
{
    return ract && !(ract[jb.ringA] || (jb.ringB >= 0 && ract[jb.ringB]));
}

// A CTA of the direct ring kernels works on a GROUP of 1, 2 or 4 jobs whose transforms have the same length M and
// the same kind (power of two / Bluestein), RF_NT / nsub threads each, side by side in shared memory: the passes of a
// short transform cannot keep 256 threads busy (M / 16 radix-16 butterflies per pass) and the ring stage is latency
// bound, so running equal-length rings together is what fills the CTA.  Control flow (number of passes and barriers)
// depends on (M, kind) only, so it is uniform over the CTA.
struct RingSub {
    RingJob job;
    int n, bsi, M, tid, nt;
    double2* buf;
    double2* scratch;
    const double2* chirp;
};

__device__ __forceinline__ RingSub ring_sub(const PlanDev& P, const RingJob* __restrict__ jobs, const int2* __restrict__ groups,
                                            double2* bufs)
{
    const int2 g = groups[blockIdx.x];   // (first job, nsub)
    RingSub S;
    S.nt = RF_NT / g.y;
    const int sub = threadIdx.x / S.nt;
    S.tid = threadIdx.x - sub * S.nt;
    S.job = jobs[g.x + sub];
    S.n = P.ring_nphi[S.job.ringA];
    S.bsi = P.ring_bs[S.job.ringA];
    S.M = S.bsi >= 0 ? P.bs[S.bsi].M : S.n;
    S.chirp = S.bsi >= 0 ? P.bs_tab + P.bs[S.bsi].chirp_off : nullptr;
    S.buf = bufs + sub * PADLEN(S.M);
    S.scratch = bufs + g.y * PADLEN(S.M) + sub * S.nt;   // used by rings shorter than nt only (M <= 2 nt)
    return S;
}

// Z[k] = Xa[k] + i Xb[k], X[k] = G[k] + conj G[n-k], G[k] = sum_{m = k mod n} w_m F_m e^{i m phi0} (alias fold), for the two
// real sequences of a job, written to buf ready for ring_idft: bit-reversed (power-of-two n) or chirp-multiplied and
// zero-padded (Bluestein).  F_m is taken as zero for m > mtop.  The spectrum is read straight from global memory, both
// components in one sweep; the phases follow from e^{i k phi0} (recurrence over the thread's k) and q = e^{i n phi0}:
// e^{i (k + j n) phi0} = e^{i k phi0} q^j, e^{i (n - k + j n) phi0} = conj(e^{i k phi0}) q^(j+1).
// Partial alias sums for UK values of k (k0 + u ks, u < UK) over the alias terms j = j0, j0 + js, ... < nterm:
//   z[u] += sum_j w e^{i (k + j n) phi0} (Fa + i Fb)[k + j n] + w conj(e^{i (kk + j n) phi0}) (conj Fa + i conj Fb)[kk + j n],
// kk = n - k (0 for k = 0).  4 UK UJ independent global loads are in flight per step.
template <bool SH, int UK, int UJ>
__device__ __forceinline__ void ring_fold(const PlanDev& P, const RingJob& job, const double2* __restrict__ Fm, const double2* __restrict__ FA,
                                          const double2* __restrict__ FB, int fs, int n, int mtop, int nterm, int k0, int ks, int j0, int js,
                                          double2 pk0, double2 step, double2 q, double2 (&z)[UK])
{   // fs: stride of m in FA / FB (1: [comp][ring][m]; 2: components interleaved, [ring][m][comp])
    // pk0 = e^{i k0 phi0}, step = e^{i ks phi0}, q = e^{i n phi0}: the phases of the first alias term follow by
    // multiplication when j0 = 0 (e^{i (n - k) phi0} = q conj e^{i k phi0}); one sincospi pair per k otherwise.
    const double2 zero = make_double2(0.0, 0.0);
    const bool hasB = job.ringB >= 0;
    const double2 qs = js == 1 ? q : ring_phase(P, job.ringA, js * n), qsc = make_double2(qs.x, -qs.y);
    double2 e1[UK], e2[UK];
#pragma unroll
    for (int u = 0; u < UK; ++u) {
        const int k = k0 + u * ks;
        z[u] = zero;
        if (j0 == 0) {
            e1[u] = u ? cmul(e1[u - 1], step) : pk0;
            e2[u] = k ? cmulc(e1[u], q) : make_double2(1.0, 0.0);     // conj(q conj e1)
        } else {
            e1[u] = e2[u] = zero;
            if (k < n) {
                e1[u] = ring_phase(P, job.ringA, k + j0 * n);
                const double2 t = ring_phase(P, job.ringA, (k ? n - k : 0) + j0 * n);
                e2[u] = make_double2(t.x, -t.y);
            }
        }
    }
    for (int jb = j0; jb < nterm; jb += UJ * js) {
        double2 fa1[UK][UJ], fa2[UK][UJ], fb1[UK][UJ], fb2[UK][UJ];
#pragma unroll
        for (int u = 0; u < UK; ++u) {
            const int k = k0 + u * ks;
#pragma unroll
            for (int v = 0; v < UJ; ++v) {
                const int j = jb + v * js;
                const int m1 = k + j * n, m2 = (k ? n - k : 0) + j * n;
                const bool v1 = k < n && m1 <= mtop, v2 = k < n && m2 <= mtop;
                fa1[u][v] = v1 ? (SH ? Fm[fm_ring_index<true>(P, job.compA, job.ringA, m1)] : FA[m1 * fs]) : zero;
                fa2[u][v] = v2 ? (SH ? Fm[fm_ring_index<true>(P, job.compA, job.ringA, m2)] : FA[m2 * fs]) : zero;
                fb1[u][v] = (hasB && v1) ? (SH ? Fm[fm_ring_index<true>(P, job.compB, job.ringB, m1)] : FB[m1 * fs]) : zero;
                fb2[u][v] = (hasB && v2) ? (SH ? Fm[fm_ring_index<true>(P, job.compB, job.ringB, m2)] : FB[m2 * fs]) : zero;
            }
        }
#pragma unroll
        for (int u = 0; u < UK; ++u) {
            const int k = k0 + u * ks;
#pragma unroll
            for (int v = 0; v < UJ; ++v) {
                const double w = (k + jb + v * js) ? 1.0 : 0.5;   // (2 - delta_m0) / 2: m = 0 only for k = 0, j = 0 (both sums)
                const double2 t1 = make_double2(fa1[u][v].x - fb1[u][v].y, fa1[u][v].y + fb1[u][v].x);    // Fa + i Fb
                const double2 t2 = make_double2(fa2[u][v].x + fb2[u][v].y, fb2[u][v].x - fa2[u][v].y);    // conj Fa + i conj Fb
                z[u] = cadd(z[u], cadd(cmul(t1, make_double2(e1[u].x * w, e1[u].y * w)), cmul(t2, make_double2(e2[u].x * w, e2[u].y * w))));
                e1[u] = cmul(e1[u], qs);
                e2[u] = cmul(e2[u], qsc);
            }
        }
    }
}

// Z[k] = Xa[k] + i Xb[k], X[k] = G[k] + conj G[n-k], G[k] = sum_{m = k mod n} w_m F_m e^{i m phi0} (alias fold), for the two
// real sequences of a job, written to buf ready for ring_idft: bit-reversed (power-of-two n) or chirp-multiplied and
// zero-padded (Bluestein).  F_m is taken as zero for m > mtop.  Both sequences of a job share phi0 (Q and U of one ring; a
// ring and its southern mirror by construction, plan.cu).  The spectrum is read straight from global memory with many
// independent loads in flight (the stage is latency bound): rings at least 4 nt long take 4 values of k per step, shorter
// ones 4 alias terms per step, and rings shorter than the thread count split the alias terms of each k over nt / n threads
// and combine the partial sums in a fixed order through `scratch` (nt entries of shared memory).
// Contains one CTA-wide barrier; all threads of the CTA must call.
template <bool SH>
__device__ __forceinline__ void ring_build_Z(const PlanDev& P, const RingSub& S, const double2* __restrict__ Fm, int mtop, double2* scratch,
                                             bool interleaved = false, bool plain = false)
{   // plain: Z_k is stored at buf[PADI(k)], k < n, as it is (no bit reversal, chirp or padding: no transform follows)
    const RingJob& job = S.job;
    const int L = P.lmax, nm = L + 1, n = S.n, lg = 31 - __clz(n);
    // spectra layout [comp][ring][m], or (block-batched Metropolis sweep) [ring][m][comp] with Q and U of one (ring, m) adjacent
    const int fs = interleaved ? 2 : 1;
    const double2* FA = interleaved ? Fm + (int64_t)job.ringA * nm * 2 + job.compA : Fm + ((int64_t)job.compA * P.nring + job.ringA) * nm;
    const double2* FB = job.ringB < 0 ? nullptr
                        : interleaved ? Fm + (int64_t)job.ringB * nm * 2 + job.compB : Fm + ((int64_t)job.compB * P.nring + job.ringB) * nm;
    const int nterm = (mtop + n) / n;   // alias terms m = k + j n <= mtop, j < nterm
    const double2 zero = make_double2(0.0, 0.0);
    const int Mz = plain ? n : S.M;
    auto put = [&](int k, double2 v) {
        if (k >= Mz) return;
        const int pos = PADI((S.bsi < 0 && !plain) ? (int)(__brev((unsigned)k) >> (32 - lg)) : k);
        if (k >= n) v = zero;
        else if (S.bsi >= 0 && !plain) v = cmul(v, __ldg(&S.chirp[k]));
        S.buf[pos] = v;
    };
    if (!SH && 2 * mtop <= n && n > S.nt) {
        // No alias term (most cap rings, the whole belt): F_m alone gives Z_m = e^{i m phi0} (Fa + i Fb)_m and
        // Z_{n-m} = e^{-i m phi0} (conj Fa + i conj Fb)_m; the walk is over m with 2 DU independent loads in flight, every one of them
        // used (the general fold below walks k and predicates off the half of its loads whose m lies above m_top).
        constexpr int DU = 8;
        double2 pm = ring_phase(P, job.ringA, S.tid);
        const double2 step = ring_phase(P, job.ringA, S.nt);
        for (int m0 = S.tid; m0 <= mtop; m0 += DU * S.nt) {
            double2 a[DU], b[DU];
#pragma unroll
            for (int u = 0; u < DU; ++u) {
                const int m = m0 + u * S.nt;
                const bool ok = m <= mtop;
                a[u] = ok ? FA[m * fs] : zero;
                b[u] = (ok && FB) ? FB[m * fs] : zero;
            }
#pragma unroll
            for (int u = 0; u < DU; ++u) {
                const int m = m0 + u * S.nt;
                if (m <= mtop) {
                    const double2 t1 = make_double2(a[u].x - b[u].y, a[u].y + b[u].x);   // Fa + i Fb
                    const double2 t2 = make_double2(a[u].x + b[u].y, b[u].x - a[u].y);   // conj Fa + i conj Fb
                    if (m == 0) put(0, make_double2(a[u].x, b[u].x));                    // weight 1/2 on both terms
                    else if (2 * m == n) put(m, cadd(cmul(t1, pm), cmulc(t2, pm)));      // the term meets its own mirror
                    else { put(m, cmul(t1, pm)); put(n - m, cmulc(t2, pm)); }
                }
                pm = cmul(pm, step);
            }
        }
        for (int k = mtop + 1 + S.tid; k < n - mtop; k += S.nt) put(k, zero);
        for (int k = n + S.tid; k < Mz; k += S.nt) put(k, zero);   // zero padding (Bluestein)
        __syncthreads();
        return;
    }
    const bool split = n <= S.nt;
    const double2 q = ring_phase(P, job.ringA, n);
    constexpr int FK = 4;   // values of k (long rings) / alias terms (short rings) per step: 4 FK loads in flight per thread
    if (split) {
        const int J = S.nt / n, kq = S.tid % n, jq = S.tid / n;
        double2 z[1] = {zero};
        if (jq < J) ring_fold<SH, 1, FK>(P, job, Fm, FA, FB, fs, n, mtop, nterm, kq, 1, jq, J, ring_phase(P, job.ringA, kq), zero, q, z);
        scratch[S.tid] = z[0];
    } else if (n >= FK * S.nt) {
        double2 pk = ring_phase(P, job.ringA, S.tid);
        const double2 step = ring_phase(P, job.ringA, S.nt), step4 = ring_phase(P, job.ringA, FK * S.nt);
        for (int k0 = S.tid; k0 < n; k0 += FK * S.nt) {
            double2 z[FK];
            ring_fold<SH, FK, 1>(P, job, Fm, FA, FB, fs, n, mtop, nterm, k0, S.nt, 0, 1, pk, step, q, z);
#pragma unroll
            for (int u = 0; u < FK; ++u) put(k0 + u * S.nt, z[u]);
            pk = cmul(pk, step4);
        }
        for (int k = S.tid + ((n - S.tid + FK * S.nt - 1) / (FK * S.nt)) * FK * S.nt; k < Mz; k += S.nt) put(k, zero);   // zero padding
    } else {
        double2 pk = ring_phase(P, job.ringA, S.tid);
        const double2 step = ring_phase(P, job.ringA, S.nt);
        for (int k0 = S.tid; k0 < n; k0 += S.nt) {
            double2 z[1];
            ring_fold<SH, 1, FK>(P, job, Fm, FA, FB, fs, n, mtop, nterm, k0, S.nt, 0, 1, pk, step, q, z);
            put(k0, z[0]);
            pk = cmul(pk, step);
        }
        for (int k = S.tid + ((n - S.tid + S.nt - 1) / S.nt) * S.nt; k < Mz; k += S.nt) put(k, zero);   // zero padding
    }
    __syncthreads();
    if (split) {
        const int J = S.nt / n;
        for (int k = S.tid; k < Mz; k += S.nt) {
            double2 v = zero;
            if (k < n) for (int i = 0; i < J; ++i) v = cadd(v, scratch[i * n + k]);
            put(k, v);
        }
    }
}

// F_m of the two real sequences of a job from the length-n DFT held in buf, m = 0..lmax:
//   Xa[k] = (Z[k] + conj Z[n-k]) / 2, Xb[k] = (Z[k] - conj Z[n-k]) / (2i), F_m = X[m mod n] e^{-i m phi0}.
// mode UNPACK_CONJ: buf[PADI(k)] = conj Z[k] (transform done as conj(idft(conj z))); UNPACK_BREV: buf holds Z[k] at the
// bit-reversed position of k (forward DIF transform of a power-of-two ring); UNPACK_PLAIN: buf[PADI(k)] = Z[k].
// chirp (UNPACK_CONJ only, nullable): buf still lacks the final Bluestein product, buf[k] chirp[k] is taken on the fly.
// sa, sb: factors of the two sequences (the transform-free path of ring_apply_kernel puts n w there).
enum { UNPACK_CONJ = 0, UNPACK_BREV = 1, UNPACK_PLAIN = 2 };
template <bool SH>
__device__ __forceinline__ void ring_unpack_F(const PlanDev& P, const RingSub& S, int mode, double2* __restrict__ Fm, int mtop,
                                              const double2* __restrict__ chirp = nullptr, double sa = 0.5, double sb = 0.5)
{
    const RingJob& job = S.job;
    const int L = P.lmax, nm = L + 1, n = S.n, lg = 31 - __clz(n);
    const double2* buf = S.buf;
    double2* FA = Fm + ((int64_t)job.compA * P.nring + job.ringA) * nm;
    double2* FB = job.ringB >= 0 ? Fm + ((int64_t)job.compB * P.nring + job.ringB) * nm : nullptr;
    double2 pa = ring_phase(P, job.ringA, S.tid);   // both sequences of a job share phi0 (plan.cu gives a ring and its mirror the same phase)
    const double2 stepa = ring_phase(P, job.ringA, S.nt);
    for (int m = S.tid; m <= mtop; m += S.nt) {
        const int k = m % n, kk = (n - k) % n;
        double2 z1, z2c;
        if (mode == UNPACK_BREV) {
            const double2 c1 = buf[PADI((int)(__brev((unsigned)k) >> (32 - lg)))], c2 = buf[PADI((int)(__brev((unsigned)kk) >> (32 - lg)))];
            z1 = c1; z2c = make_double2(c2.x, -c2.y);
        } else if (mode == UNPACK_PLAIN) {
            const double2 c1 = buf[PADI(k)], c2 = buf[PADI(kk)];
            z1 = c1; z2c = make_double2(c2.x, -c2.y);
        } else {
            double2 c1 = buf[PADI(k)], c2 = buf[PADI(kk)];
            if (chirp) { c1 = cmul(c1, __ldg(&chirp[k])); c2 = cmul(c2, __ldg(&chirp[kk])); }
            z1 = make_double2(c1.x, -c1.y); z2c = c2;
        }
        const double2 xa = make_double2(sa * (z1.x + z2c.x), sa * (z1.y + z2c.y));
        const double2 d = csub(z1, z2c);
        const double2 xb = make_double2(sb * d.y, -sb * d.x);
        if (SH) {
            Fm[fm_ring_index<true>(P, job.compA, job.ringA, m)] = cmulc(xa, pa);
            if (FB) Fm[fm_ring_index<true>(P, job.compB, job.ringB, m)] = cmulc(xb, pa);
        } else {
            FA[m] = cmulc(xa, pa);
            if (FB) FB[m] = cmulc(xb, pa);
        }
        pa = cmul(pa, stepa);
    }
}

template <bool SH>
__global__ void __launch_bounds__(RF_NT, 2)
ring_synth_kernel(PlanDev P, const RingJob* __restrict__ jobs, const int2* __restrict__ groups, const double2* __restrict__ Fm,
                  double* __restrict__ mapQ, double* __restrict__ mapU, const int* __restrict__ skip, int64_t f_stride,
                  int64_t map_stride, const int* __restrict__ mmax, int spin2, const unsigned char* __restrict__ ract,
                  const double* __restrict__ wconst)
{
    if (skip && *skip) return;
    if (group_idle(ract, jobs, groups)) return;
    extern __shared__ double2 smem[];
    // batched use (blockIdx.y = transform index): spectra at Fm + y f_stride hold m <= mmax[y] only, maps at + y map_stride
    Fm += blockIdx.y * f_stride;
    mapQ += blockIdx.y * map_stride;
    mapU += blockIdx.y * map_stride;
    const int mcap = mmax ? min(mmax[blockIdx.y], P.lmax) : P.lmax;
    double2* twq = smem;
    if (group_const(wconst, jobs, groups)) {
        // Spectral storage (Metropolis sweep, spin 2: Q and U of ONE ring with ONE weight w): the sweep only ever forms
        // w sum_j |z_j - z'_j|^2 over the ring, z = Q + i U, and the unitary DFT keeps that sum, so slot k of the ring receives
        // sqrt(n) Z_k (the unitary DFT of the pixels this launch would have produced) and no transform runs
        const RingSub S = ring_sub(P, jobs, groups, twq + (P.tw_n >> 2) + 1);
        ring_build_Z<SH>(P, S, Fm, min(mcap, ring_mtop(P, S.job.ringA, spin2)), S.scratch, mmax != nullptr, true);
        __syncthreads();
        const double sn = sqrt((double)S.n);
        double* oa = mapQ + ring_first_pixel<SH>(P, S.job.ringA);
        double* ob = mapU + ring_first_pixel<SH>(P, S.job.ringA);
        for (int k = S.tid; k < S.n; k += S.nt) {
            const double2 z = S.buf[PADI(k)];
            oa[k] = sn * z.x;
            ob[k] = sn * z.y;
        }
        return;
    }
    load_twq(P, twq);
    const RingSub S = ring_sub(P, jobs, groups, twq + (P.tw_n >> 2) + 1);
    ring_build_Z<SH>(P, S, Fm, min(mcap, ring_mtop(P, S.job.ringA, spin2)), S.scratch, mmax != nullptr);
    ring_idft(P, S.buf, twq, S.n, S.bsi, S.tid, S.nt);
    double* oa = (S.job.compA ? mapU : mapQ) + ring_first_pixel<SH>(P, S.job.ringA);
    double* ob = S.job.ringB >= 0 ? (S.job.compB ? mapU : mapQ) + ring_first_pixel<SH>(P, S.job.ringB) : nullptr;
    for (int j = S.tid; j < S.n; j += S.nt) {
        double2 z = S.buf[PADI(j)];
        if (S.bsi >= 0) z = cmul(z, __ldg(&S.chirp[j]));
        oa[j] = z.x;
        if (ob) ob[j] = z.y;
    }
}

template <bool SH>
__global__ void __launch_bounds__(RF_NT, 2)
ring_anal_kernel(PlanDev P, const RingJob* __restrict__ jobs, const int2* __restrict__ groups, const double* __restrict__ mapQ,
                 const double* __restrict__ mapU, const double* __restrict__ pixw, double2* __restrict__ Fm, const int* __restrict__ skip,
                 int spin2, const unsigned char* __restrict__ ract, int64_t f_stride, int64_t map_stride)
{
    if (skip && *skip) return;
    if (group_idle(ract, jobs, groups)) return;
    extern __shared__ double2 smem[];
    // chain batch (blockIdx.y = chain): maps at + y map_stride -> spectra at + y f_stride; the pixel weights are shared
    Fm += blockIdx.y * f_stride;
    mapQ += blockIdx.y * map_stride;
    mapU += blockIdx.y * map_stride;
    double2* twq = smem;
    load_twq(P, twq);
    const RingSub S = ring_sub(P, jobs, groups, twq + (P.tw_n >> 2) + 1);
    const RingJob& job = S.job;
    const int n = S.n;
    const int64_t sa = ring_first_pixel<SH>(P, job.ringA), sb = job.ringB >= 0 ? ring_first_pixel<SH>(P, job.ringB) : 0;
    const double* ia = (job.compA ? mapU : mapQ) + sa;
    const double* ib = job.ringB >= 0 ? (job.compB ? mapU : mapQ) + sb : nullptr;
    const int lg = 31 - __clz(n);
    // Z[k] = sum_j z_j exp(-2 pi i jk/n) = conj( idft( conj z ) )
    for (int j = S.tid; j < S.M; j += S.nt) {
        const int pos = PADI(S.bsi < 0 ? (int)(__brev((unsigned)j) >> (32 - lg)) : j);
        if (j >= n) { S.buf[pos] = make_double2(0.0, 0.0); continue; }
        double a = ia[j], b = ib ? ib[j] : 0.0;
        if (pixw) { a *= pixw[sa + j]; if (ib) b *= pixw[sb + j]; }
        double2 z = make_double2(a, -b);
        if (S.bsi >= 0) z = cmul(z, __ldg(&S.chirp[j]));
        S.buf[pos] = z;
    }
    ring_idft(P, S.buf, twq, n, S.bsi, S.tid, S.nt);
    // Bluestein: the last chirp product is taken as the spectrum is unpacked
    ring_unpack_F<SH>(P, S, UNPACK_CONJ, Fm, ring_mtop(P, job.ringA, spin2), S.bsi >= 0 ? S.chirp : nullptr);
}

// Spin-2 maps -> the storage the Metropolis sweep compares in: groups of constant-weight rings get the unitary DFT of
// z_j = Q_j + i U_j, Ztilde_k = n^-1/2 sum_j z_j e^{-2 pi i jk/n} (the counterpart of the spectral branch of ring_synth_kernel, whose
// pixels would be z_j = sum_k Z_k e^{+2 pi i jk/n} = n^-1/2 sum_k Ztilde_k e^{..}); every other ring is copied.
__global__ void __launch_bounds__(RF_NT, 2)
ring_mwg_data_kernel(PlanDev P, const RingJob* __restrict__ jobs, const int2* __restrict__ groups, const double* __restrict__ mapQ,
                     const double* __restrict__ mapU, double* __restrict__ outQ, double* __restrict__ outU, const double* __restrict__ wconst)
{
    extern __shared__ double2 smem[];
    double2* twq = smem;
    const bool spectral = group_const(wconst, jobs, groups);
    if (spectral) load_twq(P, twq);
    const RingSub S = ring_sub(P, jobs, groups, twq + (P.tw_n >> 2) + 1);
    const int n = S.n;
    const int64_t s0 = P.ring_start[S.job.ringA];
    const double* ia = mapQ + s0;
    const double* ib = mapU + s0;
    if (!spectral) {
        for (int j = S.tid; j < n; j += S.nt) { outQ[s0 + j] = ia[j]; outU[s0 + j] = ib[j]; }
        return;
    }
    const int lg = 31 - __clz(n);
    // sum_j z_j e^{-2 pi i jk/n} = conj( idft( conj z ) ), as in ring_anal_kernel
    for (int j = S.tid; j < S.M; j += S.nt) {
        const int pos = PADI(S.bsi < 0 ? (int)(__brev((unsigned)j) >> (32 - lg)) : j);
        if (j >= n) { S.buf[pos] = make_double2(0.0, 0.0); continue; }
        double2 z = make_double2(ia[j], -ib[j]);
        if (S.bsi >= 0) z = cmul(z, __ldg(&S.chirp[j]));
        S.buf[pos] = z;
    }
    ring_idft(P, S.buf, twq, n, S.bsi, S.tid, S.nt);
    const double s = rsqrt((double)n);
    for (int k = S.tid; k < n; k += S.nt) {
        double2 c = S.buf[PADI(k)];
        if (S.bsi >= 0) c = cmul(c, __ldg(&S.chirp[k]));
        outQ[s0 + k] = s * c.x;
        outU[s0 + k] = -s * c.y;
    }
}

// Ring stage of the PCG mat-vec A^T N^-1 A in ONE kernel: F_m(ring) -> pixels of the ring (kept in shared memory) ->
// times the pixel weights -> F'_m(ring), written over F_m.  Equivalent to ring_synth_kernel + ring_anal_kernel(pixw)
// without the map round trip through global memory, the second table load and the second launch.
template <bool SH>
__global__ void __launch_bounds__(RF_NT, 2)
ring_apply_kernel(PlanDev P, const RingJob* __restrict__ jobs, const int2* __restrict__ groups, double2* __restrict__ Fm,
                  const double* __restrict__ pixw, const int* __restrict__ skip, const unsigned char* __restrict__ ract, int spin2,
                  int64_t f_stride, const double* __restrict__ wconst)
{
    if (skip && *skip) return;
    if (group_idle(ract, jobs, groups)) return;
    extern __shared__ double2 smem[];
    Fm += blockIdx.y * f_stride;   // chain batch: blockIdx.y = chain, same pixel weights
    double2* twq = smem;
    if (group_const(wconst, jobs, groups)) {
        // Constant pixel weight w on each ring of the group: x_j = sum_k X_k e^{2 pi i jk/n} -> w x_j -> sum_j w x_j e^{-2 pi i jk/n}
        // = n w X_k, so F'_m = n w X_{m mod n} e^{-i m phi0} follows from the alias-folded spectrum X without any transform
        const RingSub S = ring_sub(P, jobs, groups, twq + (P.tw_n >> 2) + 1);
        const int mtop = ring_mtop(P, S.job.ringA, spin2);
        const double wA = wconst[S.job.ringA], wB = wconst[S.job.ringB >= 0 ? S.job.ringB : S.job.ringA];
        // No ring of the group aliases (2 m_top <= n: every cap ring beyond the first quarter of the cap and the whole belt): X_k is
        // the single term F_m e^{i m phi0}, the phases cancel and F'_m = n w F_m streams through registers; m = 0 keeps its real
        // part (X_0 = G_0 + conj G_0 with weight 1/2) and m = n/2 (belt rings when lmax = 2 nside) meets its own mirror term.
        bool direct = true;
        {
            const int2 g = groups[blockIdx.x];
            for (int s = 0; s < g.y; ++s) {
                const int ra = jobs[g.x + s].ringA;
                direct = direct && 2 * ring_mtop(P, ra, spin2) <= P.ring_nphi[ra];
            }
        }
        if (direct) {
            const RingJob& job = S.job;
            const double sa = (double)S.n * wA, sb = (double)S.n * wB;
            for (int m = S.tid; m <= mtop; m += S.nt) {
                const int64_t ia = fm_ring_index<SH>(P, job.compA, job.ringA, m);
                const int64_t ib = job.ringB >= 0 ? fm_ring_index<SH>(P, job.compB, job.ringB, m) : ia;
                double2 a = Fm[ia], b = job.ringB >= 0 ? Fm[ib] : make_double2(0.0, 0.0);
                if (m == 0) { a.y = 0.0; b.y = 0.0; }
                else if (2 * m == S.n) {
                    const double2 e2 = ring_phase(P, job.ringA, 2 * m);   // F + conj(F e^{2 i m phi0})
                    const double2 ta = cmul(a, e2), tb = cmul(b, e2);
                    a = make_double2(a.x + ta.x, a.y - ta.y);
                    b = make_double2(b.x + tb.x, b.y - tb.y);
                }
                Fm[ia] = make_double2(sa * a.x, sa * a.y);
                if (job.ringB >= 0) Fm[ib] = make_double2(sb * b.x, sb * b.y);
            }
            return;
        }
        ring_build_Z<SH>(P, S, Fm, mtop, S.scratch, false, true);
        __syncthreads();
        const double half_n = 0.5 * (double)S.n;
        ring_unpack_F<SH>(P, S, UNPACK_PLAIN, Fm, mtop, nullptr, half_n * wA, half_n * wB);
        return;
    }
    load_twq(P, twq);
    const RingSub S = ring_sub(P, jobs, groups, twq + (P.tw_n >> 2) + 1);
    const int n = S.n;
    const double* wa = pixw + ring_first_pixel<SH>(P, S.job.ringA);
    const double* wb = S.job.ringB >= 0 ? pixw + ring_first_pixel<SH>(P, S.job.ringB) : wa;
    const int mtop = ring_mtop(P, S.job.ringA, spin2);
    ring_build_Z<SH>(P, S, Fm, mtop, S.scratch);
    __syncthreads();
    ring_idft(P, S.buf, twq, n, S.bsi, S.tid, S.nt);
    if (S.bsi < 0) {
        // pixels z_j = a_j + i b_j in natural order -> weighted (as the first pass of the transform loads them) -> forward DIF
        // transform (bit-reversed output)
        auto weigh = [wa, wb](int j, double2 z) { return make_double2(z.x * wa[j], z.y * wb[j]); };
        fft_dif<false>(S.buf, n, twq, P.tw_n, nullptr, S.tid, S.nt, weigh);
        ring_unpack_F<SH>(P, S, UNPACK_BREV, Fm, mtop);
    } else {
        // Bluestein both ways: Z = conj(idft(conj z)); the chirp of the synthesis output, the pixel weights, the chirp of the
        // analysis input and the zero padding are applied in one pointwise pass, the last chirp as the spectrum is unpacked
        // (fusing this product into the first radix-16 pass of the next transform was measured SLOWER: 49 vs 43 us per 4096-point
        // ring; 48 more global loads inside a pass that already holds 16 complex values in registers, and spills)
        const double2* chirp = S.chirp;
        for (int j = S.tid; j < S.M; j += S.nt) {
            if (j >= n) { S.buf[PADI(j)] = make_double2(0.0, 0.0); continue; }
            const double2 c = __ldg(&chirp[j]);
            const double2 z = cmul(S.buf[PADI(j)], c);
            S.buf[PADI(j)] = cmul(make_double2(z.x * wa[j], -z.y * wb[j]), c);
        }
        ring_idft(P, S.buf, twq, n, S.bsi, S.tid, S.nt);
        ring_unpack_F<SH>(P, S, UNPACK_CONJ, Fm, mtop, chirp);
    }
    __syncthreads();
}

// ------------------------------------------------------------------ split path (rings longer than one CTA can hold)
// n = 4 n2.  Synthesis (z_j = sum_k Z_k e^{+2 pi i jk/n}, j = j2 + n2 q, k = 4a + b):
//   z_{j2 + n2 q} = sum_b i^{qb} e^{2 pi i j2 b/n} Y_b[j2],   Y_b[j2] = sum_a Z_{4a+b} e^{2 pi i j2 a/n2}
// CTA (job, b) computes Y_b with the shared-memory transform of length n2 and stores it in the scratch;
// ring_synth_combine_kernel applies the twiddles and the radix-4 butterfly and writes the pixels.
// Analysis is the transpose: CTA (job, b) loads v_b[j2] = e^{2 pi i j2 b/n} sum_q i^{qb} c_{j2 + n2 q}, transforms
// it to C_{4a+b}, and ring_anal_finish_kernel unpacks the two real sequences into F_m.
template <bool SH>
__device__ __forceinline__ double2 fold_spectrum(const PlanDev& P, const double2* __restrict__ Fm, int comp, int ring, int k, int n, int L)
{  // X_k = G_k + conj G_{n-k},  G_k = sum_{m = k mod n, m <= L} w_m F_m e^{i m phi0}
    const int kk = (n - k) % n;
    double2 g = make_double2(0.0, 0.0), h = g;
    for (int m = k; m <= L; m += n) {
        const double w = m ? 1.0 : 0.5;
        const double2 ph = ring_phase(P, ring, m);
        g = cadd(g, cmul(Fm[fm_ring_index<SH>(P, comp, ring, m)], make_double2(ph.x * w, ph.y * w)));
    }
    for (int m = kk; m <= L; m += n) {
        const double w = m ? 1.0 : 0.5;
        const double2 ph = ring_phase(P, ring, m);
        h = cadd(h, cmul(Fm[fm_ring_index<SH>(P, comp, ring, m)], make_double2(ph.x * w, ph.y * w)));
    }
    return make_double2(g.x + h.x, g.y - h.y);
}

__device__ __forceinline__ double2 mul_ipow(double2 v, int p)
{  // v * i^p
    p &= 3;
    return p == 0 ? v : p == 1 ? make_double2(-v.y, v.x) : p == 2 ? make_double2(-v.x, -v.y) : make_double2(v.y, -v.x);
}

__device__ __forceinline__ double2 unit_root(int num, int n)
{  // exp(2 pi i num / n), 0 <= num
    const int r = (int)((2LL * num) % (2LL * n));
    double s, c;
    sincospi((double)r / (double)n, &s, &c);
    return make_double2(c, s);
}

template <bool SH>
__global__ void __launch_bounds__(RF_NT, 2)
ring_synth_split_kernel(PlanDev P, const SplitJob* __restrict__ jobs, const double2* __restrict__ Fm, double2* __restrict__ scratch,
                        const int* __restrict__ skip, int spin2, const unsigned char* __restrict__ ract)
{
    if (skip && *skip) return;
    extern __shared__ double2 smem[];
    const SplitJob job = jobs[blockIdx.x >> 2];
    if (split_idle(ract, job)) return;
    const int mtop = ring_mtop(P, job.ringA, spin2);
    const int b = blockIdx.x & 3;
    const int n = P.ring_nphi[job.ringA], n2 = n >> 2, bsi = job.bs2;
    double2* twq = smem;
    double2* buf = twq + (P.tw_n >> 2) + 1;
    load_twq(P, twq);
    const int lg = 31 - __clz(n2);
    const double2* chirp = bsi >= 0 ? P.bs_tab + P.bs[bsi].chirp_off : nullptr;
    const int M = bsi >= 0 ? P.bs[bsi].M : n2;
    for (int a = threadIdx.x; a < M; a += RF_NT) {
        const int pos = PADI(bsi < 0 ? (int)(__brev((unsigned)a) >> (32 - lg)) : a);
        if (a >= n2) { buf[pos] = make_double2(0.0, 0.0); continue; }
        const int k = 4 * a + b;
        const double2 xa = fold_spectrum<SH>(P, Fm, job.compA, job.ringA, k, n, mtop);
        double2 z = xa;
        if (job.ringB >= 0) {
            const double2 xb = fold_spectrum<SH>(P, Fm, job.compB, job.ringB, k, n, mtop);
            z = make_double2(xa.x - xb.y, xa.y + xb.x);  // + i Xb
        }
        if (bsi >= 0) z = cmul(z, __ldg(&chirp[a]));
        buf[pos] = z;
    }
    ring_idft(P, buf, twq, n2, bsi);
    double2* out = scratch + job.off + (int64_t)b * n2;
    for (int j = threadIdx.x; j < n2; j += RF_NT) {
        double2 z = buf[PADI(j)];
        if (bsi >= 0) z = cmul(z, __ldg(&chirp[j]));
        out[j] = z;
    }
}

template <bool SH>
__global__ void __launch_bounds__(RF_NT)
ring_synth_combine_kernel(PlanDev P, const SplitJob* __restrict__ jobs, const double2* __restrict__ scratch, double* __restrict__ mapQ,
                          double* __restrict__ mapU, const int* __restrict__ skip, const unsigned char* __restrict__ ract)
{
    if (skip && *skip) return;
    const SplitJob job = jobs[blockIdx.x];
    if (split_idle(ract, job)) return;
    const int n = P.ring_nphi[job.ringA], n2 = n >> 2;
    const double2* Y = scratch + job.off;
    double* oa = (job.compA ? mapU : mapQ) + ring_first_pixel<SH>(P, job.ringA);
    double* ob = job.ringB >= 0 ? (job.compB ? mapU : mapQ) + ring_first_pixel<SH>(P, job.ringB) : nullptr;
    for (int j = threadIdx.x; j < n2; j += RF_NT) {
        const double2 t1 = unit_root(j, n), t2 = cmul(t1, t1), t3 = cmul(t2, t1);
        const double2 y0 = Y[j], y1 = cmul(Y[n2 + j], t1), y2 = cmul(Y[2 * n2 + j], t2), y3 = cmul(Y[3 * n2 + j], t3);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const double2 z = cadd(cadd(y0, mul_ipow(y1, q)), cadd(mul_ipow(y2, 2 * q), mul_ipow(y3, 3 * q)));
            oa[j + q * n2] = z.x;
            if (ob) ob[j + q * n2] = z.y;
        }
    }
}

template <bool SH>
__global__ void __launch_bounds__(RF_NT, 2)
ring_anal_split_kernel(PlanDev P, const SplitJob* __restrict__ jobs, const double* __restrict__ mapQ, const double* __restrict__ mapU,
                       const double* __restrict__ pixw, double2* __restrict__ scratch, const int* __restrict__ skip, const unsigned char* __restrict__ ract)
{
    if (skip && *skip) return;
    extern __shared__ double2 smem[];
    const SplitJob job = jobs[blockIdx.x >> 2];
    if (split_idle(ract, job)) return;
    const int b = blockIdx.x & 3;
    const int n = P.ring_nphi[job.ringA], n2 = n >> 2, bsi = job.bs2;
    double2* twq = smem;
    double2* buf = twq + (P.tw_n >> 2) + 1;
    load_twq(P, twq);
    const int64_t sa = ring_first_pixel<SH>(P, job.ringA), sb = job.ringB >= 0 ? ring_first_pixel<SH>(P, job.ringB) : 0;
    const double* ia = (job.compA ? mapU : mapQ) + sa;
    const double* ib = job.ringB >= 0 ? (job.compB ? mapU : mapQ) + sb : nullptr;
    const int lg = 31 - __clz(n2);
    const double2* chirp = bsi >= 0 ? P.bs_tab + P.bs[bsi].chirp_off : nullptr;
    const int M = bsi >= 0 ? P.bs[bsi].M : n2;
    for (int j = threadIdx.x; j < M; j += RF_NT) {
        const int pos = PADI(bsi < 0 ? (int)(__brev((unsigned)j) >> (32 - lg)) : j);
        if (j >= n2) { buf[pos] = make_double2(0.0, 0.0); continue; }
        double2 v = make_double2(0.0, 0.0);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int jj = j + q * n2;
            double x = ia[jj], y = ib ? ib[jj] : 0.0;
            if (pixw) { x *= pixw[sa + jj]; if (ib) y *= pixw[sb + jj]; }
            v = cadd(v, mul_ipow(make_double2(x, -y), q * b));   // c_j = conj(z_j)
        }
        if (b) v = cmul(v, unit_root(j * b, n));
        if (bsi >= 0) v = cmul(v, __ldg(&chirp[j]));
        buf[pos] = v;
    }
    ring_idft(P, buf, twq, n2, bsi);
    double2* out = scratch + job.off + (int64_t)b * n2;   // C_{4a+b} at [b][a]
    for (int a = threadIdx.x; a < n2; a += RF_NT) {
        double2 z = buf[PADI(a)];
        if (bsi >= 0) z = cmul(z, __ldg(&chirp[a]));
        out[a] = z;
    }
}

template <bool SH>
__global__ void __launch_bounds__(RF_NT)
ring_anal_finish_kernel(PlanDev P, const SplitJob* __restrict__ jobs, const double2* __restrict__ scratch, double2* __restrict__ Fm,
                        const int* __restrict__ skip, const unsigned char* __restrict__ ract)
{
    if (skip && *skip) return;
    const SplitJob job = jobs[blockIdx.x];
    if (split_idle(ract, job)) return;
    const int L = P.lmax, n = P.ring_nphi[job.ringA], n2 = n >> 2;
    const double2* Cs = scratch + job.off;
    for (int m = threadIdx.x; m <= L; m += RF_NT) {
        const int k = m % n, kk = (n - k) % n;
        const double2 c1 = Cs[(int64_t)(k & 3) * n2 + (k >> 2)], c2 = Cs[(int64_t)(kk & 3) * n2 + (kk >> 2)];
        const double2 z1 = make_double2(c1.x, -c1.y);  // Z[k]
        const double2 z2c = c2;                         // conj Z[n-k]
        const double2 xa = make_double2(0.5 * (z1.x + z2c.x), 0.5 * (z1.y + z2c.y));
        const double2 d = csub(z1, z2c);
        const double2 xb = make_double2(0.5 * d.y, -0.5 * d.x);
        Fm[fm_ring_index<SH>(P, job.compA, job.ringA, m)] = cmulc(xa, ring_phase(P, job.ringA, m));
        if (job.ringB >= 0) Fm[fm_ring_index<SH>(P, job.compB, job.ringB, m)] = cmulc(xb, ring_phase(P, job.ringB, m));
    }
}

// ------------------------------------------------------------------ host side
static int next_pow2(int v) { int p = 1; while (p < v) p <<= 1; return p; }

static int ring_M(int n) { return (n & (n - 1)) == 0 ? n : next_pow2(2 * n - 1); }

int gs_ring_setup(gs_plan* p)
{
    const int nside = p->d.nside, nring = p->d.nring, npair = p->d.npair, L = p->d.lmax;
    const size_t smem_max = 227 * 1024;
    std::vector<int> rn(nring);
    for (int r = 0; r < nring; ++r) { int i = std::min(r + 1, 4 * nside - (r + 1)); rn[r] = i < nside ? 4 * i : 4 * nside; }
    // direct path: transform buffer(s) + quarter twiddle table in one CTA; Mcap = largest power-of-two transform
    // length taken directly (two CTAs per SM).  Longer rings take the split path (n/4 per CTA).
    // (+ RF_NT entries: partial alias sums of rings shorter than their thread count, see ring_build_Z)
    auto direct_smem = [&](int M, int twn) { return (size_t)((PADLEN(M) + 16 + RF_NT) + twn / 4 + 1) * sizeof(double2); };
    int Mcap = 4;
    while (2 * direct_smem(2 * Mcap, 2 * Mcap) <= smem_max) Mcap *= 2;
    (void)L;
    if (const char* e = getenv("GS_RING_MCAP")) {  // test knob: exercise the split path at small nside
        const int v = atoi(e);
        if (v >= 4 && v < Mcap && (v & (v - 1)) == 0) Mcap = v;
    }
    auto is_split = [&](int ring) { return ring_M(rn[ring]) > Mcap; };
    std::map<int, int> n2bs;
    std::vector<BluesteinDesc> descs;
    int64_t off = 0;
    int maxMd = 4, maxMs = 4;
    auto need_len = [&](int n, int& maxM) {
        maxM = std::max(maxM, ring_M(n));
        if ((n & (n - 1)) == 0 || n2bs.count(n)) return;
        BluesteinDesc d;
        d.n = n; d.M = next_pow2(2 * n - 1); d.chirp_off = off; off += n; d.bhat_off = off; off += d.M;
        n2bs[n] = (int)descs.size();
        descs.push_back(d);
    };
    for (int r = 0; r < npair; ++r) {
        if (!is_split(r)) need_len(rn[r], maxMd);
        else {
            if (ring_M(rn[r] / 4) > Mcap) {
                gs_set_error("ring FFT: nside %d / lmax %d needs a deeper ring split than this build provides", nside, L);
                return GS_E_BADARG;
            }
            need_len(rn[r] / 4, maxMs);
        }
    }
    const int maxM = std::max(maxMd, maxMs);
    std::vector<int> rbs(nring);
    for (int r = 0; r < nring; ++r) rbs[r] = (!is_split(r) && n2bs.count(rn[r])) ? n2bs[rn[r]] : -1;
    p->d.max_M = maxM;
    p->d.tw_n = maxM;
    p->ring_smem = direct_smem(std::max(maxMd, std::min(4096, Mcap)), maxM);   // groups of short rings fill up to 4096 points
    p->split_smem = (size_t)(PADLEN(maxMs) + maxM / 4 + 1) * sizeof(double2);
    if (p->ring_smem > smem_max || p->split_smem > smem_max) {
        gs_set_error("ring FFT needs %zu bytes of shared memory (> 227 KB): nside/lmax too large for this build", p->ring_smem);
        return GS_E_BADARG;
    }
    std::vector<double2> tw(maxM);
    for (int k = 0; k < maxM; ++k) {
        long double a = 2.0L * 3.14159265358979323846264338327950288L * k / maxM;
        tw[k] = make_double2((double)cosl(a), (double)(-sinl(a)));
    }
    void* d = nullptr;
    GS_CHECK_CUDA(cudaMalloc(&d, tw.size() * sizeof(double2))); p->owned.push_back(d);
    GS_CHECK_CUDA(cudaMemcpy(d, tw.data(), tw.size() * sizeof(double2), cudaMemcpyHostToDevice));
    p->d.tw = (const double2*)d;
    GS_CHECK_CUDA(cudaMalloc(&d, std::max<size_t>(1, nring) * sizeof(int))); p->owned.push_back(d);
    GS_CHECK_CUDA(cudaMemcpy(d, rbs.data(), nring * sizeof(int), cudaMemcpyHostToDevice));
    p->d.ring_bs = (const int*)d;
    GS_CHECK_CUDA(cudaMalloc(&d, std::max<size_t>(1, descs.size()) * sizeof(BluesteinDesc))); p->owned.push_back(d);
    if (!descs.empty()) GS_CHECK_CUDA(cudaMemcpy(d, descs.data(), descs.size() * sizeof(BluesteinDesc), cudaMemcpyHostToDevice));
    p->d.bs = (const BluesteinDesc*)d;
    GS_CHECK_CUDA(cudaMalloc(&d, std::max<int64_t>(1, off) * sizeof(double2))); p->owned.push_back(d);
    p->d.bs_tab = (const double2*)d;

    GS_CHECK_CUDA(cudaFuncSetAttribute(bluestein_setup_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    GS_CHECK_CUDA(cudaFuncSetAttribute(ring_synth_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    GS_CHECK_CUDA(cudaFuncSetAttribute(ring_anal_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    GS_CHECK_CUDA(cudaFuncSetAttribute(ring_synth_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    GS_CHECK_CUDA(cudaFuncSetAttribute(ring_anal_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    GS_CHECK_CUDA(cudaFuncSetAttribute(ring_mwg_data_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    GS_CHECK_CUDA(cudaFuncSetAttribute(ring_apply_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    GS_CHECK_CUDA(cudaFuncSetAttribute(ring_apply_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    GS_CHECK_CUDA(cudaFuncSetAttribute(ring_synth_split_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    GS_CHECK_CUDA(cudaFuncSetAttribute(ring_anal_split_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    GS_CHECK_CUDA(cudaFuncSetAttribute(ring_synth_split_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    GS_CHECK_CUDA(cudaFuncSetAttribute(ring_anal_split_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    if (!descs.empty()) {
        const size_t bsm = (size_t)(PADLEN(maxM) + maxM / 4 + 1) * sizeof(double2);
        bluestein_setup_kernel<<<(int)descs.size(), RF_NT, bsm>>>(p->d, (double2*)d, (int)descs.size());
        GS_CHECK_LAUNCH();
    }

    // job lists, heaviest transforms first; sharded plans transform only the rings of the owned ring pairs
    auto cost = [&](int ring) { int n = rn[ring]; return rbs[ring] < 0 ? n : 3 * descs[rbs[ring]].M; };
    auto owned = [&](int ring) { return p->world <= 1 || std::min(ring, nring - 1 - ring) % p->world == p->rank; };
    std::vector<RingJob> j2, j0;
    std::vector<SplitJob> s2, s0;
    int64_t so2 = 0, so0 = 0;
    auto bs2_of = [&](int ring) { const int n2 = rn[ring] / 4; return n2bs.count(n2) ? n2bs[n2] : -1; };
    for (int r = 0; r < nring; ++r) {
        if (!owned(r)) continue;
        if (!is_split(r)) j2.push_back(RingJob{r, 0, r, 1});
        else { s2.push_back(SplitJob{r, 0, r, 1, bs2_of(r), 0, so2}); so2 += rn[r]; }
    }
    for (int r = 0; r < npair; ++r) {
        const int rs = nring - 1 - r;
        if (!owned(r)) continue;
        if (!is_split(r)) j0.push_back(RingJob{r, 0, rs != r ? rs : -1, 0});
        else { s0.push_back(SplitJob{r, 0, rs != r ? rs : -1, 0, bs2_of(r), 0, so0}); so0 += rn[r]; }
    }
    std::stable_sort(j2.begin(), j2.end(), [&](const RingJob& a, const RingJob& b) { return cost(a.ringA) > cost(b.ringA); });
    std::stable_sort(j0.begin(), j0.end(), [&](const RingJob& a, const RingJob& b) { return cost(a.ringA) > cost(b.ringA); });
    // groups of 1 / 2 / 4 consecutive jobs with the same transform length and kind share a CTA (see RingGroup in the
    // kernels): a pass of an M-point transform has M / 16 radix-16 butterflies, RF_NT threads need M >= 4096 alone
    const int group_points = std::min(4096, Mcap);
    auto make_groups = [&](const std::vector<RingJob>& jobs) {
        std::vector<int2> g;
        size_t i = 0;
        while (i < jobs.size()) {
            const int key = cost(jobs[i].ringA);
            const int M = ring_M(rn[jobs[i].ringA]);
            size_t e = i;
            while (e < jobs.size() && cost(jobs[e].ringA) == key) ++e;
            const int want = std::max(1, std::min(4, group_points / M));
            while (i < e) {
                int cnt = (int)std::min<size_t>(want, e - i);
                if (cnt == 3) cnt = 2;
                g.push_back(make_int2((int)i, cnt));
                i += cnt;
            }
        }
        return g;
    };
    const std::vector<int2> g2 = make_groups(j2), g0 = make_groups(j0);
    auto put = [&](const void* h, size_t bytes, void** out) -> int {
        void* q = nullptr;
        GS_CHECK_CUDA(cudaMalloc(&q, std::max<size_t>(16, bytes)));
        p->owned.push_back(q);
        if (bytes) GS_CHECK_CUDA(cudaMemcpy(q, h, bytes, cudaMemcpyHostToDevice));
        *out = q;
        return GS_OK;
    };
    int rc;
    if ((rc = put(j2.data(), j2.size() * sizeof(RingJob), (void**)&p->jobs2))) return rc;
    if ((rc = put(j0.data(), j0.size() * sizeof(RingJob), (void**)&p->jobs0))) return rc;
    if ((rc = put(s2.data(), s2.size() * sizeof(SplitJob), (void**)&p->sjobs2))) return rc;
    if ((rc = put(s0.data(), s0.size() * sizeof(SplitJob), (void**)&p->sjobs0))) return rc;
    if ((rc = put(g2.data(), g2.size() * sizeof(int2), (void**)&p->groups2))) return rc;
    if ((rc = put(g0.data(), g0.size() * sizeof(int2), (void**)&p->groups0))) return rc;
    if ((rc = put(g2.data(), g2.size() * sizeof(int2), (void**)&p->groups2_dyn))) return rc;
    if ((rc = put(g0.data(), g0.size() * sizeof(int2), (void**)&p->groups0_dyn))) return rc;
    p->ngroups2 = (int)g2.size(); p->ngroups0 = (int)g0.size();
    p->njobs2 = (int)j2.size(); p->njobs0 = (int)j0.size();
    p->nsjobs2 = (int)s2.size(); p->nsjobs0 = (int)s0.size();
    if (so2 || so0) {
        GS_CHECK_CUDA(cudaMalloc(&d, (size_t)std::max(so2, so0) * sizeof(double2)));
        p->owned.push_back(d);
        p->ring_scratch = (double2*)d;
    }
    return GS_OK;
}

int gs_ring_synth(gs_plan* p, int spin, double* mapQ, double* mapU, cudaStream_t st, const int* skip, int nc, int64_t map_stride,
                  const double* wconst)
{
    if (nc > 1 && p->world > 1) { gs_set_error("chain batches need an unsharded plan"); return GS_E_BADARG; }
    if (wconst && (spin != 2 || p->world > 1 || p->nsjobs2 > 0 || nc > 1)) { gs_set_error("spectral ring storage: spin 2, unsharded plan without split rings"); return GS_E_BADARG; }
    const int nj = spin == 0 ? p->ngroups0 : p->ngroups2, ns = spin == 0 ? p->nsjobs0 : p->nsjobs2;
    if (nc > 1 && ns > 0) {   // rings on the split path (nside >= 1024) share one scratch buffer: the chains of a batch take turns
        double2* F0 = p->Fm;
        int rc = GS_OK;
        for (int c = 0; c < nc && rc == GS_OK; ++c) {
            p->Fm = F0 + c * gs_fm_stride(p);
            rc = gs_ring_synth(p, spin, mapQ + c * map_stride, spin ? mapU + c * map_stride : mapU, st, skip, 1, 0);
        }
        p->Fm = F0;
        return rc;
    }
    const RingJob* jobs = spin == 0 ? p->jobs0 : p->jobs2;
    const int2* grp = spin == 0 ? p->groups0 : p->groups2;
    const SplitJob* sj = spin == 0 ? p->sjobs0 : p->sjobs2;
    const unsigned char* ract = p->use_act ? p->act_ring : nullptr;   // PCG mat-vec: rings without pixel weight are left out
    double* mu = spin == 0 ? mapQ : mapU;
    const bool sh = p->world > 1;
    const double2* F = sh ? p->Fx : p->Fm;
    if (ns > 0) {  // long rings first: they are the heavy ones
        if (sh) {
            ring_synth_split_kernel<true><<<4 * ns, RF_NT, p->split_smem, st>>>(p->d, sj, F, p->ring_scratch, skip, spin ? 1 : 0, ract);
            ring_synth_combine_kernel<true><<<ns, RF_NT, 0, st>>>(p->d, sj, p->ring_scratch, mapQ, mu, skip, ract);
        } else {
            ring_synth_split_kernel<false><<<4 * ns, RF_NT, p->split_smem, st>>>(p->d, sj, F, p->ring_scratch, skip, spin ? 1 : 0, ract);
            ring_synth_combine_kernel<false><<<ns, RF_NT, 0, st>>>(p->d, sj, p->ring_scratch, mapQ, mu, skip, ract);
        }
        GS_CHECK_LAUNCH();
        g_gs_launches += 2;
    }
    if (nj > 0) {
        if (sh) ring_synth_kernel<true><<<nj, RF_NT, p->ring_smem, st>>>(p->d, jobs, grp, F, mapQ, mu, skip, 0, 0, nullptr, spin ? 1 : 0, ract, nullptr);
        else ring_synth_kernel<false><<<dim3(nj, nc), RF_NT, p->ring_smem, st>>>(p->d, jobs, grp, F, mapQ, mu, skip, nc > 1 ? gs_fm_stride(p) : 0, nc > 1 ? map_stride : 0, nullptr, spin ? 1 : 0, ract, wconst);
        GS_CHECK_LAUNCH();
    }
    g_gs_launches += 1;
    return GS_OK;
}

int gs_ring_anal(gs_plan* p, int spin, const double* mapQ, const double* mapU, const double* pixw, cudaStream_t st,
                 const int* skip, int nc, int64_t map_stride)
{
    if (nc > 1 && p->world > 1) { gs_set_error("chain batches need an unsharded plan"); return GS_E_BADARG; }
    const int nj = spin == 0 ? p->ngroups0 : p->ngroups2, ns = spin == 0 ? p->nsjobs0 : p->nsjobs2;
    if (nc > 1 && ns > 0) {   // split path: one chain after the other (see gs_ring_synth)
        double2* F0 = p->Fm;
        int rc = GS_OK;
        for (int c = 0; c < nc && rc == GS_OK; ++c) {
            p->Fm = F0 + c * gs_fm_stride(p);
            rc = gs_ring_anal(p, spin, mapQ + c * map_stride, spin ? mapU + c * map_stride : mapU, pixw, st, skip, 1, 0);
        }
        p->Fm = F0;
        return rc;
    }
    const RingJob* jobs = spin == 0 ? p->jobs0 : p->jobs2;
    const int2* grp = spin == 0 ? p->groups0 : p->groups2;
    const SplitJob* sj = spin == 0 ? p->sjobs0 : p->sjobs2;
    const unsigned char* ract = p->use_act ? p->act_ring : nullptr;
    const double* mu = spin == 0 ? mapQ : mapU;
    const bool sh = p->world > 1;
    double2* F = sh ? p->Fx : p->Fm;
    if (ns > 0) {
        if (sh) {
            ring_anal_split_kernel<true><<<4 * ns, RF_NT, p->split_smem, st>>>(p->d, sj, mapQ, mu, pixw, p->ring_scratch, skip, ract);
            ring_anal_finish_kernel<true><<<ns, RF_NT, 0, st>>>(p->d, sj, p->ring_scratch, F, skip, ract);
        } else {
            ring_anal_split_kernel<false><<<4 * ns, RF_NT, p->split_smem, st>>>(p->d, sj, mapQ, mu, pixw, p->ring_scratch, skip, ract);
            ring_anal_finish_kernel<false><<<ns, RF_NT, 0, st>>>(p->d, sj, p->ring_scratch, F, skip, ract);
        }
        GS_CHECK_LAUNCH();
        g_gs_launches += 2;
    }
    if (nj > 0) {
        if (sh) ring_anal_kernel<true><<<nj, RF_NT, p->ring_smem, st>>>(p->d, jobs, grp, mapQ, mu, pixw, F, skip, spin ? 1 : 0, ract, 0, 0);
        else ring_anal_kernel<false><<<dim3(nj, nc), RF_NT, p->ring_smem, st>>>(p->d, jobs, grp, mapQ, mu, pixw, F, skip, spin ? 1 : 0, ract, nc > 1 ? gs_fm_stride(p) : 0, nc > 1 ? map_stride : 0);
        GS_CHECK_LAUNCH();
    }
    g_gs_launches += 1;
    return GS_OK;
}

// ring stage of A^T diag(pixw) A on the ring spectra in place; falls back to synthesis + weighted analysis through the
// plan's scratch maps when some rings take the split path
int gs_ring_apply(gs_plan* p, int spin, const double* pixw, cudaStream_t st, const int* skip, int nc)
{
    const int nj = spin == 0 ? p->ngroups0 : p->ngroups2, ns = spin == 0 ? p->nsjobs0 : p->nsjobs2;
    if (nc > 1 && (p->world > 1 || !pixw)) { gs_set_error("chain batches need an unsharded plan and pixel weights"); return GS_E_BADARG; }
    if (nc > 1 && ns > 0) {   // split path: the chains take turns through the plan's scratch maps
        double2* F0 = p->Fm;
        int rc = GS_OK;
        for (int c = 0; c < nc && rc == GS_OK; ++c) {
            p->Fm = F0 + c * gs_fm_stride(p);
            rc = gs_ring_apply(p, spin, pixw, st, skip, 1);
        }
        p->Fm = F0;
        return rc;
    }
    if (ns > 0 || !pixw) {
        int rc = gs_ring_synth(p, spin, p->mapQ_tmp, p->mapU_tmp, st, skip);
        if (rc) return rc;
        return gs_ring_anal(p, spin, p->mapQ_tmp, p->mapU_tmp, pixw, st, skip);
    }
    if (nj <= 0) return GS_OK;
    const RingJob* jobs = spin == 0 ? p->jobs0 : p->jobs2;
    const int2* grp = spin == 0 ? p->groups0 : p->groups2;
    // ring_wconst is filled together with the active-ring flags (gs_active_rings_build), from the weight map of this call
    const double* wconst = (p->use_act && g_gs_ring_const) ? p->ring_wconst : nullptr;
    if (wconst) grp = spin == 0 ? p->groups0_dyn : p->groups2_dyn;   // the CTAs that run transforms are dispatched first (gs_ring_order_build)
    if (p->world > 1) ring_apply_kernel<true><<<nj, RF_NT, p->ring_smem, st>>>(p->d, jobs, grp, p->Fx, pixw, skip, p->use_act ? p->act_ring : nullptr, spin ? 1 : 0, 0, nullptr);
    else ring_apply_kernel<false><<<dim3(nj, nc), RF_NT, p->ring_smem, st>>>(p->d, jobs, grp, p->Fm, pixw, skip, p->use_act ? p->act_ring : nullptr, spin ? 1 : 0, nc > 1 ? gs_fm_stride(p) : 0, wconst);
    GS_CHECK_LAUNCH();
    g_gs_launches += 1;
    return GS_OK;
}

// nb spin-2 ring syntheses in one launch: spectra F + k f_stride (m <= mmax[k]) -> maps Q/U + k map_stride
int gs_ring_order_build(gs_plan* p, cudaStream_t st)
{
    if (p->world > 1 || !p->ring_wconst) return GS_OK;
    if (p->ngroups2 > 0) ring_order_kernel<<<1, 1024, 0, st>>>(p->jobs2, p->groups2, p->ngroups2, p->act_ring, p->ring_wconst, p->groups2_dyn);
    if (p->ngroups0 > 0) ring_order_kernel<<<1, 1024, 0, st>>>(p->jobs0, p->groups0, p->ngroups0, p->act_ring, p->ring_wconst, p->groups0_dyn);
    GS_CHECK_LAUNCH();
    g_gs_launches += 2;
    return GS_OK;
}

int gs_ring_mwg_data(gs_plan* p, const double* mapQ, const double* mapU, double* outQ, double* outU, const double* wconst, cudaStream_t st)
{
    if (p->world > 1 || p->nsjobs2 > 0) { gs_set_error("spectral ring storage needs an unsharded plan without split rings"); return GS_E_BADARG; }
    if (p->ngroups2 <= 0) return GS_OK;
    ring_mwg_data_kernel<<<p->ngroups2, RF_NT, p->ring_smem, st>>>(p->d, p->jobs2, p->groups2, mapQ, mapU, outQ, outU, wconst);
    GS_CHECK_LAUNCH();
    g_gs_launches += 1;
    return GS_OK;
}

int gs_ring_synth_batch(gs_plan* p, const double2* F, int64_t f_stride, const int* mmax, double* mapQ, double* mapU,
                        int64_t map_stride, int nb, cudaStream_t st, const unsigned char* ract, const double* wconst)
{
    if (p->world > 1 || p->nsjobs2 > 0) { gs_set_error("batched ring synthesis needs an unsharded plan without split rings"); return GS_E_BADARG; }
    if (nb <= 0 || p->ngroups2 <= 0) return GS_OK;
    ring_synth_kernel<false><<<dim3(p->ngroups2, nb), RF_NT, p->ring_smem, st>>>(p->d, p->jobs2, wconst ? p->groups2_dyn : p->groups2, F, mapQ, mapU,
                                                                                 nullptr, f_stride, map_stride, mmax, 1, ract, wconst);
    GS_CHECK_LAUNCH();
    g_gs_launches += 1;
    return GS_OK;
}
