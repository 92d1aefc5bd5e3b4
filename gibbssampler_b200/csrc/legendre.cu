// Legendre stage of the spin-0 / spin-2 spherical-harmonic transforms (sm_100a, FP64).
//
// Replaces the libsharp Legendre loops behind hp.alm2map / hp.map2alm (SURVEY.md 8a rows A6, A7).
//
// One thread owns R north/south ring pairs and walks l = max(m,spin) .. lmax for ONE m with the
// normalised Wigner-d recurrence  mu_{l+1} = (a_l x -+ b_l) mu_l - mu_{l-1}  (2 DFMA per chain and
// step; table built in long double by plan.cu).  All threads of a block share m, so the a_lm
// tile (pre-multiplied by alpha_lm, the -1/2 of the E/B convention, an optional per-l filter and
// the real-layout 1/sqrt2) and the recurrence coefficients are staged once per block in shared
// memory and read back as warp-broadcast LDS.128.  The north/south symmetry
// lam^{+-}_{lm}(pi - theta) = (-1)^(l+m) lam^{-+}_{lm}(theta) halves the work: terms are
// accumulated into a symmetric and an antisymmetric part (unrolled by two in l so that the
// parity is static), north = S + A, south = S - A.
// Range: seeds ~ sin(theta)^m underflow FP64 near the poles, so every ring carries an integer
// scale (true value = v * 2^(-256 scale)); a warp runs (A) recurrence only while all its lanes are
// below 2^-900, (B) predicated accumulation while some are, (C) the unchecked fast loop.
// Analysis is the exact transpose; its sum over rings is a register fold + warp shuffle
// reduce-scatter (9 SHFL.64 per two l for 8 values), then a shared-memory sum over the warps of
// the block and one deterministic partial per 256-ring-pair chunk, combined by leg_finish_kernel.
#include <algorithm>
#include <type_traits>

#include "gs_internal.h"

#ifndef LEG_NT
#define LEG_NT 128   // threads per block
#endif
#define LEG_NW (LEG_NT / 32)
#define LEG_TL LEG_NT   // l-tile (even): one staged l per thread
#ifndef LEG_SU
#define LEG_SU 1        // synthesis kernel: multipoles staged per thread and tile (tile = LEG_SU * LEG_NT, one barrier per tile)
#endif
#define LEG_TLS (LEG_SU * LEG_NT)
#ifndef LEG_R
#define LEG_R 2      // ring pairs per thread (synthesis)
#endif
#ifndef LEG_R2
#define LEG_R2 2     // ring pairs per thread of the chain-batched synthesis (NC = 2)
#endif
#ifndef LEG_RA
#define LEG_RA 4     // ring pairs per thread (analysis); LEG_NT * LEG_RA ring pairs per partial chunk
#endif
#ifndef LEG_UA
#define LEG_UA 2     // unroll of the analysis fast loop (two reduce-scatters in flight)
#endif
#ifdef LEG_MINB_S     // minimum resident blocks per SM asked of the synthesis kernel (tuning; default: none)
#define LEG_SYNTH_BOUNDS __launch_bounds__(LEG_NT, LEG_MINB_S)
#else
#define LEG_SYNTH_BOUNDS __launch_bounds__(LEG_NT)
#endif
#define FOLD3_NB 8   // spin-2 analysis fast loop: pairs of l whose last three reduce-scatter stages are summed at once in shared memory
#define FULL 0xffffffffu
#ifndef LEG_CHK
#define LEG_CHK 4     // pairs of l between two looks at which ring groups of a warp have come alive (transition phase)
#endif
constexpr int kUnrollA = LEG_UA;

__device__ __forceinline__ double pow2i(int e) { return __hiloint2double((e + 1023) << 20, 0); }

// v != 0 normal -> mantissa in [0.5,1) (sign kept), e += exponent
__device__ __forceinline__ void renorm(double& v, int& e)
{
    int hi = __double2hiint(v), lo = __double2loint(v);
    e += ((hi >> 20) & 0x7ff) - 1022;
    v = __hiloint2double((hi & 0x800fffff) | (1022 << 20), lo);
}

// x^n = mant * 2^ex for 0 < x <= 1 (binary exponentiation with exponent tracking)
__device__ __forceinline__ void pow_scaled(double x, int n, double& mant, int& ex)
{
    double r = 0.5, b = x;
    int er = 1, eb = 0;
    renorm(b, eb);
    while (n > 0) {
        if (n & 1) { r *= b; er += eb; renorm(r, er); }
        b *= b; eb *= 2; renorm(b, eb);
        n >>= 1;
    }
    mant = r; ex = er;
}

// sin(theta_p)^m = mant 2^ex from the plan's table (built once by sinpow_build_kernel with pow_scaled: the binary
// exponentiation is a serial chain of ~2 log2(m) dependent multiplications that used to open every (pair, m) thread)
__device__ __forceinline__ void load_sinpow(const PlanDev& P, int p, int m, double& mant, int& ex)
{
    const double2 raw = __ldg(reinterpret_cast<const double2*>(P.sinpow) + (int64_t)m * P.npair + p);
    mant = raw.x;
    ex = __double2loint(raw.y);
}

__global__ void __launch_bounds__(256) sinpow_build_kernel(PlanDev P, ScaledSeed* __restrict__ tab)
{
    const int p = blockIdx.x * blockDim.x + threadIdx.x, m = blockIdx.y;
    if (p >= P.npair) return;
    ScaledSeed s;
    pow_scaled(P.sth[p], m, s.mant, s.ex);
    s.pad = 0;
    tab[(int64_t)m * P.npair + p] = s;
}

int gs_leg_build_sinpow(gs_plan* p)
{
    void* d = nullptr;
    GS_CHECK_CUDA(cudaMalloc(&d, (size_t)(p->d.lmax + 1) * p->d.npair * sizeof(ScaledSeed)));
    p->owned.push_back(d);
    sinpow_build_kernel<<<dim3((p->d.npair + 255) / 256, p->d.lmax + 1), 256>>>(p->d, (ScaledSeed*)d);
    GS_CHECK_LAUNCH();
    p->d.sinpow = (const ScaledSeed*)d;
    return GS_OK;
}

// Seeds of the recurrence at l0 = max(m, SPIN) for one ring: vp = mu^+ (m' = -2, or the spin-0
// chain), vm = mu^- (m' = +2), common scale sc.
template <int SPIN>
__device__ __forceinline__ void seed_ring(const PlanDev& P, int p, int m, double& vp, double& vm, int& sc)
{
    const double sth = P.sth[p];
    double mant; int ex;
    double fp, fm;  // plain factors multiplying mant * 2^ex
    if (SPIN == 0) {
        load_sinpow(P, p, m, mant, ex);
        ScaledSeed s = P.seed0[m];
        mant *= s.mant; ex += s.ex; fp = 1.0; fm = 0.0;
    } else {
        const double c2 = P.c2[p], s2 = P.s2[p];
        if (m >= 2) {
            load_sinpow(P, p, m, mant, ex);
            ScaledSeed s = P.seed2[m];
            mant *= s.mant; ex += s.ex;
            fp = s2 / c2; fm = c2 / s2;
        } else {
            const double n5 = 0.63078313050504001;  // sqrt(5 / (4 pi))
            mant = 1.0; ex = 0;
            if (m == 0) { fp = fm = n5 * 0.61237243569579452 * sth * sth; }  // sqrt(6)/4 sin^2
            else { fp = -n5 * sth * s2; fm = n5 * sth * c2; }
        }
    }
    // common scale from the larger chain
    double big = fmax(fabs(fp), fabs(fm)) * fabs(mant);
    int eb = ex;
    if (big == 0.0) { vp = vm = 0.0; sc = 0; return; }
    renorm(big, eb);  // true magnitude ~ 2^eb
    int shift;
    if (eb >= GS_SC_LO) { sc = 0; shift = ex; }
    else { sc = (GS_SC_LO - eb + GS_SC_K - 1) / GS_SC_K; shift = ex + GS_SC_K * sc; }
    // mant in [0.25,1], factors plain doubles: apply 2^shift in two halves to stay in range
    int h1 = shift / 2, h2 = shift - h1;
    vp = (mant * pow2i(h1)) * fp * pow2i(h2);
    vm = (mant * pow2i(h1)) * fm * pow2i(h2);
}

#define RESCALE_THR 0x1p-644   // 2^(GS_SC_LO + GS_SC_K)
#define RESCALE_MUL 0x1p-256

template <int SPIN>
struct RingState {
    double x;
    double pc, pp;  // mu^+ current / previous
    double mc, mp;  // mu^- current / previous (spin 2)
    int sc;
};

// one recurrence step with coefficients (a, b): (pc,pp) <- (new, pc)
template <int SPIN>
__device__ __forceinline__ void rec_step(RingState<SPIN>& s, double a, double b)
{
    if (SPIN == 0) {
        double t = a * s.x;
        double n = fma(t, s.pc, -s.pp);
        s.pp = s.pc; s.pc = n;
    } else {
        double tp = fma(a, s.x, b), tm = fma(a, s.x, -b);
        double np = fma(tp, s.pc, -s.pp), nm = fma(tm, s.mc, -s.mp);
        s.pp = s.pc; s.pc = np; s.mp = s.mc; s.mc = nm;
    }
}

template <int SPIN>
__device__ __forceinline__ void rescale_check(RingState<SPIN>& s)
{
    if (s.sc > 0) {
        bool big = fabs(s.pc) > RESCALE_THR;
        if (SPIN) big = big || fabs(s.mc) > RESCALE_THR;
        if (big) {
            s.pc *= RESCALE_MUL; s.pp *= RESCALE_MUL;
            if (SPIN) { s.mc *= RESCALE_MUL; s.mp *= RESCALE_MUL; }
            s.sc--;
        }
    }
}

// lambda still negligible on this ring: range-extension scale pending, or both chains below 2^LEG_SMALL_EXP.  libsharp starts to
// accumulate a ring once |lambda| passes sharp_ftol = 2^-60 (sharp_core_inc.c, iter_to_ieee): on the evanescent side of
// l ~ m / sin(theta) lambda_lm grows by orders of magnitude per few multipoles, and a term below 2^-60 of the largest one cannot
// reach the last bit of the sum.  The chains here are mu = lambda / alpha_l with alpha_l = O(1..1e-2), and the threshold is kept
// 2^90 below libsharp's; the test is an integer compare of the exponent field (no FP64 instruction).
// Between two looks (LEG_CHK pairs of l = 8 multipoles) a chain grows by at most ~2^35 (the ratio mu_{l+1} / mu_l is about
// a_l cos(theta) <= sqrt(2 m / (l - m)) right after l = m and falls to ~2 quickly), so a ring that was below 2^-150 at the last
// look has not passed 2^-115 before the next one.  Measured effect at NSIDE 512: 1-3 % of a single-chain transform, 4 % of a
// chain batch (the skipped accumulations are the larger share there).
#ifndef LEG_SMALL_EXP
#define LEG_SMALL_EXP (-150)
#endif
template <int SPIN>
__device__ __forceinline__ bool ring_dead(const RingState<SPIN>& s)
{
    constexpr int thr = (1023 + LEG_SMALL_EXP) << 20;
    bool small = (__double2hiint(s.pc) & 0x7fffffff) < thr;
    if (SPIN) small = small && (__double2hiint(s.mc) & 0x7fffffff) < thr;
    return s.sc > 0 || small;
}

// ------------------------------------------------------------------ staging of one l-tile
// Each thread fetches the (pre-scaled) a_lm pair and the recurrence coefficients of ONE l of the tile into
// registers (LEG_TL == LEG_NT); the values are stored to the other half of a double-buffered shared-memory
// tile after the current tile has been consumed, so the global-memory latency hides behind the recurrence.
template <int SPIN, bool WITH_R = true>
__device__ __forceinline__ void fetch_alm(const PlanDev& P, int m, int l, int64_t base, int64_t roff, const double* almE, const double* almB,
                                          int layout, const double* fl, const double* flB, double2& e, double2& b, double2& r)
{
    const int L = P.lmax;
    e = make_double2(0.0, 0.0); b = e; if (WITH_R) r = e;
    if (l <= L) {
        const int64_t id = base + l;
        double pre = SPIN ? -0.5 * P.alpha2[id] : P.alpha0[id];
        double preb = pre;
        if (fl) pre *= fl[l];
        if (flB) preb *= flB[l]; else preb = pre;
        if (layout == GS_ALM_COMPLEX) {
            e = reinterpret_cast<const double2*>(almE)[id];
            if (SPIN) b = reinterpret_cast<const double2*>(almB)[id];
        } else if (m == 0) {
            e.x = almE[roff + l];
            if (SPIN) b.x = almB[roff + l];
        } else {
            const int64_t off = roff + 2 * l;
            pre *= 0.70710678118654752440;
            preb *= 0.70710678118654752440;
            e.x = almE[off]; e.y = almE[off + 1];
            if (SPIN) { b.x = almB[off]; b.y = almB[off + 1]; }
        }
        e.x *= pre; e.y *= pre; b.x *= preb; b.y *= preb;
        if (SPIN) {
            // lambda^+- basis: Q_m = sum l+ (E' + iB') + l- (E' - iB'), U_m = -i [l+ (E' + iB') - l- (E' - iB')]
            // -> c1 = E'r - B'i, c2 = E'r + B'i, c3 = E'i + B'r, c4 = E'i - B'r
            const double2 c12 = make_double2(e.x - b.y, e.x + b.y), c34 = make_double2(e.y + b.x, e.y - b.x);
            e = c12; b = c34;
            if (WITH_R) r = P.rec2[id];
        } else if (WITH_R) r.x = P.rec0[id];
    }
}
// the same for the NC right-hand sides of a chain batch (chain c at almE/almB + c alm_stride): one set of recurrence coefficients
template <int SPIN, int NC>
__device__ __forceinline__ void fetch_alm_nc(const PlanDev& P, int m, int l, int64_t base, int64_t roff, const double* almE, const double* almB,
                                             int64_t alm_stride, int layout, const double* fl, const double* flB, double2 (&e)[NC], double2 (&b)[NC],
                                             double2& r)
{
    fetch_alm<SPIN, true>(P, m, l, base, roff, almE, almB, layout, fl, flB, e[0], b[0], r);
#pragma unroll
    for (int c = 1; c < NC; ++c) {
        double2 dummy;
        fetch_alm<SPIN, false>(P, m, l, base, roff, almE + c * alm_stride, SPIN ? almB + c * alm_stride : almB, layout, fl, flB, e[c], b[c], dummy);
    }
}

// Position of F_m(ring) of component comp in the ring-spectra buffer.  Unsharded: [comp][ring][m].
// Sharded (SH): [block of mk][peer = owner of the ring][comp][ring_loc][mk within the block], mk = index of m in this rank's m list.
template <bool SH>
__device__ __forceinline__ int64_t fm_index(const PlanDev& P, int comp, int ring, int m, int mk)
{
    if (SH) {
        const int blk = mk / P.sh.MLb, w = mk - blk * P.sh.MLb;
        return ((((int64_t)blk * P.sh.world + P.sh.ring_owner[ring]) * 2 + comp) * P.sh.RL + P.sh.ring_loc[ring]) * P.sh.MLb + w;
    }
    return ((int64_t)comp * P.nring + ring) * (P.lmax + 1) + m;
}
// offset such that entry (l, m) of the real layout sits at roff + (m ? 2 : 1) * l
template <bool SH>
__device__ __forceinline__ int64_t real_off(const PlanDev& P, int m, int mk, int64_t base)
{
    if (SH) return P.sh.rbase[mk] - (m ? 2 : 1) * (int64_t)m;
    return m ? 2 * base - (P.lmax + 1) : 0;
}

// ------------------------------------------------------------------ synthesis
template <int SPIN>
struct SynthAcc {
    // spin 0: (sqr,sqi) first-l-parity part, (aqr,aqi) other parity.
    // spin 2: north sums x1..x4 = sum l+ c1, l- c2, l+ c3, l- c4 ; south sums z1..z4 = sum s (l- c1, l+ c2, l- c3, l+ c4),
    //         s = +-1 alternating with l (lam^+-(pi - theta) = (-1)^(l+m) lam^-+(theta)); Q, U follow from
    //         Qr = 1+2, Qi = 3+4, Ur = 3-4, Ui = 2-1: 8 FMAs per l serve both hemispheres, no F1/F2 adds.
    double sqr, sqi, aqr, aqi;
    double sur, sui, aur, aui;
};

// accumulate one l; FIRST = same parity as the first l of this m
template <int SPIN, bool FIRST>
__device__ __forceinline__ void synth_acc(SynthAcc<SPIN>& A, double pc, double mc, double2 e, double2 b)
{
    if (SPIN == 0) {
        if (FIRST) { A.sqr = fma(e.x, pc, A.sqr); A.sqi = fma(e.y, pc, A.sqi); }
        else       { A.aqr = fma(e.x, pc, A.aqr); A.aqi = fma(e.y, pc, A.aqi); }
    } else {
        // e = (c1, c2), b = (c3, c4); north: sqr=x1 sqi=x2 sur=x3 sui=x4 ; south: aqr=z1 aqi=z2 aur=z3 aui=z4
        A.sqr = fma(pc, e.x, A.sqr); A.sqi = fma(mc, e.y, A.sqi);
        A.sur = fma(pc, b.x, A.sur); A.sui = fma(mc, b.y, A.sui);
        if (FIRST) {
            A.aqr = fma(mc, e.x, A.aqr); A.aqi = fma(pc, e.y, A.aqi);
            A.aur = fma(mc, b.x, A.aur); A.aui = fma(pc, b.y, A.aui);
        } else {
            A.aqr = fma(-mc, e.x, A.aqr); A.aqi = fma(-pc, e.y, A.aqi);
            A.aur = fma(-mc, b.x, A.aur); A.aui = fma(-pc, b.y, A.aui);
        }
    }
}

// NC > 1: chain batch.  NC right-hand sides (chain c: alm at + c alm_stride, spectra at + c fm_stride) share ONE recurrence per
// (ring pair, m) thread: 4 + 8 NC DFMA per ring pair and l instead of 12 NC (BASELINE config #5, north_star (a)).
template <int SPIN, int R, bool SH, int NC>
__global__ void LEG_SYNTH_BOUNDS
leg_synth_kernel(PlanDev P, const double* __restrict__ almE, const double* __restrict__ almB, int layout,
                 const double* __restrict__ fl, const double* __restrict__ flB, double2* __restrict__ Fm,
                 const int* __restrict__ skip, const int* __restrict__ plist, const int* __restrict__ pcount,
                 const int* __restrict__ slot0, int64_t alm_stride, int64_t fm_stride, int mk0)
{
    if (skip && *skip) return;
    const int L = P.lmax, mk = blockIdx.y + mk0, m = SH ? P.sh.mlist[mk] : mk, tid = threadIdx.x;   // mk0: first m of this launch (block-wise sharded pipeline)
    // Ring pairs run from the pole to the equator and lambda_lm is negligible on the pairs before slot0[m] (m > m_lim), so
    // for this m the grid packs the pairs from slot0[m] on: the k-th slot works on pair slot0[m] + k, or on
    // plist[slot0[m] + k] when a compacted list of the pairs with non-zero pixel weight is given (gs_active_rings_build);
    // the blocks beyond the last slot have nothing to do.
    const int s0 = slot0[m], nact = (plist ? *pcount : P.npair) - s0;
    if ((int)blockIdx.x * (LEG_NT * R) >= nact) return;
    __shared__ double2 sEb[2][NC][LEG_TLS], sBb[2][SPIN ? NC : 1][SPIN ? LEG_TLS : 1], sRb[2][LEG_TLS];
    const int l0 = m > SPIN ? m : SPIN;
    const int64_t base = (int64_t)m * (2 * L + 1 - m) / 2;
    const int64_t roff = real_off<SH>(P, m, mk, base);
    const int chunk = blockIdx.x * (LEG_NT * R);

    RingState<SPIN> st[R];
    SynthAcc<SPIN> acc[R][NC];
    int pj[R];
    bool any_act = false;
    unsigned myact = 0;   // bit j: ring pair j of this thread reaches m
#pragma unroll
    for (int j = 0; j < R; ++j) {
        const int k = chunk + ((tid >> 5) * R + j) * 32 + (tid & 31);   // warp-major: a warp owns 32 R consecutive pairs, so idle slots fill whole warps
        const int p = k < nact ? (plist ? plist[s0 + k] : s0 + k) : -1;
        pj[j] = p;
        st[j].x = 0.0; st[j].pc = st[j].pp = st[j].mc = st[j].mp = 0.0; st[j].sc = 0;
#pragma unroll
        for (int c = 0; c < NC; ++c) {
            acc[j][c].sqr = acc[j][c].sqi = acc[j][c].aqr = acc[j][c].aqi = 0.0;
            acc[j][c].sur = acc[j][c].sui = acc[j][c].aur = acc[j][c].aui = 0.0;
        }
        if (p >= 0 && m <= (SPIN ? P.mlim2[p] : P.mlim0[p])) {
            st[j].x = P.cth[p];
            seed_ring<SPIN>(P, p, m, st[j].pc, st[j].mc, st[j].sc);
            any_act = true;
            myact |= 1u << j;
        }
    }
    const bool warp_act = __any_sync(FULL, any_act);
    unsigned gact = 0;          // 32-ring groups of this warp that hold at least one ring reaching this m
#pragma unroll
    for (int j = 0; j < R; ++j) if (__any_sync(FULL, (myact >> j) & 1u)) gact |= 1u << j;
    bool all_live = false;      // set once every group accumulates and no range-extension scale is pending: fast loop from then on

#pragma unroll
    for (int u = 0; u < LEG_SU; ++u) {
        double2 e[NC], b[NC], r;
        fetch_alm_nc<SPIN, NC>(P, m, l0 + u * LEG_NT + tid, base, roff, almE, almB, alm_stride, layout, fl, flB, e, b, r);
#pragma unroll
        for (int c = 0; c < NC; ++c) { sEb[0][c][u * LEG_NT + tid] = e[c]; if (SPIN) sBb[0][c][u * LEG_NT + tid] = b[c]; }
        sRb[0][u * LEG_NT + tid] = r;
    }
    __syncthreads();
    int cur = 0;
    for (int lt = l0; lt <= L; lt += LEG_TLS, cur ^= 1) {
        const bool has_next = lt + LEG_TLS <= L;
        double2 ne[LEG_SU][NC], nb[LEG_SU][NC], nr[LEG_SU];
        if (has_next) {
#pragma unroll
            for (int u = 0; u < LEG_SU; ++u)
                fetch_alm_nc<SPIN, NC>(P, m, lt + LEG_TLS + u * LEG_NT + tid, base, roff, almE, almB, alm_stride, layout, fl, flB, ne[u], nb[u], nr[u]);
        }
        const double2 (*sE)[LEG_TLS] = sEb[cur];
        const double2 (*sB)[SPIN ? LEG_TLS : 1] = sBb[cur];
        const double2* sR = sRb[cur];
        const int ni = warp_act ? min(LEG_TLS, L - lt + 1) : 0;
        const int npr = (ni + 1) >> 1;
        int ip = 0;
        // (A/B) until every 32-ring group of the warp accumulates.  Groups come alive one after the other, equator side (high j)
        // first.  Every LEG_CHK pairs of l the warp finds the lowest group with a ring that is no longer negligible (ring_dead)
        // and runs the next pairs with the groups below it on the recurrence only (4 instead of 12 DFMA per ring pair and l;
        // no checks inside).  Lanes with a pending range-extension scale (seeds below 2^-644) take the checked path pair by pair.
        while (ip < npr && !all_live) {
            bool anys = false;
#pragma unroll
            for (int j = 0; j < R; ++j) anys = anys || st[j].sc > 0;
            if (__any_sync(FULL, anys)) {
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const int i = 2 * ip + h;
                    const double2 r = sR[i];
                    double2 e[NC], b[NC];
#pragma unroll
                    for (int c = 0; c < NC; ++c) { e[c] = sE[c][i]; b[c] = SPIN ? sB[c][i] : e[c]; }
#pragma unroll
                    for (int j = 0; j < R; ++j) {
                        const double pc = st[j].sc ? 0.0 : st[j].pc, mc = st[j].sc ? 0.0 : st[j].mc;
#pragma unroll
                        for (int c = 0; c < NC; ++c) {
                            if (h == 0) synth_acc<SPIN, true>(acc[j][c], pc, mc, e[c], b[c]);
                            else synth_acc<SPIN, false>(acc[j][c], pc, mc, e[c], b[c]);
                        }
                        rec_step<SPIN>(st[j], r.x, r.y);
                        rescale_check<SPIN>(st[j]);
                    }
                }
                ++ip;
                continue;
            }
            int jlo = R;
#pragma unroll
            for (int j = R - 1; j >= 0; --j)
                if (((gact >> j) & 1u) && __any_sync(FULL, !ring_dead<SPIN>(st[j]))) jlo = j;
            if (jlo == 0) { all_live = true; break; }
            const int ipe = min(npr, ip + LEG_CHK);
            auto run = [&](auto JLO) {
                constexpr int J0 = decltype(JLO)::value;
                for (; ip < ipe; ++ip) {
                    const int i = 2 * ip;
                    const double2 r0 = sR[i], r1 = sR[i + 1];
                    double2 e0[NC], b0[NC], e1[NC], b1[NC];
                    if (J0 < R) {
#pragma unroll
                        for (int c = 0; c < NC; ++c) {
                            e0[c] = sE[c][i]; e1[c] = sE[c][i + 1];
                            b0[c] = SPIN ? sB[c][i] : e0[c]; b1[c] = SPIN ? sB[c][i + 1] : e1[c];
                        }
                    }
#pragma unroll
                    for (int j = 0; j < R; ++j) {
                        if (j >= J0) {
#pragma unroll
                            for (int c = 0; c < NC; ++c) synth_acc<SPIN, true>(acc[j][c], st[j].pc, st[j].mc, e0[c], b0[c]);
                        }
                        rec_step<SPIN>(st[j], r0.x, r0.y);
                        if (j >= J0) {
#pragma unroll
                            for (int c = 0; c < NC; ++c) synth_acc<SPIN, false>(acc[j][c], st[j].pc, st[j].mc, e1[c], b1[c]);
                        }
                        rec_step<SPIN>(st[j], r1.x, r1.y);
                    }
                }
            };
            if (R >= 4 && jlo == 3) run(std::integral_constant<int, (R >= 4 ? 3 : R)>());
            else if (R >= 3 && jlo == 2) run(std::integral_constant<int, (R >= 3 ? 2 : R)>());
            else if (R >= 2 && jlo == 1) run(std::integral_constant<int, (R >= 2 ? 1 : R)>());
            else run(std::integral_constant<int, R>());
        }
        // (C) fast path
#pragma unroll 2
        for (; ip < npr; ++ip) {
            const int i = 2 * ip;
            const double2 r0 = sR[i], r1 = sR[i + 1];
            double2 e0[NC], b0[NC], e1[NC], b1[NC];
#pragma unroll
            for (int c = 0; c < NC; ++c) {
                e0[c] = sE[c][i]; e1[c] = sE[c][i + 1];
                b0[c] = SPIN ? sB[c][i] : e0[c]; b1[c] = SPIN ? sB[c][i + 1] : e1[c];
            }
#pragma unroll
            for (int j = 0; j < R; ++j) {
#pragma unroll
                for (int c = 0; c < NC; ++c) synth_acc<SPIN, true>(acc[j][c], st[j].pc, st[j].mc, e0[c], b0[c]);
                rec_step<SPIN>(st[j], r0.x, r0.y);
#pragma unroll
                for (int c = 0; c < NC; ++c) synth_acc<SPIN, false>(acc[j][c], st[j].pc, st[j].mc, e1[c], b1[c]);
                rec_step<SPIN>(st[j], r1.x, r1.y);
            }
        }
        if (has_next) {
#pragma unroll
            for (int u = 0; u < LEG_SU; ++u) {
#pragma unroll
                for (int c = 0; c < NC; ++c) { sEb[cur ^ 1][c][u * LEG_NT + tid] = ne[u][c]; if (SPIN) sBb[cur ^ 1][c][u * LEG_NT + tid] = nb[u][c]; }
                sRb[cur ^ 1][u * LEG_NT + tid] = nr[u];
            }
        }
        __syncthreads();
    }

    // spin 0: north = S + A, south = +-(S - A); spin 2: combine the lambda^+- sums; the south sign follows the
    // parity of the first l
    const double sg = ((l0 + m) & 1) ? -1.0 : 1.0;
#pragma unroll
    for (int j = 0; j < R; ++j) {
        const int p = pj[j];
        if (p < 0) continue;
        const int rn = p, rs = P.nring - 1 - p;
        const int64_t in = fm_index<SH>(P, 0, rn, m, mk), is = fm_index<SH>(P, 0, rs, m, mk);
#pragma unroll
        for (int c = 0; c < NC; ++c) {
            const SynthAcc<SPIN>& a = acc[j][c];
            double2* F = Fm + c * fm_stride;
            if (SPIN == 0) {
                F[in] = make_double2(a.sqr + a.aqr, a.sqi + a.aqi);
                if (rs != rn) F[is] = make_double2(sg * (a.sqr - a.aqr), sg * (a.sqi - a.aqi));
            } else {
                const int64_t cs = SH ? (int64_t)P.sh.RL * P.sh.MLb : (int64_t)P.nring * (L + 1);  // component stride
                F[in] = make_double2(a.sqr + a.sqi, a.sur + a.sui);
                F[in + cs] = make_double2(a.sur - a.sui, a.sqi - a.sqr);
                if (rs != rn) {
                    F[is] = make_double2(sg * (a.aqr + a.aqi), sg * (a.aur + a.aui));
                    F[is + cs] = make_double2(sg * (a.aur - a.aui), sg * (a.aqi - a.aqr));
                }
            }
        }
    }
}

// ------------------------------------------------------------------ block-batched synthesis (Metropolis-within-Gibbs sweep)
// The non-centred likelihood is linear in the synthesised field, so the map change of Metropolis block k is
//   dM_k = A (dfl_k (.) s),  dfl_k[l] = b_l (sqrt(C'_l) - sqrt(C_l)) on the multipoles of block k, 0 elsewhere
// (NonCenteredGibbs.py:333-355, 421-442; SURVEY.md 8f row 1).  The blocks of one spectrum partition the l axis, so ONE
// pass of the recurrence serves every block: E and B contributions are accumulated separately and flushed to the
// block's own ring-spectra slot whenever l crosses a block boundary.  lbE / lbB hold the block boundaries in l
// (block i = [lb[i], lb[i+1])); this launch covers E blocks [e0, e1) -> slots 0.., B blocks [b0, b1) -> slots (e1-e0)..;
// a slot is [nring][L+1][2] double2 (Q and U of one (ring, m) adjacent: every store completes a 32-byte sector, the
// [comp][ring][m] layout cost a DRAM fill read per half-written sector) and receives m < lb[i+1] only (the ring stage is
// told mmax per slot).
template <int R, bool DO_E, bool DO_B>
__global__ void __launch_bounds__(LEG_NT)
leg_synth_blocks_kernel(PlanDev P, const double* __restrict__ almE, const double* __restrict__ almB, const double* __restrict__ dflE,
                        const double* __restrict__ dflB, const int* __restrict__ lbE, int e0, int e1, const int* __restrict__ lbB,
                        int b0, int b1, int lend, double2* __restrict__ Fblk)
{
    // per-l staging of one tile: e = (E'r, E'i), b = (B'r, B'i), their copies times (-1)^(l+m) for the southern ring
    // (lam^+-(pi - theta) = (-1)^(l+m) lam^-+(theta)), and the recurrence coefficients
    __shared__ double2 sE[LEG_TL], sB[LEG_TL], sSE[LEG_TL], sSB[LEG_TL], sR[LEG_TL];
    extern __shared__ unsigned char sflag[];   // [2][L+2]: an E / a B block of this launch ends after multipole l
    const int L = P.lmax, m = blockIdx.y, tid = threadIdx.x;
    const int l0 = m > 2 ? m : 2;
    if (l0 >= lend) return;
    // ring pairs that reach this m, packed (see leg_synth_kernel); the ring stage reads a ring up to its m_lim only
    const int s0 = P.pmin2[m], nact = P.npair - s0;
    const int chunk = blockIdx.x * (LEG_NT * R);
    if (chunk >= nact) return;
    unsigned char* sfE = sflag;
    unsigned char* sfB = sflag + (L + 2);
    for (int i = tid; i < 2 * (L + 2); i += LEG_NT) sflag[i] = 0;
    __syncthreads();
    if (DO_E) for (int i = e0 + tid; i < e1; i += LEG_NT) { const int end = lbE[i + 1]; if (end >= 1 && end <= L + 1) sfE[end - 1] = 1; }
    if (DO_B) for (int i = b0 + tid; i < b1; i += LEG_NT) { const int end = lbB[i + 1]; if (end >= 1 && end <= L + 1) sfB[end - 1] = 1; }
    const int64_t base = (int64_t)m * (2 * L + 1 - m) / 2;
    const int64_t roff = real_off<false>(P, m, m, base);
    const int64_t nm = L + 1, cs = (int64_t)P.nring * nm, slot = 2 * cs;

    RingState<2> st[R];
    double aE[R][DO_E ? 8 : 1], aB[R][DO_B ? 8 : 1];
    int pj[R];
    bool any_act = false, all_plain = true;
#pragma unroll
    for (int j = 0; j < R; ++j) {
        const int k = chunk + ((tid >> 5) * R + j) * 32 + (tid & 31);
        const int p = k < nact ? s0 + k : -1;
        pj[j] = p;
        st[j].x = 0.0; st[j].pc = st[j].pp = st[j].mc = st[j].mp = 0.0; st[j].sc = 0;
#pragma unroll
        for (int q = 0; q < (DO_E ? 8 : 1); ++q) aE[j][q] = 0.0;
#pragma unroll
        for (int q = 0; q < (DO_B ? 8 : 1); ++q) aB[j][q] = 0.0;
        if (p >= 0 && m <= P.mlim2[p]) {
            st[j].x = P.cth[p];
            seed_ring<2>(P, p, m, st[j].pc, st[j].mc, st[j].sc);
            any_act = true;
            all_plain = all_plain && st[j].sc == 0;
        }
    }
    const bool warp_act = __any_sync(FULL, any_act);
    bool fast = __all_sync(FULL, all_plain);   // no ring of the warp carries a range-extension scale (any more)
    // blocks that end at or below the first multipole of this m receive nothing from it
    int iE = e0, iB = b0;
    if (DO_E) while (iE < e1 && lbE[iE + 1] <= l0) ++iE;
    if (DO_B) while (iB < b1 && lbB[iB + 1] <= l0) ++iB;
    // multipoles below the first block of this launch belong to blocks of another group: their sums are discarded
    const int startE = (DO_E && e1 > e0) ? lbE[e0] : -1, startB = (DO_B && b1 > b0) ? lbB[b0] : -1;

    for (int lt = l0; lt < lend; lt += LEG_TL) {
        __syncthreads();
        {
            const int l = lt + tid;
            double2 e = make_double2(0.0, 0.0), b = e, r = e;
            double sg = 1.0;
            if (l <= L) {
                const int64_t id = base + l;
                double pre = -0.5 * P.alpha2[id];
                if (m == 0) { e.x = almE[roff + l]; b.x = almB[roff + l]; }
                else {
                    const int64_t off = roff + 2 * l;
                    pre *= 0.70710678118654752440;
                    e = make_double2(almE[off], almE[off + 1]);
                    b = make_double2(almB[off], almB[off + 1]);
                }
                const double pe = pre * dflE[l], pb = pre * dflB[l];
                e.x *= pe; e.y *= pe; b.x *= pb; b.y *= pb;
                r = P.rec2[id];
                sg = ((l + m) & 1) ? -1.0 : 1.0;
            }
            sE[tid] = e; sB[tid] = b; sR[tid] = r;
            sSE[tid] = make_double2(sg * e.x, sg * e.y);
            sSB[tid] = make_double2(sg * b.x, sg * b.y);
        }
        __syncthreads();
        if (!warp_act) continue;
        const int ni = min(LEG_TL, lend - lt);
        for (int i = 0; i < ni; ++i) {
            const int l = lt + i;
            if (DO_E && l == startE) {
#pragma unroll
                for (int j = 0; j < R; ++j)
#pragma unroll
                    for (int q = 0; q < 8; ++q) aE[j][q] = 0.0;
            }
            if (DO_B && l == startB) {
#pragma unroll
                for (int j = 0; j < R; ++j)
#pragma unroll
                    for (int q = 0; q < 8; ++q) aB[j][q] = 0.0;
            }
            const double2 r = sR[i], e = sE[i], b = sB[i], se = sSE[i], sb = sSB[i];
#pragma unroll
            for (int j = 0; j < R; ++j) {
                const double pc = (fast || st[j].sc == 0) ? st[j].pc : 0.0, mc = (fast || st[j].sc == 0) ? st[j].mc : 0.0;
                if (DO_E) {   // E only: c1 = c2 = E'r, c3 = c4 = E'i
                    aE[j][0] = fma(pc, e.x, aE[j][0]); aE[j][1] = fma(mc, e.x, aE[j][1]);
                    aE[j][2] = fma(pc, e.y, aE[j][2]); aE[j][3] = fma(mc, e.y, aE[j][3]);
                    aE[j][4] = fma(mc, se.x, aE[j][4]); aE[j][5] = fma(pc, se.x, aE[j][5]);
                    aE[j][6] = fma(mc, se.y, aE[j][6]); aE[j][7] = fma(pc, se.y, aE[j][7]);
                }
                if (DO_B) {   // B only: c1 = -B'i, c2 = B'i, c3 = B'r, c4 = -B'r
                    aB[j][0] = fma(-pc, b.y, aB[j][0]); aB[j][1] = fma(mc, b.y, aB[j][1]);
                    aB[j][2] = fma(pc, b.x, aB[j][2]); aB[j][3] = fma(-mc, b.x, aB[j][3]);
                    aB[j][4] = fma(-mc, sb.y, aB[j][4]); aB[j][5] = fma(pc, sb.y, aB[j][5]);
                    aB[j][6] = fma(mc, sb.x, aB[j][6]); aB[j][7] = fma(-pc, sb.x, aB[j][7]);
                }
                rec_step<2>(st[j], r.x, r.y);
                if (!fast) rescale_check<2>(st[j]);
            }
            if (!fast) {
                bool plain = true;
#pragma unroll
                for (int j = 0; j < R; ++j) plain = plain && st[j].sc == 0;
                fast = __all_sync(FULL, plain);
            }
            // flush the block(s) that end after l
            if (DO_E && sfE[l]) {
                double2* F = Fblk + (int64_t)(iE - e0) * slot;
#pragma unroll
                for (int j = 0; j < R; ++j) {
                    const int p = pj[j];
                    double* a = aE[j];
                    if (p >= 0) {
                        const int rn = p, rs = P.nring - 1 - p;
                        double2* fn = F + ((int64_t)rn * nm + m) * 2;   // [ring][m][comp]: Q and U fill one 32-byte sector
                        fn[0] = make_double2(a[0] + a[1], a[2] + a[3]);
                        fn[1] = make_double2(a[2] - a[3], a[1] - a[0]);
                        if (rs != rn) {
                            double2* fsn = F + ((int64_t)rs * nm + m) * 2;
                            fsn[0] = make_double2(a[4] + a[5], a[6] + a[7]);
                            fsn[1] = make_double2(a[6] - a[7], a[5] - a[4]);
                        }
                    }
#pragma unroll
                    for (int q = 0; q < 8; ++q) a[q] = 0.0;
                }
                ++iE;
            }
            if (DO_B && sfB[l]) {
                double2* F = Fblk + (int64_t)((e1 - e0) + (iB - b0)) * slot;
#pragma unroll
                for (int j = 0; j < R; ++j) {
                    const int p = pj[j];
                    double* a = aB[j];
                    if (p >= 0) {
                        const int rn = p, rs = P.nring - 1 - p;
                        double2* fn = F + ((int64_t)rn * nm + m) * 2;   // [ring][m][comp]: Q and U fill one 32-byte sector
                        fn[0] = make_double2(a[0] + a[1], a[2] + a[3]);
                        fn[1] = make_double2(a[2] - a[3], a[1] - a[0]);
                        if (rs != rn) {
                            double2* fsn = F + ((int64_t)rs * nm + m) * 2;
                            fsn[0] = make_double2(a[4] + a[5], a[6] + a[7]);
                            fsn[1] = make_double2(a[6] - a[7], a[5] - a[4]);
                        }
                    }
#pragma unroll
                    for (int q = 0; q < 8; ++q) a[q] = 0.0;
                }
                ++iB;
            }
        }
    }
}

// ------------------------------------------------------------------ analysis
template <int SPIN>
struct AnalIn {
    // spin 0: (q1r,q1i) ring spectrum combined for the first-l parity, (q2r,q2i) for the other one.
    // spin 2 (lambda^+- basis): k1 = Gq.r - Gu.i, k2 = Gq.r + Gu.i, k3 = Gq.i + Gu.r, k4 = Gq.i - Gu.r of the
    //         north ring (q1r,q1i,q2r,q2i) and of the south ring (u1r,u1i,u2r,u2i; sign of the first l folded in).
    double q1r, q1i, q2r, q2i;
    double u1r, u1i, u2r, u2i;
};

// contributions of one ring pair at one l: spin 0 -> (re, im); spin 2 -> (Y1..Y4) with
//   Y1 = l+ k1n + s l- k1s, Y2 = l- k2n + s l+ k2s, Y3 = l+ k3n + s l- k3s, Y4 = l- k4n + s l+ k4s
// (E.re = Y1+Y2, E.im = Y3+Y4, B.re = Y3-Y4, B.im = Y2-Y1 are formed once per (l,m) in the finish kernel)
// Spin 2 is accumulated in a lane-permuted form.  With X = (k1n, k2s, k3n, k4s) (multiplied by lam^+) and
// Y = (k1s, k2n, k3s, k4n) (by lam^-),
//   first-parity l:  Y_c = lam^+ X_c + lam^- Y_c,   other parity:  Y_c = s_c (lam^+ X_c - lam^- Y_c),  s = (+,-,+,-),
// every slot has the same instruction pattern, so a lane may hold value c = slot ^ pi in slot `slot` for any lane constant pi
// by permuting its X, Y once.  pi = (lane bit 4, lane bit 3) makes the first two exchange stages of the reduce-scatter
// (which move half and a quarter of the values) select-free: every lane keeps the low slots and sends the high ones.
// The sign s_c is applied by the lane that ends up owning the value (flipmask in leg_anal_kernel).
template <int SPIN, bool FIRST, bool INIT>
__device__ __forceinline__ void anal_acc(double* o, const AnalIn<SPIN>& G, double pc, double mc)
{
    if constexpr (SPIN == 0) {
        const double gr = FIRST ? G.q1r : G.q2r, gi = FIRST ? G.q1i : G.q2i;
        o[0] = INIT ? gr * pc : fma(gr, pc, o[0]);
        o[1] = INIT ? gi * pc : fma(gi, pc, o[1]);
    } else {
        if (INIT) { o[0] = pc * G.q1r; o[1] = pc * G.q1i; o[2] = pc * G.q2r; o[3] = pc * G.q2i; }
        else { o[0] = fma(pc, G.q1r, o[0]); o[1] = fma(pc, G.q1i, o[1]); o[2] = fma(pc, G.q2r, o[2]); o[3] = fma(pc, G.q2i, o[3]); }
        if (FIRST) { o[0] = fma(mc, G.u1r, o[0]); o[1] = fma(mc, G.u1i, o[1]); o[2] = fma(mc, G.u2r, o[2]); o[3] = fma(mc, G.u2i, o[3]); }
        else { o[0] = fma(-mc, G.u1r, o[0]); o[1] = fma(-mc, G.u1i, o[1]); o[2] = fma(-mc, G.u2r, o[2]); o[3] = fma(-mc, G.u2i, o[3]); }
    }
}

// reduce-scatter over the warp of the values of a pair of l.
// spin 0, 4 values: afterwards lane holds the full sum of value lane >> 3.
// spin 2, v[0..3]: slots of the first l, v[4..7]: of the second.  Returns the full sum of value (h, c) = (lane bit 2, pi) in
// every lane: 9 SHFL.64, 9 DADD, one select pair.
template <int SPIN>
__device__ __forceinline__ double warp_fold(double* v, int lane)
{
    if constexpr (SPIN == 0) {
        const bool h4 = lane & 16;
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const double keep = h4 ? v[i + 2] : v[i], send = h4 ? v[i] : v[i + 2];
            v[i] = keep + __shfl_xor_sync(FULL, send, 16);
        }
        const bool h3 = lane & 8;
        const double keep = h3 ? v[1] : v[0], send = h3 ? v[0] : v[1];
        double r = keep + __shfl_xor_sync(FULL, send, 8);
        r += __shfl_xor_sync(FULL, r, 4);
        r += __shfl_xor_sync(FULL, r, 2);
        r += __shfl_xor_sync(FULL, r, 1);
        return r;
    } else {
        v[0] += __shfl_xor_sync(FULL, v[2], 16); v[1] += __shfl_xor_sync(FULL, v[3], 16);
        v[4] += __shfl_xor_sync(FULL, v[6], 16); v[5] += __shfl_xor_sync(FULL, v[7], 16);
        v[0] += __shfl_xor_sync(FULL, v[1], 8);
        v[4] += __shfl_xor_sync(FULL, v[5], 8);
        const bool h = lane & 4;
        const double keep = h ? v[4] : v[0], send = h ? v[0] : v[4];
        double r = keep + __shfl_xor_sync(FULL, send, 4);
        r += __shfl_xor_sync(FULL, r, 2);
        r += __shfl_xor_sync(FULL, r, 1);
        return r;
    }
}

#ifndef LEG_MINB_A
#define LEG_MINB_A 3   // 3 CTAs per SM: caps the unrolled fast loop at 168 registers
#endif
#ifndef LEG_RA2
#define LEG_RA2 2      // ring pairs per thread of the chain-batched analysis (NC = 2): R NC = 4 keeps the register budget
#endif
// dynamic shared memory of leg_anal_kernel<SPIN, R, SH, NC>: recurrence tile, per-warp partial sums, parked exchange values
template <int SPIN, int NC>
constexpr size_t leg_anal_smem()
{
    return sizeof(double2) * LEG_TL + sizeof(double) * LEG_NW * NC * LEG_TL * (SPIN ? 4 : 2)
           + (SPIN ? sizeof(double2) * LEG_NW * NC * FOLD3_NB * 32 : 0);
}
// NC > 1: chain batch (see leg_synth_kernel): spectra of chain c at Fm + c fm_stride, partial sums at partial + c part_stride;
// the recurrence of a (ring pair, m) thread is shared, the reduce-scatter runs once per chain.
#ifndef LEG_MINB_A2
#define LEG_MINB_A2 LEG_MINB_A   // same for the chain batch (NC = 2)
#endif
template <int SPIN, int R, bool SH, int NC>
__global__ void __launch_bounds__(LEG_NT, (NC > 1 ? LEG_MINB_A2 : LEG_MINB_A))
leg_anal_kernel(PlanDev P, const double2* __restrict__ Fm, double* __restrict__ partial, const int* __restrict__ skip,
                const int* __restrict__ plist, const int* __restrict__ pcount, const int* __restrict__ slot0, int64_t fm_stride,
                int64_t part_stride, int mk0)
{
    if (skip && *skip) return;
    const int L = P.lmax, mk = blockIdx.y + mk0, m = SH ? P.sh.mlist[mk] : mk, tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    // slots of this m: see leg_synth_kernel; leg_finish_kernel sums the chunks that hold slots only
    const int s0 = slot0[m], nact = (plist ? *pcount : P.npair) - s0;
    if ((int)blockIdx.x * (LEG_NT * R) >= nact) return;
    constexpr int NV = SPIN ? 4 : 2;   // doubles per (l,m)
    constexpr int NVAL = 2 * NV;       // values reduced per pair of l
    extern __shared__ double2 leg_dyn[];
    double2* sR = leg_dyn;                                                  // [LEG_TL]
    double* sPartAll = reinterpret_cast<double*>(leg_dyn + LEG_TL);         // [LEG_NW][NC][LEG_TL * NV]
    auto sPart = [&](int ww, int c) { return sPartAll + ((size_t)(ww * NC + c)) * (LEG_TL * NV); };
    // After the two select-free exchange stages a lane holds, for each of the two l of a pair, the sum over 4 lanes of the
    // value c = (lane bit 4, lane bit 3); what remains is a sum over the 8 lanes that differ in bits 2..0.  Instead of three
    // more dependent shuffle stages per pair of l, the fast loop parks those two numbers in shared memory and sums FOLD3_NB
    // pairs of l at a time (8 independent loads per output, no selects).  Slot of lane L for local pair q:
    // L ^ c(L) ^ ((q & 1) << 2): stores are conflict free and the 32 outputs read in one step hit 16 distinct 8-byte banks.
    double2* sFoldAll = reinterpret_cast<double2*>(sPartAll + (size_t)LEG_NW * NC * LEG_TL * NV);   // [LEG_NW][NC][FOLD3_NB * 32] (spin 2)
    const int l0 = m > SPIN ? m : SPIN;
    const int64_t base = (int64_t)m * (2 * L + 1 - m) / 2;
    // first entry (l = lt) of this block's partial sums is pbase + lt
    const int64_t pbase = SH ? (int64_t)blockIdx.x * P.sh.nalm_loc + P.sh.cbase[mk] - m : (int64_t)blockIdx.x * P.nalm + base;
    const int chunk = blockIdx.x * (LEG_NT * R);
    const bool odd0 = (l0 + m) & 1;
    const int64_t cs = SH ? (int64_t)P.sh.RL * P.sh.MLb : (int64_t)P.nring * (L + 1);  // component stride

    RingState<SPIN> st[R];
    AnalIn<SPIN> G[R][NC];
    bool any_act = false;
    unsigned myact = 0;   // bit j: ring pair j of this thread reaches m
#pragma unroll
    for (int j = 0; j < R; ++j) {
        const int k = chunk + ((tid >> 5) * R + j) * 32 + (tid & 31);   // warp-major: a warp owns 32 R consecutive pairs, so idle slots fill whole warps
        const int p = k < nact ? (plist ? plist[s0 + k] : s0 + k) : -1;
        st[j].x = 0.0; st[j].pc = st[j].pp = st[j].mc = st[j].mp = 0.0; st[j].sc = 0;
#pragma unroll
        for (int c = 0; c < NC; ++c) {
            G[j][c].q1r = G[j][c].q1i = G[j][c].q2r = G[j][c].q2i = 0.0;
            G[j][c].u1r = G[j][c].u1i = G[j][c].u2r = G[j][c].u2i = 0.0;
        }
        if (p >= 0 && m <= (SPIN ? P.mlim2[p] : P.mlim0[p])) {
            st[j].x = P.cth[p];
            seed_ring<SPIN>(P, p, m, st[j].pc, st[j].mc, st[j].sc);
            any_act = true;
            myact |= 1u << j;
            const int rn = p, rs = P.nring - 1 - p;
            const double2 z = make_double2(0.0, 0.0);
            const int64_t in = fm_index<SH>(P, 0, rn, m, mk), is = fm_index<SH>(P, 0, rs, m, mk);
#pragma unroll
            for (int c = 0; c < NC; ++c) {
                const double2* F = Fm + c * fm_stride;
                AnalIn<SPIN>& g = G[j][c];
                const double2 qn = F[in], qs = (rs != rn) ? F[is] : z;
                if (SPIN == 0) {
                    const double2 sy = make_double2(qn.x + qs.x, qn.y + qs.y), an = make_double2(qn.x - qs.x, qn.y - qs.y);
                    g.q1r = odd0 ? an.x : sy.x; g.q1i = odd0 ? an.y : sy.y;
                    g.q2r = odd0 ? sy.x : an.x; g.q2i = odd0 ? sy.y : an.y;
                } else {
                    const double2 un = F[in + cs], us = (rs != rn) ? F[is + cs] : z;
                    const double sg = odd0 ? -1.0 : 1.0;
                    g.q1r = qn.x - un.y; g.q1i = qn.x + un.y; g.q2r = qn.y + un.x; g.q2i = qn.y - un.x;
                    g.u1r = sg * (qs.x - us.y); g.u1i = sg * (qs.x + us.y);
                    g.u2r = sg * (qs.y + us.x); g.u2i = sg * (qs.y - us.x);
                    {   // (q1r,q1i,q2r,q2i) <- X = (k1n, k2s, k3n, k4s), (u1r,u1i,u2r,u2i) <- Y = (k1s, k2n, k3s, k4n), then slot = c ^ pi
                        double t = g.q1i; g.q1i = g.u1i; g.u1i = t;
                        t = g.q2i; g.q2i = g.u2i; g.u2i = t;
                        if (lane & 16) {
                            t = g.q1r; g.q1r = g.q2r; g.q2r = t;  t = g.q1i; g.q1i = g.q2i; g.q2i = t;
                            t = g.u1r; g.u1r = g.u2r; g.u2r = t;  t = g.u1i; g.u1i = g.u2i; g.u2i = t;
                        }
                        if (lane & 8) {
                            t = g.q1r; g.q1r = g.q1i; g.q1i = t;  t = g.q2r; g.q2r = g.q2i; g.q2i = t;
                            t = g.u1r; g.u1r = g.u1i; g.u1i = t;  t = g.u2r; g.u2r = g.u2i; g.u2i = t;
                        }
                    }
                }
            }
        }
    }
    const bool warp_act = __any_sync(FULL, any_act);
    unsigned gact = 0;          // 32-ring groups of this warp that hold at least one ring reaching this m
#pragma unroll
    for (int j = 0; j < R; ++j) if (__any_sync(FULL, (myact >> j) & 1u)) gact |= 1u << j;
    bool all_live = false;      // see leg_synth_kernel
    // spin 2: the lane ends up owning (h, c) = (bit 2, (bit 4, bit 3)); odd c of the second l carries a minus sign
    const int vidx = SPIN ? ((lane & 4) | ((lane >> 3) & 3)) : lane >> 3;
    const int flipmask = (SPIN && (lane & 4) && (lane & 8)) ? (int)0x80000000 : 0;   // sign flip as an integer XOR (no FP64 op)
    const bool writer = (lane & (SPIN ? 3 : 7)) == 0;

    for (int lt = l0; lt <= L; lt += LEG_TL) {
        __syncthreads();
        for (int i = tid; i < LEG_TL; i += LEG_NT) {
            const int l = lt + i;
            double2 r = make_double2(0.0, 0.0);
            if (l <= L) { if (SPIN) r = P.rec2[base + l]; else r.x = P.rec0[base + l]; }
            sR[i] = r;
        }
        __syncthreads();
        const int ni = min(LEG_TL, L - lt + 1);
        const int npr = (ni + 1) >> 1;
        int ip = 0;
        if (!warp_act) {
#pragma unroll
            for (int c = 0; c < NC; ++c) {
                double* mp = sPart(w, c);
                for (int i = lane; i < LEG_TL * NV; i += 32) mp[i] = 0.0;
            }
            ip = npr;
        }
        // (A/B) until every 32-ring group of the warp accumulates: see leg_synth_kernel.  Groups below the lowest live one run the
        // recurrence only; checked every LEG_CHK pairs of l; lanes with a pending range-extension scale go pair by pair.
        while (ip < npr && !all_live) {
            bool anys = false;
#pragma unroll
            for (int j = 0; j < R; ++j) anys = anys || st[j].sc > 0;
            if (__any_sync(FULL, anys)) {
                double v[NC][NVAL];
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const double2 r = sR[2 * ip + h];
#pragma unroll
                    for (int j = 0; j < R; ++j) {
                        const double pc = st[j].sc ? 0.0 : st[j].pc, mc = st[j].sc ? 0.0 : st[j].mc;
#pragma unroll
                        for (int c = 0; c < NC; ++c) {
                            if (h == 0) {
                                if (j == 0) anal_acc<SPIN, true, true>(v[c], G[j][c], pc, mc);
                                else anal_acc<SPIN, true, false>(v[c], G[j][c], pc, mc);
                            } else {
                                if (j == 0) anal_acc<SPIN, false, true>(v[c] + NV, G[j][c], pc, mc);
                                else anal_acc<SPIN, false, false>(v[c] + NV, G[j][c], pc, mc);
                            }
                        }
                        rec_step<SPIN>(st[j], r.x, r.y);
                        rescale_check<SPIN>(st[j]);
                    }
                }
#pragma unroll
                for (int c = 0; c < NC; ++c) {
                    const double s = warp_fold<SPIN>(v[c], lane);
                    if (writer) sPart(w, c)[ip * NVAL + vidx] = __hiloint2double(__double2hiint(s) ^ flipmask, __double2loint(s));
                }
                ++ip;
                continue;
            }
            int jlo = R;
#pragma unroll
            for (int j = R - 1; j >= 0; --j)
                if (((gact >> j) & 1u) && __any_sync(FULL, !ring_dead<SPIN>(st[j]))) jlo = j;
            if (jlo == 0) { all_live = true; break; }
            const int ipe = min(npr, ip + LEG_CHK);
            auto run = [&](auto JLO) {
                constexpr int J0 = decltype(JLO)::value;
                for (; ip < ipe; ++ip) {
                    const double2 r0 = sR[2 * ip], r1 = sR[2 * ip + 1];
                    double v[NC][NVAL];
#pragma unroll
                    for (int j = 0; j < R; ++j) {
                        if (j >= J0) {
#pragma unroll
                            for (int c = 0; c < NC; ++c) {
                                if (j == J0) anal_acc<SPIN, true, true>(v[c], G[j][c], st[j].pc, st[j].mc);
                                else anal_acc<SPIN, true, false>(v[c], G[j][c], st[j].pc, st[j].mc);
                            }
                        }
                        rec_step<SPIN>(st[j], r0.x, r0.y);
                        if (j >= J0) {
#pragma unroll
                            for (int c = 0; c < NC; ++c) {
                                if (j == J0) anal_acc<SPIN, false, true>(v[c] + NV, G[j][c], st[j].pc, st[j].mc);
                                else anal_acc<SPIN, false, false>(v[c] + NV, G[j][c], st[j].pc, st[j].mc);
                            }
                        }
                        rec_step<SPIN>(st[j], r1.x, r1.y);
                    }
                    if (J0 >= R) {   // nothing accumulates yet
                        if (lane < NVAL) {
#pragma unroll
                            for (int c = 0; c < NC; ++c) sPart(w, c)[ip * NVAL + lane] = 0.0;
                        }
                    } else {
#pragma unroll
                        for (int c = 0; c < NC; ++c) {
                            const double s = warp_fold<SPIN>(v[c], lane);
                            if (writer) sPart(w, c)[ip * NVAL + vidx] = __hiloint2double(__double2hiint(s) ^ flipmask, __double2loint(s));
                        }
                    }
                }
            };
            if (R >= 4 && jlo == 3) run(std::integral_constant<int, (R >= 4 ? 3 : R)>());
            else if (R >= 3 && jlo == 2) run(std::integral_constant<int, (R >= 3 ? 2 : R)>());
            else if (R >= 2 && jlo == 1) run(std::integral_constant<int, (R >= 2 ? 1 : R)>());
            else run(std::integral_constant<int, R>());
        }
        if constexpr (SPIN == 2) {
            const int cperm = ((lane >> 4) & 1) << 1 | ((lane >> 3) & 1);
            int ipb = ip;   // first pair of l of the batch parked in the fold buffers
            // sums the parked pairs [ipb, ipb + n) over the 8 lanes of each value and writes them to the warp's partial sums
            auto flush = [&](int n) {
                __syncwarp();
#pragma unroll
                for (int c = 0; c < NC; ++c) {
                    const double2* fbuf = sFoldAll + ((size_t)(w * NC + c)) * (FOLD3_NB * 32);
                    double* myPart = sPart(w, c);
#pragma unroll
                    for (int t = 0; t < FOLD3_NB / 4; ++t) {
                        const int o = lane + 32 * t, q = o >> 3, h = (o >> 2) & 1, cc = o & 3;
                        if (q < n) {
                            const double* e = reinterpret_cast<const double*>(fbuf + q * 32) + h;
                            const int sl0 = (((cc >> 1) << 4) | ((cc & 1) << 3)) ^ cc ^ ((q & 1) << 2);   // slot of source lane (cc, s = 0)
                            double a[8];
#pragma unroll
                            for (int k = 0; k < 8; ++k) a[k] = e[2 * (sl0 ^ k)];   // s ^ (low bits of the swizzle) runs over the same 8 slots
                            double sum = ((a[0] + a[1]) + (a[2] + a[3])) + ((a[4] + a[5]) + (a[6] + a[7]));
                            if (h && (cc & 1)) sum = -sum;
                            myPart[(ipb + q) * NVAL + h * 4 + cc] = sum;
                        }
                    }
                }
                __syncwarp();
            };
#pragma unroll kUnrollA
            for (; ip < npr; ++ip) {  // (C)
                double v[NC][NVAL];
                const double2 r0 = sR[2 * ip], r1 = sR[2 * ip + 1];
#pragma unroll
                for (int j = 0; j < R; ++j) {
#pragma unroll
                    for (int c = 0; c < NC; ++c) {
                        if (j == 0) anal_acc<SPIN, true, true>(v[c], G[j][c], st[j].pc, st[j].mc);
                        else anal_acc<SPIN, true, false>(v[c], G[j][c], st[j].pc, st[j].mc);
                    }
                    rec_step<SPIN>(st[j], r0.x, r0.y);
#pragma unroll
                    for (int c = 0; c < NC; ++c) {
                        if (j == 0) anal_acc<SPIN, false, true>(v[c] + NV, G[j][c], st[j].pc, st[j].mc);
                        else anal_acc<SPIN, false, false>(v[c] + NV, G[j][c], st[j].pc, st[j].mc);
                    }
                    rec_step<SPIN>(st[j], r1.x, r1.y);
                }
                const int q = ip - ipb;
#pragma unroll
                for (int c = 0; c < NC; ++c) {
                    double* vv = v[c];
                    vv[0] += __shfl_xor_sync(FULL, vv[2], 16); vv[1] += __shfl_xor_sync(FULL, vv[3], 16);
                    vv[4] += __shfl_xor_sync(FULL, vv[6], 16); vv[5] += __shfl_xor_sync(FULL, vv[7], 16);
                    vv[0] += __shfl_xor_sync(FULL, vv[1], 8);
                    vv[4] += __shfl_xor_sync(FULL, vv[5], 8);
                    double2* fbuf = sFoldAll + ((size_t)(w * NC + c)) * (FOLD3_NB * 32);
                    fbuf[q * 32 + (lane ^ cperm ^ ((q & 1) << 2))] = make_double2(vv[0], vv[4]);
                }
                if (q == FOLD3_NB - 1) { flush(FOLD3_NB); ipb = ip + 1; }
            }
            if (ip > ipb) flush(ip - ipb);
        } else {
#pragma unroll kUnrollA
            for (; ip < npr; ++ip) {  // (C)
                double v[NC][NVAL];
                const double2 r0 = sR[2 * ip], r1 = sR[2 * ip + 1];
#pragma unroll
                for (int j = 0; j < R; ++j) {
#pragma unroll
                    for (int c = 0; c < NC; ++c) {
                        if (j == 0) anal_acc<SPIN, true, true>(v[c], G[j][c], st[j].pc, st[j].mc);
                        else anal_acc<SPIN, true, false>(v[c], G[j][c], st[j].pc, st[j].mc);
                    }
                    rec_step<SPIN>(st[j], r0.x, r0.y);
#pragma unroll
                    for (int c = 0; c < NC; ++c) {
                        if (j == 0) anal_acc<SPIN, false, true>(v[c] + NV, G[j][c], st[j].pc, st[j].mc);
                        else anal_acc<SPIN, false, false>(v[c] + NV, G[j][c], st[j].pc, st[j].mc);
                    }
                    rec_step<SPIN>(st[j], r1.x, r1.y);
                }
#pragma unroll
                for (int c = 0; c < NC; ++c) {
                    const double s = warp_fold<SPIN>(v[c], lane);
                    if (writer) sPart(w, c)[ip * NVAL + vidx] = __hiloint2double(__double2hiint(s) ^ flipmask, __double2loint(s));
                }
            }
        }
        __syncthreads();
        // sum over the warps of the block, one deterministic partial per chunk
#pragma unroll
        for (int c = 0; c < NC; ++c) {
            double* out = partial + c * part_stride + (pbase + lt) * NV;
            for (int i = tid; i < ni * NV; i += LEG_NT) {
                double s = 0.0;
#pragma unroll
                for (int ww = 0; ww < LEG_NW; ++ww) s += sPart(ww, c)[i];
                out[i] = s;
            }
        }
    }
}

// Combine the per-chunk partials: alm = post(l,m) * sum_chunks, converted to the requested layout.
template <int SPIN, bool SH>
__global__ void leg_finish_kernel(PlanDev P, const double* __restrict__ partial, int nchunk, double* __restrict__ almE,
                                  double* __restrict__ almB, int layout, const double* __restrict__ fl, double scale,
                                  int accumulate, const int* __restrict__ skip, const int* __restrict__ pcount,
                                  const int* __restrict__ slot0, int chunk_pairs, int64_t part_stride, int64_t alm_stride)
{
    if (skip && *skip) return;
    constexpr int NV = SPIN ? 4 : 2;
    const int L = P.lmax, mk = blockIdx.y, m = SH ? P.sh.mlist[mk] : mk;
    // chain batch: blockIdx.z = chain
    partial += blockIdx.z * part_stride;
    almE += blockIdx.z * alm_stride;
    if (SPIN) almB += blockIdx.z * alm_stride;
    {   // chunks of this m that hold slots (the others were not written)
        const int nact = (pcount ? *pcount : P.npair) - slot0[m];
        nchunk = nact > 0 ? (nact + chunk_pairs - 1) / chunk_pairs : 0;
    }
    const int l = m + blockIdx.x * blockDim.x + threadIdx.x;
    if (l > L) return;
    const int64_t base = (int64_t)m * (2 * L + 1 - m) / 2, id = base + l;
    const int64_t pid = SH ? P.sh.cbase[mk] + (l - m) : id, pn = SH ? P.sh.nalm_loc : P.nalm;
    const int64_t roff = real_off<SH>(P, m, mk, base);
    double v[NV];
#pragma unroll
    for (int c = 0; c < NV; ++c) v[c] = 0.0;
    if (l >= SPIN) {
        for (int k = 0; k < nchunk; ++k) {
            const double* q = partial + ((int64_t)k * pn + pid) * NV;
#pragma unroll
            for (int c = 0; c < NV; ++c) v[c] += q[c];
        }
        if (SPIN) {  // E.re = Y1+Y2, E.im = Y3+Y4, B.re = Y3-Y4, B.im = Y2-Y1
            const double y1 = v[0], y2 = v[1], y3 = v[2], y4 = v[3];
            v[0] = y1 + y2; v[1] = y3 + y4; v[2] = y3 - y4; v[3] = y2 - y1;
        }
        double post = scale * (SPIN ? -0.5 * P.alpha2[id] : P.alpha0[id]);
        if (fl) post *= fl[l];
        if (layout == GS_ALM_REAL && m > 0) post *= 1.41421356237309504880;
#pragma unroll
        for (int c = 0; c < NV; ++c) v[c] *= post;
    }
    if (layout == GS_ALM_COMPLEX) {
        double2* E = reinterpret_cast<double2*>(almE);
        double2 e = make_double2(v[0], v[1]);
        if (accumulate) { double2 o = E[id]; e.x += o.x; e.y += o.y; }
        E[id] = e;
        if (SPIN) {
            double2* B = reinterpret_cast<double2*>(almB);
            double2 b = make_double2(v[2], v[3]);
            if (accumulate) { double2 o = B[id]; b.x += o.x; b.y += o.y; }
            B[id] = b;
        }
    } else if (m == 0) {
        almE[roff + l] = accumulate ? almE[roff + l] + v[0] : v[0];
        if (SPIN) almB[roff + l] = accumulate ? almB[roff + l] + v[2] : v[2];
    } else {
        const int64_t off = roff + 2 * l;
        almE[off] = accumulate ? almE[off] + v[0] : v[0];
        almE[off + 1] = accumulate ? almE[off + 1] + v[1] : v[1];
        if (SPIN) {
            almB[off] = accumulate ? almB[off] + v[2] : v[2];
            almB[off + 1] = accumulate ? almB[off + 1] + v[3] : v[3];
        }
    }
}

// ------------------------------------------------------------------ active rings of a pixel-weight map
// In the PCG mat-vec A^T N^-1 A the rings whose N^-1 vanishes identically (inside a galactic mask) contribute exactly
// nothing: their synthesis is multiplied by zero and their analysis input is zero.  gs_active_rings_build marks the rings
// that carry weight and compacts the ring PAIRS with at least one such ring into an ascending list, all on the device
// (no host round trip); the Legendre kernels then walk that list and the fused ring stage drops the CTAs of idle rings.
// SH: the weight map is this rank's ring-sharded local map; every rank marks its own rings in `actd` (doubles, summed over
// the ranks by the caller), the others stay zero
// wconst (unsharded, nullable): the ring's pixel weight when all its pixels carry the same one (isotropic noise outside the
// mask: every ring that the mask edge does not cut), NaN otherwise; see the transform-free path of ring_apply_kernel
template <bool SH>
__global__ void __launch_bounds__(256) ring_active_kernel(PlanDev P, const double* __restrict__ pixw, unsigned char* __restrict__ act,
                                                          double* __restrict__ actd, double* __restrict__ wconst)
{
    const int ring = blockIdx.x, n = P.ring_nphi[ring];
    if (SH && P.sh.ring_owner[ring] != P.sh.rank) { if (threadIdx.x == 0) actd[ring] = 0.0; return; }
    const double* w = pixw + (SH ? P.sh.ring_start_loc[ring] : P.ring_start[ring]);
    const double w0 = w[0];
    int any = 0, differ = 0;
    for (int j = threadIdx.x; j < n; j += blockDim.x) { const double v = w[j]; any |= (v != 0.0); differ |= !(v == w0); }
    any = __syncthreads_or(any);
    if (!SH && wconst) differ = __syncthreads_or(differ);
    if (threadIdx.x == 0) {
        if (SH) actd[ring] = any ? 1.0 : 0.0; else act[ring] = any ? 1 : 0;
        if (!SH && wconst) wconst[ring] = differ ? __longlong_as_double(0x7ff8000000000000LL) : w0;
    }
}

__global__ void ring_flags_kernel(const double* __restrict__ actd, unsigned char* __restrict__ act, int n)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) act[i] = actd[i] > 0.0 ? 1 : 0;
}

__global__ void __launch_bounds__(1024) pair_compact_kernel(PlanDev P, unsigned char* act, int* __restrict__ list,
                                                            int* __restrict__ count)
{
    __shared__ int wsum[32];
    __shared__ int base;
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    if (tid == 0) base = 0;
    __syncthreads();
    for (int p0 = 0; p0 < P.npair; p0 += 1024) {
        const int p = p0 + tid;
        const bool on = p < P.npair && (act[p] || act[P.nring - 1 - p]);
        const unsigned b = __ballot_sync(FULL, on);
        if (lane == 0) wsum[w] = __popc(b);
        __syncthreads();
        int off = base;
        for (int i = 0; i < w; ++i) off += wsum[i];
        if (on) list[off + __popc(b & ((1u << lane) - 1u))] = p;
        // the ring stage must still process (to zero) an idle ring whose mirror ring carries weight: mark pairs, not rings
        if (p < P.npair) { act[p] = on; act[P.nring - 1 - p] = on; }
        __syncthreads();
        if (tid == 0) { int t = 0; for (int i = 0; i < 32; ++i) t += wsum[i]; base += t; }
        __syncthreads();
    }
    if (tid == 0) *count = base;
}

// slot0[spin][m] = first entry k of the list with m_lim(list[k]) >= m (count when none): one warp per (spin, m)
__global__ void __launch_bounds__(256) list_slot0_kernel(PlanDev P, const int* __restrict__ list, const int* __restrict__ count,
                                                         int* __restrict__ slot0)
{
    const int L = P.lmax, wid = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (wid >= 2 * (L + 1)) return;
    const int spin2 = wid > L, m = spin2 ? wid - (L + 1) : wid, n = *count;
    const int* mlim = spin2 ? P.mlim2 : P.mlim0;
    int first = n;
    for (int k0 = 0; k0 < n && first == n; k0 += 32) {
        const int k = k0 + lane;
        const unsigned b = __ballot_sync(FULL, k < n && mlim[list[k]] >= m);
        if (b) first = k0 + __ffs(b) - 1;
    }
    if (lane == 0) slot0[wid] = first;
}

int gs_active_rings_build(gs_plan* p, const double* pixw, cudaStream_t st)
{
    if (p->world > 1) {   // ring-sharded weights: local flags, summed over the ranks (every rank builds the same lists)
        ring_active_kernel<true><<<p->d.nring, 256, 0, st>>>(p->d, pixw, p->act_ring, p->act_red, nullptr);
        GS_CHECK_LAUNCH();
        int rc = gs_shard_allreduce(p, p->act_red, p->d.nring, st);
        if (rc) return rc;
        ring_flags_kernel<<<(p->d.nring + 255) / 256, 256, 0, st>>>(p->act_red, p->act_ring, p->d.nring);
    } else {
        ring_active_kernel<false><<<p->d.nring, 256, 0, st>>>(p->d, pixw, p->act_ring, nullptr, p->ring_wconst);
    }
    pair_compact_kernel<<<1, 1024, 0, st>>>(p->d, p->act_ring, p->act_pairs, p->act_count);
    list_slot0_kernel<<<(2 * (p->d.lmax + 1) * 32 + 255) / 256, 256, 0, st>>>(p->d, p->act_pairs, p->act_count, p->act_slot0);
    GS_CHECK_LAUNCH();
    g_gs_launches += 3;
    return gs_ring_order_build(p, st);
}

// ------------------------------------------------------------------ host launchers
// nc = 1: one right-hand side (spectra in p->Fm).  nc = 2: chain batch, unsharded plans whose buffers were sized by
// gs_plan_reserve_chains: chain c reads almE/almB + c alm_stride and fills the spectra p->Fm + c gs_fm_stride(p).
int64_t gs_fm_stride(const gs_plan* p) { return (int64_t)2 * p->d.nring * (p->d.lmax + 1); }
static int anal_chunks_of(const gs_plan* p, int nc) { const int per = LEG_NT * (nc > 1 ? LEG_RA2 : LEG_RA); return (p->d.npair + per - 1) / per; }
int64_t gs_part_stride(const gs_plan* p, int nc) { return (int64_t)anal_chunks_of(p, nc) * p->d.nalm * 4; }

static int check_batch(const gs_plan* p, int nc, int layout, const char* who)
{
    if (nc == 1) return GS_OK;
    if (nc != 2) { gs_set_error("%s: chain batches run 2 right-hand sides per launch (got %d)", who, nc); return GS_E_BADARG; }
    if (p->world > 1) { gs_set_error("%s: chain batches need an unsharded plan", who); return GS_E_BADARG; }
    if (p->chain_cap < nc) { gs_set_error("%s: call gs_plan_reserve_chains(plan, %d) first", who, nc); return GS_E_BADARG; }
    (void)layout;
    return GS_OK;
}

int gs_leg_synth(gs_plan* p, int spin, const double* almE, const double* almB, int layout, const double* fl,
                 cudaStream_t st, const int* skip, const double* flB, int nc, int64_t alm_stride)
{
    const bool sh = p->world > 1;
    if (sh && layout != GS_ALM_REAL) { gs_set_error("sharded plans take the (local) real alm layout only"); return GS_E_BADARG; }
    int rc = check_batch(p, nc, layout, "gs_leg_synth");
    if (rc) return rc;
    const int rr = nc == 2 ? LEG_R2 : LEG_R;
    dim3 grid((p->d.npair + LEG_NT * rr - 1) / (LEG_NT * rr), sh ? p->d.sh.nm_loc : p->d.lmax + 1);
    const int* plist = p->use_act ? p->act_pairs : nullptr;
    const int* pcount = plist ? p->act_count : nullptr;
    const int* slot0 = plist ? p->act_slot0 + (spin ? p->d.lmax + 1 : 0) : (spin ? p->d.pmin2 : p->d.pmin0);
    const int64_t fs = gs_fm_stride(p);
    if (nc == 2) {
        if (spin == 0) leg_synth_kernel<0, LEG_R2, false, 2><<<grid, LEG_NT, 0, st>>>(p->d, almE, almB, layout, fl, flB, p->Fm, skip, plist, pcount, slot0, alm_stride, fs, 0);
        else leg_synth_kernel<2, LEG_R2, false, 2><<<grid, LEG_NT, 0, st>>>(p->d, almE, almB, layout, fl, flB, p->Fm, skip, plist, pcount, slot0, alm_stride, fs, 0);
    } else if (!sh) {
        if (spin == 0) leg_synth_kernel<0, LEG_R, false, 1><<<grid, LEG_NT, 0, st>>>(p->d, almE, almB, layout, fl, flB, p->Fm, skip, plist, pcount, slot0, 0, 0, 0);
        else leg_synth_kernel<2, LEG_R, false, 1><<<grid, LEG_NT, 0, st>>>(p->d, almE, almB, layout, fl, flB, p->Fm, skip, plist, pcount, slot0, 0, 0, 0);
    } else {
        // m-sharded -> ring-sharded (the ring stage reads p->Fx), block of m by block of m: while the all-to-all of block b runs on
        // the plan's communication stream, the Legendre kernel of block b + 1 runs on `st` (SURVEY.md 5.8).  In-process test groups
        // exchange on `st` itself (host barriers).
        const ShardDev& S = p->d.sh;
        cudaStream_t comm = st;
        cudaEvent_t* ev = nullptr;
        const bool pipelined = !p->lgroup && S.NB > 1;
        if (pipelined && (rc = gs_shard_pipeline(p, &comm, &ev))) return rc;
        for (int b = 0; b < S.NB; ++b) {
            const int mk0 = b * S.MLb, cnt = std::min(S.MLb, S.nm_loc - mk0);
            if (cnt > 0) {
                dim3 g(grid.x, cnt);
                if (spin == 0) leg_synth_kernel<0, LEG_R, true, 1><<<g, LEG_NT, 0, st>>>(p->d, almE, almB, layout, fl, flB, p->Fm, skip, plist, pcount, slot0, 0, 0, mk0);
                else leg_synth_kernel<2, LEG_R, true, 1><<<g, LEG_NT, 0, st>>>(p->d, almE, almB, layout, fl, flB, p->Fm, skip, plist, pcount, slot0, 0, 0, mk0);
                GS_CHECK_LAUNCH();
                g_gs_launches += 1;
            }
            if (pipelined) {
                GS_CHECK_CUDA(cudaEventRecord(ev[b], st));
                GS_CHECK_CUDA(cudaStreamWaitEvent(comm, ev[b], 0));
            }
            if ((rc = gs_shard_exchange_block(p, p->Fm, p->Fx, b, comm))) return rc;
        }
        if (pipelined) {
            GS_CHECK_CUDA(cudaEventRecord(ev[S.NB], comm));
            GS_CHECK_CUDA(cudaStreamWaitEvent(st, ev[S.NB], 0));
        }
        return GS_OK;
    }
    GS_CHECK_LAUNCH();
    g_gs_launches += 1;
    return GS_OK;
}

template <int SPIN, int R, bool SH, int NC>
static int launch_anal(gs_plan* p, dim3 grid, cudaStream_t st, const int* skip, const int* plist, const int* pcount, const int* slot0,
                       int64_t fs, int64_t ps, int mk0 = 0)
{
    constexpr size_t sm = leg_anal_smem<SPIN, NC>();   // opt-in size set by gs_leg_prepare at plan creation
    leg_anal_kernel<SPIN, R, SH, NC><<<grid, LEG_NT, sm, st>>>(p->d, p->Fm, p->partial, skip, plist, pcount, slot0, fs, ps, mk0);
    GS_CHECK_LAUNCH();
    return GS_OK;
}

// The analysis kernels take their tiles from dynamic shared memory (the chain batch exceeds the 48 KB default): opt in once per
// device, at plan creation, so that no attribute call happens inside a stream capture (graph-replayed PCG).
int gs_leg_prepare(gs_plan* p)
{
    (void)p;
#define GS_ANAL_ATTR(SPIN, R, SH, NC) \
    GS_CHECK_CUDA(cudaFuncSetAttribute(leg_anal_kernel<SPIN, R, SH, NC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)leg_anal_smem<SPIN, NC>()))
    GS_ANAL_ATTR(0, LEG_RA, false, 1); GS_ANAL_ATTR(2, LEG_RA, false, 1);
    GS_ANAL_ATTR(0, LEG_RA, true, 1);  GS_ANAL_ATTR(2, LEG_RA, true, 1);
    GS_ANAL_ATTR(0, LEG_RA2, false, 2); GS_ANAL_ATTR(2, LEG_RA2, false, 2);
#undef GS_ANAL_ATTR
    return GS_OK;
}

int gs_leg_anal(gs_plan* p, int spin, double* almE, double* almB, int layout, const double* fl, double scale,
                int accumulate, cudaStream_t st, const int* skip, int nc, int64_t alm_stride)
{
    const bool sh = p->world > 1;
    if (sh && layout != GS_ALM_REAL) { gs_set_error("sharded plans take the (local) real alm layout only"); return GS_E_BADARG; }
    int rc = check_batch(p, nc, layout, "gs_leg_anal");
    if (rc) return rc;
    const int nchunk = anal_chunks_of(p, nc);
    if (nchunk * nc > p->anal_chunks) { gs_set_error("gs_leg_anal: workspace too small"); return GS_E_BADARG; }
    const int nmy = sh ? p->d.sh.nm_loc : p->d.lmax + 1;
    dim3 grid(nchunk, nmy);
    dim3 fgrid((p->d.lmax + 256) / 256, nmy, nc);
    const int* plist = p->use_act ? p->act_pairs : nullptr;
    const int* pcount = plist ? p->act_count : nullptr;
    const int* slot0 = plist ? p->act_slot0 + (spin ? p->d.lmax + 1 : 0) : (spin ? p->d.pmin2 : p->d.pmin0);
    const int64_t fs = gs_fm_stride(p), ps = gs_part_stride(p, nc);
    const int cp = LEG_NT * (nc > 1 ? LEG_RA2 : LEG_RA);   // ring pairs per chunk

    if (nc == 2) {
        if (spin == 0) {
            if ((rc = launch_anal<0, LEG_RA2, false, 2>(p, grid, st, skip, plist, pcount, slot0, fs, ps))) return rc;
            leg_finish_kernel<0, false><<<fgrid, 256, 0, st>>>(p->d, p->partial, nchunk, almE, almB, layout, fl, scale, accumulate, skip, pcount, slot0, cp, ps, alm_stride);
        } else {
            if ((rc = launch_anal<2, LEG_RA2, false, 2>(p, grid, st, skip, plist, pcount, slot0, fs, ps))) return rc;
            leg_finish_kernel<2, false><<<fgrid, 256, 0, st>>>(p->d, p->partial, nchunk, almE, almB, layout, fl, scale, accumulate, skip, pcount, slot0, cp, ps, alm_stride);
        }
    } else if (!sh) {
        if (spin == 0) {
            if ((rc = launch_anal<0, LEG_RA, false, 1>(p, grid, st, skip, plist, pcount, slot0, 0, 0))) return rc;
            leg_finish_kernel<0, false><<<fgrid, 256, 0, st>>>(p->d, p->partial, nchunk, almE, almB, layout, fl, scale, accumulate, skip, pcount, slot0, cp, 0, 0);
        } else {
            if ((rc = launch_anal<2, LEG_RA, false, 1>(p, grid, st, skip, plist, pcount, slot0, 0, 0))) return rc;
            leg_finish_kernel<2, false><<<fgrid, 256, 0, st>>>(p->d, p->partial, nchunk, almE, almB, layout, fl, scale, accumulate, skip, pcount, slot0, cp, 0, 0);
        }
    } else {
        // ring-sharded (p->Fx, written by the ring analysis) -> m-sharded, block by block: the all-to-all of block b + 1 runs on the
        // communication stream while the Legendre kernel of block b runs on `st`
        const ShardDev& S = p->d.sh;
        cudaStream_t comm = st;
        cudaEvent_t* ev = nullptr;
        const bool pipelined = !p->lgroup && S.NB > 1;
        if (pipelined) {
            if ((rc = gs_shard_pipeline(p, &comm, &ev))) return rc;
            GS_CHECK_CUDA(cudaEventRecord(ev[S.NB], st));
            GS_CHECK_CUDA(cudaStreamWaitEvent(comm, ev[S.NB], 0));
        }
        for (int b = 0; b < S.NB; ++b) {
            if ((rc = gs_shard_exchange_block(p, p->Fx, p->Fm, b, comm))) return rc;
            if (pipelined) {
                GS_CHECK_CUDA(cudaEventRecord(ev[b], comm));
                GS_CHECK_CUDA(cudaStreamWaitEvent(st, ev[b], 0));
            }
            const int mk0 = b * S.MLb, cnt = std::min(S.MLb, S.nm_loc - mk0);
            if (cnt <= 0) continue;
            dim3 g(grid.x, cnt);
            if (spin == 0) rc = launch_anal<0, LEG_RA, true, 1>(p, g, st, skip, plist, pcount, slot0, 0, 0, mk0);
            else rc = launch_anal<2, LEG_RA, true, 1>(p, g, st, skip, plist, pcount, slot0, 0, 0, mk0);
            if (rc) return rc;
        }
        if (spin == 0) leg_finish_kernel<0, true><<<fgrid, 256, 0, st>>>(p->d, p->partial, nchunk, almE, almB, layout, fl, scale, accumulate, skip, pcount, slot0, cp, 0, 0);
        else leg_finish_kernel<2, true><<<fgrid, 256, 0, st>>>(p->d, p->partial, nchunk, almE, almB, layout, fl, scale, accumulate, skip, pcount, slot0, cp, 0, 0);
    }
    GS_CHECK_LAUNCH();
    g_gs_launches += 2;
    return GS_OK;
}

int gs_leg_synth_blocks(gs_plan* p, const double* almE, const double* almB, const double* dflE, const double* dflB,
                        const int* lbE, int e0, int e1, const int* lbB, int b0, int b1, int lend, double2* Fblk, cudaStream_t st)
{
    if (p->world > 1) { gs_set_error("block-batched synthesis needs an unsharded plan"); return GS_E_BADARG; }
    constexpr int RB = 2;
    dim3 grid((p->d.npair + LEG_NT * RB - 1) / (LEG_NT * RB), std::min(lend, p->d.lmax + 1));
    const size_t sm = 2 * (size_t)(p->d.lmax + 2);
    const bool doE = e1 > e0, doB = b1 > b0;
    if (!doE && !doB) return GS_OK;
    if (doE && doB) leg_synth_blocks_kernel<RB, true, true><<<grid, LEG_NT, sm, st>>>(p->d, almE, almB, dflE, dflB, lbE, e0, e1, lbB, b0, b1, lend, Fblk);
    else if (doE) leg_synth_blocks_kernel<RB, true, false><<<grid, LEG_NT, sm, st>>>(p->d, almE, almB, dflE, dflB, lbE, e0, e1, lbB, b0, b1, lend, Fblk);
    else leg_synth_blocks_kernel<RB, false, true><<<grid, LEG_NT, sm, st>>>(p->d, almE, almB, dflE, dflB, lbE, e0, e1, lbB, b0, b1, lend, Fblk);
    GS_CHECK_LAUNCH();
    g_gs_launches += 1;
    return GS_OK;
}
