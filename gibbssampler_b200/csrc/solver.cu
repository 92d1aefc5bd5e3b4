// Constrained-realization solves (SURVEY.md 8a rows A4, A5, A10, A13).
//
//   Q x = b,  Q = C^-1 + B A^T N^-1 A B   (CenteredGibbs.py:448-491 + the forked qcinv's
//   multigrid_chain.sample / opfilt_pp.fwd_op / diag_cl preconditioner / cd_solve, not vendored)
//
// Everything lives in the reference's real alm layout so that dot products are plain sums
// (= qcinv's (2 - delta_m0)-weighted complex dot).  The mat-vec is the spin-2 SHT pair of
// legendre.cu / ringfft.cu with b_l fused into the Legendre staging on both sides and N^-1 fused
// into the ring-analysis load; the vector updates are three fused HBM-bound kernels whose
// reductions finish on the device (last-block pattern, fixed summation order => bit-reproducible),
// so alpha/beta and the convergence flag never travel to the host inside the loop; once the flag
// is set every later kernel (SHT stages included) returns immediately.
#include <math.h>
#include <string.h>

#include <algorithm>

#include "gs_internal.h"
#include "spectra.cuh"

#define SV_NT 256
#define SV_GRID (148 * 4)

struct PcgState {
    double delta, pq, rr, rz, d0, alpha, beta, eps2;
    int iter, itermax, done;
    unsigned counter;
};

struct gs_pcg_ws {
    double *r[2], *p[2], *q[2];
    // r02: the solver regenerates C^-1_l and the preconditioner M_l per coefficient from per-l tables (L1-resident) and a 2-byte
    // multipole index per coefficient instead of streaming two expanded 8-byte arrays: 12 instead of 15 array passes per iteration
    const unsigned short* lof;   // [n] multipole of every coefficient of the (local) real layout
    double* ic_l[2];             // [L+1] 1 / C_l (E, B), filled by precond_kernel at the start of a solve
    double* pre_l[2];            // [L+1] M_l
    double* partials;  // SV_GRID * 2
    double* red;       // sharded plans: local sums in, all-reduced sums out (NULL on one GPU)
    PcgState* state;
    PcgState* host_state;  // pinned, two slots (the graph path of a solve keeps two polls in flight)
};

// block-level sum of NR values, then the last block to finish adds the per-block partials in a
// fixed order.  Returns true (in every thread of that last block) with the totals in tot[].
template <int NR>
__device__ bool grid_reduce(double (&v)[NR], double* partials, unsigned* counter, double (&tot)[NR])
{
    __shared__ double sm[NR][SV_NT / 32];
    __shared__ bool last;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < NR; ++k) {
        double s = v[k];
        for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) sm[k][w] = s;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
#pragma unroll
        for (int k = 0; k < NR; ++k) {
            double s = 0.0;
            for (int i = 0; i < SV_NT / 32; ++i) s += sm[k][i];
            partials[blockIdx.x * NR + k] = s;
        }
        __threadfence();
        const unsigned t = atomicInc(counter, gridDim.x - 1);
        last = (t == gridDim.x - 1);
    }
    __syncthreads();
    if (!last) return false;
    __threadfence();
#pragma unroll
    for (int k = 0; k < NR; ++k) {
        double s = 0.0;
        for (int i = threadIdx.x; i < (int)gridDim.x; i += blockDim.x) s += partials[i * NR + k];
        for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        __syncthreads();
        if (lane == 0) sm[k][w] = s;
        __syncthreads();
        double t = 0.0;
        for (int i = 0; i < SV_NT / 32; ++i) t += sm[k][i];
        tot[k] = t;
    }
    return true;
}

// diag_cl preconditioner of qcinv's opfilt_pp: M_l = 1 / (1/C_l + b_l^2 sum(N^-1)/(4 pi))
__global__ void precond_kernel(const double* __restrict__ dl, const double* __restrict__ bl, double ninv, int L,
                               double* __restrict__ invc_l, double* __restrict__ pre_l)
{
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l > L) return;
    const double ic = safe_rcp(dl_to_cl(dl[l], l));
    invc_l[l] = ic;
    pre_l[l] = safe_rcp(ic + bl[l] * bl[l] * ninv);
}

__device__ __forceinline__ void pick(int64_t i, int64_t n, int& c, int64_t& j)
{
    c = i >= n;
    j = c ? i - n : i;
}

// scalar updates that follow each reduction.  One GPU: run by the last block of the reducing kernel.
// Sharded: that block stores its local sums in W.red, the host enqueues the all-reduce and then
// pcg_scalar_kernel, so every rank applies the same update to the same numbers.
__device__ __forceinline__ void fin_init(PcgState* s, double rr, double rz)
{
    s->rr = rr; s->d0 = rr; s->delta = rz; s->iter = 0;
    s->done = (rr <= 0.0 || s->itermax <= 0) ? 1 : 0;
}
__device__ __forceinline__ void fin_apq(PcgState* s, double pq)
{
    s->pq = pq;
    s->alpha = pq != 0.0 ? s->delta / pq : 0.0;
}
__device__ __forceinline__ void fin_update(PcgState* s, double rr, double rz)
{
    s->rr = rr; s->rz = rz;
    s->beta = s->delta != 0.0 ? rz / s->delta : 0.0;
    s->delta = rz;
    s->iter += 1;
    // qcinv cd_monitors.monitor_basic: stop when <r,r> <= eps^2 <r0,r0> or iter >= iter_max
    if (rr <= s->eps2 * s->d0 || s->iter >= s->itermax) s->done = 1;
}
__global__ void pcg_scalar_kernel(gs_pcg_ws W, int stage)
{
    PcgState* s = W.state;
    if (stage == 0) fin_init(s, W.red[0], W.red[1]);
    else if (s->done) return;
    else if (stage == 1) fin_apq(s, W.red[0]);
    else fin_update(s, W.red[0], W.red[1]);
}

// r = b - q (q = Q x0, or q absent for x0 = 0), p = M r, delta = <r, M r>, d0 = rr = <r, r>
__global__ void __launch_bounds__(SV_NT)
pcg_init_kernel(gs_pcg_ws W, const double* bE, const double* bB, int have_q, int64_t n, int nc)
{
    double v[2] = {0.0, 0.0};
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < nc * n; i += (int64_t)gridDim.x * blockDim.x) {
        int c; int64_t j;
        pick(i, n, c, j);
        double r = (c ? bB : bE)[j];
        if (have_q) r -= (c ? W.q[1] : W.q[0])[j];
        const double z = (c ? W.pre_l[1] : W.pre_l[0])[W.lof[j]] * r;
        (c ? W.r[1] : W.r[0])[j] = r;
        (c ? W.p[1] : W.p[0])[j] = z;
        v[0] += r * r;
        v[1] += r * z;
    }
    double tot[2];
    if (grid_reduce<2>(v, W.partials, &W.state->counter, tot) && threadIdx.x == 0) {
        if (W.red) { W.red[0] = tot[0]; W.red[1] = tot[1]; }
        else fin_init(W.state, tot[0], tot[1]);
    }
}

// The vector kernels walk the E and B arrays with a grid stride, SV_U elements per thread and step with all loads issued
// before the first store (the arrays may alias as far as the compiler knows): enough bytes in flight to approach HBM speed.
#define SV_U 4

// q += C^-1 p ; pq = <p, q> ; alpha = delta / pq
__global__ void __launch_bounds__(SV_NT) pcg_apq_kernel(gs_pcg_ws W, int64_t n, int nc)
{
    if (W.state->done) return;
    double v[1] = {0.0};
    const int64_t stride = (int64_t)gridDim.x * blockDim.x, total = nc * n;
    for (int64_t i0 = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i0 < total; i0 += SV_U * stride) {
        double p[SV_U], q[SV_U], ic[SV_U];
#pragma unroll
        for (int k = 0; k < SV_U; ++k) {
            const int64_t i = i0 + k * stride;
            int c; int64_t j;
            pick(i, n, c, j);
            const bool ok = i < total;
            p[k] = ok ? (c ? W.p[1] : W.p[0])[j] : 0.0; q[k] = ok ? (c ? W.q[1] : W.q[0])[j] : 0.0;
            ic[k] = ok ? __ldg((c ? W.ic_l[1] : W.ic_l[0]) + W.lof[j]) : 0.0;
        }
#pragma unroll
        for (int k = 0; k < SV_U; ++k) {
            const int64_t i = i0 + k * stride;
            if (i >= total) break;
            int c; int64_t j;
            pick(i, n, c, j);
            const double qq = fma(ic[k], p[k], q[k]);
            (c ? W.q[1] : W.q[0])[j] = qq;
            v[0] += p[k] * qq;
        }
    }
    double tot[1];
    if (grid_reduce<1>(v, W.partials, &W.state->counter, tot) && threadIdx.x == 0) {
        if (W.red) W.red[0] = tot[0];
        else fin_apq(W.state, tot[0]);
    }
}

// x += alpha p ; r -= alpha q ; rr = <r,r> ; rz = <r, M r> ; beta = rz/delta ; convergence test
__global__ void __launch_bounds__(SV_NT) pcg_update_kernel(gs_pcg_ws W, double* xE, double* xB, int64_t n, int nc)
{
    if (W.state->done) return;
    const double alpha = W.state->alpha;
    double v[2] = {0.0, 0.0};
    const int64_t stride = (int64_t)gridDim.x * blockDim.x, total = nc * n;
    for (int64_t i0 = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i0 < total; i0 += SV_U * stride) {
        double x[SV_U], p[SV_U], q[SV_U], r[SV_U], pre[SV_U];
#pragma unroll
        for (int k = 0; k < SV_U; ++k) {
            const int64_t i = i0 + k * stride;
            int c; int64_t j;
            pick(i, n, c, j);
            const bool ok = i < total;
            x[k] = ok ? (c ? xB : xE)[j] : 0.0; p[k] = ok ? (c ? W.p[1] : W.p[0])[j] : 0.0; q[k] = ok ? (c ? W.q[1] : W.q[0])[j] : 0.0;
            r[k] = ok ? (c ? W.r[1] : W.r[0])[j] : 0.0; pre[k] = ok ? __ldg((c ? W.pre_l[1] : W.pre_l[0]) + W.lof[j]) : 0.0;
        }
#pragma unroll
        for (int k = 0; k < SV_U; ++k) {
            const int64_t i = i0 + k * stride;
            if (i >= total) break;
            int c; int64_t j;
            pick(i, n, c, j);
            (c ? xB : xE)[j] = fma(alpha, p[k], x[k]);
            const double rr = fma(-alpha, q[k], r[k]);
            (c ? W.r[1] : W.r[0])[j] = rr;
            v[0] += rr * rr;
            v[1] += rr * rr * pre[k];
        }
    }
    double tot[2];
    if (grid_reduce<2>(v, W.partials, &W.state->counter, tot) && threadIdx.x == 0) {
        if (W.red) { W.red[0] = tot[0]; W.red[1] = tot[1]; }
        else fin_update(W.state, tot[0], tot[1]);
    }
}

// p = M r + beta p
__global__ void __launch_bounds__(SV_NT) pcg_dir_kernel(gs_pcg_ws W, int64_t n, int nc)
{
    if (W.state->done) return;
    const double beta = W.state->beta;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x, total = nc * n;
    for (int64_t i0 = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i0 < total; i0 += SV_U * stride) {
        double p[SV_U], r[SV_U], pre[SV_U];
#pragma unroll
        for (int k = 0; k < SV_U; ++k) {
            const int64_t i = i0 + k * stride;
            int c; int64_t j;
            pick(i, n, c, j);
            const bool ok = i < total;
            p[k] = ok ? (c ? W.p[1] : W.p[0])[j] : 0.0; r[k] = ok ? (c ? W.r[1] : W.r[0])[j] : 0.0;
            pre[k] = ok ? __ldg((c ? W.pre_l[1] : W.pre_l[0]) + W.lof[j]) : 0.0;
        }
#pragma unroll
        for (int k = 0; k < SV_U; ++k) {
            const int64_t i = i0 + k * stride;
            if (i >= total) break;
            int c; int64_t j;
            pick(i, n, c, j);
            (c ? W.p[1] : W.p[0])[j] = fma(beta, p[k], pre[k] * r[k]);
        }
    }
}

__global__ void zero2_kernel(double* a, double* b, int64_t n)
{
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        a[i] = 0.0;
        b[i] = 0.0;
    }
}

// y = q + C^-1 x with C^-1 from the per-l table (warm start of a solve, gs_cr_apply_q_*); y may be q
__global__ void add_cinv_kernel(const double* q, const double* __restrict__ ic_l, const unsigned short* __restrict__ lof,
                                const double* __restrict__ x, double* y, int64_t n)
{
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        y[i] = fma(ic_l[lof[i]], x[i], q[i]);
}

__global__ void scale_map_kernel(const double* __restrict__ a, const double* __restrict__ w, double* __restrict__ out, int64_t n)
{
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) out[i] = a[i] * w[i];
}

__global__ void rhs_combine_kernel(double* rhs, const double* sic, const double* xi, const double* bdata, double resc, int64_t n)
{
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        rhs[i] = fma(resc, rhs[i], fma(sic[i], xi[i], bdata[i]));
}

// multipole of every coefficient of the real layout (unsharded: index algebra of utils.py:49-76; sharded: the plan's l_of_loc)
__global__ void lof_build_kernel(unsigned short* __restrict__ lof, const int* __restrict__ l_of_loc, int L, int64_t n)
{
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        lof[i] = (unsigned short)(l_of_loc ? l_of_loc[i] : l_of_real(i, L));
}
static bool build_lof(gs_plan* p, const unsigned short** out)
{
    void* d = nullptr;
    const int64_t n = p->nreal_loc;
    if (cudaMalloc(&d, (size_t)n * sizeof(unsigned short)) != cudaSuccess) return false;
    p->owned.push_back(d);
    lof_build_kernel<<<SV_GRID, SV_NT>>>((unsigned short*)d, p->world > 1 ? p->d.sh.l_of_loc : nullptr, p->d.lmax, n);
    if (cudaDeviceSynchronize() != cudaSuccess) return false;
    *out = (const unsigned short*)d;
    return true;
}

// ------------------------------------------------------------------ workspace
// The workspaces belong to the plan (gs_plan::pcg_ws, pcg_ws_batch, pcg_ws_teb): created on the first solve, released by
// gs_plan_destroy, which frees the device buffers recorded in p->owned and the pinned host buffers in p->owned_host and calls
// gs_pcg_ws_free for the workspace structs.  A plan is used by one host thread at a time (include/gibbs_b200.h), so no lock is
// taken.
static bool alloc_owned(gs_plan* p, double** q, size_t cnt)
{
    void* d = nullptr;
    if (cudaMalloc(&d, cnt * sizeof(double)) != cudaSuccess) return false;
    p->owned.push_back(d);
    *q = (double*)d;
    return true;
}

// the solver state on the device (in p->owned) and its pinned host copy with two slots (the graph path of a solve keeps two
// polls in flight; in p->owned_host)
static bool alloc_state(gs_plan* p, PcgState** state, PcgState** host_state)
{
    void* d = nullptr;
    if (cudaMalloc(&d, sizeof(PcgState)) != cudaSuccess) return false;
    p->owned.push_back(d);
    *state = (PcgState*)d;
    void* h = nullptr;
    if (cudaMallocHost(&h, 2 * sizeof(PcgState)) != cudaSuccess) return false;
    p->owned_host.push_back(h);
    *host_state = (PcgState*)h;
    return true;
}

static gs_pcg_ws* get_ws(gs_plan* p)
{
    if (p->pcg_ws) return (gs_pcg_ws*)p->pcg_ws;
    gs_pcg_ws* w = new gs_pcg_ws();
    const size_t n = (size_t)p->nreal_loc;
    w->red = p->world > 1 ? p->red_loc : nullptr;
    bool ok = true;
    const size_t L1 = (size_t)p->d.lmax + 1;
    for (int c = 0; c < 2 && ok; ++c)
        ok = alloc_owned(p, &w->r[c], n) && alloc_owned(p, &w->p[c], n) && alloc_owned(p, &w->q[c], n) && alloc_owned(p, &w->ic_l[c], L1) &&
             alloc_owned(p, &w->pre_l[c], L1);
    ok = ok && alloc_owned(p, &w->partials, SV_GRID * 2) && build_lof(p, &w->lof);
    ok = ok && alloc_state(p, &w->state, &w->host_state);
    if (!ok) { gs_set_error("PCG workspace allocation failed: %s", cudaGetErrorString(cudaGetLastError())); delete w; return nullptr; }
    p->pcg_ws = w;
    return w;
}

// Chain batch (gs_cr_pcg_pol_batch): two workspaces whose p and q vectors lie one batch stride (2 n doubles: E then B of a chain)
// apart, so that the chain-batched mat-vec reads / writes them as one strided array.  Allocated on the first batched solve.
static gs_pcg_ws* get_ws_batch(gs_plan* p)
{
    if (p->pcg_ws_batch) return (gs_pcg_ws*)p->pcg_ws_batch;
    gs_pcg_ws* w = new gs_pcg_ws[2]();
    const size_t n = (size_t)p->nreal_loc, L1 = (size_t)p->d.lmax + 1;
    double *P = nullptr, *Q = nullptr;
    bool ok = alloc_owned(p, &P, 4 * n) && alloc_owned(p, &Q, 4 * n);
    for (int k = 0; k < 2 && ok; ++k) {
        w[k].red = nullptr;
        for (int c = 0; c < 2 && ok; ++c) {
            w[k].p[c] = P + (2 * k + c) * n;
            w[k].q[c] = Q + (2 * k + c) * n;
            ok = alloc_owned(p, &w[k].r[c], n) && alloc_owned(p, &w[k].ic_l[c], L1) && alloc_owned(p, &w[k].pre_l[c], L1);
        }
        ok = ok && alloc_owned(p, &w[k].partials, SV_GRID * 2);
        if (ok) { if (k == 0) ok = build_lof(p, &w[0].lof); else w[1].lof = w[0].lof; }
        ok = ok && alloc_state(p, &w[k].state, &w[k].host_state);
    }
    void* d = nullptr;
    ok = ok && cudaMalloc(&d, sizeof(int)) == cudaSuccess;
    if (ok) { p->owned.push_back(d); p->pcg_alldone = (int*)d; }
    if (!ok) { gs_set_error("batched PCG workspace allocation failed: %s", cudaGetErrorString(cudaGetLastError())); delete[] w; return nullptr; }
    p->pcg_ws_batch = w;
    return w;
}

int g_gs_pcg_graph = 1;   // 1: the iterations between two convergence polls of an unsharded PCG solve are replayed from a CUDA graph
extern "C" int gs_set_pcg_graph(int on) { const int old = g_gs_pcg_graph; g_gs_pcg_graph = on ? 1 : 0; return old; }
int g_gs_ring_fused = 1;
extern "C" int gs_set_ring_fused(int fused) { const int old = g_gs_ring_fused; g_gs_ring_fused = fused ? 1 : 0; return old; }

// Rings whose N^-1 is identically zero (inside the mask) add nothing to A^T N^-1 A: the mat-vec walks the rings that carry
// weight only (gs_active_rings_build; lists rebuilt from the weight map of each solve, on the device).
int g_gs_ring_skip = 1;
// Rings on which N^-1 is constant (isotropic noise, ring not cut by the mask edge): DFT^H diag(w) DFT = n w on the alias-folded
// spectrum, so the fused ring stage of the mat-vec needs no transform there (ring_apply_kernel; flags from gs_active_rings_build).
int g_gs_ring_const = 1;
extern "C" int gs_set_ring_const(int on) { const int old = g_gs_ring_const; g_gs_ring_const = on ? 1 : 0; return old; }
extern "C" int gs_set_ring_skip(int on) { const int old = g_gs_ring_skip; g_gs_ring_skip = on ? 1 : 0; return old; }

struct ActiveRings {   // scope guard: the plan's launchers use the active lists while one of these lives
    gs_plan* p;
    bool on;
    ActiveRings(gs_plan* p_) : p(p_), on(false) {}
    int begin(const double* pixw, cudaStream_t st)
    {
        if (!g_gs_ring_skip || !pixw) return GS_OK;
        int rc = gs_active_rings_build(p, pixw, st);
        if (rc == GS_OK) { p->use_act = true; on = true; }
        return rc;
    }
    ~ActiveRings() { if (on) p->use_act = false; }
};

// q = B A^T N^-1 A B v   (C^-1 v is added by pcg_apq_kernel / the caller)
// nc = 2 (chain batch): chain c reads vE/vB + c stride and writes qE/qB + c stride; one recurrence serves both chains
static int apply_noise_op(gs_plan* p, const double* vE, const double* vB, const double* bl, const double* inv_noise,
                          double* qE, double* qB, cudaStream_t st, const int* skip, int spin = 2, int nc = 1, int64_t stride = 0)
{
    int rc;
    if ((rc = gs_leg_synth(p, spin, vE, vB, GS_ALM_REAL, bl, st, skip, nullptr, nc, stride))) return rc;
    if (g_gs_ring_fused || nc > 1) {
        if ((rc = gs_ring_apply(p, spin, inv_noise, st, skip, nc))) return rc;
    } else {
        if ((rc = gs_ring_synth(p, spin, p->mapQ_tmp, p->mapU_tmp, st, skip))) return rc;
        if ((rc = gs_ring_anal(p, spin, p->mapQ_tmp, p->mapU_tmp, inv_noise, st, skip))) return rc;
    }
    return gs_leg_anal(p, spin, qE, qB, GS_ALM_REAL, bl, 1.0, 0, st, skip, nc, stride);
}

// Start of a solve: a zeroed solver state with the stopping rule, written to the pinned host slot and copied to the device on `st`
static int pcg_state_reset(PcgState* state, PcgState* host_state, double eps, int itermax, cudaStream_t st)
{
    memset(host_state, 0, sizeof(PcgState));
    host_state->eps2 = eps * eps;
    host_state->itermax = itermax;
    GS_CHECK_CUDA(cudaMemcpyAsync(state, host_state, sizeof(PcgState), cudaMemcpyHostToDevice, st));
    return GS_OK;
}

// End of a solve: iterations and |r|/|r0| to the caller, GS_E_NOTCONVERGED if iter_max came first.  chain >= 0: the solve is
// that chain of a batch, which the message names.
static int pcg_report(const PcgState& s, double eps, int itermax, int chain, int* n_iter_out, double* resid_out)
{
    const double rel = s.d0 > 0.0 ? sqrt(s.rr / s.d0) : 0.0;
    if (n_iter_out) *n_iter_out = s.iter;
    if (resid_out) *resid_out = rel;
    if (!(s.d0 > 0.0 && s.rr > s.eps2 * s.d0)) return GS_OK;
    if (chain < 0) gs_set_error("PCG stopped at iter_max = %d with |r|/|r0| = %.3e > eps = %.1e", itermax, rel, eps);
    else gs_set_error("PCG (chain %d of the batch) stopped at iter_max = %d with |r|/|r0| = %.3e > eps = %.1e", chain, itermax, rel, eps);
    return GS_E_NOTCONVERGED;
}

// The poll loop shared by the PCG solves: `iteration(stream)` enqueues one PCG iteration whose launches take every scalar
// (alpha, beta, the done flag) from `state` on the device.  The solver state has been initialised on `st` before the call.
template <class Iteration>
static int pcg_poll_loop(gs_plan* p, cudaStream_t st, PcgState* state, PcgState* host_state, bool dist, double eps, int itermax,
                         int check_every, Iteration& iteration, int* n_iter_out, double* resid_out)
{
    // Unsharded plans: the `check_every` iterations between two polls of the convergence flag are captured ONCE per solve in a
    // CUDA graph on a stream of the plan (capture is not allowed on the legacy default stream) and replayed: one graph launch
    // instead of 7 check_every kernel launches per poll (the host side of a solve was ~2300 launches; SCALE_r01 lost 1.8 % at 8
    // GPUs to 8 processes doing that on shared cores).  gs_set_pcg_graph(0) restores plain launches.
    int rc = GS_OK;
    int launched = 0;
    bool finished = false;
    cudaGraphExec_t gexec = nullptr;
    long long launches_per_graph = 0;
    if (g_gs_pcg_graph && !dist && itermax >= check_every) {
        if (!p->work_stream) {
            cudaStream_t ws = nullptr;
            GS_CHECK_CUDA(cudaStreamCreateWithFlags(&ws, cudaStreamNonBlocking));
            p->work_stream = ws;
            cudaEvent_t ev = nullptr;
            GS_CHECK_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
            p->work_event = ev;
        }
        cudaStream_t ws = (cudaStream_t)p->work_stream;
        GS_CHECK_CUDA(cudaEventRecord((cudaEvent_t)p->work_event, st));
        GS_CHECK_CUDA(cudaStreamWaitEvent(ws, (cudaEvent_t)p->work_event, 0));
        st = ws;   // the rest of the solve runs here; every poll (and the return) synchronises it with the host
        cudaGraph_t graph = nullptr;
        const long long l0 = g_gs_launches;
        GS_CHECK_CUDA(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
        rc = GS_OK;
        for (int k = 0; k < check_every && rc == GS_OK; ++k) rc = iteration(st);
        cudaError_t ce = cudaStreamEndCapture(st, &graph);
        launches_per_graph = g_gs_launches - l0;
        g_gs_launches = l0;   // nothing ran yet: counted per replay below
        if (rc != GS_OK) { if (graph) cudaGraphDestroy(graph); return rc; }
        if (ce != cudaSuccess) { gs_set_error("PCG graph capture: %s", cudaGetErrorString(ce)); return GS_E_CUDA; }
        ce = cudaGraphInstantiate(&gexec, graph, 0);
        cudaGraphDestroy(graph);
        if (ce != cudaSuccess) { gs_set_error("PCG graph instantiate: %s", cudaGetErrorString(ce)); return GS_E_CUDA; }
    }
    if (gexec) {
        // Two batches in flight: the host enqueues batch k + 1 (graph replay + copy of the solver state + event) BEFORE it waits for the
        // state that follows batch k, so the wake-up after a poll and the next graph launch are hidden behind 8 iterations of GPU work
        // (43 polls per solve at NSIDE 512; with 8 ranks on shared host cores this was the remaining loss of the chains mode).  Once
        // the done flag is set every kernel of a later batch returns at once: at most one batch of no-ops per solve, same iterations.
        PcgState* hs = host_state;
        cudaEvent_t ev[2] = {nullptr, nullptr};
        cudaError_t ce = cudaEventCreateWithFlags(&ev[0], cudaEventDisableTiming);
        if (ce == cudaSuccess) ce = cudaEventCreateWithFlags(&ev[1], cudaEventDisableTiming);
        int cur = 0, inflight = 0;
        while (ce == cudaSuccess && !finished) {
            while (ce == cudaSuccess && inflight < 2 && launched + check_every <= itermax) {
                const int sl = (cur + inflight) & 1;
                ce = cudaGraphLaunch(gexec, st);
                if (ce == cudaSuccess) ce = cudaMemcpyAsync(hs + sl, state, sizeof(PcgState), cudaMemcpyDeviceToHost, st);
                if (ce == cudaSuccess) ce = cudaEventRecord(ev[sl], st);
                launched += check_every;
                g_gs_launches += launches_per_graph;
                ++inflight;
            }
            if (ce != cudaSuccess || inflight == 0) break;   // fewer than check_every iterations left: the loop below runs them
            ce = cudaEventSynchronize(ev[cur]);
            if (ce != cudaSuccess) break;
            --inflight;
            if (hs[cur].done || launched >= itermax) {
                if (inflight) ce = cudaStreamSynchronize(st);   // the batch behind it: no-ops after `done`, or the last iterations
                if (inflight && ce == cudaSuccess) cur ^= 1;
                hs[0] = hs[cur];
                finished = hs[0].done || launched >= itermax;
                inflight = 0;
                if (!finished) cur = 0;
                continue;
            }
            cur ^= 1;
        }
        if (ev[0]) cudaEventDestroy(ev[0]);
        if (ev[1]) cudaEventDestroy(ev[1]);
        if (ce != cudaSuccess) { cudaGraphExecDestroy(gexec); gs_set_error("PCG graph loop: %s", cudaGetErrorString(ce)); return GS_E_CUDA; }
    }
    while (!finished) {
        for (int k = 0; k < check_every && launched < itermax; ++k, ++launched)
            if ((rc = iteration(st))) { if (gexec) cudaGraphExecDestroy(gexec); return rc; }
        cudaError_t ce = cudaMemcpyAsync(host_state, state, sizeof(PcgState), cudaMemcpyDeviceToHost, st);
        if (ce == cudaSuccess) ce = cudaStreamSynchronize(st);
        if (ce != cudaSuccess) { if (gexec) cudaGraphExecDestroy(gexec); gs_set_error("PCG poll: %s", cudaGetErrorString(ce)); return GS_E_CUDA; }
        finished = host_state->done || launched >= itermax;
    }
    if (gexec) cudaGraphExecDestroy(gexec);
    return pcg_report(*host_state, eps, itermax, -1, n_iter_out, resid_out);
}

// spin 2: (E, B) system; spin 0: temperature (dl_BB, rhs_B, x_B unused)
static int cr_pcg_impl(gs_plan* p, int spin, const double* dl_EE, const double* dl_BB, const double* bl,
                       const double* inv_noise, double ninv_sum_over_4pi, const double* rhs_E,
                       const double* rhs_B, double* x_E, double* x_B, int warm_start, double eps, int itermax,
                       int check_every, int* n_iter_out, double* resid_out, void* stream)
{
    const int nc = spin ? 2 : 1;
    GS_REQUIRE(eps > 0.0 && itermax >= 0, "eps must be > 0 and itermax >= 0");
    GS_CHECK_CUDA(cudaSetDevice(p->device));
    cudaStream_t st = (cudaStream_t)stream;
    gs_pcg_ws* w = get_ws(p);
    if (!w) return GS_E_NOMEM;
    const int L = p->d.lmax;
    const int64_t n = p->nreal_loc;
    if (check_every < 1) check_every = 8;

    // per-l C^-1 and preconditioner: the vector kernels index them with the multipole of each coefficient, w->lof
    const int lb = (L + 256) / 256;
    precond_kernel<<<lb, 256, 0, st>>>(dl_EE, bl, ninv_sum_over_4pi, L, w->ic_l[0], w->pre_l[0]);
    if (nc == 2) precond_kernel<<<lb, 256, 0, st>>>(dl_BB, bl, ninv_sum_over_4pi, L, w->ic_l[1], w->pre_l[1]);
    GS_CHECK_LAUNCH();
    int rc;
    const bool dist = p->world > 1;
    ActiveRings act(p);
    if ((rc = act.begin(inv_noise, st))) return rc;

    if ((rc = pcg_state_reset(w->state, w->host_state, eps, itermax, st))) return rc;
    if (warm_start) {  // r0 = b - Q x0
        if ((rc = apply_noise_op(p, x_E, x_B, bl, inv_noise, w->q[0], w->q[1], st, nullptr, spin))) return rc;
        add_cinv_kernel<<<SV_GRID, SV_NT, 0, st>>>(w->q[0], w->ic_l[0], w->lof, x_E, w->q[0], n);
        if (nc == 2) add_cinv_kernel<<<SV_GRID, SV_NT, 0, st>>>(w->q[1], w->ic_l[1], w->lof, x_B, w->q[1], n);
    } else {
        zero2_kernel<<<SV_GRID, SV_NT, 0, st>>>(x_E, nc == 2 ? x_B : x_E, n);
    }
    pcg_init_kernel<<<SV_GRID, SV_NT, 0, st>>>(*w, rhs_E, rhs_B, warm_start ? 1 : 0, n, nc);
    GS_CHECK_LAUNCH();
    if (dist) {
        if ((rc = gs_shard_allreduce(p, w->red, 2, st))) return rc;
        pcg_scalar_kernel<<<1, 1, 0, st>>>(*w, 0);
    }

    const int* done = &w->state->done;
    // one PCG iteration: 7 launches whose arguments do not change during the solve (alpha, beta and the done flag live on the device)
    auto iteration = [&](cudaStream_t s) -> int {
        int r;
        if ((r = apply_noise_op(p, w->p[0], w->p[1], bl, inv_noise, w->q[0], w->q[1], s, done, spin))) return r;
        pcg_apq_kernel<<<SV_GRID, SV_NT, 0, s>>>(*w, n, nc);
        if (dist) {
            if ((r = gs_shard_allreduce(p, w->red, 1, s))) return r;
            pcg_scalar_kernel<<<1, 1, 0, s>>>(*w, 1);
        }
        pcg_update_kernel<<<SV_GRID, SV_NT, 0, s>>>(*w, x_E, x_B, n, nc);
        if (dist) {
            if ((r = gs_shard_allreduce(p, w->red, 2, s))) return r;
            pcg_scalar_kernel<<<1, 1, 0, s>>>(*w, 2);
        }
        pcg_dir_kernel<<<SV_GRID, SV_NT, 0, s>>>(*w, n, nc);
        GS_CHECK_LAUNCH();
        g_gs_launches += 3;
        return GS_OK;
    };
    return pcg_poll_loop(p, st, w->state, w->host_state, dist, eps, itermax, check_every, iteration, n_iter_out, resid_out);
}

extern "C" int gs_cr_pcg_pol(gs_plan* p, const double* dl_EE, const double* dl_BB, const double* bl,
                             const double* inv_noise, double ninv_sum_over_4pi, const double* rhs_E,
                             const double* rhs_B, double* x_E, double* x_B, int warm_start, double eps, int itermax,
                             int check_every, int* n_iter_out, double* resid_out, void* stream)
{
    if (!p) { gs_set_error("null plan"); return GS_E_BADARG; }
    GS_REQUIRE(dl_EE && dl_BB && bl && inv_noise && rhs_E && rhs_B && x_E && x_B, "null pointer argument");
    return cr_pcg_impl(p, 2, dl_EE, dl_BB, bl, inv_noise, ninv_sum_over_4pi, rhs_E, rhs_B, x_E, x_B, warm_start, eps, itermax,
                       check_every, n_iter_out, resid_out, stream);
}

__global__ void pcg_alldone_kernel(const PcgState* a, const PcgState* b, int* out) { *out = (a->done && b->done) ? 1 : 0; }

// Two independent chains (same data, beam and N^-1; their own D_l, right-hand sides and solutions, chain c at + c stride
// doubles, dl at + c (L+1)) solved side by side: while both are iterating, every mat-vec is ONE chain-batched launch per stage
// (leg_synth / ring_apply / leg_anal with two right-hand sides sharing the Legendre recurrence); the vector kernels, alpha,
// beta and the stopping rule stay per chain, so each chain performs exactly the iterations of its own gs_cr_pcg_pol call.
// When one chain has converged (seen at the next poll) the other continues on the single-chain kernels.
extern "C" int gs_cr_pcg_pol_batch(gs_plan* p, int n_chain, const double* dl_EE, const double* dl_BB, const double* bl,
                                   const double* inv_noise, double ninv_sum_over_4pi, const double* rhs_E,
                                   const double* rhs_B, double* x_E, double* x_B, int64_t stride, double eps, int itermax,
                                   int check_every, int* n_iter_out, double* resid_out, void* stream)
{
    if (!p) { gs_set_error("null plan"); return GS_E_BADARG; }
    GS_REQUIRE(dl_EE && dl_BB && bl && inv_noise && rhs_E && rhs_B && x_E && x_B, "null pointer argument");
    GS_REQUIRE(n_chain == 1 || n_chain == 2, "n_chain must be 1 or 2");
    const int L = p->d.lmax;
    if (n_chain == 1)
        return cr_pcg_impl(p, 2, dl_EE, dl_BB, bl, inv_noise, ninv_sum_over_4pi, rhs_E, rhs_B, x_E, x_B, 0, eps, itermax, check_every,
                           n_iter_out, resid_out, stream);
    GS_REQUIRE(p->world == 1, "chain batches need an unsharded plan");
    GS_REQUIRE(eps > 0.0 && itermax >= 0, "eps must be > 0 and itermax >= 0");
    GS_CHECK_CUDA(cudaSetDevice(p->device));
    int rc;
    if ((rc = gs_plan_reserve_chains(p, 2))) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    gs_pcg_ws* W = get_ws_batch(p);
    if (!W) return GS_E_NOMEM;
    const int64_t n = p->nreal_loc;
    if (check_every < 1) check_every = 8;
    const int lb = (L + 256) / 256;
    ActiveRings act(p);
    if ((rc = act.begin(inv_noise, st))) return rc;
    for (int k = 0; k < 2; ++k) {
        gs_pcg_ws* w = &W[k];
        precond_kernel<<<lb, 256, 0, st>>>(dl_EE + k * (L + 1), bl, ninv_sum_over_4pi, L, w->ic_l[0], w->pre_l[0]);
        precond_kernel<<<lb, 256, 0, st>>>(dl_BB + k * (L + 1), bl, ninv_sum_over_4pi, L, w->ic_l[1], w->pre_l[1]);
        GS_CHECK_LAUNCH();
        if ((rc = pcg_state_reset(w->state, w->host_state, eps, itermax, st))) return rc;
        zero2_kernel<<<SV_GRID, SV_NT, 0, st>>>(x_E + k * stride, x_B + k * stride, n);
        pcg_init_kernel<<<SV_GRID, SV_NT, 0, st>>>(*w, rhs_E + k * stride, rhs_B + k * stride, 0, n, 2);
        GS_CHECK_LAUNCH();
    }
    pcg_alldone_kernel<<<1, 1, 0, st>>>(W[0].state, W[1].state, p->pcg_alldone);
    const int64_t bstride = 2 * n;   // W[1].p[c] = W[0].p[c] + 2 n (get_ws_batch)
    bool done[2] = {false, false};
    int launched = 0;
    while (!(done[0] && done[1]) && launched < itermax) {
        for (int it = 0; it < check_every && launched < itermax; ++it, ++launched) {
            if (!done[0] && !done[1]) {
                if ((rc = apply_noise_op(p, W[0].p[0], W[0].p[1], bl, inv_noise, W[0].q[0], W[0].q[1], st, p->pcg_alldone, 2, 2, bstride))) return rc;
            } else {
                gs_pcg_ws* w = &W[done[0] ? 1 : 0];
                if ((rc = apply_noise_op(p, w->p[0], w->p[1], bl, inv_noise, w->q[0], w->q[1], st, &w->state->done, 2))) return rc;
            }
            for (int k = 0; k < 2; ++k) {
                if (done[k]) continue;
                pcg_apq_kernel<<<SV_GRID, SV_NT, 0, st>>>(W[k], n, 2);
                pcg_update_kernel<<<SV_GRID, SV_NT, 0, st>>>(W[k], x_E + k * stride, x_B + k * stride, n, 2);
                pcg_dir_kernel<<<SV_GRID, SV_NT, 0, st>>>(W[k], n, 2);
                g_gs_launches += 3;
            }
            if (!done[0] && !done[1]) { pcg_alldone_kernel<<<1, 1, 0, st>>>(W[0].state, W[1].state, p->pcg_alldone); g_gs_launches += 1; }
            GS_CHECK_LAUNCH();
        }
        for (int k = 0; k < 2; ++k) GS_CHECK_CUDA(cudaMemcpyAsync(W[k].host_state, W[k].state, sizeof(PcgState), cudaMemcpyDeviceToHost, st));
        GS_CHECK_CUDA(cudaStreamSynchronize(st));
        for (int k = 0; k < 2; ++k) done[k] = W[k].host_state->done != 0;
    }
    int ret = GS_OK;   // both chains are reported; GS_E_NOTCONVERGED if either stopped at iter_max
    for (int k = 0; k < 2; ++k)
        if (pcg_report(*W[k].host_state, eps, itermax, k, n_iter_out ? n_iter_out + k : nullptr, resid_out ? resid_out + k : nullptr))
            ret = GS_E_NOTCONVERGED;
    return ret;
}

// Temperature twin (qcinv opfilt_tt chain of ConstrainedRealization.py:40-41, run at CenteredGibbs.py:141-165 and
// NonCenteredGibbs.py:57-72): Q = C^-1 + B A^T N^-1 A B on one spin-0 field.
extern "C" int gs_cr_pcg_tt(gs_plan* p, const double* dl_TT, const double* bl, const double* inv_noise,
                            double ninv_sum_over_4pi, const double* rhs, double* x, int warm_start, double eps, int itermax,
                            int check_every, int* n_iter_out, double* resid_out, void* stream)
{
    if (!p) { gs_set_error("null plan"); return GS_E_BADARG; }
    GS_REQUIRE(dl_TT && bl && inv_noise && rhs && x, "null pointer argument");
    return cr_pcg_impl(p, 0, dl_TT, nullptr, bl, inv_noise, ninv_sum_over_4pi, rhs, nullptr, x, nullptr, warm_start, eps, itermax,
                       check_every, n_iter_out, resid_out, stream);
}

// gs_cr_apply_q_pol (spin 2) and gs_cr_apply_q_tt (spin 0: temperature in the E slots, the B arguments unused)
static int apply_q_impl(gs_plan* p, int spin, const double* dl_E, const double* dl_B, const double* bl, const double* inv_noise,
                        const double* x_E, const double* x_B, double* y_E, double* y_B, void* stream)
{
    const int nc = spin ? 2 : 1;
    GS_CHECK_CUDA(cudaSetDevice(p->device));
    cudaStream_t st = (cudaStream_t)stream;
    gs_pcg_ws* w = get_ws(p);
    if (!w) return GS_E_NOMEM;
    int rc;
    ActiveRings act(p);
    if ((rc = act.begin(inv_noise, st))) return rc;
    const int L = p->d.lmax;
    const double* dl[2] = {dl_E, dl_B};
    const double* x[2] = {x_E, x_B};
    double* y[2] = {y_E, y_B};
    for (int c = 0; c < nc; ++c)
        precond_kernel<<<(L + 256) / 256, 256, 0, st>>>(dl[c], bl, 0.0, L, w->ic_l[c], w->pre_l[c]);   // only C^-1 is read
    if ((rc = apply_noise_op(p, x_E, x_B, bl, inv_noise, w->q[0], spin ? w->q[1] : nullptr, st, nullptr, spin))) return rc;
    for (int c = 0; c < nc; ++c) add_cinv_kernel<<<SV_GRID, SV_NT, 0, st>>>(w->q[c], w->ic_l[c], w->lof, x[c], y[c], p->nreal_loc);
    GS_CHECK_LAUNCH();
    return GS_OK;
}

// gs_cr_rhs_pol (spin 2) and gs_cr_rhs_tt (spin 0: the temperature maps in the Q slots, its coefficients in the E slots, the
// U and B arguments unused).  The data term is computed from the maps when bdata_E is NULL.
static int rhs_impl(gs_plan* p, int spin, const double* dl_E, const double* dl_B, const double* bl, const double* inv_noise,
                    const double* sqrt_inv_noise, const double* bdata_E, const double* bdata_B, const double* d_Q, const double* d_U,
                    const double* xi_Q, const double* xi_U, const double* xi_E, const double* xi_B, int fluct_iter, double* rhs_E,
                    double* rhs_B, void* stream)
{
    const int nc = spin ? 2 : 1;
    GS_CHECK_CUDA(cudaSetDevice(p->device));
    cudaStream_t st = (cudaStream_t)stream;
    gs_pcg_ws* w = get_ws(p);
    if (!w) return GS_E_NOMEM;
    auto map2alm = [&](const double* mQ, const double* mU, const double* pixw, int iter, int adjoint, double* aE, double* aB) {
        return spin ? gs_map2alm_spin2(p, mQ, mU, pixw, iter, adjoint, bl, aE, aB, GS_ALM_REAL, stream)
                    : gs_map2alm_spin0(p, mQ, pixw, iter, adjoint, bl, aE, GS_ALM_REAL, stream);
    };
    int rc;
    // fluctuation term 1: utils.adjoint_synthesis_hp (utils.py:79-111) = bl * (Npix/4pi) * map2alm(iter=3)
    if ((rc = map2alm(xi_Q, xi_U, sqrt_inv_noise, fluct_iter, 0, rhs_E, rhs_B))) return rc;
    const double resc = (double)p->d.npix / (4.0 * GS_PI);
    // fluctuation term 2 and data term; use r[] / p[] of the PCG workspace as scratch
    const double* dl[2] = {dl_E, dl_B};
    for (int c = 0; c < nc; ++c)
        if ((rc = gs_plan_expand_per_l(p, dl[c], 4, w->r[c], st))) return rc;
    const double* bd[2] = {bdata_E, bdata_B};
    if (!bdata_E) {
        if ((rc = map2alm(d_Q, d_U, inv_noise, 0, 1, w->p[0], w->p[1]))) return rc;
        bd[0] = w->p[0];
        bd[1] = w->p[1];
    }
    // rhs = resc * rhs + sqrt(C^-1) xi + bdata
    const double* xi[2] = {xi_E, xi_B};
    double* rhs[2] = {rhs_E, rhs_B};
    for (int c = 0; c < nc; ++c) rhs_combine_kernel<<<SV_GRID, SV_NT, 0, st>>>(rhs[c], w->r[c], xi[c], bd[c], resc, p->nreal_loc);
    GS_CHECK_LAUNCH();
    return GS_OK;
}

extern "C" int gs_cr_apply_q_tt(gs_plan* p, const double* dl_TT, const double* bl, const double* inv_noise, const double* x,
                                double* y, void* stream)
{
    if (!p) { gs_set_error("null plan"); return GS_E_BADARG; }
    GS_REQUIRE(dl_TT && bl && inv_noise && x && y, "null pointer argument");
    return apply_q_impl(p, 0, dl_TT, nullptr, bl, inv_noise, x, nullptr, y, nullptr, stream);
}

// Right-hand side of the temperature system (CenteredGibbs.py:145-147, NonCenteredGibbs.py:61-63; RNG order xi_alm, xi_pix):
//   b = bdata + C^-1/2 xi_alm + B (Npix/4pi) map2alm_{iter}(N^-1/2 xi_pix),  bdata = B A^T N^-1 d (what qcinv adds in
//   chain.sample) passed precomputed or computed from d.
extern "C" int gs_cr_rhs_tt(gs_plan* p, const double* dl_TT, const double* bl, const double* inv_noise,
                            const double* sqrt_inv_noise, const double* bdata, const double* d, const double* xi_alm,
                            const double* xi_pix, int fluct_iter, double* rhs, void* stream)
{
    if (!p) { gs_set_error("null plan"); return GS_E_BADARG; }
    GS_REQUIRE(dl_TT && bl && inv_noise && sqrt_inv_noise && xi_alm && xi_pix && rhs, "null pointer argument");
    GS_REQUIRE(bdata || d, "need either the precomputed data term or the data map");
    GS_REQUIRE(fluct_iter >= 0, "fluct_iter must be >= 0");
    return rhs_impl(p, 0, dl_TT, nullptr, bl, inv_noise, sqrt_inv_noise, bdata, nullptr, d, nullptr, xi_pix, nullptr, xi_alm, nullptr,
                    fluct_iter, rhs, nullptr, stream);
}

// y = Q x = C^-1 x + B A^T N^-1 A B x   (qcinv opfilt_pp.fwd_op; CenteredGibbs.py:629, 651-656)
extern "C" int gs_cr_apply_q_pol(gs_plan* p, const double* dl_EE, const double* dl_BB, const double* bl,
                                 const double* inv_noise, const double* x_E, const double* x_B, double* y_E,
                                 double* y_B, void* stream)
{
    if (!p) { gs_set_error("null plan"); return GS_E_BADARG; }
    GS_REQUIRE(dl_EE && dl_BB && bl && inv_noise && x_E && x_B && y_E && y_B, "null pointer argument");
    return apply_q_impl(p, 2, dl_EE, dl_BB, bl, inv_noise, x_E, x_B, y_E, y_B, stream);
}

// Right-hand side of the masked-sky system (CenteredGibbs.py:469-483, RNG order xi_Q, xi_U, xi_E, xi_B):
//   b = B A^T N^-1 d  +  B (Npix/4pi) map2alm_{iter}(N^-1/2 xi_pix)  +  C^-1/2 xi_alm
// The first term is what qcinv's calc_prep adds inside chain.sample; it equals the reference's
// second_part_grad (CenteredGibbs.py:298-308) and may be passed precomputed (bdata_*).
extern "C" int gs_cr_rhs_pol(gs_plan* p, const double* dl_EE, const double* dl_BB, const double* bl,
                             const double* inv_noise, const double* sqrt_inv_noise, const double* bdata_E,
                             const double* bdata_B, const double* d_Q, const double* d_U, const double* xi_Q,
                             const double* xi_U, const double* xi_E, const double* xi_B, int fluct_iter,
                             double* rhs_E, double* rhs_B, void* stream)
{
    if (!p) { gs_set_error("null plan"); return GS_E_BADARG; }
    GS_REQUIRE(dl_EE && dl_BB && bl && inv_noise && sqrt_inv_noise && xi_Q && xi_U && xi_E && xi_B && rhs_E && rhs_B,
               "null pointer argument");
    GS_REQUIRE((bdata_E && bdata_B) || (d_Q && d_U), "need either the precomputed data term or the data maps");
    GS_REQUIRE(fluct_iter >= 0, "fluct_iter must be >= 0");
    return rhs_impl(p, 2, dl_EE, dl_BB, bl, inv_noise, sqrt_inv_noise, bdata_E, bdata_B, d_Q, d_U, xi_Q, xi_U, xi_E, xi_B, fluct_iter,
                    rhs_E, rhs_B, stream);
}

// ------------------------------------------------------------------ joint T/E/B system on a cut sky
// qcinv's joint T+P filter (opfilt_tp upstream; not vendored, restated here): the (T, E, B) coefficients of every (l, m) are
// coupled by the per-l prior C_l = [[TT, TE, 0], [TE, EE, 0], [0, 0, BB]], the data by two pixel weight maps:
//   Q = C^-1 + B A^T N^-1 A B,   A B x = (alm2map_spin0(b x_T), alm2map_spin2(b x_E, b x_B)),  N^-1 = diag(N_T^-1, N_P^-1, N_P^-1)
// The mat-vec is the spin-0 mat-vec of the TT solve on x_T with N_T^-1 followed by the spin-2 mat-vec of the E/B solve on
// (x_E, x_B) with N_P^-1; the vector kernels take one coefficient of all three fields per thread, because T_j and E_j meet in
// the 2x2 block of C^-1 and of the preconditioner.  Singular blocks follow safe_inv: a zero field inverts to zero, a block with
// C^TE = 0 inverts field by field, and a TE block with zero determinant gives a zero C^-1 block.

// Per-l tables of the joint solve: [ic_TT, ic_TE, ic_EE, ic_BB, M_TT, M_TE, M_EE, M_BB] for every l (8 doubles)
#define TEB_TAB 8

struct TebWs {
    double *r[3], *p[3], *q[3];   // T, E, B
    const unsigned short* lof;     // multipole of every coefficient (shared with gs_pcg_ws)
    double* tab;                   // [L+1][TEB_TAB]
    double* partials;              // SV_GRID * 2
    PcgState* state;
    PcgState* host_state;          // pinned, two slots
};

// inverse of the symmetric 2x2 [[a, b], [b, d]] (safe_inv convention above)
__device__ __forceinline__ void inv2x2(double a, double b, double d, double& i11, double& i12, double& i22)
{
    if (b == 0.0) { i11 = safe_rcp(a); i12 = 0.0; i22 = safe_rcp(d); return; }
    const double det = a * d - b * b;
    const double id = safe_rcp(det);
    i11 = d * id; i12 = -b * id; i22 = a * id;
}

// One thread per l: C_l^-1 and the diag_cl preconditioner M_l = (C_l^-1 + diag(b_l^2 nT, b_l^2 nP, b_l^2 nP))^-1,
// nX = sum(N_X^-1) / (4 pi)
__global__ void teb_tables_kernel(const double* __restrict__ dlTT, const double* __restrict__ dlTE, const double* __restrict__ dlEE,
                                  const double* __restrict__ dlBB, const double* __restrict__ bl, double nT, double nP, int L,
                                  double* __restrict__ tab)
{
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l > L) return;
    double i11, i12, i22;
    inv2x2(dl_to_cl(dlTT[l], l), dl_to_cl(dlTE[l], l), dl_to_cl(dlEE[l], l), i11, i12, i22);
    const double ibb = safe_rcp(dl_to_cl(dlBB[l], l));
    const double b2 = bl[l] * bl[l];
    double m11, m12, m22;
    inv2x2(i11 + b2 * nT, i12, i22 + b2 * nP, m11, m12, m22);
    double* t = tab + (int64_t)l * TEB_TAB;
    t[0] = i11; t[1] = i12; t[2] = i22; t[3] = ibb;
    t[4] = m11; t[5] = m12; t[6] = m22; t[7] = safe_rcp(ibb + b2 * nP);
}

// the four entries of a per-l block (off 0: C^-1, off 4: M) through the read-only cache
__device__ __forceinline__ double4 teb_blk(const double* tab, int l, int off)
{
    const double2 u = __ldg((const double2*)(tab + l * TEB_TAB + off));
    const double2 v = __ldg((const double2*)(tab + l * TEB_TAB + off + 2));
    return make_double4(u.x, u.y, v.x, v.y);
}

// y = q + K v with the per-l block K = (tt, te, ee, bb) on (T, E) and B
__device__ __forceinline__ void teb_mul_add(const double4& k, double vT, double vE, double vB, double qT, double qE, double qB,
                                            double& yT, double& yE, double& yB)
{
    yT = fma(k.x, vT, fma(k.y, vE, qT));
    yE = fma(k.y, vT, fma(k.z, vE, qE));
    yB = fma(k.w, vB, qB);
}

// Each thread takes TEB_U coefficients j (grid stride), T, E and B of each; all loads are issued before the first store.
#define TEB_U 2

// r = b - (q + C^-1 x)  (warm start; q = B A^T N^-1 A B x) or r = b ; p = M r ; delta = <r, M r> ; d0 = rr = <r, r>
__global__ void __launch_bounds__(SV_NT)
teb_init_kernel(TebWs W, const double* bT, const double* bE, const double* bB, const double* xT, const double* xE, const double* xB,
                int have_q, int64_t n)
{
    double v[2] = {0.0, 0.0};
    for (int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; j < n; j += (int64_t)gridDim.x * blockDim.x) {
        const int l = W.lof[j];
        double rT = bT[j], rE = bE[j], rB = bB[j];
        if (have_q) {
            double yT, yE, yB;
            teb_mul_add(teb_blk(W.tab, l, 0), xT[j], xE[j], xB[j], W.q[0][j], W.q[1][j], W.q[2][j], yT, yE, yB);
            rT -= yT; rE -= yE; rB -= yB;
        }
        double zT, zE, zB;
        teb_mul_add(teb_blk(W.tab, l, 4), rT, rE, rB, 0.0, 0.0, 0.0, zT, zE, zB);
        W.r[0][j] = rT; W.r[1][j] = rE; W.r[2][j] = rB;
        W.p[0][j] = zT; W.p[1][j] = zE; W.p[2][j] = zB;
        v[0] += rT * rT + rE * rE + rB * rB;
        v[1] += rT * zT + rE * zE + rB * zB;
    }
    double tot[2];
    if (grid_reduce<2>(v, W.partials, &W.state->counter, tot) && threadIdx.x == 0) fin_init(W.state, tot[0], tot[1]);
}

// pq = <p, q + C^-1 p> ; alpha = delta / pq.  q keeps B A^T N^-1 A B p: teb_update_kernel adds C^-1 p again on the fly (same
// arithmetic), which saves the store of q and its second read.
__global__ void __launch_bounds__(SV_NT) teb_apq_kernel(TebWs W, int64_t n)
{
    if (W.state->done) return;
    double v[1] = {0.0};
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t j0 = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; j0 < n; j0 += TEB_U * stride) {
        double p[TEB_U][3], q[TEB_U][3];
        double4 ic[TEB_U];
#pragma unroll
        for (int k = 0; k < TEB_U; ++k) {
            const int64_t j = j0 + k * stride;
            const bool ok = j < n;
#pragma unroll
            for (int c = 0; c < 3; ++c) { p[k][c] = ok ? W.p[c][j] : 0.0; q[k][c] = ok ? W.q[c][j] : 0.0; }
            ic[k] = ok ? teb_blk(W.tab, W.lof[j], 0) : make_double4(0.0, 0.0, 0.0, 0.0);
        }
#pragma unroll
        for (int k = 0; k < TEB_U; ++k) {
            double yT, yE, yB;
            teb_mul_add(ic[k], p[k][0], p[k][1], p[k][2], q[k][0], q[k][1], q[k][2], yT, yE, yB);
            v[0] += p[k][0] * yT + p[k][1] * yE + p[k][2] * yB;
        }
    }
    double tot[1];
    if (grid_reduce<1>(v, W.partials, &W.state->counter, tot) && threadIdx.x == 0) fin_apq(W.state, tot[0]);
}

// x += alpha p ; r -= alpha (q + C^-1 p) ; rr = <r, r> ; rz = <r, M r> ; beta = rz / delta ; convergence test
__global__ void __launch_bounds__(SV_NT) teb_update_kernel(TebWs W, double* xT, double* xE, double* xB, int64_t n)
{
    if (W.state->done) return;
    const double alpha = W.state->alpha;
    double* const x[3] = {xT, xE, xB};
    double v[2] = {0.0, 0.0};
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t j0 = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; j0 < n; j0 += TEB_U * stride) {
        double xv[TEB_U][3], p[TEB_U][3], q[TEB_U][3], r[TEB_U][3];
        double4 ic[TEB_U], m[TEB_U];
#pragma unroll
        for (int k = 0; k < TEB_U; ++k) {
            const int64_t j = j0 + k * stride;
            const bool ok = j < n;
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                xv[k][c] = ok ? x[c][j] : 0.0; p[k][c] = ok ? W.p[c][j] : 0.0;
                q[k][c] = ok ? W.q[c][j] : 0.0; r[k][c] = ok ? W.r[c][j] : 0.0;
            }
            const int l = ok ? W.lof[j] : 0;
            ic[k] = teb_blk(W.tab, l, 0);
            m[k] = teb_blk(W.tab, l, 4);
        }
#pragma unroll
        for (int k = 0; k < TEB_U; ++k) {
            const int64_t j = j0 + k * stride;
            if (j >= n) break;
            double y[3], z[3];
            teb_mul_add(ic[k], p[k][0], p[k][1], p[k][2], q[k][0], q[k][1], q[k][2], y[0], y[1], y[2]);
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                x[c][j] = fma(alpha, p[k][c], xv[k][c]);
                r[k][c] = fma(-alpha, y[c], r[k][c]);
                W.r[c][j] = r[k][c];
            }
            teb_mul_add(m[k], r[k][0], r[k][1], r[k][2], 0.0, 0.0, 0.0, z[0], z[1], z[2]);
            v[0] += r[k][0] * r[k][0] + r[k][1] * r[k][1] + r[k][2] * r[k][2];
            v[1] += r[k][0] * z[0] + r[k][1] * z[1] + r[k][2] * z[2];
        }
    }
    double tot[2];
    if (grid_reduce<2>(v, W.partials, &W.state->counter, tot) && threadIdx.x == 0) fin_update(W.state, tot[0], tot[1]);
}

// p = M r + beta p
__global__ void __launch_bounds__(SV_NT) teb_dir_kernel(TebWs W, int64_t n)
{
    if (W.state->done) return;
    const double beta = W.state->beta;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t j0 = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; j0 < n; j0 += TEB_U * stride) {
        double p[TEB_U][3], r[TEB_U][3];
        double4 m[TEB_U];
#pragma unroll
        for (int k = 0; k < TEB_U; ++k) {
            const int64_t j = j0 + k * stride;
            const bool ok = j < n;
#pragma unroll
            for (int c = 0; c < 3; ++c) { p[k][c] = ok ? W.p[c][j] : 0.0; r[k][c] = ok ? W.r[c][j] : 0.0; }
            m[k] = teb_blk(W.tab, ok ? W.lof[j] : 0, 4);
        }
#pragma unroll
        for (int k = 0; k < TEB_U; ++k) {
            const int64_t j = j0 + k * stride;
            if (j >= n) break;
            double bp[3];
#pragma unroll
            for (int c = 0; c < 3; ++c) bp[c] = beta * p[k][c];
            double o[3];
            teb_mul_add(m[k], r[k][0], r[k][1], r[k][2], bp[0], bp[1], bp[2], o[0], o[1], o[2]);
#pragma unroll
            for (int c = 0; c < 3; ++c) W.p[c][j] = o[c];
        }
    }
}

// y = q + C^-1 x  (gs_cr_apply_q_teb)
__global__ void teb_add_cinv_kernel(TebWs W, const double* xT, const double* xE, const double* xB, double* yT, double* yE, double* yB,
                                    int64_t n)
{
    for (int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; j < n; j += (int64_t)gridDim.x * blockDim.x) {
        double a, b, c;
        teb_mul_add(teb_blk(W.tab, W.lof[j], 0), xT[j], xE[j], xB[j], W.q[0][j], W.q[1][j], W.q[2][j], a, b, c);
        yT[j] = a; yE[j] = b; yB[j] = c;
    }
}

// rhs = resc rhs + F xi_alm + bdata, F = L^-T on (T, E) with C^TE block = L L^T (lower Cholesky), 1/sqrt(C^BB) on B:
// F F^T = C^-1, so the prior term has covariance C^-1.  A field with C = 0 gets F = 0 (safe_inv, as mode 4 of gs_expand_per_l).
__global__ void teb_rhs_combine_kernel(const unsigned short* __restrict__ lof, const double* __restrict__ dlTT,
                                       const double* __restrict__ dlTE, const double* __restrict__ dlEE,
                                       const double* __restrict__ dlBB, const double* xiT, const double* xiE, const double* xiB,
                                       const double* bdT, const double* bdE, const double* bdB, double resc, double* rT, double* rE,
                                       double* rB, int64_t n)
{
    for (int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; j < n; j += (int64_t)gridDim.x * blockDim.x) {
        const int l = lof[j];
        const double a = dl_to_cl(dlTT[l], l), b = dl_to_cl(dlTE[l], l), d = dl_to_cl(dlEE[l], l), e = dl_to_cl(dlBB[l], l);
        double fTT, fTE, fEE;
        if (b == 0.0) {
            fTT = a != 0.0 ? sqrt(1.0 / a) : 0.0;
            fTE = 0.0;
            fEE = d != 0.0 ? sqrt(1.0 / d) : 0.0;
        } else {
            const double l11 = sqrt(a), l21 = b / l11, l22 = sqrt(d - l21 * l21);
            fTT = 1.0 / l11;
            fTE = -l21 / (l11 * l22);
            fEE = 1.0 / l22;
        }
        const double fBB = e != 0.0 ? sqrt(1.0 / e) : 0.0;
        const double xt = xiT[j], xe = xiE[j], xb = xiB[j];
        rT[j] = fma(resc, rT[j], fma(fTT, xt, fma(fTE, xe, bdT[j])));
        rE[j] = fma(resc, rE[j], fma(fEE, xe, bdE[j]));
        rB[j] = fma(resc, rB[j], fma(fBB, xb, bdB[j]));
    }
}

static TebWs* get_ws_teb(gs_plan* p)
{
    if (p->pcg_ws_teb) return (TebWs*)p->pcg_ws_teb;
    gs_pcg_ws* base = get_ws(p);   // for its per-coefficient multipole index
    if (!base) return nullptr;
    TebWs* w = new TebWs();
    const size_t n = (size_t)p->nreal_loc;
    bool ok = true;
    for (int c = 0; c < 3 && ok; ++c) ok = alloc_owned(p, &w->r[c], n) && alloc_owned(p, &w->p[c], n) && alloc_owned(p, &w->q[c], n);
    ok = ok && alloc_owned(p, &w->tab, (size_t)TEB_TAB * (p->d.lmax + 1)) && alloc_owned(p, &w->partials, SV_GRID * 2);
    w->lof = base->lof;
    ok = ok && alloc_state(p, &w->state, &w->host_state);
    if (!ok) { gs_set_error("joint T/E/B workspace allocation failed: %s", cudaGetErrorString(cudaGetLastError())); delete w; return nullptr; }
    p->pcg_ws_teb = w;
    return w;
}

void gs_pcg_ws_free(gs_plan* p)
{
    delete (gs_pcg_ws*)p->pcg_ws;
    delete[] (gs_pcg_ws*)p->pcg_ws_batch;
    delete (TebWs*)p->pcg_ws_teb;
    p->pcg_ws = p->pcg_ws_batch = p->pcg_ws_teb = nullptr;
}

// Two weight maps, one set of plan-wide ring flags: the Legendre and ring launchers read act_ring / act_pairs / act_slot0 /
// ring_wconst and the dynamic group order from the plan, and ring_apply_kernel takes the weight of a constant-weight ring from
// ring_wconst, not from the map.  So the joint solve builds the flags of N_P^-1 in the plan's own set and those of N_T^-1 in
// p->flags_T, once per call, and swaps the two sets while it enqueues the spin-0 half (the launch arguments are fixed at enqueue
// time, graph capture included).  When both weight maps are the same array the plan's set serves both halves.
static void swap_flags(gs_plan* p)
{
    RingFlags& f = p->flags_T;
    std::swap(p->act_ring, f.act_ring);
    std::swap(p->act_pairs, f.act_pairs);
    std::swap(p->act_count, f.act_count);
    std::swap(p->act_slot0, f.act_slot0);
    std::swap(p->ring_wconst, f.ring_wconst);
    std::swap(p->groups0_dyn, f.groups0_dyn);
    std::swap(p->groups2_dyn, f.groups2_dyn);
}

static int alloc_flags_T(gs_plan* p)
{
    RingFlags& f = p->flags_T;
    if (f.act_ring) return GS_OK;
    const int L1 = p->d.lmax + 1;
    auto alloc = [&](void** q, size_t bytes) { void* d = nullptr; if (cudaMalloc(&d, std::max<size_t>(16, bytes)) != cudaSuccess) return false; p->owned.push_back(d); *q = d; return true; };
    bool ok = alloc((void**)&f.act_ring, (size_t)p->d.nring) && alloc((void**)&f.act_pairs, (size_t)p->d.npair * sizeof(int)) &&
              alloc((void**)&f.act_count, sizeof(int)) && alloc((void**)&f.act_slot0, (size_t)2 * L1 * sizeof(int)) &&
              alloc((void**)&f.ring_wconst, (size_t)p->d.nring * sizeof(double)) &&
              alloc((void**)&f.groups0_dyn, (size_t)p->ngroups0 * sizeof(int2)) && alloc((void**)&f.groups2_dyn, (size_t)p->ngroups2 * sizeof(int2));
    if (!ok) { memset(&f, 0, sizeof(f)); gs_set_error("ring flag allocation failed: %s", cudaGetErrorString(cudaGetLastError())); return GS_E_NOMEM; }
    return GS_OK;
}

struct TebRings {   // scope guard: both flag sets of one joint call; the plan's own set afterwards as before
    gs_plan* p;
    ActiveRings act;
    bool two;       // the spin-0 half runs on p->flags_T
    TebRings(gs_plan* p_) : p(p_), act(p_), two(false) {}
    int begin(const double* invT, const double* invP, cudaStream_t st)
    {
        int rc = act.begin(invP, st);
        if (rc || !act.on || invT == invP) return rc;
        if ((rc = alloc_flags_T(p))) return rc;
        swap_flags(p);
        rc = gs_active_rings_build(p, invT, st);
        swap_flags(p);
        two = rc == GS_OK;
        return rc;
    }
};

// q = B A^T N^-1 A B v on (T, E, B): the spin-0 half on N_T^-1, then the spin-2 half on N_P^-1
static int teb_noise_op(gs_plan* p, TebRings& tr, const double* vT, const double* vE, const double* vB, const double* bl,
                        const double* invT, const double* invP, double* qT, double* qE, double* qB, cudaStream_t st, const int* skip)
{
    if (tr.two) swap_flags(p);
    int rc = apply_noise_op(p, vT, nullptr, bl, invT, qT, nullptr, st, skip, 0);
    if (tr.two) swap_flags(p);
    if (rc) return rc;
    return apply_noise_op(p, vE, vB, bl, invP, qE, qB, st, skip, 2);
}

static int teb_unsharded(gs_plan* p, const char* who)
{
    if (p->world > 1) {
        gs_set_error("%s: the joint T/E/B solve needs an unsharded plan (this plan is sharded over %d ranks)", who, p->world);
        return GS_E_BADARG;
    }
    return GS_OK;
}

// Joint twin of gs_cr_pcg_pol / gs_cr_pcg_tt (include/gibbs_b200.h): one poll loop, one CUDA graph per solve
extern "C" int gs_cr_pcg_teb(gs_plan* p, const double* dl_TT, const double* dl_TE, const double* dl_EE, const double* dl_BB,
                             const double* bl, const double* inv_noise_T, const double* inv_noise_P, double ninvT_sum_over_4pi,
                             double ninvP_sum_over_4pi, const double* rhs_T, const double* rhs_E, const double* rhs_B, double* x_T,
                             double* x_E, double* x_B, int warm_start, double eps, int itermax, int check_every, int* n_iter_out,
                             double* resid_out, void* stream)
{
    if (!p) { gs_set_error("null plan"); return GS_E_BADARG; }
    GS_REQUIRE(dl_TT && dl_TE && dl_EE && dl_BB && bl && inv_noise_T && inv_noise_P && rhs_T && rhs_E && rhs_B && x_T && x_E && x_B,
               "null pointer argument");
    GS_REQUIRE(eps > 0.0 && itermax >= 0, "eps must be > 0 and itermax >= 0");
    int rc;
    if ((rc = teb_unsharded(p, __func__))) return rc;
    GS_CHECK_CUDA(cudaSetDevice(p->device));
    cudaStream_t st = (cudaStream_t)stream;
    TebWs* w = get_ws_teb(p);
    if (!w) return GS_E_NOMEM;
    const int L = p->d.lmax;
    const int64_t n = p->nreal_loc;
    if (check_every < 1) check_every = 8;
    teb_tables_kernel<<<(L + 256) / 256, 256, 0, st>>>(dl_TT, dl_TE, dl_EE, dl_BB, bl, ninvT_sum_over_4pi, ninvP_sum_over_4pi, L, w->tab);
    GS_CHECK_LAUNCH();
    TebRings tr(p);
    if ((rc = tr.begin(inv_noise_T, inv_noise_P, st))) return rc;

    if ((rc = pcg_state_reset(w->state, w->host_state, eps, itermax, st))) return rc;
    if (warm_start) {  // r0 = b - Q x0
        if ((rc = teb_noise_op(p, tr, x_T, x_E, x_B, bl, inv_noise_T, inv_noise_P, w->q[0], w->q[1], w->q[2], st, nullptr))) return rc;
    } else {
        zero2_kernel<<<SV_GRID, SV_NT, 0, st>>>(x_T, x_E, n);
        zero2_kernel<<<SV_GRID, SV_NT, 0, st>>>(x_B, x_B, n);
    }
    teb_init_kernel<<<SV_GRID, SV_NT, 0, st>>>(*w, rhs_T, rhs_E, rhs_B, x_T, x_E, x_B, warm_start ? 1 : 0, n);
    GS_CHECK_LAUNCH();

    const int* done = &w->state->done;
    // one PCG iteration: the spin-0 and spin-2 mat-vecs, then 3 vector kernels; every argument is fixed for the whole solve
    auto iteration = [&](cudaStream_t s) -> int {
        int r;
        if ((r = teb_noise_op(p, tr, w->p[0], w->p[1], w->p[2], bl, inv_noise_T, inv_noise_P, w->q[0], w->q[1], w->q[2], s, done))) return r;
        teb_apq_kernel<<<SV_GRID, SV_NT, 0, s>>>(*w, n);
        teb_update_kernel<<<SV_GRID, SV_NT, 0, s>>>(*w, x_T, x_E, x_B, n);
        teb_dir_kernel<<<SV_GRID, SV_NT, 0, s>>>(*w, n);
        GS_CHECK_LAUNCH();
        g_gs_launches += 3;
        return GS_OK;
    };
    return pcg_poll_loop(p, st, w->state, w->host_state, false, eps, itermax, check_every, iteration, n_iter_out, resid_out);
}

extern "C" int gs_cr_apply_q_teb(gs_plan* p, const double* dl_TT, const double* dl_TE, const double* dl_EE, const double* dl_BB,
                                 const double* bl, const double* inv_noise_T, const double* inv_noise_P, const double* x_T,
                                 const double* x_E, const double* x_B, double* y_T, double* y_E, double* y_B, void* stream)
{
    if (!p) { gs_set_error("null plan"); return GS_E_BADARG; }
    GS_REQUIRE(dl_TT && dl_TE && dl_EE && dl_BB && bl && inv_noise_T && inv_noise_P && x_T && x_E && x_B && y_T && y_E && y_B,
               "null pointer argument");
    int rc;
    if ((rc = teb_unsharded(p, __func__))) return rc;
    GS_CHECK_CUDA(cudaSetDevice(p->device));
    cudaStream_t st = (cudaStream_t)stream;
    TebWs* w = get_ws_teb(p);
    if (!w) return GS_E_NOMEM;
    const int L = p->d.lmax;
    teb_tables_kernel<<<(L + 256) / 256, 256, 0, st>>>(dl_TT, dl_TE, dl_EE, dl_BB, bl, 0.0, 0.0, L, w->tab);
    GS_CHECK_LAUNCH();
    TebRings tr(p);
    if ((rc = tr.begin(inv_noise_T, inv_noise_P, st))) return rc;
    if ((rc = teb_noise_op(p, tr, x_T, x_E, x_B, bl, inv_noise_T, inv_noise_P, w->q[0], w->q[1], w->q[2], st, nullptr))) return rc;
    teb_add_cinv_kernel<<<SV_GRID, SV_NT, 0, st>>>(*w, x_T, x_E, x_B, y_T, y_E, y_B, p->nreal_loc);
    GS_CHECK_LAUNCH();
    return GS_OK;
}

// b = B A^T N^-1 d + B (Npix/4pi) map2alm_{iter}(N^-1/2 xi_pix) + F xi_alm  (the two pixel terms as in gs_cr_rhs_tt / _pol)
extern "C" int gs_cr_rhs_teb(gs_plan* p, const double* dl_TT, const double* dl_TE, const double* dl_EE, const double* dl_BB,
                             const double* bl, const double* inv_noise_T, const double* sqrt_inv_noise_T, const double* inv_noise_P,
                             const double* sqrt_inv_noise_P, const double* bdata_T, const double* bdata_E, const double* bdata_B,
                             const double* d_I, const double* d_Q, const double* d_U, const double* xi_I, const double* xi_Q,
                             const double* xi_U, const double* xi_T, const double* xi_E, const double* xi_B, int fluct_iter,
                             double* rhs_T, double* rhs_E, double* rhs_B, void* stream)
{
    if (!p) { gs_set_error("null plan"); return GS_E_BADARG; }
    GS_REQUIRE(dl_TT && dl_TE && dl_EE && dl_BB && bl && inv_noise_T && sqrt_inv_noise_T && inv_noise_P && sqrt_inv_noise_P && xi_I &&
               xi_Q && xi_U && xi_T && xi_E && xi_B && rhs_T && rhs_E && rhs_B, "null pointer argument");
    GS_REQUIRE((bdata_T && bdata_E && bdata_B) || (d_I && d_Q && d_U), "need either the precomputed data terms or the data maps");
    GS_REQUIRE(fluct_iter >= 0, "fluct_iter must be >= 0");
    int rc;
    if ((rc = teb_unsharded(p, __func__))) return rc;
    GS_CHECK_CUDA(cudaSetDevice(p->device));
    cudaStream_t st = (cudaStream_t)stream;
    TebWs* w = get_ws_teb(p);
    if (!w) return GS_E_NOMEM;
    if ((rc = gs_map2alm_spin0(p, xi_I, sqrt_inv_noise_T, fluct_iter, 0, bl, rhs_T, GS_ALM_REAL, stream))) return rc;
    if ((rc = gs_map2alm_spin2(p, xi_Q, xi_U, sqrt_inv_noise_P, fluct_iter, 0, bl, rhs_E, rhs_B, GS_ALM_REAL, stream))) return rc;
    const double* bd[3] = {bdata_T, bdata_E, bdata_B};
    if (!bdata_T || !bdata_E || !bdata_B) {   // data terms into the r vectors of the workspace
        if ((rc = gs_map2alm_spin0(p, d_I, inv_noise_T, 0, 1, bl, w->r[0], GS_ALM_REAL, stream))) return rc;
        if ((rc = gs_map2alm_spin2(p, d_Q, d_U, inv_noise_P, 0, 1, bl, w->r[1], w->r[2], GS_ALM_REAL, stream))) return rc;
        for (int c = 0; c < 3; ++c) bd[c] = w->r[c];
    }
    const double resc = (double)p->d.npix / (4.0 * GS_PI);
    teb_rhs_combine_kernel<<<SV_GRID, SV_NT, 0, st>>>(w->lof, dl_TT, dl_TE, dl_EE, dl_BB, xi_T, xi_E, xi_B, bd[0], bd[1], bd[2], resc,
                                                      rhs_T, rhs_E, rhs_B, p->nreal_loc);
    GS_CHECK_LAUNCH();
    return GS_OK;
}

// Times the parts of one joint PCG iteration with CUDA events on `stream` (average of nrep, after one warm-up): ms_out[0] the
// spin-0 half of the mat-vec (N_T^-1), [1] the spin-2 half (N_P^-1), [2..4] the vector kernels teb_apq / teb_update / teb_dir on
// the joint workspace, zero-filled, with the analysis workspace overwritten before each (the arrays come from HBM, not L2).
// The vector kernels' reductions go to a scratch state, so no solver state changes.
extern "C" int gs_profile_matvec_teb(gs_plan* p, const double* bl, const double* inv_noise_T, const double* inv_noise_P, int nrep,
                                     float* ms_out, void* stream)
{
    if (!p) { gs_set_error("null plan"); return GS_E_BADARG; }
    GS_REQUIRE(bl && inv_noise_T && inv_noise_P && ms_out && nrep >= 1, "bad arguments");
    int rc;
    if ((rc = teb_unsharded(p, __func__))) return rc;
    GS_CHECK_CUDA(cudaSetDevice(p->device));
    cudaStream_t st = (cudaStream_t)stream;
    TebWs* w = get_ws_teb(p);
    if (!w) return GS_E_NOMEM;
    const int64_t n = p->nreal_loc;
    for (int c = 0; c < 3; ++c) {
        double* arrs[3] = {w->r[c], w->p[c], w->q[c]};
        for (double* a : arrs) GS_CHECK_CUDA(cudaMemsetAsync(a, 0, (size_t)n * sizeof(double), st));
    }
    GS_CHECK_CUDA(cudaMemsetAsync(w->tab, 0, (size_t)TEB_TAB * (p->d.lmax + 1) * sizeof(double), st));
    double* x[3] = {p->almE_tmp, p->almB_tmp, p->almE_tmp2};
    for (double* a : x) GS_CHECK_CUDA(cudaMemsetAsync(a, 0, (size_t)n * sizeof(double), st));
    PcgState* scratch = nullptr;
    GS_CHECK_CUDA(cudaMalloc(&scratch, sizeof(PcgState)));
    GS_CHECK_CUDA(cudaMemsetAsync(scratch, 0, sizeof(PcgState), st));
    TebWs v = *w;
    v.state = scratch;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    double acc[5] = {0, 0, 0, 0, 0};
    const size_t flush_bytes = (size_t)p->anal_chunks * (size_t)p->d.nalm * 4 * sizeof(double);
    {
        TebRings tr(p);
        rc = tr.begin(inv_noise_T, inv_noise_P, st);
        if (rc == GS_OK && (cudaEventCreate(&e0) != cudaSuccess || cudaEventCreate(&e1) != cudaSuccess)) rc = GS_E_CUDA;
        for (int k = 0; k < 5 && rc == GS_OK; ++k) {
            for (int rep = -1; rep < nrep && rc == GS_OK; ++rep) {
                // the flush, and a fresh scratch state: a reduction on zero vectors marks it converged, which would turn
                // every later launch into an early exit
                if (k >= 2 && (cudaMemsetAsync(p->partial, 0, flush_bytes, st) != cudaSuccess ||
                               cudaMemsetAsync(scratch, 0, sizeof(PcgState), st) != cudaSuccess)) { rc = GS_E_CUDA; break; }
                cudaEventRecord(e0, st);
                if (k == 0) {
                    if (tr.two) swap_flags(p);
                    rc = apply_noise_op(p, w->p[0], nullptr, bl, inv_noise_T, w->q[0], nullptr, st, nullptr, 0);
                    if (tr.two) swap_flags(p);
                } else if (k == 1) {
                    rc = apply_noise_op(p, w->p[1], w->p[2], bl, inv_noise_P, w->q[1], w->q[2], st, nullptr, 2);
                } else if (k == 2) {
                    teb_apq_kernel<<<SV_GRID, SV_NT, 0, st>>>(v, n);
                } else if (k == 3) {
                    teb_update_kernel<<<SV_GRID, SV_NT, 0, st>>>(v, x[0], x[1], x[2], n);
                } else {
                    teb_dir_kernel<<<SV_GRID, SV_NT, 0, st>>>(v, n);
                }
                cudaEventRecord(e1, st);
                if (cudaEventSynchronize(e1) != cudaSuccess) { rc = GS_E_CUDA; break; }
                float ms = 0;
                cudaEventElapsedTime(&ms, e0, e1);
                if (rep >= 0) acc[k] += ms;
            }
        }
    }
    if (rc == GS_E_CUDA) gs_set_error("gs_profile_matvec_teb: %s", cudaGetErrorString(cudaGetLastError()));
    for (int k = 0; k < 5; ++k) ms_out[k] = (float)(acc[k] / nrep);
    if (e0) cudaEventDestroy(e0);
    if (e1) cudaEventDestroy(e1);
    cudaFree(scratch);
    return rc;
}

// ------------------------------------------------------------------ measurement helpers (bench.py)
long long g_gs_launches = 0;
extern "C" long long gs_launch_count(void) { return g_gs_launches; }

// Times the stages of one PCG mat-vec with CUDA events on `st`, averaged over nrep: ms_out[0] Legendre synthesis, then the ring
// stage (split_ring: ring synthesis and ring analysis with N^-1 as two stages; otherwise the fused ring stage), then Legendre
// analysis + finish.  n_chain right-hand sides at x / y + c stride (doubles) per launch; the times are for the whole batch.
static int profile_matvec(gs_plan* p, int n_chain, int64_t stride, bool split_ring, const double* x_E, const double* x_B,
                          const double* bl, const double* inv_noise, double* y_E, double* y_B, int nrep, float* ms_out,
                          cudaStream_t st, const char* who)
{
    const int ns = split_ring ? 4 : 3;
    cudaEvent_t ev[5];
    for (int i = 0; i <= ns; ++i) GS_CHECK_CUDA(cudaEventCreate(&ev[i]));
    double acc[4] = {0, 0, 0, 0};
    int rc;
    {
        ActiveRings act(p);   // as in the PCG: rings without weight are skipped unless gs_set_ring_skip(0)
        rc = act.begin(inv_noise, st);
        for (int r = 0; r < nrep && rc == GS_OK; ++r) {
            int e = 0;
            cudaEventRecord(ev[e++], st);
            rc = gs_leg_synth(p, 2, x_E, x_B, GS_ALM_REAL, bl, st, nullptr, nullptr, n_chain, stride);
            cudaEventRecord(ev[e++], st);
            if (split_ring) {
                if (!rc) rc = gs_ring_synth(p, 2, p->mapQ_tmp, p->mapU_tmp, st);
                cudaEventRecord(ev[e++], st);
                if (!rc) rc = gs_ring_anal(p, 2, p->mapQ_tmp, p->mapU_tmp, inv_noise, st);
            } else if (!rc) {
                rc = gs_ring_apply(p, 2, inv_noise, st, nullptr, n_chain);
            }
            cudaEventRecord(ev[e++], st);
            if (!rc) rc = gs_leg_anal(p, 2, y_E, y_B, GS_ALM_REAL, bl, 1.0, 0, st, nullptr, n_chain, stride);
            cudaEventRecord(ev[e], st);
            if (cudaEventSynchronize(ev[e]) != cudaSuccess) { gs_set_error("%s: %s", who, cudaGetErrorString(cudaGetLastError())); rc = GS_E_CUDA; break; }
            for (int i = 0; i < ns; ++i) { float ms = 0; cudaEventElapsedTime(&ms, ev[i], ev[i + 1]); acc[i] += ms; }
        }
    }
    for (int i = 0; i < ns; ++i) ms_out[i] = (float)(acc[i] / nrep);
    for (int i = 0; i <= ns; ++i) cudaEventDestroy(ev[i]);
    return rc;
}

// Times the four kernels of one PCG mat-vec (Legendre synthesis, ring synthesis, ring analysis with
// fused N^-1, Legendre analysis + finish) with CUDA events on the launching stream; ms_out[0..3]
// receive the average duration of each stage over nrep repetitions.
extern "C" int gs_profile_matvec(gs_plan* p, const double* x_E, const double* x_B, const double* bl,
                                 const double* inv_noise, double* y_E, double* y_B, int nrep, float* ms_out,
                                 void* stream)
{
    if (!p) { gs_set_error("null plan"); return GS_E_BADARG; }
    GS_REQUIRE(x_E && x_B && bl && inv_noise && y_E && y_B && ms_out && nrep >= 1, "bad arguments");
    GS_CHECK_CUDA(cudaSetDevice(p->device));
    const int rc = profile_matvec(p, 1, 0, !g_gs_ring_fused, x_E, x_B, bl, inv_noise, y_E, y_B, nrep, ms_out, (cudaStream_t)stream,
                                  __func__);
    // fused ring stage (the PCG's own path): reported as stage 1, stage 2 = 0
    if (g_gs_ring_fused) { ms_out[3] = ms_out[2]; ms_out[2] = 0.0f; }
    return rc;
}

// gs_profile_matvec for a chain batch: n_chain (1 or 2) right-hand sides at x / y + c stride (doubles) per launch; the fused ring
// stage only.  ms_out[0] Legendre synthesis, [1] fused ring stage, [2] Legendre analysis + finish, each for the WHOLE batch.
extern "C" int gs_profile_matvec_batch(gs_plan* p, int n_chain, const double* x_E, const double* x_B, int64_t stride,
                                       const double* bl, const double* inv_noise, double* y_E, double* y_B, int nrep,
                                       float* ms_out, void* stream)
{
    if (!p) { gs_set_error("null plan"); return GS_E_BADARG; }
    GS_REQUIRE(x_E && x_B && bl && inv_noise && y_E && y_B && ms_out && nrep >= 1 && (n_chain == 1 || n_chain == 2), "bad arguments");
    GS_CHECK_CUDA(cudaSetDevice(p->device));
    int rc;
    if (n_chain > 1 && (rc = gs_plan_reserve_chains(p, n_chain))) return rc;
    return profile_matvec(p, n_chain, stride, false, x_E, x_B, bl, inv_noise, y_E, y_B, nrep, ms_out, (cudaStream_t)stream, __func__);
}

// Times the three vector kernels of one PCG iteration (q += C^-1 p with <p,q>; x, r update with <r,r>, <r,Mr>; p = M r + beta p)
// on the plan's own workspace, zero-filled, with CUDA events on `stream`: ms_out[0..2] = average of nrep launches each.  The
// reductions run as in the solver but their results go to a scratch buffer, so no solver state changes.
extern "C" int gs_profile_pcg_vectors(gs_plan* p, int spin, int nrep, float* ms_out, void* stream)
{
    if (!p) { gs_set_error("null plan"); return GS_E_BADARG; }
    GS_REQUIRE(ms_out && nrep >= 1 && (spin == 0 || spin == 2), "bad arguments");
    GS_CHECK_CUDA(cudaSetDevice(p->device));
    cudaStream_t st = (cudaStream_t)stream;
    gs_pcg_ws* w = get_ws(p);
    if (!w) return GS_E_NOMEM;
    const int nc = spin ? 2 : 1;
    const int64_t n = p->nreal_loc;
    for (int c = 0; c < 2; ++c) {
        double* arrs[3] = {w->r[c], w->p[c], w->q[c]};
        for (double* a : arrs) GS_CHECK_CUDA(cudaMemsetAsync(a, 0, (size_t)n * sizeof(double), st));
        double* tabs[2] = {w->ic_l[c], w->pre_l[c]};   // per-l tables
        for (double* a : tabs) GS_CHECK_CUDA(cudaMemsetAsync(a, 0, (size_t)(p->d.lmax + 1) * sizeof(double), st));
    }
    GS_CHECK_CUDA(cudaMemsetAsync(p->almE_tmp, 0, (size_t)n * sizeof(double), st));
    GS_CHECK_CUDA(cudaMemsetAsync(p->almB_tmp, 0, (size_t)n * sizeof(double), st));
    GS_CHECK_CUDA(cudaMemsetAsync(w->state, 0, sizeof(PcgState), st));
    double* red = nullptr;   // the reductions land here: the solver state (done flag, alpha, beta = 0) stays untouched
    GS_CHECK_CUDA(cudaMalloc(&red, 2 * sizeof(double)));
    gs_pcg_ws v = *w;
    v.red = red;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    int rc = GS_OK;
    if (cudaEventCreate(&e0) != cudaSuccess || cudaEventCreate(&e1) != cudaSuccess) rc = GS_E_CUDA;
    // between launches the analysis partials (> L2 at the bench size) are overwritten, as the Legendre / ring kernels do
    // between the vector kernels of a real iteration: the arrays come from HBM, not from the 126 MB L2
    const size_t flush_bytes = (size_t)p->anal_chunks * (size_t)(p->world > 1 ? p->d.sh.nalm_loc : p->d.nalm) * 4 * sizeof(double);
    for (int k = 0; k < 3 && rc == GS_OK; ++k) {
        double acc = 0.0;
        for (int rep = -2; rep < nrep; ++rep) {   // two warm-up launches
            if (cudaMemsetAsync(p->partial, 0, flush_bytes, st) != cudaSuccess) { rc = GS_E_CUDA; break; }
            cudaEventRecord(e0, st);
            if (k == 0) pcg_apq_kernel<<<SV_GRID, SV_NT, 0, st>>>(v, n, nc);
            else if (k == 1) pcg_update_kernel<<<SV_GRID, SV_NT, 0, st>>>(v, p->almE_tmp, p->almB_tmp, n, nc);
            else pcg_dir_kernel<<<SV_GRID, SV_NT, 0, st>>>(v, n, nc);
            cudaEventRecord(e1, st);
            if (cudaEventSynchronize(e1) != cudaSuccess) { rc = GS_E_CUDA; break; }
            float ms = 0;
            cudaEventElapsedTime(&ms, e0, e1);
            if (rep >= 0) acc += ms;
        }
        ms_out[k] = (float)(acc / nrep);
    }
    if (rc == GS_E_CUDA) gs_set_error("gs_profile_pcg_vectors: %s", cudaGetErrorString(cudaGetLastError()));
    if (e0) cudaEventDestroy(e0);
    if (e1) cudaEventDestroy(e1);
    cudaFree(red);
    if (rc) return rc;
    GS_CHECK_LAUNCH();
    return GS_OK;
}

// FP64 FMA throughput of the device (MEASURED_PEAKS.json holds no FP64 figure).  16 independent sums per thread in the
// operand pattern of the Legendre kernels, sum += x_k * y_j with register operands that change during the loop (three
// distinct register pairs per DFMA; scripts/ubench/dfma_operands.cu compares patterns: this one is the highest the pipe
// delivers, 36.9 TFLOP/s on B200 = 99 % of 148 x 64 x 2 x 1.965 GHz); 148 x 8 CTAs of 128 threads; TFLOP/s, best of 5.
__global__ void __launch_bounds__(128) dfma_peak_kernel(double* out, int iters, double a, double b)
{
    double v[16], w[4], u[4];
#pragma unroll
    for (int k = 0; k < 16; ++k) v[k] = threadIdx.x * 1e-3 + k;
#pragma unroll
    for (int k = 0; k < 4; ++k) { w[k] = a + 1e-9 * k; u[k] = b * (k + 1); }
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int k = 0; k < 16; ++k) v[k] = fma(w[k & 3], u[k >> 2], v[k]);
        w[i & 3] = fma(w[i & 3], a, b * 1e-30);   // keeps the multiplicands live (1 of 17 DFMAs, counted)
    }
    double s = 0;
#pragma unroll
    for (int k = 0; k < 16; ++k) s += v[k];
    if (s == 123.456) out[0] = s;
}

extern "C" int gs_measure_fp64_peak(double* tflops_out, void* stream)
{
    GS_REQUIRE(tflops_out, "null output");
    cudaStream_t st = (cudaStream_t)stream;
    double* d = nullptr;
    GS_CHECK_CUDA(cudaMalloc(&d, 8));
    cudaEvent_t e0, e1;
    GS_CHECK_CUDA(cudaEventCreate(&e0));
    GS_CHECK_CUDA(cudaEventCreate(&e1));
    const int iters = 1 << 14, grid = 148 * 8;
    double best = 0.0;
    for (int r = 0; r < 6; ++r) {
        cudaEventRecord(e0, st);
        dfma_peak_kernel<<<grid, 128, 0, st>>>(d, iters, 0.999999, 1e-9);
        cudaEventRecord(e1, st);
        GS_CHECK_CUDA(cudaEventSynchronize(e1));
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        const double tf = 2.0 * 17.0 * iters * (double)grid * 128.0 / (ms * 1e-3) * 1e-12;
        if (r > 0 && tf > best) best = tf;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(d);
    *tflops_out = best;
    return GS_OK;
}

extern "C" int gs_constant_rings(gs_plan* p, int* count_out)
{
    if (!p) { gs_set_error("null plan"); return GS_E_BADARG; }
    GS_REQUIRE(count_out, "null output");
    *count_out = 0;
    if (!p->ring_wconst) return GS_OK;   // sharded plans do not flag constant rings
    GS_CHECK_CUDA(cudaSetDevice(p->device));
    std::vector<double> w(p->d.nring);
    GS_CHECK_CUDA(cudaMemcpy(w.data(), p->ring_wconst, w.size() * sizeof(double), cudaMemcpyDeviceToHost));
    for (double v : w) *count_out += (v == v);
    return GS_OK;
}

extern "C" int gs_active_ring_pairs(gs_plan* p, int* active_out, int* total_out)
{
    if (!p) { gs_set_error("null plan"); return GS_E_BADARG; }
    GS_REQUIRE(active_out && total_out, "null output");
    GS_CHECK_CUDA(cudaSetDevice(p->device));
    GS_CHECK_CUDA(cudaMemcpy(active_out, p->act_count, sizeof(int), cudaMemcpyDeviceToHost));
    *total_out = p->d.npair;
    return GS_OK;
}
