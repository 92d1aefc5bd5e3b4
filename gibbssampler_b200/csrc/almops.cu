// Harmonic-space array utilities (HBM-bound, one pass each).  Replace the reference's
// variance_expension.pyx / utils.py helpers and the healpy per-l helpers (SURVEY.md 8a rows A3, A8, A11).
#include <algorithm>

#include "gs_internal.h"

#define EW_NT 256

static inline int ew_blocks(int64_t n) { return (int)std::min<int64_t>((n + EW_NT - 1) / EW_NT, 148 * 16); }

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

// l of entry i of the real layout ((L+1)^2 doubles)
__device__ __forceinline__ int l_of_real_index(int64_t i, int L)
{
    if (i <= L) return (int)i;
    int l, m;
    lm_of_index((i + L + 1) >> 1, L, l, m);
    return l;
}

// ---- utils.real_to_complex / complex_to_real (utils.py:49-76, variance_expension.pyx:65-100)
__global__ void real_to_complex_kernel(const double* __restrict__ r, double2* __restrict__ c, int L, int64_t nalm)
{
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < nalm; i += (int64_t)gridDim.x * blockDim.x) {
        if (i <= L) c[i] = make_double2(r[i], 0.0);
        else {
            const int64_t o = 2 * i - (L + 1);
            // utils.py:59 divides a complex array by np.sqrt(2): numpy's complex division multiplies by the
            // rounded reciprocal 1.0 / sqrt(2) (one ulp below the correctly rounded 1/sqrt2)
            const double scl = 1.0 / 1.4142135623730951;
            c[i] = make_double2(r[o] * scl, r[o + 1] * scl);
        }
    }
}

__global__ void complex_to_real_kernel(const double2* __restrict__ c, double* __restrict__ r, int L, int64_t nalm)
{
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < nalm; i += (int64_t)gridDim.x * blockDim.x) {
        const double2 v = c[i];
        if (i <= L) r[i] = v.x;
        else {
            const int64_t o = 2 * i - (L + 1);
            r[o] = v.x * 1.41421356237309504880;
            r[o + 1] = v.y * 1.41421356237309504880;
        }
    }
}

// ---- per-l array -> real layout.  mode 0: copy x_l (GibbsSampler.compute_bl_map, GibbsSampler.py:64-74,
// config.generate_var_cl config.py:75-84); mode 1: D_l -> C_l = D_l 2 pi / (l(l+1)), l = 0 copied
// (utils.generate_var_cl_cython utils.py:114-137, variance_expension.pyx:8-33); mode 2: 1/C_l where C_l != 0
// else 0; mode 3: sqrt(C_l); mode 4: sqrt(1/C_l) where C_l != 0 else 0.
__device__ __forceinline__ double per_l_value(const double* x, int l, int mode)
{
    double v = x[l];
    if (mode == 0) return v;
    if (l != 0) v = v * 2.0 * 3.14159265358979323846 / ((double)l * (double)(l + 1));
    if (mode == 1) return v;
    if (mode == 3) return sqrt(v);
    const double inv = (v != 0.0) ? 1.0 / v : 0.0;
    return mode == 2 ? inv : sqrt(inv);
}

__global__ void expand_per_l_kernel(const double* __restrict__ x, double* __restrict__ out, int L, int mode)
{
    const int64_t nre = (int64_t)(L + 1) * (L + 1);
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < nre; i += (int64_t)gridDim.x * blockDim.x)
        out[i] = per_l_value(x, l_of_real_index(i, L), mode);
}

// ---- utils.unfold_bins (utils.py:150-162): np.repeat(binned, diff(bins))
__global__ void unfold_bins_kernel(const double* __restrict__ binned, const int* __restrict__ bins, int nbins,
                                   double* __restrict__ out, int nout)
{
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < nout; i += gridDim.x * blockDim.x) {
        const int l = bins[0] + i;  // output position i corresponds to multipole bins[0] + i
        int lo = 0, hi = nbins - 1;
        while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (bins[mid] <= l) lo = mid; else hi = mid - 1; }
        out[i] = binned[lo];
    }
}

// ---- hp.almxfl: a_lm * f_l, either layout, out may alias in
__global__ void almxfl_kernel(const double* __restrict__ in, double* __restrict__ out, const double* __restrict__ fl, int L,
                              int layout, int64_t n, const int* __restrict__ lof)
{
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        if (layout == GS_ALM_REAL) out[i] = in[i] * fl[lof ? lof[i] : l_of_real_index(i, L)];
        else {
            int l, m;
            lm_of_index(i, L, l, m);
            const double f = fl[l];
            const double2 v = reinterpret_cast<const double2*>(in)[i];
            reinterpret_cast<double2*>(out)[i] = make_double2(v.x * f, v.y * f);
        }
    }
}

// ---- hp.alm2cl: one warp per l, lanes stride over m; deterministic shuffle reduction
__global__ void alm2cl_kernel(const double* __restrict__ alm, int layout, int L, double* __restrict__ cl)
{
    const int l = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (l > L) return;
    double s = 0.0;
    for (int m = lane; m <= l; m += 32) {
        const int64_t id = (int64_t)m * (2 * L + 1 - m) / 2 + l;
        if (layout == GS_ALM_COMPLEX) {
            const double2 v = reinterpret_cast<const double2*>(alm)[id];
            s += (m ? 2.0 : 1.0) * (v.x * v.x + v.y * v.y);
        } else if (m == 0) s += alm[l] * alm[l];
        else { const int64_t o = 2 * id - (L + 1); s += alm[o] * alm[o] + alm[o + 1] * alm[o + 1]; }
    }
    for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) cl[l] = s / (2.0 * l + 1.0);
}

// r = a * w - b  (residual map of the Jacobi-refined analysis); w nullable
__global__ void map_residual_kernel(const double* __restrict__ a, const double* __restrict__ w, const double* b, double* r,
                                    int64_t n)
{
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        r[i] = (w ? a[i] * w[i] : a[i]) - b[i];
}

// ------------------------------------------------------------------ C ABI
#define STREAM(s) ((cudaStream_t)(s))

extern "C" int gs_real_to_complex(const double* real_alm, double* complex_alm, int lmax, void* stream)
{
    GS_REQUIRE(real_alm && complex_alm && lmax >= 0, "bad arguments");
    const int64_t n = gs_nalm(lmax);
    real_to_complex_kernel<<<ew_blocks(n), EW_NT, 0, STREAM(stream)>>>(real_alm, (double2*)complex_alm, lmax, n);
    GS_CHECK_LAUNCH();
    return GS_OK;
}

extern "C" int gs_complex_to_real(const double* complex_alm, double* real_alm, int lmax, void* stream)
{
    GS_REQUIRE(real_alm && complex_alm && lmax >= 0, "bad arguments");
    const int64_t n = gs_nalm(lmax);
    complex_to_real_kernel<<<ew_blocks(n), EW_NT, 0, STREAM(stream)>>>((const double2*)complex_alm, real_alm, lmax, n);
    GS_CHECK_LAUNCH();
    return GS_OK;
}

int gs_launch_expand_per_l(const double* x, int lmax, int mode, double* out, cudaStream_t st)
{
    expand_per_l_kernel<<<ew_blocks((int64_t)(lmax + 1) * (lmax + 1)), EW_NT, 0, st>>>(x, out, lmax, mode);
    GS_CHECK_LAUNCH();
    return GS_OK;
}

extern "C" int gs_expand_per_l(const double* x, int lmax, int mode, double* out, void* stream)
{
    GS_REQUIRE(x && out && lmax >= 0 && mode >= 0 && mode <= 4, "bad arguments");
    expand_per_l_kernel<<<ew_blocks((int64_t)(lmax + 1) * (lmax + 1)), EW_NT, 0, STREAM(stream)>>>(x, out, lmax, mode);
    GS_CHECK_LAUNCH();
    return GS_OK;
}

extern "C" int gs_unfold_bins(const double* binned, const int* bins, int nbins, double* out, int nout, void* stream)
{
    GS_REQUIRE(binned && bins && out && nbins >= 1 && nout >= 0, "bad arguments");
    if (nout == 0) return GS_OK;
    unfold_bins_kernel<<<ew_blocks(nout), EW_NT, 0, STREAM(stream)>>>(binned, bins, nbins, out, nout);
    GS_CHECK_LAUNCH();
    return GS_OK;
}

extern "C" int gs_almxfl(const double* alm, int layout, int lmax, const double* fl, double* out, void* stream)
{
    GS_REQUIRE(alm && fl && out && lmax >= 0 && (layout == GS_ALM_COMPLEX || layout == GS_ALM_REAL), "bad arguments");
    const int64_t n = layout == GS_ALM_REAL ? (int64_t)(lmax + 1) * (lmax + 1) : gs_nalm(lmax);
    almxfl_kernel<<<ew_blocks(n), EW_NT, 0, STREAM(stream)>>>(alm, out, fl, lmax, layout, n, nullptr);
    GS_CHECK_LAUNCH();
    return GS_OK;
}

extern "C" int gs_alm2cl(const double* alm, int layout, int lmax, double* cl, void* stream)
{
    GS_REQUIRE(alm && cl && lmax >= 0 && (layout == GS_ALM_COMPLEX || layout == GS_ALM_REAL), "bad arguments");
    alm2cl_kernel<<<(lmax + 8) / 8, 256, 0, STREAM(stream)>>>(alm, layout, lmax, cl);
    GS_CHECK_LAUNCH();
    return GS_OK;
}

// ---- SHT entry points (compose the Legendre and ring stages)
static int check_plan(gs_plan* p)
{
    if (!p) { gs_set_error("null plan"); return GS_E_BADARG; }
    cudaError_t e = cudaSetDevice(p->device);
    if (e != cudaSuccess) { gs_set_error("cudaSetDevice: %s", cudaGetErrorString(e)); return GS_E_CUDA; }
    return GS_OK;
}

extern "C" int gs_alm2map_spin0(gs_plan* p, const double* alm, int layout, const double* fl, double* map, void* stream)
{
    int rc = check_plan(p);
    if (rc) return rc;
    GS_REQUIRE(alm && map && (layout == GS_ALM_COMPLEX || layout == GS_ALM_REAL), "bad arguments");
    if ((rc = gs_leg_synth(p, 0, alm, nullptr, layout, fl, STREAM(stream)))) return rc;
    return gs_ring_synth(p, 0, map, nullptr, STREAM(stream));
}

extern "C" int gs_alm2map_spin2(gs_plan* p, const double* almE, const double* almB, int layout, const double* fl,
                                double* mapQ, double* mapU, void* stream)
{
    int rc = check_plan(p);
    if (rc) return rc;
    GS_REQUIRE(almE && almB && mapQ && mapU && (layout == GS_ALM_COMPLEX || layout == GS_ALM_REAL), "bad arguments");
    if ((rc = gs_leg_synth(p, 2, almE, almB, layout, fl, STREAM(stream)))) return rc;
    return gs_ring_synth(p, 2, mapQ, mapU, STREAM(stream));
}

extern "C" int gs_alm2map_spin2_fl2(gs_plan* p, const double* almE, const double* almB, int layout, const double* flE,
                                    const double* flB, double* mapQ, double* mapU, void* stream)
{
    int rc = check_plan(p);
    if (rc) return rc;
    GS_REQUIRE(almE && almB && mapQ && mapU && flE && flB && (layout == GS_ALM_COMPLEX || layout == GS_ALM_REAL), "bad arguments");
    if ((rc = gs_leg_synth(p, 2, almE, almB, layout, flE, STREAM(stream), nullptr, flB))) return rc;
    return gs_ring_synth(p, 2, mapQ, mapU, STREAM(stream));
}

static int map2alm_impl(gs_plan* p, int spin, const double* mapQ, const double* mapU, const double* pixw, int iter,
                        int adjoint, const double* fl, double* almE, double* almB, int layout, cudaStream_t st)
{
    const double scale = adjoint ? 1.0 : 4.0 * 3.14159265358979323846 / (double)p->d.npix;
    if (adjoint) iter = 0;
    const double* fl0 = iter > 0 ? nullptr : fl;
    int rc;
    if ((rc = gs_ring_anal(p, spin, mapQ, mapU, pixw, st))) return rc;
    if ((rc = gs_leg_anal(p, spin, almE, almB, layout, fl0, scale, 0, st))) return rc;
    for (int it = 0; it < iter; ++it) {  // a += map2alm0(f - alm2map(a))
        if ((rc = gs_leg_synth(p, spin, almE, almB, layout, nullptr, st))) return rc;
        if ((rc = gs_ring_synth(p, spin, p->mapQ_tmp, p->mapU_tmp, st))) return rc;
        map_residual_kernel<<<ew_blocks(p->npix_loc), EW_NT, 0, st>>>(mapQ, pixw, p->mapQ_tmp, p->mapQ_tmp, p->npix_loc);
        if (spin) map_residual_kernel<<<ew_blocks(p->npix_loc), EW_NT, 0, st>>>(mapU, pixw, p->mapU_tmp, p->mapU_tmp, p->npix_loc);
        GS_CHECK_LAUNCH();
        if ((rc = gs_ring_anal(p, spin, p->mapQ_tmp, p->mapU_tmp, nullptr, st))) return rc;
        if ((rc = gs_leg_anal(p, spin, almE, almB, layout, nullptr, scale, 1, st))) return rc;
    }
    if (iter > 0 && fl) {
        const int64_t n = layout == GS_ALM_REAL ? p->nreal_loc : p->d.nalm;
        const int* lof = p->world > 1 ? p->d.sh.l_of_loc : nullptr;
        almxfl_kernel<<<ew_blocks(n), EW_NT, 0, st>>>(almE, almE, fl, p->d.lmax, layout, n, lof);
        if (spin) almxfl_kernel<<<ew_blocks(n), EW_NT, 0, st>>>(almB, almB, fl, p->d.lmax, layout, n, lof);
        GS_CHECK_LAUNCH();
    }
    return GS_OK;
}

extern "C" int gs_map2alm_spin0(gs_plan* p, const double* map, const double* pixw, int iter, int adjoint,
                                const double* fl, double* alm, int layout, void* stream)
{
    int rc = check_plan(p);
    if (rc) return rc;
    GS_REQUIRE(map && alm && iter >= 0 && (layout == GS_ALM_COMPLEX || layout == GS_ALM_REAL), "bad arguments");
    return map2alm_impl(p, 0, map, nullptr, pixw, iter, adjoint, fl, alm, nullptr, layout, STREAM(stream));
}

extern "C" int gs_map2alm_spin2(gs_plan* p, const double* mapQ, const double* mapU, const double* pixw, int iter,
                                int adjoint, const double* fl, double* almE, double* almB, int layout, void* stream)
{
    int rc = check_plan(p);
    if (rc) return rc;
    GS_REQUIRE(mapQ && mapU && almE && almB && iter >= 0 && (layout == GS_ALM_COMPLEX || layout == GS_ALM_REAL), "bad arguments");
    return map2alm_impl(p, 2, mapQ, mapU, pixw, iter, adjoint, fl, almE, almB, layout, STREAM(stream));
}

// ---- chain-batched SHTs (BASELINE config #5: "alm2map + map2alm ... batched over chains"; north_star (a))
// n_chain right-hand sides, chain c at alm + c alm_stride / map + c map_stride (strides in doubles), are transformed two per
// launch: the two chains of a pair share ONE Legendre recurrence per (ring pair, m) thread (4 + 8 K DFMA per ring pair and l
// instead of 12 K, K = 2); an odd last chain takes the single-chain kernels.  Same results as n_chain separate calls.
extern "C" int gs_alm2map_batch(gs_plan* p, int spin, int n_chain, const double* almE, const double* almB, int64_t alm_stride,
                                int layout, const double* fl, double* mapQ, double* mapU, int64_t map_stride, void* stream)
{
    int rc = check_plan(p);
    if (rc) return rc;
    GS_REQUIRE((spin == 0 || spin == 2) && n_chain >= 1 && almE && mapQ && (spin == 0 || (almB && mapU)) &&
               (layout == GS_ALM_COMPLEX || layout == GS_ALM_REAL), "bad arguments");
    if (n_chain > 1 && (rc = gs_plan_reserve_chains(p, 2))) return rc;
    cudaStream_t st = STREAM(stream);
    for (int c = 0; c < n_chain; c += 2) {
        const int nc = n_chain - c >= 2 ? 2 : 1;
        const double* e = almE + c * alm_stride;
        const double* b = spin ? almB + c * alm_stride : nullptr;
        double* q = mapQ + c * map_stride;
        double* u = spin ? mapU + c * map_stride : nullptr;
        if ((rc = gs_leg_synth(p, spin, e, b, layout, fl, st, nullptr, nullptr, nc, alm_stride))) return rc;
        if ((rc = gs_ring_synth(p, spin, q, u, st, nullptr, nc, map_stride))) return rc;
    }
    return GS_OK;
}

// map2alm(iter = 0) (adjoint = 0: weight 4 pi / Npix, adjoint = 1: A^T) of n_chain map sets; pixw (optional) multiplies the pixels
extern "C" int gs_map2alm_batch(gs_plan* p, int spin, int n_chain, const double* mapQ, const double* mapU, int64_t map_stride,
                                const double* pixw, int adjoint, const double* fl, double* almE, double* almB, int64_t alm_stride,
                                int layout, void* stream)
{
    int rc = check_plan(p);
    if (rc) return rc;
    GS_REQUIRE((spin == 0 || spin == 2) && n_chain >= 1 && almE && mapQ && (spin == 0 || (almB && mapU)) &&
               (layout == GS_ALM_COMPLEX || layout == GS_ALM_REAL), "bad arguments");
    if (n_chain > 1 && (rc = gs_plan_reserve_chains(p, 2))) return rc;
    cudaStream_t st = STREAM(stream);
    const double scale = adjoint ? 1.0 : 4.0 * 3.14159265358979323846 / (double)p->d.npix;
    for (int c = 0; c < n_chain; c += 2) {
        const int nc = n_chain - c >= 2 ? 2 : 1;
        const double* q = mapQ + c * map_stride;
        const double* u = spin ? mapU + c * map_stride : nullptr;
        double* e = almE + c * alm_stride;
        double* b = spin ? almB + c * alm_stride : nullptr;
        if ((rc = gs_ring_anal(p, spin, q, u, pixw, st, nullptr, nc, map_stride))) return rc;
        if ((rc = gs_leg_anal(p, spin, e, b, layout, fl, scale, 0, st, nullptr, nc, alm_stride))) return rc;
    }
    return GS_OK;
}
