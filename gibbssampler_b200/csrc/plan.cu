// Plan: HEALPix RING geometry, FP64 recurrence tables (computed on the host in long double),
// ring-FFT tables and workspace.  Replaces the geometry / sharp-plan setup hidden inside every
// hp.alm2map / hp.map2alm call of the reference (SURVEY.md 2.2).
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>

#include "gs_internal.h"

static thread_local char g_err[512] = "";

void gs_set_error(const char* fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

extern "C" const char* gs_last_error_string(void) { return g_err; }
extern "C" int gs_version(void) { return 100; }

static const long double PI_L = 3.14159265358979323846264338327950288L;

template <typename T>
static int upload(gs_plan* p, const std::vector<T>& h, const T** dptr)
{
    void* d = nullptr;
    size_t bytes = std::max<size_t>(h.size(), 1) * sizeof(T);
    GS_CHECK_CUDA(cudaMalloc(&d, bytes));
    p->owned.push_back(d);
    if (!h.empty()) GS_CHECK_CUDA(cudaMemcpy(d, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice));
    *dptr = (const T*)d;
    return GS_OK;
}

template <typename T>
static int dev_alloc(gs_plan* p, size_t count, T** dptr)
{
    void* d = nullptr;
    GS_CHECK_CUDA(cudaMalloc(&d, std::max<size_t>(count, 1) * sizeof(T)));
    p->owned.push_back(d);
    *dptr = (T*)d;
    return GS_OK;
}

static ScaledSeed to_seed(long double v)
{
    ScaledSeed s;
    int e = 0;
    long double m = frexpl(v, &e);
    s.mant = (double)m;
    s.ex = e;
    s.pad = 0;
    return s;
}

// Highest m whose lambda_lm (l <= lmax) is non-negligible at a ring with the given sin/cos(theta).
// Same functional form as the pruning rule of libsharp (lambda_lm is evanescent for
// m > l sin(theta)); verified against the unpruned CPU oracle in tests/test_sht_gpu.py.
static int mlim_of(int lmax, int spin, long double sth, long double cth)
{
    long double ofs = lmax * 0.01L;
    if (ofs < 100.0L) ofs = 100.0L;
    long double b = -2.0L * spin * fabsl(cth);
    long double t1 = lmax * sth + ofs;
    long double c = (long double)spin * spin - t1 * t1;
    long double discr = b * b - 4 * c;
    if (discr <= 0) return lmax;
    long double res = (-b + sqrtl(discr)) / 2.0L;
    if (res > lmax) res = lmax;
    return (int)(res + 0.5L);
}

static int build_tables(gs_plan* p)
{
    const int nside = p->d.nside, L = p->d.lmax;
    const int npair = 2 * nside, nring = 4 * nside - 1;
    const int64_t ns = nside, npix = 12 * ns * ns, ncap = 2 * ns * (ns - 1);
    p->d.npair = npair;
    p->d.nring = nring;
    p->d.npix = npix;
    p->d.nalm = gs_nalm(L);

    // ---- ring geometry (HEALPix RING scheme) ----
    std::vector<double> cth(npair), sth(npair), c2(npair), s2(npair);
    std::vector<int> mlim0(npair), mlim2(npair);
    std::vector<int> rn(nring), rq(nring), rden(nring);
    std::vector<int64_t> rstart(nring);
    for (int i = 1; i <= npair; ++i) {
        long double z, omz, st;
        int nphi, q, den;
        int64_t start;
        if (i < nside) {
            omz = (long double)i * i / (3.0L * ns * ns);
            z = 1.0L - omz;
            st = sqrtl(omz * (1.0L + z));
            nphi = 4 * i;
            q = 1;
            den = 4 * i;
            start = 2 * (int64_t)i * (i - 1);
        } else {
            z = 4.0L / 3.0L - 2.0L * i / (3.0L * ns);
            omz = 1.0L - z;
            st = sqrtl(omz * (1.0L + z));
            nphi = 4 * nside;
            // HEALPix pix2ang_ring: phi_j = (j - fodd) pi / (2 nside), fodd = 1/2 when (ring + nside) is even, else 1:
            // half-pixel shift on rings nside, nside + 2, ...; the other belt rings start at phi = 0
            q = (i - nside + 1) & 1;
            den = 4 * nside;
            start = ncap + (int64_t)(i - nside) * 4 * ns;
        }
        cth[i - 1] = (double)z;
        sth[i - 1] = (double)st;
        s2[i - 1] = (double)(0.5L * omz);
        c2[i - 1] = (double)(0.5L * (1.0L + z));
        mlim0[i - 1] = mlim_of(L, 0, st, z);
        mlim2[i - 1] = mlim_of(L, 2, st, z);
        rn[i - 1] = nphi; rq[i - 1] = q; rden[i - 1] = den; rstart[i - 1] = start;
        int is = 4 * nside - i;  // mirror ring (1-based)
        if (is != i) {
            rn[is - 1] = nphi; rq[is - 1] = q; rden[is - 1] = den;
            rstart[is - 1] = npix - start - nphi;
        }
    }
    int rc;
    if ((rc = upload(p, cth, &p->d.cth))) return rc;
    if ((rc = upload(p, sth, &p->d.sth))) return rc;
    if ((rc = upload(p, c2, &p->d.c2))) return rc;
    if ((rc = upload(p, s2, &p->d.s2))) return rc;
    if ((rc = upload(p, mlim0, &p->d.mlim0))) return rc;
    if ((rc = upload(p, mlim2, &p->d.mlim2))) return rc;
    {   // first ring pair (pole -> equator) that reaches a given m: the Legendre kernels pack the pairs from there on
        std::vector<int> pmin0(L + 1, npair), pmin2(L + 1, npair);
        for (int m = 0; m <= L; ++m) {
            for (int q = 0; q < npair; ++q) if (mlim0[q] >= m) { pmin0[m] = q; break; }
            for (int q = 0; q < npair; ++q) if (mlim2[q] >= m) { pmin2[m] = q; break; }
        }
        if ((rc = upload(p, pmin0, &p->d.pmin0))) return rc;
        if ((rc = upload(p, pmin2, &p->d.pmin2))) return rc;
    }
    if ((rc = upload(p, rn, &p->d.ring_nphi))) return rc;
    if ((rc = upload(p, rq, &p->d.ring_phq))) return rc;
    if ((rc = upload(p, rden, &p->d.ring_phden))) return rc;
    if ((rc = upload(p, rstart, &p->d.ring_start))) return rc;

    // ---- per-m seed factors ----
    std::vector<ScaledSeed> seed0(L + 1), seed2(L + 1);
    {
        long double v = 1.0L;  // prod_{k<=m} sqrt((2k-1)/(2k)) as v * 2^e
        int e = 0;
        for (int m = 0; m <= L; ++m) {
            if (m > 0) {
                v *= sqrtl((2.0L * m - 1.0L) / (2.0L * m));
                int t;
                v = frexpl(v, &t);
                e += t;
            }
            long double sgn = (m & 1) ? -1.0L : 1.0L;
            long double f0 = sgn * v * sqrtl((2.0L * m + 1.0L) / (4.0L * PI_L));
            seed0[m] = to_seed(f0);
            seed0[m].ex += e;
            long double f2 = 0.0L;
            if (m >= 2) f2 = f0 * sqrtl((long double)m * (m - 1) / ((long double)(m + 1) * (m + 2)));
            seed2[m] = to_seed(f2);
            seed2[m].ex += e;
        }
    }
    if ((rc = upload(p, seed0, &p->d.seed0))) return rc;
    if ((rc = upload(p, seed2, &p->d.seed2))) return rc;

    // ---- recurrence tables ----
    // lam_{l+1} = A_l (x - B_l) lam_l - C_l lam_{l-1}; with lam_l = alpha_l mu_l and
    // alpha_{l+1} = C_l alpha_{l-1}:  mu_{l+1} = (a_l x - b_l) mu_l - mu_{l-1},
    // a_l = A_l alpha_l / alpha_{l+1}, b_l = a_l B_l.  (two FMAs per step; alpha folded into a_lm)
    const int64_t nalm = p->d.nalm;
    std::vector<double> rec0(nalm, 0.0), alpha0(nalm, 0.0), alpha2(nalm, 0.0);
    std::vector<double2> rec2(nalm, make_double2(0.0, 0.0));
    for (int spin = 0; spin <= 2; spin += 2) {
        for (int m = 0; m <= L; ++m) {
            int l0 = std::max(m, spin);
            if (l0 > L) continue;
            int64_t base = (int64_t)m * (2 * L + 1 - m) / 2;
            long double a_prev = 1.0L, a_cur = 1.0L;  // alpha_{l-1}, alpha_l
            const long double mp = (long double)spin;   // |m'|
            for (int l = l0; l <= L; ++l) {
                if (spin == 0) alpha0[base + l] = (double)a_cur; else alpha2[base + l] = (double)a_cur;
                if (l == L) break;
                long double ll = l, L1 = l + 1.0L, mm = m;
                long double den = sqrtl((L1 * L1 - mm * mm) * (L1 * L1 - mp * mp));
                long double f = L1 * (2.0L * ll + 1.0L) / den;
                long double A = sqrtl((2.0L * ll + 3.0L) / (2.0L * ll + 1.0L)) * f;
                long double B = (l == 0) ? 0.0L : mm * mp / (ll * L1);
                long double a_next;
                if (l == l0) a_next = 1.0L;
                else {
                    long double Cc = sqrtl((2.0L * ll + 3.0L) / (2.0L * ll - 1.0L)) * f *
                                     sqrtl((ll * ll - mm * mm) * (ll * ll - mp * mp)) / (ll * (2.0L * ll + 1.0L));
                    a_next = Cc * a_prev;
                }
                long double a = A * a_cur / a_next;
                if (spin == 0) rec0[base + l] = (double)a;
                else rec2[base + l] = make_double2((double)a, (double)(a * B));
                a_prev = a_cur;
                a_cur = a_next;
            }
        }
    }
    if ((rc = upload(p, rec0, &p->d.rec0))) return rc;
    if ((rc = upload(p, alpha0, &p->d.alpha0))) return rc;
    if ((rc = upload(p, rec2, &p->d.rec2))) return rc;
    if ((rc = upload(p, alpha2, &p->d.alpha2))) return rc;
    return GS_OK;
}

static int plan_create_impl(gs_plan** out, int nside, int lmax, int device, int rank, int world, const char* nccl_id,
                            void* lgroup = nullptr)
{
    if (!out) { gs_set_error("gs_plan_create: null output"); return GS_E_BADARG; }
    *out = nullptr;
    // the ring stage takes a ring whole or as four sub-transforms of n/4 points (ringfft.cu, gs_ring_setup).  A belt ring's
    // quarter has nside points; unless that is a power of two it runs as a Bluestein transform of next_pow2(2 nside - 1)
    // points, and one CTA holds at most 4096: nside <= 2048.  Refused here, before any table is built on the device.
    GS_REQUIRE(nside >= 1 && nside <= GS_NSIDE_MAX, "nside out of range [1, 2048]: rings longer than 8192 pixels need a deeper ring split");
    GS_REQUIRE(lmax >= 2 && lmax <= 4 * nside, "lmax must satisfy 2 <= lmax <= 4 nside");
    GS_REQUIRE(world >= 1 && rank >= 0 && rank < world, "need 0 <= rank < world");
    GS_REQUIRE(world <= 2 * nside && world <= (lmax + 2) / 2, "more ranks than ring pairs or m pairs");
    if (device >= 0) GS_CHECK_CUDA(cudaSetDevice(device));
    int dev = 0;
    GS_CHECK_CUDA(cudaGetDevice(&dev));
    gs_plan* p = new gs_plan();
    memset(&p->d, 0, sizeof(p->d));
    p->device = dev;
    p->d.nside = nside;
    p->d.lmax = lmax;
    p->jobs0 = p->jobs2 = nullptr;
    p->groups0 = p->groups2 = nullptr;
    p->groups0_dyn = p->groups2_dyn = nullptr;
    p->ngroups0 = p->ngroups2 = 0;
    p->sjobs0 = p->sjobs2 = nullptr;
    p->nsjobs0 = p->nsjobs2 = 0;
    p->ring_scratch = nullptr;
    p->act_ring = nullptr;
    p->ring_wconst = nullptr;
    p->act_pairs = nullptr;
    p->act_count = nullptr;
    p->act_slot0 = nullptr;
    p->act_red = nullptr;
    p->use_act = false;
    p->mwg_F = nullptr;
    p->mwg_maps = nullptr;
    p->mwg_group = 0;
    p->mwg_small = nullptr;
    p->mwg_data = nullptr;
    p->mwg_meta = nullptr;
    p->world = world;
    p->rank = rank;
    p->comm = nullptr;
    p->lgroup = lgroup;
    p->pcg_ws = nullptr;
    p->pcg_ws_batch = nullptr;
    p->pcg_alldone = nullptr;
    p->pcg_ws_teb = nullptr;
    memset(&p->flags_T, 0, sizeof(p->flags_T));
    p->work_stream = nullptr;
    p->work_event = nullptr;
    p->comm_stream = nullptr;
    p->chain_cap = 1;
    p->Fx = nullptr;
    p->red_loc = nullptr;
    p->d.sh.world = 1;
    int rc = build_tables(p);
    if (rc == GS_OK) rc = gs_leg_build_sinpow(p);
    if (rc == GS_OK) rc = gs_leg_prepare(p);
    const int64_t nm = lmax + 1;
    p->nreal_loc = nm * nm;
    p->npix_loc = p->d.npix;
    if (rc == GS_OK && world > 1) rc = gs_shard_build(p, rank, world, nccl_id);
    if (rc == GS_OK) rc = gs_ring_setup(p);
    if (rc == GS_OK) {
        const size_t nfm = world > 1 ? (size_t)world * 2 * p->d.sh.RL * p->d.sh.ML : (size_t)2 * p->d.nring * nm;   // ML = NB MLb
        rc = dev_alloc(p, nfm, &p->Fm);
        if (rc == GS_OK && world > 1) rc = dev_alloc(p, nfm, &p->Fx);
        // the padding entries of the spectra buffers are exchanged but never read; keep them finite
        if (rc == GS_OK) cudaMemset(p->Fm, 0, nfm * sizeof(double2));
        if (rc == GS_OK && world > 1) cudaMemset(p->Fx, 0, nfm * sizeof(double2));
        // analysis: ring pairs are split in chunks of >= 128 per block (see legendre.cu)
        p->anal_chunks = (p->d.npair + 127) / 128;
        const size_t nalm_part = world > 1 ? (size_t)p->d.sh.nalm_loc : (size_t)p->d.nalm;
        if (rc == GS_OK) rc = dev_alloc(p, (size_t)p->anal_chunks * nalm_part * 4, &p->partial);
        if (rc == GS_OK) rc = dev_alloc(p, (size_t)p->d.nring, &p->act_ring);
        if (rc == GS_OK) rc = dev_alloc(p, (size_t)p->d.npair, &p->act_pairs);
        if (rc == GS_OK) rc = dev_alloc(p, (size_t)1, &p->act_count);
        if (rc == GS_OK) rc = dev_alloc(p, (size_t)2 * (lmax + 1), &p->act_slot0);
        if (rc == GS_OK) rc = dev_alloc(p, (size_t)p->d.nring, &p->act_red);
        if (rc == GS_OK && world <= 1) rc = dev_alloc(p, (size_t)p->d.nring, &p->ring_wconst);
        if (rc == GS_OK) rc = dev_alloc(p, (size_t)p->npix_loc, &p->mapQ_tmp);
        if (rc == GS_OK) rc = dev_alloc(p, (size_t)p->npix_loc, &p->mapU_tmp);
        const size_t nre = (size_t)p->nreal_loc;  // big enough for either layout
        if (rc == GS_OK) rc = dev_alloc(p, nre, &p->almE_tmp);
        if (rc == GS_OK) rc = dev_alloc(p, nre, &p->almB_tmp);
        if (rc == GS_OK) rc = dev_alloc(p, nre, &p->almE_tmp2);
        if (rc == GS_OK) rc = dev_alloc(p, nre, &p->almB_tmp2);
    }
    if (rc == GS_OK) {
        cudaError_t e = cudaDeviceSynchronize();
        if (e != cudaSuccess) { gs_set_error("plan setup: %s", cudaGetErrorString(e)); rc = GS_E_CUDA; }
    }
    if (rc != GS_OK) { gs_plan_destroy(p); return rc; }
    *out = p;
    return GS_OK;
}

extern "C" int gs_plan_create(gs_plan** out, int nside, int lmax, int device)
{
    return plan_create_impl(out, nside, lmax, device, 0, 1, nullptr);
}

extern "C" int gs_plan_create_sharded(gs_plan** out, int nside, int lmax, int device, int rank, int world,
                                      const char* nccl_id128_host)
{
    return plan_create_impl(out, nside, lmax, device, rank, world, nccl_id128_host);
}

extern "C" int gs_plan_create_sharded_local(gs_plan** out, int nside, int lmax, int device, int rank, int world,
                                            void* local_group)
{
    if (!local_group) { gs_set_error("null local group"); return GS_E_BADARG; }
    return plan_create_impl(out, nside, lmax, device, rank, world, nullptr, local_group);
}

// Chain batches (BASELINE config #5 "batched over chains", north_star (a)): size the ring-spectra and analysis partial-sum
// buffers for n_chain right-hand sides that share one Legendre recurrence per launch.  Unsharded plans, n_chain <= 2 per launch.
extern "C" int gs_plan_reserve_chains(gs_plan* p, int n_chain)
{
    if (!p) { gs_set_error("null plan"); return GS_E_BADARG; }
    GS_REQUIRE(n_chain >= 1 && n_chain <= 2, "n_chain must be 1 or 2");
    GS_REQUIRE(p->world == 1, "chain batches need an unsharded plan");
    if (n_chain <= p->chain_cap) return GS_OK;
    GS_CHECK_CUDA(cudaSetDevice(p->device));
    const int64_t nm = p->d.lmax + 1;
    const size_t nfm = (size_t)n_chain * 2 * p->d.nring * nm;
    double2* F = nullptr;
    int rc = dev_alloc(p, nfm, &F);
    if (rc) return rc;
    GS_CHECK_CUDA(cudaMemset(F, 0, nfm * sizeof(double2)));
    // every chain of a batch takes ceil(npair / 256) chunks of partial sums (legendre.cu: LEG_NT * LEG_RA2 ring pairs per chunk)
    const int chunks = std::max(p->anal_chunks, n_chain * ((p->d.npair + 255) / 256));
    double* part = nullptr;
    if (chunks > p->anal_chunks) {
        rc = dev_alloc(p, (size_t)chunks * p->d.nalm * 4, &part);
        if (rc) return rc;
        p->partial = part;
        p->anal_chunks = chunks;
    }
    GS_CHECK_CUDA(cudaDeviceSynchronize());
    p->Fm = F;   // the single-chain buffer stays in p->owned until the plan is destroyed
    p->chain_cap = n_chain;
    return GS_OK;
}

extern "C" int gs_plan_destroy(gs_plan* p)
{
    if (!p) return GS_OK;
    gs_pcg_ws_free(p);
    gs_shard_free(p);
    for (void* e : p->comm_events) cudaEventDestroy((cudaEvent_t)e);
    if (p->comm_stream) cudaStreamDestroy((cudaStream_t)p->comm_stream);
    if (p->work_event) cudaEventDestroy((cudaEvent_t)p->work_event);
    if (p->work_stream) cudaStreamDestroy((cudaStream_t)p->work_stream);
    for (void* d : p->owned) cudaFree(d);
    for (void* h : p->owned_host) cudaFreeHost(h);
    cudaFree(p->mwg_F);
    cudaFree(p->mwg_maps);
    cudaFree(p->mwg_small);
    cudaFree(p->mwg_data);
    cudaFree(p->mwg_meta);
    delete p;
    return GS_OK;
}

extern "C" int gs_plan_nside(const gs_plan* p) { return p ? p->d.nside : 0; }
extern "C" int gs_plan_lmax(const gs_plan* p) { return p ? p->d.lmax : 0; }
extern "C" int64_t gs_plan_npix(const gs_plan* p) { return p ? p->d.npix : 0; }
extern "C" int64_t gs_plan_nalm(const gs_plan* p) { return p ? p->d.nalm : 0; }
extern "C" int64_t gs_plan_nreal(const gs_plan* p) { return p ? (int64_t)(p->d.lmax + 1) * (p->d.lmax + 1) : 0; }
