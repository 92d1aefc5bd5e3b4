// m-sharded spherical-harmonic transforms over the GPUs of one node (SURVEY.md 8e row 2, BASELINE config #4).
//
// The reference runs one chain per SLURM task and has no multi-GPU transform; this is the single-chain
// strategy for NSIDE >= 1024: the Legendre stage is partitioned over m, the ring-FFT / pixel stage over
// ring pairs, and the ring spectra F_m(theta_r) are transposed between the two partitions by ONE all-to-all
// of equal-sized chunks per transform (NCCL grouped send/recv over NVLink).  alm vectors stay m-sharded
// in a compact local real layout, maps (data, N^-1, mask) stay ring-sharded, the PCG dot products are a
// 2-scalar all-reduce per reduction.
//
// Partition (pure functions of (nside, lmax, world), identical on every rank):
//   m     : pairs {j, L - j}, j < ceil((L+1)/2), have constant Legendre cost -> pair j goes to rank j mod W
//   rings : ring pair p (north ring p, south ring nring-1-p; N/S kept together for the parity trick)
//           goes to rank p mod W, which balances the ring lengths of the polar caps
// NCCL is resolved at run time (dlopen of the libnccl.so.2 that torch already loaded), so the library has
// no link-time dependency and single-GPU use never touches it.
#include <dlfcn.h>
#include <nccl.h>
#include <pthread.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "gs_internal.h"
#include "spectra.cuh"

// ---------------------------------------------------------------- NCCL, resolved lazily
namespace {
struct NcclApi {
    ncclResult_t (*GetUniqueId)(ncclUniqueId*);
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int);
    ncclResult_t (*CommDestroy)(ncclComm_t);
    ncclResult_t (*GroupStart)();
    ncclResult_t (*GroupEnd)();
    ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t);
    ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t);
    ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t);
    const char* (*GetErrorString)(ncclResult_t);
    bool ok;
};
NcclApi g_nccl = {};

bool nccl_load()
{
    if (g_nccl.ok) return true;
    void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);  // torch's copy when it is already in the process
    if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!h) { gs_set_error("NCCL not found: %s", dlerror()); return false; }
#define GS_SYM(field, name)                                                         \
    *(void**)(&g_nccl.field) = dlsym(h, name);                                      \
    if (!g_nccl.field) { gs_set_error("NCCL symbol %s missing", name); return false; }
    GS_SYM(GetUniqueId, "ncclGetUniqueId")
    GS_SYM(CommInitRank, "ncclCommInitRank")
    GS_SYM(CommDestroy, "ncclCommDestroy")
    GS_SYM(GroupStart, "ncclGroupStart")
    GS_SYM(GroupEnd, "ncclGroupEnd")
    GS_SYM(Send, "ncclSend")
    GS_SYM(Recv, "ncclRecv")
    GS_SYM(AllReduce, "ncclAllReduce")
    GS_SYM(GetErrorString, "ncclGetErrorString")
#undef GS_SYM
    g_nccl.ok = true;
    return true;
}
}  // namespace

#define GS_CHECK_NCCL(expr)                                                                      \
    do {                                                                                         \
        ncclResult_t _r = (expr);                                                                \
        if (_r != ncclSuccess) {                                                                 \
            gs_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, g_nccl.GetErrorString(_r)); \
            return GS_E_NCCL;                                                                    \
        }                                                                                        \
    } while (0)

// ---------------------------------------------------------------- in-process group (tests on ONE GPU)
// `world` sharded plans on the same device, each driven by its own host thread and stream.  The all-to-all
// is a host barrier + device-to-device copies, the all-reduce a host barrier + a fixed-order sum, so the
// sharded kernels, the sharded PCG and their index tables can be verified on a single-GPU box.  Not a
// performance path: production groups are NCCL communicators (one process per GPU).
struct gs_local_group {
    int world;
    pthread_barrier_t bar;
    std::vector<const double2*> send;
    std::vector<std::vector<double>> red;
};

extern "C" int gs_local_group_create(void** out, int world)
{
    GS_REQUIRE(out && world >= 1, "bad arguments");
    gs_local_group* g = new gs_local_group();
    g->world = world;
    pthread_barrier_init(&g->bar, nullptr, (unsigned)world);
    g->send.assign(world, nullptr);
    g->red.assign(world, std::vector<double>());
    *out = g;
    return GS_OK;
}

extern "C" int gs_local_group_destroy(void* group)
{
    gs_local_group* g = (gs_local_group*)group;
    if (!g) return GS_OK;
    pthread_barrier_destroy(&g->bar);
    delete g;
    return GS_OK;
}

static int local_exchange(gs_plan* p, const double2* send, double2* recv, int blk, cudaStream_t st)
{
    gs_local_group* g = (gs_local_group*)p->lgroup;
    const ShardDev& S = p->d.sh;
    const size_t chunk = (size_t)2 * S.RL * S.MLb, b0 = (size_t)blk * S.world * chunk;
    GS_CHECK_CUDA(cudaStreamSynchronize(st));
    g->send[S.rank] = send;
    pthread_barrier_wait(&g->bar);
    for (int r = 0; r < S.world; ++r)
        GS_CHECK_CUDA(cudaMemcpyAsync(recv + b0 + r * chunk, g->send[r] + b0 + S.rank * chunk, chunk * sizeof(double2), cudaMemcpyDeviceToDevice, st));
    GS_CHECK_CUDA(cudaStreamSynchronize(st));
    pthread_barrier_wait(&g->bar);
    return GS_OK;
}

static int local_allreduce(gs_plan* p, double* buf, int n, cudaStream_t st)
{
    gs_local_group* g = (gs_local_group*)p->lgroup;
    const int rank = p->d.sh.rank;
    g->red[rank].resize(n);
    GS_CHECK_CUDA(cudaMemcpyAsync(g->red[rank].data(), buf, n * sizeof(double), cudaMemcpyDeviceToHost, st));
    GS_CHECK_CUDA(cudaStreamSynchronize(st));
    pthread_barrier_wait(&g->bar);
    std::vector<double> tot(n, 0.0);
    for (int r = 0; r < g->world; ++r) for (int i = 0; i < n; ++i) tot[i] += g->red[r][i];
    GS_CHECK_CUDA(cudaMemcpyAsync(buf, tot.data(), n * sizeof(double), cudaMemcpyHostToDevice, st));
    GS_CHECK_CUDA(cudaStreamSynchronize(st));
    pthread_barrier_wait(&g->bar);
    return GS_OK;
}

// ---------------------------------------------------------------- partition (host, no GPU needed)
static int ring_nphi_of(int nside, int ring)  // 0-based ring
{
    const int i = std::min(ring + 1, 4 * nside - (ring + 1));
    return i < nside ? 4 * i : 4 * nside;
}

extern "C" int gs_shard_partition_m(int lmax, int world, int rank, int* out)
{
    if (lmax < 0 || world < 1 || rank < 0 || rank >= world) return GS_E_BADARG;
    std::vector<int> v;
    const int npairs = (lmax + 2) / 2;  // ceil((L+1)/2)
    for (int j = rank; j < npairs; j += world) {
        v.push_back(j);
        if (lmax - j != j) v.push_back(lmax - j);
    }
    std::sort(v.begin(), v.end());
    if (out) std::copy(v.begin(), v.end(), out);
    return (int)v.size();
}

extern "C" int gs_shard_partition_rings(int nside, int world, int rank, int* out)
{
    if (nside < 1 || world < 1 || rank < 0 || rank >= world) return GS_E_BADARG;
    const int npair = 2 * nside, nring = 4 * nside - 1;
    std::vector<int> v;
    for (int p = rank; p < npair; p += world) {
        v.push_back(p);
        if (nring - 1 - p != p) v.push_back(nring - 1 - p);
    }
    std::sort(v.begin(), v.end());
    if (out) std::copy(v.begin(), v.end(), out);
    return (int)v.size();
}

// global real-layout index ((L+1)^2 numbering, utils.py:49-76) of every entry of rank's local real layout:
// owned m ascending; m = 0 contributes l = 0..L, m > 0 contributes (sqrt2 Re, sqrt2 Im) for l = m..L
extern "C" int64_t gs_shard_real_index(int lmax, int world, int rank, int64_t* out)
{
    const int nm = gs_shard_partition_m(lmax, world, rank, nullptr);
    if (nm < 0) return nm;
    std::vector<int> ml(nm);
    gs_shard_partition_m(lmax, world, rank, ml.data());
    int64_t n = 0;
    for (int m : ml) {
        const int64_t base = (int64_t)m * (2 * lmax + 1 - m) / 2;
        for (int l = m; l <= lmax; ++l) {
            if (m == 0) { if (out) out[n] = l; n += 1; }
            else {
                const int64_t o = 2 * (base + l) - (lmax + 1);
                if (out) { out[n] = o; out[n + 1] = o + 1; }
                n += 2;
            }
        }
    }
    return n;
}

// global RING pixel index of every pixel of rank's local map (owned rings ascending)
extern "C" int64_t gs_shard_pixel_index(int nside, int world, int rank, int64_t* out)
{
    const int nr = gs_shard_partition_rings(nside, world, rank, nullptr);
    if (nr < 0) return nr;
    std::vector<int> rl(nr);
    gs_shard_partition_rings(nside, world, rank, rl.data());
    const int nring = 4 * nside - 1;
    std::vector<int64_t> start(nring + 1, 0);
    for (int r = 0; r < nring; ++r) start[r + 1] = start[r] + ring_nphi_of(nside, r);
    int64_t n = 0;
    for (int r : rl) {
        const int np = ring_nphi_of(nside, r);
        if (out) for (int j = 0; j < np; ++j) out[n + j] = start[r] + j;
        n += np;
    }
    return n;
}

template <typename T>
static int up(gs_plan* p, const std::vector<T>& h, const T** dptr)
{
    void* d = nullptr;
    GS_CHECK_CUDA(cudaMalloc(&d, std::max<size_t>(h.size(), 1) * sizeof(T)));
    p->owned.push_back(d);
    if (!h.empty()) GS_CHECK_CUDA(cudaMemcpy(d, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice));
    *dptr = (const T*)d;
    return GS_OK;
}

// Fills p->d.sh, the host lists and the communicator.  Called by gs_plan_create_sharded after the
// geometry tables exist and before the ring job lists are built.
int gs_shard_build(gs_plan* p, int rank, int world, const char* nccl_id)
{
    const int L = p->d.lmax, nside = p->d.nside, nring = p->d.nring;
    ShardDev& S = p->d.sh;
    S.world = world;
    S.rank = rank;
    std::vector<int> m_owner(L + 1), m_loc(L + 1), ring_owner(nring), ring_loc(nring);
    std::vector<int64_t> ring_start_loc(nring);
    int ML = 0, RL = 0;
    for (int r = 0; r < world; ++r) {
        std::vector<int> ml(gs_shard_partition_m(L, world, r, nullptr));
        gs_shard_partition_m(L, world, r, ml.data());
        for (size_t k = 0; k < ml.size(); ++k) { m_owner[ml[k]] = r; m_loc[ml[k]] = (int)k; }
        ML = std::max(ML, (int)ml.size());
        std::vector<int> rl(gs_shard_partition_rings(nside, world, r, nullptr));
        gs_shard_partition_rings(nside, world, r, rl.data());
        int64_t off = 0;
        for (size_t k = 0; k < rl.size(); ++k) {
            ring_owner[rl[k]] = r; ring_loc[rl[k]] = (int)k; ring_start_loc[rl[k]] = off;
            off += ring_nphi_of(nside, rl[k]);
        }
        RL = std::max(RL, (int)rl.size());
        if (r == rank) { p->h_mlist = ml; p->h_rings = rl; p->npix_loc = off; }
    }
    // blocks of m for the pipelined all-to-all (GS_SHARD_NB = 1..16).  Default 1 = one exchange per transform: measured on 2 B200 at
    // NSIDE 1024 / lmax 2048 the pipeline with 4 blocks is SLOWER (SHT pair 4.45 vs 4.24 ms; the all-to-all alone 0.32 vs 0.23 ms):
    // the exposed exchange is ~5 % per direction, less than what four Legendre launches (four tails) sharing the SMs with the NCCL
    // kernels cost.  The blocked layout and the stream / event pipeline stay available for larger worlds or slower links.
    int NB = 1;
    if (const char* e = getenv("GS_SHARD_NB")) { const int v = atoi(e); if (v >= 1 && v <= 16) NB = std::min(v, std::max(ML, 1)); }
    const int MLb = (ML + NB - 1) / NB;
    S.NB = NB;
    S.MLb = MLb;
    S.ML = NB * MLb;
    S.RL = RL;
    S.nm_loc = (int)p->h_mlist.size();
    std::vector<int64_t> m_base(L + 1);
    for (int m = 0; m <= L; ++m) {
        const int blk = m_loc[m] / MLb, w = m_loc[m] - blk * MLb;
        m_base[m] = (((int64_t)blk * world + m_owner[m]) * 2 * RL) * MLb + w;
    }
    std::vector<int64_t> cbase(S.nm_loc), rbase(S.nm_loc);
    std::vector<int> lof;
    int64_t nc = 0, nr = 0;
    for (int k = 0; k < S.nm_loc; ++k) {
        const int m = p->h_mlist[k];
        cbase[k] = nc; rbase[k] = nr;
        nc += L - m + 1;
        nr += (m ? 2 : 1) * (int64_t)(L - m + 1);
        for (int l = m; l <= L; ++l) { lof.push_back(l); if (m) lof.push_back(l); }
    }
    S.nalm_loc = nc;
    p->nreal_loc = nr;
    int rc;
    if ((rc = up(p, p->h_mlist, &S.mlist))) return rc;
    if ((rc = up(p, cbase, &S.cbase))) return rc;
    if ((rc = up(p, rbase, &S.rbase))) return rc;
    if ((rc = up(p, m_owner, &S.m_owner))) return rc;
    if ((rc = up(p, m_loc, &S.m_loc))) return rc;
    if ((rc = up(p, m_base, &S.m_base))) return rc;
    if ((rc = up(p, ring_owner, &S.ring_owner))) return rc;
    if ((rc = up(p, ring_loc, &S.ring_loc))) return rc;
    if ((rc = up(p, ring_start_loc, &S.ring_start_loc))) return rc;
    if ((rc = up(p, lof, &S.l_of_loc))) return rc;
    void* d = nullptr;
    GS_CHECK_CUDA(cudaMalloc(&d, 8 * sizeof(double)));
    p->owned.push_back(d);
    p->red_loc = (double*)d;

    if (p->lgroup) return GS_OK;  // in-process group: no communicator
    if (!nccl_load()) return GS_E_NCCL;
    if (!nccl_id) { gs_set_error("sharded plan needs the NCCL unique id of the group"); return GS_E_BADARG; }
    ncclUniqueId id;
    static_assert(sizeof(id) == 128, "ncclUniqueId is 128 bytes");
    memcpy(&id, nccl_id, sizeof(id));
    ncclComm_t comm = nullptr;
    GS_CHECK_NCCL(g_nccl.CommInitRank(&comm, world, id, rank));
    p->comm = comm;
    return GS_OK;
}

void gs_shard_free(gs_plan* p)
{
    if (p->comm && g_nccl.ok) g_nccl.CommDestroy((ncclComm_t)p->comm);
    p->comm = nullptr;
}

int gs_shard_exchange_block(gs_plan* p, const double2* send, double2* recv, int blk, cudaStream_t st)
{
    if (p->lgroup) return local_exchange(p, send, recv, blk, st);
    const ShardDev& S = p->d.sh;
    const size_t chunk = (size_t)2 * S.RL * S.MLb, b0 = (size_t)blk * S.world * chunk;  // double2 per peer and block
    ncclComm_t comm = (ncclComm_t)p->comm;
    GS_CHECK_NCCL(g_nccl.GroupStart());
    for (int r = 0; r < S.world; ++r) {
        GS_CHECK_NCCL(g_nccl.Send(send + b0 + r * chunk, 2 * chunk, ncclDouble, r, comm, st));
        GS_CHECK_NCCL(g_nccl.Recv(recv + b0 + r * chunk, 2 * chunk, ncclDouble, r, comm, st));
    }
    GS_CHECK_NCCL(g_nccl.GroupEnd());
    return GS_OK;
}

int gs_shard_exchange(gs_plan* p, const double2* send, double2* recv, cudaStream_t st)
{
    for (int b = 0; b < p->d.sh.NB; ++b) {
        int rc = gs_shard_exchange_block(p, send, recv, b, st);
        if (rc) return rc;
    }
    return GS_OK;
}

int gs_shard_pipeline(gs_plan* p, cudaStream_t* comm, cudaEvent_t** events)
{
    if (!p->comm_stream) {
        cudaStream_t s = nullptr;
        GS_CHECK_CUDA(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
        p->comm_stream = s;
        for (int i = 0; i <= p->d.sh.NB; ++i) {
            cudaEvent_t e = nullptr;
            GS_CHECK_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
            p->comm_events.push_back(e);
        }
    }
    *comm = (cudaStream_t)p->comm_stream;
    *events = reinterpret_cast<cudaEvent_t*>(p->comm_events.data());
    return GS_OK;
}

// Average duration (ms, CUDA events on `stream`) of ONE ring <-> m all-to-all of the plan's spectra buffers, timed alone
// (collective: every rank calls it with the same nrep).  bench.py reports it next to the Legendre stages of config #4.
extern "C" int gs_profile_exchange(gs_plan* p, int nrep, float* ms_out, void* stream)
{
    if (!p) { gs_set_error("null plan"); return GS_E_BADARG; }
    GS_REQUIRE(ms_out && nrep >= 1, "bad arguments");
    if (p->world <= 1) { *ms_out = 0.0f; return GS_OK; }
    GS_CHECK_CUDA(cudaSetDevice(p->device));
    cudaStream_t st = (cudaStream_t)stream;
    cudaEvent_t e0, e1;
    GS_CHECK_CUDA(cudaEventCreate(&e0));
    GS_CHECK_CUDA(cudaEventCreate(&e1));
    int rc = gs_shard_exchange(p, p->Fm, p->Fx, st);   // warm-up
    cudaEventRecord(e0, st);
    for (int r = 0; r < nrep && rc == GS_OK; ++r) rc = gs_shard_exchange(p, p->Fm, p->Fx, st);
    cudaEventRecord(e1, st);
    if (rc == GS_OK && cudaEventSynchronize(e1) != cudaSuccess) { gs_set_error("gs_profile_exchange: %s", cudaGetErrorString(cudaGetLastError())); rc = GS_E_CUDA; }
    float ms = 0.0f;
    if (rc == GS_OK) cudaEventElapsedTime(&ms, e0, e1);
    *ms_out = ms / nrep;
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    return rc;
}

int gs_shard_allreduce(gs_plan* p, double* buf, int n, cudaStream_t st)
{
    if (p->lgroup) return local_allreduce(p, buf, n, st);
    GS_CHECK_NCCL(g_nccl.AllReduce(buf, buf, (size_t)n, ncclDouble, ncclSum, (ncclComm_t)p->comm, st));
    return GS_OK;
}

// ---------------------------------------------------------------- per-l helpers on the local real layout
__global__ void expand_per_l_shard_kernel(const double* __restrict__ x, const int* __restrict__ lof, double* __restrict__ out,
                                          int64_t n, int mode)
{
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        out[i] = per_l_value(x, lof[i], mode);
}

int gs_plan_expand_per_l(gs_plan* p, const double* x, int mode, double* out, cudaStream_t st)
{
    if (p->world <= 1) return gs_launch_expand_per_l(x, p->d.lmax, mode, out, st);
    const int64_t n = p->nreal_loc;
    const int nb = (int)std::min<int64_t>((n + 255) / 256, 148 * 16);
    expand_per_l_shard_kernel<<<std::max(nb, 1), 256, 0, st>>>(x, p->d.sh.l_of_loc, out, n, mode);
    GS_CHECK_LAUNCH();
    return GS_OK;
}

// sum_m |a_lm|^2 over the owned m (real layout: plain squares), one warp per l
__global__ void alm2cl_shard_kernel(PlanDev P, const double* __restrict__ alm, double* __restrict__ cl)
{
    const int L = P.lmax, l = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (l > L) return;
    double s = 0.0;
    for (int k = lane; k < P.sh.nm_loc; k += 32) {
        const int m = P.sh.mlist[k];
        if (m > l) break;  // mlist ascending
        const int64_t o = P.sh.rbase[k] + (m ? 2 : 1) * (int64_t)(l - m);
        s += alm[o] * alm[o];
        if (m) s += alm[o + 1] * alm[o + 1];
    }
    for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) cl[l] = s;
}

__global__ void cl_norm_kernel(double* cl, int L)
{
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l <= L) cl[l] /= (2.0 * l + 1.0);
}

// ---------------------------------------------------------------- C ABI
extern "C" int gs_nccl_unique_id(char* id128_host)
{
    GS_REQUIRE(id128_host, "null output");
    if (!nccl_load()) return GS_E_NCCL;
    ncclUniqueId id;
    GS_CHECK_NCCL(g_nccl.GetUniqueId(&id));
    memcpy(id128_host, &id, sizeof(id));
    return GS_OK;
}

extern "C" int gs_plan_world(const gs_plan* p) { return p ? p->world : 0; }
extern "C" int gs_plan_rank(const gs_plan* p) { return p ? p->rank : 0; }
extern "C" int64_t gs_plan_nreal_local(const gs_plan* p) { return p ? p->nreal_loc : 0; }
extern "C" int64_t gs_plan_npix_local(const gs_plan* p) { return p ? p->npix_loc : 0; }

extern "C" int gs_shard_expand_per_l(gs_plan* p, const double* x, int mode, double* out, void* stream)
{
    if (!p) { gs_set_error("null plan"); return GS_E_BADARG; }
    GS_REQUIRE(x && out && mode >= 0 && mode <= 4, "bad arguments");
    GS_CHECK_CUDA(cudaSetDevice(p->device));
    return gs_plan_expand_per_l(p, x, mode, out, (cudaStream_t)stream);
}

extern "C" int gs_shard_alm2cl(gs_plan* p, const double* alm_loc, double* cl, void* stream)
{
    if (!p) { gs_set_error("null plan"); return GS_E_BADARG; }
    GS_REQUIRE(alm_loc && cl, "bad arguments");
    GS_CHECK_CUDA(cudaSetDevice(p->device));
    cudaStream_t st = (cudaStream_t)stream;
    const int L = p->d.lmax;
    if (p->world <= 1) return gs_alm2cl(alm_loc, GS_ALM_REAL, L, cl, stream);
    alm2cl_shard_kernel<<<(L + 8) / 8, 256, 0, st>>>(p->d, alm_loc, cl);
    GS_CHECK_LAUNCH();
    int rc = gs_shard_allreduce(p, cl, L + 1, st);
    if (rc) return rc;
    cl_norm_kernel<<<(L + 256) / 256, 256, 0, st>>>(cl, L);
    GS_CHECK_LAUNCH();
    return GS_OK;
}

// sum over ranks of n doubles in place (e.g. sum(N^-1) of the ring-sharded noise map)
extern "C" int gs_shard_allreduce_sum(gs_plan* p, double* buf, int n, void* stream)
{
    if (!p) { gs_set_error("null plan"); return GS_E_BADARG; }
    GS_REQUIRE(buf && n >= 1, "bad arguments");
    if (p->world <= 1) return GS_OK;
    GS_CHECK_CUDA(cudaSetDevice(p->device));
    return gs_shard_allreduce(p, buf, n, (cudaStream_t)stream);
}
