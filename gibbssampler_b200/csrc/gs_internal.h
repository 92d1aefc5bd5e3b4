// Internal declarations shared by the CUDA translation units of libgibbs_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <string>
#include <vector>

#include "../../include/gibbs_b200.h"

// ---------------------------------------------------------------- errors
void gs_set_error(const char* fmt, ...);
#define GS_CHECK_CUDA(expr)                                                                  \
    do {                                                                                     \
        cudaError_t _e = (expr);                                                             \
        if (_e != cudaSuccess) {                                                             \
            gs_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
            return GS_E_CUDA;                                                                \
        }                                                                                    \
    } while (0)
#define GS_CHECK_LAUNCH() GS_CHECK_CUDA(cudaGetLastError())
#define GS_REQUIRE(cond, msg)                                \
    do {                                                     \
        if (!(cond)) {                                       \
            gs_set_error("%s: %s", __func__, msg);           \
            return GS_E_BADARG;                              \
        }                                                    \
    } while (0)

// ---------------------------------------------------------------- scaled-recurrence constants
// true lambda = v * 2^(-GS_SC_K * scale); contributions with true |lambda| < 2^GS_SC_LO are dropped.
#define GS_SC_LO (-900)
#define GS_SC_K 256

struct ScaledSeed {  // value = mant * 2^ex
    double mant;
    int ex;
    int pad;
};

// One Bluestein descriptor per distinct non-power-of-two ring length.
struct BluesteinDesc {
    int n;            // ring length
    int M;            // power-of-two convolution length >= 2n-1
    int64_t chirp_off;  // offset (in double2) of c_j = exp(i pi j^2 / n), j < n
    int64_t bhat_off;   // offset (in double2) of DIF-ordered FFT_M(conj chirp, wrapped) / M
};

struct RingJob {  // one complex DFT = two real ring sequences of equal length
    int ringA, compA;  // 0-based ring index, component (0 = Q/T, 1 = U)
    int ringB, compB;  // ringB = -1: no second sequence
};

// m-sharded transform over `world` GPUs (SURVEY.md 8e, BASELINE config #4): every rank owns a set of m
// (Legendre stage, all rings) and a set of ring pairs (ring-FFT / pixel stage, all m); the ring spectra
// F_m(theta_r) travel between the two partitions in buffers laid out [peer][comp][RL][ML] (double2), so
// that one all-to-all of equal-sized chunks performs the ring <-> m transpose:
//   element (ring, m) lives at ((peer * 2 + comp) * RL + ring_loc[ring]) * ML + m_loc[m]
//   with peer = ring_owner[ring] on the m-sharded side and peer = m_owner[m] on the ring-sharded side.
struct ShardDev {
    int world, rank;
    int nm_loc;       // m owned by this rank
    int ML, RL;       // per-rank m / ring counts, padded to the maximum over ranks (ML = NB * MLb)
    // r02: the local m are cut in NB blocks of MLb so that the all-to-all can run block by block, overlapped with the Legendre
    // stage of the neighbouring block: element (ring, m) lives at
    //   ((((blk * world + peer) * 2 + comp) * RL + ring_loc[ring]) * MLb + (mloc % MLb),  blk = mloc / MLb
    // with mloc = index of m in its owner's list; peer as above.  NB = 1 is the single-exchange layout.
    int NB, MLb;
    const int64_t* m_base;   // [L+1] ring-sharded side: ((blk * world + m_owner[m]) * 2 * RL) * MLb + (m_loc[m] % MLb)
    int64_t nalm_loc; // complex coefficients owned: sum over owned m of (L - m + 1)
    const int* mlist;        // [nm_loc] owned m, ascending
    const int64_t* cbase;    // [nm_loc] index of (l = m) in the local complex numbering
    const int64_t* rbase;    // [nm_loc] offset of (l = m) in the local real layout
    const int* m_owner;      // [L+1]
    const int* m_loc;        // [L+1] index of m in its owner's mlist
    const int* ring_owner;   // [nring]
    const int* ring_loc;     // [nring] index of the ring in its owner's ring list
    const int64_t* ring_start_loc;  // [nring] first pixel of the ring in its owner's local map
    const int* l_of_loc;     // [nreal_loc] multipole of every entry of the local real layout
};

// A ring too long for one CTA's shared memory (nside >= 2048) is transformed as 4 interleaved
// sub-transforms of length n/4 (one CTA each, decimation by 4) that meet in a global scratch buffer.
struct SplitJob {
    int ringA, compA, ringB, compB;
    int bs2;       // Bluestein descriptor of the sub-length n/4, or -1 (power of two)
    int pad;
    int64_t off;   // offset (double2) of this job's n scratch entries
};

// Device-side view of a plan (plain pointers; passed by value to kernels).
struct PlanDev {
    int nside, lmax, nring, npair;
    int64_t npix, nalm;
    // ring pairs p = 0..npair-1 <-> north ring p+1 (p = npair-1 is the equator)
    const double* cth;   // cos(theta)
    const double* sth;   // sin(theta)
    const double* c2;    // cos^2(theta/2)
    const double* s2;    // sin^2(theta/2)
    const int* mlim0;    // last m with a non-negligible lambda_lm on this ring pair (spin 0)
    const int* mlim2;    // same for spin 2
    const int* pmin0;    // [lmax+1] first pair p with mlim0[p] >= m (npair when none)
    const int* pmin2;    // same for spin 2
    // per-m seed factors
    const ScaledSeed* seed0;  // (-1)^m prod sqrt((2k-1)/2k) sqrt((2m+1)/4pi)
    const ScaledSeed* seed2;  // ... * sqrt(m(m-1)/((m+1)(m+2)))  (m >= 2)
    const ScaledSeed* sinpow; // [lmax+1][npair] sin(theta_pair)^m as mant 2^ex (built on the device at plan creation)
    // recurrence tables indexed like healpy alm: idx(l,m) = m(2L+1-m)/2 + l
    const double* rec0;   // a_l (spin 0)
    const double* alpha0; // alpha_l (spin 0)
    const double2* rec2;  // (a_l, b_l) (spin 2)
    const double* alpha2; // alpha_l (spin 2)
    // rings 0..nring-1
    const int* ring_nphi;
    const int64_t* ring_start;
    const int* ring_phq;   // phi0 = pi * ring_phq / ring_phden
    const int* ring_phden;
    const int* ring_bs;    // Bluestein descriptor index or -1 (power-of-two ring)
    const BluesteinDesc* bs;
    const double2* bs_tab; // pooled chirp / bhat tables
    const double2* tw;     // exp(-2 pi i k / tw_n), k < tw_n
    int tw_n;
    int max_M;
    ShardDev sh;           // world == 1: unused
};

// One set of ring flags built from one weight map (gs_active_rings_build): the plan's own set lives in the gs_plan fields of
// the same names; the joint T/E/B solve keeps a second set for N_T^-1 here and swaps it in while its spin-0 half is enqueued.
struct RingFlags {
    unsigned char* act_ring;
    int* act_pairs;
    int* act_count;
    int* act_slot0;
    double* ring_wconst;
    int2* groups0_dyn;
    int2* groups2_dyn;
};

struct gs_plan {
    int device;
    PlanDev d;
    // sharding (world == 1: nreal_loc = (L+1)^2, npix_loc = npix, no communicator)
    int world, rank;
    int64_t nreal_loc, npix_loc;
    void* comm;         // ncclComm_t
    void* lgroup;       // gs_local_group* (in-process test group) or NULL
    double2* Fx;        // second spectra buffer (all-to-all peer of Fm) on sharded plans
    double* red_loc;    // 4 doubles: local partial sums / all-reduced sums of the sharded PCG
    std::vector<int> h_mlist, h_rings;
    std::vector<void*> owned;  // device allocations to free
    // job lists (device) for the ring-FFT stage
    RingJob* jobs2;  // spin 2: (Q,U) of each ring, heavy first
    int njobs2;
    RingJob* jobs0;  // spin 0: (north, south) ring of each pair
    int njobs0;
    int2* groups2;   // CTA work list: (first job, 1 | 2 | 4 jobs of equal transform length) over jobs2 / jobs0
    int ngroups2;
    int2* groups0;
    int ngroups0;
    // the same lists reordered for the weight map of the current call (gs_ring_order_build): groups that need transforms first
    int2* groups2_dyn;
    int2* groups0_dyn;
    SplitJob* sjobs2;   // rings of the spin-2 / spin-0 lists that take the split path (empty below nside 2048)
    int nsjobs2;
    SplitJob* sjobs0;
    int nsjobs0;
    double2* ring_scratch;
    size_t split_smem;
    // block-batched Metropolis sweep workspace (allocated on first use)
    double2* mwg_F;      // [G][2][nring][L+1]
    double* mwg_maps;    // [G][2][npix]  (Q maps of all blocks, then U maps)
    int mwg_group;       // G
    double* mwg_small;   // reduction partials, likelihood pair, per-l filters
    double* mwg_data;    // [2][npix] the data maps with the constant-weight rings in spectral storage (gs_ring_mwg_data)
    int* mwg_meta;       // bins / block boundaries / per-block mmax / flags (re-uploaded when the blocking changes)
    std::vector<int> mwg_meta_host;
    // rings / ring pairs that carry a non-zero pixel weight (gs_active_rings_build); use_act = the Legendre and fused
    // ring kernels launched through gs_leg_synth / gs_leg_anal / gs_ring_apply walk these lists (PCG mat-vec only)
    unsigned char* act_ring;  // [nring] 1 = some pixel weight of the ring is non-zero
    int* act_pairs;           // [npair] ascending list of pairs with an active north or south ring
    int* act_count;           // device int: entries of act_pairs
    double* act_red;          // [nring] sharded plans: ring flags as doubles for the sum over ranks
    int* act_slot0;           // [2][lmax+1] (spin 0, spin 2): first entry of act_pairs whose pair reaches m
    double* ring_wconst;      // [nring] the pixel weight of a ring whose weights are all equal, NaN for any other ring (unsharded plans)
    bool use_act;
    // workspace
    double2* Fm;        // [2][nring][lmax+1] ring spectra
    double* partial;    // analysis partial sums [nchunk][nalm][4]
    int anal_chunks;
    int chain_cap;      // right-hand sides the spectra / partial-sum buffers hold (1; gs_plan_reserve_chains raises it)
    size_t ring_smem;   // dynamic shared memory of the ring-FFT kernels
    // scratch maps / alms for iter>0 analysis and solvers
    double* mapQ_tmp;
    double* mapU_tmp;
    double* almE_tmp;
    double* almB_tmp;
    double* almE_tmp2;
    double* almB_tmp2;
    void* pcg_ws;       // gs_pcg_ws* (solver.cu): PCG vectors / state of this plan, allocated on the first solve
    void* pcg_ws_batch; // gs_pcg_ws[2]: workspaces of a two-chain batch (gs_cr_pcg_pol_batch), allocated on first use
    int* pcg_alldone;   // device flag: both chains of the batch have converged
    void* pcg_ws_teb;   // TebWs* (solver.cu): vectors / state of the joint T/E/B solve, allocated on its first use
    RingFlags flags_T;  // second ring-flag set of the joint T/E/B solve (N_T^-1); all NULL until its first use
    void* comm_stream;  // cudaStream_t the block-wise all-to-all of a sharded plan runs on (NULL until first used)
    std::vector<void*> comm_events;   // cudaEvent_t: NB + 1 of them
    void* work_stream;  // cudaStream_t of the plan for graph-captured solves (NULL until first used)
    void* work_event;   // cudaEvent_t ordering work_stream after the caller's stream
};

extern int g_gs_ring_const;       // 1: rings of constant pixel weight take the transform-free path of ring_apply_kernel (PCG mat-vec)
extern int g_gs_ring_skip;        // 1: rings whose pixel weights vanish identically are left out (PCG mat-vec, Metropolis sweep)
extern int g_gs_ring_fused;       // 1: the PCG mat-vec runs its ring stage as one fused kernel (ring_apply_kernel)
extern long long g_gs_launches;  // kernels launched by this library (bench.py's gpu_launches)
static inline int64_t gs_nalm(int lmax) { return (int64_t)(lmax + 1) * (lmax + 2) / 2; }

// legendre.cu
// `skip` (nullable device int): when *skip != 0 the kernels return immediately (device-side early exit)
// nc = 2: chain batch (two right-hand sides share one recurrence; chain c at alm + c alm_stride, spectra at p->Fm + c gs_fm_stride(p));
// needs gs_plan_reserve_chains(p, 2) and an unsharded plan
int gs_leg_synth(gs_plan* p, int spin, const double* almE, const double* almB, int layout, const double* fl,
                 cudaStream_t st, const int* skip = nullptr, const double* flB = nullptr, int nc = 1, int64_t alm_stride = 0);
int gs_leg_anal(gs_plan* p, int spin, double* almE, double* almB, int layout, const double* fl, double scale,
                int accumulate, cudaStream_t st, const int* skip = nullptr, int nc = 1, int64_t alm_stride = 0);
int64_t gs_fm_stride(const gs_plan* p);            // double2 entries of one chain's ring spectra
int64_t gs_part_stride(const gs_plan* p, int nc);  // doubles of one chain's analysis partial sums
int gs_active_rings_build(gs_plan* p, const double* pixw, cudaStream_t st);
int gs_leg_build_sinpow(gs_plan* p);
int gs_leg_prepare(gs_plan* p);   // per-device kernel attributes (dynamic shared memory opt-in)
// ringfft.cu
int gs_ring_setup(gs_plan* p);
// nc > 1 (chain batch): chain c uses the spectra p->Fm + c gs_fm_stride(p) and the maps + c map_stride
// wconst (spin 2, unsharded, no split rings; see gs_ring_mwg_data): rings with a constant pixel weight are written in spectral storage
int gs_ring_synth(gs_plan* p, int spin, double* mapQ, double* mapU, cudaStream_t st, const int* skip = nullptr, int nc = 1,
                  int64_t map_stride = 0, const double* wconst = nullptr);
int gs_ring_anal(gs_plan* p, int spin, const double* mapQ, const double* mapU, const double* pixw, cudaStream_t st,
                 const int* skip = nullptr, int nc = 1, int64_t map_stride = 0);
int gs_ring_apply(gs_plan* p, int spin, const double* pixw, cudaStream_t st, const int* skip = nullptr, int nc = 1);
int gs_ring_synth_batch(gs_plan* p, const double2* F, int64_t f_stride, const int* mmax, double* mapQ, double* mapU,
                        int64_t map_stride, int nb, cudaStream_t st, const unsigned char* ract = nullptr, const double* wconst = nullptr);
// Spectral storage of constant-weight rings (Metropolis sweep): out = the Q/U maps with every ring whose wconst is a number replaced
// by the unitary DFT of its pixels z_j = Q_j + i U_j (Re in the Q slots, Im in the U slots); other rings are copied.
// Launch order of the ring groups for the current weight map (after gs_active_rings_build filled act_ring / ring_wconst): groups with a
// ring that needs its transforms first (they are the long CTAs), then constant-weight groups, then idle ones; stable within a class
int gs_ring_order_build(gs_plan* p, cudaStream_t st);
int gs_ring_mwg_data(gs_plan* p, const double* mapQ, const double* mapU, double* outQ, double* outU, const double* wconst, cudaStream_t st);
// legendre.cu: block-batched spin-2 synthesis for the Metropolis-within-Gibbs sweep (see leg_synth_blocks_kernel)
int gs_leg_synth_blocks(gs_plan* p, const double* almE, const double* almB, const double* dflE, const double* dflB,
                        const int* lbE, int e0, int e1, const int* lbB, int b0, int b1, int lend, double2* Fblk, cudaStream_t st);
// almops.cu
int gs_launch_expand_per_l(const double* x, int lmax, int mode, double* out, cudaStream_t st);
// expansion over the plan's (possibly sharded) real layout
int gs_plan_expand_per_l(gs_plan* p, const double* x, int mode, double* out, cudaStream_t st);
// solver.cu
void gs_pcg_ws_free(gs_plan* p);
// shard.cu
int gs_shard_build(gs_plan* p, int rank, int world, const char* nccl_id);
void gs_shard_free(gs_plan* p);
// all-to-all of the spectra buffers (ring <-> m transpose): send -> recv, all NB blocks (chunk = 2 RL MLb double2 per peer and block)
int gs_shard_exchange(gs_plan* p, const double2* send, double2* recv, cudaStream_t st);
// one block of it (collective; blocks must be exchanged in the same order on every rank)
int gs_shard_exchange_block(gs_plan* p, const double2* send, double2* recv, int blk, cudaStream_t st);
// streams / events of the pipelined exchange (NCCL plans): comm stream and NB + 1 events, created on first use
int gs_shard_pipeline(gs_plan* p, cudaStream_t* comm, cudaEvent_t** events);
// in-place sum over ranks of n doubles (device)
int gs_shard_allreduce(gs_plan* p, double* buf, int n, cudaStream_t st);
