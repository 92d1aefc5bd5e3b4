// One C call per chain for the centred polarised full-sky sampler (BASELINE config #1; SURVEY.md 8b gs_gibbs_step_centered,
// 7.1 step 4 "CUDA-graph the iteration"):
//
//   GibbsSampler.run_polarization (GibbsSampler.py:118-180) with
//     constrained_sampler.sample  = PolarizedCenteredConstrainedRealization.sample_no_mask (CenteredGibbs.py:317-353)
//     cls_sampler.sample          = PolarizedCenteredClsSampler.sample (CenteredGibbs.py:54-93)
//     utils.unfold_bins           (utils.py:150-162)
//
// At NSIDE 64 an iteration is ~10 us of kernel work; driven from Python (one ctypes call per kernel) it costs ~280 us.  Here
// the iteration is three kernels that read the iteration number from device memory (history row, Philox stream ids), captured
// ONCE in a CUDA graph and replayed n_iter times: the binned D_l history fills on the device and crosses PCIe once.
#include <algorithm>
#include <vector>

#include "gs_internal.h"
#include "rng.cuh"
#include "spectra.cuh"

struct ChainDev {
    int L, nbE, nbB;
    const int* binsE;      // nbE + 1 edges
    const int* binsB;
    const int* binofE;     // [L+1] bin of multipole l (-1 outside the binning)
    const int* binofB;
    const double* bl;
    const double* dE;      // data alm (real layout)
    const double* dB;
    double w;              // Npix / (noise 4 pi)
    double* histE;         // [n_iter + 1][nbE]
    double* histB;
    double* almE;          // current sky (real layout)
    double* almB;
    double* clE;           // [L+1] hp.alm2cl of the current sky
    double* clB;
    unsigned long long* it;  // iteration counter
    unsigned long long seed;
};

__global__ void gstep_binof_kernel(const int* __restrict__ bins, int nb, int L, int* __restrict__ binof)
{
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l > L) return;
    binof[l] = l >= bins[0] && l < bins[nb] ? bin_of(bins, nb, l) : -1;
}

// constrained realization: diagonal solve + draw for E and B (CenteredGibbs.py:317-353); D_l of this iteration = history row `it`
__global__ void __launch_bounds__(256) gstep_cr_kernel(ChainDev C)
{
    const unsigned long long it = *C.it;
    const int L = C.L;
    const int64_t n = (int64_t)(L + 1) * (L + 1);
    const Philox ph(C.seed);
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int l = l_of_real(i, L);
        const double b = C.bl[l];
        double n0, n1;
        box_muller(ph((uint64_t)i, RNG_CR | it), n0, n1);
#pragma unroll
        for (int pol = 0; pol < 2; ++pol) {
            const int bin = (pol ? C.binofB : C.binofE)[l];
            const double ic = safe_rcp(dl_to_cl(bin >= 0 ? (pol ? C.histB + it * C.nbB : C.histE + it * C.nbE)[bin] : 0.0, l));
            const double sigma = 1.0 / (C.w * b * b + ic);
            const double d = (pol ? C.dB : C.dE)[i];
            (pol ? C.almB : C.almE)[i] = sigma * (b * (C.w * d)) + (pol ? n1 : n0) * sqrt(sigma);
        }
    }
}

// hp.alm2cl on the real layout (every entry of multipole l has variance C_l): one warp per (l, pol)
__global__ void __launch_bounds__(256) gstep_cl_kernel(ChainDev C)
{
    const int L = C.L, wid = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (wid >= 2 * (L + 1)) return;
    const int pol = wid > L, l = pol ? wid - (L + 1) : wid;
    const double s = warp_sum(alm2cl_real_lane(pol ? C.almB : C.almE, l, L, lane));
    if (lane == 0) (pol ? C.clB : C.clE)[l] = s / (2.0 * l + 1.0);
}

// inverse-gamma draw per bin (CenteredGibbs.py:54-79) into history row it + 1; the last thread advances the counter
__global__ void __launch_bounds__(128) gstep_cls_kernel(ChainDev C)
{
    const unsigned long long it = *C.it;
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < C.nbE + C.nbB) {
        const int pol = t >= C.nbE, b = pol ? t - C.nbE : t;
        const int* bins = pol ? C.binsB : C.binsE;
        double beta, alpha = ig_bin_stats(pol ? C.clB : C.clE, bins[b], bins[b + 1], beta);
        if (b == 0) alpha = 1.0;
        const double g = alpha > 0.0 ? gamma_mt(alpha, Philox(C.seed), RNG_GAMMA | (it << 21) | ((uint64_t)pol << 20) | (uint64_t)b) : 1.0;
        (pol ? C.histB + (it + 1) * C.nbB : C.histE + (it + 1) * C.nbE)[b] = (b < 2) ? 0.0 : beta / g;
    }
}
__global__ void gstep_advance_kernel(unsigned long long* it) { *it += 1; }

extern "C" int gs_gibbs_run_centered_fullsky(int lmax, int64_t npix, double noise_pol, const double* bl, const double* d_E,
                                             const double* d_B, const int* bins_EE, int nbins_EE, const int* bins_BB, int nbins_BB,
                                             const double* init_EE, const double* init_BB, int n_iter, uint64_t seed,
                                             double* hist_EE, double* hist_BB, double* last_E, double* last_B, int use_graph,
                                             void* stream)
{
    GS_REQUIRE(lmax >= 2 && npix > 0 && noise_pol > 0.0 && bl && d_E && d_B && bins_EE && bins_BB && init_EE && init_BB && hist_EE && hist_BB,
               "bad arguments");
    GS_REQUIRE(nbins_EE >= 1 && nbins_BB >= 1 && n_iter >= 0 && n_iter < (1 << 30), "bad arguments");
    // the loop runs on a stream of its own (stream capture is not allowed on the legacy default stream), ordered after `stream`
    cudaStream_t user = (cudaStream_t)stream, st = nullptr;
    cudaEvent_t ready = nullptr;
    GS_CHECK_CUDA(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    GS_CHECK_CUDA(cudaEventCreateWithFlags(&ready, cudaEventDisableTiming));
    GS_CHECK_CUDA(cudaEventRecord(ready, user));
    GS_CHECK_CUDA(cudaStreamWaitEvent(st, ready, 0));
    const int L = lmax;
    const int64_t n = (int64_t)(L + 1) * (L + 1);
    // scratch: [almE, almB (unless given)] [clE, clB] [binofE, binofB] [it]
    double* scratch = nullptr;
    const size_t nd = (size_t)(2 * n + 2 * (L + 1) + 2);
    GS_CHECK_CUDA(cudaMalloc(&scratch, nd * sizeof(double) + (size_t)2 * (L + 1) * sizeof(int)));
    ChainDev C;
    C.L = L; C.nbE = nbins_EE; C.nbB = nbins_BB;
    C.binsE = bins_EE; C.binsB = bins_BB;
    C.almE = last_E ? last_E : scratch;
    C.almB = last_B ? last_B : scratch + n;
    C.clE = scratch + 2 * n; C.clB = C.clE + (L + 1);
    C.it = reinterpret_cast<unsigned long long*>(C.clB + (L + 1));
    int* binof = reinterpret_cast<int*>(scratch + nd);
    C.binofE = binof; C.binofB = binof + (L + 1);
    C.bl = bl; C.dE = d_E; C.dB = d_B;
    C.w = (double)npix / (noise_pol * 4.0 * GS_PI);
    C.histE = hist_EE; C.histB = hist_BB;
    C.seed = seed;
    int rc = GS_OK;
    auto fail = [&](cudaError_t e, const char* what) { gs_set_error("gs_gibbs_run_centered_fullsky: %s: %s", what, cudaGetErrorString(e)); rc = GS_E_CUDA; };
    cudaError_t e;
    if ((e = cudaMemsetAsync(C.it, 0, sizeof(unsigned long long), st)) != cudaSuccess) fail(e, "memset");
    gstep_binof_kernel<<<(L + 256) / 256, 256, 0, st>>>(bins_EE, nbins_EE, L, binof);
    gstep_binof_kernel<<<(L + 256) / 256, 256, 0, st>>>(bins_BB, nbins_BB, L, binof + (L + 1));
    if (rc == GS_OK && (e = cudaMemcpyAsync(hist_EE, init_EE, nbins_EE * sizeof(double), cudaMemcpyDeviceToDevice, st)) != cudaSuccess) fail(e, "copy");
    if (rc == GS_OK && (e = cudaMemcpyAsync(hist_BB, init_BB, nbins_BB * sizeof(double), cudaMemcpyDeviceToDevice, st)) != cudaSuccess) fail(e, "copy");
    const int g_cr = (int)std::min<int64_t>((n + 255) / 256, 148 * 8), g_cl = (2 * (L + 1) * 32 + 255) / 256, g_cls = (nbins_EE + nbins_BB + 127) / 128;
    auto iteration = [&]() {
        gstep_cr_kernel<<<g_cr, 256, 0, st>>>(C);
        gstep_cl_kernel<<<g_cl, 256, 0, st>>>(C);
        gstep_cls_kernel<<<g_cls, 128, 0, st>>>(C);
        gstep_advance_kernel<<<1, 1, 0, st>>>(C.it);
    };
    if (rc == GS_OK && n_iter > 0) {
        if (use_graph) {
            cudaGraph_t graph = nullptr;
            cudaGraphExec_t exec = nullptr;
            if ((e = cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal)) != cudaSuccess) fail(e, "begin capture");
            if (rc == GS_OK) {
                iteration();
                if ((e = cudaStreamEndCapture(st, &graph)) != cudaSuccess) fail(e, "end capture");
            }
            if (rc == GS_OK && (e = cudaGraphInstantiate(&exec, graph, 0)) != cudaSuccess) fail(e, "instantiate");
            for (int k = 0; k < n_iter && rc == GS_OK; ++k)
                if ((e = cudaGraphLaunch(exec, st)) != cudaSuccess) fail(e, "graph launch");
            if (exec) cudaGraphExecDestroy(exec);
            if (graph) cudaGraphDestroy(graph);
        } else {
            for (int k = 0; k < n_iter; ++k) iteration();
            if ((e = cudaGetLastError()) != cudaSuccess) fail(e, "launch");
        }
        g_gs_launches += 4LL * n_iter;
    }
    if ((e = cudaStreamSynchronize(st)) != cudaSuccess && rc == GS_OK) fail(e, "synchronize");
    cudaFree(scratch);
    cudaEventDestroy(ready);
    cudaStreamDestroy(st);
    return rc;
}
