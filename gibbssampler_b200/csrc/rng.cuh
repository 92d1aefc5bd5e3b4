// Device random numbers of the samplers: Philox4x32-10 counter RNG, its stream domains, Box-Muller normals and
// Marsaglia-Tsang gamma variates.
#pragma once
#include <math.h>
#include <stdint.h>

// ------------------------------------------------------------------ Philox4x32-10 counter RNG
struct Philox {
    uint32_t k0, k1;
    __device__ Philox(uint64_t seed) : k0((uint32_t)seed), k1((uint32_t)(seed >> 32)) {}
    __device__ uint4 operator()(uint64_t ctr, uint64_t stream) const
    {
        uint32_t c0 = (uint32_t)ctr, c1 = (uint32_t)(ctr >> 32), c2 = (uint32_t)stream, c3 = (uint32_t)(stream >> 32);
        uint32_t a = k0, b = k1;
#pragma unroll
        for (int r = 0; r < 10; ++r) {
            const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
            const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
            const uint32_t n0 = hi1 ^ c1 ^ a, n2 = hi0 ^ c3 ^ b;
            c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
            a += 0x9E3779B9u; b += 0xBB67AE85u;
        }
        return make_uint4(c0, c1, c2, c3);
    }
};

__device__ __forceinline__ double u01(uint32_t hi, uint32_t lo)
{  // uniform in (0,1): 53 random bits, centred
    const uint64_t x = (((uint64_t)hi << 32) | lo) >> 11;
    return ((double)x + 0.5) * 0x1p-53;
}

__device__ __forceinline__ void box_muller(uint4 r, double& n0, double& n1)
{
    const double u1 = u01(r.x, r.y), u2 = u01(r.z, r.w);
    const double rad = sqrt(-2.0 * log(u1));
    double s, c;
    sincospi(2.0 * u2, &s, &c);
    n0 = rad * c;
    n1 = rad * s;
}

// Stream domains: the top byte of a Philox stream id names its consumer, so no consumer walks into another one's streams however
// long a chain runs (the counters of gs_randn / gs_randu stay below 2^56).  Each consumer keeps its own id layout, and changing one
// changes every chain history:
//   RNG_CR       normals of the fused chain (gibbs_step.cu): RNG_CR | it
//   RNG_GAMMA    gs_cls_invgamma: ((call << 20) + b) & RNG_ID_MASK; the fused chain, on its own seed word: (it << 21) | (pol << 20) | b
//   RNG_WISHART  inverse-Wishart draws (teb.cu): ((call << 22) + 4 k) & RNG_ID_MASK, then + 0 / 1 / 2
constexpr uint64_t RNG_CR = 0x43ull << 56, RNG_GAMMA = 0x47ull << 56, RNG_WISHART = 0x57ull << 56;
constexpr uint64_t RNG_ID_MASK = 0x00ffffffffffffffull;

// ------------------------------------------------------------------ inverse-gamma C_l draw
// Marsaglia-Tsang Gamma(a,1), a > 0, one thread per draw with its own Philox stream
__device__ inline double gamma_mt(double a, const Philox& ph, uint64_t stream)
{
    uint64_t ctr = 0;
    double boost = 1.0;
    if (a < 1.0) {
        const uint4 r = ph(ctr++, stream);
        boost = pow(u01(r.x, r.y), 1.0 / a);
        a += 1.0;
    }
    const double d = a - 1.0 / 3.0, c = 1.0 / sqrt(9.0 * d);
    for (int it = 0; it < 1000; ++it) {
        double x, x2;
        box_muller(ph(ctr++, stream), x, x2);
        const uint4 r = ph(ctr++, stream);
        const double u = u01(r.x, r.y);
        double v = 1.0 + c * x;
        if (v <= 0.0) { x = x2; v = 1.0 + c * x; if (v <= 0.0) continue; }
        v = v * v * v;
        if (log(u) < 0.5 * x * x + d * (1.0 - v + log(v))) return boost * d * v;
    }
    return boost * d;
}
