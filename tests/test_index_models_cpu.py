"""CPU models of the two pieces of index algebra in the CUDA kernels that no other CPU test can see.  They restate, in numpy,
exactly what the device code does lane by lane / thread by thread, so that a change of the scheme has to be made (and
argued) in two places:

* the spin-2 analysis reduce-scatter (legendre.cu: anal_acc, the select-free exchange stages, the swizzled shared-memory
  park + batched sum over FOLD3_NB pairs of l in the fast loop of leg_anal_kernel): every (l-parity h, value c) must come out as the sum over the 32 lanes, at the index the
  kernel writes (h * 4 + c), with the sign flip of (h = 1, odd c);
* the complex-coefficient decode c -> (l, m) of loglik_alm_partial_kernel (sampler.cu) and its real-layout offsets
  (utils.py:49-76 of the reference: r[l] for m = 0, r[2 i - (L+1)], r[2 i - (L+1) + 1] for i > L)."""
import math

import numpy as np


def test_analysis_reduce_scatter_model():
    rng = np.random.default_rng(0)
    NB = 8                                   # FOLD3_NB pairs of l per batch
    # true per-lane contributions y[q][lane][h][c] (already summed over the R ring pairs of the lane, signs of the
    # lambda^+- basis applied): the kernel computes s_c * y for (h = 1, odd c) and flips it back at the end
    y = rng.standard_normal((NB, 32, 2, 4))
    sgn = np.ones((2, 4))
    sgn[1, 1] = sgn[1, 3] = -1.0
    out = np.zeros((NB, 8))
    buf = np.zeros((NB, 32, 2))              # sFold: [q][slot] -> (h = 0 value, h = 1 value)
    for q in range(NB):
        # registers v[slot] of every lane: slot s holds value c = s ^ pi(lane), pi = (bit 4, bit 3)
        v = np.zeros((32, 8))
        for lane in range(32):
            pi = ((lane >> 4) & 1) << 1 | ((lane >> 3) & 1)
            for h in range(2):
                for s in range(4):
                    c = s ^ pi
                    v[lane, 4 * h + s] = sgn[h, c] * y[q, lane, h, c]
        # stage xor 16: every lane keeps slots 0, 1 and adds the partner's slots 2, 3 (both l of the pair)
        w = v.copy()
        for lane in range(32):
            p = lane ^ 16
            for base in (0, 4):
                w[lane, base + 0] = v[lane, base + 0] + v[p, base + 2]
                w[lane, base + 1] = v[lane, base + 1] + v[p, base + 3]
        v = w.copy()
        # stage xor 8: keep slot 0, add the partner's slot 1
        for lane in range(32):
            p = lane ^ 8
            for base in (0, 4):
                w[lane, base + 0] = v[lane, base + 0] + v[p, base + 1]
        v = w
        # park (v[0], v[4]) at the swizzled slot
        for lane in range(32):
            cperm = ((lane >> 4) & 1) << 1 | ((lane >> 3) & 1)
            slot = lane ^ cperm ^ ((q & 1) << 2)
            buf[q, slot] = (v[lane, 0], v[lane, 4])
        assert len({lane ^ (((lane >> 4) & 1) << 1 | ((lane >> 3) & 1)) ^ ((q & 1) << 2) for lane in range(32)}) == 32   # conflict free
    # flush: output o = lane + 32 t -> (q, h, c); 8 entries s0 ^ k
    for t in range(NB // 4):
        banks = []
        for lane in range(32):
            o = lane + 32 * t
            q, h, c = o >> 3, (o >> 2) & 1, o & 3
            s0 = (((c >> 1) << 4) | ((c & 1) << 3)) ^ c ^ ((q & 1) << 2)
            a = [buf[q, s0 ^ k, h] for k in range(8)]
            total = ((a[0] + a[1]) + (a[2] + a[3])) + ((a[4] + a[5]) + (a[6] + a[7]))
            if h and (c & 1):
                total = -total
            out[q, h * 4 + c] = total
            banks.append(((q * 32 + s0) * 2 + h) % 16)        # 8-byte bank of the k = 0 load
        # 32 loads of 8 bytes need two wavefronts at best: every bank is hit exactly twice
        assert sorted(np.bincount(banks, minlength=16)) == [2] * 16
    ref = y.sum(axis=1).reshape(NB, 8)                        # [q][h * 4 + c]
    assert np.allclose(out, ref, rtol=1e-13, atol=1e-13)


def _decode(c, L):
    t = 2.0 * L + 3.0
    m = int((t - math.sqrt(max(t * t - 8.0 * c, 0.0))) * 0.5)
    m = max(0, min(m, L))
    while m > 0 and m * (2 * L + 3 - m) // 2 > c:
        m -= 1
    while m < L and (m + 1) * (2 * L + 3 - (m + 1)) // 2 <= c:
        m += 1
    return m, c - m * (2 * L + 1 - m) // 2


def test_complex_coefficient_decode_and_real_offsets():
    for L in (0, 1, 2, 3, 8, 33, 128):
        n = (L + 1) * (L + 2) // 2
        seen = np.zeros((L + 1) ** 2, dtype=int)
        for c in range(n):
            m, l = _decode(c, L)
            assert 0 <= m <= l <= L and c == m * (2 * L + 1 - m) // 2 + l      # healpy index (utils.py:123)
            if m == 0:
                seen[l] += 1
            else:
                off = 2 * c - (L + 1)
                seen[off] += 1
                seen[off + 1] += 1
        assert np.all(seen == 1)                                                 # every real-layout entry exactly once
    # ends of the range at the bench size, where the float sqrt is least exact
    L = 4096
    n = (L + 1) * (L + 2) // 2
    for c in list(range(0, 3000)) + list(range(n - 3000, n)) + list(range(0, n, 9973)):
        m, l = _decode(c, L)
        assert 0 <= m <= l <= L and c == m * (2 * L + 1 - m) // 2 + l
