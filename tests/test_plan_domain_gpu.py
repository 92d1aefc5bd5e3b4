"""The transforms and the PCG operator over the whole (NSIDE, lmax) domain gs_plan_create accepts (1 <= NSIDE <= 2048,
2 <= lmax <= 4 NSIDE), against the long-double oracle (oracle/sht_oracle.c: generic HEALPix geometry, mixed-radix reference
FFT, m % n alias folding) to the FP64 bar of 1e-10 relative.

What the rest of the suite leaves out and this file covers:
  * NSIDE that is not a power of two (even, odd, prime): the 2 NSIDE + 1 belt rings of 4 NSIDE pixels leave the radix-4
    path for Bluestein, with the half-pixel shift on every other belt ring;
  * lmax = 4 NSIDE (every belt ring alias-folded up to m = n), lmax << NSIDE (Legendre pruning and the fold without alias
    terms on almost every ring) and the healpy default lmax = 3 NSIDE - 1;
  * the ring-stage variants (fused ring stage, ring skip, constant-weight rings, forced split path, chain batches, local
    sharded groups, spectral ring storage of the Metropolis sweep) at those sizes, under a mask that leaves rings idle,
    constant and cut;
  * lmax = 3 NSIDE - 1 and 4 NSIDE at NSIDE 1024 / 1536 / 2048 through the sampled direct sums of tests/sampled_sht.py."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import reference_logic as R
from oracle import sht as O

pytestmark = pytest.mark.gpu

RTOL = 1e-10

NONPOW2 = [3, 5, 6, 7, 12, 24, 48, 96, 100, 127]


def _lmaxes(nside):
    small = [nside // 8] if nside // 8 >= 2 else []
    return sorted({2, *small, 3 * nside - 1, 4 * nside})


GRID = [(n, l) for n in NONPOW2 for l in _lmaxes(n)] + [(1, 4), (2, 8), (8, 32), (64, 256), (128, 512), (256, 2), (512, 7),
                                                        pytest.param(512, 2047, marks=pytest.mark.slow)]
# one odd NSIDE, one NSIDE = 2 mod 4, NSIDE 100 at lmax = 4 NSIDE
VARIANT_GRID = [(7, 20), (6, 24), (100, 400)]
SETTERS = ("gs_set_ring_fused", "gs_set_ring_skip", "gs_set_ring_const", "gs_set_pcg_graph")


@pytest.fixture
def ring_flags():
    """The library's global switches as the test found them, restored whatever the test does."""
    from gibbssampler_b200 import _lib
    L = _lib.lib()
    saved = {}
    for s in SETTERS:
        saved[s] = getattr(L, s)(1)
        getattr(L, s)(saved[s])
    try:
        yield L
    finally:
        for s, v in saved.items():
            getattr(L, s)(v)


def dev(x):
    return torch.as_tensor(np.ascontiguousarray(x), device="cuda")


def host(x):
    return x.cpu().numpy()


def relerr(got, ref):
    return float(np.abs(got - ref).max() / np.abs(ref).max())


def rand_alm(lmax, rng, lmin=0):
    a = rng.standard_normal(O.nalm(lmax)) + 1j * rng.standard_normal(O.nalm(lmax))
    a[:lmax + 1] = a[:lmax + 1].real
    ell = np.concatenate([np.arange(m, lmax + 1) for m in range(lmax + 1)])
    a[ell < lmin] = 0
    return a


def to_real(a, lmax):
    r = np.empty((lmax + 1) ** 2)
    r[:lmax + 1] = a[:lmax + 1].real
    r[lmax + 1::2] = a[lmax + 1:].real * np.sqrt(2)
    r[lmax + 2::2] = a[lmax + 1:].imag * np.sqrt(2)
    return r


def kind_of(nside):
    """long double up to NSIDE 128; the FP64 OpenMP build above (a few seconds per transform at NSIDE 512)"""
    return "ld" if nside <= 128 else "f64"


def ring_index(nside):
    n = np.r_[4 * np.arange(1, nside), np.full(2 * nside + 1, 4 * nside), 4 * np.arange(nside - 1, 0, -1)]
    return np.repeat(np.arange(4 * nside - 1), n)


def mask_weights(nside):
    """N^-1 that leaves rings idle (|z| < 0.08 everywhere, and the southern cap below z = -0.75), constant (a different
    constant north and south) and cut (a longitude-dependent band edge between |z| = 0.08 and 0.43)."""
    th, ph = O.pix_angles(nside)
    z = np.cos(th)
    half = 0.08 + 0.35 * np.exp(-(np.angle(np.exp(1j * ph)) / 0.7) ** 2)
    return 20.0 * (np.abs(z) > half) * (z > -0.75) * (1.0 + 0.5 * (z > 0))


def ring_kinds(nside, w):
    """(idle, constant, cut) ring counts of a weight map; idle rings count as constant (their weight is the constant 0)"""
    ring = ring_index(nside)
    idle = const = cut = 0
    for r in range(4 * nside - 1):
        v = w[ring == r]
        if np.ptp(v) == 0.0:
            const += 1
            idle += v[0] == 0.0
        else:
            cut += 1
    return idle, const, cut


def test_mask_of_the_variant_grid_has_idle_constant_and_cut_rings():
    for nside, _ in VARIANT_GRID:
        idle, const, cut = ring_kinds(nside, mask_weights(nside))
        assert idle > 0 and const > idle and cut > 0, (nside, idle, const, cut)


# ------------------------------------------------------------------------------------------------------------- (a) transforms
@pytest.mark.parametrize("nside,lmax", GRID)
def test_transforms_vs_oracle(nside, lmax):
    from gibbssampler_b200 import _lib
    from gibbssampler_b200._dev import ptr, stream
    from gibbssampler_b200.sht import Plan
    kind = kind_of(nside)
    plan = Plan.get(nside, lmax) if nside <= 128 else Plan(nside, lmax)
    rng = np.random.default_rng(1000 * nside + lmax)
    npix = 12 * nside ** 2
    # synthesis, spin 0 and spin 2, both alm layouts
    a = rand_alm(lmax, rng)
    ref = O.alm2map(a, nside, lmax, kind=kind)
    assert relerr(host(plan.alm2map(dev(a))), ref) < RTOL
    assert relerr(host(plan.alm2map(dev(to_real(a, lmax)))), ref) < RTOL
    e, b = rand_alm(lmax, rng, 2), rand_alm(lmax, rng, 2)
    rq, ru = O.alm2map_spin2(e, b, nside, lmax, kind=kind)
    for x, y in ((e, b), (to_real(e, lmax), to_real(b, lmax))):
        q, u = plan.alm2map_spin2(dev(x), dev(y))
        assert relerr(host(q), rq) < RTOL and relerr(host(u), ru) < RTOL
    # separate E and B filters (gs_alm2map_spin2_fl2)
    flE, flB = rng.uniform(0.5, 1.5, lmax + 1), rng.uniform(-1.0, 1.0, lmax + 1)
    fq, fu = O.alm2map_spin2(O.almxfl(e, flE, lmax), O.almxfl(b, flB, lmax), nside, lmax, kind=kind)
    q, u = torch.empty(npix, dtype=torch.float64, device="cuda"), torch.empty(npix, dtype=torch.float64, device="cuda")
    ed, bd, fe, fb = dev(e), dev(b), dev(flE), dev(flB)
    _lib.check(_lib.lib().gs_alm2map_spin2_fl2(plan._h, ptr(ed), ptr(bd), 0, ptr(fe), ptr(fb), ptr(q), ptr(u), stream()))
    assert relerr(host(q), fq) < RTOL and relerr(host(u), fu) < RTOL
    # analysis: iter 0 and 3 with pixel weights and a filter, and the adjoint in the real layout
    mq, mu = rng.standard_normal(npix), rng.standard_normal(npix)
    w = rng.uniform(0.0, 2.0, npix)
    bl = O.gauss_beam(np.radians(120.0 / nside), lmax)
    for it in (0, 3):
        ra = O.almxfl(O.map2alm(mq * w, nside, lmax, iter=it, kind=kind), bl, lmax)
        assert relerr(host(plan.map2alm(dev(mq), iter=it, pixw=dev(w), fl=dev(bl))), ra) < RTOL
        re_, rb_ = O.map2alm_spin2(mq * w, mu * w, nside, lmax, iter=it, kind=kind)
        ge, gb = plan.map2alm_spin2(dev(mq), dev(mu), iter=it, pixw=dev(w), fl=dev(bl))
        assert relerr(host(ge), O.almxfl(re_, bl, lmax)) < RTOL and relerr(host(gb), O.almxfl(rb_, bl, lmax)) < RTOL
    ra = to_real(O.map2alm(mq, nside, lmax, adjoint=True, kind=kind), lmax)
    assert relerr(host(plan.map2alm(dev(mq), adjoint=True, real_layout=True)), ra) < RTOL
    ae, ab = O.map2alm_spin2(mq, mu, nside, lmax, adjoint=True, kind=kind)
    ge, gb = plan.map2alm_spin2(dev(mq), dev(mu), adjoint=True, real_layout=True)
    assert relerr(host(ge), to_real(ae, lmax)) < RTOL and relerr(host(gb), to_real(ab, lmax)) < RTOL


# --------------------------------------------------------------------------------------------------- (b) ring-stage variants
def _operator(plan, lmax, spin, w, seed=3):
    from gibbssampler_b200 import _lib
    from gibbssampler_b200._dev import f64, ptr, stream
    L = _lib.lib()
    rng = np.random.default_rng(seed)
    nre = (lmax + 1) ** 2
    ell = np.arange(lmax + 1)
    dl, bl = f64(np.where(ell >= 2, 1.0 + 0.1 * ell, 0.0)), f64(np.exp(-1e-4 * ell * (ell + 1.0)))
    invn = f64(w)
    xe, xb = f64(rng.standard_normal(nre)), f64(rng.standard_normal(nre))
    ye, yb = torch.zeros_like(xe), torch.zeros_like(xb)
    if spin == 2:
        _lib.check(L.gs_cr_apply_q_pol(plan._h, ptr(dl), ptr(dl), ptr(bl), ptr(invn), ptr(xe), ptr(xb), ptr(ye), ptr(yb), stream()))
    else:
        _lib.check(L.gs_cr_apply_q_tt(plan._h, ptr(dl), ptr(bl), ptr(invn), ptr(xe), ptr(ye), stream()))
    torch.cuda.synchronize()
    nconst = C.c_int(-1)
    _lib.check(L.gs_constant_rings(plan._h, C.byref(nconst)))
    return host(ye), host(yb), nconst.value


def _operator_oracle(nside, lmax, spin, w, seed=3):
    rng = np.random.default_rng(seed)
    nre = (lmax + 1) ** 2
    ell = np.arange(lmax + 1)
    dl, bl = np.where(ell >= 2, 1.0 + 0.1 * ell, 0.0), np.exp(-1e-4 * ell * (ell + 1.0))
    xe, xb = rng.standard_normal(nre), rng.standard_normal(nre)
    blm, ic = R.expand_per_l(bl), R.safe_inv(R.generate_var_cl(dl))
    if spin == 2:
        q, u = R.synth_pol(xe * blm, xb * blm, nside, lmax, "ld")
        ae, ab = R.adjoint_pol(q * w, u * w, nside, lmax, 0, "ld")
        return ic * xe + blm * ae, ic * xb + blm * ab
    t = O.alm2map(R.real_to_complex(xe * blm), nside, lmax)
    at = R.complex_to_real(O.map2alm(t * w, nside, lmax, adjoint=True))
    return ic * xe + blm * at, np.zeros(nre)


@pytest.mark.parametrize("spin", [2, 0])
@pytest.mark.parametrize("nside,lmax", VARIANT_GRID)
def test_ring_stage_variants_vs_oracle_under_a_mask(nside, lmax, spin, ring_flags):
    """Every combination of gs_set_ring_fused / gs_set_ring_skip / gs_set_ring_const gives the operator of the default state
    to rounding and the oracle operator to 1e-10; with constant rings on, gs_constant_rings counts the constant rings of the map."""
    from gibbssampler_b200.sht import Plan
    L = ring_flags
    plan = Plan.get(nside, lmax)
    w = mask_weights(nside)
    _, nconst_map, _ = ring_kinds(nside, w)
    re_, rb_ = _operator_oracle(nside, lmax, spin, w)
    for s in SETTERS[:3]:
        getattr(L, s)(1)
    base = _operator(plan, lmax, spin, w)
    assert base[2] == nconst_map
    for fused in (1, 0):
        for skip in (1, 0):
            for const in (1, 0):
                L.gs_set_ring_fused(fused)
                L.gs_set_ring_skip(skip)
                L.gs_set_ring_const(const)
                ye, yb, _ = _operator(plan, lmax, spin, w)
                tag = (fused, skip, const)
                assert relerr(ye, re_) < RTOL, tag
                assert np.abs(ye - base[0]).max() <= 1e-12 * np.abs(base[0]).max(), tag
                if spin == 2:
                    assert relerr(yb, rb_) < RTOL, tag
                    assert np.abs(yb - base[1]).max() <= 1e-12 * np.abs(base[1]).max(), tag


# ---------------------------------------------------------------------------------------------------- (c) forced split path
SPLIT_CASES = [(12, 48, 64), (12, 35, 64), (24, 96, 64), (24, 71, 128), (7, 28, 16)]


def _split_plan(nside, lmax, mcap, monkeypatch):
    from gibbssampler_b200.sht import Plan
    monkeypatch.setenv("GS_RING_MCAP", str(mcap))
    try:
        return Plan(nside, lmax)
    finally:
        monkeypatch.delenv("GS_RING_MCAP")


@pytest.mark.parametrize("nside,lmax,mcap", SPLIT_CASES)
def test_forced_split_path_with_bluestein_sub_transforms(nside, lmax, mcap, monkeypatch):
    """GS_RING_MCAP < 4 NSIDE sends the belt rings (4 NSIDE pixels, not a power of two) through the split path, whose four
    sub-transforms of NSIDE points are Bluestein transforms themselves: both directions, both spins, against the unforced plan
    (1e-12) and the oracle (1e-10)."""
    from gibbssampler_b200.sht import Plan
    ref = Plan.get(nside, lmax)
    plan = _split_plan(nside, lmax, mcap, monkeypatch)
    rng = np.random.default_rng(7 + nside + mcap)
    npix = 12 * nside ** 2
    e, b, t = rand_alm(lmax, rng, 2), rand_alm(lmax, rng, 2), rand_alm(lmax, rng)
    rq, ru = O.alm2map_spin2(e, b, nside, lmax)
    q0, u0 = ref.alm2map_spin2(dev(e), dev(b))
    q1, u1 = plan.alm2map_spin2(dev(e), dev(b))
    assert relerr(host(q1), host(q0)) < 1e-12 and relerr(host(u1), host(u0)) < 1e-12
    assert relerr(host(q1), rq) < RTOL and relerr(host(u1), ru) < RTOL
    t0, t1 = ref.alm2map(dev(t)), plan.alm2map(dev(t))
    assert relerr(host(t1), host(t0)) < 1e-12 and relerr(host(t1), O.alm2map(t, nside, lmax)) < RTOL
    fq, fu = rng.standard_normal(npix), rng.standard_normal(npix)
    w = rng.uniform(0.5, 1.5, npix)
    re_, rb_ = O.map2alm_spin2(fq * w, fu * w, nside, lmax)
    e0, b0 = ref.map2alm_spin2(dev(fq), dev(fu), pixw=dev(w))
    e1, b1 = plan.map2alm_spin2(dev(fq), dev(fu), pixw=dev(w))
    assert relerr(host(e1), host(e0)) < 1e-12 and relerr(host(b1), host(b0)) < 1e-12
    assert relerr(host(e1), re_) < RTOL and relerr(host(b1), rb_) < RTOL
    ra = O.map2alm(fq, nside, lmax, adjoint=True)
    a0, a1 = ref.map2alm(dev(fq), adjoint=True), plan.map2alm(dev(fq), adjoint=True)
    assert relerr(host(a1), host(a0)) < 1e-12 and relerr(host(a1), ra) < RTOL


def test_forced_split_keeps_twelve_pixel_rings_direct(monkeypatch):
    """NSIDE 3 with GS_RING_MCAP = 16: every belt ring has 12 pixels, whose quarter (3 points) would be a Bluestein
    transform of M = 8 on the split path, shorter than the radix-16 pass that applies its chirp spectrum: the synthesis came
    out unrelated to the oracle (relative error 2.5 at NSIDE 7 / lmax 28).  Such rings stay on the direct path."""
    nside, lmax = 3, 12
    plan = _split_plan(nside, lmax, 16, monkeypatch)
    rng = np.random.default_rng(12)
    e, b, t = rand_alm(lmax, rng, 2), rand_alm(lmax, rng, 2), rand_alm(lmax, rng)
    rq, ru = O.alm2map_spin2(e, b, nside, lmax)
    q, u = plan.alm2map_spin2(dev(e), dev(b))
    assert relerr(host(q), rq) < RTOL and relerr(host(u), ru) < RTOL
    assert relerr(host(plan.alm2map(dev(t))), O.alm2map(t, nside, lmax)) < RTOL
    f = rng.standard_normal(12 * nside ** 2)
    assert relerr(host(plan.map2alm(dev(f), adjoint=True)), O.map2alm(f, nside, lmax, adjoint=True)) < RTOL


# ------------------------------------------------------------------------------------- (d) chain batches, local sharded groups
@pytest.mark.parametrize("k", [2, 3])
@pytest.mark.parametrize("nside,lmax,mcap", [(12, 48, 0), (7, 20, 0), (12, 48, 64)])
def test_chain_batches_equal_single_calls(nside, lmax, mcap, k, monkeypatch):
    """k chains per call equal k single calls; with mcap the belt rings take the split path, where the chains of a batch take
    turns on the shared scratch buffer."""
    from gibbssampler_b200.sht import Plan
    plan = _split_plan(nside, lmax, mcap, monkeypatch) if mcap else Plan(nside, lmax)
    rng = np.random.default_rng(31 * nside + k)
    npix = 12 * nside ** 2
    es = np.stack([to_real(rand_alm(lmax, rng, 2), lmax) for _ in range(k)])
    bs = np.stack([to_real(rand_alm(lmax, rng, 2), lmax) for _ in range(k)])
    ts = np.stack([to_real(rand_alm(lmax, rng), lmax) for _ in range(k)])
    fq, fu = rng.standard_normal((k, npix)), rng.standard_normal((k, npix))
    w = rng.uniform(0.5, 1.5, npix)
    single = [[host(v) for v in plan.alm2map_spin2(dev(es[c]), dev(bs[c]))] + [host(plan.alm2map(dev(ts[c])))]
              + [host(v) for v in plan.map2alm_spin2(dev(fq[c]), dev(fu[c]), pixw=dev(w), real_layout=True)]
              + [host(plan.map2alm(dev(fq[c]), adjoint=True, real_layout=True))] for c in range(k)]
    q, u = plan.alm2map_spin2_batch(dev(es), dev(bs))
    t = plan.alm2map_batch(dev(ts))
    ge, gb = plan.map2alm_spin2_batch(dev(fq), dev(fu), pixw=dev(w), real_layout=True)
    g0 = plan.map2alm_batch(dev(fq), adjoint=True, real_layout=True)
    for c in range(k):
        for got, ref in zip((q[c], u[c], t[c], ge[c], gb[c], g0[c]), single[c]):
            assert relerr(host(got), ref) < 1e-12, c
        rq, ru = O.alm2map_spin2(R.real_to_complex(es[c]), R.real_to_complex(bs[c]), nside, lmax)
        assert relerr(host(q[c]), rq) < RTOL and relerr(host(u[c]), ru) < RTOL


@pytest.mark.parametrize("nside,lmax,world", [(12, 48, 2), (12, 35, 3), (7, 28, 3), (6, 2, 2)])
def test_local_group_transforms_match_single_gpu(nside, lmax, world):
    from gibbssampler_b200.sharded import ShardedPlan, run_local_group
    from gibbssampler_b200.sht import Plan
    from tests.test_shard_gpu import full_inputs
    ref = Plan.get(nside, lmax)
    e, b, q, u, w, fl = full_inputs(nside, lmax, 17 + nside)
    want = dict(sq=ref.alm2map_spin2(e, b, fl=fl)[0], su=ref.alm2map_spin2(e, b, fl=fl)[1],
                s0=ref.alm2map(e, fl=fl), t0=ref.map2alm(q, adjoint=True, real_layout=True))
    want["ae"], want["ab"] = ref.map2alm_spin2(q, u, adjoint=True, pixw=w, fl=fl, real_layout=True)
    want["je"], want["jb"] = ref.map2alm_spin2(q, u, iter=3, real_layout=True)
    plans = ShardedPlan.local_group(nside, lmax, world)

    def work(p):
        le, lb = p.local_alm(e), p.local_alm(b)
        lq, lu, lw = p.local_map(q), p.local_map(u), p.local_map(w)
        out = {}
        out["sq"], out["su"] = p.alm2map_spin2(le, lb, fl=fl)
        out["ae"], out["ab"] = p.map2alm_spin2(lq, lu, adjoint=True, pixw=lw, fl=fl, real_layout=True)
        out["je"], out["jb"] = p.map2alm_spin2(lq, lu, iter=3, real_layout=True)
        out["s0"] = p.alm2map(le, fl=fl)
        out["t0"] = p.map2alm(lq, adjoint=True, real_layout=True)
        return out

    res = run_local_group(plans, work)
    for key, ref_v in want.items():
        out = torch.zeros_like(ref_v)
        for p, r in zip(plans, res):
            out[p.pixel_index if key in ("sq", "su", "s0") else p.real_index] = r[key]
        assert float((out - ref_v).abs().max() / ref_v.abs().max()) < RTOL, key


# ------------------------------------------------------------------------------------------------- (e) PCG operator and solve
def _teb_inputs(nside, lmax, seed):
    from tests.teb_oracle import TPProblem
    rng = np.random.default_rng(seed)
    npix = 12 * nside ** 2
    w = mask_weights(nside)
    wT = w * np.where(np.cos(O.pix_angles(nside)[0]) > 0.5, rng.uniform(0.5, 1.5, npix), 1.0)   # T: rough northern cap
    d = [rng.standard_normal(npix) for _ in range(3)]
    fwhm = 240.0 / nside
    return TPProblem(nside, lmax, d[0], d[1], d[2], wT, w, fwhm), wT, w


@pytest.mark.parametrize("nside,lmax", [(7, 28), (6, 17), (12, 48), (100, 400)])
def test_pcg_operators_vs_oracle(nside, lmax, ring_flags):
    """gs_cr_apply_q_tt / _pol / _teb against TTProblem / PolProblem / TPProblem.apply_Q, with the library's default ring
    shortcuts on, under a mask with idle, constant and cut rings and different T and P weights."""
    from gibbssampler_b200 import _lib
    from gibbssampler_b200._dev import f64, ptr, stream
    from gibbssampler_b200.sht import Plan
    from tests import teb_problem as T
    L = ring_flags
    for s in SETTERS[:3]:
        getattr(L, s)(1)
    plan = Plan.get(nside, lmax)
    prob, wT, wP = _teb_inputs(nside, lmax, 5 + nside)
    dls = T.spectra(lmax)
    n = (lmax + 1) ** 2
    rng = np.random.default_rng(9)
    x = [rng.standard_normal(n) for _ in range(3)]
    xd = [f64(v) for v in x]
    y = [torch.zeros(n, dtype=torch.float64, device="cuda") for _ in range(3)]
    d = {k: f64(v) for k, v in dls.items()}
    bl, invT, invP = f64(prob.bl_gauss), f64(wT), f64(wP)
    _lib.check(L.gs_cr_apply_q_tt(plan._h, ptr(d["TT"]), ptr(bl), ptr(invT), ptr(xd[0]), ptr(y[0]), stream()))
    ref = prob.tt.apply_Q(R.generate_var_cl(dls["TT"]), x[0])
    assert relerr(host(y[0]), ref) < RTOL
    _lib.check(L.gs_cr_apply_q_pol(plan._h, ptr(d["EE"]), ptr(d["BB"]), ptr(bl), ptr(invP), ptr(xd[1]), ptr(xd[2]), ptr(y[1]),
                                   ptr(y[2]), stream()))
    re_, rb_ = prob.pol.apply_Q(dls["EE"], dls["BB"], x[1], x[2])
    assert relerr(host(y[1]), re_) < RTOL and relerr(host(y[2]), rb_) < RTOL
    _lib.check(L.gs_cr_apply_q_teb(plan._h, ptr(d["TT"]), ptr(d["TE"]), ptr(d["EE"]), ptr(d["BB"]), ptr(bl), ptr(invT), ptr(invP),
                                   *[ptr(v) for v in xd], *[ptr(v) for v in y], stream()))
    got, want = np.concatenate([host(v) for v in y]), np.concatenate(prob.apply_Q(dls, tuple(x)))
    assert relerr(got, want) < RTOL


def test_pcg_pol_solve_vs_dense_solve():
    """gs_cr_pcg_pol at NSIDE 5 / lmax 20 = 4 NSIDE (belt rings Bluestein and alias-folded) against a dense solve of the oracle's Q"""
    from gibbssampler_b200 import _lib
    from gibbssampler_b200._dev import f64, ptr, stream
    from gibbssampler_b200.sht import Plan
    nside, lmax = 5, 20
    prob, _, wP = _teb_inputs(nside, lmax, 41)
    pol = prob.pol
    ell = np.arange(lmax + 1)
    dlE, dlB = np.where(ell >= 2, 1.0 + 0.1 * ell, 0.0), np.where(ell >= 2, 0.3 + 0.02 * ell, 0.0)
    n = (lmax + 1) ** 2
    keep = np.ones(2 * n, bool)
    keep[[0, 1, lmax + 1, lmax + 2, n, n + 1, n + lmax + 1, n + lmax + 2]] = False   # l < 2: Q and b vanish there
    rng = np.random.default_rng(4)
    bvec = rng.standard_normal(2 * n) * keep
    Q = pol.dense_Q(dlE, dlB)
    ref = np.zeros(2 * n)
    ref[keep] = np.linalg.solve(Q[np.ix_(keep, keep)], bvec[keep])
    plan = Plan.get(nside, lmax)
    L = _lib.lib()
    xe, xb = torch.zeros(n, dtype=torch.float64, device="cuda"), torch.zeros(n, dtype=torch.float64, device="cuda")
    nit, res = C.c_int(0), C.c_double(0)
    be, bb = f64(bvec[:n]), f64(bvec[n:])
    de, db, bl, invn = f64(dlE), f64(dlB), f64(pol.bl_gauss), f64(wP)   # held until the solve has read them
    _lib.check(L.gs_cr_pcg_pol(plan._h, ptr(de), ptr(db), ptr(bl), ptr(invn), float(np.sum(wP) / (4 * np.pi)), ptr(be), ptr(bb),
                               ptr(xe), ptr(xb), 0, 1e-12, 4000, 8, C.byref(nit), C.byref(res), stream()))
    assert 0 < nit.value < 4000 and res.value <= 1.01e-12
    got = np.concatenate([host(xe), host(xb)])
    assert np.abs(got - ref).max() <= 1e-8 * np.abs(ref).max()


def test_pcg_teb_solve_vs_dense_solve():
    """gs_cr_pcg_teb at NSIDE 3 / lmax 12 = 4 NSIDE against a dense solve of the oracle's joint Q"""
    from gibbssampler_b200 import _lib
    from gibbssampler_b200._dev import f64, ptr, stream
    from gibbssampler_b200.sht import Plan
    from tests import teb_problem as T
    nside, lmax = 3, 12
    prob, wT, wP = _teb_inputs(nside, lmax, 43)
    dls = T.spectra(lmax)
    n = (lmax + 1) ** 2
    act = T.active(lmax)
    rng = np.random.default_rng(6)
    bvec = rng.standard_normal(3 * n) * act
    Q = prob.dense_Q(dls)
    ref = np.zeros(3 * n)
    ref[act] = np.linalg.solve(Q[np.ix_(act, act)], bvec[act])
    plan = Plan.get(nside, lmax)
    L = _lib.lib()
    d = {k: f64(v) for k, v in dls.items()}
    b = [f64(v) for v in np.split(bvec, 3)]
    x = [torch.zeros(n, dtype=torch.float64, device="cuda") for _ in range(3)]
    nit, res = C.c_int(0), C.c_double(0)
    bl, invT, invP = f64(prob.bl_gauss), f64(wT), f64(wP)   # held until the solve has read them
    _lib.check(L.gs_cr_pcg_teb(plan._h, ptr(d["TT"]), ptr(d["TE"]), ptr(d["EE"]), ptr(d["BB"]), ptr(bl),
                               ptr(invT), ptr(invP), float(np.sum(wT) / (4 * np.pi)), float(np.sum(wP) / (4 * np.pi)),
                               *[ptr(v) for v in b], *[ptr(v) for v in x], 0, 1e-12, 4000, 8, C.byref(nit), C.byref(res), stream()))
    assert 0 < nit.value < 4000 and res.value <= 1.01e-12
    got = np.concatenate([host(v) for v in x])
    assert np.abs(got - ref).max() <= 1e-8 * np.abs(ref).max()


# ------------------------------------------------------------------------------------------------------- (f) Metropolis sweep
@pytest.mark.parametrize("nside,lmax", [(12, 35), (7, 28)])
def test_batched_sweep_with_constant_rings_equals_per_block_sweep(nside, lmax, ring_flags):
    """gs_mwg_sweep_blocks with gs_set_ring_const on (constant rings kept as ring spectra, Bluestein belt rings) against the
    per-block path (one gs_alm2map_spin2_fl2 per block): same accept decisions and the same spectra, under a mask with cut rings."""
    from tests.test_cr_gpu import make_problem
    from tests.test_mwg_blocks_gpu import binned_start, build
    L = ring_flags
    L.gs_set_ring_skip(1)
    L.gs_set_ring_const(1)
    P = make_problem(nside, lmax, seed=3)
    mask = (mask_weights(nside) != 0).astype(float)
    P["dQ"], P["dU"], P["mask"] = P["dQ"] * mask, P["dU"] * mask, mask
    ee = np.arange(0, lmax + 2)
    cut = (3 * lmax) // 4
    bb = np.concatenate([np.arange(0, cut), np.arange(cut, lmax + 1, 3)])
    bb[-1] = lmax + 1
    bins = {"EE": ee, "BB": bb}
    blocks = {"EE": [2, len(ee) // 2, len(ee) - 1], "BB": np.concatenate([[2, cut // 2], np.arange(cut // 2 + 1, len(bb))])}
    rng = np.random.default_rng(11)
    s_nc = {p: rng.standard_normal((lmax + 1) ** 2) for p in ("EE", "BB")}
    start = binned_start(P, bins)
    res = []
    for batched in (False, True):
        nc = build(P, bins, blocks, 1, 0, batched)
        assert nc.batched_blocks == batched
        np.random.seed(77)
        res.append(nc.sample(s_nc, {k: v.copy() for k, v in start.items()}))
    (d0, a0), (d1, a1) = res
    assert a0["EE"] == a1["EE"] and a0["BB"] == a1["BB"]
    assert 0 < sum(a0["BB"]) + sum(a0["EE"]) < len(a0["BB"]) + len(a0["EE"])
    for p in ("EE", "BB"):
        assert np.array_equal(d0[p], d1[p])
    nconst = C.c_int(-1)
    L.gs_constant_rings(nc.plan._h, C.byref(nconst))
    assert 0 < nconst.value < 4 * nside - 1


# ------------------------------------------------------------------------------------------------------------ (g) large sizes
LARGE = [(1024, 3071), (1536, 3071), pytest.param(1024, 4096, marks=pytest.mark.slow),
         pytest.param(1536, 6144, marks=pytest.mark.slow), pytest.param(2048, 6143, marks=pytest.mark.slow),
         pytest.param(2048, 8192, marks=pytest.mark.slow)]


def _large_rings(nside, lmax, ms, step):
    """poles, the cap/belt boundaries, the equator, every `step`-th ring, and the rings on both sides of the pruning boundary
    m = m_lim(theta) of every sampled m (northern hemisphere; the south mirrors it)"""
    nring = 4 * nside - 1
    rings = (set(range(1, 41)) | set(range(nring - 39, nring + 1)) | set(range(1, nring + 1, step))
             | set(range(nside - 3, nside + 4)) | set(range(2 * nside - 2, 2 * nside + 3)) | set(range(3 * nside - 3, 3 * nside + 4)))
    sth = np.array([O.ring_info(nside, r)[1] for r in range(1, 2 * nside + 1)])
    for m in ms:
        if m < 100:
            continue
        # mlim_of (plan.cu): m_lim = lmax sin(theta) + max(100, lmax / 100) for spin 0; first ring that reaches m
        reach = np.nonzero(lmax * sth + max(100.0, 0.01 * lmax) >= m)[0]
        if len(reach):
            r0 = int(reach[0]) + 1
            rings |= {r for r in range(r0 - 2, r0 + 3) if 1 <= r <= nring} | {nring + 1 - r for r in range(r0 - 2, r0 + 3) if 1 <= r <= nring}
    return sorted(rings)


@pytest.mark.parametrize("nside,lmax", LARGE)
def test_sampled_sums_at_large_sizes(nside, lmax):
    """lmax = 3 NSIDE - 1 and 4 NSIDE at NSIDE 1024 and 2048, and NSIDE 1536 (belt rings of 6144 pixels: split path with
    Bluestein sub-transforms of 1536 points), against the direct sums of tests/sampled_sht.py (aliasing included)."""
    from gibbssampler_b200.sht import Plan
    from tests import sampled_sht as S
    plan = Plan(nside, lmax)
    rng = np.random.default_rng(nside + lmax)
    ms = S.sampled_m(lmax)
    rings = _large_rings(nside, lmax, ms, 23)
    e, b, t, coef = S.sampled_alm(lmax, ms, rng)
    q, u = (host(x) for x in plan.alm2map_spin2(dev(e), dev(b)))
    tm = host(plan.alm2map(dev(t)))
    worst = S.synthesis_error(nside, lmax, ms, coef, rings, q, u, tm, rng, npick=16)
    assert worst < RTOL, worst
    nring = 4 * nside - 1
    trings = [1, 2, 37, nside - 1, nside, nside + 1, 2 * nside, 3 * nside + 1, nring - 5, nring]
    fq, fu, geo = S.ring_supported_maps(nside, trings, rng)
    ge, gb = (host(x) for x in plan.map2alm_spin2(dev(fq), dev(fu), adjoint=True))
    gt = host(plan.map2alm(dev(fq), adjoint=True))
    worst = S.analysis_error(nside, lmax, ms, trings, fq, fu, geo, ge, gb, gt)
    assert worst < RTOL, worst
