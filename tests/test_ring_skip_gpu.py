"""Masked rings in the PCG mat-vec A^T N^-1 A: rings whose N^-1 vanishes identically are left out of the Legendre and ring
kernels (gs_set_ring_skip, default on).  The operator and the PCG solution must equal the all-rings path to rounding and the
oracle operator to 1e-10, for equatorial bands (whole ring pairs idle), one-sided caps (one ring of a pair idle), masks that
leave whole CTA chunks empty, an all-zero weight map, and weight maps without any idle ring."""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _ring_z(nside):
    from oracle import sht as O
    th, _ = O.pix_angles(nside)
    return np.cos(th)


def _weights(kind, nside, rng):
    z = _ring_z(nside)
    npix = z.size
    w = rng.uniform(0.5, 2.0, npix)
    if kind == "band":            # galactic band: both rings of the equatorial pairs idle
        w *= np.abs(z) > 0.3
    elif kind == "south":         # southern cap masked: one ring of each polar pair idle
        w *= z > -0.5
    elif kind == "north_only":    # only a polar cap observed: most pairs half idle, equatorial pairs idle
        w *= z > 0.6
    elif kind == "holes":         # point-source holes: no idle ring
        w *= rng.uniform(size=npix) > 0.1
    elif kind == "zero":
        w *= 0.0
    elif kind == "full":
        pass
    else:
        raise ValueError(kind)
    return w


def _apply(nside, lmax, spin, w, skip, seed=3):
    from gibbssampler_b200 import _lib
    from gibbssampler_b200._dev import f64, ptr, stream
    from gibbssampler_b200.sht import Plan
    L = _lib.lib()
    rng = np.random.default_rng(seed)
    nre = (lmax + 1) ** 2
    ell = np.arange(lmax + 1)
    dl = f64(np.where(ell >= 2, 1.0 + 0.1 * ell, 0.0))
    bl = f64(np.exp(-1e-4 * ell * (ell + 1.0)))
    invn = f64(w)
    xe, xb = f64(rng.standard_normal(nre)), f64(rng.standard_normal(nre))
    ye, yb = torch.empty_like(xe), torch.empty_like(xb)
    plan = Plan.get(nside, lmax)
    old = L.gs_set_ring_skip(1 if skip else 0)
    try:
        if spin == 2:
            _lib.check(L.gs_cr_apply_q_pol(plan._h, ptr(dl), ptr(dl), ptr(bl), ptr(invn), ptr(xe), ptr(xb), ptr(ye), ptr(yb), stream()))
        else:
            _lib.check(L.gs_cr_apply_q_tt(plan._h, ptr(dl), ptr(bl), ptr(invn), ptr(xe), ptr(ye), stream()))
            yb.zero_()
        torch.cuda.synchronize()
        act, tot = C.c_int(-1), C.c_int(-1)
        if skip:
            _lib.check(L.gs_active_ring_pairs(plan._h, C.byref(act), C.byref(tot)))
    finally:
        L.gs_set_ring_skip(old)
    return ye.cpu().numpy(), yb.cpu().numpy(), act.value, tot.value


@pytest.mark.parametrize("kind", ["band", "south", "north_only", "holes", "zero", "full"])
@pytest.mark.parametrize("nside,lmax", [(8, 16), (32, 64), (128, 256), (512, 700)])
@pytest.mark.parametrize("spin", [2, 0])
def test_skipping_idle_rings_leaves_the_operator_unchanged(kind, nside, lmax, spin):
    rng = np.random.default_rng(11)
    w = _weights(kind, nside, rng)
    a = _apply(nside, lmax, spin, w, True)
    b = _apply(nside, lmax, spin, w, False)
    # expected number of active pairs straight from the weight map
    npair, nring = 2 * nside, 4 * nside - 1
    z = _ring_z(nside)
    starts = np.concatenate([[0], np.cumsum(np.r_[4 * np.arange(1, nside), np.full(2 * nside + 1, 4 * nside), 4 * np.arange(nside - 1, 0, -1)])])
    ring_on = np.array([np.any(w[starts[r]:starts[r + 1]] != 0.0) for r in range(nring)])
    expect = sum(bool(ring_on[p] or ring_on[nring - 1 - p]) for p in range(npair))
    assert (a[2], a[3]) == (expect, npair)
    for u, v in zip(a[:2], b[:2]):
        assert np.abs(u - v).max() <= 1e-12 * max(1.0, np.abs(v).max())
    del z


def test_skipping_operator_vs_oracle():
    from oracle import reference_logic as R
    nside, lmax = 16, 40
    rng = np.random.default_rng(5)
    w = _weights("band", nside, rng)
    nre = (lmax + 1) ** 2
    ell = np.arange(lmax + 1)
    dl = np.where(ell >= 2, 1.0 + 0.1 * ell, 0.0)
    bl = np.exp(-1e-4 * ell * (ell + 1.0))
    xr = np.random.default_rng(3)
    xe, xb = xr.standard_normal(nre), xr.standard_normal(nre)
    ye, yb, act, tot = _apply(nside, lmax, 2, w, True)
    assert 0 < act < tot
    blm = R.expand_per_l(bl)
    q, u = R.synth_pol(xe * blm, xb * blm, nside, lmax, "ld")
    ae, ab = R.adjoint_pol(q * w, u * w, nside, lmax, 0, "ld")
    ic = R.safe_inv(R.generate_var_cl(dl))
    re, rb = ic * xe + blm * ae, ic * xb + blm * ab
    assert np.abs(ye - re).max() <= 1e-10 * np.abs(re).max()
    assert np.abs(yb - rb).max() <= 1e-10 * np.abs(rb).max()


@pytest.mark.parametrize("kind,setter", [("band", "gs_set_ring_skip"), ("south", "gs_set_ring_skip")])
def test_pcg_solution_with_and_without_skipping(kind, setter):
    """Same solve with idle-ring skipping on and off."""
    from gibbssampler_b200 import _lib, utils
    from gibbssampler_b200.CenteredGibbs import PolarizedCenteredConstrainedRealization
    from oracle import sht as O
    L = _lib.lib()
    nside, lmax = 32, 64
    npix, nre = 12 * nside * nside, (lmax + 1) ** 2
    rng = np.random.default_rng(9)
    mask = (_weights(kind, nside, rng) != 0).astype(float)
    noise = np.full(npix, 0.05)
    ell = np.arange(lmax + 1)
    dls = {"EE": np.where(ell >= 2, 1.0 + 0.05 * ell, 0.0), "BB": np.where(ell >= 2, 0.3 + 0.01 * ell, 0.0)}
    fwhm = 3.0
    dQ, dU = rng.standard_normal(npix) * mask, rng.standard_normal(npix) * mask
    bl_map = utils.expand_per_l(O.gauss_beam(np.radians(fwhm), lmax))
    xi = (rng.standard_normal(npix), rng.standard_normal(npix), rng.standard_normal(nre), rng.standard_normal(nre))
    out = []
    old_const = L.gs_set_ring_const(0)   # isotropic noise: keep the transform-free path of constant rings (tests/test_ring_const_gpu.py) out of this A/B
    for skip in (1, 0):
        old = getattr(L, setter)(skip)
        try:
            cr = PolarizedCenteredConstrainedRealization({"Q": dQ, "U": dU}, noise * 1e4, noise, bl_map, lmax, npix, fwhm, mask=mask)
            sol, _ = cr.sample_mask(dls, xi)
            out.append((np.concatenate([np.asarray(sol["EE"]), np.asarray(sol["BB"])]), cr.last_pcg_iterations))
        finally:
            getattr(L, setter)(old)
    L.gs_set_ring_const(old_const)
    (xa, ia), (xb_, ib) = out
    assert abs(ia - ib) <= 1
    # skipping re-associates the sums of the mat-vec, so the two solves to the reference's eps = 1e-5 follow slightly different
    # conjugate-gradient trajectories: they agree to the tolerance of the solve, not to rounding
    assert np.abs(xa - xb_).max() <= 1e-5 * np.abs(xb_).max()
