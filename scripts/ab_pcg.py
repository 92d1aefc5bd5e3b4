"""A/B timing of one masked-sky PCG solve (NSIDE 512 / lmax 1024, the bench system) with a library switch on and off.
usage: python scripts/ab_pcg.py [gs_set_ring_skip | gs_set_ring_fused]"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from gibbssampler_b200 import _dev, _lib, utils  # noqa: E402
from gibbssampler_b200.CenteredGibbs import PolarizedCenteredConstrainedRealization as CR  # noqa: E402
from gibbssampler_b200.sht import Plan  # noqa: E402

setter = sys.argv[1] if len(sys.argv) > 1 else "gs_set_ring_skip"
nside, lmax = 512, 1024
npix, nre = 12 * nside ** 2, (lmax + 1) ** 2
L = _lib.lib()
plan = Plan.get(nside, lmax)
dlE, dlB = bench.fiducial(lmax)
bl = _dev.gauss_beam(np.radians(0.5), lmax)
noise_var = 0.04 * npix / 786432.0
mask = bench.make_mask(nside)
rng = _dev.Rng("philox", seed=1234)
sE = rng.normal(nre) * utils.expand_per_l(_dev.f64(dlE), 3)
sB = rng.normal(nre) * utils.expand_per_l(_dev.f64(dlB), 3)
q, u = plan.alm2map_spin2(sE, sB, fl=_dev.f64(bl))
md = _dev.f64(mask)
dQ = (q + rng.normal(npix) * np.sqrt(noise_var)) * md
dU = (u + rng.normal(npix) * np.sqrt(noise_var)) * md
noise_pol = torch.full((npix,), noise_var, dtype=torch.float64, device="cuda")
cr = CR({"Q": dQ, "U": dU}, noise_pol * 1e4, noise_pol, utils.expand_per_l(_dev.f64(bl), 0), lmax, npix, 0.5, mask=mask, rng="philox", seed=7)
dls = {"EE": _dev.f64(dlE), "BB": _dev.f64(dlB)}
xi = [rng.normal(npix), rng.normal(npix), rng.normal(nre), rng.normal(nre)]
for on in (1, 0, 1, 0):
    old = getattr(L, setter)(on)
    cr.sample_mask(dls, xi=xi)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(2):
        cr.sample_mask(dls, xi=xi)
    e1.record()
    torch.cuda.synchronize()
    getattr(L, setter)(old)
    print("%s(%d): %.2f ms per solve, %d iterations" % (setter, on, e0.elapsed_time(e1) / 2, cr.last_pcg_iterations), flush=True)
