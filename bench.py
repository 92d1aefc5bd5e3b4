#!/usr/bin/env python
"""bench.py -- Gibbs iterations/s (and spin-2 SHT pairs/s) of the constrained-realization +
C_l-sampling Gibbs step on synthetic CMB polarisation skies (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W          # this repo (sm_100a kernels)
  python bench.py --impl reference --gpus N ...          # the reference CPU path (oracle port) on host cores

A step = one Gibbs iteration of the centred polarised masked-sky sampler
(PolarizedCenteredConstrainedRealization.sample_mask: RHS draw + PCG solve, then
PolarizedCenteredClsSampler.sample), one independent chain per GPU (weak scaling, no data-path
collective).  Workload (SURVEY.md 8d): NSIDE 512, lmax 1024, analytic fiducial spectra
D^EE_l = exp(-(l/1200)^2) + 0.02, D^BB_l = 0.05 (l/80)^-0.5 exp(-(l/1500)^2) + 1e-3 (l >= 2),
Gaussian 0.5 deg beam, white noise sigma^2_pol = 0.04 uK^2 (NSIDE 256) scaled with Npix, galactic
band mask f_sky = 0.8 with a 2 deg cosine edge; data synthetic, seeds fixed.  Every run also measures the same
sampler under a galactic-plane-like mask whose edge depends on the longitude (--mask galplane; key `galplane_mask`
of the JSON line): the band cuts no ring, that one cuts a third of them (see make_mask).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

REF_BUDGET_S = 1500.0   # wall-clock budget of the reference arm (the driver's limit per arm is 1800 s)


def pixel_z(nside):
    """cos(theta) of every RING pixel (HEALPix geometry, vectorised)."""
    npix = 12 * nside * nside
    z = np.empty(npix)
    i = np.arange(1, nside)
    start = 2 * i * (i - 1)
    zc = 1 - i * i / (3.0 * nside * nside)
    for ii, s, zz in zip(i, start, zc):
        z[s:s + 4 * ii] = zz
        z[npix - s - 4 * ii:npix - s] = -zz
    ib = np.arange(nside, 3 * nside + 1)
    ncap = 2 * nside * (nside - 1)
    zb = 4.0 / 3 - 2 * ib / (3.0 * nside)
    z[ncap:npix - ncap] = np.repeat(zb, 4 * nside)
    return z


def fiducial(lmax):
    ell = np.arange(lmax + 1, dtype=np.float64)
    dlE = np.where(ell >= 2, np.exp(-(ell / 1200.0) ** 2) + 0.02, 0.0)
    dlB = np.where(ell >= 2, 0.05 * (np.maximum(ell, 1) / 80.0) ** -0.5 * np.exp(-(ell / 1500.0) ** 2) + 1e-3, 0.0)
    return dlE, dlB


def pixel_phi(nside):
    """Longitude of every RING pixel (HEALPix geometry: caps (j + 1/2) pi / (2 i), belt rings alternately shifted)."""
    npix = 12 * nside * nside
    phi = np.empty(npix)
    for i in range(1, nside):
        s = 2 * i * (i - 1)
        p = (np.arange(4 * i) + 0.5) * np.pi / (2 * i)
        phi[s:s + 4 * i] = p
        phi[npix - s - 4 * i:npix - s] = p
    ncap = 2 * nside * (nside - 1)
    ib = np.arange(nside, 3 * nside + 1)
    shift = 0.5 * ((ib - nside + 1) & 1)
    phi[ncap:npix - ncap] = ((np.arange(4 * nside)[None, :] + shift[:, None]) * np.pi / (2 * nside)).ravel()
    return phi


MASK_KINDS = ("band", "galplane")
MASK_KIND = "band"   # --mask; read by every make_mask(nside) of this run (both arms, config #4)
MASK_NOTE = {
    "band": "the synthetic input SURVEY.md 8(d) names (and BENCH_r01 ran): axisymmetric galactic band |b| < 11.5 deg, cos taper 2 deg, "
            "f_sky 0.8.  No ring is cut by its edge, so with isotropic noise every ring has ONE pixel weight and the transform-free ring "
            "paths (gs_set_ring_const) serve the whole sky: see the galplane_mask entry for a mask that cuts rings",
    "galplane": "stand-in for the shape of the reference's HFI GalPlane 80 % mask (config.py:26): |b| < b0(l), bulge at l = 0 + ripples "
                "(half width 3 to 33 deg), cos taper 2 deg, f_sky 0.8; its edge CUTS 735 of the 2047 rings at NSIDE 512 (they keep their "
                "FFTs), 994 instead of 883 ring pairs carry weight, and the PCG needs about 3 % more iterations",
}


def make_mask(nside, fsky=0.8, kind=None, edge_deg=2.0):
    """Synthetic stand-in for the reference's sky mask (config.py:26: HFI_Mask_GalPlane-apo0_2048_R2 80 %, a mask of the galactic
    plane in galactic coordinates), cos-tapered over edge_deg, mean = fsky.
    "band" (default; the input SURVEY.md 8(d) names): the axisymmetric band |b| < asin(1 - fsky); no ring is cut, every ring has one
    weight.  "galplane": |b| < b0(l) with a bulge around l = 0 and ripples (half width between about 3 and 33 degrees), so the
    rings near the plane are CUT by the mask edge while the polar caps and the high-latitude belt stay whole, as under the Planck
    mask."""
    kind = kind or MASK_KIND
    z = pixel_z(nside)
    b = np.degrees(np.arcsin(np.abs(z)))        # |latitude|
    if kind == "band":
        b0 = np.degrees(np.arcsin(1.0 - fsky))  # band |b| < b0 removes 1 - fsky of the sky
        t = np.clip((b - b0) / edge_deg + 0.5, 0.0, 1.0)
        return 0.5 * (1 - np.cos(np.pi * t))
    if kind != "galplane":
        raise ValueError("mask kind %r" % (kind,))
    def edge_of(ns):
        phi = pixel_phi(ns)
        dl = np.degrees(phi) - 360.0 * (phi > np.pi)                 # longitude in (-180, 180]
        return 22.0 * np.exp(-(dl / 40.0) ** 2) + 3.0 * np.cos(3 * phi + 1.0) + 1.5 * np.cos(7 * phi + 0.5)

    def mask_for(c, bb, shape):
        t = np.clip((bb - (c + shape)) / edge_deg + 0.5, 0.0, 1.0)
        return 0.5 * (1 - np.cos(np.pi * t))
    ns = min(nside, 128)                                             # base half width c: mean(mask) = fsky, solved at NSIDE <= 128
    bs = b if ns == nside else np.degrees(np.arcsin(np.abs(pixel_z(ns))))
    ss = edge_of(ns)
    lo, hi = 0.0, 40.0
    for _ in range(40):
        c = 0.5 * (lo + hi)
        if mask_for(c, bs, ss).mean() > fsky:
            lo = c
        else:
            hi = c
    return mask_for(0.5 * (lo + hi), b, ss if ns == nside else edge_of(nside))


def bins_for(lmax):
    """EE: one multipole per bin; BB: the shipped Planck-like scheme (config.py:45-46) scaled to lmax."""
    ee = np.arange(0, lmax + 2)
    cut = int(round(396 * lmax / 512))
    tail = np.unique(np.round(np.array([396, 398, 400, 402, 406, 410, 415, 420, 425, 430, 435, 440, 445, 460, 475, 495, 513])
                              * lmax / 512).astype(int))
    tail = tail[tail > cut]
    bb = np.concatenate([np.arange(0, cut + 1), tail])
    bb[-1] = lmax + 1
    return {"EE": ee, "BB": bb}


def blocks_for(lmax, bins, l_cut):
    """Metropolis blocks over the BINNED arrays: EE one block, BB one wide block then one bin per block (the shipped
    scheme, config.py:51-52: [2, 279] + arange(280, n_bins), scaled to lmax); the first block starts at the first
    non-centred bin (l >= l_cut)."""
    first = {p: int(np.searchsorted(np.asarray(bins[p]), max(l_cut, 2), side="left")) for p in ("EE", "BB")}
    nb_bb = len(bins["BB"])
    wide = int(round(279 * lmax / 512))
    return {"EE": np.array([first["EE"], len(bins["EE"]) - 1]),
            "BB": np.concatenate([[first["BB"], wide], np.arange(wide + 1, nb_bb)])}


def proposal_variances_for(lmax, bins, dlE, dlB, noise_var, npix, bl, fsky=0.8):
    """Cosmic-variance-like proposal variances per bin, indexed from bin 2 (config.py:196-197)."""
    ell = np.arange(lmax + 1, dtype=np.float64)
    nl = noise_var * 4 * np.pi / npix * ell * (ell + 1) / (2 * np.pi) / np.maximum(bl, 1e-30) ** 2
    out = {}
    for pol, dl in (("EE", dlE), ("BB", dlB)):
        var_l = 2.0 / ((2 * ell + 1) * fsky) * (dl + nl) ** 2
        e = np.asarray(bins[pol])
        v = np.array([var_l[e[i]:e[i + 1]].sum() / (e[i + 1] - e[i]) ** 2 for i in range(len(e) - 1)])
        out[pol] = 0.3 * v[2:]
    return out


L_CUT = 5  # PNCP: multipoles below l_cut stay centred (recovered config: l_cut = 5)


class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.samples = index, False, []

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(s[0]) for s in self.samples if s[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(len(s) > 2 + k and s[2 + k].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": float(self.samples[0][1]), "reasons": reasons,
                "samples": len(self.samples)}


def cpu_problem(args):
    """The benchmark workload restated for the CPU arm: same spectra, beam, noise level, mask, bins, Metropolis blocks and
    proposal variances as the GPU arm (its own realisation of sky and noise, numpy seed 1234), as the oracle's PolProblem /
    PNCPPol on the vectorised SHT (oracle/sht_fast.c) with the numpy twins of the reference's O(L^2) Python loops."""
    from oracle import reference_logic as R
    from oracle import sht as O
    import scipy.stats  # noqa: F401  (imported here so that no timed step pays for it)
    nside, lmax = args.nside, args.lmax
    npix, nre = 12 * nside * nside, (lmax + 1) ** 2
    dlE, dlB = fiducial(lmax)
    fwhm = 0.5 * (512 // nside) if nside < 512 else 0.5
    bl = O.gauss_beam(np.radians(fwhm), lmax)
    noise_var = 0.04 * npix / 786432.0
    mask = make_mask(nside)
    rng = np.random.default_rng(1234)
    bl_map = R.expand_per_l_vec(bl)
    sE = rng.standard_normal(nre) * np.sqrt(R.generate_var_cl_vec(dlE))
    sB = rng.standard_normal(nre) * np.sqrt(R.generate_var_cl_vec(dlB))
    q, u = R.synth_pol(sE * bl_map, sB * bl_map, nside, lmax, "fast")
    dQ = (q + rng.standard_normal(npix) * np.sqrt(noise_var)) * mask
    dU = (u + rng.standard_normal(npix) * np.sqrt(noise_var)) * mask
    prob = R.PolProblem(nside, lmax, dQ, dU, mask / noise_var, fwhm, kind="fast", vectorised=True)
    bins = bins_for(lmax)
    blocks = blocks_for(lmax, bins, L_CUT)
    pv = proposal_variances_for(lmax, bins, dlE, dlB, noise_var, npix, bl)
    binned = {pol: np.array([dl[bins[pol][i]:bins[pol][i + 1]].mean() for i in range(len(bins[pol]) - 1)])
              for pol, dl in (("EE", dlE), ("BB", dlB))}
    return prob, bins, blocks, pv, binned


def cpu_centered_iteration(prob, bins, binned):
    """One CenteredGibbs iteration on the CPU restatement: sample_mask (CenteredGibbs.py:448-491) + the inverse-gamma draw
    (CenteredGibbs.py:54-93).  Returns (binned, PCG iterations)."""
    from oracle import reference_logic as R
    from scipy.stats import invgamma
    lmax = prob.lmax
    dls = {k: R.unfold_bins(binned[k], bins[k]) for k in ("EE", "BB")}
    xi = [np.random.normal(size=n) for n in (prob.npix, prob.npix, (lmax + 1) ** 2, (lmax + 1) ** 2)]
    bE, bB = prob.rhs(dls["EE"], dls["BB"], *xi)
    sE, sB, it, _ = prob.pcg(dls["EE"], dls["BB"], bE, bB, eps=1e-5)
    out = {}
    for pol, s in (("EE", sE), ("BB", sB)):
        al, be = R.cls_alpha_beta(s, bins[pol], lmax)
        d = be * invgamma.rvs(a=al)
        d[:2] = 0
        out[pol] = d
    return out, it


def host_threads():
    """torchrun exports OMP_NUM_THREADS=1 to its workers; a CPU arm is ONE process that owns the host, so give the OpenMP
    oracle every core (the library reads the variable when it is first loaded)."""
    if "TORCHELASTIC_RUN_ID" in os.environ or os.environ.get("OMP_NUM_THREADS") == "1":
        os.environ["OMP_NUM_THREADS"] = str(os.cpu_count() or 1)
    # numpy's BLAS pool (the PCG dot products) would spin on the same cores as the OpenMP SHT threads: keep BLAS serial
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(limits=1, user_api="blas")
    except Exception:
        pass


def cpu_host_info():
    """Threads, vector ISA and measured DFMA peak of the host cores (all cores busy), for the GFLOP/s-per-core figure."""
    import ctypes as C
    from oracle import sht as O
    lib = O._fast()
    lib.orf_fma_peak_gflops_per_core.restype = C.c_double
    lib.orf_fma_peak_gflops_per_core.argtypes = [C.c_double]
    return {"threads": int(lib.orf_num_threads()), "simd_bits": int(lib.orf_simd_bits()),
            "dfma_peak_gflops_per_core": float(lib.orf_fma_peak_gflops_per_core(1.0))}


def cpu_pair_seconds(nside, lmax, reps, seed=0):
    """Seconds per spin-2 SHT pair (alm2map_spin2 + A^T) of the vectorised CPU port on all host cores, best of reps."""
    from oracle import sht as O
    rng = np.random.default_rng(seed)
    n = O.nalm(lmax)
    e = rng.standard_normal(n) + 1j * rng.standard_normal(n)
    b = rng.standard_normal(n) + 1j * rng.standard_normal(n)
    ts = []
    for _ in range(reps + 1):
        t0 = time.perf_counter()
        q, u = O.alm2map_spin2(e, b, nside, lmax, kind="fast")
        O.map2alm_spin2(q, u, nside, lmax, adjoint=True, kind="fast")
        ts.append(time.perf_counter() - t0)
    return float(np.min(ts[1:]))


def legendre_flops(nside, lmax):
    """SURVEY.md 8d: algorithmic flops of one spin-2 Legendre transform (unpruned): 26 per (ring pair, l, m)."""
    nring = 4 * nside - 1
    n_lm2 = sum(lmax - max(m, 2) + 1 for m in range(lmax + 1))
    return 26.0 * ((nring + 1) // 2) * n_lm2


def python_overhead_term(args, n_blocks):
    """The live reference calls the PURE-PYTHON utils.generate_var_cl (utils.py:114-147; the Cython import is commented out,
    utils.py:5) twice per constrained realization and twice per likelihood evaluation: its cost per Gibbs iteration, timed on
    the restatement of that loop (oracle.reference_logic.generate_var_cl), stated separately and NOT part of `value`."""
    from oracle import reference_logic as R
    dl = fiducial(args.lmax)[0]
    t0 = time.perf_counter()
    R.generate_var_cl(dl)
    t = time.perf_counter() - t0
    calls = 2 + (2 * (n_blocks + 1) if args.sampler == "pncp" else 0)
    return {"generate_var_cl_s_per_call": t, "calls_per_iteration": calls, "s_per_iteration": t * calls,
            "note": "pure-Python O(lmax^2) loop of the live reference (utils.py:114-147), excluded from value: the CPU arm uses "
                    "its vectorised twin, i.e. what the reference's compiled Cython version (variance_expension.pyx:8-33) would cost"}


def cpu_baseline_sample(args, n_pcg, n_blocks):
    """cpu_baseline leg of the GPU arm (rank 0, N = 1): a BOUNDED sample of the same workload on the host cores, about
    10-30 s of CPU work: the RHS, a PCG solve cut after `n_cap` iterations and `n_lik` likelihood evaluations of the
    Metropolis sweep are timed on the CPU restatement and scaled to the iteration counts the GPU run measured.
    (`bench.py --impl reference` runs whole iterations instead.)"""
    host_threads()
    from oracle import reference_logic as R
    prob, bins, blocks, pv, binned = cpu_problem(args)
    host = cpu_host_info()
    pair_s = cpu_pair_seconds(args.nside, args.lmax, 2)
    lmax = args.lmax
    dls = {k: R.unfold_bins(binned[k], bins[k]) for k in ("EE", "BB")}
    np.random.seed(99)
    xi = [np.random.normal(size=n) for n in (prob.npix, prob.npix, (lmax + 1) ** 2, (lmax + 1) ** 2)]
    t0 = time.perf_counter()
    bE, bB = prob.rhs(dls["EE"], dls["BB"], *xi)
    t_rhs = time.perf_counter() - t0
    n_cap = max(4, min(n_pcg, int(8.0 / max(pair_s, 1e-3))))
    t0 = time.perf_counter()
    sE, sB, it, _ = prob.pcg(dls["EE"], dls["BB"], bE, bB, eps=1e-5, itermax=n_cap)
    t_pcg_it = (time.perf_counter() - t0) / max(it, 1)
    t_lik, n_lik = 0.0, 0
    if args.sampler == "pncp":
        n_lik = 8
        s = {"EE": sE, "BB": sB}
        t0 = time.perf_counter()
        for _ in range(n_lik):
            R.nc_loglik(binned, bins, s, prob, L_CUT)
        t_lik = (time.perf_counter() - t0) / n_lik
    t_iter = t_rhs + n_pcg * t_pcg_it + (n_blocks + 1) * t_lik if args.sampler == "pncp" else t_rhs + n_pcg * t_pcg_it
    gf_core = 2 * legendre_flops(args.nside, args.lmax) / pair_s * 1e-9 / host["threads"]
    return {"value": 1.0 / t_iter, "unit": "it/s", "cores": host["threads"], "kind": "port",
            "sample": "bounded: RHS (%.2f s) + %d PCG iterations (%.3f s each) + %d likelihood evaluations (%.3f s each) of the CPU "
                      "restatement (oracle/reference_logic.py on oracle/sht_fast.c) at the full NSIDE/lmax, scaled to the %d PCG "
                      "iterations and %d Metropolis tests + 1 of the GPU run" % (t_rhs, it, t_pcg_it, n_lik, t_lik, n_pcg, n_blocks),
            "sht_pair_s": pair_s, "pairs_per_s": 1.0 / pair_s, "sht_gflops_per_core": gf_core, "simd_bits": host["simd_bits"],
            "dfma_peak_gflops_per_core": host["dfma_peak_gflops_per_core"],
            "sht_fraction_of_host_dfma_peak": gf_core / host["dfma_peak_gflops_per_core"] if host["dfma_peak_gflops_per_core"] else None,
            "reference_python_overhead": python_overhead_term(args, n_blocks)}


def run_reference(args):
    """Reference arm: the reference's own CPU algorithm for the path, on the box's host cores.  healpy / qcinv cannot be
    installed here, so it is the oracle restatement (PolProblem.rhs + .pcg to eps 1e-5, inverse-gamma draw, blocked
    Metropolis sweep with one full spin-2 synthesis per block: oracle/reference_logic.py) on the vectorised SHT port
    (oracle/sht_fast.c).  A timed step is ONE REAL Gibbs iteration at the full NSIDE / lmax; the warm-up steps page the
    tables in and spin the thread pool up with one SHT pair each (a CPU arm has nothing else to warm)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    host_threads()
    from oracle import reference_logic as R
    t_start = time.perf_counter()
    prob, bins, blocks, pv, binned = cpu_problem(args)
    pncp = args.sampler == "pncp"
    n_blocks = len(blocks["EE"]) + len(blocks["BB"]) - 2 if pncp else 0
    host = cpu_host_info()
    pair_s = None
    for _ in range(max(args.warmup, 1)):
        pair_s = cpu_pair_seconds(args.nside, args.lmax, 1)
    np.random.seed(4321)
    pn = R.PNCPPol(prob, bins, blocks, pv, L_CUT) if pncp else None
    t_steps, its, acc = [], [], []
    budget = float(os.environ.get("GS_REF_BUDGET_S", REF_BUDGET_S))
    for k in range(args.steps):
        if t_steps and (time.perf_counter() - t_start) + 1.15 * max(t_steps) > budget:
            break    # out of wall-clock budget: report the iterations that were really run (steps < requested)
        t0 = time.perf_counter()
        if pncp:
            binned, a, _ = pn.iteration(binned)
            its.append(pn.last_pcg_iterations)
            acc.append((sum(a["EE"]) + sum(a["BB"])) / max(1, len(a["EE"]) + len(a["BB"])))
        else:
            binned, it = cpu_centered_iteration(prob, bins, binned)
            its.append(it)
        t_steps.append(time.perf_counter() - t0)
    done = len(t_steps)
    t_iter = float(np.sum(t_steps)) / done
    val = 1.0 / t_iter
    f2 = legendre_flops(args.nside, args.lmax)
    gf_core = 2 * f2 / pair_s * 1e-9 / host["threads"]
    line = {
        "impl": "reference", "metric": "gibbs_iters_per_s", "value": val, "unit": "it/s", "n_gpus": args.gpus, "steps": done,
        "warmup": args.warmup, "ms_per_step": 1e3 * t_iter, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": workload_config(args),
        "steps_requested": args.steps, "seconds_per_step": t_steps, "pcg_iterations_per_step": its,
        "sht_pairs_per_s": 1.0 / pair_s,
        "cpu_baseline": {"value": val, "unit": "it/s", "cores": host["threads"], "kind": "port",
                         "sample": "%d full Gibbs iterations of the CPU restatement at the full NSIDE/lmax (none extrapolated): RHS with "
                                   "map2alm(iter=3), PCG to eps 1e-5 (%s iterations), inverse-gamma draw%s; SHT = oracle/sht_fast.c on all host cores"
                                   % (done, its, ", %d-block Metropolis sweep with one spin-2 synthesis per block" % n_blocks if pncp else ""),
                         "sht_pair_s": pair_s, "sht_gflops_per_core": gf_core, "simd_bits": host["simd_bits"],
                         "dfma_peak_gflops_per_core": host["dfma_peak_gflops_per_core"],
                         "sht_fraction_of_host_dfma_peak": gf_core / host["dfma_peak_gflops_per_core"] if host["dfma_peak_gflops_per_core"] else None,
                         "reference_python_overhead": python_overhead_term(args, n_blocks)},
        "e2e": {"value": val, "unit": "it/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    if pncp:
        line["mwg"] = {"blocks": n_blocks, "mean_accept_rate": float(np.mean(acc)) if acc else None}
    print(json.dumps(line), flush=True)


def chain_seed(rank):
    """Philox seed of the chain owned by `rank` (same data on every rank, independent chains)."""
    return 1000 + rank


def reduce_max_ms(ms_tensor, world):
    """Max over ranks of the device-timed duration (ms); no-op for one rank."""
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(ms_tensor, op=dist.ReduceOp.MAX)
    return float(ms_tensor.item())


def whole_job_value(world, steps, ms):
    """Whole-job throughput: steps of all ranks / max-over-ranks time."""
    return world * steps / (ms * 1e-3)


def pncp_block_count(lmax):
    b = blocks_for(lmax, bins_for(lmax), L_CUT)
    return len(b["EE"]) + len(b["BB"]) - 2


def workload_config(args):
    if args.sampler == "pncp":
        wl = ("PNCP polarised masked sky (BASELINE config #3): PCG constrained realization (eps 1e-5, diag_cl precond) + inverse-gamma "
              "draw of l < %d + blocked Metropolis-within-Gibbs sweep of l >= %d (%d blocks); one independent chain per GPU"
              % (L_CUT, L_CUT, pncp_block_count(args.lmax)))
    else:
        wl = ("CenteredGibbs polarised masked sky: PCG constrained realization (eps 1e-5, diag_cl precond) + inverse-gamma C_l draw; "
              "one independent chain per GPU")
    return {"workload": wl, "sampler": args.sampler,
            "nside": args.nside, "lmax": args.lmax, "fsky": 0.8, "mask": MASK_KIND + ": " + MASK_NOTE[MASK_KIND], "noise": "isotropic (noise_covar * ones, as config.py)",
            "beam_fwhm_deg": 0.5 * max(1, 512 // args.nside) if args.nside < 512 else 0.5,
            "pcg": "eps 1e-5, diag_cl preconditioner, cold start", "chains_per_gpu": 1,
            "l2_policy": "inputs larger than L2: each PCG iteration streams the 67 MB ring-spectra intermediate, 50 MB of maps and 100 MB of "
                         "recurrence/alm vectors (126 MB L2)"}


def run_sharded(args):
    """BASELINE config #4 as its own run (--mode sharded): see sharded_measure."""
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    line = sharded_measure(args.nside, args.lmax, args.steps, args.warmup)
    if line is not None:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def sharded_measure(nside, lmax, steps, warmup):
    """BASELINE config #4: a single CenteredGibbs chain with the m-sharded SHT (NCCL all-to-all ring<->m transpose)
    over all ranks of the (already initialised) process group; strong scaling, value = iterations/s of that one chain.
    Returns the JSON object on rank 0, None elsewhere."""
    import torch
    import torch.distributed as dist
    from gibbssampler_b200 import _dev, _lib, utils
    from gibbssampler_b200.CenteredGibbs import PolarizedCenteredClsSampler, PolarizedCenteredConstrainedRealization
    from gibbssampler_b200.sharded import ShardedPlan
    from gibbssampler_b200.sht import Plan

    class A:
        pass
    args = A()
    args.nside, args.lmax, args.steps, args.warmup = nside, lmax, steps, warmup
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dev = torch.device("cuda", local)
    npix, nre = 12 * nside * nside, (lmax + 1) ** 2
    L = _lib.lib()
    plan = ShardedPlan(nside, lmax) if world > 1 else Plan.get(nside, lmax)
    dlE, dlB = fiducial(lmax)
    fwhm = 0.5 * (512 / nside)
    bl = _dev.gauss_beam(np.radians(fwhm), lmax)
    noise_var = 0.04 * npix / 786432.0
    mask = make_mask(nside)
    # synthetic sky generated shard-locally with the sharded transform (same construction as the chains mode)
    data_rng = _dev.Rng("philox", seed=1234 + 17 * rank)
    sE = data_rng.normal(plan.nreal) * plan.expand_per_l(_dev.f64(dlE), 3)
    sB = data_rng.normal(plan.nreal) * plan.expand_per_l(_dev.f64(dlB), 3)
    q, u = plan.alm2map_spin2(sE, sB, fl=_dev.f64(bl))
    mask_loc = plan.local_map(_dev.f64(mask))
    dQ = (q + data_rng.normal(plan.npix) * np.sqrt(noise_var)) * mask_loc
    dU = (u + data_rng.normal(plan.npix) * np.sqrt(noise_var)) * mask_loc
    bins = bins_for(lmax)
    bl_map = plan.expand_per_l(_dev.f64(bl), 0)
    cr = PolarizedCenteredConstrainedRealization({"Q": dQ, "U": dU}, noise_var * 1e4, noise_var, bl_map, lmax, npix, fwhm,
                                                 mask=mask, rng="philox", seed=5000 + rank, plan=plan)
    cls = PolarizedCenteredClsSampler({"Q": dQ, "U": dU}, lmax, nside, bins, bl_map, noise_var, rng="philox", seed=99,
                                      plan=plan if world > 1 else None)
    state = {"binned": {pol: _dev.f64(np.array([dl[bins[pol][i]:bins[pol][i + 1]].mean() for i in range(len(bins[pol]) - 1)]))
                        for pol, dl in (("EE", dlE), ("BB", dlB))}}
    pcg_its = []

    def step():
        b = state["binned"]
        dls = {"EE": utils.unfold_bins(b["EE"], bins["EE"]), "BB": utils.unfold_bins(b["BB"], bins["BB"])}
        sky, _ = cr.sample_mask(dls)
        pcg_its.append(cr.last_pcg_iterations)
        state["binned"] = cls.sample(sky)

    clocks = ClockSampler(local)
    clocks.start()
    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    launches0 = L.gs_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.barrier()
    ms_total = reduce_max_ms(ms, world)
    launches = int(L.gs_launch_count() - launches0)
    clocks.stop_flag = True
    clocks.join(timeout=2)
    # stage timing of one mat-vec (the all-to-alls are inside the Legendre-stage calls on sharded plans)
    x_e, x_b = data_rng.normal(plan.nreal), data_rng.normal(plan.nreal)
    y_e, y_b = torch.empty_like(x_e), torch.empty_like(x_b)
    ms4 = (C.c_float * 4)()
    for nrep in (3, 20):
        _lib.check(L.gs_profile_matvec(plan._h, _dev.ptr(x_e), _dev.ptr(x_b), _dev.ptr(cr.bl_gauss_d), _dev.ptr(cr.inv_noise_pol),
                                       _dev.ptr(y_e), _dev.ptr(y_b), nrep, ms4, _dev.stream()))
    st = torch.tensor(list(ms4), device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(st, op=dist.ReduceOp.MAX)
    st = [float(x) for x in st.tolist()]
    a2a_ms = C.c_float(0.0)
    if world > 1:
        _lib.check(L.gs_profile_exchange(plan._h, 10, C.byref(a2a_ms), _dev.stream()))
    a2a = torch.tensor([a2a_ms.value], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(a2a, op=dist.ReduceOp.MAX)
    a2a_ms = float(a2a.item())
    its = pcg_its[args.warmup:]
    n_pcg = int(round(float(np.mean(its)))) if its else 0
    nring = 4 * nside - 1
    n_lm2 = sum(lmax - max(m, 2) + 1 for m in range(lmax + 1))
    f2 = 26.0 * ((nring + 1) // 2) * n_lm2
    exch_bytes = 2 * 16.0 * nring * (lmax + 1) * (world - 1) / max(world, 1) / max(world, 1)  # sent per GPU and transform
    if rank == 0:
        line = {
            "metric": "gibbs_iters_per_s", "value": args.steps / (ms_total * 1e-3), "unit": "it/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "CenteredGibbs polarised masked sky, ONE chain, m-sharded SHT with NCCL all-to-all ring<->m transpose "
                                   "(PCG eps 1e-5, diag_cl precond) + inverse-gamma C_l draw", "nside": nside, "lmax": lmax, "fsky": 0.8, "mask": MASK_KIND,
                       "beam_fwhm_deg": fwhm, "parallelism": "m-shard x%d" % world,
                       "l2_policy": "inputs larger than L2"},
            "pcg_iterations_mean": n_pcg, "gpu_launches": launches, "sht_pair_ms": sum(st), "sht_pairs_per_s": 1e3 / sum(st),
            "stage_ms": {"leg_synth+a2a": st[0], "ring_synth": st[1], "ring_anal": st[2], "a2a+leg_anal": st[3]},
            "a2a_ms_alone": a2a_ms, "a2a_blocks": int(os.environ.get("GS_SHARD_NB", "1")),
            "a2a_note": "GS_SHARD_NB=k > 1 runs the ring <-> m all-to-all block of m by block of m on a communication stream, overlapped "
                        "with the Legendre kernels of the neighbouring blocks (default 1: one exchange per transform; 4 blocks "
                        "measured slower on 2 GPUs at NSIDE 1024, profiles/shard_overlap_r02.txt)", "legendre_ms_without_a2a": {"leg_synth": st[0] - a2a_ms, "leg_anal": st[3] - a2a_ms},
            "exposed_communication_fraction_of_pair": 2 * a2a_ms / sum(st) if sum(st) > 0 else None,
            "legendre_tflops_all_gpus": 2 * f2 / (max(st[0] + st[3] - 2 * a2a_ms, 1e-9) * 1e-3) * 1e-12,
            "a2a_bytes_sent_per_gpu_per_transform": exch_bytes,
            "clocks": clocks.summary(), "pcg_iterations_per_step": its,
        }
        return line
    return None


DUMP_BYTES = 60_000_000   # --dump-outputs writes at most this many bytes of data (with the .npy headers, under 64 MB)


def dump_outputs(dirname, arrays):
    """Writes each array as dirname/<name>.npy in float64.  When together they exceed DUMP_BYTES, every array larger than its
    share of that budget is cut to the entries at sorted positions drawn with numpy seed 0: the same positions for the same
    arguments, so the files of two builds compare entry for entry."""
    arrays = {k: np.asarray(v, dtype=np.float64).ravel() for k, v in arrays.items()}
    share = DUMP_BYTES // 8 // len(arrays)
    over = sum(a.size for a in arrays.values()) * 8 > DUMP_BYTES
    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        if over and a.size > share:
            a = a[np.sort(np.random.default_rng(0).choice(a.size, share, replace=False))]
        np.save(os.path.join(dirname, name + ".npy"), a)


def main():
    sys.dont_write_bytecode = True   # the tree may be read-only: nothing imported from it is cached there
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--nside", type=int, default=512)
    ap.add_argument("--lmax", type=int, default=1024)
    ap.add_argument("--pcg-iters", type=int, default=0)
    ap.add_argument("--mask", default="band", choices=list(MASK_KINDS), help="synthetic sky mask, f_sky 0.8 (see make_mask)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-other-mask", "--no-band-mask", dest="no_other_mask", action="store_true",
                    help="skip the secondary measurement under the other synthetic mask (galplane when --mask band, and vice versa)")
    ap.add_argument("--no-chain-batch", action="store_true", help="skip the secondary measurement with two chains per GPU")
    ap.add_argument("--no-config4", action="store_true", help="N >= 2: skip the m-sharded single-chain measurement (BASELINE config #4)")
    ap.add_argument("--config4-nside", type=int, default=2048)
    ap.add_argument("--sampler", default="pncp", choices=["pncp", "centered"],
                    help="pncp (default): BASELINE config #3, partially non-centred polarised masked-sky sampler = PCG constrained "
                         "realization + low-l inverse-gamma draw + high-l blocked Metropolis sweep; centered: CenteredGibbs "
                         "(PCG constrained realization + inverse-gamma draw)")
    ap.add_argument("--mode", default="chains", choices=["chains", "sharded"],
                    help="chains: one independent chain per GPU (weak scaling, the default and the driver's contract); "
                         "sharded: ONE chain whose SHTs are m-sharded over the GPUs (BASELINE config #4, strong scaling)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned to the caller (rank 0's chain) as DIR/<name>.npy: "
                         "alm_EE/BB (constrained realization), binned_dl_EE/BB, accept_EE/BB (Metropolis blocks, pncp), pcg_iterations")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.mode != "chains"):
        ap.error("--dump-outputs writes the outputs of the default path (--impl b200 --mode chains)")
    global MASK_KIND
    MASK_KIND = args.mask
    if args.impl == "reference":
        return run_reference(args)
    if args.mode == "sharded":
        return run_sharded(args)

    import torch
    import torch.distributed as dist
    from gibbssampler_b200 import _dev, _lib, utils
    from gibbssampler_b200.CenteredGibbs import PolarizedCenteredClsSampler, PolarizedCenteredConstrainedRealization
    from gibbssampler_b200.sht import Plan

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    nside, lmax = args.nside, args.lmax
    npix, nre = 12 * nside * nside, (lmax + 1) ** 2
    L = _lib.lib()
    dev = torch.device("cuda", local)

    # ---- synthetic sky (generated with the library's own kernels; same data on every rank, different chains)
    plan = Plan.get(nside, lmax)
    dlE, dlB = fiducial(lmax)
    fwhm = 0.5 * (512 // nside) if nside < 512 else 0.5
    bl = _dev.gauss_beam(np.radians(fwhm), lmax)
    noise_var = 0.04 * npix / 786432.0
    mask = make_mask(nside)
    data_rng = _dev.Rng("philox", seed=1234)
    sE = data_rng.normal(nre) * utils.expand_per_l(_dev.f64(dlE), 3)
    sB = data_rng.normal(nre) * utils.expand_per_l(_dev.f64(dlB), 3)
    q, u = plan.alm2map_spin2(sE, sB, fl=_dev.f64(bl))
    mask_d = _dev.f64(mask)
    skyQ = q + data_rng.normal(npix) * np.sqrt(noise_var)
    skyU = u + data_rng.normal(npix) * np.sqrt(noise_var)
    dQ, dU = skyQ * mask_d, skyU * mask_d
    bins = bins_for(lmax)
    bl_map = utils.expand_per_l(_dev.f64(bl), 0)
    noise_pol = torch.full((npix,), noise_var, dtype=torch.float64, device=dev)
    pncp = args.sampler == "pncp"
    n_blocks = 0
    if pncp:
        from gibbssampler_b200.PNCP import PNCPClsSampler, PNCPConstrainedRealization
        blocks = blocks_for(lmax, bins, L_CUT)
        n_blocks = len(blocks["EE"]) + len(blocks["BB"]) - 2
        pv = proposal_variances_for(lmax, bins, dlE, dlB, noise_var, npix, bl)
        cr = PNCPConstrainedRealization({"Q": dQ, "U": dU}, noise_pol * 1e4, noise_pol, bl_map, lmax, npix, fwhm, mask=mask,
                                        rng="philox", seed=chain_seed(rank), ula=False, l_cut=L_CUT)
        cls = PNCPClsSampler({"Q": dQ, "U": dU}, lmax, nside, bins, bl_map, noise_pol * 1e4, noise_pol, blocks, pv, L_CUT, n_iter=1,
                             mask=mask, rng=cr.rng)
    else:
        cr = PolarizedCenteredConstrainedRealization({"Q": dQ, "U": dU}, noise_pol * 1e4, noise_pol, bl_map, lmax, npix, fwhm,
                                                     mask=mask, rng="philox", seed=chain_seed(rank))
        cls = PolarizedCenteredClsSampler({"Q": dQ, "U": dU}, lmax, nside, bins, bl_map, noise_pol, mask=mask, rng=cr.rng)

    def binned_init():
        out = {}
        for pol, dl in (("EE", dlE), ("BB", dlB)):
            e = bins[pol]
            out[pol] = _dev.f64(np.array([dl[e[i]:e[i + 1]].mean() for i in range(len(e) - 1)]))
        return out

    state = {"binned": binned_init()}
    pcg_its = []

    accepts = []

    def unfold(b):
        return {"EE": utils.unfold_bins(b["EE"], bins["EE"]), "BB": utils.unfold_bins(b["BB"], bins["BB"])}

    def make_step(cr, cls, state, pcg_its, accepts):
        def step():
            b = state["binned"]
            sky, _ = cr.sample_mask(unfold(b))
            pcg_its.append(cr.last_pcg_iterations)
            state["sky"] = sky
            if not pncp:
                state["binned"] = cls.sample(sky)
                return
            b = cls.sample_low_l(sky, b)                       # PNCPGibbs.run_polarization, one iteration
            mixed = cr.to_mixed(sky, unfold(b))
            b, acc = cls.sample_high_l(mixed, b)
            accepts.append((sum(acc["EE"]) + sum(acc["BB"])) / max(1, len(acc["EE"]) + len(acc["BB"])))
            state["binned"], state["accept"] = b, acc
        return step
    step_device = make_step(cr, cls, state, pcg_its, accepts)

    h2d = d2h = 0

    def step_e2e():
        """The same iteration through the reference-facing sample() calls with HOST (numpy) arrays."""
        nonlocal h2d, d2h
        b = state["binned_host"]
        dls = {"EE": np.repeat(b["EE"], np.diff(bins["EE"])), "BB": np.repeat(b["BB"], np.diff(bins["BB"]))}
        sky, _ = cr.sample_mask(dls)                  # H2D: D_l; D2H: alms (numpy out)
        nb = len(b["EE"]) + len(b["BB"])
        if not pncp:
            state["binned_host"] = cls.sample(sky)    # H2D: alms; D2H: binned D_l
            h2d = 8 * (2 * (lmax + 1) + 2 * nre)
            d2h = 8 * (2 * nre + nb)
            return
        sky_d = {k: _dev.f64(v) for k, v in sky.items()}                            # H2D: alms
        b_d = cls.sample_low_l(sky_d, {k: _dev.f64(v) for k, v in b.items()})       # H2D: binned D_l
        mixed = {k: v.cpu().numpy() for k, v in cr.to_mixed(sky_d, unfold(b_d)).items()}   # D2H: mixed alms
        b_h = {k: v.cpu().numpy() for k, v in b_d.items()}                          # D2H: binned D_l
        b, _ = cls.sample_high_l(mixed, b_h)          # H2D: mixed alms, binned; D2H: binned + accept flags
        state["binned_host"] = b
        h2d = 8 * (2 * (lmax + 1) + 2 * nre) + 8 * (2 * nre + nb) + 8 * (2 * nre + nb)
        d2h = 8 * (2 * nre) + 8 * (2 * nre + nb) + 8 * nb + 4 * n_blocks

    counted = {}

    def timed(fn, nwarm, nsteps):
        for _ in range(nwarm):
            fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n0 = L.gs_launch_count()
        e0.record()
        for _ in range(nsteps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        counted["launches"] = int(L.gs_launch_count() - n0)     # kernels of this library launched inside the timed region
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.barrier()
        return reduce_max_ms(ms, world)

    clocks = ClockSampler(local)
    clocks.start()
    pcg_its.clear()
    ms_total = timed(step_device, args.warmup, args.steps)
    if args.dump_outputs and rank == 0:   # now: the passes below run the same sampler again
        last = {"alm_" + p: state["sky"][p].cpu() for p in ("EE", "BB")}
        last.update({"binned_dl_" + p: state["binned"][p].cpu() for p in ("EE", "BB")})
        if pncp:
            last.update({"accept_" + p: state["accept"][p] for p in ("EE", "BB")})
        last["pcg_iterations"] = [pcg_its[-1]]
        dump_outputs(args.dump_outputs, last)
    launches = counted["launches"]
    its_timed = pcg_its[args.warmup:]
    clocks.stop_flag = True
    clocks.join(timeout=2)

    state["binned_host"] = {k: v.cpu().numpy() for k, v in state["binned"].items()}
    ms_e2e = timed(step_e2e, 1, max(1, args.steps))
    e2e_val = whole_job_value(world, max(1, args.steps), ms_e2e)

    value = whole_job_value(world, args.steps, ms_total)
    n_pcg = int(round(float(np.mean(its_timed)))) if its_timed else 0

    # ---- secondary measurement: the same sampler under the OTHER synthetic mask.  The default (band) mask cuts no ring, so with
    # isotropic noise every ring has one weight and neither the mat-vec's ring stage nor the sweep runs an FFT; the galactic-plane-like
    # mask cuts 735 rings, which keep their transforms: both numbers belong next to each other.
    other_kind = "galplane" if MASK_KIND == "band" else "band"
    other_mask = None
    if not args.no_other_mask:
        mask_b = make_mask(nside, kind=other_kind)
        mb_d = _dev.f64(mask_b)
        dQb, dUb = skyQ * mb_d, skyU * mb_d
        if pncp:
            crb = PNCPConstrainedRealization({"Q": dQb, "U": dUb}, noise_pol * 1e4, noise_pol, bl_map, lmax, npix, fwhm, mask=mask_b,
                                             rng="philox", seed=chain_seed(rank), ula=False, l_cut=L_CUT)
            clsb = PNCPClsSampler({"Q": dQb, "U": dUb}, lmax, nside, bins, bl_map, noise_pol * 1e4, noise_pol, blocks, pv, L_CUT, n_iter=1,
                                  mask=mask_b, rng=crb.rng)
        else:
            crb = PolarizedCenteredConstrainedRealization({"Q": dQb, "U": dUb}, noise_pol * 1e4, noise_pol, bl_map, lmax, npix, fwhm,
                                                          mask=mask_b, rng="philox", seed=chain_seed(rank))
            clsb = PolarizedCenteredClsSampler({"Q": dQb, "U": dUb}, lmax, nside, bins, bl_map, noise_pol, mask=mask_b, rng=crb.rng)
        st_b, its_b = {"binned": binned_init()}, []
        ms_b = timed(make_step(crb, clsb, st_b, its_b, []), args.warmup, args.steps)
        other_mask = {"mask": other_kind + ": " + MASK_NOTE[other_kind], "value": whole_job_value(world, args.steps, ms_b), "unit": "it/s",
                      "ms_per_step": ms_b / args.steps, "pcg_iterations_per_step": its_b[args.warmup:], "gpu_launches": counted["launches"]}
        del crb, clsb, dQb, dUb

    # ---- secondary measurement: TWO chains per GPU whose PCG mat-vecs run as chain batches (one Legendre recurrence for both
    # right-hand sides: gs_cr_pcg_pol_batch; BASELINE config #5 / north_star (a) "batched over chains").  `value` above stays the
    # one-chain-per-GPU configuration of BASELINE config #3; this is reported next to it.
    chain_batch = None
    if not args.no_chain_batch:
        from gibbssampler_b200.CenteredGibbs import sample_mask_batch
        if pncp:
            cr2 = PNCPConstrainedRealization({"Q": dQ, "U": dU}, noise_pol * 1e4, noise_pol, bl_map, lmax, npix, fwhm, mask=mask,
                                             rng="philox", seed=chain_seed(rank) + 500, ula=False, l_cut=L_CUT)
            cls2 = PNCPClsSampler({"Q": dQ, "U": dU}, lmax, nside, bins, bl_map, noise_pol * 1e4, noise_pol, blocks, pv, L_CUT, n_iter=1,
                                  mask=mask, rng=cr2.rng)
        else:
            cr2 = PolarizedCenteredConstrainedRealization({"Q": dQ, "U": dU}, noise_pol * 1e4, noise_pol, bl_map, lmax, npix, fwhm,
                                                          mask=mask, rng="philox", seed=chain_seed(rank) + 500)
            cls2 = PolarizedCenteredClsSampler({"Q": dQ, "U": dU}, lmax, nside, bins, bl_map, noise_pol, mask=mask, rng=cr2.rng)
        cr2.inv_noise_pol = cr.inv_noise_pol
        pair = [(cr, cls), (cr2, cls2)]
        pstate = [state["binned"], binned_init()]
        pair_its = []

        def step_pair():
            outs = sample_mask_batch([c for c, _ in pair], [unfold(b) for b in pstate])
            pair_its.append([c.last_pcg_iterations for c, _ in pair])
            for k, ((c, s), (sky, _)) in enumerate(zip(pair, outs)):
                if not pncp:
                    pstate[k] = s.sample(sky)
                    continue
                b = s.sample_low_l(sky, pstate[k])
                mixed = c.to_mixed(sky, unfold(b))
                pstate[k], _ = s.sample_high_l(mixed, b)

        ms_pair = timed(step_pair, max(1, args.warmup - 1), args.steps)
        xx = data_rng.normal(4 * nre).reshape(2, 2, nre)
        yy = torch.empty_like(xx)
        ms3 = (C.c_float * 3)()
        for nrep in (3, 20):
            _lib.check(L.gs_profile_matvec_batch(plan._h, 2, _dev.ptr(xx[0, 0]), _dev.ptr(xx[0, 1]), 2 * nre, _dev.ptr(cr.bl_gauss_d),
                                                 _dev.ptr(cr.inv_noise_pol), _dev.ptr(yy[0, 0]), _dev.ptr(yy[0, 1]), nrep, ms3, _dev.stream()))
        chain_batch = {"chains_per_gpu": 2, "value": whole_job_value(world, 2 * args.steps, ms_pair), "unit": "it/s",
                       "ms_per_step_of_two_chains": ms_pair / args.steps, "gpu_launches": counted["launches"],
                       "pcg_iterations_per_step": pair_its[max(1, args.warmup - 1):],
                       "pcg_matvec_two_chains_ms": {"leg_synth": ms3[0], "ring_apply_fused": ms3[1], "leg_anal": ms3[2], "total": sum(ms3)},
                       "note": "two independent chains per GPU; their PCG solves share the Legendre recurrences (two right-hand sides per "
                               "launch, 4 + 8 K DFMA per ring pair and multipole instead of 12 K); C_l sampling per chain"}

    # ---- per-kernel timing of one PCG mat-vec (CUDA events on the launching stream) + roofline
    x_e, x_b = data_rng.normal(nre), data_rng.normal(nre)
    y_e, y_b = torch.empty_like(x_e), torch.empty_like(x_b)
    def profile_matvec(skip_idle_rings):
        ms4 = (C.c_float * 4)()
        old = L.gs_set_ring_skip(1 if skip_idle_rings else 0)
        try:
            for nrep in (3, 20):
                _lib.check(L.gs_profile_matvec(plan._h, _dev.ptr(x_e), _dev.ptr(x_b), _dev.ptr(cr.bl_gauss_d), _dev.ptr(cr.inv_noise_pol),
                                               _dev.ptr(y_e), _dev.ptr(y_b), nrep, ms4, _dev.stream()))
        finally:
            L.gs_set_ring_skip(old)
        if ms4[2] == 0.0:   # the PCG's ring stage is one kernel (synthesis -> N^-1 -> analysis per ring)
            return {"leg_synth": ms4[0], "ring_apply_fused": ms4[1], "leg_anal": ms4[3]}
        return {"leg_synth": ms4[0], "ring_synth": ms4[1], "ring_anal": ms4[2], "leg_anal": ms4[3]}

    # all rings: the spin-2 SHT pair of the metric and the launch the roofline is quoted on; idle rings skipped: the mat-vec
    # as the PCG of this workload runs it (rings wholly inside the mask carry N^-1 = 0 and are left out)
    stage_ms = profile_matvec(False)
    old_const = L.gs_set_ring_const(0)
    matvec_tr_ms = profile_matvec(True)     # every ring with weight through its transforms (the mat-vec of r01 / r02a)
    L.gs_set_ring_const(old_const)
    matvec_ms = profile_matvec(True)
    act, tot, nconst = C.c_int(0), C.c_int(0), C.c_int(0)
    _lib.check(L.gs_active_ring_pairs(plan._h, C.byref(act), C.byref(tot)))
    _lib.check(L.gs_constant_rings(plan._h, C.byref(nconst)))
    fused_ring = "ring_apply_fused" in stage_ms
    pair_ms = sum(stage_ms.values())
    peak = C.c_double(0.0)
    _lib.check(L.gs_measure_fp64_peak(C.byref(peak), _dev.stream()))
    nring = 4 * nside - 1
    n_lm2 = sum(lmax - max(m, 2) + 1 for m in range(lmax + 1))
    f2 = 26.0 * ((nring + 1) // 2) * n_lm2                 # SURVEY.md 8d: flops of one spin-2 Legendre transform (unpruned)
    dom = max(("leg_synth", "leg_anal"), key=lambda k: stage_ms[k])
    ach = f2 / (stage_ms[dom] * 1e-3) * 1e-12

    def ncu_traffic(prefix):
        """DRAM bytes per launch (read + write) of the kernel from the committed ncu --set full capture, or None."""
        for fn in ("traffic_r02.json", "traffic_r01.json"):   # this round's capture first (the ring kernel was last captured in r01)
            try:
                t = json.load(open(os.path.join(ROOT, "profiles", fn)))["kernels"]
                k = next(v for name, v in t.items() if name.startswith(prefix))
                return k["dram_bytes_read"] + k["dram_bytes_write"]
            except Exception:
                continue
        return None

    at_bench_size = nside == 512 and lmax == 1024
    roofline = {"kernel": "leg_anal_kernel<2,4,0,1>" if dom == "leg_anal" else "leg_synth_kernel<2,2,0,1>", "bound": "fp64",
                "achieved": ach, "peak": peak.value, "unit": "TFLOP/s", "frac": ach / peak.value if peak.value else None,
                "traffic": ncu_traffic(dom + "_kernel") if at_bench_size else None,
                "traffic_source": "profiles/traffic_r02.json (ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum per launch)",
                "peak_source": "DFMA microkernel measured in this run (MEASURED_PEAKS.json has no FP64 figure; nominal 37.2 TFLOP/s)",
                "algorithmic_flops_per_launch": f2, "ms_per_launch": stage_ms[dom],
                "both_legendre_kernels_tflops": 2 * f2 / ((stage_ms["leg_synth"] + stage_ms["leg_anal"]) * 1e-3) * 1e-12}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        hbm_peak, hbm_src = peaks["hbm_gbs"], "MEASURED_PEAKS.json"
    except Exception:
        hbm_peak, hbm_src = 6650.0, "fallback"
    if fused_ring:
        # ring spectra (Q,U) read and written in place + the N^-1 map; the pixels never leave shared memory
        ring_bytes = 2 * 2 * 16.0 * nring * (lmax + 1) + 8.0 * npix
        ring_ms, ring_kernel = stage_ms["ring_apply_fused"], "ring_apply_kernel"
    else:
        ring_bytes = 2 * 16.0 * nring * (lmax + 1) + 2 * 8.0 * npix      # ring spectra (Q,U) + maps (Q,U), one direction
        ring_ms = max(stage_ms["ring_synth"], stage_ms["ring_anal"])
        ring_kernel = "ring_synth_kernel" if stage_ms["ring_synth"] >= stage_ms["ring_anal"] else "ring_anal_kernel"
    roofline_hbm = {"kernel": ring_kernel, "bound": "hbm", "achieved": ring_bytes / (ring_ms * 1e-3) * 1e-9,
                    "peak": hbm_peak, "unit": "GB/s", "frac": ring_bytes / (ring_ms * 1e-3) * 1e-9 / hbm_peak,
                    "traffic": ncu_traffic(ring_kernel) if at_bench_size else None,
                    "peak_source": hbm_src, "algorithmic_bytes_per_launch": ring_bytes,
                    "note": "every ring through its transforms (random-like weights): the ring stage of a stand-alone SHT pair"}
    if fused_ring and "ring_apply_fused" in matvec_ms:
        # the same kernel as the PCG of this workload launches it: idle ring pairs dropped, constant-weight rings without transforms
        frac_active = 2.0 * act.value / nring
        pcg_ring_bytes = ring_bytes * frac_active
        roofline_hbm["as_run_by_the_pcg"] = {
            "ms": matvec_ms["ring_apply_fused"], "algorithmic_bytes_per_launch": pcg_ring_bytes,
            "achieved": pcg_ring_bytes / (matvec_ms["ring_apply_fused"] * 1e-3) * 1e-9,
            "frac": pcg_ring_bytes / (matvec_ms["ring_apply_fused"] * 1e-3) * 1e-9 / hbm_peak,
            "constant_weight_rings": nconst.value, "rings_with_weight": 2 * act.value, "rings": nring}

    # the HBM-bound vector kernels of one PCG iteration (algorithmic bytes: 4 + 7 + 4 arrays of 8 N_re bytes per field)
    ms3 = (C.c_float * 3)()
    _lib.check(L.gs_profile_pcg_vectors(plan._h, 2, 20, ms3, _dev.stream()))
    # r02: C^-1_l and M_l come from per-l tables through a 2-byte multipole index per coefficient: 3 + 6 + 3 passes over 8 N_re bytes
    # per field (+ the index) instead of 4 + 7 + 4
    vec_bytes = [(3 * 8.0 + 2.0) * 2 * nre, (6 * 8.0 + 2.0) * 2 * nre, (3 * 8.0 + 2.0) * 2 * nre]

    def copy_gbs(total_bytes, nrep=20):
        """A plain device copy that moves the same number of bytes (half read, half written), timed like the kernels above: each
        launch alone after a write larger than L2.  What a launch of this SIZE can reach on this GPU (the 6.5 TB/s of
        MEASURED_PEAKS.json is a 4 GiB copy; a 50-100 MB launch lasts 10-20 us and pays its ramp and tail)."""
        nn = int(total_bytes // 16)
        a, b = torch.zeros(nn, dtype=torch.float64, device=dev), torch.empty(nn, dtype=torch.float64, device=dev)
        flush = torch.empty(20_000_000, dtype=torch.float64, device=dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        acc = 0.0
        for rep in range(-2, nrep):
            flush.fill_(0.0)
            e0.record()
            b.copy_(a)
            e1.record()
            e1.synchronize()
            if rep >= 0:
                acc += e0.elapsed_time(e1)
        return 16.0 * nn / (acc / nrep * 1e-3) * 1e-9
    copy_same = [copy_gbs(vb) for vb in vec_bytes]
    roofline_pcg = {"kernel": "pcg_apq + pcg_update + pcg_dir", "bound": "hbm",
                    "achieved": sum(vec_bytes) / (sum(ms3) * 1e-3) * 1e-9, "peak": hbm_peak, "unit": "GB/s",
                    "frac": sum(vec_bytes) / (sum(ms3) * 1e-3) * 1e-9 / hbm_peak, "traffic": None, "peak_source": hbm_src,
                    "algorithmic_bytes_per_iteration": sum(vec_bytes), "survey_minimum_bytes_per_iteration": 10 * 2 * 8.0 * nre,
                    "frac_of_peak_on_survey_minimum": 10 * 2 * 8.0 * nre / (sum(ms3) * 1e-3) * 1e-9 / hbm_peak,
                    "ms": {"pcg_apq": ms3[0], "pcg_update": ms3[1], "pcg_dir": ms3[2]},
                    "gb_per_s": {"pcg_apq": vec_bytes[0] / ms3[0] * 1e-6, "pcg_update": vec_bytes[1] / ms3[1] * 1e-6,
                                 "pcg_dir": vec_bytes[2] / ms3[2] * 1e-6},
                    "copy_of_the_same_size_gb_per_s": {"pcg_apq": copy_same[0], "pcg_update": copy_same[1], "pcg_dir": copy_same[2]},
                    "frac_of_same_size_copy": sum(vec_bytes) / (sum(ms3) * 1e-3) * 1e-9
                                              / (sum(vec_bytes) / sum(vb / cs for vb, cs in zip(vec_bytes, copy_same))),
                    "note": "each launch timed alone after a write of the 134 MB analysis workspace (L2 flushed), as inside a PCG iteration; "
                            "copy_of_the_same_size = torch copy_ moving as many bytes, timed the same way: the attainable rate of a launch "
                            "of 50-100 MB"}

    # the SHT pair is timed on EVERY rank; the whole-job pairs/s uses the slowest rank's time
    pair_t = torch.tensor([pair_ms], device=dev, dtype=torch.float64)
    pair_ms_max = reduce_max_ms(pair_t, world)

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_baseline = cpu_baseline_sample(args, n_pcg, n_blocks)

    # ---- BASELINE config #4 on the same ranks (N >= 2): ONE chain at NSIDE 2048 / lmax 4096 whose SHTs are m-sharded over
    # the GPUs with an NCCL all-to-all ring <-> m transpose (strong scaling); reported next to the chains-per-GPU value
    config4 = None
    if world > 1 and not args.no_config4:
        try:
            torch.cuda.empty_cache()
            config4 = sharded_measure(args.config4_nside, 2 * args.config4_nside, 2, 1)
        except Exception as e:   # the headline measurement above stands on its own
            config4 = {"error": "%s: %s" % (type(e).__name__, e)} if rank == 0 else None

    if rank == 0:
        line = {
            "metric": "gibbs_iters_per_s", "value": value, "unit": "it/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": workload_config(args), "pcg_iterations_mean": n_pcg,
            "e2e": {"value": e2e_val, "unit": "it/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": launches, other_kind + "_mask": other_mask, "chain_batch": chain_batch, "config4_m_sharded": config4,
            "sht_pairs_per_s": world * 1e3 / pair_ms_max, "sht_pair_ms": pair_ms_max, "stage_ms": stage_ms,
            "pcg_matvec": {"ms": sum(matvec_ms.values()), "stage_ms": matvec_ms, "active_ring_pairs": act.value, "ring_pairs": tot.value,
                           "constant_weight_rings": nconst.value, "rings": 4 * nside - 1,
                           "stage_ms_all_transforms": matvec_tr_ms,
                           "note": "mat-vec of the PCG: ring pairs wholly inside the mask (N^-1 = 0) are skipped, exact; rings whose N^-1 is "
                                   "one number (isotropic noise, ring not cut by the mask edge; idle rings count) skip their FFTs: n w times "
                                   "the alias-folded spectrum (gs_set_ring_const); stage_ms_all_transforms = the same mat-vec with that off"},
            "roofline": roofline, "roofline_hbm": roofline_hbm, "roofline_pcg": roofline_pcg, "cpu_baseline": cpu_baseline, "clocks": clocks.summary(),
            "pcg_iterations_per_step": its_timed,
        }
        if pncp:
            line["mwg"] = {"blocks": n_blocks, "mean_accept_rate": float(np.mean(accepts[args.warmup:])) if accepts[args.warmup:] else None,
                           "path": "gs_mwg_sweep_blocks (one Legendre pass per block group + batched ring FFT)"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
