"""Joint T/E/B constrained realization on a cut sky (gs_cr_pcg_teb) at NSIDE 512 / lmax 1024: PCG iterations and time of the
masked joint solve, the mat-vec split into its spin-0 half, spin-2 half and vector kernels (CUDA events,
gs_profile_matvec_teb), the vector kernels' bytes and share of HBM peak, masked JointGibbs iterations per second, and the E/B-only
solve on the same P mask for context.  T mask: bench.make_mask "galplane"; P mask: "band".  With --bins planck it measures the
binned joint sampler instead (planck_bins): masked JointGibbs it/s with bins, and the binned C_l step alone (CUDA events) next to
the per-l one.  Writes one JSON line (stdout, and --out if given).  Needs a GPU."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.dont_write_bytecode = True
import bench  # noqa: E402
from gibbssampler_b200 import _dev, _lib, utils  # noqa: E402
from gibbssampler_b200.JointSampler import JointClsSampler, JointConstrainedRealization, JointGibbs  # noqa: E402
from gibbssampler_b200.sht import Plan  # noqa: E402

HBM_PEAK = 7.7e12   # B/s, one B200 (data sheet); the share below is bytes moved / kernel time / this
TT_FORMULA = "D^TT_l = 30 (exp(-(l/900)^2) + 0.05), D^TE_l = 0.5 sqrt(D^TT_l D^EE_l) cos(l/60) for l >= 2 (0 below); " \
             "D^EE_l, D^BB_l = bench.fiducial"


def fiducial_teb(lmax):
    ell = np.arange(lmax + 1, dtype=np.float64)
    ee, bb = bench.fiducial(lmax)
    tt = np.where(ell >= 2, 30.0 * (np.exp(-(ell / 900.0) ** 2) + 0.05), 0.0)
    te = 0.5 * np.sqrt(tt * ee) * np.cos(ell / 60.0)
    return {"TT": tt, "TE": te, "EE": ee, "BB": bb}


def planck_bins(lmax):
    """TT/TE/EE: one multipole per bin up to l = 30, then bins of width 10 (the last one ends at lmax + 1); BB: the Planck-like
    edges of bench.bins_for."""
    tt = np.unique(np.concatenate([np.arange(0, min(lmax, 30) + 1), np.arange(40, lmax + 1, 10), [lmax + 1]]))
    return {"TT": tt, "BB": np.asarray(bench.bins_for(lmax)["BB"])}


def cuda_ms(fn, nrep):
    """mean time of fn() between two CUDA events over nrep calls, after one warm-up call"""
    fn()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(nrep):
        fn()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / nrep


def binned_report(a, data, noise_T, noise_P, fwhm, maskT, maskP, dls):
    """masked JointGibbs with planck_bins (it/s) and the C_l step alone, binned and per l"""
    lmax = a.lmax
    bins = planck_bins(lmax)
    binned = {k: dls[k][bins["BB" if k == "BB" else "TT"][:-1]] for k in dls}   # D at the first multipole of each bin
    gs = JointGibbs(data, noise_T, noise_P, fwhm, a.nside, lmax, n_iter=1, mask=maskT, mask_pol=maskP, bins=bins, seed=11)
    gs.run(binned)
    gs.n_iter = a.gibbs_iters
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    gs.run(binned)
    torch.cuda.synchronize()
    gibbs_s = time.perf_counter() - t0
    unfolded = {k: utils.unfold_bins(v, bins["BB" if k == "BB" else "TT"]) for k, v in binned.items()}
    sky, _ = gs.constrained_sampler.sample(unfolded)
    per_l = JointClsSampler(lmax, seed=12)
    ch = gs.cls_sampler.empirical(sky)
    nt = len(bins["TT"]) - 1
    out = [torch.empty(nt, dtype=torch.float64, device="cuda") for _ in range(3)]
    e_tt = _dev.i32(bins["TT"])
    L = _lib.lib()

    def kernel():
        _lib.check(L.gs_cls_invwishart_binned(*[_dev.ptr(ch[k]) for k in ("TT", "TE", "EE")], lmax, _dev.ptr(e_tt), nt, None,
                                              gs.cls_sampler.rng.seed, 1, *[_dev.ptr(o) for o in out], _dev.stream()))

    return {
        "what": "binned joint T/E/B sampler: masked JointGibbs(bins=) and the binned C_l step (gs_cls_invwishart_binned + "
                "gs_cls_invgamma)",
        "nside": a.nside, "lmax": lmax, "beam_fwhm_deg": fwhm,
        "mask_T": "bench.make_mask galplane, f_sky 0.8", "mask_P": "bench.make_mask band, f_sky 0.8",
        "noise": "isotropic per pixel: noise_P = %.4g (bench.py), noise_T = noise_P / 2" % noise_P,
        "spectra": TT_FORMULA, "pcg_eps": gs.constrained_sampler.pcg_accuracy,
        "bins": "TT/TE/EE: one l per bin to l = 30, width 10 above (%d bins); BB: bench.bins_for (%d bins)"
                % (nt, len(bins["BB"]) - 1),
        "joint_gibbs_binned_it_per_s": round(a.gibbs_iters / gibbs_s, 3), "joint_gibbs_iters_timed": a.gibbs_iters,
        "cl_step_ms": {"binned": round(cuda_ms(lambda: gs.cls_sampler.sample(sky), a.nrep), 4),
                       "per_l": round(cuda_ms(lambda: per_l.sample(sky), a.nrep), 4),
                       "invwishart_binned_kernel": round(cuda_ms(kernel, a.nrep), 4)},
        "cl_step_note": "CUDA events around nrep calls after one warm-up: JointClsSampler.sample (4 cross spectra, the TT/TE/EE "
                        "draw, the BB draw and their host-side launches) and the binned inverse-Wishart launch alone",
        "nrep": a.nrep,
    }


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=20).stdout.strip().splitlines()[0]
        name, plim, smax = [x.strip() for x in out.split(",")]
        return {"device": name, "power_limit_w": float(plim), "sm_clock_max_mhz": float(smax)}
    except Exception as e:   # the device name still comes from torch
        return {"device": torch.cuda.get_device_name(), "power_limit_w": None, "nvidia_smi": repr(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nside", type=int, default=512)
    ap.add_argument("--lmax", type=int, default=1024)
    ap.add_argument("--solves", type=int, default=3)
    ap.add_argument("--gibbs-iters", type=int, default=4)
    ap.add_argument("--nrep", type=int, default=20)
    ap.add_argument("--bins", choices=("none", "planck"), default="none")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("teb_timing.py needs a GPU")
    nside, lmax = a.nside, a.lmax
    npix, n = 12 * nside ** 2, (lmax + 1) ** 2
    L = _lib.lib()
    plan = Plan.get(nside, lmax)
    fwhm = 0.5
    bl = _dev.gauss_beam(np.radians(fwhm), lmax)
    noise_P = 0.04 * npix / 786432.0          # bench.py's polarisation noise per pixel
    noise_T = 0.5 * noise_P
    dls = fiducial_teb(lmax)
    # simulated sky: (T, E) correlated per l through the lower Cholesky factor of the TE block, B independent
    rng = np.random.default_rng(1234)
    f = np.array([2 * np.pi / (l * (l + 1)) if l else 0.0 for l in range(lmax + 1)])
    a_, b_, d_ = dls["TT"] * f, dls["TE"] * f, dls["EE"] * f
    l11 = np.sqrt(a_)
    l21 = np.divide(b_, l11, out=np.zeros_like(b_), where=l11 > 0)
    l22 = np.sqrt(np.maximum(d_ - l21 ** 2, 0.0))
    from oracle import reference_logic as R
    lof = R.l_of_real_layout(lmax)
    z = rng.standard_normal((3, n))
    sT, sE, sB = l11[lof] * z[0], l21[lof] * z[0] + l22[lof] * z[1], np.sqrt(dls["BB"] * f)[lof] * z[2]
    dev = lambda x: torch.as_tensor(np.ascontiguousarray(x), device="cuda")
    mI = plan.alm2map(dev(sT), fl=bl)
    mQ, mU = plan.alm2map_spin2(dev(sE), dev(sB), fl=bl)
    maskT, maskP = bench.make_mask(nside, 0.8, "galplane"), bench.make_mask(nside, 0.8, "band")
    data = {"I": (mI + dev(rng.standard_normal(npix) * np.sqrt(noise_T))) * dev(maskT),
            "Q": (mQ + dev(rng.standard_normal(npix) * np.sqrt(noise_P))) * dev(maskP),
            "U": (mU + dev(rng.standard_normal(npix) * np.sqrt(noise_P))) * dev(maskP)}
    if a.bins == "planck":
        res = binned_report(a, data, noise_T, noise_P, fwhm, maskT, maskP, dls)
        res.update(gpu_info())
        emit(res, a.out)
        return
    cr = JointConstrainedRealization(data, noise_T, noise_P, bl, lmax, npix, mask=maskT, mask_pol=maskP, seed=7)
    dd = {k: dev(v) for k, v in dls.items()}

    # masked joint solve (PCG eps 1e-6, the sampler's default); one warm-up solve
    its, ms = [], []
    for k in range(a.solves + 1):
        rhs = cr.build_rhs(dls)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        cr.solve(dls, *rhs)
        torch.cuda.synchronize()
        if k:
            ms.append((time.perf_counter() - t0) * 1e3)
            its.append(cr.last_pcg_iterations)
    # mat-vec split
    out5 = (C.c_float * 5)()
    _lib.check(L.gs_profile_matvec_teb(plan._h, _dev.ptr(cr.bl), _dev.ptr(cr.inv_noise_T), _dev.ptr(cr.inv_noise_P), a.nrep, out5,
                                       _dev.stream()))
    spin0, spin2, apq, upd, dirk = [float(x) for x in out5]
    arrays = {"apq": 6, "update": 18, "dir": 9}   # arrays of 8 n bytes each kernel reads or writes (T, E, B)
    vec_ms = apq + upd + dirk
    vec_bytes = 8.0 * n * sum(arrays.values())
    # E/B-only solve on the same P mask, on the E/B part of the joint right-hand side
    rhs = cr.build_rhs(dls)
    xe, xb = torch.empty(n, dtype=torch.float64, device="cuda"), torch.empty(n, dtype=torch.float64, device="cuda")
    eb_ms, eb_its = [], []
    for k in range(a.solves + 1):
        nit, res = C.c_int(0), C.c_double(0.0)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        rc = L.gs_cr_pcg_pol(plan._h, _dev.ptr(dd["EE"]), _dev.ptr(dd["BB"]), _dev.ptr(cr.bl), _dev.ptr(cr.inv_noise_P),
                             cr.ninvP_sum_over_4pi, _dev.ptr(rhs[1]), _dev.ptr(rhs[2]), _dev.ptr(xe), _dev.ptr(xb), 0, cr.pcg_accuracy,
                             cr.pcg_itermax, 8, C.byref(nit), C.byref(res), _dev.stream())
        torch.cuda.synchronize()
        if rc not in (0, -3):
            _lib.check(rc)
        if k:
            eb_ms.append((time.perf_counter() - t0) * 1e3)
            eb_its.append(nit.value)
    # masked JointGibbs: CR + inverse-Wishart / inverse-gamma C_l step per iteration (one warm-up iteration)
    gs = JointGibbs(data, noise_T, noise_P, fwhm, nside, lmax, n_iter=1, mask=maskT, mask_pol=maskP, seed=11)
    gs.run(dls)
    gs.n_iter = a.gibbs_iters
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    gs.run(dls)
    torch.cuda.synchronize()
    gibbs_s = time.perf_counter() - t0
    res = {
        "what": "joint T/E/B masked constrained realization (gs_cr_pcg_teb)",
        "nside": nside, "lmax": lmax, "beam_fwhm_deg": fwhm,
        "mask_T": "bench.make_mask galplane, f_sky 0.8", "mask_P": "bench.make_mask band, f_sky 0.8",
        "noise": "isotropic per pixel: noise_P = %.4g (bench.py), noise_T = noise_P / 2" % noise_P,
        "spectra": TT_FORMULA, "pcg_eps": cr.pcg_accuracy,
        "joint_solve": {"iterations": its, "ms": [round(x, 2) for x in ms], "ms_median": round(float(np.median(ms)), 2)},
        "matvec_ms": {"spin0_half_T": round(spin0, 4), "spin2_half_P": round(spin2, 4), "vectors": round(vec_ms, 4),
                      "vector_kernels": {"apq": round(apq, 4), "update": round(upd, 4), "dir": round(dirk, 4)}},
        "vector_bytes_per_iteration": int(vec_bytes),
        "vector_bytes_note": "33 arrays of 8 (lmax+1)^2 bytes: apq reads p, q (6); update reads x, p, q, r and writes x, r (18); "
                             "dir reads p, r and writes p (9); per-l tables and the 2-byte l index are not counted",
        "vector_hbm_fraction": round(vec_bytes / (vec_ms * 1e-3) / HBM_PEAK, 3) if vec_ms > 0 else None,
        "hbm_peak_assumed_Bps": HBM_PEAK,
        "eb_only_solve_same_P_mask": {"iterations": eb_its, "ms": [round(x, 2) for x in eb_ms],
                                      "ms_median": round(float(np.median(eb_ms)), 2)},
        "joint_gibbs_it_per_s": round(a.gibbs_iters / gibbs_s, 3), "joint_gibbs_iters_timed": a.gibbs_iters,
        "per_iteration_ms_estimate": round(spin0 + spin2 + vec_ms, 4),
    }
    res.update(gpu_info())
    emit(res, a.out)


def emit(res, out):
    line = json.dumps(res)
    print(line)
    if out:
        os.makedirs(os.path.dirname(out) or ".", exist_ok=True)
        with open(out, "a") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
