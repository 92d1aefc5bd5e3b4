"""Blackwell-Rao estimator timing on one GPU: the fused GEMM + log-mean-exp (gs_br_logmeanexp) against the torch composition
torch.logsumexp(c[:, None] + S^T W + e, 0) on the same inputs, alternated in the same run, and the per-bin marginals.

sigma is synthetic (no chain): for each sample, (2l+1) Chat_l ~ Wishart(2l+1, C_l) for the (TT, TE; TE, EE) block and
(2l+1) Chat_l / C_l ~ chi^2_{2l+1} for BB, around bench.fiducial (EE, BB; TT = 30 EE, TE = 0.5 sqrt(TT EE)), fixed seed.
Shapes: (A) N = 65536 samples, M = 8192 models, joint per l, l = 2..31; (B) the same with M = 1 (one parameter-MCMC call);
(C) N = 16384, M = 4096, TT/TE/EE one l per bin to 30 and width 10 above to 1024, BB edges of bench.bins_for(1024);
(D) marginals, N = 65536, EE per l to 1024, 256 grid points.  Writes one JSON line per shape to --out."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
from gibbssampler_b200 import _lib  # noqa: E402
from gibbssampler_b200._dev import ptr, stream  # noqa: E402
from gibbssampler_b200.BlackwellRao import BlackwellRao  # noqa: E402


def fiducial_cl(lmax):
    ell = np.arange(lmax + 1, dtype=np.float64)
    dlE, dlB = bench.fiducial(lmax)
    dlT = 30.0 * dlE
    dlTE = 0.5 * np.sqrt(dlT * dlE)
    f = np.where(ell >= 2, 2 * np.pi / np.maximum(ell * (ell + 1), 1), 0.0)
    return {"TT": dlT * f, "TE": dlTE * f, "EE": dlE * f, "BB": dlB * f}


def draw_sigma(n, lmax, rng, keys=("TT", "TE", "EE", "BB")):
    cl = fiducial_cl(lmax)
    out = {k: np.zeros((n, lmax + 1)) for k in keys}
    for l in range(2, lmax + 1):
        k = 2 * l + 1
        if "TT" in keys:
            # Bartlett: k Chat = Lc A A^T Lc^T, A = [[sqrt(chi2_k), 0], [N(0,1), sqrt(chi2_{k-1})]]
            cov = np.array([[cl["TT"][l], cl["TE"][l]], [cl["TE"][l], cl["EE"][l]]])
            lc = np.linalg.cholesky(cov)
            a11, a21, a22 = np.sqrt(rng.chisquare(k, n)), rng.standard_normal(n), np.sqrt(rng.chisquare(k - 1, n))
            b00, b10, b11 = lc[0, 0] * a11, lc[1, 0] * a11 + lc[1, 1] * a21, lc[1, 1] * a22
            out["TT"][:, l], out["TE"][:, l], out["EE"][:, l] = b00 * b00 / k, b00 * b10 / k, (b10 * b10 + b11 * b11) / k
        elif "EE" in keys:
            out["EE"][:, l] = cl["EE"][l] * rng.chisquare(k, n) / k
        if "BB" in keys:
            out["BB"][:, l] = cl["BB"][l] * rng.chisquare(k, n) / k
    return out


def models(br, m, rng):
    """m models scattered by 3 % around the mean of the sample conditional modes"""
    out = {}
    for k in br.keys:
        nb = br.nbins[k]
        e = br.edges[k]
        sig = br.sigma[k].mean(0).cpu().numpy()
        ell = np.arange(len(sig))
        dl = sig * ell * (ell + 1) / (2 * np.pi)
        base = np.array([dl[e[b]:e[b + 1]].mean() for b in range(nb)])
        base[:2] = 1.0
        scale = 0.03 if k != "TE" else 0.01
        out[k] = base[None, :] * (1 + scale * rng.standard_normal((m, nb)))
    return out


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as exc:  # reported, not guessed
        q = "unavailable (%s)" % exc
    return name, q


def time_pair(fused, ref, reps):
    """alternate fused / ref, CUDA events around each call -> (fused ms list, ref ms list)"""
    tf, tr = [], []
    for _ in range(reps):
        for fn, acc in ((fused, tf), (ref, tr)):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            acc.append(a.elapsed_time(b))
    return tf, tr


def back_to_back(fn, reps):
    """ms per call over reps calls enqueued back to back between two events (one synchronisation)"""
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def kernel_times(fn, reps):
    """device time per call of every br_* kernel (torch.profiler, CUDA activity), microseconds"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        if "br_" in ev.key:
            t = getattr(ev, "device_time_total", None)
            out[ev.key.split("(")[0]] = (t if t is not None else ev.cuda_time_total) / reps
    return out


def gemm_case(name, br, m, rng, reps, warmup, peak):
    dls = models(br, m, rng)
    f = br._features(None)
    dev = f["S"].device
    K, N = f["K"], br.n
    # model features once, outside the timed window (they are O(M K))
    W = torch.empty((K, m), dtype=torch.float64, device=dev)
    e = torch.empty(m, dtype=torch.float64, device=dev)
    L = _lib.lib()
    x = {k: torch.as_tensor(v, device=dev) for k, v in dls.items()}
    r0, first = 0, True
    scratch = torch.empty(max(max(br.nbins.values()) * m, int(L.gs_br_logmeanexp_scratch(N, m))), dtype=torch.float64, device=dev)
    for (kind, keys), (b0, b1), nr, ed in zip(br.groups, f["sel"], f["rows"], f["edges"]):
        cols = [x[k][:, b0:b1].contiguous() for k in keys] + [None] * (3 - len(keys))
        _lib.check(L.gs_br_model_features(kind, ptr(cols[0]), ptr(cols[1]), ptr(cols[2]), m, br.ncl, ptr(ed), b1 - b0, ptr(W[r0]), ptr(e),
                                          0 if first else 1, ptr(scratch), stream()))
        r0 += nr
        first = False
    logl = torch.empty(m, dtype=torch.float64, device=dev)
    neff = torch.empty(m, dtype=torch.float64, device=dev)
    S, c = f["S"], f["c"]

    def fused():
        _lib.check(L.gs_br_logmeanexp(ptr(S), ptr(c), N, ptr(W), ptr(e), m, K, ptr(scratch), ptr(logl), ptr(neff), stream()))

    out_ref = {}

    def ref():
        out_ref["v"] = torch.logsumexp(c[:, None] + S.T @ W + e[None, :], 0) - np.log(N)

    for _ in range(warmup):
        fused()
        ref()
    torch.cuda.synchronize()
    diff = float((logl - out_ref["v"]).abs().max())
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    ref()
    torch.cuda.synchronize()
    ref_peak = torch.cuda.max_memory_allocated() - base
    torch.cuda.reset_peak_memory_stats()
    fused()
    torch.cuda.synchronize()
    fused_peak = torch.cuda.max_memory_allocated() - base
    tf, tr = time_pair(fused, ref, reps)
    bf, br_ = back_to_back(fused, reps), back_to_back(ref, reps)
    kern = kernel_times(fused, reps)
    fl = 2.0 * N * m * K
    mf, mr = float(np.median(tf)), float(np.median(tr))
    return {"fused_ms_back_to_back": bf, "torch_ms_back_to_back": br_, "kernel_us_per_call": kern,
            "fused_fp64_tflops_kernel": fl / (sum(v for k, v in kern.items() if "logmeanexp" in k) * 1e-6) * 1e-12, "case": name, "N": N, "M": m, "K": K, "reps": reps, "fused_ms_median": mf, "fused_ms_min": float(np.min(tf)),
            "torch_ms_median": mr, "torch_ms_min": float(np.min(tr)), "speedup_vs_torch": mr / mf,
            "fused_fp64_tflops": fl / (mf * 1e-3) * 1e-12, "fused_fraction_of_measured_fp64_peak": fl / (mf * 1e-3) * 1e-12 / peak,
            "torch_peak_extra_bytes": int(ref_peak), "fused_peak_extra_bytes": int(fused_peak),
            "max_abs_diff_fused_vs_torch": diff, "median_n_eff": float(neff.median())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "br_timing_r05.jsonl"))
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--cases", default="ABCD")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("br_timing.py measures on the GPU: no CUDA device")
    torch.cuda.set_device(0)
    rng = np.random.default_rng(2025)
    peak = C.c_double(0.0)
    _lib.check(_lib.lib().gs_measure_fp64_peak(C.byref(peak), stream()))
    name, q = gpu_info()
    head = {"gpu": name, "power_limit_and_max_sm_clock": q, "measured_fp64_peak_tflops": peak.value}
    lines = []
    if "A" in a.cases or "B" in a.cases:
        br = BlackwellRao(draw_sigma(65536, 31, rng), None)
        if "A" in a.cases:
            lines.append(gemm_case("A_grid_scan_joint_l2-31", br, 8192, rng, a.reps, a.warmup, peak.value))
        if "B" in a.cases:
            lines.append(gemm_case("B_one_mcmc_call_joint_l2-31", br, 1, rng, a.reps, a.warmup, peak.value))
        del br
    if "C" in a.cases:
        lmax = 1024
        tt = np.concatenate([np.arange(0, 31), np.arange(31, lmax + 1, 10)[1:], [lmax + 1]])
        bins = {"TT": np.unique(tt), "BB": bench.bins_for(lmax)["BB"]}
        br = BlackwellRao(draw_sigma(16384, lmax, rng), bins)
        lines.append(gemm_case("C_planck_like_joint", br, 4096, rng, a.reps, a.warmup, peak.value))
        del br
    if "D" in a.cases:
        lmax = 1024
        br = BlackwellRao(draw_sigma(65536, lmax, rng, keys=("EE",)), None)
        grid = torch.linspace(0.5, 1.5, 256, dtype=torch.float64, device="cuda")
        for _ in range(a.warmup):
            br.marginal("EE", grid)
        ts = []
        for _ in range(a.reps):
            s, t = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            out = br.marginal("EE", grid)
            t.record()
            t.synchronize()
            ts.append(s.elapsed_time(t))
        lines.append({"case": "D_marginals_EE_per_l_to_1024", "N": br.n, "bins": lmax - 1, "G": 256, "reps": a.reps,
                      "marginal_ms_median": float(np.median(ts)), "marginal_ms_min": float(np.min(ts)),
                      "finite": bool(torch.isfinite(out[2:]).all())})
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        for ln in lines:
            ln = dict(head, **ln)
            fh.write(json.dumps(ln) + "\n")
            print(json.dumps(ln))


if __name__ == "__main__":
    main()
