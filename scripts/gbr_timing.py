"""Gaussianized Blackwell-Rao timing on one GPU: the fused mixture-CDF transform (gs_gbr_transform) against the torch composition
(gammaincc / gammainc over an N x M x B tensor, ndtri, logsumexp) where that fits in memory, and BR's median n_eff at the same
models.  sigma is synthetic, drawn as in scripts/br_timing.py.  Cases:
(A) construction: N = 65536 samples, per-l TT, l = 2..29, 65536 models standing in for the chain's D rows (N x N x B evaluations);
(B) one parameter-MCMC call, M = 1, the same bins;
(C) M = 8192 models, joint TT/EE/BB (TE marginalised), l = 2..31, N = 65536;
(D) wide alpha: the Planck-like bins of scripts/teb_timing.py --bins planck (TT one l to 30, width 10 above to 1024; BB edges
    of bench.bins_for(1024)), N = 16384, M = 1024.
Writes one JSON line per case to --out, with the GPU name, power limit and max SM clock read in the same run."""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import bench  # noqa: E402
from br_timing import back_to_back, draw_sigma, gpu_info, models  # noqa: E402
from gibbssampler_b200.BlackwellRao import BlackwellRao  # noqa: E402


def kernel_times(fn, reps):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        if "gbr_" in ev.key:
            t = getattr(ev, "device_time_total", None)
            out[ev.key.split("(")[0]] = (t if t is not None else ev.cuda_time_total) / reps
    return out


def torch_transform(br, key, d):
    """the torch composition of one key: x (M, nb), logm (M, nb) from an N x M x nb tensor"""
    gi, kind, comp = br._group_of(key)
    f = br._features(None)
    r0 = sum(f["rows"][:gi])
    e = br.edges[key]
    nb = br.nbins[key] - 2
    ell = [(e[b], e[b + 1]) for b in range(2, nb + 2)]
    if kind == 0:
        alpha = torch.tensor([sum((2 * l + 1) / 2 for l in range(a, b)) - 1 for a, b in ell], dtype=torch.float64, device="cuda")
        beta = f["S"][r0:r0 + nb]
    else:
        alpha = torch.tensor([(sum(2 * l + 1 for l in range(a, b)) - 4) / 2 for a, b in ell], dtype=torch.float64, device="cuda")
        beta = 0.5 * f["S"][r0 + comp:r0 + 3 * nb:3]
    t = beta.T[:, None, :] / d[None, :, :]                  # (N, M, nb)
    a = alpha[None, None, :].expand_as(t)
    N = t.shape[0]
    F = torch.special.gammaincc(a, t).sum(0) / N
    G = torch.special.gammainc(a, t).sum(0) / N
    x = torch.where(F <= 0.5, torch.special.ndtri(F), -torch.special.ndtri(G))
    lp = alpha * torch.log(t) - t - torch.lgamma(alpha) - torch.log(d)[None]
    return x, torch.logsumexp(lp, 0) - np.log(N)


def case(name, br, dls, keys, reps, warmup, torch_ok):
    d = {k: torch.as_tensor(np.asarray(dls[k])[:, 2:], device="cuda").contiguous() for k in keys}
    M = next(iter(d.values())).shape[0]

    def fused():
        return [br._transform(k, d[k]) for k in keys]
    for _ in range(warmup):
        fused()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fused()
    torch.cuda.synchronize()
    first = time.perf_counter() - t0
    ms = back_to_back(fused, reps) if first < 2.0 else first * 1e3
    kern = kernel_times(fused, reps if first < 2.0 else 1)
    evals = br.n * M * sum(br.nbins[k] - 2 for k in keys)
    line = {"case": name, "N": br.n, "M": M, "bins": {k: br.nbins[k] - 2 for k in keys}, "reps": reps,
            "fused_ms_back_to_back": ms, "kernel_us_per_call": kern, "incomplete_gamma_evals": evals,
            "incomplete_gamma_evals_per_s_kernel": evals / (sum(kern.values()) * 1e-6) if kern else None}
    if torch_ok:
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        ref = [torch_transform(br, k, d[k]) for k in keys]
        torch.cuda.synchronize()
        line["torch_peak_extra_bytes"] = int(torch.cuda.max_memory_allocated() - base)
        line["torch_ms_back_to_back"] = back_to_back(lambda: [torch_transform(br, k, d[k]) for k in keys], max(1, reps // 4))
        fin = [torch.isfinite(r[0]) & torch.isfinite(o[0]) for r, o in zip(ref, out)]
        line["max_abs_diff_x_vs_torch"] = max(float((r[0] - o[0])[f].abs().max()) for r, o, f in zip(ref, out, fin))
        line["max_abs_diff_logm_vs_torch"] = max(float((r[1] - o[1])[f].abs().max()) for r, o, f in zip(ref, out, fin))
    else:
        line["torch"] = "not run: the N x M x B tensor does not fit"
    if M <= 8192:
        full = {k: np.asarray(dls[k]) for k in br.keys if k in dls}
        if br.joint:
            full["TE"] = np.asarray(dls["TE"])
        _, neff = br.logpdf(full, n_eff=True)
        line["br_median_n_eff"] = float(np.median(neff))
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "gbr_timing_r06.jsonl"))
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--cases", default="ABCD")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("gbr_timing.py measures on the GPU: no CUDA device")
    torch.cuda.set_device(0)
    rng = np.random.default_rng(2026)
    name, q = gpu_info()
    head = {"gpu": name, "power_limit_and_max_sm_clock": q}
    lines = []
    if "A" in a.cases or "B" in a.cases:
        br = BlackwellRao({"TT": 30.0 * draw_sigma(65536, 29, rng, keys=("EE",))["EE"]}, None)
        if "A" in a.cases:
            lines.append(case("A_construction_tt_l2-29", br, models(br, 65536, rng), ("TT",), 1, 0, False))
        if "B" in a.cases:
            lines.append(case("B_one_mcmc_call_tt_l2-29", br, models(br, 1, rng), ("TT",), a.reps * 10, a.warmup, True))
        del br
    if "C" in a.cases:
        br = BlackwellRao(draw_sigma(65536, 31, rng), None)
        lines.append(case("C_grid_joint_tt_ee_bb_l2-31", br, models(br, 8192, rng), ("TT", "EE", "BB"), a.reps, a.warmup, False))
        del br
    if "D" in a.cases:
        lmax = 1024
        tt = np.concatenate([np.arange(0, 31), np.arange(31, lmax + 1, 10)[1:], [lmax + 1]])
        bins = {"TT": np.unique(tt), "BB": bench.bins_for(lmax)["BB"]}
        br = BlackwellRao(draw_sigma(16384, lmax, rng), bins)
        lines.append(case("D_planck_like_wide_alpha", br, models(br, 1024, rng), ("TT", "EE", "BB"), a.reps, a.warmup, False))
        del br
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        for ln in lines:
            ln = dict(head, **ln)
            fh.write(json.dumps(ln) + "\n")
            print(json.dumps(ln), flush=True)


if __name__ == "__main__":
    main()
