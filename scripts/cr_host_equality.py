"""Seeded outputs of the constrained-realization host entry points on a masked sky, for bit-for-bit comparison of two builds.

    python scripts/cr_host_equality.py OUT_DIR [--nside 64,512]     # writes OUT_DIR/nside<N>/*.npy and results.json
    python scripts/cr_host_equality.py --compare DIR_A DIR_B         # exit status 1 unless every file is byte-identical

GIBBS_B200_LIB selects the library, so the same script runs against two builds.  Per NSIDE (lmax = 2 NSIDE): gs_cr_apply_q_tt /
_pol, gs_cr_rhs_tt / _pol with the data term passed in and computed from the maps, and gs_cr_pcg_tt / _pol / _pol_batch (two
chains) stopped at iter_max, with their return codes, iteration counts, residuals and error messages."""
import argparse
import ctypes as C
import filecmp
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from gibbssampler_b200 import _dev, _lib  # noqa: E402
from gibbssampler_b200.sht import Plan  # noqa: E402

ITERMAX = 12   # well short of convergence at eps = 1e-12: every solve stops at iter_max


def run(nside, out):
    os.makedirs(out, exist_ok=True)
    L = _lib.lib()
    lmax = 2 * nside
    npix, nre = 12 * nside ** 2, (lmax + 1) ** 2
    plan = Plan.get(nside, lmax)
    h, ptr, st = plan._h, _dev.ptr, _dev.stream()
    g = np.random.default_rng(nside)
    fidE, fidB = bench.fiducial(lmax)
    dlE, dlB = _dev.f64(fidE), _dev.f64(fidB)
    dlE2, dlB2 = _dev.f64(np.stack([fidE, 0.8 * fidE])), _dev.f64(np.stack([fidB, 1.5 * fidB]))   # [chain][l]
    bl = _dev.f64(_dev.gauss_beam(np.radians(60.0 / nside), lmax))
    # cut, constant-weight and empty rings: every ring class of the mat-vec
    mask = bench.make_mask(nside, kind="galplane")
    invn = _dev.f64(mask * 25.0)
    sinvn = torch.sqrt(invn)
    ninv = float(invn.sum().item()) / (4 * np.pi)

    def vec(n):
        return _dev.f64(g.standard_normal(n))

    x, xE, xB = vec(nre), vec(nre), vec(nre)
    dI, dQ, dU = vec(npix) * _dev.f64(mask), vec(npix) * _dev.f64(mask), vec(npix) * _dev.f64(mask)
    xiI, xiQ, xiU = vec(npix), vec(npix), vec(npix)
    xiT, xiE, xiB = vec(nre), vec(nre), vec(nre)
    bdT, bdE, bdB = vec(nre), vec(nre), vec(nre)
    res = {}
    arrays = {}

    def empty():
        return torch.empty(nre, dtype=torch.float64, device="cuda")

    def record(name, rc, **a):
        torch.cuda.synchronize()
        res[name] = {"rc": int(rc)}
        if rc:
            res[name]["error"] = L.gs_last_error_string().decode()
        for k, v in a.items():
            arrays["%s_%s" % (name, k)] = v

    y = empty()
    record("apply_q_tt", L.gs_cr_apply_q_tt(h, ptr(dlE), ptr(bl), ptr(invn), ptr(x), ptr(y), st), y=y)
    yE, yB = empty(), empty()
    record("apply_q_pol", L.gs_cr_apply_q_pol(h, ptr(dlE), ptr(dlB), ptr(bl), ptr(invn), ptr(xE), ptr(xB), ptr(yE), ptr(yB), st), yE=yE, yB=yB)
    for with_bdata in (True, False):
        tag = "bdata" if with_bdata else "maps"
        r = empty()
        rc = L.gs_cr_rhs_tt(h, ptr(dlE), ptr(bl), ptr(invn), ptr(sinvn), ptr(bdT) if with_bdata else None, None if with_bdata else ptr(dI),
                            ptr(xiT), ptr(xiI), 3, ptr(r), st)
        record("rhs_tt_" + tag, rc, rhs=r)
        rE, rB = empty(), empty()
        bd = (ptr(bdE), ptr(bdB), None, None) if with_bdata else (None, None, ptr(dQ), ptr(dU))
        rc = L.gs_cr_rhs_pol(h, ptr(dlE), ptr(dlB), ptr(bl), ptr(invn), ptr(sinvn), *bd, ptr(xiQ), ptr(xiU), ptr(xiE), ptr(xiB), 3,
                             ptr(rE), ptr(rB), st)
        record("rhs_pol_" + tag, rc, rhsE=rE, rhsB=rB)

    nit, rr = C.c_int(0), C.c_double(0.0)
    s = empty()
    rc = L.gs_cr_pcg_tt(h, ptr(dlE), ptr(bl), ptr(invn), ninv, ptr(bdT), ptr(s), 0, 1e-12, ITERMAX, 8, C.byref(nit), C.byref(rr), st)
    record("pcg_tt", rc, x=s)
    res["pcg_tt"].update(iters=nit.value, resid=rr.value.hex())
    sE, sB = empty(), empty()
    rc = L.gs_cr_pcg_pol(h, ptr(dlE), ptr(dlB), ptr(bl), ptr(invn), ninv, ptr(bdE), ptr(bdB), ptr(sE), ptr(sB), 0, 1e-12, ITERMAX, 8,
                         C.byref(nit), C.byref(rr), st)
    record("pcg_pol", rc, xE=sE, xB=sB)
    res["pcg_pol"].update(iters=nit.value, resid=rr.value.hex())
    rhs2 = torch.stack([torch.stack([bdE, bdB]), torch.stack([bdB, bdE])])   # [chain][E, B][nre]
    x2 = torch.empty_like(rhs2)
    nit2, rr2 = (C.c_int * 2)(), (C.c_double * 2)()
    rc = L.gs_cr_pcg_pol_batch(h, 2, ptr(dlE2), ptr(dlB2), ptr(bl), ptr(invn), ninv, ptr(rhs2[0, 0]), ptr(rhs2[0, 1]), ptr(x2[0, 0]),
                               ptr(x2[0, 1]), 2 * nre, 1e-12, ITERMAX, 8, nit2, rr2, st)
    record("pcg_pol_batch", rc, x=x2)
    res["pcg_pol_batch"].update(iters=list(nit2), resid=[v.hex() for v in rr2])

    for k, v in arrays.items():
        np.save(os.path.join(out, k + ".npy"), v.cpu().numpy())
    with open(os.path.join(out, "results.json"), "w") as f:
        json.dump(res, f, indent=1, sort_keys=True)
    print(json.dumps({"nside": nside, **{k: (v["rc"], v.get("iters")) for k, v in res.items()}}), flush=True)


def compare(a, b):
    bad, n = [], 0
    for dirpath, _, files in os.walk(a):
        for fn in files:
            pa = os.path.join(dirpath, fn)
            pb = os.path.join(b, os.path.relpath(pa, a))
            n += 1
            if not os.path.exists(pb) or not filecmp.cmp(pa, pb, shallow=False):
                bad.append(os.path.relpath(pa, a))
    for dirpath, _, files in os.walk(b):
        for fn in files:
            if not os.path.exists(os.path.join(a, os.path.relpath(os.path.join(dirpath, fn), b))):
                bad.append(os.path.relpath(os.path.join(dirpath, fn), b))
    print(json.dumps({"files": n, "differ": sorted(set(bad))}))
    return 1 if bad or n == 0 else 0


if __name__ == "__main__":
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("out", nargs="?")
    ap.add_argument("--nside", default="64,512")
    ap.add_argument("--compare", nargs=2, metavar=("DIR_A", "DIR_B"))
    args = ap.parse_args()
    if args.compare:
        sys.exit(compare(*args.compare))
    if not args.out:
        ap.error("OUT_DIR is required")
    for ns in (int(v) for v in args.nside.split(",")):
        run(ns, os.path.join(args.out, "nside%d" % ns))
