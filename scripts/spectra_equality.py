"""Seeded outputs of every entry point that uses the per-l spectrum helpers (csrc/spectra.cuh), for bit-for-bit comparison of two
builds.

    python scripts/spectra_equality.py OUT_DIR [--nside 64,512]     # writes OUT_DIR/nside<N>/*.npy and results.json
    python scripts/spectra_equality.py --compare DIR_A DIR_B         # exit status 1 unless every file is byte-identical

GIBBS_B200_LIB selects the library, so the same script runs against two builds.  Per NSIDE (lmax = 2 NSIDE): gs_alm2cl in both
layouts and gs_alm2cl_cross; gs_expand_per_l modes 0-4, gs_unfold_bins, gs_expand_var_cl_3x3; gs_cls_invgamma with Philox and
with injected variates, with alpha_out / beta_out; gs_cls_invwishart and gs_cls_invwishart_binned (also on a broken binning);
gs_gibbs_run_centered_fullsky with and without the graph; gs_cr_direct modes 0 / 1, gs_cr_direct_pix, gs_aux_s_update,
gs_pncp_factor, gs_mala_sigma, gs_ula_nomask; gs_cr_apply_q_teb, gs_cr_rhs_teb and gs_cr_pcg_teb stopped at iter_max on a
masked sky; gs_br_sample_features / gs_br_model_features for both kinds."""
import argparse
import ctypes as C
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
import bench  # noqa: E402
from cr_host_equality import compare  # noqa: E402
from gibbssampler_b200 import _dev, _lib  # noqa: E402
from gibbssampler_b200._lib import GS_ALM_COMPLEX, GS_ALM_REAL  # noqa: E402
from gibbssampler_b200.sht import Plan  # noqa: E402

ITERMAX = 12   # well short of convergence at eps = 1e-12: the solve stops at iter_max
GS_BR_IG, GS_BR_IW = 0, 1


def run(nside, out):
    os.makedirs(out, exist_ok=True)
    L = _lib.lib()
    lmax = 2 * nside
    npix, nre, ncl = 12 * nside ** 2, (lmax + 1) ** 2, lmax + 1
    nalm = (lmax + 1) * (lmax + 2) // 2
    ptr, st = _dev.ptr, _dev.stream()
    g = np.random.default_rng(1000 + nside)
    fidE, fidB = bench.fiducial(lmax)
    fidT = 8.0 * fidE
    fidTE = 0.4 * np.sqrt(fidT * fidE)
    dlT, dlTE, dlE, dlB = (_dev.f64(v) for v in (fidT, fidTE, fidE, fidB))
    bl = _dev.f64(_dev.gauss_beam(np.radians(60.0 / nside), lmax))
    res, arrays = {}, {}

    def vec(n, scale=1.0):
        return _dev.f64(scale * g.standard_normal(n))

    def zeros(n):
        return torch.zeros(n, dtype=torch.float64, device="cuda")

    def record(name, rc, **a):
        torch.cuda.synchronize()
        res[name] = {"rc": int(rc)}
        if rc:
            res[name]["error"] = L.gs_last_error_string().decode()
        for k, v in a.items():
            arrays["%s_%s" % (name, k)] = v

    # ---- alm2cl
    xr, yr, xc = vec(nre), vec(nre), vec(2 * nalm)
    cl = zeros(ncl)
    record("alm2cl_real", L.gs_alm2cl(ptr(xr), GS_ALM_REAL, lmax, ptr(cl), st), cl=cl)
    cl = zeros(ncl)
    record("alm2cl_complex", L.gs_alm2cl(ptr(xc), GS_ALM_COMPLEX, lmax, ptr(cl), st), cl=cl)
    cl = zeros(ncl)
    record("alm2cl_cross", L.gs_alm2cl_cross(ptr(xr), ptr(yr), lmax, ptr(cl), st), cl=cl)

    # ---- per-l expansions (a zero and a negative entry exercise the safe reciprocal and the NaN of sqrt)
    x = fidE.copy()
    x[5], x[7] = 0.0, -1.0
    xd = _dev.f64(x)
    for mode in range(5):
        o = zeros(nre)
        record("expand_per_l_%d" % mode, L.gs_expand_per_l(ptr(xd), lmax, mode, ptr(o), st), out=o)
    edges = np.concatenate([[0, 1, 2], np.arange(3, lmax + 1, 7), [lmax + 1]]).astype(np.int32)
    edges = np.unique(edges)
    bins = _dev.i32(edges)
    nb = len(edges) - 1
    binned = vec(nb)
    o = zeros(lmax + 1)
    record("unfold_bins", L.gs_unfold_bins(ptr(binned), ptr(bins), nb, ptr(o), lmax + 1, st), out=o)
    dls9 = vec(9 * ncl)
    o = zeros(9 * nre)
    record("expand_var_cl_3x3", L.gs_expand_var_cl_3x3(ptr(dls9), lmax, ptr(o), st), out=o)

    # ---- inverse-gamma / inverse-Wishart C_l steps
    clhat = _dev.f64(np.abs(g.standard_normal(ncl)) * fidE * 2 * np.pi / np.maximum(np.arange(ncl) * (np.arange(ncl) + 1), 1))
    for inj in (False, True):
        o, a, b = zeros(nb), zeros(nb), zeros(nb)
        gi = _dev.f64(g.gamma(3.0, size=nb)) if inj else None
        rc = L.gs_cls_invgamma(ptr(clhat), ptr(bins), nb, ptr(gi), 1234 + nside, 7, ptr(o), ptr(a), ptr(b), st)
        record("cls_invgamma_%s" % ("inject" if inj else "philox"), rc, dl=o, alpha=a, beta=b)
    o = zeros(nb)
    record("cls_invgamma_noout", L.gs_cls_invgamma(ptr(clhat), ptr(bins), nb, None, 99, 3, ptr(o), None, None, st), dl=o)
    ctt, cte, cee = (_dev.f64(np.abs(v) * 1e-3) for v in (fidT, fidTE, fidE))
    cte = cte * 0.5
    ott, ote, oee = zeros(ncl), zeros(ncl), zeros(ncl)
    rc = L.gs_cls_invwishart(ptr(ctt), ptr(cte), ptr(cee), lmax, None, 55, 2, ptr(ott), ptr(ote), ptr(oee), st)
    record("cls_invwishart", rc, tt=ott, te=ote, ee=oee)
    for tag, e in (("good", edges), ("broken", np.concatenate([edges[:4], [edges[5], edges[4]], edges[6:]]).astype(np.int32))):
        ott, ote, oee = zeros(nb), zeros(nb), zeros(nb)
        rc = L.gs_cls_invwishart_binned(ptr(ctt), ptr(cte), ptr(cee), lmax, ptr(_dev.i32(e)), nb, None, 56, 4, ptr(ott), ptr(ote),
                                        ptr(oee), st)
        record("cls_invwishart_binned_" + tag, rc, tt=ott, te=ote, ee=oee)

    # ---- the fused centred chain
    noise = 0.01
    dEa, dBa = vec(nre, 0.1), vec(nre, 0.01)
    binsE = _dev.i32(edges)
    n_iter = 20
    for use_graph in (0, 1):
        hE, hB = zeros((n_iter + 1) * nb), zeros((n_iter + 1) * nb)
        lE, lB = zeros(nre), zeros(nre)
        initE = _dev.f64(np.concatenate([[0, 0], np.full(nb - 2, 0.5)]))
        initB = _dev.f64(np.concatenate([[0, 0], np.full(nb - 2, 0.05)]))
        rc = L.gs_gibbs_run_centered_fullsky(lmax, npix, noise, ptr(bl), ptr(dEa), ptr(dBa), ptr(binsE), nb, ptr(binsE), nb, ptr(initE),
                                             ptr(initB), n_iter, 777 + nside, ptr(hE), ptr(hB), ptr(lE), ptr(lB), use_graph, st)
        record("gibbs_run_graph%d" % use_graph, rc, histE=hE, histB=hB, lastE=lE, lastB=lB)

    # ---- diagonal full-sky draws
    w = npix / (noise * 4 * np.pi)
    d_alm, xi, bsum, badj = vec(nre, 0.1), vec(nre), vec(nre), vec(nre)
    for mode in (0, 1):
        o = zeros(nre)
        record("cr_direct_%d" % mode, L.gs_cr_direct(ptr(dlE), ptr(bl), ptr(d_alm), ptr(xi), w, lmax, mode, ptr(o), st), out=o)
    for l_cut, zl in ((lmax + 1, 0), (0, 0), (lmax // 3, 1)):
        o = zeros(nre)
        rc = L.gs_cr_direct_pix(ptr(dlE), ptr(bl), ptr(bsum), ptr(xi), w, lmax, l_cut, zl, ptr(o), st)
        record("cr_direct_pix_%d_%d" % (l_cut, zl), rc, out=o)
    for alpha in (0.0, 0.7):
        s = vec(nre)
        record("aux_s_update_%g" % alpha, L.gs_aux_s_update(ptr(badj), ptr(dlE), ptr(bl), ptr(xi), 3.5, alpha, lmax, ptr(s), st), s=s)
    for mode in (0, 1):
        o = zeros(ncl)
        record("pncp_factor_%d" % mode, L.gs_pncp_factor(ptr(xd), lmax, lmax // 4, mode, ptr(o), st), out=o)
    o = zeros(nre)
    record("mala_sigma", L.gs_mala_sigma(ptr(dlE), ptr(bl), w, lmax, ptr(o), st), out=o)
    s_old, s_new, scratch, lr = vec(nre, 0.1), zeros(nre), zeros(592), zeros(1)
    rc = L.gs_ula_nomask(ptr(dlE), ptr(bl), ptr(d_alm), ptr(s_old), ptr(xi), w, 0.02, lmax, ptr(s_new), ptr(scratch), ptr(lr), st)
    record("ula_nomask", rc, s_new=s_new, log_ratio=lr)

    # ---- joint T/E/B on a cut sky
    plan = Plan.get(nside, lmax)
    h = plan._h
    mask = bench.make_mask(nside, kind="galplane")
    invnT, invnP = _dev.f64(mask * 4.0), _dev.f64(mask * 25.0)
    sinvnT, sinvnP = torch.sqrt(invnT), torch.sqrt(invnP)
    nT, nP = float(invnT.sum().item()) / (4 * np.pi), float(invnP.sum().item()) / (4 * np.pi)
    teb = (ptr(dlT), ptr(dlTE), ptr(dlE), ptr(dlB), ptr(bl))
    xT, xE, xB = vec(nre), vec(nre), vec(nre)
    yT, yE, yB = zeros(nre), zeros(nre), zeros(nre)
    rc = L.gs_cr_apply_q_teb(h, *teb, ptr(invnT), ptr(invnP), ptr(xT), ptr(xE), ptr(xB), ptr(yT), ptr(yE), ptr(yB), st)
    record("apply_q_teb", rc, yT=yT, yE=yE, yB=yB)
    dI, dQ, dU = (vec(npix) * _dev.f64(mask) for _ in range(3))
    xiI, xiQ, xiU = vec(npix), vec(npix), vec(npix)
    xiT, xiE, xiB = vec(nre), vec(nre), vec(nre)
    rT, rE, rB = zeros(nre), zeros(nre), zeros(nre)
    rc = L.gs_cr_rhs_teb(h, *teb, ptr(invnT), ptr(sinvnT), ptr(invnP), ptr(sinvnP), None, None, None, ptr(dI), ptr(dQ), ptr(dU),
                         ptr(xiI), ptr(xiQ), ptr(xiU), ptr(xiT), ptr(xiE), ptr(xiB), 3, ptr(rT), ptr(rE), ptr(rB), st)
    record("rhs_teb", rc, rT=rT, rE=rE, rB=rB)
    sT, sE, sB = zeros(nre), zeros(nre), zeros(nre)
    nit, rr = C.c_int(0), C.c_double(0.0)
    rc = L.gs_cr_pcg_teb(h, *teb, ptr(invnT), ptr(invnP), nT, nP, ptr(rT), ptr(rE), ptr(rB), ptr(sT), ptr(sE), ptr(sB), 0, 1e-12,
                         ITERMAX, 8, C.byref(nit), C.byref(rr), st)
    record("pcg_teb", rc, xT=sT, xE=sE, xB=sB)
    res["pcg_teb"].update(iters=nit.value, resid=rr.value.hex())

    # ---- Blackwell-Rao features (bins 2.. of the chain's binning; one broken bin at the end)
    nsamp, nmod = 300, 40
    be = edges[2:].copy()
    be_bad = np.concatenate([be, [be[-1] + 5]]).astype(np.int32)   # last bin runs past ncl: NaN
    nbb = len(be_bad) - 1
    bins_br = _dev.i32(be_bad)
    sig = [_dev.f64(np.abs(g.standard_normal((nsamp, ncl))) * 1e-3 + 1e-4) for _ in range(3)]
    sig[1] = sig[1] * 0.1
    mods = [_dev.f64(np.abs(g.standard_normal((nmod, nbb))) + 0.1) for _ in range(3)]
    mods[1] = mods[1] * 0.1
    for kind, tag, f in ((GS_BR_IG, "ig", 1), (GS_BR_IW, "iw", 3)):
        S, c, scr = zeros(f * nbb * nsamp), zeros(nsamp), zeros(nbb * nsamp)
        rc = L.gs_br_sample_features(kind, ptr(sig[0]), ptr(sig[1]), ptr(sig[2]), nsamp, ncl, ptr(bins_br), nbb, ptr(S), ptr(c), 0,
                                     ptr(scr), st)
        record("br_sample_features_" + tag, rc, S=S, c=c)
        W, e, scr = zeros(f * nbb * nmod), zeros(nmod), zeros(nbb * nmod)
        rc = L.gs_br_model_features(kind, ptr(mods[0]), ptr(mods[1]), ptr(mods[2]), nmod, ncl, ptr(bins_br), nbb, ptr(W), ptr(e), 0,
                                    ptr(scr), st)
        record("br_model_features_" + tag, rc, W=W, e=e)

    for k, v in arrays.items():
        np.save(os.path.join(out, k + ".npy"), v.cpu().numpy())
    with open(os.path.join(out, "results.json"), "w") as f:
        json.dump(res, f, indent=1, sort_keys=True)
    # pcg_teb returns GS_E_NOTCONVERGED: it is stopped at iter_max on purpose
    print(json.dumps({"nside": nside, "calls": len(res), "nonzero_rc": sorted(k for k, v in res.items() if v["rc"])}), flush=True)


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
