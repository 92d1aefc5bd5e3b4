"""Several chains per GPU, stepped in lockstep so that their constrained realizations run as chain batches.

The reference runs one chain per process (SLURM array, job-script.sh:6); every process repeats the Legendre recurrences of
hp.alm2map / hp.map2alm inside its PCG.  Two chains on one GPU can share them: `run_chains` steps K Gibbs objects of this
package (CenteredGibbs or PNCPGibbs, polarised, masked sky, same data / mask / noise / plan, their own seeds) together and
draws their sky maps with `sample_mask_batch` (gs_cr_pcg_pol_batch: two right-hand sides per launch, 4 + 8 K instead of
12 K DFMA per ring pair and multipole); the C_l steps stay per chain.  Every chain performs exactly the PCG iterations of
its own solve and returns what its own run() would return.
"""
import time

import numpy as np
import torch

from . import _dev
from ._dev import f64
from .CenteredGibbs import sample_mask_batch


def _cls_step(g, skymap, binned):
    """The C_l part of one iteration of g.run_polarization (GibbsSampler.py:160-166 / recovered PNCPGibbs.run)."""
    if hasattr(g.cls_sampler, "sample_low_l"):          # PNCP: centred low l, non-centred Metropolis high l
        binned = g.cls_sampler.sample_low_l(skymap, binned)
        all_dls = {"EE": g._unfold(binned, "EE"), "BB": g._unfold(binned, "BB")}
        mixed = g.constrained_sampler.to_mixed(skymap, all_dls)
        binned, acc = g.cls_sampler.sample_high_l(mixed, binned)
        return binned, acc
    return g.cls_sampler.sample(dict(skymap)), None


def run_chains(gibbs, dls_init):
    """gibbs: list of 1..N CenteredGibbs / PNCPGibbs objects (polarization=True, a mask, the same data and plan);
    dls_init: one binned {"EE", "BB"} start per chain.  Chains are paired (0, 1), (2, 3), ...; an odd last chain runs alone.
    Returns one (h_dls, accept, t_cr, t_cls) tuple per chain, as the chain's own run()."""
    assert len(gibbs) == len(dls_init) and len(gibbs) >= 1
    if any(getattr(g, "keep_sigma", False) for g in gibbs):
        raise ValueError("run_chains does not record the sky spectra: run chains built with keep_sigma=True through their own run()")
    n_iter = gibbs[0].n_iter
    assert all(g.n_iter == n_iter and g.polarization for g in gibbs)
    K = len(gibbs)
    binned = [{k: f64(v) for k, v in d.items()} for d in dls_init]
    hist = [{"EE": [_dev.to_host(b["EE"])], "BB": [_dev.to_host(b["BB"])]} for b in binned]
    accept = [{"EE": [], "BB": []} for _ in range(K)]
    t_cr, t_cls = [[] for _ in range(K)], [[] for _ in range(K)]
    for _ in range(n_iter):
        t0 = time.perf_counter()
        sky = [None] * K
        for a in range(0, K, 2):
            idx = list(range(a, min(a + 2, K)))
            dls = [{"EE": gibbs[i]._unfold(binned[i], "EE"), "BB": gibbs[i]._unfold(binned[i], "BB")} for i in idx]
            for i, (s, _) in zip(idx, sample_mask_batch([gibbs[i].constrained_sampler for i in idx], dls)):
                sky[i] = s
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / K
        for i in range(K):
            t0 = time.perf_counter()
            binned[i], acc = _cls_step(gibbs[i], sky[i], binned[i])
            torch.cuda.synchronize()
            t_cr[i].append(dt)
            t_cls[i].append(time.perf_counter() - t0)
            if acc is not None:
                accept[i]["EE"].append(acc["EE"])
                accept[i]["BB"].append(acc["BB"])
            hist[i]["EE"].append(_dev.to_host(binned[i]["EE"]))
            hist[i]["BB"].append(_dev.to_host(binned[i]["BB"]))
    out = []
    for i in range(K):
        h = {k: np.array(v) for k, v in hist[i].items()}
        acc = {k: np.array(v) for k, v in accept[i].items()} if accept[i]["EE"] else np.ones(n_iter)
        out.append((h, acc, np.array(t_cr[i]), np.array(t_cls[i])))
    return out
