"""Drop-in for the array helpers of the reference's utils.py / variance_expension.pyx, executed by
the sm_100a kernels of almops.cu.  Inputs may be numpy arrays (results come back as numpy) or CUDA
tensors (results stay in HBM).  lmax is inferred from the array length like the Cython versions do
(variance_expension.pyx:70,89) instead of from the global config.L_MAX_SCALARS (utils.py:57,71)."""
import numpy as np
import torch

from . import _dev, _lib
from ._dev import f64, ptr, stream
from ._lib import check, GS_ALM_COMPLEX, GS_ALM_REAL
from .sht import Plan


def _ret(t, like):
    return t if isinstance(like, torch.Tensor) else t.cpu().numpy()


def real_to_complex(alms):
    """utils.real_to_complex (utils.py:49-60)."""
    r = f64(alms)
    lmax = _dev.lmax_from_real(r.numel())
    c = torch.empty((lmax + 1) * (lmax + 2) // 2, dtype=torch.complex128, device=r.device)
    check(_lib.lib().gs_real_to_complex(ptr(r), ptr(c), lmax, stream()))
    return _ret(c, alms)


def complex_to_real(alms):
    """utils.complex_to_real (utils.py:63-76)."""
    c = alms if isinstance(alms, torch.Tensor) else torch.as_tensor(np.ascontiguousarray(alms, dtype=np.complex128))
    c = c.to(device=_dev.device(), dtype=torch.complex128).contiguous()
    lmax = _dev.lmax_from_complex(c.numel())
    r = torch.empty((lmax + 1) ** 2, dtype=torch.float64, device=c.device)
    check(_lib.lib().gs_complex_to_real(ptr(c), ptr(r), lmax, stream()))
    return _ret(r, alms)


def expand_per_l(x, mode=0):
    x_ = f64(x)
    lmax = x_.numel() - 1
    out = torch.empty((lmax + 1) ** 2, dtype=torch.float64, device=x_.device)
    check(_lib.lib().gs_expand_per_l(ptr(x_), lmax, int(mode), ptr(out), stream()))
    return _ret(out, x)


def generate_var_cl(cls_):
    """utils.generate_var_cl (utils.py:139-147): takes D_l (despite the name), returns the diagonal of
    C in the real alm layout."""
    return expand_per_l(cls_, 1)


def dls_to_cls_array(lmax):
    """Per-l factor that turns D_l into C_l: 2 pi / (l (l+1)), and 0 at l = 0."""
    return np.array([2 * np.pi / (l * (l + 1)) if l != 0 else 0 for l in range(lmax + 1)])


def unfold_bins(binned_cls_, bins):
    """utils.unfold_bins (utils.py:150-162): np.repeat(binned, diff(bins))."""
    b = f64(binned_cls_)
    edges = np.asarray(_dev.to_host(bins), dtype=np.int64)
    nbins = len(edges) - 1
    assert b.numel() == nbins, "need one value per bin"
    nout = int(edges[-1] - edges[0])
    out = torch.empty(nout, dtype=torch.float64, device=b.device)
    check(_lib.lib().gs_unfold_bins(ptr(b), ptr(_dev.i32(edges)), nbins, ptr(out), nout, stream()))
    return _ret(out, binned_cls_)


def remove_monopole_dipole_contributions(alms):
    """variance_expension.remove_monopole_dipole_contributions (variance_expension.pyx:103-111): zeroes the real-layout
    entries 0, 1, L+1, L+2 IN PLACE and returns the array, like the Cython function does with its memoryview."""
    if isinstance(alms, torch.Tensor) and alms.is_cuda:
        lmax = _dev.lmax_from_real(alms.numel())
        assert alms.dtype == torch.float64 and alms.is_contiguous()
        check(_lib.lib().gs_remove_monopole_dipole(ptr(alms), lmax, stream()))
        return alms
    a = np.asarray(alms)
    lmax = _dev.lmax_from_real(a.size)
    a[[0, 1, lmax + 1, lmax + 2]] = 0.0
    return alms


def synthesis_hp(alms, nside):
    """variance_expension.synthesis_hp (variance_expension.pyx:114-123): real-layout alm -> map."""
    a = f64(alms)
    plan = Plan.get(nside, _dev.lmax_from_real(a.numel()))
    return _ret(plan.alm2map(a), alms)


def adjoint_synthesis_hp(map, bl_map=None, nside=None, lmax=None, iter=3):
    """utils.adjoint_synthesis_hp (utils.py:79-111): (Npix/4pi) * complex_to_real(map2alm(iter=3)) [* bl_map].
    `map` is one map or a list [I, Q, U]; lmax defaults to 2 nside as in config.py:21."""
    pol = isinstance(map, (list, tuple)) and len(map) == 3
    first = map[1] if pol else map
    npix = int(first.shape[0]) if hasattr(first, "shape") else len(first)
    nside = nside or int(round((npix / 12) ** 0.5))
    if lmax is None:
        lmax = _dev.lmax_from_real(len(bl_map)) if bl_map is not None else 2 * nside
    plan = Plan.get(nside, lmax)
    resc = npix / (4 * np.pi)
    blm = f64(bl_map) if bl_map is not None else None
    if pol:
        t = plan.map2alm(f64(map[0]), iter=iter, real_layout=True) * resc
        e, b = plan.map2alm_spin2(f64(map[1]), f64(map[2]), iter=iter, real_layout=True)
        outs = [t, e * resc, b * resc]
        if blm is not None:
            outs = [o * blm for o in outs]
        return tuple(_ret(o, first) for o in outs)
    a = plan.map2alm(f64(map), iter=iter, real_layout=True) * resc
    if blm is not None:
        a = a * blm
    return _ret(a, map)
