"""ctypes loader of libgibbs_b200.so (the C ABI declared in include/gibbs_b200.h).

There is no CPU fallback: if the CUDA library has not been built the import of any compute
entry point fails loudly.  Build it with ``python -c "import __graft_entry__ as g; g.build()"``
or ``make -C gibbssampler_b200/csrc``.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("GIBBS_B200_LIB") or os.path.join(_HERE, "csrc", "_build", "libgibbs_b200.so")

GS_ALM_COMPLEX = 0
GS_ALM_REAL = 1

_lib = None

_vp = C.c_void_p
_i = C.c_int
_d = C.c_double
_i64 = C.c_int64

# name -> (restype, argtypes); mirrors include/gibbs_b200.h one to one
SIGNATURES = {
    "gs_last_error_string": (C.c_char_p, []),
    "gs_version": (_i, []),
    "gs_plan_create": (_i, [C.POINTER(_vp), _i, _i, _i]),
    "gs_plan_destroy": (_i, [_vp]),
    "gs_plan_reserve_chains": (_i, [_vp, _i]),
    "gs_plan_nside": (_i, [_vp]),
    "gs_plan_lmax": (_i, [_vp]),
    "gs_plan_npix": (_i64, [_vp]),
    "gs_plan_nalm": (_i64, [_vp]),
    "gs_plan_nreal": (_i64, [_vp]),
    "gs_alm2map_spin0": (_i, [_vp, _vp, _i, _vp, _vp, _vp]),
    "gs_alm2map_spin2": (_i, [_vp, _vp, _vp, _i, _vp, _vp, _vp, _vp]),
    "gs_map2alm_spin0": (_i, [_vp, _vp, _vp, _i, _i, _vp, _vp, _i, _vp]),
    "gs_map2alm_spin2": (_i, [_vp, _vp, _vp, _vp, _i, _i, _vp, _vp, _vp, _i, _vp]),
    "gs_alm2map_batch": (_i, [_vp, _i, _i, _vp, _vp, _i64, _i, _vp, _vp, _vp, _i64, _vp]),
    "gs_map2alm_batch": (_i, [_vp, _i, _i, _vp, _vp, _i64, _vp, _i, _vp, _vp, _vp, _i64, _i, _vp]),
    "gs_real_to_complex": (_i, [_vp, _vp, _i, _vp]),
    "gs_complex_to_real": (_i, [_vp, _vp, _i, _vp]),
    "gs_expand_per_l": (_i, [_vp, _i, _i, _vp, _vp]),
    "gs_unfold_bins": (_i, [_vp, _vp, _i, _vp, _i, _vp]),
    "gs_almxfl": (_i, [_vp, _i, _i, _vp, _vp, _vp]),
    "gs_alm2cl": (_i, [_vp, _i, _i, _vp, _vp]),
    "gs_alm2map_spin2_fl2": (_i, [_vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp]),
    "gs_cr_rhs_pol": (_i, [_vp] * 14 + [_i, _vp, _vp, _vp]),
    "gs_cr_pcg_pol": (_i, [_vp, _vp, _vp, _vp, _vp, _d, _vp, _vp, _vp, _vp, _i, _d, _i, _i,
                           C.POINTER(_i), C.POINTER(_d), _vp]),
    "gs_cr_pcg_pol_batch": (_i, [_vp, _i, _vp, _vp, _vp, _vp, _d, _vp, _vp, _vp, _vp, _i64, _d, _i, _i,
                                 C.POINTER(_i), C.POINTER(_d), _vp]),
    "gs_set_pcg_graph": (_i, [_i]),
    "gs_cr_apply_q_pol": (_i, [_vp] * 10),
    "gs_cr_rhs_tt": (_i, [_vp] * 9 + [_i, _vp, _vp]),
    "gs_cr_pcg_tt": (_i, [_vp, _vp, _vp, _vp, _d, _vp, _vp, _i, _d, _i, _i, C.POINTER(_i), C.POINTER(_d), _vp]),
    "gs_cr_apply_q_tt": (_i, [_vp] * 7),
    "gs_cr_rhs_teb": (_i, [_vp] * 22 + [_i, _vp, _vp, _vp, _vp]),
    "gs_cr_pcg_teb": (_i, [_vp] * 8 + [_d, _d] + [_vp] * 6 + [_i, _d, _i, _i, C.POINTER(_i), C.POINTER(_d), _vp]),
    "gs_cr_apply_q_teb": (_i, [_vp] * 15),
    "gs_gibbs_run_centered_fullsky": (_i, [_i, _i64, _d, _vp, _vp, _vp, _vp, _i, _vp, _i, _vp, _vp, _i, C.c_uint64, _vp, _vp, _vp, _vp,
                                           _i, _vp]),
    "gs_cr_direct": (_i, [_vp, _vp, _vp, _vp, _d, _i, _i, _vp, _vp]),
    "gs_cr_direct_pix": (_i, [_vp, _vp, _vp, _vp, _d, _i, _i, _i, _vp, _vp]),
    "gs_cls_invgamma": (_i, [_vp, _vp, _i, _vp, C.c_uint64, C.c_uint64, _vp, _vp, _vp, _vp]),
    "gs_truncnorm_propose": (_i, [_vp, _vp, _i, _vp, _vp, _vp]),
    "gs_truncnorm_logpdf": (_i, [_vp, _vp, _vp, _i, _vp, _vp]),
    "gs_loglik_pix": (_i, [_vp, _vp, _vp, _vp, _vp, _i64, _vp, _vp, _vp]),
    "gs_loglik_alm": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _d, _vp, _vp, _vp]),
    "gs_randn": (_i, [_vp, _i64, C.c_uint64, C.c_uint64, _vp]),
    "gs_randu": (_i, [_vp, _i64, C.c_uint64, C.c_uint64, _vp]),
    "gs_sum": (_i, [_vp, _i64, _vp, _vp, _vp]),
    "gs_mwg_filters": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _vp, _i, _i, _i, _i, _vp, _i, _i, _vp, _vp, _vp]),
    "gs_mwg_accept": (_i, [_vp, _vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "gs_mwg_sweep_blocks": (_i, [_vp] * 9 + [_vp, _i, _vp, _i, _vp, _i, _vp, _i, _i, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp]),
    "gs_mul": (_i, [_vp, _vp, _vp, _i64, _vp]),
    "gs_aux_v_update": (_i, [_vp, _vp, _vp, _vp, _d, _d, _vp, _vp, _i64, _vp]),
    "gs_aux_s_update": (_i, [_vp, _vp, _vp, _vp, _d, _d, _i, _vp, _vp]),
    "gs_pncp_factor": (_i, [_vp, _i, _i, _i, _vp, _vp]),
    "gs_mala_sigma": (_i, [_vp, _vp, _d, _i, _vp, _vp]),
    "gs_mala_grad": (_i, [_vp, _vp, _vp, _vp, _vp, _i64, _vp]),
    "gs_mala_propose": (_i, [_vp, _vp, _vp, _vp, _d, _vp, _i64, _vp]),
    "gs_mala_logq": (_i, [_vp, _vp, _vp, _vp, _d, _i64, _vp, _vp, _vp]),
    "gs_dot3": (_i, [_vp, _vp, _vp, _i64, _vp, _vp, _vp]),
    "gs_ula_nomask": (_i, [_vp, _vp, _vp, _vp, _vp, _d, _d, _i, _vp, _vp, _vp, _vp]),
    "gs_remove_monopole_dipole": (_i, [_vp, _i, _vp]),
    "gs_expand_var_cl_3x3": (_i, [_vp, _i, _vp, _vp]),
    "gs_inv_chol_3x3": (_i, [_vp, _vp, _i, _vp, _vp, _vp]),
    "gs_matvec_3x3": (_i, [_vp, _vp, _vp, _i, _vp, _vp]),
    "gs_alm2cl_cross": (_i, [_vp, _vp, _i, _vp, _vp]),
    "gs_cls_invwishart": (_i, [_vp, _vp, _vp, _i, _vp, C.c_uint64, C.c_uint64, _vp, _vp, _vp, _vp]),
    "gs_cls_invwishart_binned": (_i, [_vp, _vp, _vp, _i, _vp, _i, _vp, C.c_uint64, C.c_uint64, _vp, _vp, _vp, _vp]),
    "gs_nccl_unique_id": (_i, [C.c_char_p]),
    "gs_plan_create_sharded": (_i, [C.POINTER(_vp), _i, _i, _i, _i, _i, C.c_char_p]),
    "gs_local_group_create": (_i, [C.POINTER(_vp), _i]),
    "gs_local_group_destroy": (_i, [_vp]),
    "gs_plan_create_sharded_local": (_i, [C.POINTER(_vp), _i, _i, _i, _i, _i, _vp]),
    "gs_plan_world": (_i, [_vp]),
    "gs_plan_rank": (_i, [_vp]),
    "gs_plan_nreal_local": (_i64, [_vp]),
    "gs_plan_npix_local": (_i64, [_vp]),
    "gs_shard_partition_m": (_i, [_i, _i, _i, _vp]),
    "gs_shard_partition_rings": (_i, [_i, _i, _i, _vp]),
    "gs_shard_real_index": (_i64, [_i, _i, _i, _vp]),
    "gs_shard_pixel_index": (_i64, [_i, _i, _i, _vp]),
    "gs_shard_expand_per_l": (_i, [_vp, _vp, _i, _vp, _vp]),
    "gs_shard_alm2cl": (_i, [_vp, _vp, _vp, _vp]),
    "gs_shard_allreduce_sum": (_i, [_vp, _vp, _i, _vp]),
    "gs_launch_count": (C.c_longlong, []),
    "gs_profile_matvec": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, C.POINTER(C.c_float), _vp]),
    "gs_profile_exchange": (_i, [_vp, _i, C.POINTER(C.c_float), _vp]),
    "gs_profile_matvec_batch": (_i, [_vp, _i, _vp, _vp, _i64, _vp, _vp, _vp, _vp, _i, C.POINTER(C.c_float), _vp]),
    "gs_measure_fp64_peak": (_i, [C.POINTER(_d), _vp]),
    "gs_profile_pcg_vectors": (_i, [_vp, _i, _i, C.POINTER(C.c_float), _vp]),
    "gs_profile_matvec_teb": (_i, [_vp, _vp, _vp, _vp, _i, C.POINTER(C.c_float), _vp]),
    "gs_set_ring_fused": (_i, [_i]),
    "gs_set_ring_skip": (_i, [_i]),
    "gs_set_ring_const": (_i, [_i]),
    "gs_constant_rings": (_i, [_vp, C.POINTER(_i)]),
    "gs_active_ring_pairs": (_i, [_vp, C.POINTER(_i), C.POINTER(_i)]),
}


class GibbsB200Error(RuntimeError):
    pass


def lib():
    """The loaded C-ABI library; raises if it was never built (no fallback path exists)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise GibbsB200Error(
                "libgibbs_b200.so not found at %s: the CUDA extension is not built "
                "(run __graft_entry__.build()); gibbssampler_b200 has no CPU fallback" % LIB_PATH)
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(l, name)
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def check(rc):
    if rc != 0:
        msg = lib().gs_last_error_string()
        raise GibbsB200Error("libgibbs_b200 error %d: %s" % (rc, msg.decode() if msg else "?"))
