"""CPU (-m "not gpu"): gs_plan_create refuses NSIDE above what the ring stage can build (GS_NSIDE_MAX = 2048) before any
device work, with a message that names the limit, and leaves the output handle NULL.  Runs without a GPU: the refusal comes
from the argument check, not from a failed allocation."""
import ctypes as C
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_header_states_the_nside_limit():
    hdr = open(os.path.join(ROOT, "include", "gibbs_b200.h")).read()
    assert re.search(r"#define\s+GS_NSIDE_MAX\s+2048\b", hdr)


@pytest.mark.parametrize("nside,lmax", [(2049, 4096), (8192, 16384), (4096, 8192), (2049, 2)])
def test_plan_create_refuses_nside_above_2048(nside, lmax):
    from gibbssampler_b200 import _lib
    lib = _lib.lib()
    sentinel = C.c_void_p(0x1234)
    p = C.c_void_p(sentinel.value)
    assert lib.gs_plan_create(C.byref(p), nside, lmax, -1) == -1            # GS_E_BADARG
    assert p.value is None                                                  # *out = NULL
    msg = lib.gs_last_error_string()
    assert b"2048" in msg and b"nside" in msg, msg
    p = C.c_void_p(sentinel.value)
    assert lib.gs_plan_create_sharded(C.byref(p), nside, lmax, -1, 0, 1, None) == -1
    assert p.value is None and b"2048" in lib.gs_last_error_string()


def test_lmax_bounds_still_checked_at_the_nside_limit():
    """The nside check comes first; at an accepted nside the lmax bound 2 <= lmax <= 4 nside still refuses."""
    from gibbssampler_b200 import _lib
    lib = _lib.lib()
    p = C.c_void_p()
    assert lib.gs_plan_create(C.byref(p), 2048, 8193, -1) == -1
    assert b"lmax" in lib.gs_last_error_string() and p.value is None
    assert lib.gs_plan_create(C.byref(p), 2048, 1, -1) == -1
    assert b"lmax" in lib.gs_last_error_string() and p.value is None
