"""The reference's own compiled Cython kernels (oracle/_ref, built from variance_expension.pyx of a reference checkout
by oracle/build_ref.py) against the oracle restatement (CPU) and the sm_100a kernels (GPU): index work bit-exact.
The repository holds no reference source: without oracle/_ref these tests skip."""
import os
import sys

import numpy as np
import pytest

from oracle import reference_logic as R

REF = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "_ref")


def ref_module():
    if not os.path.isdir(REF):
        pytest.skip("oracle/_ref not built (python oracle/build_ref.py <reference checkout>)")
    if REF not in sys.path:
        sys.path.insert(0, REF)
    try:
        import variance_expension as ve
    except ImportError as e:
        pytest.skip("oracle/_ref extension not importable: %s" % e)
    return ve


@pytest.mark.parametrize("L", [2, 3, 4, 7, 128, 512])
def test_oracle_matches_reference_cython(L):
    ve = ref_module()
    rng = np.random.default_rng(L)
    dl = rng.uniform(0.1, 3.0, L + 1)
    assert np.array_equal(np.asarray(ve.generate_var_cl_cython(dl)), R.generate_var_cl(dl))
    r = rng.standard_normal((L + 1) ** 2)
    c = np.asarray(ve.real_to_complex(r))
    # the Cython twin multiplies by 1/sqrt2 (variance_expension.pyx:86,98) where utils.py:59 divides: same index map
    assert np.allclose(c, R.real_to_complex(r), rtol=1e-15, atol=0)
    assert np.array_equal(np.asarray(ve.complex_to_real(c)), R.complex_to_real(c))
    z = np.asarray(ve.remove_monopole_dipole_contributions(r.copy()))
    assert np.array_equal(np.nonzero(z == 0)[0], np.array([0, 1, L + 1, L + 2]))


@pytest.mark.gpu
@pytest.mark.parametrize("L", [2, 3, 4, 7, 128, 512])
def test_gpu_kernels_match_reference_cython(L):
    ve = ref_module()
    from gibbssampler_b200 import utils
    rng = np.random.default_rng(100 + L)
    dl = rng.uniform(0.1, 3.0, L + 1)
    ref = np.asarray(ve.generate_var_cl_cython(dl))
    got = utils.generate_var_cl(dl)
    assert np.allclose(got, ref, rtol=1e-15, atol=0)
    # integer indexing bit-exact: expand the identity l -> l and compare positions
    ell = np.arange(L + 1, dtype=float)
    pos_ref = np.asarray(ve.generate_var_cl_cython(ell * (ell + 1) / (2 * np.pi) * np.where(ell > 0, ell, 1)))  # C_l = l (l>0)
    assert np.array_equal(np.rint(pos_ref[L + 1:]), utils.expand_per_l(ell, 0)[L + 1:])
    r = rng.standard_normal((L + 1) ** 2)
    c = np.asarray(ve.real_to_complex(r))
    assert np.allclose(utils.real_to_complex(r), c, rtol=1e-15, atol=0)
    assert np.array_equal(utils.complex_to_real(c), np.asarray(ve.complex_to_real(c)))
