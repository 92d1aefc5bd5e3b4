"""Compiles the reference's own Cython kernels (variance_expension.pyx) FROM WHERE THEY LIE in a checkout
of the reference into oracle/_ref/ (git-ignored), for tests/test_ref_cython.py:

    python oracle/build_ref.py <reference checkout>

TEST INFRASTRUCTURE ONLY.  No reference source is copied into the repository: Cython is pointed at
<reference checkout>/variance_expension.pyx and writes its generated C and the extension into oracle/_ref/.
The file needs language_level=2 (C-integer '/' at .pyx:14,42,90) and imports
healpy._healpy_sph_transform_lib._alm2map at module level (.pyx:2); a 2-line stub package in oracle/_ref/
satisfies that import (synthesis_hp is not used by the tests)."""
import os
import subprocess
import sys
import sysconfig

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "_ref")


def main():
    if len(sys.argv) != 2:
        print("usage: python oracle/build_ref.py <reference checkout>")
        return 2
    src = os.path.join(sys.argv[1], "variance_expension.pyx")
    if not os.path.exists(src):
        print("%s not found" % src)
        return 1
    os.makedirs(os.path.join(OUT, "healpy"), exist_ok=True)
    with open(os.path.join(OUT, "healpy", "__init__.py"), "w") as f:
        f.write("# stub: healpy is not installable here (oracle/build_ref.py)\n")
    with open(os.path.join(OUT, "healpy", "_healpy_sph_transform_lib.py"), "w") as f:
        f.write("def _alm2map(*a, **k):\n    raise RuntimeError('healpy stub')\n")
    import numpy as np
    cfile = os.path.join(OUT, "variance_expension.c")
    subprocess.check_call([sys.executable, "-m", "cython", "-2", "-o", cfile, src])
    ext = sysconfig.get_config_var("EXT_SUFFIX")
    so = os.path.join(OUT, "variance_expension" + ext)
    inc = [sysconfig.get_paths()["include"], np.get_include()]
    cmd = ["gcc", "-O2", "-fPIC", "-shared", "-w", cfile, "-o", so] + ["-I" + i for i in inc]
    subprocess.check_call(cmd)
    print("built", so)
    return 0


if __name__ == "__main__":
    sys.exit(main())
