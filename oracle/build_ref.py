"""Compile the REFERENCE's own CPU inverse solver into oracle/_ref/ (test infrastructure).

Source (read where it lies, never copied into the repo):
    $FINCFLOW_REFERENCE/fastflow/utils/fastflow_inverse/solve_parallel_mc.pyx
where FINCFLOW_REFERENCE names a checkout of aditya-v-kallappa/FInCFlow.
It is the default ``PaddedConv2d.reverse`` of the reference
(fastflow/layers/conv.py:109-163 -> solve_parallel, .pyx:77-126).  The shipped .so
files are cp37/cp39; the .pyx compiles unchanged with Cython 3 / numpy 2 / py3.12.

As in the reference's setup.py (fastflow/utils/fastflow_inverse/setup.py:1-5) no
``-fopenmp`` is passed, so ``prange`` runs on ONE thread -- that is the reference
as shipped.  Outputs (generated .c, .so) go only to oracle/_ref/, which is
git-ignored.

Without a reference checkout this script is a no-op and a previously built file, if
any, is used.
"""
from __future__ import annotations

import glob
import os
import subprocess
import sys
import sysconfig

HERE = os.path.dirname(os.path.abspath(__file__))
REFERENCE = os.environ.get("FINCFLOW_REFERENCE", "")
REF_PYX = os.path.join(REFERENCE, "fastflow", "utils", "fastflow_inverse", "solve_parallel_mc.pyx") if REFERENCE else ""
OUT_DIR = os.path.join(HERE, "_ref")
MOD = "solve_parallel_mc"


def built_path():
    hits = glob.glob(os.path.join(OUT_DIR, MOD + "*.so"))
    return hits[0] if hits else None


def build(force: bool = False):
    if not os.path.exists(REF_PYX):
        return built_path()  # no reference checkout: use what an earlier build left
    have = built_path()
    if have and not force and os.path.getmtime(have) >= os.path.getmtime(REF_PYX):
        return have
    import numpy as np

    os.makedirs(OUT_DIR, exist_ok=True)
    c_file = os.path.join(OUT_DIR, MOD + ".c")
    subprocess.check_call([sys.executable, "-m", "cython", "-3", REF_PYX, "-o", c_file])
    ext = sysconfig.get_config_var("EXT_SUFFIX")
    so = os.path.join(OUT_DIR, MOD + ext)
    subprocess.check_call([
        "gcc", "-O2", "-fPIC", "-shared", "-w",
        "-DNPY_NO_DEPRECATED_API=NPY_1_7_API_VERSION",
        "-I" + sysconfig.get_paths()["include"], "-I" + np.get_include(),
        c_file, "-o", so,
    ])
    return so


def load():
    """Import the compiled reference solver; returns the module or None."""
    so = build()
    if not so:
        return None
    import importlib.util

    spec = importlib.util.spec_from_file_location(MOD, so)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


if __name__ == "__main__":
    print(build(force="--force" in sys.argv))
