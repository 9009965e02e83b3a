"""Build libfincflow_b200.so (the C-ABI CUDA library) in-tree for sm_100a.

    python -m fincflow_b200.build [--force] [--verbose]

nvcc cross-compiles without a GPU.  The .so is git-ignored but travels to the GPU box
with the gpurun snapshot.  CUDA runtime is linked statically so the library has no
dependency on torch's bundled runtime and loads with plain ctypes.
"""
from __future__ import annotations

import concurrent.futures as cf
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT_DIR = os.path.join(HERE, "lib")
LIB = os.path.join(OUT_DIR, "libfincflow_b200.so")
SOURCES = [f"finc_inverse_rw_{adj}c{c}k{k}.cu" for c, k in ((12, 5), (12, 3), (6, 5), (6, 3), (4, 5), (3, 5), (4, 3),
                                                            (3, 3), (2, 5), (2, 3), (1, 5), (1, 3))
           for adj in ("", "adj_")] + [  # heaviest first; each inverse family with its adjoint
    "finc_inverse_rw_multi.cu", "finc_api.cu", "finc_naive.cu", "finc_conv.cu", "finc_inverse.cu", "finc_inverse_wave.cu", "finc_inverse_rw.cu",
    "finc_wgrad.cu", "finc_collective.cu", "finc_affine.cu", "finc_chain.cu", "tc_api.cu", "tc_wgrad.cu",
    *[f"tc_igemm_nhwc_p{p}_c{c}.cu" for p in (3, 1) for c in (1, 2, 4)], "tc_igemm_rows_p3.cu", "tc_igemm_rows_p1.cu"] + [
    f"finc_inverse_wave_c{c}.cu" for c in (24, 12, 6, 4, 3, 2, 1)] + [  # heaviest first
    f"finc_conv_c{c}.cu" for c in (0, 6, 24, 12, 4, 3, 2, 1)]
HEADERS = [os.path.join(CSRC, "finc_common.cuh"), os.path.join(CSRC, "finc_inverse_wave.cuh"), os.path.join(CSRC, "finc_inverse_rw.cuh"), os.path.join(CSRC, "finc_conv.cuh"),
           os.path.join(os.path.dirname(HERE), "include", "fincflow_b200.h")]

NVCC_FLAGS = [
    "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
    "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr", "-Xptxas", "-v",
]


def _nvcc():
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found: cannot build libfincflow_b200.so")
    return exe


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def _deps(src, seen=None):
    """the source plus every header it includes (transitively, quoted includes only)"""
    import re

    seen = set() if seen is None else seen
    src = os.path.normpath(src)
    if src in seen or not os.path.exists(src):
        return seen
    seen.add(src)
    with open(src) as f:
        for inc in re.findall(r'^\s*#include\s+"([^"]+)"', f.read(), flags=re.M):
            _deps(os.path.join(os.path.dirname(src), inc), seen)
    return seen


def _compile(src, obj, verbose):
    cmd = [_nvcc(), *NVCC_FLAGS, "-ccbin", "g++", "-c", src, "-o", obj]
    p = subprocess.run(cmd, capture_output=True, text=True)
    log = obj + ".log"
    with open(log, "w") as f:
        f.write(" ".join(cmd) + "\n" + p.stdout + p.stderr)
    if p.returncode != 0:
        raise RuntimeError(f"nvcc failed for {src}:\n{p.stderr[-4000:]}")
    if verbose:
        print(p.stderr)
    return obj


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OUT_DIR, exist_ok=True)
    objs, jobs = [], []
    for s in SOURCES:
        src = os.path.join(CSRC, s)
        obj = os.path.join(OUT_DIR, s.replace(".cu", ".o"))
        objs.append(obj)
        if force or _stale(obj, sorted(_deps(src))):
            jobs.append((src, obj))
    if jobs:
        with cf.ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 4)) as ex:
            list(ex.map(lambda j: _compile(j[0], j[1], verbose), jobs))
    if jobs or not os.path.exists(LIB):
        cmd = [_nvcc(), "-shared", "-cudart", "static", "-ccbin", "g++", "-o", LIB, *objs]
        subprocess.check_call(cmd)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
