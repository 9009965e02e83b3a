"""Compile the REFERENCE's own CUDA inverse extensions into oracle/_ref/ (test infrastructure).

Sources (read where they lie in the reference checkout named by FINCFLOW_REFERENCE, never copied, never modified):
    $FINCFLOW_REFERENCE/fastflow/utils/fastflow_cuda_inverse/cinc_cuda_level{1,2}.cpp
    $FINCFLOW_REFERENCE/fastflow/utils/fastflow_cuda_inverse/cinc_cuda_kernel_level{1,2}.cu
They are the pybind modules `cinc_cuda_level1` / `cinc_cuda_level2` the reference JIT-builds at
import time (fastflow/fastflow.py:9-10, layers/conv.py:11-12): one function
`inverse(input, kernel, output) -> [output]` (cinc_cuda_level2.cpp:19-32), (H+W-1)*Cq launches each
followed by cudaDeviceSynchronize (cinc_cuda_kernel_level2.cu:98-132).

Under torch 2.x the .cu files need ONE missing ATen overload, supplied by the pre-included
oracle/ref_cuda_shim.h instead of patching the source.  nvcc cross-compiles for sm_100 without a GPU;
the .so files land in oracle/_ref/ (git-ignored) and are used by tests/test_gpu_reference_cuda.py and
bench.py's `gpu_reference` block as the reference's GPU path.

Without a reference checkout build() only returns files an earlier build left.
"""
from __future__ import annotations

import glob
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
REFERENCE = os.environ.get("FINCFLOW_REFERENCE", "")
REF_DIR = os.path.join(REFERENCE, "fastflow", "utils", "fastflow_cuda_inverse") if REFERENCE else ""
OUT_DIR = os.path.join(HERE, "_ref")
SHIM = os.path.join(HERE, "ref_cuda_shim.h")
LEVELS = {1: "cinc_cuda_level1", 2: "cinc_cuda_level2"}


def built_path(level: int):
    hits = glob.glob(os.path.join(OUT_DIR, LEVELS[level], LEVELS[level] + "*.so"))
    return hits[0] if hits else None


def build(level: int = 2, force: bool = False):
    name = LEVELS[level]
    srcs = [os.path.join(REF_DIR, f"{name}.cpp"), os.path.join(REF_DIR, f"cinc_cuda_kernel_level{level}.cu")]
    if not REF_DIR or not all(os.path.exists(s) for s in srcs):
        return built_path(level)  # no reference checkout: use what an earlier build left
    have = built_path(level)
    if have and not force and os.path.getmtime(have) >= max(os.path.getmtime(s) for s in srcs + [SHIM]):
        return have
    os.environ.setdefault("TORCH_CUDA_ARCH_LIST", "10.0")
    from torch.utils import cpp_extension

    out = os.path.join(OUT_DIR, name)
    os.makedirs(out, exist_ok=True)
    cpp_extension.load(name=name, sources=srcs, build_directory=out, verbose=False, is_python_module=False,
                       extra_cflags=["-O2", "-w"], extra_cuda_cflags=["-O2", "-w", "-include", SHIM])
    return built_path(level)


def load(level: int = 2):
    """import the compiled reference extension (torch must be importable); None if it was never built"""
    so = build(level)
    if not so:
        return None
    import importlib.util

    import torch  # noqa: F401  (the extension links against libtorch)

    spec = importlib.util.spec_from_file_location(LEVELS[level], so)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


if __name__ == "__main__":
    for lv in (1, 2):
        print(build(lv, force="--force" in sys.argv))
