"""CPU tests of the drop-in boundary: the C-ABI library builds for sm_100a, loads without a
GPU, exports every symbol include/fincflow_b200.h declares, and the host layer refuses to
run anywhere but on the CUDA kernels (no fallback)."""
import ctypes
import os
import re

import pytest
import torch

from conftest import REPO


@pytest.fixture(scope="module")
def lib_path():
    from fincflow_b200 import build

    return build.build()


def _header_functions():
    src = open(os.path.join(REPO, "include", "fincflow_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(finc_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol(lib_path):
    lib = ctypes.CDLL(lib_path)
    names = _header_functions()
    assert len(names) >= 11
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/fincflow_b200.h but not exported"
    from fincflow_b200 import _native

    assert sorted(_native.SYMBOLS) == names


def _header_prototypes():
    """{name: (return type, [parameter types])} of every function prototype in the header, types as written"""
    src = open(os.path.join(REPO, "include", "fincflow_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    protos = {}
    for ret, name, params in re.findall(r"([A-Za-z_][\w \t]*?\**)\s*\b(finc_[a-z0-9_]+)\s*\(([^)]*)\)\s*;", src):
        types = [re.sub(r"\s*\b\w+$", "", p.strip()) for p in params.split(",") if p.strip() not in ("", "void")]
        protos[name] = (ret.strip(), types)
    return protos


def _ctype_of(decl, structs):
    """the ctypes type a C type of the header binds to"""
    from fincflow_b200 import _native

    decl = " ".join(decl.replace("const", " ").replace("*", " * ").split())
    if decl == "char *":
        return ctypes.c_char_p
    if decl.endswith("*"):
        base = decl[:-1].strip()
        return ctypes.POINTER(getattr(_native, base)) if base in structs else ctypes.c_void_p
    return {"int": ctypes.c_int, "unsigned": ctypes.c_uint, "long": ctypes.c_long, "size_t": ctypes.c_size_t,
            "float": ctypes.c_float}[decl]


def test_signature_table_matches_the_header():
    """return type and the number and C type of every parameter of every header function, against the binding's
    one signature table"""
    from fincflow_b200 import _native

    src = open(os.path.join(REPO, "include", "fincflow_b200.h")).read()
    structs = set(re.findall(r"typedef struct (\w+)", src))
    protos = _header_prototypes()
    assert sorted(protos) == _header_functions() == sorted(_native._SIGNATURES)
    for name, (ret, params) in protos.items():
        restype, argtypes = _native._SIGNATURES[name]
        assert restype is _ctype_of(ret, structs), (name, ret, restype)
        want = [_ctype_of(p, structs) for p in params]
        assert len(argtypes) == len(want), (name, len(argtypes), len(want))
        for k, (got, exp) in enumerate(zip(argtypes, want)):
            assert got is exp, f"{name} parameter {k} ({params[k]}): {got} bound, {exp} declared"


def test_abi_version_and_error_strings(lib_path):
    from fincflow_b200 import _native

    lib = _native.load()
    assert lib.finc_abi_version() == 1
    assert b"bad argument" in lib.finc_error_string(-1)
    assert b"workspace" in lib.finc_error_string(-2)
    # argument validation happens before any CUDA call, so it is testable without a GPU
    assert lib.finc_forward_f32(None, None, None, None, 1, 4, 3, 8, 8, 3, 3, 0xE4, 0, None) == -1
    assert lib.finc_inverse_f32(None, None, None, 1, 17, 3, 8, 8, 3, 3, 0, 0, None) == -1  # G > 16
    assert lib.finc_backward_weight_workspace_bytes(256, 4, 3, 16, 16, 3, 3) >= 4096
    assert lib.finc_backward_weight_workspace_bytes(0, 4, 3, 16, 16, 3, 3) >= 4096   # B = 0: no plan, no division
    # tensor-core entry points: sizes are host arithmetic, bad arguments are rejected before any CUDA call
    assert lib.finc_coupling_prepared_bytes(12, 512, 0) > 4 * (2 * 512 * 64 + 2 * 512 * 512 + 2 * 9 * 16 * 512)
    assert lib.finc_coupling_prepared_bytes(12, 512, 1) > lib.finc_coupling_prepared_bytes(12, 512, 0)
    assert lib.finc_coupling_prepared_bytes(12, 16, 0) == 0 and lib.finc_coupling_prepared_bytes(13, 512, 0) == 0
    assert lib.finc_coupling_prepared_bytes(12, 96, 0) > 0 and lib.finc_coupling_prepared_bytes(12, 96, 1) == 0
    assert lib.finc_coupling_backward_workspace_bytes(256, 12, 16, 16, 512) > 0
    assert lib.finc_tc_wgrad_workspace_bytes(65536, 512, 512) > 0 and lib.finc_tc_wgrad_workspace_bytes(100, 512, 100) == 0
    assert lib.finc_slogdet_inverse_f32(None, None, None, 3, 200, None) == -1
    assert lib.finc_coupling_workspace_bytes(256, 12, 16, 16, 512) >= 4 * 256 * 256 * (64 + 512 + 512)
    assert lib.finc_coupling_apply_f32(None, None, None, None, None, 0, 1, 12, 8, 8, 512, 0, 0, None) == -1
    assert lib.finc_tc_conv_nhwc_f32(None, None, None, None, None, 1, 8, 8, 32, 32, 9, 0, 0, None) == -1
    assert lib.finc_tc_conv_weights_bytes(512, 6, 9, 1) == 2 * 512 * 64 * 4
    # glue entry points: the edges they refuse, before any CUDA call
    f, nil = ctypes.c_float, ctypes.c_void_p(16)   # a non-null, 16-byte aligned pointer that is never dereferenced
    assert lib.finc_affine1x1_f32(nil, nil, None, ctypes.c_void_p(32), 1, 4097, 16, None) == -1        # C > 4096
    assert lib.finc_affine1x1_backward_weight_workspace_bytes(1, 4097, 16) == 0
    assert lib.finc_slogdet_inverse_f32(nil, nil, nil, 3, 129, None) == -1                           # C > 128
    assert lib.finc_preprocess_f32(nil, None, nil, None, 1, 10, f(0.5), 0, None) == -1               # alpha >= 0.5
    assert lib.finc_squeeze_f32(nil, ctypes.c_void_p(64), 1, 3, 7, 8, None) == -1                    # odd H
    assert lib.finc_squeeze_f32(nil, ctypes.c_void_p(64), 1, 3, 8, 7, None) == -1                    # odd W
    assert lib.finc_squeeze_f32(ctypes.c_void_p(20), ctypes.c_void_p(64), 1, 3, 8, 8, None) == -1    # x 4-byte aligned
    # a workspace one float too small for the tiled affine weight gradient: FINC_E_WORKSPACE, nothing launched
    need = lib.finc_affine1x1_backward_weight_workspace_bytes(2, 16, 64)
    assert need > 64
    assert lib.finc_affine1x1_backward_weight_f32(nil, nil, nil, None, nil, need - 4, 2, 16, 64, None) == -2


def test_sass_is_sm100a_with_bulk_tma(lib_path):
    """the tiled kernels must really be Blackwell code using the TMA bulk-copy engine"""
    import shutil
    import subprocess

    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    out = subprocess.run([cuobjdump, "-sass", lib_path], capture_output=True, text=True).stdout
    assert "sm_100a" in out
    assert "UBLKCP" in out  # cp.async.bulk global<->shared
    assert "SYNCS" in out   # mbarrier
    # tensor-core path: tcgen05.mma / tcgen05.ld / TMA tensor-map loads and stores
    # (/opt/skills/guides/B200_PROFILING.md "What proves a Blackwell-native kernel")
    for mnemonic in ("UTCHMMA", "LDTM", "UTMALDG", "UTMASTG", "UTCBAR"):
        assert mnemonic in out, mnemonic
    assert "HMMA.16" not in out and "HGMMA" not in out   # no legacy mma.sync / wgmma paths


def test_no_cpu_fallback():
    from fincflow_b200 import _native
    from fincflow_b200.fastflow import FastFlowUnit
    from fincflow_b200.layers.conv import PaddedConv2d

    with pytest.raises(_native.FincNativeError):
        FastFlowUnit(8, 8, (3, 3))(torch.randn(2, 8, 4, 4))
    with pytest.raises(_native.FincNativeError):
        PaddedConv2d(3, 3, (3, 3), order="BR").reverse(torch.randn(2, 3, 4, 4))


def test_product_never_imports_the_oracle():
    pkg = os.path.join(REPO, "fincflow_b200")
    for root, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(root, f)).read()
                assert "oracle" not in txt.lower() or f == "build.py", f"{f} mentions the oracle"


def test_layer_api_matches_reference_surface():
    """names/attributes a reference user relies on (SURVEY.md 8b)"""
    from fincflow_b200.fastflow import FastFlowUnit
    from fincflow_b200.layers.conv import PaddedConv2d
    from fincflow_b200.layers.flowlayer import FlowLayer

    conv = PaddedConv2d(3, 3, (3, 3), order="TR")
    assert isinstance(conv, FlowLayer)
    assert conv.pad == (0, 2, 2, 0) and conv.order == "TR" and conv.kernel_size == (3, 3)
    assert list(conv.state_dict().keys()) == ["conv.weight"]
    w = conv.conv.weight.data
    # stored orientation of TR: corner tap (kH-1, 0): unit diagonal, zero above it
    for o in range(3):
        assert w[o, o, 2, 0] == 1.0 and (w[o, o + 1:, 2, 0] == 0).all()
    assert conv.mask.sum() == conv.mask.numel() - 3 * 4 // 2
    unit = FastFlowUnit(12, 12, (3, 3))
    assert sorted(unit.state_dict().keys()) == sorted(
        f"conv_{q}.conv.weight" for q in ("tl", "tr", "bl", "br"))
    other = FastFlowUnit(12, 12, 3)
    other.load_state_dict(unit.state_dict())
    assert torch.equal(other.weight, unit.weight)
    assert unit.conv_br.conv.weight.shape == (3, 3, 3, 3) and unit.conv_br.order == "BR"
    with pytest.raises(AssertionError):
        FastFlowUnit(6, 6, (3, 3))


def test_every_kernel_belongs_to_exactly_one_census(lib_path):
    """every kernel entry of the library (template instantiations from the symbol table, the others from their
    __device_stub__ symbols) belongs to exactly one of the three census family maps: FInC
    (test_gpu_kernel_variants.py), tensor-core (test_gpu_tc_variants.py) and glue (test_gpu_glue_variants.py), so a
    new kernel anywhere has to be claimed by a census.  Cross-checked against cuobjdump's function count."""
    import shutil
    import subprocess

    if not (shutil.which("nm") and shutil.which("c++filt")):
        pytest.skip("nm / c++filt not available")
    from test_gpu_glue_variants import GLUE_FAMILIES, kernel_entries
    from test_gpu_kernel_variants import FAMILIES
    from test_gpu_tc_variants import TC_FAMILIES

    entries = kernel_entries(lib_path)
    maps = {"finc": FAMILIES, "tc": TC_FAMILIES, "glue": GLUE_FAMILIES}
    owners = {}
    for name, args in entries:
        owners[(name, args)] = [m for m, fams in maps.items() if name in fams.values()]
    unclaimed = sorted(e for e, o in owners.items() if not o)
    assert not unclaimed, f"kernels no census claims: {unclaimed}"
    assert all(len(o) == 1 for o in owners.values())
    counts = {m: sum(1 for o in owners.values() if o == [m]) for m in maps}
    print(f"\n[library census] {len(entries)} kernel entries: {counts}")
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if os.path.exists(cuobjdump):
        out = subprocess.run([cuobjdump, "-res-usage", lib_path], capture_output=True, text=True).stdout
        functions = set(re.findall(r"^\s*Function (\S+?):", out, flags=re.M))
        assert len(functions) == len(entries), (len(functions), len(entries))
