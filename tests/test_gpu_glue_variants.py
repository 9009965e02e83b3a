"""The glue and fall-back kernels of the library against float64 references, with a census of the kernels that ran.

test_gpu_kernel_variants.py and test_gpu_tc_variants.py take a census of the hot-path template families.  Every
other kernel in the library is glue: the per-pixel affine map of each flow step (ActNorm + Conv1x1) and its weight
gradient, the inverse for groups the register-window and wavefront kernels do not cover (inverse_warp_kernel<CP>),
the generic kernels of FINC_FLAG_NAIVE, the preprocessing, log-density, log-det, mask, squeeze and Adam kernels,
the small matrix inverse of the 1x1 convolutions, and the helpers of the tensor-core coupling and dense inverse.

Each recipe below reaches one of them and asserts, under torch.profiler, that exactly that kernel ran.  References
are float64 PyTorch on the GPU or the float64 FInC oracle.  test_every_glue_kernel_is_exercised runs every recipe
and requires each glue kernel in the library's symbol table to have been launched, except those in UNREACHABLE.
test_native_abi.py checks, without a GPU, that every kernel entry of the library belongs to exactly one of the
three censuses.
"""
import functools
import json
import math
import os
import re
import subprocess
import tempfile

import numpy as np
import pytest
import torch

from oracle import finc_oracle as fo
from test_gpu_inverse_grad import adjoint_oracle
from test_gpu_kernel_variants import check_guarded, guarded, kernels_in, launched

pytestmark = pytest.mark.gpu

ORDERS = (0, 1, 2, 3)
G = len(ORDERS)
EPS32 = 2.0 ** -24

_ANON = "finc::(anonymous namespace)::"
GLUE_FAMILIES = {
    # finc_affine.cu
    "affine": _ANON + "affine1x1_kernel",
    "affine_split": _ANON + "affine1x1_split_kernel",
    "affine_generic": _ANON + "affine1x1_generic_kernel",
    "affine_wgrad": _ANON + "affine1x1_wgrad_kernel",
    "affine_wgrad_finish": _ANON + "affine1x1_wgrad_finish_kernel",
    "affine_wgrad_generic": _ANON + "affine1x1_wgrad_generic_kernel",
    "preprocess": "finc::preprocess_kernel",
    "slogdet_inverse": "finc::slogdet_inverse_kernel",
    # finc_inverse.cu
    "inverse_warp": _ANON + "inverse_warp_kernel",
    # finc_naive.cu
    "conv_naive": "finc::conv_naive_kernel",
    "inverse_naive": "finc::inverse_naive_kernel",
    "wgrad_naive": "finc::wgrad_naive_kernel",
    "mask": "finc::mask_kernel",
    "logdet": "finc::logdet_kernel",
    "gaussian_logp": "finc::gaussian_logp_kernel",
    "squeeze": "finc::squeeze_kernel",
    "adam": "finc::adam_kernel",
    "adam_tick": "finc::adam_tick_kernel",
    # weight tables of the FInC kernels, the multi-level inverse, the collective
    "conv_prepare": _ANON + "conv_prepare_kernel",
    "wave_prepare": _ANON + "wave_prepare_kernel",
    "inverse_rw_multi": "finc::rw::inverse_rw_multi_kernel",
    "allreduce_adam": _ANON + "allreduce_adam_kernel",
    # tc_api.cu, tc_wgrad.cu: helpers of the tensor-core coupling layer and dense inverse
    **{f"tc_{k}": f"finc::tc::{k}_kernel" for k in (
        "split_weights", "im2col3x3", "rowsum_reduce", "coupling_gather", "coupling_bwd_weights",
        "coupling_bwd_pointwise", "coupling_bwd_expand", "coupling_bwd_col2im", "colsum_partial", "colsum_final",
        "wgrad_unpack", "coupling_vectors", "wgrad_reduce")},
    "dense_inverse_weights": "dense_inverse_weights_kernel",   # extern "C": unmangled
    "dense_identity": "dense_identity_kernel",
}

# glue kernels no recipe here may launch, with the reason (from the code)
UNREACHABLE = {
    ("allreduce_adam", ()): "spin-waits on the signal flags of its peer ranks (finc_collective.cu); a single "
                            "process cannot launch it without hanging.  tests/multirank_check.py runs it",
}


def glue_launched(fn):
    return launched(fn, GLUE_FAMILIES)


# ---- the library's kernel entries (no GPU needed) ------------------------------------------------------------------
def _demangle(names):
    out = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True, check=True).stdout
    return out.splitlines()


def library_kernels(lib_path=None):
    """the demangled names of every kernel entry in the library: template instantiations from the demangled symbol
    table (`void <name><args>(...)`), the others from their `__device_stub__` symbols.  A name ending in `_kernel`
    alone is not enough: finc::rw::(anonymous namespace)::multi_kernel() is a host function."""
    if lib_path is None:
        from fincflow_b200 import _native

        lib_path = _native.LIB_PATH
    names = set()
    plain = subprocess.run(["nm", lib_path], capture_output=True, text=True, check=True).stdout
    stubs = sorted({m.group(1) for m in re.finditer(r"__device_stub_(_Z\w+)", plain)})
    names.update(_demangle(stubs))
    demangled = subprocess.run(["nm", "-C", lib_path], capture_output=True, text=True, check=True).stdout
    for line in demangled.splitlines():
        m = re.match(r"^\w+ [tTwW] void ((?:\w+::|\(anonymous namespace\)::)*\w+_kernel<.*)$", line)
        if m:
            names.add(m.group(1))
    return names


def kernel_entries(lib_path=None):
    """{(qualified name, template arguments)} of every kernel entry in the library"""
    from test_gpu_kernel_variants import _template_args

    out = set()
    for name in library_kernels(lib_path):
        base = re.match(r"(?:\w+::|\(anonymous namespace\)::)*\w+", name).group(0)
        rest = name[len(base):]
        out.add((base, _template_args(rest)[0] if rest.startswith("<") else ()))
    return out


# ---- float64 comparisons on the GPU (the formulas of conftest.rel_err and conftest.elementwise_close) ------------
def rel64(got, want):
    got, want = got.double(), want.double()
    return float((got - want).abs().max() / max(float(want.abs().max()), 1e-30))


def close64(got, want, rtol=1e-5, floor=1e-1):
    got, want = got.double(), want.double()
    return bool(((got - want).abs() <= rtol * (want.abs() + floor * want.abs().max())).all())


def npy(t):
    return t.detach().double().cpu().numpy()


@pytest.fixture(scope="module")
def nat():
    from fincflow_b200 import _native

    _native.load()
    return _native


def _sms():
    from fincflow_b200 import _native

    return _native.sm_count()


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def offset_copy(t, offset):
    """a contiguous copy of `t` starting `offset` floats past a 16-byte boundary"""
    buf = torch.empty(t.numel() + 4, device="cuda")
    v = buf[offset:offset + t.numel()].view(t.shape)
    v.copy_(t)
    return v


def expect_one(fn, key, what=""):
    out, ran = glue_launched(fn)
    assert ran == {key}, (what, ran)
    return out


# ================================================================================================================
# affine1x1_kernel<C, VEC>, affine1x1_split_kernel<C>, affine1x1_generic_kernel  (finc_affine.cu, launch_affine1x1)
# ================================================================================================================
AFFINE_C = (4, 8, 12, 16, 24, 32, 48, 96)        # the specialised channel counts
AFFINE_GENERIC_C = (1, 3, 5, 10, 100, 256)
# layouts: (H, W), float offset of x and y; the vector width the layout allows (rows start at multiples of HW floats)
AFFINE_LAYOUTS = {
    "v4": ((16, 16), 0),     # HW % 4 == 0, 16-byte aligned: float4
    "v2off": ((16, 16), 2),  # 8-byte aligned: float2
    "v1off": ((16, 16), 1),  # 4-byte aligned: scalar
    "v2hw": ((14, 15), 0),   # HW % 4 == 2: float2
    "v1hw": ((15, 15), 0),   # HW odd: scalar
}


def affine_vec(H, W, offset):
    hw = H * W
    if hw % 4 == 0 and offset % 4 == 0:
        return 4
    return 2 if hw % 2 == 0 and offset % 2 == 0 else 1


def affine_vmax(C):
    return 1 if C >= 96 else 2 if C >= 32 else 4


def affine_big_batch(C, H, W, vec):
    """the smallest batch (+ 3) at which launch_affine1x1 takes the vectorised kernel: B * HW / min(vec, vmax)
    pixel-vectors >= SMs * 512 (below that, the split kernel)"""
    per_image = (H * W) // min(vec, affine_vmax(C))
    return -(-_sms() * 512 // per_image) + 3


@functools.lru_cache(maxsize=None)
def _affine_params(C):
    g = _gen(7000 + C)
    A = torch.randn(C, C, device="cuda", generator=g) / math.sqrt(C)
    b = torch.randn(C, device="cuda", generator=g)
    return A, b


@functools.lru_cache(maxsize=4)
def _affine_images(C, B, H, W):
    return torch.randn(B, C, H, W, device="cuda", generator=_gen(C * 7 + B + H * W))


def affine_ref(x, A, b):
    y = torch.einsum("oi,nihw->nohw", A.double(), x.double())
    return y if b is None else y + b.double().view(1, -1, 1, 1)


def run_affine(nat, x, A, b, offset, key, what):
    """y = A x + b with x and y `offset` floats past a 16-byte boundary, y inside sentinel guards; only `key` ran"""
    xs = offset_copy(x, offset) if offset else x
    buf, view = guarded(tuple(x.shape), offset)
    expect_one(lambda: nat.affine1x1(xs, A, b, out=view), key, what)
    check_guarded(buf, view, offset, what)
    return view.clone()


def check_affine(y, x, A, b, what):
    want = affine_ref(x, A, b)
    assert rel64(y, want) <= 1e-5, (what, rel64(y, want))
    assert close64(y, want), what


@pytest.mark.parametrize("C", AFFINE_C)
def test_affine1x1_variants(nat, C):
    """every layout at a batch past the threshold runs affine1x1_kernel<C, min(vec, vmax)>; the same images alone run
    affine1x1_split_kernel<C>.  All kernels compute each output as the same bias-first fmaf chain over i ascending,
    so the images they share come out bit-identical, and within 1e-5 of float64.  With and without bias."""
    A, b = _affine_params(C)
    for hw, layouts in (((16, 16), ("v4", "v2off", "v1off")), ((14, 15), ("v2hw",)), ((15, 15), ("v1hw",))):
        H, W = hw
        vmax_here = max(min(affine_vec(H, W, AFFINE_LAYOUTS[n][1]), affine_vmax(C)) for n in layouts)
        B = affine_big_batch(C, H, W, vmax_here)
        x = _affine_images(C, B, H, W)
        alone = {}
        for bias in (b, None):
            for off in (0, 1):
                alone[(off, bias is None)] = run_affine(nat, x[:3].contiguous(), A, bias, off, ("affine_split", (C,)),
                                                         f"C{C} {hw} alone offset {off} bias {bias is not None}")
            assert torch.equal(alone[(0, bias is None)], alone[(1, bias is None)])
            check_affine(alone[(0, bias is None)], x[:3], A, bias, f"C{C} split")
        for name in layouts:
            off = AFFINE_LAYOUTS[name][1]
            vec = min(affine_vec(H, W, off), affine_vmax(C))
            for bias in ((b, None) if name in ("v4", "v1hw") else (b,)):
                what = f"C{C} {name} B{B} bias {bias is not None}"
                y = run_affine(nat, x, A, bias, off, ("affine", (C, vec)), what)
                assert torch.equal(y[:3], alone[(0, bias is None)]), what + ": differs from the split kernel"
                check_affine(y, x, A, bias, what)
                del y


@pytest.mark.parametrize("C", AFFINE_GENERIC_C)
def test_affine1x1_generic(nat, C):
    """channel counts without a specialisation: affine1x1_generic_kernel, with and without bias, odd and unaligned
    layouts, and (C = 256) more elements than its grid covers in one pass"""
    A, b = _affine_params(C)
    for B, H, W, off in ((3, 5, 7, 0), (2, 16, 16, 1), (9 if C < 256 else 4, 32, 32, 2)):
        x = torch.randn(B, C, H, W, device="cuda", generator=_gen(C + B))
        outs = []
        for bias in (b, None):
            for o in sorted({0, off}):
                y = run_affine(nat, x, A, bias, o, ("affine_generic", ()), f"C{C} B{B} {H}x{W} offset {o}")
                check_affine(y, x, A, bias, f"C{C} generic")
                outs.append((bias is None, y))
        for nb, y in outs:
            ref = next(v for k, v in outs if k == nb)
            assert torch.equal(y, ref)


# ================================================================================================================
# affine1x1_wgrad_kernel + _finish_kernel (C % 4 == 0, C <= 108), affine1x1_wgrad_generic_kernel (finc_affine.cu)
# ================================================================================================================
AW_PT = 64   # pixels per tile (kAwPT)


def affine_wgrad_plan(C):
    """(tiled, slices, rounds) of launch_affine1x1_wgrad: tiled when C % 4 == 0 and (C/4)^2 <= 3 * 256; a 4x4 block
    of (o, i) per thread and round; slices = clamp(256 / (C/4)^2, 1, 16) threads share a block's pixels"""
    nblk = (C // 4) ** 2
    if C % 4 or nblk > 768:
        return False, 0, 0
    return True, max(1, min(256 // nblk, AW_PT // 4)), -(-nblk // 256)


# slices 16 (C <= 16), 10, 7, 4, 2 (C = 20, 24, 32, 40), 1 from C = 48; a third round from (C/4)^2 > 512 (C >= 92),
# which also needs over 48 KB of dynamic shared memory (2 * C * 68 floats); C = 112 and odd C: generic
AW_C = (4, 16, 20, 24, 32, 40, 48, 92, 108, 112, 6, 13)
AW_SHAPES = [  # B, H, W, offset
    (1, 7, 7, 0),      # one tile (49 pixels), HW % 4 != 0: scalar staging
    (3, 10, 10, 0),    # 300 pixels: a short last tile, float4 staging
    (37, 32, 32, 0),   # 592 tiles: more than the 2 * SMs CTAs, float4 staging
    (37, 32, 32, 1),   # unaligned: scalar staging
    (5, 9, 11, 0),     # odd HW
]


def test_affine_wgrad_plan_covers_every_feature():
    plans = {C: affine_wgrad_plan(C) for C in AW_C}
    assert {p[1] for p in plans.values() if p[0]} == {16, 10, 7, 4, 2, 1}
    assert any(p[2] == 3 for p in plans.values()) and any(not p[0] for p in plans.values())
    assert any(2 * C * (AW_PT + 4) * 4 > 48 * 1024 for C, p in plans.items() if p[0])


@pytest.mark.parametrize("C", AW_C)
def test_affine1x1_backward_weight(nat, C):
    """dA = sum dy x^T and db = sum dy against float64, element-wise within 2e-6 of sum |dy_o| |x_i| (the bound of an
    fp32 sum of products in any order, with margin); the tiled and the generic kernel; deterministic; want_bias=False
    gives the same dA; B = 0 gives zeros"""
    tiled, _, _ = affine_wgrad_plan(C)
    keys = {("affine_wgrad", ()), ("affine_wgrad_finish", ())} if tiled else {("affine_wgrad_generic", ())}
    for B, H, W, off in AW_SHAPES:
        g = _gen(C * 100 + B + off)
        x = offset_copy(torch.randn(B, C, H, W, device="cuda", generator=g), off)
        dy = offset_copy(torch.randn(B, C, H, W, device="cuda", generator=g), off)
        (dA, db), ran = glue_launched(lambda: nat.affine1x1_backward_weight(dy, x))
        assert ran == keys, (C, B, H, W, off, ran)
        what = f"C{C} B{B} {H}x{W} offset {off}"
        x64, d64 = x.double().flatten(2), dy.double().flatten(2)
        want = torch.einsum("nop,nip->oi", d64, x64)
        bound = 2e-6 * torch.einsum("nop,nip->oi", d64.abs(), x64.abs())
        assert bool(((dA.double() - want).abs() <= bound).all()), (what, float((dA.double() - want).abs().max()))
        want_b = d64.sum((0, 2))
        assert bool(((db.double() - want_b).abs() <= 2e-6 * d64.abs().sum((0, 2))).all()), what
        dA2, db2 = nat.affine1x1_backward_weight(dy, x)
        assert torch.equal(dA2, dA) and torch.equal(db2, db), what + ": not deterministic"
        dA3, none = nat.affine1x1_backward_weight(dy, x, want_bias=False)
        assert none is None and torch.equal(dA3, dA), what
    e = torch.empty(0, C, 4, 4, device="cuda")
    dA0, db0 = nat.affine1x1_backward_weight(e, e)
    assert not bool(dA0.any()) and not bool(db0.any())


# ================================================================================================================
# inverse_warp_kernel<CP>  (finc_inverse.cu, launch_inverse_fast)
# ================================================================================================================
WARP_CP = (1, 2, 3, 4, 6, 8, 12, 16, 24, 32)


def _optin():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).shared_memory_per_block_optin


def warp_plan(B, Gn, C, H, W, kh, kw, aligned=True, sms=None, optin=None):
    """launch_inverse_fast restated: None when it refuses the shape, else its schedule (CP, gsplit, S, T, bulk, warps,
    CTAs).  The tests use it to state what each shape exercises; the kernel itself is asserted by name."""
    sms = _sms() if sms is None else sms
    optin = _optin() if optin is None else optin
    CP = next((o for o in WARP_CP if C <= o), 0)
    tile = C * H * W
    if CP == 0 or tile * 4 > 96 * 1024:
        return None
    CPP = CP if CP <= 2 else -(-CP // 4) * 4
    wk_per_g = kh * kw * C * CPP
    budget = optin - 4096 if optin > 8192 else 0
    if wk_per_g * Gn * 4 <= budget // 2:
        gsplit, wk = 0, wk_per_g * Gn
    elif wk_per_g * 4 <= budget // 2:
        gsplit, wk = 1, wk_per_g
    else:
        return None
    bulk = int(tile % 4 == 0 and aligned)
    WL = min(W, 32)
    T = 32 // WL
    stride = -(-tile // 4) * 4
    if T > 1 and WL % 4 == 0:
        while stride % 32 != WL % 32:
            stride += 4
    wk_bytes = -(-wk // 32) * 32 * 4
    stage = T * stride * 4
    nbT = -(-B // T)
    n_items = nbT if gsplit else nbT * Gn
    ctas = max(1, sms // Gn if gsplit else sms)
    ctas = min(ctas, n_items)
    ipc = -(-n_items // ctas)
    S = nw = 0
    for s in (3, 2, 1):
        n = min((budget - wk_bytes) // (s * stage + s * 8), 16)
        want = min(ipc, 16)
        if n >= (1 if s == 1 else min(want, 8)):
            S, nw = s, n
            break
    if nw < 1:
        return None
    if ipc <= nw:
        S = 1
    while nw > 1 and (nw - 1) * ctas >= n_items:
        nw -= 1
    return {"CP": CP, "gsplit": gsplit, "S": S, "T": T, "bulk": bulk, "warps": nw, "ctas": ctas}


# C, (kh, kw), H, W, a large batch.  Every CP with C = CP, and the padded C = 5, 7, 11, 15, 23, 31.
WARP_CASES = [
    (1, (3, 3), 16, 16, 1300), (2, (3, 3), 8, 8, 1300), (3, (3, 3), 12, 12, 700), (4, (3, 3), 6, 40, 300),
    (5, (3, 3), 8, 8, 900), (6, (5, 5), 8, 8, 400), (7, (3, 3), 8, 8, 1300), (8, (3, 3), 8, 8, 2000),
    (11, (3, 3), 8, 8, 300), (12, (3, 3), 8, 8, 1500), (15, (3, 3), 8, 8, 300), (16, (3, 3), 8, 8, 300),
    (23, (3, 3), 4, 4, 300), (24, (3, 3), 4, 4, 300), (31, (3, 3), 8, 8, 64), (32, (3, 3), 8, 8, 64),
    (4, (2, 2), 8, 8, 300), (4, (1, 3), 8, 8, 300), (6, (3, 2), 9, 9, 300), (3, (4, 4), 12, 12, 300),
]
WARP_DEFAULT_C = (8, 16, 32)   # no register-window or wavefront kernel: the default path takes inverse_warp_kernel


def warp_schedules(C, k, H, W, B):
    """(tag, batch, groups, offset, in place) runs of one case; every run shares images 0..2 of groups 0 and 1"""
    runs = [("big", B, G, 0, False), ("one", 1, G, 0, False), ("ragged", 5, G, 0, False),
            ("lanes", B, G, 1, False), ("two_groups", 3, 2, 0, False), ("in_place", 5, G, 0, True)]
    return runs


def _warp_id(c):
    C, k, H, W, B = c
    return f"C{C}_k{k[0]}x{k[1]}_{H}x{W}"


@functools.lru_cache(maxsize=2)
def _warp_data(C, k, H, W, B):
    rng = np.random.default_rng(C * 31 + k[0] * 7 + k[1] + H)
    w = fo.init_unit_weight(C, k, rng, std=0.05)
    x = rng.standard_normal((B, G * C, H, W)).astype(np.float32)
    z = fo.forward(x, w.astype(np.float64), ORDERS).astype(np.float32)
    return torch.from_numpy(w).cuda(), torch.from_numpy(x).cuda(), torch.from_numpy(z).cuda()


def test_inverse_warp_schedules_cover_the_planner():
    """the planner arithmetic the cases rely on, at this device's SM count and shared-memory limit: gsplit, 1, 2 and
    3 stages, bulk and lane copies, T > 1 with a ragged last item and W > 32 all occur"""
    seen = {"gsplit": set(), "S": set(), "bulk": set(), "ragged_T": False, "wide": False}
    for C, k, H, W, B in WARP_CASES:
        for tag, b, g, off, _ in warp_schedules(C, k, H, W, B):
            p = warp_plan(b, g, C, H, W, *k, aligned=off == 0)
            assert p is not None, (C, k, H, W, tag)
            seen["gsplit"].add(p["gsplit"])
            seen["S"].add(p["S"])
            seen["bulk"].add(p["bulk"])
            seen["ragged_T"] |= p["T"] > 1 and b % p["T"] != 0
            seen["wide"] |= W > 32
    assert seen["gsplit"] == {0, 1} and seen["S"] == {1, 2, 3} and seen["bulk"] == {0, 1}, seen
    assert seen["ragged_T"] and seen["wide"]
    # C = 32, k = 3, G = 4: 4 * 9 * 32 * 32 floats of weights = 147 KB, over half the budget: one group per CTA row
    assert warp_plan(64, 4, 32, 8, 8, 3, 3)["gsplit"] == 1 and warp_plan(3, 2, 32, 8, 8, 3, 3)["gsplit"] == 0


def launch_dims(fn, name_part):
    """(grid, block) of the kernels whose name contains `name_part`, from the profiler's chrome trace (None when the
    trace does not carry them)"""
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        torch.zeros(1, device="cuda").add_(1)
        torch.cuda.synchronize()
        fn()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f).get("traceEvents", [])
    dims = [(e.get("args", {}).get("grid"), e.get("args", {}).get("block")) for e in events
            if e.get("cat") == "kernel" and name_part in e.get("name", "")]
    return dims if dims and all(g is not None for g, _ in dims) else None


@pytest.mark.parametrize("case", WARP_CASES, ids=_warp_id)
def test_inverse_warp_variants(nat, case):
    """inverse_warp_kernel<CP> under FINC_FLAG_GENERIC_TILED (and by default for C = 8, 16, 32) over its schedules:
    the batch (stages S), one image, a ragged last item, lane copies (unaligned), two groups (no gsplit where four
    need it) and in place.  The per-pixel FMA order does not depend on the schedule, so every run gives the same bits
    on the images they share; the oracle on the first and last images; the forward round trip; guard zones."""
    C, k, H, W, B = case
    w, x, z = _warp_data(C, k, H, W, B)
    plan = warp_plan(B, G, C, H, W, *k)
    key = ("inverse_warp", (plan["CP"],))
    flag_sets = [nat.FLAG_GENERIC_TILED] + ([0] if C in WARP_DEFAULT_C else [])
    shared = []
    for tag, b, g, off, in_place in warp_schedules(C, k, H, W, B):
        zs = z[:b, :g * C].contiguous()
        ws = w[:g * C].contiguous()
        orders = nat.pack_orders(ORDERS[:g])
        for flags in flag_sets:
            what = f"{tag} flags {flags}"
            if in_place:
                buf, view = guarded(tuple(zs.shape), off)
                view.copy_(zs)
                expect_one(lambda: nat.inverse(view, ws, g, orders, flags=flags, out=view), key, what)
            else:
                src = offset_copy(zs, off) if off else zs
                buf, view = guarded(tuple(zs.shape), off)
                expect_one(lambda: nat.inverse(src, ws, g, orders, flags=flags, out=view), key, what)
            check_guarded(buf, view, off, what)
            shared.append((what, view[:3, :2 * C].clone()))
            if tag == "big":
                back = view
    base_what, base = shared[0]
    for what, o in shared[1:]:
        assert torch.equal(o, base[:o.shape[0]]), f"{what} differs from {base_what}"
    assert float((back - x).abs().max()) <= 1e-4, "inverse(forward(x)) != x"
    sel = torch.cat([z[:3], z[-3:]])
    want = torch.from_numpy(fo.inverse(npy(sel), npy(w), ORDERS)).cuda()
    got = torch.cat([back[:3], back[-3:]])
    assert rel64(got, want) <= 1e-5 and close64(got, want)


def test_inverse_warp_gsplit_grid(nat):
    """C = 32, k = 3, G = 4 runs one group per grid row (grid.y == G): its weights do not fit twice in the budget"""
    w, x, z = _warp_data(32, (3, 3), 8, 8, 64)
    assert warp_plan(64, G, 32, 8, 8, 3, 3)["gsplit"] == 1
    dims = launch_dims(lambda: nat.inverse(z, w, flags=nat.FLAG_GENERIC_TILED), "inverse_warp_kernel")
    if dims is None:
        pytest.skip("the profiler trace carries no launch dimensions")
    assert len(dims) == 1 and dims[0][0][1] == G, dims


def test_inverse_warp_refuses_7x7_at_32_channels(nat):
    """C = 32, k = 7: 49 * 32 * 32 floats of weights per group (200 KB) are over half the shared-memory budget, so
    even one group per CTA is refused and the generic inverse_naive_kernel<false> runs; it matches the oracle"""
    assert warp_plan(2, G, 32, 8, 8, 7, 7) is None
    w, x, z = _warp_data(32, (7, 7), 8, 8, 2)
    got = expect_one(lambda: nat.inverse(z, w), ("inverse_naive", (0,)))
    want = fo.inverse(npy(z), npy(w), ORDERS)
    assert float((got - x).abs().max()) <= 1e-4
    assert rel64(got, torch.from_numpy(want).cuda()) <= 1e-5


# ================================================================================================================
# slogdet_inverse_kernel (finc_affine.cu)
# ================================================================================================================
SLOGDET_C = (1, 2, 3, 5, 31, 32, 33, 64, 65, 77, 78, 96, 127, 128)


def _slogdet_batch(C, n, seed):
    """n well-conditioned matrices (random orthogonal x diag(exp(0.3 N))), of them: rows rotated by C/2 (pivots from
    another warp's rows once C > 64), entries of equal magnitude (Hadamard-like sign patterns: ties), negative
    determinants, and scales 1e-3 and 1e3"""
    g = torch.Generator().manual_seed(seed)
    q, _ = torch.linalg.qr(torch.randn(n, C, C, generator=g, dtype=torch.float64))
    m = q * torch.exp(0.3 * torch.randn(n, 1, C, generator=g, dtype=torch.float64))
    k = max(1, n // 8)
    dom = torch.eye(C, dtype=torch.float64) * 4 + 0.1 * torch.randn(k, C, C, generator=g, dtype=torch.float64)
    m[:k] = dom.roll(C // 2, dims=1)          # diagonally dominant, rows rotated: pivot of column j at row j + C/2
    if C & (C - 1) == 0:                       # Sylvester-Hadamard: every candidate pivot ties in magnitude
        h = torch.ones(1, 1, dtype=torch.float64)
        while h.shape[0] < C:
            h = torch.cat([torch.cat([h, h], 1), torch.cat([h, -h], 1)], 0)
        m[k:2 * k] = h
    m[2 * k:3 * k, 0] *= -1                    # negative determinants
    m[3 * k:4 * k] *= 1e3
    m[4 * k:5 * k] *= 1e-3
    return m


@pytest.mark.parametrize("C", SLOGDET_C)
def test_slogdet_inverse(nat, C):
    """log|det W| within 4e-6 * C (+1e-6 relative) of float64 and W W^-1 within 2e-4 of I, up to C = 128, including
    the opt-in shared-memory path (C >= 78); C = 129 is refused"""
    n = 2000 if C <= 33 else 300
    m64 = _slogdet_batch(C, n, C)
    W = m64.float().cuda()
    ld, Wi = expect_one(lambda: nat.slogdet_inverse(W), ("slogdet_inverse", ()))
    want = torch.linalg.slogdet(W.double())[1]
    err = (ld.double() - want).abs()
    assert bool((err <= 4e-6 * C + 1e-6 * want.abs()).all()), float(err.max())
    eye = torch.eye(C, dtype=torch.float64, device="cuda")
    res = float((W.double() @ Wi.double() - eye).abs().max())   # the matrices have condition numbers below ~10
    assert res <= 2e-4, res


def test_slogdet_inverse_rejects_129(nat):
    with pytest.raises(nat.FincNativeError):
        nat.slogdet_inverse(torch.eye(129, device="cuda").unsqueeze(0))


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two CUDA devices")
def test_slogdet_inverse_large_c_on_two_devices(nat):
    """the opt-in shared-memory limit (C >= 78) is raised per device: a call on a second device after one on the
    first still launches"""
    m = _slogdet_batch(96, 16, 5).float()
    for dev in ("cuda:0", "cuda:1"):
        W = m.to(dev)
        ld, Wi = nat.slogdet_inverse(W)
        want = torch.linalg.slogdet(W.double())[1]
        assert float((ld.double() - want).abs().max()) <= 4e-6 * 96 + 1e-6 * float(want.abs().max())


# ================================================================================================================
# preprocess_kernel (finc_affine.cu)
# ================================================================================================================
PRE_D = (1, 255, 256, 257, 784, 3072, 12288)


def preprocess_ref(x, u, alpha):
    s = 1.0 - 2.0 * alpha
    p = ((x.double() + u.double()) / 256.0 + alpha) * s
    lp, lq = torch.log(p), torch.log1p(-p)
    D = x[0].numel()
    return lp - lq, (-lp - lq).flatten(1).sum(1) + D * (math.log(s) - math.log(256.0)), p, (lp.abs() + lq.abs())


@pytest.mark.parametrize("D", PRE_D)
def test_preprocess(nat, D):
    """y = logit(((x + u) / 256 + alpha)(1 - 2 alpha)) element-wise within 4 eps/(1-p) + 4 eps (|log p| + |log(1-p)|)
    of float64 (the conditioning of the fp32 formula as p -> 1) and the log-det within 1e-6 of the sum of the
    magnitudes of its terms plus the sum of those bounds; noise None gives the bits of zero noise; without log-det,
    the same y"""
    for B in (1, 37):
        for alpha in (1e-6, 0.05):
            g = _gen(D + B)
            x = torch.randint(0, 256, (B, D), device="cuda", generator=g).float()
            x[0, 0] = 255.0
            u = torch.rand(B, D, device="cuda", generator=g)
            u[0, 0] = 0.999
            (y, ld) = expect_one(lambda: nat.preprocess(x, u, alpha), ("preprocess", ()))
            y64, ld64, p, mag = preprocess_ref(x, u, alpha)
            bound = 4 * EPS32 / (1 - p) + 4 * EPS32 * mag
            assert bool(((y.double() - y64).abs() <= bound).all()), (B, alpha, float((y.double() - y64).abs().max()))
            # the log-det sums the same ill-conditioned log(1 - p) terms: their bounds add up
            terms = mag.flatten(1).sum(1) + D * abs(math.log(1 - 2 * alpha) - math.log(256.0))
            ld_err = (ld.double() - ld64).abs()
            assert bool((ld_err <= 1e-6 * terms + bound.flatten(1).sum(1)).all()), (B, alpha, float(ld_err.max()))
            y0, ld0 = nat.preprocess(x, None, alpha)
            yz, ldz = nat.preprocess(x, torch.zeros_like(u), alpha)
            assert torch.equal(y0, yz) and torch.equal(ld0, ldz)
            yn, none = nat.preprocess(x, u, alpha, want_logdet=False)
            assert none is None and torch.equal(yn, y)


@pytest.mark.parametrize("alpha", (1e-6, 0.05, 0.25))
def test_preprocess_reverse_returns_every_integer(nat, alpha):
    x = torch.arange(256, device="cuda", dtype=torch.float32).repeat(3, 1)
    for u in (0.25, 0.5, 0.75):
        y, _ = nat.preprocess(x, torch.full_like(x, u), alpha)
        back = expect_one(lambda: nat.preprocess(y, alpha=alpha, reverse=True)[0], ("preprocess", ()))
        assert torch.equal(back, x), (u, int((back != x).sum()))


# ================================================================================================================
# gaussian_logp_kernel (finc_naive.cu)
# ================================================================================================================
G_CAP = 148 * 8   # launch_gaussian_logp's grid cap: each CTA loops over images beyond it


@pytest.mark.parametrize("D", (1, 31, 3072, 12288))
def test_gaussian_logp(nat, D):
    """logp = -|z|^2 / 2 - D log(2 pi) / 2 + logdet within 1e-6 of the magnitude of its terms; dz is exactly
    float32(dz_scale) * z; batches below, at and above the grid cap"""
    for B in (1, 7, G_CAP, G_CAP + 1, 3001):
        g = _gen(B * 7 + D)
        z = torch.randn(B, D, device="cuda", generator=g)
        for with_ld in (False, True):
            ld = 100 * torch.randn(B, device="cuda", generator=g) if with_ld else None
            scale = -1.0 / (3 * D)
            logp, dz = expect_one(lambda: nat.gaussian_logp(z, ld, dz_scale=scale), ("gaussian_logp", ()))
            sq = z.double().pow(2).sum(1)
            want = -0.5 * sq - 0.5 * D * math.log(2 * math.pi) + (ld.double() if with_ld else 0)
            mag = 0.5 * sq + 0.5 * D * math.log(2 * math.pi) + (ld.double().abs() if with_ld else 0)
            assert bool(((logp.double() - want).abs() <= 1e-6 * mag).all()), (B, D, with_ld)
            assert torch.equal(dz, z * torch.tensor(scale, dtype=torch.float32, device="cuda"))
            logp2, none = nat.gaussian_logp(z, ld)
            assert none is None and torch.equal(logp2, logp)


# ================================================================================================================
# logdet_kernel, mask_kernel (finc_naive.cu)
# ================================================================================================================
def _corner(o, k):
    """the stored position of the corner tap of a group of order `o` (fo.init_weight: (-1, -1), flipped per order)"""
    return (0 if o & 2 else k[0] - 1), (0 if o & 1 else k[1] - 1)


def _corner_diag(w, Gn, C, k, orders):
    return np.array([w[g * C + c, c][_corner(orders[g], k)] for g in range(Gn) for c in range(C)], dtype=np.float64)


def _random_diag_weight(Gn, C, k, seed, orders):
    """a FInC weight with corner-tap diagonals of random magnitude and sign"""
    rng = np.random.default_rng(seed)
    w = fo.init_unit_weight(C, k, rng, orders=orders)
    for g, o in enumerate(orders):
        d = rng.uniform(0.3, 3.0, C) * rng.choice([-1.0, 1.0], C)
        for c in range(C):
            w[(g * C + c, c) + _corner(o, k)] = d[c]
    return w


@pytest.mark.parametrize("Gn,C", [(4, 3), (4, 80), (16, 20)])
def test_logdet_kernel(nat, Gn, C):
    """finc_logdet_f32 and the generic forward with FINC_FLAG_LOGDET_ACCUMULATE against fo.logdet, at B > 256 and
    G * C up to 320 (more than one value per thread), non-unit and negative diagonals"""
    rng = np.random.default_rng(C)
    orders = tuple(int(o) for o in rng.integers(0, 4, Gn))
    k = (3, 3)
    w = _random_diag_weight(Gn, C, k, C + Gn, orders)
    H, W, B = 3, 5, 300
    want = fo.logdet(w, H, W, orders)
    wd = torch.from_numpy(w).cuda()
    packed = nat.pack_orders(orders)
    got = expect_one(lambda: nat.logdet(wd, B, H, W, Gn, packed), ("logdet", ()))
    mag = H * W * float(np.abs(np.log(np.abs(_corner_diag(w, Gn, C, k, orders)))).sum())
    assert float((got.double() - want).abs().max()) <= 1e-6 * mag, (float(got[0]), want)
    assert bool((got == got[0]).all())
    x = torch.randn(B, Gn * C, H, W, device="cuda", generator=_gen(C))
    acc0 = torch.randn(B, device="cuda")
    acc = acc0.clone()
    _, ran = glue_launched(lambda: nat.forward(x, wd, Gn, packed, True, nat.FLAG_NAIVE | nat.FLAG_LOGDET_ACCUMULATE,
                                               logdet_out=acc))
    assert ran == {("conv_naive", ()), ("logdet", ())}, ran
    assert torch.equal(acc, acc0 + got)


@pytest.mark.parametrize("k", [(1, 3), (2, 2), (3, 3), (5, 5), (3, 5)], ids=lambda k: f"{k[0]}x{k[1]}")
def test_apply_grad_mask(nat, k):
    """masked entries (corner tap, i >= o) become exactly +0, every other entry keeps its bits; G = 1 .. 16 with
    random orders, G * C * C > 256"""
    rng = np.random.default_rng(k[0] * 10 + k[1])
    for Gn, C in ((1, 17), (2, 12), (5, 8), (16, 5), (16, 1)):
        orders = tuple(int(o) for o in rng.integers(0, 4, Gn))
        dw = torch.randn(Gn * C, C, *k, device="cuda", generator=_gen(Gn * C))
        dw[dw.abs() < 0.1] = -0.0
        before = dw.clone()
        expect_one(lambda: nat.apply_grad_mask_(dw, Gn, nat.pack_orders(orders)), ("mask", ()))
        masked = torch.from_numpy(fo.apply_grad_mask(np.ones(tuple(dw.shape), np.float32), orders) == 0).cuda()
        assert int(masked.sum()) == Gn * C * (C + 1) // 2
        got = dw.cpu().numpy()
        m = masked.cpu().numpy()
        assert (got[m] == 0).all() and not np.signbit(got[m]).any()
        assert torch.equal(dw[~masked].view(torch.int32), before[~masked].view(torch.int32))


# ================================================================================================================
# the generic kernels under FINC_FLAG_NAIVE (finc_naive.cu)
# ================================================================================================================
NAIVE_CASES = [(3, (3, 3), 7, 9), (5, (2, 3), 6, 5), (2, (5, 5), 8, 8)]


@pytest.mark.parametrize("case", NAIVE_CASES, ids=lambda c: f"C{c[0]}_k{c[1][0]}x{c[1][1]}")
def test_naive_kernels(nat, case):
    """forward, backward-input, inverse, adjoint and weight gradient (masked, NO_MASK, NEGATE, ACCUMULATE, B = 0)
    through the generic kernels against the oracle"""
    C, k, H, W = case
    rng = np.random.default_rng(C)
    w = fo.init_unit_weight(C, k, rng)
    B = 3
    x = rng.standard_normal((B, G * C, H, W)).astype(np.float32)
    dz = rng.standard_normal((B, G * C, H, W)).astype(np.float32)
    wd, xd, dzd = (torch.from_numpy(a).cuda() for a in (w, x, dz))
    N = nat.FLAG_NAIVE
    z, _ = expect_one(lambda: nat.forward(xd, wd, flags=N, want_logdet=False), ("conv_naive", ()))
    want = fo.forward(x, w, ORDERS)
    assert rel64(z, torch.from_numpy(want).cuda()) <= 1e-5
    dx = expect_one(lambda: nat.backward_input(dzd, wd, flags=N), ("conv_naive", ()))
    assert rel64(dx, torch.from_numpy(fo.backward_input(dz, w, ORDERS)).cuda()) <= 1e-5
    zf = torch.from_numpy(want.astype(np.float32)).cuda()
    xi = expect_one(lambda: nat.inverse(zf, wd, flags=N), ("inverse_naive", (0,)))
    assert rel64(xi, torch.from_numpy(fo.inverse(npy(zf), w, ORDERS)).cuda()) <= 1e-5
    assert float((xi - xd).abs().max()) <= 1e-4
    adj = expect_one(lambda: nat.inverse_adjoint(dzd, wd, flags=N), ("inverse_naive", (1,)))
    assert rel64(adj, torch.from_numpy(adjoint_oracle(dz.astype(np.float64), w, ORDERS)).cuda()) <= 1e-5
    masked_ref = fo.backward_weight(dz, x, k, ORDERS)
    raw_ref = fo.backward_weight(dz, x, k, ORDERS, apply_mask=False)
    dw = expect_one(lambda: nat.backward_weight(dzd, xd, k, flags=N), ("wgrad_naive", ()))
    assert rel64(dw, torch.from_numpy(masked_ref).cuda()) <= 1e-5
    masked = fo.apply_grad_mask(np.ones(w.shape, np.float32), ORDERS) == 0
    d = dw.cpu().numpy()
    assert (d[masked] == 0).all() and not np.signbit(d[masked]).any()
    raw = nat.backward_weight(dzd, xd, k, flags=N | nat.FLAG_NO_MASK)
    assert rel64(raw, torch.from_numpy(raw_ref).cuda()) <= 1e-5
    neg = nat.backward_weight(dzd, xd, k, flags=N | nat.FLAG_NEGATE)
    assert torch.equal(neg, -dw)   # masked entries stay +0: 0 is not negated
    old = torch.randn(dw.shape, device="cuda")
    acc = old.clone()
    nat.backward_weight(dzd, xd, k, flags=N | nat.FLAG_ACCUMULATE, out=acc)
    assert torch.equal(acc, old + dw)
    e = torch.empty(0, G * C, H, W, device="cuda")
    zeros = expect_one(lambda: nat.backward_weight(e, e, k, flags=N, out=torch.full_like(dw, 7.0)), ("wgrad_naive", ()))
    assert not bool(zeros.any())
    acc = old.clone()
    nat.backward_weight(e, e, k, flags=N | nat.FLAG_ACCUMULATE, out=acc)
    assert torch.equal(acc, old)


# ================================================================================================================
# census-only recipes: kernels value-checked elsewhere (test_gpu_tc*.py, test_gpu_stack.py, test_gpu_flow.py, ...)
# ================================================================================================================
def _census_coupling(nat):
    from test_gpu_tc_variants import LOGSCALE

    C, width, B, H, W = 12, 128, 2, 8, 8
    g = torch.Generator().manual_seed(3)
    ci = C // 2
    p = [torch.randn(width, ci, 3, 3, generator=g) / (9 * ci) ** 0.5, 0.1 * torch.randn(width, generator=g),
         torch.randn(width, width, 1, 1, generator=g) / width ** 0.5, 0.1 * torch.randn(width, generator=g),
         0.5 * torch.randn(C, width, 3, 3, generator=g) / (9 * width) ** 0.5, 0.1 * torch.randn(C, generator=g),
         0.1 * torch.randn(C, generator=g)]
    p = [t.cuda() for t in p]
    x = torch.randn(B, C, H, W, generator=g).cuda()
    blob = nat.coupling_prepare(*p, LOGSCALE, with_backward=True)
    ws = torch.empty(nat.coupling_workspace_bytes(B, C, H, W, width), dtype=torch.uint8, device="cuda")
    y, _ = nat.coupling_apply(x, blob, width, workspace=ws)
    nat.coupling_backward(x, torch.randn_like(x), torch.randn(B, device="cuda"), blob, ws, width)
    ws2 = torch.empty_like(ws)
    nat.coupling_apply(y, blob, width, reverse=True, want_logdet=True, workspace=ws2)
    nat.coupling_backward(y, torch.randn_like(x), torch.randn(B, device="cuda"), blob, ws2, width,
                          flags=nat.FLAG_COUPLING_REVERSE)


def _census_dense(nat):
    w = torch.from_numpy(fo.init_unit_weight(4, (3, 3), np.random.default_rng(0))).cuda()
    nat.inverse_dense_prepare(w, 4, 4)


def _census_tc_wgrad(nat):
    P = torch.randn(20000, 64, device="cuda", generator=_gen(1))
    nat.tc_wgrad(P, torch.randn(20000, 64, device="cuda", generator=_gen(2)))


def _census_prepare(nat):
    w = torch.stack([torch.from_numpy(fo.init_unit_weight(3, (3, 3), np.random.default_rng(u))) for u in range(2)])
    w = w.cuda().contiguous()
    for kind in (nat.PREP_FORWARD, nat.PREP_BACKWARD_INPUT, nat.PREP_INVERSE):
        nb = nat.prepared_weights_bytes(kind, 8, G, 3, 16, 16, 3, 3)
        assert nb > 0, kind
        nat.prepare_weights(w, torch.empty((2, nb), dtype=torch.uint8, device="cuda"), kind, 8, 16, 16)


def _census_inverse_multi(nat):
    from test_gpu_inverse_multi import CIFAR, _level

    levels = []
    for i, (C, H, W) in enumerate(CIFAR):
        z, t = _level(8, C, H, W, 2, i)
        levels.append((z, t, (3, 3), range(1, -1, -1), None))
    nat.inverse_chain_multi(levels)


def _census_squeeze_adam(nat):
    x = torch.randn(2, 3, 8, 8, device="cuda")
    nat.unsqueeze(nat.squeeze(x))
    n = 1000
    nat.adam_step_(torch.randn(n, device="cuda"), torch.randn(n, device="cuda"), torch.zeros(n, device="cuda"),
                   torch.zeros(n, device="cuda"), torch.zeros(1, device="cuda"))


CENSUS_ONLY = [_census_coupling, _census_dense, _census_tc_wgrad, _census_prepare, _census_inverse_multi,
               _census_squeeze_adam]


# ================================================================================================================
# census: every glue kernel in the library is launched by some recipe, or is listed in UNREACHABLE
# ================================================================================================================
def _census_value_recipes(nat):
    """one launch of each recipe of the value tests above, at their smallest shapes (each profiled on its own)"""
    out = []
    for C in AFFINE_C:
        A, b = _affine_params(C)
        for off, H, W in ((0, 16, 16), (2, 16, 16), (1, 16, 16)):
            vec = min(affine_vec(H, W, off), affine_vmax(C))
            x = _affine_images(C, affine_big_batch(C, H, W, vec), H, W)
            out.append(lambda x=x, A=A, b=b, off=off: nat.affine1x1(offset_copy(x, off), A, b,
                                                                    out=guarded(tuple(x.shape), off)[1]))
        out.append(lambda C=C, A=A, b=b: nat.affine1x1(torch.randn(1, C, 4, 4, device="cuda"), A, b))
    out.append(lambda: nat.affine1x1(torch.randn(1, 5, 4, 4, device="cuda"), *_affine_params(5)))
    for C in (4, 6):
        out.append(lambda C=C: nat.affine1x1_backward_weight(torch.randn(2, C, 8, 8, device="cuda"),
                                                             torch.randn(2, C, 8, 8, device="cuda")))
    for C, k, H, W, _ in WARP_CASES:
        if C in WARP_CP:
            w, _, z = _warp_data(C, k, H, W, 3)
            out.append(lambda z=z, w=w: nat.inverse(z, w, flags=nat.FLAG_GENERIC_TILED))
    out.append(lambda: nat.slogdet_inverse(torch.eye(5, device="cuda").expand(3, 5, 5).contiguous()))
    out.append(lambda: nat.preprocess(torch.zeros(2, 10, device="cuda")))
    out.append(lambda: nat.gaussian_logp(torch.randn(2, 10, device="cuda"), dz_scale=1.0))
    w3 = torch.from_numpy(fo.init_unit_weight(3, (3, 3), np.random.default_rng(1))).cuda()
    x3 = torch.randn(2, 12, 5, 5, device="cuda")
    out.append(lambda: nat.logdet(w3, 2, 5, 5))
    out.append(lambda: nat.apply_grad_mask_(torch.randn(12, 3, 3, 3, device="cuda"), G, nat.ORDERS_UNIT))
    out.append(lambda: nat.forward(x3, w3, flags=nat.FLAG_NAIVE))
    out.append(lambda: nat.inverse(x3, w3, flags=nat.FLAG_NAIVE))
    out.append(lambda: nat.inverse_adjoint(x3, w3, flags=nat.FLAG_NAIVE))
    out.append(lambda: nat.backward_weight(x3, x3, (3, 3), flags=nat.FLAG_NAIVE))
    return out


def test_every_glue_kernel_is_exercised(nat):
    compiled = {e for e in kernels_in(library_kernels(), GLUE_FAMILIES)}
    assert {f for f, _ in compiled} == set(GLUE_FAMILIES), "a glue kernel family is missing from the symbol table"
    observed = set()
    for fn in _census_value_recipes(nat) + [functools.partial(f, nat) for f in CENSUS_ONLY]:
        observed |= glue_launched(fn)[1]
    unreachable = set(UNREACHABLE)
    print(f"\n[glue census] compiled {len(compiled)}, observed {len(observed & compiled)}, "
          f"unreachable {len(unreachable)}")
    assert unreachable <= compiled, unreachable - compiled
    assert not (observed & unreachable), observed & unreachable
    assert observed <= compiled, f"kernels ran that the symbol table does not list: {observed - compiled}"
    missing = compiled - unreachable - observed
    assert not missing, f"compiled but reached by no recipe: {sorted(missing)}"
    assert len(observed) + len(unreachable) == len(compiled)
