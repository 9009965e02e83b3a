"""Every compiled instantiation of the FInC kernel templates against the float64 oracle, with a census of the
kernels that actually ran.

The hot path is a family of template instantiations, and a host planner picks one per call from the shape, the
batch size and the pointer alignment:

    conv_cta_kernel<CT, OB, WT, KH, KW, RB>      forward and backward-input      (finc_conv.cu, finc_conv_c<N>.cu)
    wgrad_kernel<OB, WT, KH, KW>                 weight gradient                 (finc_wgrad.cu)
    inverse_rw_kernel<C, KH, KW, P, MT, ADJ>     inverse and its adjoint         (finc_inverse_rw*.cu)
    chain_kernel<CT, OB, WT>                     chains of units                 (finc_chain.cu)
    inverse_wave_kernel<C, KH, KW, P>            shared-memory wavefront inverse (finc_inverse_wave*.cu)

Each case below is a *recipe*: a shape, an output alignment and the per-call planner knobs (FINC_CONV_OB,
FINC_WG_FORCE, FINC_CHAIN_IPB, FINC_RW_P / _NSTK / _T / _S / _WARPS) that reach one instantiation.  Every value a
recipe forces is one the planner itself could choose.  Each launch runs under torch.profiler and the test asserts
that exactly the intended instantiation ran: a forced plan the host refuses falls back to another kernel, and that
must fail, not pass by accident.  test_every_compiled_instantiation_is_exercised lists the instantiations compiled
into the library (its symbol table) and requires every one of them to be reached by some recipe, except those in
UNREACHABLE, each with the reason the planner can never select it.
"""
import functools
import math
import re
import subprocess

import numpy as np
import pytest
import torch

from conftest import elementwise_close, rel_err
from oracle import finc_oracle as fo
from test_gpu_inverse_grad import adjoint_oracle

pytestmark = pytest.mark.gpu

REL_TOL = 1e-5
RT_TOL = 1e-4
ORDERS = (0, 1, 2, 3)   # a FastFlowUnit: one group per padding corner
G = len(ORDERS)

# ---- kernel census ---------------------------------------------------------------------------------------------
# demangled names, e.g. `void finc::conv::conv_cta_kernel<12, 1, 2, 3, 3, 1>(finc::conv::ConvArgs)`
FAMILIES = {
    "conv": "finc::conv::conv_cta_kernel",
    "wgrad": "finc::(anonymous namespace)::wgrad_kernel",
    "inverse_rw": "finc::rw::inverse_rw_kernel",
    "chain": "finc::chain::chain_kernel",
    "inverse_wave": "finc::wave::inverse_wave_kernel",
}

# compiled instantiations the planners can never select, with the reason (from the code)
UNREACHABLE = {
    ("wgrad", (1, 2, 5, 5)): "dispatched, but make_plan (finc_wgrad.cu) takes WT = 2 only when kW - 1 <= 2",
    ("wgrad", (2, 2, 5, 5)): "dispatched, but make_plan (finc_wgrad.cu) takes WT = 2 only when kW - 1 <= 2",
}


def _arg(v):
    v = " ".join(v.split())
    if v in ("true", "false"):
        return int(v == "true")
    return int(v) if re.fullmatch(r"-?\d+", v) else v   # a type argument stays a string


def _template_args(s):
    """the arguments of the template argument list `s` starts with ("<...>", nesting allowed) and its length"""
    depth, args, start = 0, [], 1
    for i, ch in enumerate(s):
        if ch == "<":
            depth += 1
        elif ch == ">":
            depth -= 1
            if depth == 0:
                args.append(s[start:i])
                return tuple(_arg(a) for a in args), i + 1
        elif ch == "," and depth == 1:
            args.append(s[start:i])
            start = i + 1
    raise ValueError(f"unbalanced template arguments in {s!r}")


def kernels_in(names, families=FAMILIES):
    """{(family, template arguments)} of the kernel families in `families` (name -> qualified kernel name, by
    default the five FInC families) among kernel names.  Bools read as 0 / 1 and type arguments as strings; a
    kernel that is not a template (its name followed by its parameter list, or an unmangled extern "C" name alone)
    has the arguments ()."""
    pattern = re.compile(r"(?<![\w:])(" + "|".join(re.escape(p) for p in families.values()) + r")(?=[<(]|$)")
    family_of = {p: f for f, p in families.items()}
    found = set()
    for name in names:
        for m in pattern.finditer(name):
            rest = name[m.end():]
            args = _template_args(rest)[0] if rest.startswith("<") else ()
            found.add((family_of[m.group(1)], args))
    return found


def launched(fn, families=FAMILIES):
    """(fn(), the set of kernel instantiations of `families` it launched)"""
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    # a PyTorch kernel first: when the session opens with a new CUPTI activity buffer ("Activity Buffer Request"), a
    # CUDA-only profile of a lone kernel was seen to lose that kernel's record; with CPU activities and a warm-up
    # kernel ahead of it, it was recorded
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        torch.zeros(1, device="cuda").add_(1)
        torch.cuda.synchronize()
        out = fn()
        torch.cuda.synchronize()
    return out, kernels_in((e.key for e in prof.key_averages()), families)


def compiled_instantiations(families=FAMILIES):
    """the instantiations of `families` in the library's symbol table (their host stubs)"""
    from fincflow_b200 import _native

    syms = subprocess.run(["nm", "-C", _native.LIB_PATH], capture_output=True, text=True, check=True).stdout
    return kernels_in(syms.splitlines(), families)


@pytest.fixture(scope="module")
def nat():
    from fincflow_b200 import _native

    _native.load()
    return _native


def npy(t):
    return t.detach().double().cpu().numpy()


def _sms():
    from fincflow_b200 import _native

    return _native.sm_count()


# ---- sentinel-guarded outputs ------------------------------------------------------------------------------------
GUARD, SENT = 4096, 12345.678


def guarded(shape, offset=0):
    """(buffer, view): `shape` inside a sentinel-filled buffer, `offset` floats past a 16-byte boundary"""
    n = math.prod(shape)
    buf = torch.full((n + 2 * GUARD + 4,), SENT, device="cuda")
    return buf, buf[GUARD + offset:GUARD + offset + n].view(shape)


def check_guarded(buf, view, offset, what):
    n = view.numel()
    torch.cuda.synchronize()
    assert bool((buf[:GUARD + offset] == SENT).all()), what + ": write before the output"
    assert bool((buf[GUARD + offset + n:] == SENT).all()), what + ": write past the output"
    assert not bool((view == SENT).any()), what + ": output left unwritten"


def set_knobs(mp, knobs, names):
    for k in names:
        mp.delenv(k, raising=False)
    for k, v in knobs.items():
        mp.setenv(k, str(v))


class Recipe:
    """one instantiation and how to reach it: `knobs` (environment, read per call) and `launch(nat, inputs)`"""

    def __init__(self, family, args, knobs, make, launch, id_, **meta):
        self.expect = (family, tuple(args))
        self.knobs, self.make, self.launch, self.id, self.meta = knobs, make, launch, id_, meta

    def __repr__(self):
        return self.id


def unit_weight(C, k, seed, diag=None):
    """[G*C, C, k, k] FastFlowUnit weight (numpy); `diag` replaces the corner-tap diagonal of group 0, channel 0"""
    w = fo.init_unit_weight(C, (k, k), np.random.default_rng(seed))
    if diag is not None:
        w[0, 0, k - 1, k - 1] = diag   # group 0 pads top-left: its corner tap is (k-1, k-1)
    return w


@functools.lru_cache(maxsize=None)
def _inputs(B, C, H, W, k, seed, diag=None):
    """device inputs of one shape (cached: the census and the variant tests share them)"""
    g = torch.Generator().manual_seed(seed)
    w = unit_weight(C, k, seed, diag)
    x = torch.randn(B, G * C, H, W, generator=g)
    dz = torch.randn(B, G * C, H, W, generator=g)
    return {"w": torch.from_numpy(w).cuda(), "x": x.cuda(), "dz": dz.cuda()}


# ================================================================================================================
# inverse_rw_kernel<C, K, K, P, MT, ADJ>
# ================================================================================================================
RW_KNOBS = ("FINC_RW_P", "FINC_RW_NSTK", "FINC_RW_T", "FINC_RW_S", "FINC_RW_WARPS")
# every compiled (C, k, P) family with a tile it covers (P * WP <= 32, WP = the power of two >= W)
RW_FAMILIES = [  # C, k, P, H, W
    (1, 3, 1, 16, 16), (2, 3, 1, 14, 14), (3, 3, 1, 16, 16), (4, 3, 1, 14, 14), (4, 3, 2, 14, 14),
    (6, 3, 1, 8, 8), (6, 3, 2, 7, 7), (12, 3, 1, 8, 8), (12, 3, 4, 8, 8),
    (1, 5, 1, 12, 12), (2, 5, 1, 16, 16), (3, 5, 1, 10, 10), (4, 5, 2, 14, 14), (6, 5, 2, 8, 8), (12, 5, 4, 6, 6),
]
RW_B = 37   # not a multiple of NSTK * T for any forced NSTK * T > 1


def _wp(W):
    wp = 4
    while wp < W:
        wp *= 2
    return wp


def rw_schedules(P, W):
    """scheduling knobs to sweep for one (C, k, P): stacks per warp, tiles per stack (T > 1 runs the MT
    instantiation), pipeline stages and warps per CTA.  The first entry is the planner's own choice."""
    nmax = 32 // (_wp(W) * P)
    return [
        {},
        {"FINC_RW_NSTK": 1, "FINC_RW_T": 1, "FINC_RW_S": 1, "FINC_RW_WARPS": 1},
        {"FINC_RW_NSTK": nmax, "FINC_RW_T": 1, "FINC_RW_S": 2, "FINC_RW_WARPS": 2},
        {"FINC_RW_NSTK": nmax, "FINC_RW_T": 2, "FINC_RW_S": 2, "FINC_RW_WARPS": 2},
        {"FINC_RW_NSTK": max(1, nmax // 2), "FINC_RW_T": 4, "FINC_RW_S": 1, "FINC_RW_WARPS": 8},
        {"FINC_RW_NSTK": 1, "FINC_RW_T": 8, "FINC_RW_S": 2, "FINC_RW_WARPS": 3},
    ]


def _rw_make(B, C, H, W, k):
    def make():
        d = _inputs(B, C, H, W, k, 1000 * C + 10 * k + H)
        w = d["w"]
        z = _z_of(B, C, H, W, k)
        return {"w": w, "z": z, "dx": d["dz"]}
    return make


@functools.lru_cache(maxsize=None)
def _z_of(B, C, H, W, k):
    """z = forward(x) in float64, rounded to float32: inverse(z) must give back x"""
    d = _inputs(B, C, H, W, k, 1000 * C + 10 * k + H)
    return torch.from_numpy(fo.forward(npy(d["x"]), npy(d["w"]), ORDERS).astype(np.float32)).cuda()


def _rw_launch(adj, offset):
    def launch(nat, inp, out=None):
        src = inp["dx"] if adj else inp["z"]
        if offset:   # input and output 4 bytes past a 16-byte boundary: no TMA bulk copies
            sbuf = torch.empty(src.numel() + 4, device="cuda")
            src = sbuf[offset:offset + src.numel()].view_as(src)
            src.copy_(inp["dx"] if adj else inp["z"])
        if out is None:
            out = guarded(tuple(src.shape), offset)[1]
        fn = nat.inverse_adjoint if adj else nat.inverse
        return fn(src, inp["w"], G, nat.ORDERS_UNIT, out=out)
    return launch


def rw_recipes():
    out = []
    for C, k, P, H, W in RW_FAMILIES:
        for adj in (0, 1):
            tag = f"{'adj' if adj else 'inv'}_C{C}_k{k}_P{P}_{H}x{W}"
            for i, sched in enumerate(rw_schedules(P, W)):
                mt = int(sched.get("FINC_RW_T", 1) > 1)
                out.append(Recipe("inverse_rw", (C, k, k, P, mt, adj), {"FINC_RW_P": P, **sched},
                                  _rw_make(RW_B, C, H, W, k), _rw_launch(adj, 0), f"{tag}_s{i}",
                                  fam=(C, k, P, H, W), adj=adj, sched=i, offset=0))
            out.append(Recipe("inverse_rw", (C, k, k, P, 0, adj), {"FINC_RW_P": P}, _rw_make(RW_B, C, H, W, k),
                              _rw_launch(adj, 1), f"{tag}_unaligned", fam=(C, k, P, H, W), adj=adj, sched=-1, offset=1))
    return out


RW_RECIPES = rw_recipes()


def _rw_group(C, k, P, H, W, adj):
    return [r for r in RW_RECIPES if r.meta["fam"] == (C, k, P, H, W) and r.meta["adj"] == adj]


@pytest.mark.parametrize("adj", [0, 1], ids=["inverse", "adjoint"])
@pytest.mark.parametrize("fam", RW_FAMILIES, ids=lambda f: "C{}_k{}_P{}_{}x{}".format(*f))
def test_inverse_rw_variants(nat, monkeypatch, fam, adj):
    """one (C, k, P) family, as inverse or adjoint, over its scheduling parameters (NSTK, T, S, WARPS; T > 1 is the
    multi-tile MT instantiation) and once unaligned: every schedule is the intended instantiation, writes exactly
    its output, and gives the same bits (the per-pixel arithmetic depends only on P), which match the float64
    oracle and invert the forward (or backward-input) map"""
    C, k, P, H, W = fam
    outs = []
    for r in _rw_group(C, k, P, H, W, adj):
        inp = r.make()
        set_knobs(monkeypatch, r.knobs, RW_KNOBS)
        off = r.meta["offset"]
        buf, view = guarded(tuple(inp["z"].shape), off)
        _, ran = launched(lambda: r.launch(nat, inp, out=view))
        assert ran == {r.expect}, (r.id, ran)
        check_guarded(buf, view, off, r.id)
        outs.append((r.id, view.clone()))
    set_knobs(monkeypatch, {}, RW_KNOBS)
    base_id, base = outs[0]
    for rid, o in outs[1:]:
        assert torch.equal(o, base), f"{rid} differs from {base_id}"
    inp = _rw_group(C, k, P, H, W, adj)[0].make()
    w = npy(inp["w"])
    if adj:
        want = adjoint_oracle(npy(inp["dx"]), w, ORDERS)
        back = nat.backward_input(base, inp["w"])           # A^T (A^-T dx) = dx
        assert float((back - inp["dx"]).abs().max()) <= RT_TOL
    else:
        want = fo.inverse(npy(inp["z"]), w, ORDERS)
        x = _inputs(RW_B, C, H, W, k, 1000 * C + 10 * k + H)["x"]
        assert float((base - x).abs().max()) <= RT_TOL        # inverse(forward(x)) = x
    assert rel_err(npy(base), want) <= REL_TOL
    assert elementwise_close(npy(base), want)


# planner-chosen variants at the batch sizes that select them (no knobs)
RW_NATURAL = [  # C, k, H, W, batch (None: 2 * SMs + 11), expected P
    (4, 3, 14, 14, None, 1),   # C = 4 picks P = 1 once B * G * WP / 32 >= 4 * SMs
    (6, 3, 20, 20, 37, 1),     # W > 16: P = 2 does not fit the warp
]


@pytest.mark.parametrize("adj", [0, 1], ids=["inverse", "adjoint"])
@pytest.mark.parametrize("case", RW_NATURAL, ids=lambda c: "C{}_k{}_{}x{}".format(*c[:4]))
def test_inverse_rw_planner_choices(nat, monkeypatch, case, adj):
    """shapes whose batch or width makes the planner itself pick a variant the rest of the suite does not reach;
    the oracle on the first and last images (the last item is the ragged one)"""
    C, k, H, W, B, P = case
    set_knobs(monkeypatch, {}, RW_KNOBS)
    B = B or 2 * _sms() + 11
    r = Recipe("inverse_rw", (C, k, k, P, 0, adj), {}, _rw_make(B, C, H, W, k), _rw_launch(adj, 0), "natural")
    inp = r.make()
    buf, view = guarded(tuple(inp["z"].shape))
    _, ran = launched(lambda: r.launch(nat, inp, out=view))
    assert ran == {r.expect}, ran
    check_guarded(buf, view, 0, "natural")
    src = inp["dx"] if adj else inp["z"]
    sel = torch.cat([src[:3], src[-3:]])
    got = torch.cat([view[:3], view[-3:]])
    want = adjoint_oracle(npy(sel), npy(inp["w"]), ORDERS) if adj else fo.inverse(npy(sel), npy(inp["w"]), ORDERS)
    assert rel_err(npy(got), want) <= REL_TOL and elementwise_close(npy(got), want)


# ================================================================================================================
# conv_cta_kernel<CT, OB, WT, K, K, RB>
# ================================================================================================================
CONV_KNOBS = ("FINC_CONV_OB",)
CONV_OBS = {1: [1], 2: [2, 1], 3: [3, 1], 4: [4, 2], 6: [6, 3, 2], 12: [4, 2, 1], 24: [4, 2, 1],
            0: [6, 4, 3, 2, 1]}     # output blocks instantiated per channel count (finc_conv_c<N>.cu; 0 = generic C)
CONV_HW = {1: 16, 2: 16, 3: 16, 4: 12, 6: 8, 12: 8, 24: 8, 0: 8}
CONV_GENERIC_C = 18   # not a specialised channel count, and every generic output block divides it (or pads: 4)
WT_OFFSET = {4: 0, 2: 2, 1: 1}   # output 16-, 8- or 4-byte aligned


def conv_variants():
    out = []
    for ct, obs in CONV_OBS.items():
        for ob in obs:
            for wt in ((4, 2, 1) if ct == 0 else (4, 2)):
                for k in ((2, 3, 5) if ct == 0 else (3, 5)):
                    out.append((ct, ob, wt, k, 1))
                    if 1 <= ct <= 3 and ob == ct and wt == 4 and k == 3:
                        out.append((ct, ob, wt, k, 2))
    return out


def _conv_recipe(v):
    ct, ob, wt, k, rb = v
    C = ct or CONV_GENERIC_C
    H = W = 32 if rb == 2 else CONV_HW[ct]

    def make():
        # RB = 2 (two output rows per sub-item) once spread * nob * H * nstrip >= 4 * 16 * 32, spread = B * G / SMs
        B = 2 * _sms() + 17 if rb == 2 else 9
        return _inputs(B, C, H, W, k, 7 * C + k + rb, diag=1.7)

    def launch(nat, inp, out=None, flags=0, logdet_out=None, transpose=False):
        if out is None:   # the output alignment selects WT
            out = guarded(tuple(inp["x"].shape), WT_OFFSET[wt])[1]
        if transpose:
            return nat.backward_input(inp["dz"], inp["w"], G, nat.ORDERS_UNIT, flags=flags, out=out)
        return nat.forward(inp["x"], inp["w"], G, nat.ORDERS_UNIT, True, flags, out=out, logdet_out=logdet_out)

    return Recipe("conv", (ct, ob, wt, k, k, rb), {"FINC_CONV_OB": ob}, make, launch,
                  f"CT{ct}_OB{ob}_WT{wt}_k{k}_RB{rb}", offset=WT_OFFSET[wt])


CONV_RECIPES = [_conv_recipe(v) for v in conv_variants()]


@pytest.mark.parametrize("r", CONV_RECIPES, ids=lambda r: r.id)
def test_conv_variant(nat, monkeypatch, r):
    """forward (+ logdet) and backward-input of one instantiation against the float64 oracle.

    conv_sub accumulates each output as fmaf(w, x, acc) over (input channel, kernel row, kernel column) in that
    order, starting from 0, whatever OB, WT and RB are (they only choose how many outputs a lane holds; padding
    reads +0 from the zero strip or a column predicate alike), so every variant is also bit-identical to the
    default plan of the same shape."""
    inp = r.make()
    off = r.meta["offset"]
    shape = tuple(inp["x"].shape)
    B, _, H, W = shape
    k = r.expect[1][3]
    set_knobs(monkeypatch, r.knobs, CONV_KNOBS)
    res = {}
    for tr in (False, True):
        buf, view = guarded(shape, off)
        _, ran = launched(lambda: r.launch(nat, inp, out=view, transpose=tr))
        assert ran == {r.expect}, (tr, ran)
        check_guarded(buf, view, off, f"{r.id} transpose={tr}")
        res[tr] = view.clone()
    ld = r.launch(nat, inp)[1]
    # determinism, the half-GPU plan and the logdet accumulator: same instantiation, same bits
    again = r.launch(nat, inp)[0]
    assert torch.equal(again, res[False])
    (half, _), ran = launched(lambda: r.launch(nat, inp, flags=nat.FLAG_HALF_GPU))
    assert ran == {r.expect}, ran
    assert torch.equal(half, res[False])
    acc0 = torch.randn(B, device="cuda")
    acc = acc0.clone()
    r.launch(nat, inp, flags=nat.FLAG_LOGDET_ACCUMULATE, logdet_out=acc)
    assert torch.equal(acc, acc0 + ld)
    set_knobs(monkeypatch, {}, CONV_KNOBS)
    z_default, _ = nat.forward(inp["x"], inp["w"])
    assert torch.equal(res[False], z_default)
    assert torch.equal(res[True], nat.backward_input(inp["dz"], inp["w"]))
    w = npy(inp["w"])
    z_want = fo.forward(npy(inp["x"]), w, ORDERS)
    dx_want = fo.backward_input(npy(inp["dz"]), w, ORDERS)
    assert rel_err(npy(res[False]), z_want) <= REL_TOL and elementwise_close(npy(res[False]), z_want)
    assert rel_err(npy(res[True]), dx_want) <= REL_TOL and elementwise_close(npy(res[True]), dx_want)
    ld_want = fo.logdet(w, H, W, ORDERS)
    assert abs(ld_want - H * W * np.log(np.float32(1.7))) < 1e-9 * H * W
    assert rel_err(npy(ld), np.full(B, ld_want)) <= REL_TOL


# ================================================================================================================
# wgrad_kernel<OB, WT, K, K>
# ================================================================================================================
WG_KNOBS = ("FINC_WG_FORCE",)
WG_CASES = [  # OB, WT, k, C, B, Z, CH (0 = free).  WT = 4: 8x8 tiles, WT = 2: 6x6.  B = 1: one batch slice (X = 1)
    (1, 4, 3, 3, 1, 1, 0), (1, 4, 3, 3, 37, 2, 4), (1, 2, 3, 3, 1, 1, 0), (1, 2, 3, 3, 37, 2, 4),
    (2, 4, 3, 4, 1, 1, 0), (2, 4, 3, 4, 37, 2, 4), (2, 2, 3, 4, 1, 1, 0), (2, 2, 3, 4, 37, 2, 4),
    (3, 4, 3, 6, 1, 1, 0), (3, 4, 3, 6, 37, 2, 4), (3, 2, 3, 6, 1, 1, 0), (3, 2, 3, 6, 37, 2, 4),
    (4, 4, 3, 7, 1, 1, 0), (4, 4, 3, 10, 37, 2, 4), (4, 2, 3, 7, 1, 1, 0), (4, 2, 3, 10, 37, 2, 4),  # padded last block
    (6, 4, 3, 6, 1, 1, 0), (6, 4, 3, 12, 37, 2, 4), (6, 4, 3, 24, 37, 2, 0), (6, 2, 3, 6, 1, 1, 0), (6, 2, 3, 12, 37, 2, 4),
    (1, 4, 5, 2, 1, 1, 0), (1, 4, 5, 3, 37, 2, 4), (2, 4, 5, 2, 1, 1, 0), (2, 4, 5, 4, 37, 2, 4),
]


def _wg_recipe(case):
    ob, wt, k, C, B, z, ch = case
    H = W = 8 if wt == 4 else 6

    def make():
        return _inputs(B, C, H, W, k, 31 * C + B + k)

    def launch(nat, inp, out=None, flags=0, workspace=None):
        return nat.backward_weight(inp["dz"], inp["x"], (k, k), G, nat.ORDERS_UNIT, flags, out=out, workspace=workspace)

    return Recipe("wgrad", (ob, wt, k, k), {"FINC_WG_FORCE": f"{ob},{z},{ch}"}, make, launch,
                  f"OB{ob}_WT{wt}_k{k}_C{C}_B{B}_Z{z}_CH{ch}", ksize=k)


WG_RECIPES = [_wg_recipe(c) for c in WG_CASES]


@pytest.mark.parametrize("r", WG_RECIPES, ids=lambda r: r.id)
def test_wgrad_variant(nat, monkeypatch, r):
    """masked and unmasked weight gradient of one instantiation against the float64 oracle; masked entries are
    exactly +0; FLAG_ACCUMULATE adds into `out`; a reused workspace (FLAG_WORKSPACE_CLEAN) gets its tickets back
    to zero and the same bits every call; the quarter-GPU plan"""
    inp = r.make()
    k = r.meta["ksize"]
    wshape = tuple(inp["w"].shape)
    set_knobs(monkeypatch, r.knobs, WG_KNOBS)   # before any workspace is sized: it is planned under the same knobs
    buf, view = guarded(wshape)
    _, ran = launched(lambda: r.launch(nat, inp, out=view))
    assert ran == {r.expect}, ran
    check_guarded(buf, view, 0, r.id)
    dw = view.clone()
    buf, view = guarded(wshape)
    _, ran = launched(lambda: r.launch(nat, inp, out=view, flags=nat.FLAG_NO_MASK))
    assert ran == {r.expect}, ran
    check_guarded(buf, view, 0, r.id + " unmasked")
    raw = view.clone()
    init = torch.randn(wshape, device="cuda")
    acc = init.clone()
    r.launch(nat, inp, out=acc, flags=nat.FLAG_ACCUMULATE)
    assert torch.equal(acc, init + dw)
    B, _, H, W = inp["x"].shape
    ws = nat.new_workspace(nat.backward_weight_workspace_bytes(B, G, wshape[1], H, W, k, k), "cuda")
    for _ in range(3):
        assert torch.equal(r.launch(nat, inp, workspace=ws), dw)
    torch.cuda.synchronize()
    assert not bool(ws[:4096].any()), "ticket counters left dirty"
    quarter, ran = launched(lambda: r.launch(nat, inp, flags=nat.FLAG_QUARTER_GPU))
    assert ran == {r.expect}, ran
    set_knobs(monkeypatch, {}, WG_KNOBS)
    dz, x = npy(inp["dz"]), npy(inp["x"])
    want = fo.backward_weight(dz, x, (k, k), ORDERS)
    want_raw = fo.backward_weight(dz, x, (k, k), ORDERS, apply_mask=False)
    for got, ref in ((dw, want), (raw, want_raw), (quarter, want)):
        assert rel_err(npy(got), ref) <= REL_TOL and elementwise_close(npy(got), ref)
    masked = fo.apply_grad_mask(np.ones(wshape, dtype=np.float32), ORDERS) == 0
    d = dw.cpu().numpy()
    assert masked.any() and (d[masked] == 0).all() and not np.signbit(d[masked]).any()
    assert not (raw.cpu().numpy()[masked] == 0).all()


# ================================================================================================================
# chain_kernel<CT, OB, WT>
# ================================================================================================================
CHAIN_KNOBS = ("FINC_CHAIN_IPB",)
CHAIN_OB = {1: 1, 2: 2, 3: 3, 6: 2, 12: 1, 24: 4}   # finc_chain_f32's output block per channel count
CHAIN_HW = {4: 8, 2: 6, 1: 5}                       # W % 4 == 0, W % 4 == 2, W odd
CHAIN_B, CHAIN_U = 37, 3


def chain_largest_ipb(C, H, W, B, affine):
    """the largest images-per-block make_plan (finc_chain.cu) considers: <= 32 and <= B, with two CTAs per SM
    possible (<= 100 KB of shared memory) -- the smem formula restated from make_plan"""
    ob = CHAIN_OB[C]
    nob, obp = -(-C // ob), (ob if ob <= 2 else -(-ob // 4) * 4)
    tile, wk, gc = C * H * W, G * C * 9 * nob * obp, G * C

    def smem(ipb):
        blk = (ipb * G * tile + 31) & ~31
        return 4 * (((wk + 31) & ~31) + (((gc * gc + gc + 31) & ~31) if affine else 0) + 32 + 2 * (blk + 32)) + 192

    best = 1
    for ipb in range(2, min(32, B) + 1):
        if smem(ipb) > 100 * 1024:
            break
        best = ipb
    return best


def _chain_make(C, H, W):
    def make():
        torch.manual_seed(C * 100 + W)
        w = torch.stack([torch.from_numpy(unit_weight(C, 3, 50 + u + C)) for u in range(CHAIN_U)]).cuda().contiguous()
        A = (torch.linalg.qr(torch.randn(CHAIN_U, G * C, G * C))[0]
             * torch.exp(0.1 * torch.randn(CHAIN_U, 1, G * C))).cuda().contiguous()
        return {"w": w, "x": torch.randn(CHAIN_B, G * C, H, W, device="cuda"), "A": A,
                "b": torch.randn(CHAIN_U, G * C, device="cuda")}
    return make


def _chain_launch(mode):
    def launch(nat, inp, out=None):
        w, x = inp["w"], inp["x"]
        out = torch.empty((CHAIN_U,) + tuple(x.shape), device="cuda") if out is None else out
        if mode == "forward":
            return nat.chain(x, w, out)
        if mode == "transpose":
            return nat.chain(x, w, out, units=range(CHAIN_U - 1, -1, -1), transpose=True)
        return nat.chain(x, w, out, A=inp["A"], bias=inp["b"])
    return launch


def chain_recipes():
    out = []
    for C, ob in CHAIN_OB.items():
        for wt, hw in CHAIN_HW.items():
            for mode in ("forward", "transpose", "affine"):
                for ipb in ("1", "planner", "largest"):
                    out.append(Recipe("chain", (C, ob, wt), {}, _chain_make(C, hw, hw), _chain_launch(mode),
                                      f"C{C}_WT{wt}_{mode}_ipb-{ipb}", C=C, hw=hw, mode=mode, ipb=ipb))
    return out


def _chain_knobs(r):
    if r.meta["ipb"] == "planner":
        return {}
    if r.meta["ipb"] == "1":
        return {"FINC_CHAIN_IPB": 1}
    hw = r.meta["hw"]
    return {"FINC_CHAIN_IPB": chain_largest_ipb(r.meta["C"], hw, hw, CHAIN_B, r.meta["mode"] == "affine")}


CHAIN_RECIPES = chain_recipes()
for _r in CHAIN_RECIPES:
    _r.knobs = _chain_knobs(_r)


@pytest.mark.parametrize("r", CHAIN_RECIPES, ids=lambda r: r.id)
def test_chain_variant(nat, monkeypatch, r):
    """one chain_kernel instantiation at a forced images-per-block: bit-identical to the per-unit forward /
    backward-input launches, within 2e-6 of forward + affine1x1 with the affine glue; unit 0 against the oracle"""
    inp = r.make()
    set_knobs(monkeypatch, r.knobs, CHAIN_KNOBS)
    out, ran = launched(lambda: r.launch(nat, inp))
    assert ran == {r.expect}, ran
    set_knobs(monkeypatch, {}, CHAIN_KNOBS)
    w, x, mode = inp["w"], inp["x"], r.meta["mode"]
    cur = x
    if mode == "transpose":
        for u in reversed(range(CHAIN_U)):
            cur = nat.backward_input(cur, w[u])
            assert torch.equal(out[u], cur), f"unit {u}"
        want0 = None
    else:
        for u in range(CHAIN_U):
            cur, _ = nat.forward(cur, w[u])
            if mode == "affine":
                cur = nat.affine1x1(cur, inp["A"][u], inp["b"][u])
                assert rel_err(npy(out[u]), npy(cur)) <= 2e-6, f"unit {u}"
            else:
                assert torch.equal(out[u], cur), f"unit {u}"
        want0 = fo.forward(npy(x), npy(w[0]), ORDERS)
        if mode == "affine":
            want0 = np.einsum("oc,bchw->bohw", npy(inp["A"][0]), want0) + npy(inp["b"][0])[None, :, None, None]
    if want0 is not None:
        assert rel_err(npy(out[0]), want0) <= REL_TOL


# ================================================================================================================
# inverse_wave_kernel<C, K, K, P>
# ================================================================================================================
WAVE_P = {1: [1, 2, 4, 8], 2: [1, 2, 4, 8], 3: [1, 2, 4, 8], 4: [1, 2, 4, 8], 6: [1, 2, 4, 8], 12: [2, 4, 8], 24: [4, 8]}
WAVE_W = {1: 32, 2: 16, 4: 8, 8: 4}   # the planner takes the largest P <= 8 with W * P <= 32


def _wave_recipe(C, k, P):
    W = WAVE_W[P]
    H = 6 if W == 32 else min(W, 8)

    def make():
        d = _inputs(5, C, H, W, k, 300 + C + P + k)
        return {"w": d["w"], "z": d["x"]}

    def launch(nat, inp, out=None):
        return nat.inverse(inp["z"], inp["w"], G, nat.ORDERS_UNIT, flags=nat.FLAG_WAVE_SMEM, out=out)

    return Recipe("inverse_wave", (C, k, k, P), {}, make, launch, f"C{C}_k{k}_P{P}_{H}x{W}")


WAVE_RECIPES = [_wave_recipe(C, k, P) for C, ps in WAVE_P.items() for k in (3, 5) for P in ps]


@pytest.mark.parametrize("r", WAVE_RECIPES, ids=lambda r: r.id)
def test_inverse_wave_variant(nat, r):
    inp = r.make()
    buf, view = guarded(tuple(inp["z"].shape))
    _, ran = launched(lambda: r.launch(nat, inp, out=view))
    assert ran == {r.expect}, ran
    check_guarded(buf, view, 0, r.id)
    want = fo.inverse(npy(inp["z"]), npy(inp["w"]), ORDERS)
    assert rel_err(npy(view), want) <= REL_TOL and elementwise_close(npy(view), want)


# ================================================================================================================
# census: compiled == exercised + UNREACHABLE
# ================================================================================================================
ALL_RECIPES = RW_RECIPES + CONV_RECIPES + WG_RECIPES + CHAIN_RECIPES + WAVE_RECIPES
ALL_KNOBS = RW_KNOBS + CONV_KNOBS + WG_KNOBS + CHAIN_KNOBS


def test_every_compiled_instantiation_is_exercised(nat, monkeypatch):
    """every instantiation in the library's symbol table is launched by some recipe above, or is listed in
    UNREACHABLE with the reason the planner cannot select it.  Runs every recipe once under the profiler (no
    oracle), so the result does not depend on which other tests ran."""
    compiled = compiled_instantiations()
    assert {f for f, _ in compiled} == set(FAMILIES), "a kernel family is missing from the symbol table"

    def run_all():
        for r in ALL_RECIPES:
            set_knobs(monkeypatch, r.knobs, ALL_KNOBS)
            r.launch(nat, r.make())
        set_knobs(monkeypatch, {}, ALL_KNOBS)

    _, observed = launched(run_all)
    unreachable = set(UNREACHABLE)
    print(f"\n[census] compiled {len(compiled)}, observed {len(observed & compiled)}, unreachable {len(unreachable)}")
    assert unreachable <= compiled, f"UNREACHABLE lists instantiations that are not compiled: {unreachable - compiled}"
    assert not (observed & unreachable), f"UNREACHABLE instantiations ran: {observed & unreachable}"
    assert observed <= compiled, f"kernels ran that the symbol table does not list: {observed - compiled}"
    missing = compiled - unreachable - observed
    assert not missing, f"compiled but reached by no recipe: {sorted(missing)}"
    assert len(observed) + len(unreachable) == len(compiled)
