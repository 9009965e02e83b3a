"""Every compiled instantiation of the tensor-core GEMM templates against a float64 reference, with a census of the
kernels that actually ran.

The tensor-core path (csrc/tc_igemm.cuh, csrc/tc_wgrad.cuh, csrc/tc_api.cu) does nearly all the FLOPs of a whole
flow, and it is built from three template families:

    igemm_kernel<BN, NPASS, EPI = 0 (NHWC), CL, EW>   channels-last convolutions          pick_bn_nhwc, cluster_size
    igemm_kernel<BN, NPASS, EPI = 2 (ROWS), 1, EW>    coupling's third conv (BN 144), its backward dA1 (BN 64),
                                                      dense inverse (BN 64 / 128 by n % 128)
    wgrad_kernel<BN, NPASS, EW>                       weight-gradient GEMM                 pick_bn_wgrad

Each case below is a recipe: a shape plus knobs (FINC_TC_CLUSTER, read per call, and FINC_FLAG_TF32_1PASS) that
reaches one instantiation.  Each launch runs under torch.profiler and the test asserts that exactly the intended
instantiations ran, so a cluster size the planner lowers, or a BN it does not pick, fails instead of passing on
another kernel.  test_every_compiled_tc_instantiation_is_exercised lists the instantiations in the library's
symbol table and requires each to be reached by some recipe, except those in UNREACHABLE.

References are float64 PyTorch on the same inputs (F.conv2d, P^T Q, the coupling formulas) or the float64 FInC
oracle (dense inverse).  3xTF32 must be within 2e-6 max-norm relative for a GEMM (1e-5 for the coupling layer);
single-pass TF32 within 2e-3 and worse than 1e-7, which proves the single pass really ran.
"""
import functools

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import elementwise_close, rel_err
from oracle import finc_oracle as fo
from test_gpu_kernel_variants import GUARD, SENT, check_guarded, compiled_instantiations, guarded, launched, set_knobs

pytestmark = pytest.mark.gpu

TC_FAMILIES = {"igemm": "finc::tc::igemm_kernel", "wgrad": "finc::tc::wgrad_kernel"}
KNOBS = ("FINC_TC_CLUSTER",)
NHWC, ROWS = 0, 2        # tc_igemm.cuh: enum Epi
TOL3, TOL1, FLOOR1 = 2e-6, 2e-3, 1e-7

# compiled instantiations no caller can select, with the reason (from the code)
_NO_ROWS_CALLER = ("no caller of `launch_igemm_rows` passes BN 16 or 32 (`tc_api.cu`: 144 coupling apply, "
                   "64 coupling backward, 64/128 dense inverse)")
UNREACHABLE = {("igemm", (bn, p, ROWS, 1, 4)): _NO_ROWS_CALLER for bn in (16, 32) for p in (1, 3)}


def ew(bn):
    """epilogue warps of an instantiation (tc_igemm_*.cu, tc_wgrad.cu): 8 from BN = 128 up"""
    return 8 if bn >= 128 else 4


def igemm(bn, npass, epi, cl=1):
    return ("igemm", (bn, npass, epi, cl, ew(bn)))


def wgrad(bn, npass):
    return ("wgrad", (bn, npass, ew(bn)))


def pick_bn_nhwc(npad):   # tc_api.cu
    return 128 if npad % 128 == 0 else 64 if npad % 64 == 0 else 32


def pick_bn_wgrad(n):     # tc_api.cu
    return 160 if n % 160 == 0 else 128 if n % 128 == 0 else 64 if n % 64 == 0 else 0


def tc_launched(fn):
    return launched(fn, TC_FAMILIES)


def flags_of(nat, npass):
    return nat.FLAG_TF32_1PASS if npass == 1 else 0


def check_accuracy(got, want, npass, what, tol3=TOL3, tol1=TOL1):
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    e = rel_err(got, want)
    if npass == 3:
        assert e <= tol3, (what, e)
        assert elementwise_close(got, want), what
    else:
        assert FLOOR1 < e <= tol1, (what, e)


def ru(v, m):
    return (v + m - 1) // m * m


@pytest.fixture(scope="module")
def nat():
    from fincflow_b200 import _native

    _native.load()
    return _native


class Case:
    """a recipe: `knobs` (environment), `expect` (the set of tensor-core instantiations one call launches) and
    `run(nat)`, the bare launch the census uses"""

    def __init__(self, id_, knobs, expect, run, **meta):
        self.id, self.knobs, self.expect, self.run, self.meta = id_, knobs, set(expect), run, meta

    def __repr__(self):
        return self.id


# ================================================================================================================
# igemm_kernel<BN, NPASS, 0, CL, EW>: channels-last convolutions through finc_tc_conv_nhwc_f32
# ================================================================================================================
# Per BN, three shapes (B, H, W, Cin, N, taps, relu, mask).  N picks BN through Npad = round_up(N, 32).  The first
# two have a pixel-tile count that is not a multiple of 2 or 4 (cluster-padding tiles) and partial tiles (H, W
# not powers of two, W > 128, 1x1 images); 27, 3 and 9 k-blocks leave the last TMEM partial short of kFlush.
# The third has more tiles than the GPU has CTAs at every CL, so CTAs go round the persistent loop.
NHWC_SHAPES = {
    32: [(5, 7, 9, 72, 80, 9, True, False),          # Npad 96, 5 tiles, Cin_pad 96: 27 k-blocks
         (300, 1, 1, 32, 150, 1, False, True),       # Npad 160, 1x1 images: 128 per tile, 3 tiles
         (64, 16, 16, 96, 96, 1, True, False)],      # 128 pixel tiles x 3 N tiles
    64: [(1, 3, 300, 40, 40, 9, True, False),        # W > 128: 3 x 3 tiles, Cin_pad 64
         (7, 6, 10, 96, 64, 1, False, True),         # 7 tiles, 3 k-blocks
         (64, 16, 16, 64, 192, 1, True, False)],     # 128 x 3 tiles
    128: [(9, 7, 7, 80, 100, 9, True, False),        # two 8x8 images per tile, 5 tiles, 27 k-blocks
          (9, 12, 20, 32, 256, 1, False, True),      # 27 tiles x 2 N tiles
          (64, 16, 16, 512, 512, 1, True, False)],   # 128 x 4 tiles
}
NHWC_CL = {32: (1, 2), 64: (1, 2, 4), 128: (1, 2, 4)}   # instantiated (cluster_size never gives CL = 4 at BN = 32)


def _tiles(B, H, W):
    """pixel tiles of make_geom (tc_api.cu)"""
    p2 = lambda v: 1 << (v - 1).bit_length()
    wb = min(p2(W), 128)
    hb = min(p2(H), 128 // wb)
    nb = 128 // (wb * hb)
    return -(-W // wb) * -(-H // hb) * -(-B // nb)


@functools.lru_cache(maxsize=None)
def _nhwc_data(shape):
    """device inputs of one shape and the float64 reference (cached: every instantiation shares them)"""
    B, H, W, Cin, N, taps, relu, mask = shape
    k = 3 if taps == 9 else 1
    Cp, Np = ru(Cin, 32), ru(N, 32)
    g = torch.Generator().manual_seed(B * 7919 + H * 131 + W * 17 + Cin + N)
    x = torch.randn(B, Cin, H, W, generator=g)
    w = torch.randn(N, Cin, k, k, generator=g) / (Cin * taps) ** 0.5
    bias = torch.zeros(Np)
    bias[:N] = torch.randn(N, generator=g)
    xz = torch.zeros(B, H, W, Cp)
    xz[..., :Cin] = x.permute(0, 2, 3, 1)
    xg = xz.clone()      # finite garbage in the padded input channels: the prepared weights are zero there
    xg[..., Cin:] = 1e3 * torch.randn(B, H, W, Cp - Cin, generator=g)
    m = torch.randn(B, H, W, Np, generator=g) if mask else None
    ref = F.conv2d(x.cuda().double(), w.cuda().double(), bias[:N].cuda().double(), padding=k // 2).permute(0, 2, 3, 1)
    if relu:
        ref = F.relu(ref)
    if mask:
        ref = ref * (m[..., :N].cuda() > 0)
    d = {"xz": xz, "xg": xg, "w": w, "bias": bias, "mask": m}
    d = {k_: (v.cuda() if v is not None else None) for k_, v in d.items()}
    from fincflow_b200 import _native

    d["wp"] = _native.tc_conv_prepare_weights(d["w"], 0)
    d["ref"] = ref.cpu().numpy()
    return d


def _nhwc_run(nat, shape, npass, x=None, out=None):
    B, H, W, Cin, N, taps, relu, mask = shape
    d = _nhwc_data(shape)
    return nat.tc_conv_nhwc(d["xg"] if x is None else x, d["wp"], d["bias"], ru(N, 32), taps, relu=relu,
                            relu_mask=d["mask"], flags=flags_of(nat, npass), out=out)


def nhwc_cases():
    out = []
    for bn, shapes in NHWC_SHAPES.items():
        for si, shape in enumerate(shapes):
            assert pick_bn_nhwc(ru(shape[4], 32)) == bn
            for npass in (3, 1):
                for cl in NHWC_CL[bn]:
                    assert _tiles(*shape[:3]) >= cl
                    out.append(Case(f"BN{bn}_P{npass}_CL{cl}_s{si}", {"FINC_TC_CLUSTER": cl}, [igemm(bn, npass, NHWC, cl)],
                                    functools.partial(_nhwc_run, shape=shape, npass=npass), shape=shape, npass=npass,
                                    cl=cl, bn=bn))
    return out


NHWC_CASES = nhwc_cases()


@pytest.mark.parametrize("c", NHWC_CASES, ids=repr)
def test_igemm_nhwc_variant(nat, monkeypatch, c):
    """one channels-last instantiation on one shape: exactly it ran; it writes exactly its output (16-byte aligned,
    inside sentinel guard zones); padded output channels are exactly 0; garbage in the padded input channels gives
    the same bits as zeros; two runs give the same bits; CL = 2 and 4 give the same bits as CL = 1 (each tile's MMA
    sequence and partial-sum order do not depend on which CTA of the cluster loaded which weight slice: the slices
    land at the same shared-memory rows, and BN / CL % 8 == 0 keeps the swizzle phase); float64 F.conv2d"""
    shape, npass, cl = c.meta["shape"], c.meta["npass"], c.meta["cl"]
    B, H, W, Cin, N, taps, relu, mask = shape
    d = _nhwc_data(shape)
    oshape = (B, H, W, ru(N, 32))
    set_knobs(monkeypatch, c.knobs, KNOBS)
    buf, view = guarded(oshape)
    _, ran = tc_launched(lambda: c.run(nat, out=view))
    assert ran == c.expect, (c.id, ran)
    check_guarded(buf, view, 0, c.id)
    y = view.clone()
    assert torch.equal(c.run(nat), y), "two runs differ"
    if Cin % 32:
        assert torch.equal(c.run(nat, x=d["xz"]), y), "the padded input channels changed the result"
    assert bool((y[..., N:] == 0).all()), "padded output channels are not 0"
    if cl > 1:
        set_knobs(monkeypatch, {"FINC_TC_CLUSTER": 1}, KNOBS)
        y1, ran = tc_launched(lambda: c.run(nat))
        assert ran == {igemm(c.meta["bn"], npass, NHWC, 1)}, ran
        assert torch.equal(y, y1), f"CL = {cl} differs from CL = 1"
    set_knobs(monkeypatch, {}, KNOBS)
    check_accuracy(y[..., :N].cpu().numpy(), d["ref"], npass, c.id)


# cluster sizes the planner must lower (cluster_size, tc_api.cu): (shape, forced CL, CL that runs)
CL_LOWERED = [
    (NHWC_SHAPES[32][0], 4, 2),                        # BN = 32 has no CL = 4
    ((1, 8, 16, 32, 64, 1, True, False), 2, 1),        # one pixel tile
    (NHWC_SHAPES[128][0], 3, 1),                       # 128 % 3 != 0
    (NHWC_SHAPES[128][1], 8, 4),                       # 27 tiles, but no CL = 8 instantiation: capped at 4
]


@pytest.mark.parametrize("case", CL_LOWERED, ids=lambda c: f"BN{pick_bn_nhwc(ru(c[0][4], 32))}_force{c[1]}")
def test_cluster_knob_is_lowered_to_an_instantiated_size(nat, monkeypatch, case):
    """FINC_TC_CLUSTER is read per call; a size the kernel cannot take runs the largest one it can, with the
    same bits as CL = 1"""
    shape, force, runs = case
    bn = pick_bn_nhwc(ru(shape[4], 32))
    set_knobs(monkeypatch, {"FINC_TC_CLUSTER": force}, KNOBS)
    y, ran = tc_launched(lambda: _nhwc_run(nat, shape, 3))
    assert ran == {igemm(bn, 3, NHWC, runs)}, ran
    set_knobs(monkeypatch, {}, KNOBS)
    y1, ran = tc_launched(lambda: _nhwc_run(nat, shape, 3))
    assert ran == {igemm(bn, 3, NHWC, 1)}, ran
    assert torch.equal(y, y1)


# ================================================================================================================
# igemm_kernel<144, NPASS, 2, 1, 8>: the coupling layer's third convolution (finc_coupling_apply_f32)
# ================================================================================================================
COUPLING_C = (12, 24, 48, 64, 96)     # N3pad = 16, 32, 48, 64, 96: one to six N tiles of 144 columns
COUPLING_WIDTHS = (32, 96, 512)
LOGSCALE = 3.0


def _coupling_shape(C):
    return (16, 16, 16) if C == 96 else (3, 6, 10)   # C = 96: 32 pixel tiles x 6 N tiles, more than one per CTA


@functools.lru_cache(maxsize=None)
def _coupling_data(C, width, with_backward=False):
    from fincflow_b200 import _native

    B, H, W = _coupling_shape(C)
    g = torch.Generator().manual_seed(C * 1000 + width)
    ci = C // 2
    p = {
        "w1": torch.randn(width, ci, 3, 3, generator=g) / (9 * ci) ** 0.5, "b1": 0.1 * torch.randn(width, generator=g),
        "w2": torch.randn(width, width, 1, 1, generator=g) / width ** 0.5, "b2": 0.1 * torch.randn(width, generator=g),
        "w3": 0.5 * torch.randn(C, width, 3, 3, generator=g) / (9 * width) ** 0.5,
        "b3": 0.1 * torch.randn(C, generator=g), "logs3": 0.1 * torch.randn(C, generator=g),
    }
    p = {k: v.cuda() for k, v in p.items()}
    x = torch.randn(B, C, H, W, generator=g).cuda()
    blob = _native.coupling_prepare(p["w1"], p["b1"], p["w2"], p["b2"], p["w3"], p["b3"], p["logs3"], LOGSCALE,
                                    with_backward=with_backward)
    return p, x, blob


def coupling_ref(x, p, reverse=False):
    """layers/coupling.py in float64: y (or the reverse map's x) and the per-image logdet"""
    x = x.double()
    q = {k: v.double() for k, v in p.items()}
    ci = x.shape[1] // 2
    x1, x2 = x[:, :ci], x[:, ci:]
    h = F.relu(F.conv2d(x1, q["w1"], q["b1"], padding=1))
    h = F.relu(F.conv2d(h, q["w2"], q["b2"]))
    h = F.conv2d(h, q["w3"], q["b3"], padding=1) * torch.exp(LOGSCALE * q["logs3"]).view(1, -1, 1, 1)
    log_s, t = 2.0 * torch.tanh(h[:, ::2] / 2.0), h[:, 1::2]
    y2 = (x2 - t) * torch.exp(-log_s) if reverse else x2 * torch.exp(log_s) + t
    return torch.cat([x1, y2], dim=1), log_s.flatten(1).sum(-1)


def coupling_cases():
    out = []
    for C in COUPLING_C:
        for width in COUPLING_WIDTHS:
            for npass in (3, 1):
                expect = [igemm(pick_bn_nhwc(width), npass, NHWC), igemm(144, npass, ROWS)]

                def run(nat, C=C, width=width, npass=npass):
                    _, x, blob = _coupling_data(C, width)
                    return nat.coupling_apply(x, blob, width, flags=flags_of(nat, npass))

                out.append(Case(f"C{C}_w{width}_P{npass}", {}, expect, run, C=C, width=width, npass=npass))
    return out


COUPLING_CASES = coupling_cases()


@pytest.mark.parametrize("c", COUPLING_CASES, ids=repr)
def test_igemm_rows_coupling_apply(nat, monkeypatch, c):
    """ROWS BN = 144 through the coupling layer, forward (logdet on, off and accumulated) and reverse, against the
    float64 formulas; the first half of the channels passes through exactly"""
    C, width, npass = c.meta["C"], c.meta["width"], c.meta["npass"]
    p, x, blob = _coupling_data(C, width)
    f = flags_of(nat, npass)
    set_knobs(monkeypatch, {}, KNOBS)
    buf, view = guarded(tuple(x.shape))
    (y, ld), ran = tc_launched(lambda: nat.coupling_apply(x, blob, width, flags=f, out=view))
    assert ran == c.expect, ran
    check_guarded(buf, view, 0, c.id)
    y = y.clone()
    y_nold, ld_none = nat.coupling_apply(x, blob, width, want_logdet=False, flags=f)
    assert ld_none is None and torch.equal(y_nold, y)
    acc0 = torch.randn(x.shape[0], device="cuda")
    acc = acc0.clone()
    nat.coupling_apply(x, blob, width, logdet_out=acc, flags=f | nat.FLAG_LOGDET_ACCUMULATE)
    assert torch.equal(acc, acc0 + ld)
    buf, view = guarded(tuple(x.shape))
    (xr, _), ran = tc_launched(lambda: nat.coupling_apply(x, blob, width, reverse=True, flags=f, out=view))
    assert ran == c.expect, ran
    check_guarded(buf, view, 0, c.id + " reverse")
    ci = C // 2
    assert torch.equal(y[:, :ci], x[:, :ci]) and torch.equal(xr[:, :ci], x[:, :ci])
    y64, ld64 = coupling_ref(x, p)
    xr64, _ = coupling_ref(x, p, reverse=True)
    check_accuracy(y[:, ci:].cpu(), y64[:, ci:].cpu(), npass, "y", tol3=1e-5)
    check_accuracy(xr[:, ci:].cpu(), xr64[:, ci:].cpu(), npass, "reverse", tol3=1e-5)
    e = rel_err(ld.cpu().numpy(), ld64.cpu().numpy())
    assert e <= (1e-5 if npass == 3 else 1e-2), ("logdet", e)


# ================================================================================================================
# igemm_kernel<64, NPASS, 2, 1, 4>: dA1 of the coupling backward (finc_coupling_backward_f32)
# ================================================================================================================
COUPLING_BWD = [(12, 128), (24, 256), (48, 128)]   # C, width (the backward needs width % 128 == 0)


def _coupling_bwd_expect(C, width, npass):
    k1pad, ldy = ru(9 * (C // 2), 64), ru(9 * ru(C, 16), 160)
    return [igemm(64, npass, ROWS), igemm(pick_bn_nhwc(width), npass, NHWC)] + [
        wgrad(pick_bn_wgrad(n), npass) for n in (ldy, width, k1pad)]


def _coupling_bwd_run(nat, C, width, npass):
    """the backward's launch and its inputs.  The forward that saves the activations always runs in 3xTF32: from a
    single-pass forward, a ReLU whose input is near 0 can switch against the float64 reference and pass (or drop)
    a whole gradient element, which says nothing about the backward's GEMMs"""
    p, x, blob = _coupling_data(C, width, True)
    B, _, H, W = x.shape
    ws = torch.empty(nat.coupling_workspace_bytes(B, C, H, W, width), dtype=torch.uint8, device="cuda")
    nat.coupling_apply(x, blob, width, workspace=ws)
    g = torch.Generator(device="cuda").manual_seed(C + width)
    dy = torch.randn(x.shape, device="cuda", generator=g)
    dld = torch.randn(B, device="cuda", generator=g)
    return lambda: nat.coupling_backward(x, dy, dld, blob, ws, width, flags=flags_of(nat, npass)), (x, dy, dld, p)


def coupling_bwd_cases():
    return [Case(f"C{C}_w{width}_P{npass}", {}, _coupling_bwd_expect(C, width, npass),
                 lambda nat, C=C, width=width, npass=npass: _coupling_bwd_run(nat, C, width, npass)[0](),
                 C=C, width=width, npass=npass)
            for C, width in COUPLING_BWD for npass in (3, 1)]


COUPLING_BWD_CASES = coupling_bwd_cases()


@pytest.mark.parametrize("c", COUPLING_BWD_CASES, ids=repr)
def test_igemm_rows_coupling_backward(nat, monkeypatch, c):
    """ROWS BN = 64 (and the backward's wgrad / backward-data GEMMs) against float64 autograd of the formulas"""
    C, width, npass = c.meta["C"], c.meta["width"], c.meta["npass"]
    set_knobs(monkeypatch, {}, KNOBS)
    go, (x, dy, dld, p) = _coupling_bwd_run(nat, C, width, npass)
    got, ran = tc_launched(go)
    assert ran == c.expect, ran
    x64 = x.double().requires_grad_(True)
    p64 = {k: v.double().requires_grad_(True) for k, v in p.items()}
    y64, ld64 = coupling_ref(x64, p64)
    want = torch.autograd.grad([y64, ld64], [x64] + [p64[k] for k in ("w1", "b1", "w2", "b2", "w3", "b3", "logs3")],
                               [dy.double(), dld.double()])
    # single pass: three chained TF32 GEMMs (dY -> dh2 -> dh1 -> dA1) before dx, hence the wider bound
    errs = {name: rel_err(a.cpu().numpy(), b.cpu().numpy())
            for name, a, b in zip(("dx", "dw1", "db1", "dw2", "db2", "dw3", "db3", "dlogs3"), got, want)}
    assert [a.shape for a in got] == [b.shape for b in want]
    assert max(errs.values()) <= (2e-5 if npass == 3 else 2e-2), errs


# ================================================================================================================
# igemm_kernel<64 | 128, NPASS, 2, 1, EW>: the dense inverse (finc_inverse_dense_f32), BN = 128 iff n % 128 == 0
# ================================================================================================================
DENSE = [  # C, H, W, G, B, k;  n = C * H * W
    (4, 4, 4, 1, 129, 3),     # n = 64
    (12, 4, 4, 2, 1, 3),      # n = 192
    (3, 8, 8, 4, 129, 5),     # n = 192
    (4, 4, 4, 16, 129, 3),    # n = 64, sixteen groups
    (8, 4, 4, 1, 1, 3),       # n = 128
    (4, 8, 8, 2, 129, 5),     # n = 256
    (16, 8, 8, 4, 129, 3),    # n = 1024
    (2, 8, 8, 16, 129, 3),    # n = 128, sixteen groups
]


@functools.lru_cache(maxsize=None)
def _dense_data(C, H, W, G, B, k):
    from fincflow_b200 import _native

    rng = np.random.default_rng(C * 100 + H + 7 * G + B)
    orders = tuple(int(o) for o in rng.integers(0, 4, G))
    w = np.concatenate([fo.init_weight(C, (k, k), o, rng) for o in orders], axis=0)
    z = rng.standard_normal((B, G * C, H, W)).astype(np.float32)
    packed = sum(o << (2 * g) for g, o in enumerate(orders))
    wd = torch.from_numpy(w).cuda()
    blob = _native.inverse_dense_prepare(wd, H, W, G, packed)
    return torch.from_numpy(z).cuda(), blob, fo.inverse(z, w, orders)


def dense_cases():
    out = []
    for case in DENSE:
        C, H, W, G, B, k = case
        bn = 128 if C * H * W % 128 == 0 else 64
        for npass in (3, 1):
            def run(nat, case=case, npass=npass, out=None):
                z, blob, _ = _dense_data(*case)
                return nat.inverse_dense(z, blob, case[3], flags=flags_of(nat, npass), out=out)

            out.append(Case(f"n{C * H * W}_C{C}_G{G}_B{B}_k{k}_P{npass}", {}, [igemm(bn, npass, ROWS)], run, case=case,
                            npass=npass))
    return out


DENSE_CASES = dense_cases()


@pytest.mark.parametrize("c", DENSE_CASES, ids=repr)
def test_igemm_rows_dense_inverse(nat, monkeypatch, c):
    """ROWS BN = 64 / 128 through the dense inverse: random corner orders, G up to 16, batch tails; against the
    float64 oracle, inside guard zones, deterministic"""
    set_knobs(monkeypatch, {}, KNOBS)
    z, _, want = _dense_data(*c.meta["case"])
    buf, view = guarded(tuple(z.shape))
    _, ran = tc_launched(lambda: c.run(nat, out=view))
    assert ran == c.expect, ran
    check_guarded(buf, view, 0, c.id)
    assert torch.equal(c.run(nat), view)
    check_accuracy(view.cpu().numpy(), want, c.meta["npass"], c.id, tol3=1e-5)


# ================================================================================================================
# wgrad_kernel<BN, NPASS, EW> through finc_tc_wgrad_f32
# ================================================================================================================
WGRAD = [  # np, M, N, ldP - M, ldQ - N, ld_dW - N
    (1000, 96, 160, 0, 0, 0),        # BN 160, 32 slices
    (77, 200, 320, 4, 32, 8),        # strided P, Q and dW; a partial last k-block
    (96, 2048, 1760, 0, 0, 0),       # 16 x 11 tiles > SMs: CTAs take a second work item
    (5000, 1, 128, 3, 0, 4),         # BN 128, M = 1
    (30, 256, 384, 0, 64, 16),       # one k-block: a single slice
    (96, 2048, 1536, 0, 0, 0),       # 16 x 12 tiles
    (1000, 200, 64, 4, 0, 4),        # BN 64
    (33, 96, 448, 0, 0, 0),          # 7 N tiles, two k-blocks
    (96, 2048, 704, 0, 0, 0),        # 16 x 11 tiles
]


@functools.lru_cache(maxsize=None)
def _wgrad_data(np_, M, N, xp, xq):
    g = torch.Generator().manual_seed(np_ + M + N)
    P = torch.randn(np_, M + xp, generator=g)
    Q = torch.randn(np_, N + xq, generator=g)
    P[:, M:] = 1e3 * torch.randn(np_, xp, generator=g)   # columns past M / N are not part of the operands
    Q[:, N:] = 1e3 * torch.randn(np_, xq, generator=g)
    ref = (P[:, :M].double().t() @ Q[:, :N].double()).numpy()
    return P.cuda(), Q.cuda(), ref


def wgrad_cases():
    out = []
    for case in WGRAD:
        np_, M, N, xp, xq, xd = case
        for npass in (3, 1):
            def run(nat, case=case, npass=npass, out=None, flags=0):
                np_, M, N, xp, xq, _ = case
                P, Q, _ = _wgrad_data(np_, M, N, xp, xq)
                return nat.tc_wgrad(P, Q, M=M, N=N, flags=flags_of(nat, npass) | flags, out=out)

            out.append(Case(f"np{np_}_M{M}_N{N}_ld{xp}-{xq}-{xd}_P{npass}", {}, [wgrad(pick_bn_wgrad(N), npass)], run,
                            case=case, npass=npass))
    return out


WGRAD_CASES = wgrad_cases()


@pytest.mark.parametrize("c", WGRAD_CASES, ids=repr)
def test_wgrad_variant(nat, monkeypatch, c):
    """one wgrad instantiation: exactly it ran; dW written through a strided view leaves its padding columns and the
    guard zones untouched; FINC_FLAG_ACCUMULATE gives exactly old + fresh (fp32, `*d + s`); deterministic;
    float64 P^T Q"""
    np_, M, N, xp, xq, xd = c.meta["case"]
    _, _, ref = _wgrad_data(np_, M, N, xp, xq)
    set_knobs(monkeypatch, {}, KNOBS)
    ld = N + xd
    buf, full = guarded((M, ld))
    view = full[:, :N]
    _, ran = tc_launched(lambda: c.run(nat, out=view))
    assert ran == c.expect, ran
    torch.cuda.synchronize()
    assert bool((buf[:GUARD] == SENT).all()) and bool((buf[GUARD + M * ld:] == SENT).all()), "write outside dW"
    assert bool((full[:, N:] == SENT).all()), "write into the padding columns of dW"
    assert not bool((view == SENT).any()), "dW left unwritten"
    dw = view.clone()
    assert torch.equal(c.run(nat), dw), "two runs differ"
    old = torch.randn(M, ld, device="cuda")
    acc = old.clone()
    c.run(nat, out=acc[:, :N], flags=nat.FLAG_ACCUMULATE)
    want = old.cpu()
    want[:, :N] = want[:, :N] + dw.cpu()
    assert torch.equal(acc.cpu(), want), "ACCUMULATE is not old + fresh"
    check_accuracy(dw.cpu().numpy(), ref, c.meta["npass"], c.id)


# ================================================================================================================
# census: compiled == exercised + UNREACHABLE
# ================================================================================================================
ALL_CASES = NHWC_CASES + COUPLING_CASES + COUPLING_BWD_CASES + DENSE_CASES + WGRAD_CASES


def test_every_compiled_tc_instantiation_is_exercised(nat, monkeypatch):
    """every tensor-core instantiation in the library's symbol table is launched by some recipe above, or is listed
    in UNREACHABLE with the reason no caller selects it.  Runs every recipe once under the profiler (no reference),
    so the result does not depend on which other tests ran."""
    compiled = compiled_instantiations(TC_FAMILIES)
    assert {f for f, _ in compiled} == set(TC_FAMILIES), "a tensor-core family is missing from the symbol table"

    def run_all():
        for c in ALL_CASES:
            set_knobs(monkeypatch, c.knobs, KNOBS)
            c.run(nat)
        set_knobs(monkeypatch, {}, KNOBS)

    _, observed = tc_launched(run_all)
    expected = set().union(*(c.expect for c in ALL_CASES))
    unreachable = set(UNREACHABLE)
    print(f"\n[tc census] compiled {len(compiled)}, launched {len(observed & compiled)}, unreachable {len(unreachable)}")
    assert observed == expected, f"recipes ran {observed - expected}, missed {expected - observed}"
    assert unreachable <= compiled, f"UNREACHABLE lists instantiations that are not compiled: {unreachable - compiled}"
    assert not (observed & unreachable), f"UNREACHABLE instantiations ran: {observed & unreachable}"
    assert observed <= compiled, f"kernels ran that the symbol table does not list: {observed - compiled}"
    missing = compiled - unreachable - observed
    assert not missing, f"compiled but reached by no recipe: {sorted(missing)}"
    assert len(observed) + len(unreachable) == len(compiled)
