"""The differentiable sampling direction (run on the B200 box: `pytest -m gpu`).

  * finc_inverse_adjoint_f32: dz = A^-T dx for the map A that finc_inverse_f32 inverts, on every register-window
    family of the inverse and on the generic kernel;
  * FINC_FLAG_NEGATE of the weight-gradient kernels;
  * autograd through PaddedConv2d / FastFlowUnit / FincStack .reverse and a whole FastFlow.reverse, against a
    float64 PyTorch reference: the fixed-point solve x <- z - (F(x) - x), F = F.pad + conv2d with the corner
    constants of the inverse (unit diagonal, nothing above it) substituted, iterated (H+W-1)*C times -- the
    dependency chains of the triangular system are never longer, so the iteration is the exact solve.
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import rel_err
from oracle import finc_oracle as fo
from test_gpu_parity import INVERSE_KERNEL_CASES

pytestmark = pytest.mark.gpu

REL_TOL = 1e-5
ORDERS = ("TL", "TR", "BL", "BR")
CODE = {"TL": 0, "TR": 1, "BL": 2, "BR": 3}


@pytest.fixture(scope="module")
def nat():
    from fincflow_b200 import _native

    _native.load()
    return _native


@pytest.fixture
def fp32_convs():
    """the reference's conv2d in true fp32 (cuDNN would otherwise use TF32 products)"""
    old = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32 = old


def npy(t):
    return t.detach().double().cpu().numpy()


def unit_weight(CT, k, seed=0):
    from fincflow_b200.fastflow import FastFlowUnit

    torch.manual_seed(seed)
    return FastFlowUnit(CT, CT, (k, k)).weight.detach().cuda()


def adjoint_oracle(dx, w, orders):
    """float64 A^-T dx per group: a FInC inverse with w''[o, i, a, b] = w[C-1-i, C-1-o, kH-1-a, kW-1-b], the opposite
    corner and the channels reversed"""
    G, C = len(orders), w.shape[1]
    out = np.empty(dx.shape, dtype=np.float64)
    for g, o in enumerate(orders):
        code = CODE[o] if isinstance(o, str) else int(o)
        w2 = w[g * C:(g + 1) * C][::-1, ::-1].transpose(1, 0, 2, 3)[:, :, ::-1, ::-1]
        out[:, g * C:(g + 1) * C] = fo.inverse(dx[:, g * C:(g + 1) * C][:, ::-1], w2, orders=[code ^ 3])[:, ::-1]
    return out


# ---- kernel -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", INVERSE_KERNEL_CASES, ids=lambda s: "B{}C{}_{}x{}_k{}".format(*s))
def test_adjoint_kernel(nat, shape):
    """register-window adjoint: inverts backward_input, is the transpose of inverse(), equals the generic kernel and
    the float64 oracle, runs in place bit for bit, and never reads w[o, i>=o, corner]"""
    B, CT, H, W, k = shape
    w = unit_weight(CT, k, B + CT + k)
    torch.manual_seed(B + k)
    dx = torch.randn(B, CT, H, W, device="cuda")
    z = torch.randn(B, CT, H, W, device="cuda")
    g = nat.inverse_adjoint(dx, w)
    assert rel_err(npy(nat.backward_input(g, w)), npy(dx)) <= REL_TOL
    lhs = (g.double() * z.double()).flatten(1).sum(1)
    rhs = (dx.double() * nat.inverse(z, w).double()).flatten(1).sum(1)
    assert rel_err(lhs.cpu().numpy(), rhs.cpu().numpy()) <= REL_TOL
    assert rel_err(npy(nat.inverse_adjoint(dx, w, flags=nat.FLAG_NAIVE)), npy(g)) <= REL_TOL
    sel = torch.cat([dx[:3], dx[-3:]]) if B > 6 else dx
    got = torch.cat([g[:3], g[-3:]]) if B > 6 else g
    assert rel_err(npy(got), adjoint_oracle(npy(sel), npy(w), ORDERS)) <= REL_TOL
    buf = dx.clone()
    nat.inverse_adjoint(buf, w, out=buf)
    assert torch.equal(buf, g)
    # the corner diagonal is taken as 1 and the entries above it are never read
    C = CT // 4
    w2 = w.clone()
    for q, o in enumerate(ORDERS):
        a, b = (0 if CODE[o] & 2 else k - 1), (0 if CODE[o] & 1 else k - 1)
        blk = w2[q * C:(q + 1) * C, :, a, b]
        blk += torch.triu(torch.full((C, C), 0.37, device="cuda"))
    assert torch.equal(nat.inverse_adjoint(dx, w2), g)


@pytest.mark.parametrize("order", ORDERS)
@pytest.mark.parametrize("shape", [(64, 3, 16, 16, 3), (5, 12, 8, 8, 3), (9, 2, 7, 11, 5), (3, 24, 8, 8, 3),
                                   (2, 3, 40, 36, 3), (4, 5, 6, 6, 3), (3, 2, 9, 9, 4)],
                         ids=lambda s: "B{}C{}_{}x{}_k{}".format(*s))
def test_adjoint_single_group(nat, order, shape):
    """G = 1 (PaddedConv2d) for every order; covers the generic kernel (C = 24 and 5, W > 32, even k)"""
    from fincflow_b200.layers.conv import PaddedConv2d

    B, C, H, W, k = shape
    torch.manual_seed(C * H + k)
    w = PaddedConv2d(C, C, (k, k), order=order).conv.weight.detach().cuda()
    po = nat.pack_orders([order])
    dx = torch.randn(B, C, H, W, device="cuda")
    g = nat.inverse_adjoint(dx, w, 1, po)
    assert rel_err(npy(nat.backward_input(g, w, 1, po)), npy(dx)) <= REL_TOL
    assert rel_err(npy(g), adjoint_oracle(npy(dx), npy(w), [order])) <= REL_TOL
    assert rel_err(npy(nat.inverse_adjoint(dx, w, 1, po, flags=nat.FLAG_NAIVE)), npy(g)) <= REL_TOL


@pytest.mark.parametrize("order", ORDERS)
def test_adjoint_dense_solve(nat, order):
    """tiny shapes: exactly np.linalg.solve(M^T, dx) with M the dense matrix of the convolution"""
    from fincflow_b200.layers.conv import PaddedConv2d

    C, H, W, k = 3, 4, 5, 3
    torch.manual_seed(CODE[order])
    w = PaddedConv2d(C, C, (k, k), order=order).conv.weight.detach().cuda()
    dx = torch.randn(2, C, H, W, device="cuda")
    g = nat.inverse_adjoint(dx, w, 1, nat.pack_orders([order]))
    M = fo.dense_matrix(npy(w), H, W, order)
    want = np.linalg.solve(M.T, npy(dx).reshape(2, -1).T).T.reshape(2, C, H, W)
    assert rel_err(npy(g), want) <= REL_TOL


def test_adjoint_edge_inputs(nat):
    """B = 0, unaligned and non-contiguous tensors (no TMA path), and the refused prepared flag"""
    w = unit_weight(12, 3)
    B, CT, H, W = 37, 12, 16, 16
    assert nat.inverse_adjoint(torch.empty(0, CT, H, W, device="cuda"), w).shape == (0, CT, H, W)
    torch.manual_seed(1)
    dx = torch.randn(B, CT, H, W, device="cuda")
    g = nat.inverse_adjoint(dx, w)
    n = dx.numel()
    src = torch.empty(n + 1, device="cuda")
    src[1:] = dx.flatten()
    dst = torch.empty(n + 1, device="cuda")
    out = dst[1:].view(B, CT, H, W)
    nat.inverse_adjoint(src[1:].view(B, CT, H, W), w, out=out)     # 4-byte aligned only
    assert torch.equal(out, g)
    wide = torch.randn(B, 2 * CT, H, W, device="cuda")
    wide[:, 1::2] = dx
    assert torch.equal(nat.inverse_adjoint(wide[:, 1::2], w), g)  # non-contiguous
    lib = nat.load()
    assert lib.finc_inverse_adjoint_f32(dx.data_ptr(), w.data_ptr(), g.data_ptr(), B, 4, 3, H, W, 3, 3,
                                        nat.ORDERS_UNIT, nat.FLAG_PREPARED, None) == -3


# ---- FINC_FLAG_NEGATE ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("naive", [False, True], ids=["tiled", "naive"])
@pytest.mark.parametrize("shape", [(256, 12, 16, 16, 3), (300, 48, 4, 4, 3), (64, 24, 8, 8, 5), (16, 96, 4, 4, 3)],
                         ids=lambda s: "B{}C{}_{}x{}_k{}".format(*s))
def test_negate_flag(nat, naive, shape):
    from fincflow_b200.layers.conv import finc_grad_mask

    B, CT, H, W, k = shape
    torch.manual_seed(B + CT)
    dz = torch.randn(B, CT, H, W, device="cuda")
    x = torch.randn(B, CT, H, W, device="cuda")
    base = nat.FLAG_NAIVE if naive else 0
    plain = nat.backward_weight(dz, x, (k, k), flags=base)
    neg = nat.backward_weight(dz, x, (k, k), flags=base | nat.FLAG_NEGATE)
    assert torch.equal(neg, -plain)
    masked = torch.cat([finc_grad_mask(CT // 4, (k, k), o) for o in ORDERS]).cuda() == 0
    assert bool((neg[masked] == 0).all()) and not bool(torch.signbit(neg[masked]).any())   # +0, not -0
    init = torch.randn_like(plain)
    acc = init.clone()
    nat.backward_weight(dz, x, (k, k), flags=base | nat.FLAG_NEGATE | nat.FLAG_ACCUMULATE, out=acc)
    assert torch.equal(acc, init + (-plain))


def test_negate_flag_batched(nat):
    B, CT, H, W, U = 256, 12, 16, 16, 3
    torch.manual_seed(3)
    dz = torch.randn(U, B, CT, H, W, device="cuda")
    x = torch.randn(U, B, CT, H, W, device="cuda")
    plain = torch.empty(U, CT, CT // 4, 3, 3, device="cuda")
    neg = torch.empty_like(plain)
    nat.backward_weight_batched(dz, x, plain, (3, 3))
    nat.backward_weight_batched(dz, x, neg, (3, 3), flags=nat.FLAG_NEGATE)
    assert torch.equal(neg, -plain)
    acc = torch.randn_like(plain)
    want = acc + (-plain)
    nat.backward_weight_batched(dz, x, acc, (3, 3), flags=nat.FLAG_NEGATE | nat.FLAG_ACCUMULATE)
    assert torch.equal(acc, want)


# ---- autograd -----------------------------------------------------------------------------------------------------
def _pad(order, k):
    kH, kW = k
    return {"TL": (kW - 1, 0, kH - 1, 0), "TR": (0, kW - 1, kH - 1, 0),
            "BL": (kW - 1, 0, 0, kH - 1), "BR": (0, kW - 1, 0, kH - 1)}[order]


def ref_inverse(z, w, orders):
    """differentiable float64 solve of the inverse (see the module docstring), one group per order"""
    G, C = len(orders), w.shape[1]
    k = tuple(w.shape[2:])
    H, W = z.shape[2], z.shape[3]
    outs = []
    for g, order in enumerate(orders):
        code = CODE[order]
        a, b = (0 if code & 2 else k[0] - 1), (0 if code & 1 else k[1] - 1)
        keep = torch.ones_like(w[:C])
        keep[:, :, a, b] = torch.tril(torch.ones(C, C, dtype=w.dtype, device=w.device), -1)
        const = torch.zeros_like(w[:C])
        const[:, :, a, b] = torch.eye(C, dtype=w.dtype, device=w.device)
        wg = w[g * C:(g + 1) * C] * keep + const
        zg = z[:, g * C:(g + 1) * C]
        x = zg
        for _ in range((H + W - 1) * C):
            x = zg - (F.conv2d(F.pad(x, _pad(order, k)), wg) - x)
        outs.append(x)
    return torch.cat(outs, 1)


def _grads(fn, z, w, r):
    z = z.detach().clone().requires_grad_()
    w = w.detach().clone().requires_grad_()
    x = fn(z, w)
    gz, gw = torch.autograd.grad((x * r).sum(), (z, w))
    return x, gz, gw


def _check_against_ref(fn, z, w, orders, masked, same_bits=True):
    r = torch.randn_like(z)
    x, gz, gw = _grads(fn, z, w, r)
    _, rz, rw = _grads(lambda zz, ww: ref_inverse(zz.double(), ww.double(), orders), z, w, r.double())
    assert rel_err(npy(gz), npy(rz)) <= REL_TOL
    assert rel_err(npy(gw), npy(rw)) <= REL_TOL
    assert bool((gw[masked] == 0).all()) and bool((rw[masked] == 0).all())
    if same_bits:
        with torch.no_grad():
            assert torch.equal(x, fn(z, w))     # the same bits with and without autograd
    return gz, gw


@pytest.mark.parametrize("order", ORDERS)
@pytest.mark.parametrize("mask_in_backward", [False, True])
def test_padded_conv_reverse_grad(fp32_convs, order, mask_in_backward):
    from fincflow_b200.layers.conv import PaddedConv2d

    torch.manual_seed(CODE[order])
    layer = PaddedConv2d(3, 3, (3, 3), order=order, mask_in_backward=mask_in_backward).cuda()
    z = torch.randn(6, 3, 10, 12, device="cuda")
    masked = layer.mask.cuda() == 0

    def fn(zz, ww):   # the layer's reverse with ww as its weight (keeps the graph to ww)
        del layer.conv.weight
        layer.conv.weight = ww
        return layer.reverse(zz)[0]

    _check_against_ref(fn, z, layer.conv.weight.detach().clone(), [order], masked)
    del layer.conv.weight
    layer.conv.weight = torch.nn.Parameter(torch.randn(3, 3, 3, 3, device="cuda"))
    assert not layer.reverse(z)[0].requires_grad      # a latent without grad: no graph, as before


@pytest.mark.parametrize("dense", [False, True], ids=["wavefront", "dense_reverse"])
def test_fastflow_unit_reverse_grad(fp32_convs, dense):
    from fincflow_b200.fastflow import FastFlowUnit
    from fincflow_b200.layers.conv import finc_grad_mask

    torch.manual_seed(7)
    unit = FastFlowUnit(12, 12, (3, 3)).cuda()
    unit.dense_reverse = dense
    w0 = unit.weight.detach().clone()
    z = torch.randn(5, 12, 8, 8, device="cuda")
    masked = torch.cat([finc_grad_mask(3, (3, 3), o) for o in ORDERS]).cuda() == 0

    def fn(zz, ww):
        del unit.weight
        unit.weight = ww
        return unit.reverse(zz)

    # a latent with grad runs the wavefront forward (dense_reverse or not): the same bits as the wavefront without
    # autograd; dense_reverse without autograd runs the dense table
    _check_against_ref(fn, z, w0, list(ORDERS), masked, same_bits=not dense)
    unit.weight = torch.nn.Parameter(w0.clone())
    zg = z.clone().requires_grad_()
    xg = unit.reverse(zg)
    assert xg.requires_grad and torch.equal(xg, _wavefront(unit, z))
    # a latent without grad: no graph, even though the weight is a parameter (sampling code gets plain tensors)
    x = unit.reverse(z)
    assert not x.requires_grad
    with torch.no_grad():
        assert torch.equal(x, unit.reverse(z))


def _wavefront(unit, z):
    from fincflow_b200 import _native

    return _native.inverse(z, unit.weight.detach())


def _ref_dw(z, w, orders, r):
    w = w.detach().double().clone().requires_grad_()
    (rw,) = torch.autograd.grad((ref_inverse(z.double(), w, orders) * r.double()).sum(), (w,))
    return rw


@pytest.mark.parametrize("order", ORDERS)
def test_weight_only_grad_padded_conv(fp32_convs, order):
    """a latent without grad inside weight_grad_in_reverse: the weight gets its gradient, the output its usual bits"""
    from fincflow_b200 import weight_grad_in_reverse
    from fincflow_b200.layers.conv import PaddedConv2d

    torch.manual_seed(20 + CODE[order])
    layer = PaddedConv2d(3, 3, (3, 3), order=order).cuda()
    z = torch.randn(6, 3, 10, 12, device="cuda")
    r = torch.randn_like(z)
    with weight_grad_in_reverse():
        x = layer.reverse(z)[0]
    assert x.requires_grad
    with torch.no_grad():
        assert torch.equal(x, layer.reverse(z)[0])
    (gw,) = torch.autograd.grad((x * r).sum(), (layer.conv.weight,))
    rw = _ref_dw(z, layer.conv.weight, [order], r)
    assert rel_err(npy(gw), npy(rw)) <= REL_TOL
    masked = layer.mask.cuda() == 0
    assert bool((gw[masked] == 0).all())


@pytest.mark.parametrize("dense", [False, True], ids=["wavefront", "dense_reverse"])
def test_weight_only_grad_fastflow_unit(fp32_convs, dense):
    """dense_reverse keeps its dense forward inside the Function (same bits as without autograd); the weight gradient
    comes from the adjoint wavefront"""
    from fincflow_b200 import weight_grad_in_reverse
    from fincflow_b200.fastflow import FastFlowUnit

    torch.manual_seed(21)
    unit = FastFlowUnit(12, 12, (3, 3)).cuda()
    unit.dense_reverse = dense
    z = torch.randn(5, 12, 8, 8, device="cuda")
    r = torch.randn_like(z)
    with weight_grad_in_reverse():
        x = unit.reverse(z)
    assert x.requires_grad
    with torch.no_grad():
        want = unit.reverse(z)
    assert torch.equal(x, want)
    if dense:
        assert not torch.equal(x, _wavefront(unit, z))   # really the dense table, not the wavefront
    (gw,) = torch.autograd.grad((x * r).sum(), (unit.weight,))
    assert rel_err(npy(gw), npy(_ref_dw(z, unit.weight, list(ORDERS), r))) <= REL_TOL


def test_weight_only_grad_finc_stack(fp32_convs):
    from fincflow_b200 import weight_grad_in_reverse
    from fincflow_b200.stack import FincStack, LevelSpec

    torch.manual_seed(22)
    stack = FincStack([LevelSpec(12, 8, 8, 3, (3, 3))]).cuda()
    z = torch.randn(6, 12, 8, 8, device="cuda")
    r = torch.randn_like(z)
    assert not stack.reverse(z).requires_grad          # outside the context: a plain tensor, as before
    with weight_grad_in_reverse():
        x = stack.reverse(z)
    with torch.no_grad():
        assert torch.equal(x, stack.reverse(z))
    (gflat,) = torch.autograd.grad((x * r).sum(), (stack.flat,))
    flat = stack.flat.detach().double().clone().requires_grad_()
    xr = z.double()
    for u in reversed(range(3)):
        xr = ref_inverse(xr, stack.unit_weight(0, u, flat), list(ORDERS))
    (rflat,) = torch.autograd.grad((xr * r.double()).sum(), (flat,))
    assert rel_err(npy(gflat), npy(rflat)) <= REL_TOL


@pytest.mark.parametrize("C", [3, 12, 48])
def test_conv1x1_inverse_fn_grad(C):
    """the glue's W^-1 Function: forward = finc_slogdet_inverse_f32, gradient = float64 torch.linalg.inv autograd"""
    from fincflow_b200.flows import _InverseFn

    torch.manual_seed(C)
    W = (torch.linalg.qr(torch.randn(C, C))[0] + 0.1 * torch.randn(C, C)).cuda()
    R = torch.randn(C, C, device="cuda")
    Wf = W.clone().requires_grad_()
    Winv = _InverseFn.apply(Wf)
    (g,) = torch.autograd.grad((Winv * R).sum(), (Wf,))
    Wd = W.double().requires_grad_()
    (gd,) = torch.autograd.grad((torch.linalg.inv(Wd) * R.double()).sum(), (Wd,))
    assert rel_err(npy(Winv), npy(torch.linalg.inv(W.double()))) <= 1e-5
    assert rel_err(npy(g), npy(gd)) <= 1e-5


def test_quadrant_view_reverse_grad(fp32_convs):
    from fincflow_b200.fastflow import FastFlowUnit

    torch.manual_seed(8)
    unit = FastFlowUnit(12, 12, (3, 3)).cuda()
    z = torch.randn(4, 3, 8, 8, device="cuda", requires_grad=True)
    r = torch.randn_like(z)
    x = unit.conv_br.reverse(z)[0]
    gz, gw = torch.autograd.grad((x * r).sum(), (z, unit.weight))
    w_br = unit.weight.detach()[9:12].clone().requires_grad_()
    zr = z.detach().clone().requires_grad_()
    rz, rw = torch.autograd.grad((ref_inverse(zr.double(), w_br.double(), ["BR"]) * r.double()).sum(), (zr, w_br))
    assert rel_err(npy(gz), npy(rz)) <= REL_TOL
    assert rel_err(npy(gw[9:12]), npy(rw)) <= REL_TOL
    assert bool((gw[:9] == 0).all())


def test_finc_stack_reverse_grad(fp32_convs):
    from fincflow_b200.stack import FincStack, LevelSpec

    torch.manual_seed(9)
    stack = FincStack([LevelSpec(12, 8, 8, 3, (3, 3))]).cuda()
    z = torch.randn(6, 12, 8, 8, device="cuda", requires_grad=True)
    r = torch.randn_like(z)
    x = stack.reverse(z)
    with torch.no_grad():
        assert torch.equal(x, stack.reverse(z))
    gz, gflat = torch.autograd.grad((x * r).sum(), (z, stack.flat))
    flat = stack.flat.detach().double().clone().requires_grad_()
    zr = z.detach().double().clone().requires_grad_()
    xr = zr
    for u in reversed(range(3)):
        xr = ref_inverse(xr, stack.unit_weight(0, u, flat), list(ORDERS))
    rz, rflat = torch.autograd.grad((xr * r.double()).sum(), (zr, flat))
    assert rel_err(npy(gz), npy(rz)) <= REL_TOL
    assert rel_err(npy(gflat), npy(rflat)) <= REL_TOL


def test_fastflow_reverse_grad_whole_flow(fp32_convs, monkeypatch):
    """every parameter and every latent gets the gradient of the PyTorch-reference flow (FInC inverse: the float64
    fixed-point solve; ActNorm / Conv1x1 reverse: the unfused layers, torch.inverse and F.conv2d); none is None or
    zero.  Plain latents inside weight_grad_in_reverse give the parameters the same gradients."""
    from fincflow_b200 import weight_grad_in_reverse
    import fincflow_b200.fastflow as ffmod
    from fincflow_b200 import flows

    torch.manual_seed(10)
    model = flows.FastFlow(n_blocks=2, block_size=2, image_size=(1, 28, 28), final_steps=1, width=32,
                           actnorm=True).cuda()
    x = torch.randint(0, 256, (4, 1, 28, 28), device="cuda").float()
    with torch.no_grad():
        zs, _ = model(x)                                       # initialises ActNorm
        for m in model.modules():
            if isinstance(m, flows.Coupling):                  # Conv2dZero starts at 0: coupling grads would be 0
                m.net[4].weight.normal_(0, 0.02)
                m.net[4].bias.normal_(0, 0.1)
                m.net[4].logs.normal_(0, 0.1)
    zs = [torch.randn_like(z) for z in zs]
    params = [p for p in model.parameters()]
    outs = {}
    with weight_grad_in_reverse():
        img0 = model.reverse(zs=zs, quantize=False)
        w8 = torch.randn(img0.shape, device="cuda", generator=torch.Generator(device="cuda").manual_seed(11))
        plain = torch.autograd.grad((img0 * w8).sum(), params)
    for name in ("ours", "ref"):
        if name == "ref":
            monkeypatch.setattr(ffmod, "finc_inverse",     # (FastFlowUnit.reverse: G = 4, the unit's orders)
                                lambda z, w, G=4, orders=None, dense=None: ref_inverse(
                                    z.double(), w.double(), ORDERS).float())
            monkeypatch.setattr(flows.GlowStep, "fused", False)
        lat = [z.clone().requires_grad_() for z in zs]
        img = model.reverse(zs=lat, quantize=False)
        r = torch.Generator(device="cuda").manual_seed(11)
        w8 = torch.randn(img.shape, device="cuda", generator=r)
        outs[name] = (img, torch.autograd.grad((img * w8).sum(), params + lat, allow_unused=True))
    img, ours = outs["ours"]
    _, ref = outs["ref"]
    assert rel_err(npy(img), npy(outs["ref"][0])) <= 1e-4
    for (pname, _), a, b in zip(list(model.named_parameters()) + [(f"zs[{i}]", None) for i in range(len(zs))],
                                ours, ref):
        assert a is not None and b is not None, pname
        assert float(a.abs().max()) > 0, pname
        assert rel_err(npy(a), npy(b)) <= 1e-4, (pname, rel_err(npy(a), npy(b)))
    for (pname, _), a, b in zip(model.named_parameters(), plain, ref):
        assert rel_err(npy(a), npy(b)) <= 1e-4, ("plain latents", pname, rel_err(npy(a), npy(b)))
    # the default keeps the floor (integer image, zero gradient)
    with torch.no_grad():
        q = model.reverse(zs=zs)
    assert torch.equal(q, q.floor())
