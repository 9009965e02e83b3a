"""GPU vs GPU: our inverse kernels against the REFERENCE's own CUDA extension
(fastflow/utils/fastflow_cuda_inverse/cinc_cuda_kernel_level{1,2}.cu, compiled unmodified for sm_100 by
oracle/build_ref_cuda.py into oracle/_ref/), driven exactly like the reference's call sites
(FastFlowUnit.reverse_level2, fastflow/fastflow.py:78-100; PaddedConv2d.reverse_cuda,
layers/conv.py:191-218).  north_star: "Outputs must match the reference's own PyTorch/cinc_cuda
implementation ... <= 1e-5 relative, <= 1e-4 max-abs round trip".

The reference kernel launches `threads(B)` per block, so B <= 1024, and maps diagonals assuming
H <= W (cinc_cuda_kernel_level2.cu:90-112); the cases stay inside that envelope.

The live comparison needs the reference's extensions, built only from a reference checkout
(FINCFLOW_REFERENCE).  Without them each test checks the same kernels against the reference's
stored outputs in tests/golden (its own FastFlowUnit / PaddedConv2d reverse, make_golden.py) at the
stored case closest to the live one: same channels and kernel, and the same image size where one
was stored."""
import numpy as np
import pytest
import torch

from conftest import rel_err

pytestmark = pytest.mark.gpu


def _ref(level):
    """the reference's compiled extension, or None when it was not built"""
    from oracle import build_ref_cuda

    return build_ref_cuda.load(level)


def _elementwise_ok(a, b, rtol=1e-5):
    """|a - b| <= rtol * (|b| + 0.1 max|b|): element-wise relative with an absolute floor of 1e-6 max|b|
    (two fp32 evaluations of the recurrence in different orders differ by a few 1e-7 absolute on
    elements that cancel to ~0, whatever their magnitude)"""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return bool((np.abs(a - b) <= rtol * (np.abs(b) + 1e-1 * np.abs(b).max())).all())


def _reference_unit_reverse(ext, unit, z):
    """fastflow/fastflow.py:78-100, line by line, on the reference's own extension"""
    k_tl = unit.conv_tl.conv.weight.data
    k_tr = torch.flip(unit.conv_tr.conv.weight.data, [3])
    k_bl = torch.flip(unit.conv_bl.conv.weight.data, [2])
    k_br = torch.flip(unit.conv_br.conv.weight.data, [2, 3])
    kernel = torch.cat([k_tl, k_tr, k_bl, k_br], dim=0).contiguous()
    o_tl, o_tr, o_bl, o_br = torch.chunk(z, 4, dim=1)
    x = torch.cat([o_tl, torch.flip(o_tr, [3]), torch.flip(o_bl, [2]), torch.flip(o_br, [2, 3])], dim=1).contiguous()
    y = torch.zeros_like(x)
    y = ext.inverse(x, kernel, y)[0]
    o_tl, o_tr, o_bl, o_br = torch.chunk(y, 4, dim=1)
    return torch.cat([o_tl, torch.flip(o_tr, [3]), torch.flip(o_bl, [2]), torch.flip(o_br, [2, 3])], dim=1)


# unit shapes of the BASELINE configs (SURVEY.md section 8 shape table), B <= 1024
UNIT_CASES = [
    (64, 4, 14, 14, 3),                                                       # cfg1 / cfg2 level 0
    (128, 8, 7, 7, 3),                                                        # cfg2 final level
    (256, 12, 16, 16, 3), (256, 24, 8, 8, 3), (256, 48, 4, 4, 3),             # cfg3
    (512, 12, 16, 16, 3),                                                     # cfg4 (per-GPU batch)
    (64, 12, 32, 32, 3), (64, 24, 16, 16, 3), (64, 48, 8, 8, 3), (64, 96, 4, 4, 3),    # cfg5, k = 3
    (32, 12, 32, 32, 5), (32, 48, 8, 8, 5), (32, 96, 4, 4, 5),                # cfg5, k = 5
    (3, 8, 5, 9, 3), (1024, 4, 6, 6, 3),                                      # H < W, the reference's batch limit
]


# UNIT_CASES -> the stored reference case used without the extension
STORED_UNIT = {
    (4, 14, 14, 3): "unit_C1_H14_W14_k3x3_B2", (8, 7, 7, 3): "unit_C2_H7_W7_k3x3_B2",
    (12, 16, 16, 3): "unit_C3_H16_W16_k3x3_B2", (24, 8, 8, 3): "unit_C6_H8_W8_k3x3_B2",
    (48, 4, 4, 3): "unit_C12_H4_W4_k3x3_B2", (12, 32, 32, 3): "unit_C3_H32_W32_k3x3_B1",
    (24, 16, 16, 3): "unit_C6_H16_W16_k3x3_B1", (48, 8, 8, 3): "unit_C12_H8_W8_k3x3_B1",
    (96, 4, 4, 3): "unit_C24_H4_W4_k3x3_B1", (12, 32, 32, 5): "unit_C3_H16_W16_k5x5_B1",
    (48, 8, 8, 5): "unit_C12_H4_W4_k5x5_B1", (96, 4, 4, 5): "unit_C24_H4_W4_k5x5_B1",
    (8, 5, 9, 3): "unit_C2_H5_W9_k2x3_B2", (4, 6, 6, 3): "unit_C1_H4_W4_k2x2_B3",
}


def _check_stored_unit(golden, name):
    """our unit inverse against the reference's stored reverse of the same weights and latents"""
    from fincflow_b200.fastflow import FastFlowUnit

    c = golden.case(name)
    C, k = c["w"].shape[0], tuple(c["w"].shape[2:])
    unit = FastFlowUnit(C, C, k).cuda()
    with torch.no_grad():
        unit.weight.copy_(torch.from_numpy(c["w"]))
        ours = unit.reverse(torch.from_numpy(c["zs"]).cuda()).cpu().numpy()
        rt = unit.reverse(torch.from_numpy(c["z"]).cuda()).cpu().numpy()
    assert rel_err(ours, c["x_from_zs"]) <= 1e-5
    assert _elementwise_ok(ours, c["x_from_zs"])
    assert np.abs(rt - c["x"]).max() <= 1e-4 and np.abs(c["x_rt"] - c["x"]).max() <= 1e-4


@pytest.mark.parametrize("case", UNIT_CASES)
def test_unit_inverse_matches_reference_cuda_kernel(case, golden):
    from fincflow_b200.fastflow import FastFlowUnit

    ext = _ref(2)
    B, C, H, W, k = case
    if ext is None:
        _check_stored_unit(golden, STORED_UNIT[(C, H, W, k)])
        return
    torch.manual_seed(B + C + H)
    unit = FastFlowUnit(C, C, (k, k)).cuda()
    x = torch.randn(B, C, H, W, device="cuda")
    with torch.no_grad():
        z, _ = unit(x)
        ours = unit.reverse(z)
        theirs = _reference_unit_reverse(ext, unit, z)
    assert rel_err(ours.cpu().numpy(), theirs.cpu().numpy()) <= 1e-5
    assert _elementwise_ok(ours.cpu().numpy(), theirs.cpu().numpy())
    assert float((ours - x).abs().max()) <= 1e-4 and float((theirs - x).abs().max()) <= 1e-4
    # sampling input (z ~ N(0, 1), not a forward image)
    zs = torch.randn(B, C, H, W, device="cuda")
    with torch.no_grad():
        a, b = unit.reverse(zs), _reference_unit_reverse(ext, unit, zs)
    assert rel_err(a.cpu().numpy(), b.cpu().numpy()) <= 1e-5


@pytest.mark.parametrize("order", ["TL", "TR", "BL", "BR"])
def test_single_conv_inverse_matches_reference_level1_kernel(order, golden):
    """PaddedConv2d.reverse_cuda (layers/conv.py:191-218): flips to TL form, level-1 extension, flips back"""
    from fincflow_b200.layers.conv import PaddedConv2d

    ext = _ref(1)
    if ext is None:   # the reference's stored PaddedConv2d reverse at the same shape
        c = golden.case(f"conv_{order}_C4_H14_W14_k3x3_B2")
        conv = PaddedConv2d(4, 4, (3, 3), order=order).cuda()
        with torch.no_grad():
            conv.conv.weight.copy_(torch.from_numpy(c["w"]))
            ours, _ = conv.reverse(torch.from_numpy(c["zs"]).cuda())
        assert rel_err(ours.cpu().numpy(), c["x_from_zs"]) <= 1e-5
        assert _elementwise_ok(ours.cpu().numpy(), c["x_from_zs"])
        return
    torch.manual_seed(11)
    conv = PaddedConv2d(4, 4, (3, 3), order=order).cuda()
    x = torch.randn(64, 4, 14, 14, device="cuda")
    dims = {"TL": [], "TR": [3], "BL": [2], "BR": [2, 3]}[order]
    with torch.no_grad():
        z, _ = conv(x)
        ours, _ = conv.reverse(z)
        kern = (torch.flip(conv.conv.weight.data, dims) if dims else conv.conv.weight.data).contiguous()
        zin = (torch.flip(z, dims) if dims else z).contiguous()
        y = ext.inverse(zin, kern, torch.zeros_like(zin))[0]
        theirs = torch.flip(y, dims) if dims else y
    assert rel_err(ours.cpu().numpy(), theirs.cpu().numpy()) <= 1e-5
    assert _elementwise_ok(ours.cpu().numpy(), theirs.cpu().numpy())
    assert float((ours - x).abs().max()) <= 1e-4


def test_reference_forward_path_on_gpu_matches():
    """the reference's forward is F.pad + conv2d (layers/conv.py:102-107); with TF32 off on the GPU
    it must agree with our fused kernel (north_star: "reference's own PyTorch ... implementation")"""
    import torch.nn.functional as F

    from fincflow_b200.fastflow import FastFlowUnit

    old = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        torch.manual_seed(2)
        unit = FastFlowUnit(24, 24, (3, 3)).cuda()
        x = torch.randn(256, 24, 8, 8, device="cuda", requires_grad=True)
        z, _ = unit(x)
        dz = torch.randn_like(z)
        z.backward(dz)
        xr = x.detach().clone().requires_grad_(True)
        pads = {"tl": (2, 0, 2, 0), "tr": (0, 2, 2, 0), "bl": (2, 0, 0, 2), "br": (0, 2, 0, 2)}
        outs = []
        ws = []
        for q, xq in zip(("tl", "tr", "bl", "br"), torch.chunk(xr, 4, dim=1)):
            w = getattr(unit, f"conv_{q}").conv.weight.detach().clone().requires_grad_(True)
            ws.append(w)
            outs.append(F.conv2d(F.pad(xq, pads[q], "constant", 0), w))
        zr = torch.cat(outs, dim=1)
        zr.backward(dz)
        assert rel_err(z.detach().cpu().numpy(), zr.detach().cpu().numpy()) <= 1e-5
        assert rel_err(x.grad.cpu().numpy(), xr.grad.cpu().numpy()) <= 1e-5
        raw = torch.cat([w.grad for w in ws], 0)
        unit2_grad = unit.weight.grad.clone()
        unit.reset_gradients()
        masks = torch.cat([getattr(unit, f"conv_{q}").mask for q in ("tl", "tr", "bl", "br")], 0).cuda()
        assert rel_err(unit.weight.grad.cpu().numpy(), (raw * masks).cpu().numpy()) <= 1e-5
        assert rel_err(unit2_grad.cpu().numpy(), raw.cpu().numpy()) <= 1e-5   # raw before reset_gradients()
    finally:
        torch.backends.cudnn.allow_tf32 = old
