"""CPU checks of the differentiable coupling reverse and FastFlow.sample_with_log_prob: the C ABI flag, argument
validation of finc_coupling_backward_f32 (it happens before any CUDA call), the public signatures, and the reverse
log-determinants of the PyTorch formulas (Coupling, Preprocess) on CPU tensors."""
import inspect
import os
import re

import pytest
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from fincflow_b200 import _native, build

    build.build()
    return _native.load()


def header_flags():
    with open(os.path.join(REPO, "include", "fincflow_b200.h")) as f:
        return {m.group(1): int(m.group(2)) for m in re.finditer(r"#define FINC_FLAG_(\w+) (\d+)u", f.read())}


def test_coupling_reverse_flag_matches_header():
    from fincflow_b200 import _native

    flags = header_flags()
    assert flags["COUPLING_REVERSE"] == _native.FLAG_COUPLING_REVERSE == 8192
    others = [v for k, v in flags.items() if k != "COUPLING_REVERSE"]
    assert all(v & 8192 == 0 for v in others)                # a bit of its own


def test_coupling_backward_reverse_argument_validation(lib):
    from fincflow_b200 import _native

    f = lib.finc_coupling_backward_f32
    args = [None] * 6 + [0] + [None] * 8 + [2, 12, 8, 8, 128]
    assert f(*args, _native.FLAG_COUPLING_REVERSE, None) == -1          # null pointers: FINC_E_BADARG
    assert f(*args, 0, None) == -1


def test_public_signatures():
    from fincflow_b200.flows import FastFlow

    assert str(inspect.signature(FastFlow.reverse)) == "(self, n_samples=1, zs=None, z_std=1.0, quantize=True)"
    assert str(inspect.signature(FastFlow.sample)) == "(self, n_samples, context=None)"
    assert str(inspect.signature(FastFlow.sample_with_log_prob)) == "(self, n_samples=1, zs=None)"


def test_coupling_reverse_logdet_formulas():
    """CPU tensors keep the PyTorch formulas: the reverse log-det is minus the forward's at the reconstructed input"""
    from fincflow_b200.flows import Coupling

    torch.manual_seed(0)
    cp = Coupling((12, 6, 6), width=32).double()
    with torch.no_grad():
        cp.net[4].weight.normal_(0, 0.02)
        cp.net[4].bias.normal_(0, 0.1)
        cp.net[4].logs.normal_(0, 0.1)
    y = torch.randn(3, 12, 6, 6, dtype=torch.float64)
    x, ld = cp.reverse_and_logdet(y)
    assert torch.equal(x, cp.reverse(y))
    y2, ld_fwd = cp(x)
    assert torch.allclose(y2, y, atol=1e-12) and torch.allclose(ld, -ld_fwd, atol=1e-12)
    assert x.requires_grad and ld.requires_grad        # parameters require grad: a graph, as the formulas give
    with torch.no_grad():
        assert not cp.reverse_and_logdet(y)[1].requires_grad


def test_preprocess_reverse_logdet():
    """minus the Normalization and LogitTransform terms of the forward at the image the reverse returns"""
    from fincflow_b200.flows import Preprocess

    pre = Preprocess((3, 4, 4))
    torch.manual_seed(1)
    z = torch.randn(2, 3, 4, 4, dtype=torch.float64, requires_grad=True)
    img, ld = pre.reverse_and_logdet(z)
    assert torch.equal(img, pre.reverse(z, quantize=False))
    pre.layers[0].fixed_noise = torch.zeros_like(img)
    z2, ld_fwd = pre(img.detach())
    assert torch.allclose(z2, z.detach(), atol=1e-9) and torch.allclose(ld.detach(), -ld_fwd, rtol=1e-12)
    (g,) = torch.autograd.grad(ld.sum(), (z,))
    assert bool(torch.isfinite(g).all()) and float(g.abs().max()) > 0
