"""CPU checks of the differentiable sampling direction: argument validation of finc_inverse_adjoint_f32 (it happens
before any CUDA call) and Preprocess.reverse without the final floor."""
import ctypes

import pytest
import torch


@pytest.fixture(scope="module")
def lib():
    from fincflow_b200 import _native, build

    build.build()
    return _native.load()


def test_inverse_adjoint_argument_validation(lib):
    from fincflow_b200 import _native

    f = lib.finc_inverse_adjoint_f32
    w = ctypes.c_void_p(256)   # never dereferenced: every call below returns before touching the device
    assert f(None, None, None, 1, 4, 3, 8, 8, 3, 3, 0xE4, 0, None) == -1                   # null weights
    assert f(None, w, None, 1, 4, 3, 8, 8, 3, 3, 0xE4, 0, None) == -1                      # null dx / dz
    assert f(None, w, None, 1, 17, 3, 8, 8, 3, 3, 0, 0, None) == -1                        # G > 16
    assert f(None, w, None, -1, 4, 3, 8, 8, 3, 3, 0xE4, 0, None) == -1                     # B < 0
    assert f(None, w, None, 1, 4, 0, 8, 8, 3, 3, 0xE4, 0, None) == -1                      # C = 0
    assert f(None, w, None, 0, 4, 3, 8, 8, 3, 3, 0xE4, 0, None) == 0                       # B = 0: no-op
    assert f(w, w, w, 1, 4, 3, 8, 8, 3, 3, 0xE4, _native.FLAG_PREPARED, None) == -3        # no prepared tables
    assert _native.FLAG_NEGATE == 4096


def test_inverse_adjoint_rejects_cpu_tensors(lib):
    from fincflow_b200 import _native
    from fincflow_b200.ops import finc_inverse

    w = torch.zeros(12, 3, 3, 3, requires_grad=True)
    with pytest.raises(_native.FincNativeError):
        _native.inverse_adjoint(torch.randn(2, 12, 4, 4), w.detach())
    with pytest.raises(_native.FincNativeError):
        finc_inverse(torch.randn(2, 12, 4, 4, requires_grad=True), w)


def test_preprocess_reverse_without_floor():
    from fincflow_b200.flows import Preprocess

    pre = Preprocess((3, 4, 4))
    torch.manual_seed(0)
    y = torch.randn(2, 3, 4, 4, requires_grad=True)
    cont = pre.reverse(y, quantize=False)
    a = pre.alpha
    want = (torch.sigmoid(y) / (1 - 2 * a) - a) * 256
    assert torch.allclose(cont, want, rtol=1e-6, atol=1e-4)
    assert torch.equal(pre.reverse(y.detach()), cont.detach().floor())    # default: the integer image
    (g,) = torch.autograd.grad(cont.sum(), (y,))
    assert bool((g > 0).all())
