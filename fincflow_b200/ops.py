"""torch.autograd glue over the C ABI: Functions for the fused FInC convolution and its inverse."""
from __future__ import annotations

import contextlib
import threading

import torch

from . import _native

_tls = threading.local()


@contextlib.contextmanager
def weight_grad_in_reverse(enabled=True):
    """Inside this context (this thread) every reverse records a graph when autograd is on and its latent OR its
    weights require grad -- e.g. training a flow on samples of plain noise (reverse-KL: `stack.reverse(torch.randn(...))`
    with a loss on the weights).  Outside it, a reverse records only when its latent requires grad: a reverse of a
    detached latent returns a plain tensor even though the weights are parameters, as it always has, so sampling code
    under grad mode that hands the samples to numpy keeps working.  Output values are the same bits either way."""
    old = getattr(_tls, "weight_grad", False)
    _tls.weight_grad = bool(enabled)
    try:
        yield
    finally:
        _tls.weight_grad = old


def reverse_records(latent, *params):
    """whether a reverse step records a graph (see weight_grad_in_reverse)"""
    if not torch.is_grad_enabled():
        return False
    if latent.requires_grad:
        return True
    return getattr(_tls, "weight_grad", False) and any(p.requires_grad for p in params)


class FincConvFunction(torch.autograd.Function):
    """z, logdet = FInC conv of x [B, G*C, H, W] with packed weights [G*C, C, kH, kW].

    forward  -> finc_forward_f32            (reference: layers/conv.py:102-107, fastflow.py:31-50)
    backward -> finc_backward_input_f32 + finc_backward_weight_f32
                (reference: cuDNN dgrad/wgrad via autograd; mask: layers/conv.py:98-99)
    `mask_dw=True` applies the FInC gradient mask inside the weight-gradient kernel;
    `False` returns the raw gradient exactly as autograd does in the reference, to be
    masked later by reset_gradients()/clear_grad (train/experiment.py:246-250 masks AFTER
    the optional gradient clipping).
    """

    @staticmethod
    def forward(ctx, x, w, G, orders, mask_dw, want_logdet):
        z, logdet = _native.forward(x, w, G, orders, want_logdet)
        ctx.save_for_backward(x, w)
        ctx.G, ctx.orders, ctx.mask_dw = G, orders, mask_dw
        if logdet is None:
            logdet = x.new_zeros(())
        ctx.mark_non_differentiable(logdet)
        return z, logdet

    @staticmethod
    def backward(ctx, dz, _dlogdet):
        x, w = ctx.saved_tensors
        dx = dw = None
        if ctx.needs_input_grad[0]:
            dx = _native.backward_input(dz, w, ctx.G, ctx.orders)
        if ctx.needs_input_grad[1]:
            flags = 0 if ctx.mask_dw else _native.FLAG_NO_MASK
            dw = _native.backward_weight(dz, x, (w.shape[2], w.shape[3]), ctx.G, ctx.orders, flags)
        return dx, dw, None, None, None, None


def finc_conv(x, w, G=4, orders=_native.ORDERS_UNIT, mask_dw=False, want_logdet=True):
    z, logdet = FincConvFunction.apply(x, w, G, orders, mask_dw, want_logdet)
    return z, (logdet if want_logdet else None)


class FincInverseFunction(torch.autograd.Function):
    """x = A(w)^-1 z, the FInC inverse (sampling direction), differentiable in z and w.

    forward  -> finc_inverse_f32 (or, given `dense`, FastFlowUnit.dense_reverse's table of the same w:
                finc_inverse_dense_f32)
    backward -> g = A^-T dx by finc_inverse_adjoint_f32 (one launch: the same wavefront swept from the opposite
                corner), then dz = g and dw = -wgrad(g, x) by finc_backward_weight_f32 with FINC_FLAG_NEGATE, always
                masked: the inverse never reads w[o, i>=o, corner], so their derivative is 0 whatever the layer's
                mask_in_backward says (reset_gradients re-masks idempotently).
    """

    @staticmethod
    def forward(ctx, z, w, G, orders, dense=None):
        x = _native.inverse(z, w, G, orders) if dense is None else _native.inverse_dense(z.contiguous(), dense, G)
        ctx.save_for_backward(x, w)
        ctx.G, ctx.orders = G, orders
        return x

    @staticmethod
    def backward(ctx, dx):
        x, w = ctx.saved_tensors
        g = _native.inverse_adjoint(dx, w, ctx.G, ctx.orders)
        dw = None
        if ctx.needs_input_grad[1]:
            dw = _native.backward_weight(g, x, (w.shape[2], w.shape[3]), ctx.G, ctx.orders, _native.FLAG_NEGATE)
        return (g if ctx.needs_input_grad[0] else None), dw, None, None, None


def finc_inverse(z, w, G=4, orders=_native.ORDERS_UNIT, dense=None):
    """x with forward(x) == z.

    Differentiable in z and w whenever it records a graph (reverse_records: autograd on and z requires grad, or w
    does inside weight_grad_in_reverse): it is then FincInverseFunction, whose backward is one adjoint wavefront
    launch (+ one weight-gradient launch when w needs a gradient).  Otherwise the result is a plain tensor.  x is bit
    for bit the same either way.  `dense`: a dense-inverse table of w (FastFlowUnit.dense_reverse) that the forward
    runs instead of the wavefront.
    """
    if reverse_records(z, w):
        return FincInverseFunction.apply(z, w, G, orders, dense)
    with torch.no_grad():
        if dense is not None:
            return _native.inverse_dense(z.contiguous(), dense, G)
        return _native.inverse(z, w, G, orders)
