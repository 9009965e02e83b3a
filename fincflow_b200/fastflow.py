"""FastFlowUnit -- four corner-padded FInC convolutions on the four channel quarters, fused.

Drop-in for the reference's fastflow/fastflow.py:13-100: same constructor
(`FastFlowUnit(in_channels, out_channels, kernel_size)`, out_channels ignored,
in_channels % 4 == 0), same sub-module names (`conv_tl/tr/bl/br`, each exposing
`.conv.weight`, `.mask`, `.order`, `reset_gradients()`), same state-dict keys
(`conv_tl.conv.weight`, ...), `forward(x, context=None) -> (out, logdet)`,
`reverse(x, context=None) -> out` (bare tensor, fastflow.py:100; differentiable, which the reference's reverse is not: see
ops.finc_inverse).

B200-first differences (results identical):
  * the four weights live in ONE packed parameter `weight` [4*Cq, Cq, kH, kW] in their
    stored (flipped) orientation, so forward / backward / inverse are one kernel launch each
    over the whole [B, 4Cq, H, W] tensor -- no chunk, pad, flip, cat or zeros_like copies;
  * the gradient mask is applied by the weight-gradient kernel (mask_in_backward=True) or
    by one launch in reset_gradients(), never by uploading a CPU mask.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from . import _native
from .layers.conv import ORDERS, finc_grad_mask, init_finc_weight_
from .ops import finc_conv, finc_inverse


class _ConvHandle(nn.Module):
    """`.weight` view of one quadrant, so `unit.conv_tl.conv.weight` keeps working."""

    def __init__(self, unit, q):
        super().__init__()
        object.__setattr__(self, "_unit", unit)  # not registered: avoids a module cycle
        self._q = q

    @property
    def weight(self):
        u = self._unit
        return u.weight[self._q * u.cq:(self._q + 1) * u.cq]

    @property
    def bias(self):
        return None


class _QuadrantView(nn.Module):
    """Stands where the reference has a PaddedConv2d sub-module (fastflow.py:24-27)."""

    def __init__(self, unit, q):
        super().__init__()
        object.__setattr__(self, "_unit", unit)
        self._q = q
        self.order = ORDERS[q]
        self.kernel_size = unit.kernel_size
        self.conv = _ConvHandle(unit, q)
        self.mask = finc_grad_mask(unit.cq, unit.kernel_size, self.order)

    def get_mask(self):
        return self.mask

    def reset_gradients(self):
        if self._q == 0:  # one launch masks all four quadrants
            self._unit.reset_gradients()

    def forward(self, x, context=None):
        u = self._unit
        w = self.conv.weight.contiguous()
        z, _ = finc_conv(x, w, 1, _native.pack_orders([self.order]), u.mask_in_backward, False)
        return z, 0.0

    def reverse(self, x, context=None):
        w = self.conv.weight.contiguous()
        return finc_inverse(x, w, 1, _native.pack_orders([self.order])), 0


class FastFlowUnit(nn.Module):
    def __init__(self, in_channels, out_channels=None, kernel_size=(3, 3), mask_in_backward=False,
                 logdet_mode="float"):
        super().__init__()
        if isinstance(kernel_size, int) or len(kernel_size) == 1:
            k = kernel_size if isinstance(kernel_size, int) else kernel_size[0]
            kernel_size = (k, k)
        assert in_channels % 4 == 0, "Input channels have to be a multiple of 4"
        self.in_channels = in_channels
        self.cq = in_channels // 4
        self.kernel_size = tuple(kernel_size)
        self.mask_in_backward = mask_in_backward
        self.logdet_mode = logdet_mode
        self.weight = nn.Parameter(torch.empty(4 * self.cq, self.cq, *self.kernel_size))
        self.reset_parameters()
        self.conv_tl = _QuadrantView(self, 0)
        self.conv_tr = _QuadrantView(self, 1)
        self.conv_bl = _QuadrantView(self, 2)
        self.conv_br = _QuadrantView(self, 3)
        self._register_state_dict_hook(_split_weight_hook)
        self._register_load_state_dict_pre_hook(_merge_weight_hook, with_module=True)

    def reset_parameters(self):
        for q, order in enumerate(ORDERS):  # same RNG order as the reference: TL, TR, BL, BR
            init_finc_weight_(self.weight.data[q * self.cq:(q + 1) * self.cq], order)

    def reset_gradients(self):
        g = self.weight.grad
        if g is not None and not self.mask_in_backward:
            _native.apply_grad_mask_(g, 4, _native.ORDERS_UNIT)

    def forward(self, x, context=None):
        want = self.logdet_mode == "tensor"
        if torch.is_grad_enabled() and self.weight.requires_grad:
            self._dense_key = None   # a training forward: the dense-inverse table may be stale after the next update
        z, logdet = finc_conv(x, self.weight, 4, _native.ORDERS_UNIT, self.mask_in_backward, want)
        return z, (logdet if want else 0.0)  # reference: 0.0 + 0.0 + 0.0 + 0.0 (fastflow.py:34-50)

    # opt-in (class or instance attribute): sampling with FIXED weights runs x = L^-1 z as one block-diagonal
    # tensor-core GEMM when the tile is small (n = Cq*H*W <= 1024); L^-1 is cached per weight version.  Pays for
    # 4x4 / 8x8 tiles and k=5 (2-11x over the wavefront kernel at B >= 1024), not for 16x16 tiles at k=3.
    dense_reverse = False

    def _dense_table(self, H, W):
        key = (self.weight.data_ptr(), self.weight._version, H, W)
        if getattr(self, "_dense_key", None) != key:
            self._dense_blob = _native.inverse_dense_prepare(self.weight.detach().contiguous(), H, W)
            self._dense_key = key
        return self._dense_blob

    def reverse(self, x, context=None):
        if (self.dense_reverse and x.is_cuda and not (torch.is_grad_enabled() and x.requires_grad)
                and _native.inverse_dense_bytes(4, self.cq, x.shape[2], x.shape[3]) > 0):
            # (a graph for the weight alone -- weight_grad_in_reverse -- keeps the dense forward; its backward is the
            # adjoint wavefront)
            return finc_inverse(x, self.weight, 4, _native.ORDERS_UNIT,
                                dense=self._dense_table(int(x.shape[2]), int(x.shape[3])))
        return finc_inverse(x, self.weight, 4, _native.ORDERS_UNIT)

    def logdet(self, x, context=None):
        if self.logdet_mode == "tensor":
            return _native.logdet(self.weight.detach(), x.shape[0], x.shape[2], x.shape[3])
        return 0.0


_QNAMES = ("conv_tl", "conv_tr", "conv_bl", "conv_br")


def _split_weight_hook(module, state_dict, prefix, local_metadata):
    """emit the reference's keys `<prefix>conv_{tl,tr,bl,br}.conv.weight`"""
    w = state_dict.pop(prefix + "weight")
    for q, name in enumerate(_QNAMES):
        state_dict[f"{prefix}{name}.conv.weight"] = w[q * module.cq:(q + 1) * module.cq].clone()


def _merge_weight_hook(module, state_dict, prefix, local_metadata, strict, missing_keys, unexpected_keys,
                       error_msgs):
    keys = [f"{prefix}{name}.conv.weight" for name in _QNAMES]
    if all(k in state_dict for k in keys):
        state_dict[prefix + "weight"] = torch.cat([state_dict.pop(k) for k in keys], dim=0)


def clear_grad(module):
    """`model.apply(clear_grad)` of the reference (train/experiment.py:16-18,250)."""
    from .layers.conv import PaddedConv2d

    if isinstance(module, (FastFlowUnit, PaddedConv2d)):
        module.reset_gradients()
