"""Multi-scale FInC flows (MNIST / CIFAR-10 / ImageNet32 / ImageNet64 shapes).

The model definition of the reference's maintained scripts
(fastflow/fastflow_{mnist,cifar,imagenet,imagenet64}_multi_gpu.py: Preprocess, GlowStep,
FastFlowStep, FastFlowLevel, FastFlow) rebuilt around the B200 FInC kernels:

  * `FastFlowUnit` and `Squeeze` run on the sm_100a kernels behind the C ABI;
  * the Glow glue (ActNorm, Conv1x1, Coupling, SplitPrior, preprocessing) stays plain PyTorch
    (SURVEY.md section 8f: "next" rows) with the reference's formulas
    (layers/actnorm.py:14-64, conv1x1.py:9-43, coupling.py:9-105, normalize.py:18-31,
    transforms.py:11-18, dequantize.py:13-19);
  * the base density is the closed form -0.5|z|^2 - d/2 log(2 pi) on the input's own device
    instead of a dense d x d MultivariateNormal pinned to cuda:0 (train/losses.py:17-45).

Sub-module and parameter names are the reference's, so its checkpoints load with
`load_state_dict` (e.g. `fastflow_levels.0.fastflow_level.1.fastflow_step.fastflow_unit.conv_tl.conv.weight`,
`...glow_unit.glow_step.conv1x1.W`, `...coupling.net.4.logs`).
"""
from __future__ import annotations

import math
from collections import OrderedDict

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _native
from .fastflow import FastFlowUnit
from .ops import reverse_records
from .layers.flowlayer import FlowLayer, PreprocessingFlowLayer


# ---------------------------------------------------------------------------------------------
# glue layers
# ---------------------------------------------------------------------------------------------
class _SqueezeFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        return _native.squeeze(x)

    @staticmethod
    def backward(ctx, g):
        return _native.unsqueeze(g)


class _UnsqueezeFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        return _native.unsqueeze(x)

    @staticmethod
    def backward(ctx, g):
        return _native.squeeze(g)


class Squeeze(FlowLayer):
    """space-to-depth, out channel 4c + 2dh + dw (layers/squeeze.py:5-39) on finc_squeeze_f32"""

    def forward(self, input, context=None):
        return _SqueezeFn.apply(input), self.logdet(input, context)

    def reverse(self, input, context=None):
        return _UnsqueezeFn.apply(input)

    def logdet(self, input, context=None):
        return input.new_zeros(len(input))


class Dequantization(PreprocessingFlowLayer):
    """x + u, u ~ U[0,1) (layers/dequantize.py:13-19).  `fixed_noise` pins u for parity tests
    (the reference draws it from the CPU generator on every forward)."""

    def __init__(self):
        super().__init__()
        self.fixed_noise = None

    def forward(self, input, context=None):
        u = self.fixed_noise if self.fixed_noise is not None else torch.rand_like(input)
        return input + u.to(input.device), input.new_zeros(len(input))

    def reverse(self, input, context=None):
        return input.floor()

    def logdet(self, input, context=None):
        return input.new_zeros(len(input))


class Normalization(PreprocessingFlowLayer):
    def __init__(self, translation, scale):
        super().__init__()
        self.register_buffer("translation", torch.Tensor([translation]))
        self.register_buffer("scale", torch.Tensor([scale]))

    def forward(self, input, context=None):
        return (input - self.translation) / self.scale, self.logdet(input, context)

    def reverse(self, input, context=None):
        return input * self.scale + self.translation

    def logdet(self, input, context=None):
        N, C, H, W = input.size()
        return (-C * H * W * torch.log(self.scale)).expand(N)


class LogitTransform(PreprocessingFlowLayer):
    def forward(self, input, context=None):
        return torch.log(input) - torch.log(1 - input), self.logdet(input, context)

    def reverse(self, input, context=None):
        return torch.sigmoid(input)

    def logdet(self, input, context=None):
        return (-torch.log(input) - torch.log(1 - input)).flatten(start_dim=1).sum(-1)


class ActNorm(FlowLayer):
    """layers/actnorm.py:14-64.  `sync_init`: under torch.distributed the data-dependent initialisation uses
    the moments of the GLOBAL batch (all-reduced count / sum / sum of squares), so that every replica of a
    data-parallel job starts with the same translation / log_scale (the reference initialises from
    replica 0's shard inside nn.DataParallel: layers/actnorm.py:17-23)."""

    sync_init = True

    def __init__(self, n_dims):
        super().__init__()
        self.n_dims = n_dims
        self.translation = nn.Parameter(torch.zeros(n_dims))
        self.log_scale = nn.Parameter(torch.zeros(n_dims))
        self.register_buffer("initialized", torch.tensor(0))
        self._ready = False   # host copy of `initialized`: checking the device buffer costs a stream sync per call

    def is_initialized(self):
        if not self._ready:
            self._ready = bool(self.initialized)
        return self._ready

    @staticmethod
    def _moments(input):
        dims = [0, 2, 3]
        import torch.distributed as dist

        if ActNorm.sync_init and dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            n = torch.tensor([float(input.numel() // input.shape[1])], device=input.device, dtype=torch.float64)
            s = input.double().sum(dim=dims)
            ss = input.double().pow(2).sum(dim=dims)
            packed = torch.cat([n, s, ss])
            dist.all_reduce(packed)
            n, s, ss = packed[0], packed[1:1 + s.numel()], packed[1 + s.numel():]
            mean = s / n
            var = (ss - n * mean * mean) / (n - 1)          # unbiased, like torch.std
            return mean.to(input.dtype), var.clamp_min(0).sqrt().to(input.dtype)
        return input.mean(dim=dims), input.std(dim=dims)

    def forward(self, input, context=None):
        if not self.is_initialized():  # data-dependent init on the first batch (actnorm.py:17-23)
            with torch.no_grad():
                mean, std = self._moments(input)
                self.translation.data.copy_(mean)
                self.log_scale.data.copy_(torch.log(std + 1e-8))
                self.initialized.fill_(1)
                self._ready = True
        t, ls = self.translation.view(1, -1, 1, 1), self.log_scale.view(1, -1, 1, 1)
        return (input - t) * torch.exp(-ls), self.logdet(input, context)

    def reverse(self, input, context=None):
        assert self.is_initialized()
        t, ls = self.translation.view(1, -1, 1, 1), self.log_scale.view(1, -1, 1, 1)
        return input * torch.exp(ls) + t

    def logdet(self, input, context=None):
        H, W = input.shape[2:]
        return -self.log_scale.sum().expand(input.size(0)) * H * W


class Conv1x1(FlowLayer):
    def __init__(self, n_channels):
        super().__init__()
        self.n_channels = n_channels
        q = torch.linalg.qr(torch.randn(n_channels, n_channels))[0]
        self.W = nn.Parameter(q.contiguous())

    def forward(self, x, context=None):
        _, _, H, W = x.size()
        ldj = H * W * torch.slogdet(self.W)[1]
        return F.conv2d(x, self.W.view(self.n_channels, self.n_channels, 1, 1)), ldj

    def reverse(self, z, context=None):
        return F.conv2d(z, torch.inverse(self.W).view(self.n_channels, self.n_channels, 1, 1))

    def logdet(self, input, context=None):
        return input.shape[2] * input.shape[3] * torch.slogdet(self.W)[1]


class Conv2dZero(nn.Module):
    def __init__(self, in_channels, out_channels, logscale_factor=3):
        super().__init__()
        self.logscale_factor = logscale_factor
        self.weight = nn.Parameter(torch.zeros(out_channels, in_channels, 3, 3))
        self.bias = nn.Parameter(torch.zeros(out_channels))
        self.logs = nn.Parameter(torch.zeros(out_channels))

    def forward(self, input):
        out = F.conv2d(input, self.weight, self.bias, padding=1)
        return out * torch.exp(self.logs * self.logscale_factor).view(1, -1, 1, 1)


class Coupling(FlowLayer):
    """Affine coupling (layers/coupling.py:44-105).  On CUDA the whole layer -- both 3x3 convolutions,
    the 1x1, the ReLUs, exp(3 logs), the tanh-bounded scale, the affine map and the per-image
    log-determinant -- runs on the tensor-core path (finc_coupling_apply_f32: tcgen05 3xTF32
    implicit GEMMs, hidden activations channels-last, never seen by PyTorch).  Shapes the path does
    not cover (e.g. width % 32 != 0) and CPU tensors use the PyTorch formulas below.

    `precision`: "fp32" = 3xTF32 split products with fp32 accumulation (matches an fp32 reference
    to ~1e-6); "tf32" = single-pass TF32 products, PyTorch's default conv precision (~5e-4)."""

    tensor_core = True      # class-wide switch (tests compare both paths)
    precision = "fp32"

    def __init__(self, input_size, width=512):
        super().__init__()
        self.n_channels = input_size[0]
        self.half_channels = self.n_channels // 2
        self.width = width
        self.net = nn.Sequential(nn.Conv2d(self.half_channels, width, 3, padding=1), nn.ReLU(),
                                 nn.Conv2d(width, width, 1), nn.ReLU(), Conv2dZero(width, self.n_channels))
        self._blob = None
        self._blob_key = None

    # ---- tensor-core path -------------------------------------------------------------------------
    def _params(self):
        n = self.net
        return (n[0].weight, n[0].bias, n[2].weight, n[2].bias, n[4].weight, n[4].bias, n[4].logs)

    def _use_tc(self, x):
        return (self.tensor_core and x.is_cuda and x.dtype == torch.float32 and x.dim() == 4
                and _native.coupling_prepared_bytes(self.n_channels, self.width) > 0)

    def prepared(self, with_backward=False, training=False):
        """hi / lo split weight blob.  Evaluation (no_grad) reuses it while no parameter changed: the cache is
        keyed on (data_ptr, `_version`) of every parameter -- in-place updates, load_state_dict and most optimizers
        bump `_version`.  torch.optim.Adam(fused=True) does NOT (measured: version 0 -> 0 after step()), so a
        training forward (`training=True`) never trusts the cache: it always rebuilds the blob and leaves the
        cache invalid, and the first evaluation after an optimizer step rebuilds it once more.  `with_backward`
        adds the transposed weights of the backward pass."""
        ps = self._params()
        key = None if training else (with_backward,) + tuple((p.data_ptr(), p._version) for p in ps)
        if training or self._blob is None or key != self._blob_key or self._blob.device != ps[0].device:
            self._blob = _native.coupling_prepare(*[p.detach() for p in ps], self.net[4].logscale_factor,
                                                  out=self._blob if self._blob is not None
                                                  and self._blob.device == ps[0].device else None,
                                                  with_backward=with_backward)
            self._blob_key = key
        return self._blob

    def _flags(self):
        return _native.FLAG_TF32_1PASS if self.precision == "tf32" else 0

    # ---- reference formulas (CPU tensors / uncovered shapes / autograd) ----------------------------
    def _st(self, x):
        x1, x2 = x[:, :self.half_channels], x[:, self.half_channels:]
        h = self.net(x1)
        log_s = 2.0 * torch.tanh(h[:, ::2] / 2.0)
        return x1, x2, log_s, h[:, 1::2]

    def _formulas(self, x, reverse):
        """(y, the direction's log-det [B]): forward y2 = x2 exp(log_s) + t, sum log_s; reverse
        y2 = (x2 - t) exp(-log_s), -sum log_s"""
        x1, x2, log_s, t = self._st(x)
        ld = log_s.flatten(start_dim=1).sum(-1)
        if reverse:
            return torch.cat([x1, (x2 - t) * torch.exp(-log_s)], dim=1), -ld
        return torch.cat([x1, x2 * torch.exp(log_s) + t], dim=1), ld

    def forward(self, input, context=None):
        if self._use_tc(input):
            return _CouplingFn.apply(input, self, False, True, *self._params())
        return self._formulas(input, False)

    def _reverse(self, input, want_logdet):
        if self._use_tc(input):
            # a graph exactly when the formulas below would record one
            if torch.is_grad_enabled() and (input.requires_grad or any(p.requires_grad for p in self._params())):
                return _CouplingFn.apply(input, self, True, want_logdet, *self._params())
            return _native.coupling_apply(input, self.prepared(), self.width, reverse=True, want_logdet=want_logdet,
                                          flags=self._flags())
        y, ld = self._formulas(input, True)
        return y, (ld if want_logdet else None)

    def reverse(self, input, context=None):
        return self._reverse(input, False)[0]

    def reverse_and_logdet(self, input):
        """(reverse(input), log|det| of the reverse map [B]) = (x, -sum log_s): minus the forward's log-det at x"""
        return self._reverse(input, True)

    def logdet(self, input, context=None):
        return self.forward(input, context)[1]


class _CouplingFn(torch.autograd.Function):
    """Coupling.forward, or with `reverse` its reverse (and the reverse's log-det -sum log_s when `want_logdet`; None
    otherwise), with the backward on the tensor-core kernels: finc_coupling_apply_f32, then one
    finc_coupling_backward_f32 on the kept workspace (the channels-last hidden activations), with
    FINC_FLAG_COUPLING_REVERSE for the reverse.  Widths the backward kernels do not cover (width % 128 != 0)
    recompute through the PyTorch formulas instead."""

    @staticmethod
    def forward(ctx, x, module, reverse, want_logdet, *params):
        ctx.module, ctx.reverse = module, reverse
        B, C, H, W = x.shape
        train = any(ctx.needs_input_grad)
        ctx.native = train and _native.coupling_prepared_bytes(C, module.width, True) > 0
        ws = None
        if ctx.native:
            ws = torch.empty(_native.coupling_workspace_bytes(B, C, H, W, module.width), dtype=torch.uint8, device=x.device)
        blob = module.prepared(with_backward=ctx.native, training=train)
        y, logdet = _native.coupling_apply(x, blob, module.width, reverse=reverse, want_logdet=want_logdet,
                                           flags=module._flags(), workspace=ws)
        ctx.save_for_backward(x)
        ctx.ws, ctx.blob = ws, blob
        return y, logdet

    @staticmethod
    def backward(ctx, dy, dlogdet):
        (x,) = ctx.saved_tensors
        m = ctx.module
        if ctx.native:
            if dy is None:
                dy = torch.zeros_like(x)
            flags = m._flags() | (_native.FLAG_COUPLING_REVERSE if ctx.reverse else 0)
            grads = _native.coupling_backward(x, dy.contiguous(), dlogdet, ctx.blob, ctx.ws, m.width, flags=flags)
            ctx.ws = None
            return (grads[0], None, None, None, *grads[1:])
        ps = m._params()
        with torch.enable_grad():
            xi = x.detach().requires_grad_(ctx.needs_input_grad[0])
            y, ld = m._formulas(xi, ctx.reverse)
            wanted = [xi] if ctx.needs_input_grad[0] else []
            wanted += [p for p, need in zip(ps, ctx.needs_input_grad[4:]) if need]
            outs, gouts = [y], [dy]
            if dlogdet is not None:    # None: a reverse without its log-det
                outs.append(ld)
                gouts.append(dlogdet)
            grads = list(torch.autograd.grad(outs, wanted, gouts, allow_unused=True))
        dx = grads.pop(0) if ctx.needs_input_grad[0] else None
        dps = [grads.pop(0) if need else None for need in ctx.needs_input_grad[4:]]
        return (dx, None, None, None, *dps)


class GaussianPrior(nn.Module):
    """standard normal over `size`; closed form, device follows the input / `device`"""

    is_standard_normal = True  # FlowSequential then fuses log_prob + logdet into finc_gaussian_logp_f32

    def __init__(self, size):
        super().__init__()
        self.size = tuple(size)
        self.dim = int(math.prod(size))
        self.register_buffer("_anchor", torch.zeros(()), persistent=False)

    def log_prob(self, input, context=None):
        return -0.5 * input.reshape(input.shape[0], -1).pow(2).sum(1) - 0.5 * self.dim * math.log(2 * math.pi)

    def forward(self, input, context=None):
        return -self.log_prob(input, context).sum(-1)

    def sample(self, n_samples, context=None):
        x = torch.randn(n_samples, *self.size, device=self._anchor.device)
        return x, self.log_prob(x)


class SplitPrior(FlowLayer):
    """Coupling, then the second half of the channels is modelled by the prior
    (fastflow_cifar_multi_gpu.py:41-75)"""

    def __init__(self, size, width=512):
        super().__init__()
        self.n_channels = size[0]
        self.transform = Coupling(size, width=width)
        self.base = GaussianPrior((self.n_channels // 2, size[1], size[2]))

    def forward(self, input, context=None):
        x, ldj = self.transform(input, context)
        x1, x2 = x[:, :self.n_channels // 2], x[:, self.n_channels // 2:]
        return x1, x2, self.base.log_prob(x2) + ldj

    def _reverse(self, input, x2, want_logdet):
        """(x, minus the term the forward adds: the coupling's reverse log-det - log N(x2); None unless `want_logdet`)"""
        if x2 is None:
            x2 = torch.randn_like(input)
        x, ld = self.transform._reverse(torch.cat([input, x2], dim=1), want_logdet)
        return x, (ld - self.base.log_prob(x2) if want_logdet else None)

    def reverse(self, input, x2=None, context=None):
        return self._reverse(input, x2, False)[0]

    def reverse_and_logdet(self, input, x2=None):
        return self._reverse(input, x2, True)

    def logdet(self, input, context=None):
        return self.forward(input, context)[2]


# ---------------------------------------------------------------------------------------------
# flow
# ---------------------------------------------------------------------------------------------
class Preprocess(nn.Module):
    """Dequantization, Normalization(0, 256), Normalization(-alpha, 1/(1-2 alpha)), LogitTransform
    (fastflow_cifar_multi_gpu.py:162-186).  On CUDA the four layers and their log-determinants are ONE
    kernel (finc_preprocess_f32); the sub-modules stay for the reference's state-dict keys
    (`preprocess.layers.1.translation`, ...) and for CPU tensors."""

    fused = True

    def __init__(self, size):
        super().__init__()
        self.alpha = alpha = 1e-6
        self.layers = nn.Sequential(Dequantization(), Normalization(0, 256),
                                    Normalization(-alpha, 1 / (1 - 2 * alpha)), LogitTransform())

    def forward(self, x):
        if self.fused and x.is_cuda and x.dtype == torch.float32 and not x.requires_grad:
            deq = self.layers[0]
            u = deq.fixed_noise.to(x.device) if deq.fixed_noise is not None else torch.rand_like(x)
            return _native.preprocess(x, u, self.alpha)
        return _forward_layers(self.layers, x)

    def _reverse(self, x, want_logdet, quantize=False):
        """(reverse(x, quantize), log|det| of that map or None unless `want_logdet`).  The log-det is that of the
        continuous image (quantize=False): the Normalization and LogitTransform terms of the forward, negated, each at
        the forward's input; Dequantization adds 0."""
        if quantize and self.fused and x.is_cuda and x.dtype == torch.float32 and not torch.is_grad_enabled():
            return _native.preprocess(x, None, self.alpha, reverse=True)[0], None
        return _reverse_layers(self.layers if quantize else self.layers[1:], x, want_logdet)

    def reverse(self, x, quantize=True):
        """`quantize=False` stops before Dequantization's floor and returns the continuous image in [0, 256), whose
        gradient reaches the latents and the parameters (the floored image has zero gradient everywhere)."""
        return self._reverse(x, False, quantize)[0]

    def reverse_and_logdet(self, x):
        return self._reverse(x, True)


def _forward_layers(layers, x):
    """x through the layers' forward, and the sum of their log-determinants"""
    logdet = 0
    for layer in layers:
        x, ld = layer(x)
        logdet = logdet + ld
    return x, logdet


def _reverse_layers(layers, x, want_logdet):
    """x through the layers' reverse, last layer first, and (None unless `want_logdet`) the sum of their reverse
    log-determinants.  Each term is minus what the layer's forward adds, evaluated where the forward evaluates it (the
    forward's input = the reverse's output): the layer's own `_reverse` where it has one, -layer.logdet(output)
    otherwise.  Without `want_logdet` no layer's logdet runs: some launch kernels or allocate."""
    logdet = 0 if want_logdet else None
    for layer in reversed(layers):
        if hasattr(layer, "_reverse"):
            x, ld = layer._reverse(x, want_logdet)
        else:
            x = layer.reverse(x)
            ld = -layer.logdet(x) if want_logdet else None
        if want_logdet:
            logdet = logdet + ld
    return x, logdet


class GlowStep(nn.Module):
    def __init__(self, size, actnorm=False, width=512):
        super().__init__()
        d = OrderedDict()
        if actnorm:
            d["actnorm"] = ActNorm(size[0])
        d["conv1x1"] = Conv1x1(size[0])
        d["coupling"] = Coupling(size, width)
        self.glow_step = nn.Sequential(d)

    fused = True  # ActNorm + Conv1x1 as one finc_affine1x1_f32 launch on CUDA tensors

    def forward(self, x):
        if self.fused and x.is_cuda:
            return _fused_glow_forward(self, x)
        return _forward_layers(self.glow_step, x)

    def _reverse(self, x, want_logdet):
        if self.fused and x.is_cuda:
            return _fused_glow_reverse(self, x, want_logdet)
        return _reverse_layers(self.glow_step, x, want_logdet)

    def reverse(self, x):
        return self._reverse(x, False)[0]

    def reverse_and_logdet(self, x):
        return self._reverse(x, True)


class _Affine1x1Fn(torch.autograd.Function):
    """y = A x + b per pixel on finc_affine1x1_f32; backward-data = the same kernel with A^T;
    dA = sum dy x^T and db = sum dy on finc_affine1x1_backward_weight_f32."""

    @staticmethod
    def forward(ctx, x, A, b):
        x = x.contiguous()
        A = A.contiguous()
        ctx.save_for_backward(x, A)
        ctx.has_bias = b is not None
        return _native.affine1x1(x, A, None if b is None else b.contiguous())

    @staticmethod
    def backward(ctx, dy):
        x, A = ctx.saved_tensors
        dy = dy.contiguous()
        dx = _native.affine1x1(dy, A.t().contiguous()) if ctx.needs_input_grad[0] else None
        dA = db = None
        if ctx.needs_input_grad[1] or (ctx.has_bias and ctx.needs_input_grad[2]):
            dA, db = _native.affine1x1_backward_weight(dy, x, want_bias=ctx.has_bias)
        return dx, dA, db


class _InverseFn(torch.autograd.Function):
    """W^-1 of one Conv1x1 weight on finc_slogdet_inverse_f32 (the same bits as the cached reverse constants of
    _glue_constants); backward -W^-T g W^-T"""

    @staticmethod
    def forward(ctx, W):
        Winv = _native.slogdet_inverse(W.unsqueeze(0).contiguous())[1][0]
        ctx.save_for_backward(Winv)
        return Winv

    @staticmethod
    def backward(ctx, g):
        # -W^-T g W^-T as two finc_affine1x1_f32 products (a C x C matrix is one image of C channels, C pixels)
        (Winv,) = ctx.saved_tensors
        C = Winv.shape[0]
        P = _native.affine1x1(g.contiguous().view(1, C, C), Winv.t().contiguous())[0]     # W^-T g
        return -_native.affine1x1(P.t().contiguous().view(1, C, C), Winv)[0].t()          # (W^-1 P^T)^T = P W^-T


class _SlogdetFn(torch.autograd.Function):
    """log|det W_i| of a stack of Conv1x1 weights on finc_slogdet_inverse_f32; backward g_i * W_i^-T"""

    @staticmethod
    def forward(ctx, Ws):
        ld, Winv = _native.slogdet_inverse(Ws)
        ctx.save_for_backward(Winv)
        return ld

    @staticmethod
    def backward(ctx, g):
        (Winv,) = ctx.saved_tensors
        return g.view(-1, 1, 1) * Winv.transpose(1, 2)


def _native_slogdet(W):
    """whether finc_slogdet_inverse_f32 takes the Conv1x1 weight(s) W: CUDA, at most 128 channels"""
    return W.is_cuda and W.shape[-1] <= 128


def _affine_map(act, conv, reverse, want_logdet=False, ld_w=None):
    """(M, bias, ld_pix): one direction of [ActNorm +] Conv1x1 as the per-pixel affine map M x + bias, and the
    log|det| per pixel of the forward map, ld_w - sum log_s where ld_w = log|det W|.
      forward: M = A = W exp(-log_s)[None, :], bias = -A t; ld_pix from the caller's `ld_w`, None without one;
      reverse: M = A^-1 = exp(log_s)[:, None] W^-1, bias = t; ld_pix when `want_logdet`, None otherwise.
    bias is None without ActNorm.  Differentiable under grad, where W^-1 and log|det W| take one
    finc_slogdet_inverse_f32 call each (_InverseFn, _SlogdetFn); under no_grad (_glue_constants) they come from one
    call together, the same bits."""
    W = M = conv.W
    if reverse:
        if not _native_slogdet(W):
            M = torch.inverse(W)
            ld_w = torch.slogdet(W)[1] if want_logdet else None
        elif torch.is_grad_enabled():
            M = _InverseFn.apply(W)
            ld_w = _SlogdetFn.apply(W.unsqueeze(0))[0] if want_logdet else None
        else:
            ld, Winv = _native.slogdet_inverse(W.unsqueeze(0).contiguous())
            M, ld_w = Winv[0], (ld[0] if want_logdet else None)
    if act is None:
        return M, None, ld_w
    ld_pix = None if ld_w is None else ld_w - act.log_scale.sum()
    if reverse:
        return torch.exp(act.log_scale).unsqueeze(1) * M, act.translation, ld_pix
    A = W * torch.exp(-act.log_scale).unsqueeze(0)
    return A, -(A @ act.translation), ld_pix


def _glue_constants(self):
    """(A, b, scalar logdet per pixel, A^-1, reverse bias) of [ActNorm +] Conv1x1, cached on the parameter
    versions.  Used under no_grad (evaluation / sampling): slogdet, inverse and the small products then run
    once per weight update instead of once per call (torch.slogdet alone is an LU factorisation + a host sync)."""
    gs = self.glow_step
    act = getattr(gs, "actnorm", None)
    conv = gs.conv1x1
    ps = [conv.W] + ([act.translation, act.log_scale] if act is not None else [])
    key = tuple((p.data_ptr(), p._version) for p in ps)
    if getattr(self, "_glue_key", None) != key:
        with torch.no_grad():
            Ainv, binv, ld_pix = _affine_map(act, conv, True, want_logdet=True)
            A, b, _ = _affine_map(act, conv, False)
        self._glue = tuple(None if t is None else t.detach().contiguous() for t in (A, b, ld_pix, Ainv, binv))
        self._glue_key = key
    return self._glue


def _fused_glow_forward(self, x):
    """GlowStep.forward with [ActNorm +] Conv1x1 as ONE per-pixel affine kernel (SURVEY.md 8f row 1);
    same values and log-determinants as the layer-by-layer path (actnorm.py:14-64, conv1x1.py:18-43)."""
    gs = self.glow_step
    act = getattr(gs, "actnorm", None)
    conv = gs.conv1x1
    B, _, H, W = x.shape
    if act is not None and not act.is_initialized():
        x, ld0 = act(x)                     # data-dependent init needs the un-fused statistics once
        y = _Affine1x1Fn.apply(x, conv.W, None)
        y, ld = gs.coupling(y)
        return y, ld0 + H * W * torch.slogdet(conv.W)[1] + ld
    if not torch.is_grad_enabled():
        A, b, ld_pix, _, _ = _glue_constants(self)
        y = _native.affine1x1(x.contiguous(), A, b)
        y, ld = gs.coupling(y)
        return y, ld + (H * W) * ld_pix
    self._glue_key = None   # training forward: the cached evaluation constants may not be trusted afterwards
                            # (torch's fused Adam updates parameters without bumping their version counters)
    ld_w = conv.__dict__.pop("_ld_batched", None)     # set by FastFlow.forward: one batched LU per level
    if ld_w is None:
        ld_w = torch.slogdet(conv.W)[1]
    A, b, ld_pix = _affine_map(act, conv, False, ld_w=ld_w)
    y = _Affine1x1Fn.apply(x, A, b)
    y, ld = gs.coupling(y)
    return y, ld + (H * W) * ld_pix


def _fused_glow_reverse(self, z, want_logdet):
    """(x, its reverse log-det: the coupling's and minus H*W*ld_pix, the affine term the forward adds; None unless
    `want_logdet`)"""
    gs = self.glow_step
    act = getattr(gs, "actnorm", None)
    assert act is None or act.is_initialized()
    x, ld = gs.coupling._reverse(z, want_logdet)
    HW = z.shape[2] * z.shape[3]
    act_ps = [act.translation, act.log_scale] if act is not None else []
    if reverse_records(x, gs.conv1x1.W, *act_ps):
        Ainv, binv, ld_pix = _affine_map(act, gs.conv1x1, True, want_logdet)
        y = _Affine1x1Fn.apply(x, Ainv, binv)
    else:
        _, _, ld_pix, Ainv, binv = _glue_constants(self)
        y = _native.affine1x1(x.contiguous(), Ainv, binv)
    return y, (ld - HW * ld_pix if want_logdet else None)


class FastFlowStep(nn.Module):
    def __init__(self, size, actnorm=False, kernel_size=(3, 3), width=512, mask_in_backward=True):
        super().__init__()
        # mask_in_backward=True applies the FInC gradient mask inside the weight-gradient kernel.  The reference clips
        # the gradient norm over the UNMASKED gradients and masks afterwards (train/experiment.py:243-250): pass
        # False (and call clear_grad / reset_gradients after clipping) when that ordering matters.
        self.fastflow_step = nn.Sequential(OrderedDict([
            ("fastflow_unit", FastFlowUnit(size[0], size[0], kernel_size, mask_in_backward=mask_in_backward)),
            ("glow_unit", GlowStep(size, actnorm, width))]))

    fused = True  # evaluation: FastFlowUnit + [ActNorm +] Conv1x1 as ONE finc_chain_f32 launch (SURVEY.md 8f row 1)

    def forward(self, x):
        unit, glow = self.fastflow_step.fastflow_unit, self.fastflow_step.glow_unit
        act = getattr(glow.glow_step, "actnorm", None)
        if (self.fused and glow.fused and not torch.is_grad_enabled() and x.is_cuda and x.dtype == torch.float32
                and (act is None or act.is_initialized()) and x.is_contiguous() and x.data_ptr() % 16 == 0
                and unit.weight.data_ptr() % 16 == 0 and unit.weight.is_contiguous()
                and _native.chain_supported(4, unit.cq, x.shape[2], x.shape[3], unit.kernel_size, True)):
            # z = FInC(x) never leaves shared memory: y = A z + b is written, then the coupling layer
            A, b, ld_pix, _, _ = _glue_constants(glow)
            if b is None:   # no ActNorm: plain Conv1x1
                b = getattr(self, "_zero_bias", None)
                if b is None or b.device != x.device:
                    b = self._zero_bias = torch.zeros(A.shape[0], device=x.device)
            H, W = x.shape[2], x.shape[3]
            y = _native.chain(x, unit.weight.detach().unsqueeze(0), torch.empty_like(x),
                              A=A.unsqueeze(0), bias=b.unsqueeze(0))
            y, ld = glow.glow_step.coupling(y)
            ld = ld + (H * W) * ld_pix
            if unit.logdet_mode == "tensor":   # otherwise the unit reports 0.0 like the reference (fastflow.py:34-50)
                ld = ld + unit.logdet(x)
            return y, ld
        return _forward_layers(self.fastflow_step, x)

    def _reverse(self, x, want_logdet):
        return _reverse_layers(self.fastflow_step, x, want_logdet)

    def reverse(self, x):
        return self._reverse(x, False)[0]

    def reverse_and_logdet(self, x):
        return self._reverse(x, True)


class FastFlowLevel(nn.Module):
    def __init__(self, size, block_size=16, actnorm=False, kernel_size=(3, 3), width=512, mask_in_backward=True):
        super().__init__()
        size = (size[0] * 4, size[1] // 2, size[2] // 2)
        self.fastflow_level = nn.ModuleList([Squeeze(),
                                             *[FastFlowStep(size, actnorm, kernel_size, width, mask_in_backward)
                                               for _ in range(block_size)],
                                             SplitPrior(size, width)])

    def forward(self, x):
        logdet, z = 0, None
        for layer in self.fastflow_level:
            if isinstance(layer, SplitPrior):
                x, z, ld = layer(x)
            else:
                x, ld = layer(x)
            logdet = logdet + ld
        return x, z, logdet

    def _reverse(self, x, z, want_logdet):
        *layers, split = self.fastflow_level
        x, ld = split._reverse(x, z, want_logdet)
        x, ld_rest = _reverse_layers(layers, x, want_logdet)
        return x, (ld + ld_rest if want_logdet else None)

    def reverse(self, x, z=None):
        return self._reverse(x, z, False)[0]

    def reverse_and_logdet(self, x, z=None):
        return self._reverse(x, z, True)


class FastFlow(nn.Module):
    """forward(x) -> (zs, logp[B]); reverse(n_samples, zs) -> x; sample(n); reconstruct(x)
    (fastflow_cifar_multi_gpu.py:295-387).  `final_steps=None` = block_size (CIFAR / ImageNet32
    scripts); the MNIST and ImageNet64 scripts use ONE final step (`final_steps=1`)."""

    def __init__(self, n_blocks=2, block_size=16, image_size=(1, 28, 28), actnorm=False, kernel_size=(3, 3),
                 final_steps=None, width=512, mask_in_backward=True):
        super().__init__()
        C_in, H, W = image_size
        self.output_size = (C_in * 2 ** (n_blocks + 1), H // 2 ** n_blocks, W // 2 ** n_blocks)
        self.preprocess = Preprocess(image_size)
        self.fastflow_levels = nn.ModuleList([
            FastFlowLevel((C_in * 2 ** i, H // 2 ** i, W // 2 ** i), block_size, actnorm, kernel_size, width,
                          mask_in_backward)
            for i in range(n_blocks - 1)])
        self.squeeze = Squeeze()
        n_final = block_size if final_steps is None else final_steps
        self.fastflow_step = nn.Sequential(*[FastFlowStep(self.output_size, actnorm, kernel_size, width, mask_in_backward)
                                             for _ in range(n_final)])
        self.base_distribution = GaussianPrior(self.output_size)

    def _batched_slogdets(self):
        """training path: log|det W| of every Conv1x1 in ONE batched LU per channel count (3 calls for the
        CIFAR-10 flow instead of 48; each torch.slogdet is a cuSOLVER factorisation with a host round trip)"""
        groups = {}
        for mod in self.modules():
            if isinstance(mod, Conv1x1):
                groups.setdefault(mod.n_channels, []).append(mod)
        for n_ch, convs in groups.items():
            Ws = torch.stack([c.W for c in convs])
            lds = _SlogdetFn.apply(Ws) if _native_slogdet(Ws) else torch.linalg.slogdet(Ws)[1]
            for i, c in enumerate(convs):
                c._ld_batched = lds[i]

    def forward(self, x, context=None):
        zs = []
        if torch.is_grad_enabled() and x.is_cuda and GlowStep.fused:
            self._batched_slogdets()
        x, logdet = self.preprocess(x)
        for level in self.fastflow_levels:
            x, z, ld = level(x)
            logdet = logdet + ld
            zs.append(z)
        x, ld = self.squeeze(x)
        logdet = logdet + ld
        for step in self.fastflow_step:
            x, ld = step(x)
            logdet = logdet + ld
        zs.append(x)
        return zs, logdet + self.base_distribution.log_prob(x)

    def reverse(self, n_samples=1, zs=None, z_std=1.0, quantize=True):
        """x = the flow's inverse of the latents `zs` (sampled when None).  Differentiable in `zs` and every parameter
        the inverse uses (ops.finc_inverse says when a graph is recorded); `quantize=False` returns the continuous image before the final floor, which has zero gradient
        (Preprocess.reverse)."""
        return self._reverse(n_samples, zs, False, quantize)[0]

    def sample_with_log_prob(self, n_samples=1, zs=None):
        """(x, log_q[B]): x = reverse(n_samples, zs, quantize=False), the continuous image, and log_q its log-density
        under the model in nats, log N(every latent, the split-prior ones drawn inside included) - log|det dx/dz|.
        This is model.log_prob(x) with zero dequantisation noise, without a second pass.  Differentiable in `zs` and
        the parameters wherever reverse() records a graph (reverse-KL: E_q[log q(x) - log p*(x)])."""
        return self._reverse(n_samples, zs, True)

    def _reverse(self, n_samples, zs, want_logdet, quantize=False):
        """(reverse(n_samples, zs, quantize=quantize), log_q or None unless `want_logdet`).  Latents not given are drawn
        in this order: the base sample first, then the split priors from the last level to the first."""
        if zs is None:
            zs = [self.base_distribution.sample(n_samples)[0]]
        x, logdet = _reverse_layers(self.fastflow_step, zs[-1], want_logdet)
        x = self.squeeze.reverse(x)
        for i, level in enumerate(reversed(self.fastflow_levels)):
            x, ld = level._reverse(x, None if len(zs) == 1 else zs[-i - 2], want_logdet)
            if want_logdet:
                logdet = logdet + ld
        x, ld = self.preprocess._reverse(x, want_logdet, quantize)
        if not want_logdet:
            return x, None
        return x, self.base_distribution.log_prob(zs[-1]) - (logdet + ld)

    def log_prob(self, x, bits_per_pixel=False):
        """bits_per_pixel: per IMAGE dimension (x[0].numel()).  The reference divides by `zs[0].numel()`, a
        batch-sized latent tensor (fastflow_cifar_multi_gpu.py log_prob), so its printed value scales with the batch
        size and is not comparable; its training metric (train/experiment.py:279-295) agrees with this one."""
        zs, logp = self.forward(x)
        return logp / (math.log(2) * x[0].numel()) if bits_per_pixel else logp

    def sample(self, n_samples, context=None):
        x = self.reverse(n_samples=n_samples)
        return x, x

    def reconstruct(self, x, context=None):
        zs, _ = self.forward(x)
        return self.reverse(n_samples=x.shape[0], zs=[zs[-1]])

    def reconstruct_exact(self, x):
        """true inverse: feeds the split-off latents back (test_layers.py:304-348 reconstruct_ff)"""
        zs, _ = self.forward(x)
        return self.reverse(n_samples=x.shape[0], zs=zs)


class InferenceSession:
    """Likelihood evaluation and sampling of a trained flow as CUDA graphs.

    An eager forward of the CIFAR-10 flow issues ~1900 kernel launches (48 steps x FInC unit, affine glue,
    six coupling launches, log-determinant adds); the host needs ~26 ms to enqueue what the GPU executes in
    ~12 ms.  The session captures `model.forward` / `model.reverse` once per batch size into a CUDA graph
    (static input / output buffers, weights read in place) and replays it.  Weights must not change between
    capture and replay; call `reset()` after loading new ones.  The reference samples one layer at a time
    from Python (train/experiment.py:327-337)."""

    def __init__(self, model):
        self.model = model.eval()
        self._eval, self._sample = {}, {}

    def reset(self):
        self._eval.clear()
        self._sample.clear()

    @staticmethod
    def _capture(fn, warm=2):
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side), torch.no_grad():
            for _ in range(warm):          # lazy initialisations (weight blobs, glue constants, workspaces)
                fn()
        torch.cuda.current_stream().wait_stream(side)
        g = torch.cuda.CUDAGraph()
        with torch.no_grad(), torch.cuda.graph(g):
            out = fn()
        return g, out

    def log_prob(self, x):
        """(zs, logp[B]) like model.forward(x); the returned tensors are the session's static buffers"""
        key = tuple(x.shape)
        if key not in self._eval:
            buf = x.clone()
            g, out = self._capture(lambda: self.model(buf))
            self._eval[key] = (g, buf, out)
        g, buf, out = self._eval[key]
        buf.copy_(x)
        g.replay()
        return out

    def sample(self, n_samples):
        """x [n, C, H, W] like model.sample(n)[0]; latents are drawn inside the graph"""
        if n_samples not in self._sample:
            g, out = self._capture(lambda: self.model.sample(n_samples)[0])
            self._sample[n_samples] = (g, out)
        g, out = self._sample[n_samples]
        g.replay()
        return out


def set_fp32_parity(enabled: bool = True):
    """The reference ran full fp32 (CUDA 10.2 / cuDNN 7.6 predate TF32).  The glue layers here
    are PyTorch convolutions whose cuDNN default is TF32 (~5e-4 relative); call this to get the
    reference's numerics in the glue as well.  The FInC kernels are always fp32 FMA."""
    torch.backends.cudnn.allow_tf32 = not enabled
    torch.backends.cuda.matmul.allow_tf32 = not enabled


def clear_grad(module):
    from .fastflow import clear_grad as _cg

    _cg(module)


# builders with the reference scripts' settings (SURVEY.md section 8 shape table)
def fastflow_mnist(**kw):
    return FastFlow(n_blocks=2, block_size=16, image_size=(1, 28, 28), final_steps=1, **kw)


def fastflow_cifar10(**kw):
    return FastFlow(n_blocks=3, block_size=16, image_size=(3, 32, 32), **kw)


def fastflow_imagenet32(**kw):
    return FastFlow(n_blocks=3, block_size=48, image_size=(3, 32, 32), **kw)


def fastflow_imagenet64(kernel_size=(3, 3), **kw):
    return FastFlow(n_blocks=4, block_size=48, image_size=(3, 64, 64), final_steps=1, kernel_size=kernel_size, **kw)
