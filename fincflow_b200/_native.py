"""ctypes binding of libfincflow_b200.so (include/fincflow_b200.h) for torch tensors.

PyTorch is plumbing here: it owns device memory and streams; every kernel on the FInC hot
path is our own sm_100a code behind the C ABI.  There is NO CPU fallback: a missing
library or a non-CUDA tensor raises.
"""
from __future__ import annotations

import ctypes
import os
import threading

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libfincflow_b200.so")

ORDER_CODE = {"TL": 0, "TR": 1, "BL": 2, "BR": 3}
ORDERS_UNIT = 0xE4  # TL | TR<<2 | BL<<4 | BR<<6   (fastflow/fastflow.py:24-27)

FLAG_NAIVE = 1
FLAG_NO_MASK = 2
FLAG_ACCUMULATE = 4
FLAG_LOGDET_ACCUMULATE = 8
FLAG_GENERIC_TILED = 16
FLAG_WORKSPACE_CLEAN = 32
FLAG_PREPARED = 64
FLAG_CHAIN_TRANSPOSE = 2048
FLAG_QUARTER_GPU = 128
FLAG_HALF_GPU = 256
FLAG_WAVE_SMEM = 512
FLAG_TF32_1PASS = 1024
FLAG_NEGATE = 4096
FLAG_COUPLING_REVERSE = 8192
PREP_FORWARD, PREP_BACKWARD_INPUT, PREP_INVERSE = 0, 1, 2

# every symbol declared in include/fincflow_b200.h
SYMBOLS = (
    "finc_abi_version", "finc_error_string", "finc_set_device", "finc_sm_count",
    "finc_forward_f32", "finc_backward_input_f32", "finc_backward_weight_workspace_bytes",
    "finc_backward_weight_f32", "finc_inverse_f32", "finc_inverse_adjoint_f32", "finc_apply_grad_mask_f32", "finc_logdet_f32",
    "finc_gaussian_logp_f32", "finc_debug_timestamps", "finc_prepared_weights_bytes", "finc_prepare_weights_f32",
    "finc_squeeze_f32", "finc_unsqueeze_f32", "finc_adam_step_f32", "finc_allreduce_adam_f32", "finc_affine1x1_f32",
    "finc_affine1x1_backward_weight_workspace_bytes", "finc_affine1x1_backward_weight_f32",
    "finc_preprocess_f32", "finc_slogdet_inverse_f32", "finc_tc_conv_weights_bytes", "finc_tc_conv_prepare_weights_f32", "finc_tc_conv_nhwc_f32",
    "finc_tc_wgrad_workspace_bytes", "finc_tc_wgrad_f32", "finc_coupling_prepared_bytes", "finc_coupling_workspace_bytes", "finc_coupling_prepare_f32",
    "finc_coupling_apply_f32", "finc_coupling_backward_workspace_bytes", "finc_coupling_backward_f32",
    "finc_inverse_dense_bytes", "finc_inverse_dense_scratch_bytes", "finc_inverse_dense_prepare_f32",
    "finc_inverse_dense_f32", "finc_chain_supported", "finc_chain_f32", "finc_inverse_chain_f32",
    "finc_inverse_chain_multi_f32",
    "finc_backward_weight_batched_workspace_bytes", "finc_backward_weight_batched_f32",
)

_lib = None
_tls = threading.local()
launch_count = 0  # kernels of ours enqueued through this module (bench.py's gpu_launches)


class FincNativeError(RuntimeError):
    pass


class FincInverseLevel(ctypes.Structure):
    """include/fincflow_b200.h: FincInverseLevel (the arguments of finc_inverse_chain_f32)"""
    _fields_ = [("z", ctypes.c_void_p), ("prepared", ctypes.c_void_p), ("prepared_stride_bytes", ctypes.c_size_t),
                ("x", ctypes.c_void_p)] + [(n, ctypes.c_int) for n in ("B", "G", "C", "H", "W", "kH", "kW")] + [
                ("orders", ctypes.c_uint), ("n_units", ctypes.c_int), ("u_first", ctypes.c_int), ("u_step", ctypes.c_int)]


def load():
    """Load the CUDA library; fails loudly if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise FincNativeError(
            f"{LIB_PATH} is missing: build it with `python -m fincflow_b200.build` "
            "(or __graft_entry__.build()).  fincflow_b200 has no CPU or PyTorch fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    i, u, p, sz = ctypes.c_int, ctypes.c_uint, ctypes.c_void_p, ctypes.c_size_t
    dims = [i] * 7
    lib.finc_abi_version.restype = i
    lib.finc_error_string.restype = ctypes.c_char_p
    lib.finc_error_string.argtypes = [i]
    lib.finc_set_device.argtypes = [i]
    lib.finc_sm_count.restype = i
    lib.finc_forward_f32.argtypes = [p, p, p, p, *dims, u, u, p]
    lib.finc_backward_input_f32.argtypes = [p, p, p, *dims, u, u, p]
    lib.finc_backward_weight_workspace_bytes.restype = sz
    lib.finc_backward_weight_workspace_bytes.argtypes = dims
    lib.finc_backward_weight_f32.argtypes = [p, p, p, p, sz, *dims, u, u, p]
    lib.finc_inverse_f32.argtypes = [p, p, p, *dims, u, u, p]
    lib.finc_inverse_adjoint_f32.argtypes = [p, p, p, *dims, u, u, p]
    lib.finc_apply_grad_mask_f32.argtypes = [p, i, i, i, i, u, p]
    lib.finc_logdet_f32.argtypes = [p, p, *dims, u, p]
    lib.finc_gaussian_logp_f32.argtypes = [p, p, p, p, ctypes.c_float, i, ctypes.c_long, p]
    lib.finc_adam_step_f32.restype = i
    lib.finc_adam_step_f32.argtypes = [p, p, p, p, p] + [ctypes.c_float] * 4 + [ctypes.c_long, p]
    lib.finc_allreduce_adam_f32.restype = i
    lib.finc_allreduce_adam_f32.argtypes = [p] * 7 + [ctypes.c_float] * 5 + [ctypes.c_long, i, i, p]
    lib.finc_squeeze_f32.restype = i
    lib.finc_squeeze_f32.argtypes = [p, p, i, i, i, i, p]
    lib.finc_unsqueeze_f32.restype = i
    lib.finc_unsqueeze_f32.argtypes = [p, p, i, i, i, i, p]
    lib.finc_affine1x1_f32.restype = i
    lib.finc_affine1x1_f32.argtypes = [p, p, p, p, i, i, ctypes.c_long, p]
    lib.finc_affine1x1_backward_weight_workspace_bytes.restype = sz
    lib.finc_affine1x1_backward_weight_workspace_bytes.argtypes = [i, i, ctypes.c_long]
    lib.finc_affine1x1_backward_weight_f32.restype = i
    lib.finc_affine1x1_backward_weight_f32.argtypes = [p, p, p, p, p, sz, i, i, ctypes.c_long, p]
    lib.finc_prepared_weights_bytes.restype = sz
    lib.finc_prepared_weights_bytes.argtypes = [i] + dims
    lib.finc_prepare_weights_f32.restype = i
    lib.finc_prepare_weights_f32.argtypes = [p, p, i, i, sz, sz, *dims, u, p]
    lib.finc_slogdet_inverse_f32.restype = i
    lib.finc_slogdet_inverse_f32.argtypes = [p, p, p, i, i, p]
    lib.finc_preprocess_f32.restype = i
    lib.finc_preprocess_f32.argtypes = [p, p, p, p, i, ctypes.c_long, ctypes.c_float, i, p]
    lib.finc_tc_conv_weights_bytes.restype = sz
    lib.finc_tc_conv_weights_bytes.argtypes = [i, i, i, i]
    lib.finc_tc_conv_prepare_weights_f32.restype = i
    lib.finc_tc_conv_prepare_weights_f32.argtypes = [p, p, i, i, i, i, p]
    lib.finc_tc_conv_nhwc_f32.restype = i
    lib.finc_tc_conv_nhwc_f32.argtypes = [p, p, p, p, p, i, i, i, i, i, i, i, u, p]
    lib.finc_tc_wgrad_workspace_bytes.restype = sz
    lib.finc_tc_wgrad_workspace_bytes.argtypes = [ctypes.c_long, i, i]
    lib.finc_tc_wgrad_f32.restype = i
    lib.finc_tc_wgrad_f32.argtypes = [p, p, p, p, sz, ctypes.c_long, i, i, i, i, i, u, p]
    lib.finc_coupling_prepared_bytes.restype = sz
    lib.finc_coupling_prepared_bytes.argtypes = [i, i, i]
    lib.finc_coupling_workspace_bytes.restype = sz
    lib.finc_coupling_workspace_bytes.argtypes = [i, i, i, i, i]
    lib.finc_coupling_prepare_f32.restype = i
    lib.finc_coupling_prepare_f32.argtypes = [p] * 7 + [ctypes.c_float, p, i, i, i, p]
    lib.finc_inverse_dense_bytes.restype = sz
    lib.finc_inverse_dense_bytes.argtypes = [i, i, i, i]
    lib.finc_inverse_dense_scratch_bytes.restype = sz
    lib.finc_inverse_dense_scratch_bytes.argtypes = [i, i, i, i]
    lib.finc_inverse_dense_prepare_f32.restype = i
    lib.finc_inverse_dense_prepare_f32.argtypes = [p, p, p, sz, i, i, i, i, i, i, u, p]
    lib.finc_inverse_dense_f32.restype = i
    lib.finc_inverse_dense_f32.argtypes = [p, p, p, i, i, i, i, i, u, p]
    lib.finc_backward_weight_batched_workspace_bytes.restype = ctypes.c_size_t
    lib.finc_backward_weight_batched_workspace_bytes.argtypes = [i, i, i, i, i, i, i, i]
    lib.finc_backward_weight_batched_f32.restype = i
    lib.finc_backward_weight_batched_f32.argtypes = [p, p, p, p, ctypes.c_size_t, i, i, i, i, i, i, i, u, u, i,
                                                     ctypes.c_long, ctypes.c_long, ctypes.c_long, p]
    lib.finc_inverse_chain_f32.restype = i
    lib.finc_inverse_chain_f32.argtypes = [p, p, ctypes.c_size_t, p, i, i, i, i, i, i, i, u, i, i, i, p]
    lib.finc_inverse_chain_multi_f32.restype = i
    lib.finc_inverse_chain_multi_f32.argtypes = [ctypes.POINTER(FincInverseLevel), i, p]
    lib.finc_chain_supported.restype = i
    lib.finc_chain_supported.argtypes = [i, i, i, i, i, i, i]
    lib.finc_chain_f32.restype = i
    lib.finc_chain_f32.argtypes = [p, p, ctypes.c_long, p, ctypes.c_long, p, p, p, i, i, i, i, i, i, i, u, i, i, i, u, p]
    lib.finc_coupling_backward_workspace_bytes.restype = sz
    lib.finc_coupling_backward_workspace_bytes.argtypes = [i, i, i, i, i]
    lib.finc_coupling_backward_f32.restype = i
    lib.finc_coupling_backward_f32.argtypes = [p] * 6 + [sz] + [p] * 8 + [i, i, i, i, i, u, p]
    lib.finc_coupling_apply_f32.restype = i
    lib.finc_coupling_apply_f32.argtypes = [p, p, p, p, p, sz, i, i, i, i, i, i, u, p]
    for f in ("finc_set_device", "finc_forward_f32", "finc_backward_input_f32", "finc_backward_weight_f32",
              "finc_inverse_f32", "finc_inverse_adjoint_f32", "finc_apply_grad_mask_f32", "finc_logdet_f32", "finc_gaussian_logp_f32"):
        getattr(lib, f).restype = i
    if lib.finc_abi_version() != 1:
        raise FincNativeError("libfincflow_b200.so ABI version mismatch; rebuild")
    _lib = lib
    return lib


def pack_orders(orders) -> int:
    v = 0
    for g, o in enumerate(orders):
        v |= (ORDER_CODE[o] if isinstance(o, str) else int(o)) << (2 * g)
    return v


def _check(rc: int, what: str, launches: int = 1):
    global launch_count
    launch_count += launches
    if rc != 0:
        msg = load().finc_error_string(rc).decode()
        raise FincNativeError(f"{what} failed: {msg} (code {rc})")


def _prep(t: torch.Tensor, name: str) -> torch.Tensor:
    if not t.is_cuda:
        raise FincNativeError(f"{name} must be a CUDA tensor: fincflow_b200 has no CPU path")
    if t.dtype != torch.float32:
        raise FincNativeError(f"{name} must be float32, got {t.dtype}")
    return t if t.is_contiguous() else t.contiguous()


def _bind_device(t: torch.Tensor):
    """make the tensor's device the current CUDA device of this thread.  Checked against the runtime on every call
    (torch.cuda.current_device() is a cudaGetDevice): a cached value goes stale when torch switches devices
    (torch.cuda.set_device, leaving a `with torch.cuda.device(i)` block)."""
    dev = t.device.index
    if torch.cuda.current_device() != dev:
        _check(load().finc_set_device(dev), "finc_set_device", 0)


def _stream(t: torch.Tensor) -> int:
    return torch.cuda.current_stream(t.device).cuda_stream


def _dims(x: torch.Tensor, w: torch.Tensor, G: int):
    B, CT, H, W = x.shape
    if CT % G != 0:
        raise FincNativeError(f"channels {CT} not divisible by groups {G}")
    C = CT // G
    if tuple(w.shape[:2]) != (G * C, C):
        raise FincNativeError(f"weight shape {tuple(w.shape)} does not match [G*C={G * C}, C={C}, kH, kW]")
    return B, G, C, H, W, int(w.shape[2]), int(w.shape[3])


def _dims_prepared(x, G, ksize):
    B, CT, H, W = x.shape
    return B, G, CT // G, H, W, int(ksize[0]), int(ksize[1])


def forward(x, w, G=4, orders=ORDERS_UNIT, want_logdet=True, flags=0, out=None, logdet_out=None, prepared=None,
            ksize=None):
    """z, logdet[B] (or None).  C ABI: finc_forward_f32.  With `logdet_out` and
    FLAG_LOGDET_ACCUMULATE the layer's logdet is added into a running [B] accumulator.
    `prepared` (a table from prepare_weights, with `ksize`) replaces `w`; no logdet then."""
    x = _prep(x, "x")
    if prepared is not None:
        d, w, flags = _dims_prepared(x, G, ksize), prepared, flags | FLAG_PREPARED
    else:
        w = _prep(w, "weight")
        d = _dims(x, w, G)
    _bind_device(x)
    z = torch.empty_like(x) if out is None else out
    if logdet_out is not None:
        logdet, want_logdet = logdet_out, True
    else:
        logdet = torch.empty(d[0], dtype=torch.float32, device=x.device) if want_logdet else None
    _check(load().finc_forward_f32(x.data_ptr(), w.data_ptr(), z.data_ptr(),
                                   logdet.data_ptr() if want_logdet else None,
                                   *d, orders, flags, _stream(x)), "finc_forward_f32")
    return z, logdet


def backward_input(dz, w, G=4, orders=ORDERS_UNIT, flags=0, out=None, prepared=None, ksize=None):
    dz = _prep(dz, "dz")
    if prepared is not None:
        d, w, flags = _dims_prepared(dz, G, ksize), prepared, flags | FLAG_PREPARED
    else:
        w = _prep(w, "weight")
        d = _dims(dz, w, G)
    _bind_device(dz)
    dx = torch.empty_like(dz) if out is None else out
    _check(load().finc_backward_input_f32(dz.data_ptr(), w.data_ptr(), dx.data_ptr(), *d, orders, flags,
                                          _stream(dz)), "finc_backward_input_f32")
    return dx


def backward_weight_workspace_bytes(B, G, C, H, W, kH, kW) -> int:
    return int(load().finc_backward_weight_workspace_bytes(B, G, C, H, W, kH, kW))


def new_workspace(nbytes, device):
    """zero-initialised workspace for backward_weight(workspace=...); the kernels leave its
    ticket counters zero, so it can be reused by stream-ordered calls without a memset"""
    return torch.zeros(max(int(nbytes), 4096), dtype=torch.uint8, device=device)


def backward_weight(dz, x, ksize, G=4, orders=ORDERS_UNIT, flags=0, out=None, workspace=None):
    """Masked dW [G*C, C, kH, kW] (FLAG_NO_MASK for the raw gradient).  `out` may be a view
    into a flat gradient bucket; FLAG_ACCUMULATE adds into it."""
    dz, x = _prep(dz, "dz"), _prep(x, "x")
    B, CT, H, W = x.shape
    C = CT // G
    kH, kW = ksize
    _bind_device(x)
    if out is None:
        out = torch.empty((G * C, C, kH, kW), dtype=torch.float32, device=x.device)
    elif not (out.is_cuda and out.is_contiguous() and out.dtype == torch.float32 and out.numel() == G * C * C * kH * kW):
        raise FincNativeError("backward_weight: `out` must be a contiguous float32 CUDA tensor of G*C*C*kH*kW elements")
    lib = load()
    if workspace is None:
        nbytes = lib.finc_backward_weight_workspace_bytes(B, G, C, H, W, kH, kW)
        ws = torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=x.device)
    else:
        ws = workspace  # caller-owned, zero-initialised once (see new_workspace): skips the memset node
        flags |= FLAG_WORKSPACE_CLEAN
    _check(lib.finc_backward_weight_f32(dz.data_ptr(), x.data_ptr(), out.data_ptr(), ws.data_ptr(), ws.numel(),
                                        B, G, C, H, W, kH, kW, orders, flags, _stream(x)),
           "finc_backward_weight_f32")
    return out


def inverse(z, w, G=4, orders=ORDERS_UNIT, flags=0, out=None, prepared=None, ksize=None):
    z = _prep(z, "z")
    if prepared is not None:
        d, w, flags = _dims_prepared(z, G, ksize), prepared, flags | FLAG_PREPARED
    else:
        w = _prep(w, "weight")
        d = _dims(z, w, G)
    _bind_device(z)
    x = torch.empty_like(z) if out is None else out
    _check(load().finc_inverse_f32(z.data_ptr(), w.data_ptr(), x.data_ptr(), *d, orders, flags, _stream(z)),
           "finc_inverse_f32")
    return x


def inverse_adjoint(dx, w, G=4, orders=ORDERS_UNIT, flags=0, out=None):
    """dz = A^-T dx, the adjoint of inverse() (x = A^-1 z): <dx, inverse(z)> == <inverse_adjoint(dx), z>.
    `out` may be `dx` (in place).  C ABI: finc_inverse_adjoint_f32."""
    dx = _prep(dx, "dx")
    w = _prep(w, "weight")
    d = _dims(dx, w, G)
    _bind_device(dx)
    dz = torch.empty_like(dx) if out is None else out
    _check(load().finc_inverse_adjoint_f32(dx.data_ptr(), w.data_ptr(), dz.data_ptr(), *d, orders, flags, _stream(dx)),
           "finc_inverse_adjoint_f32")
    return dz


def apply_grad_mask_(dw, G, orders):
    if not dw.is_contiguous():
        raise FincNativeError("apply_grad_mask_: dw must be contiguous (in-place operation)")
    dw = _prep(dw, "dw")
    _bind_device(dw)
    C, kH, kW = int(dw.shape[1]), int(dw.shape[2]), int(dw.shape[3])
    _check(load().finc_apply_grad_mask_f32(dw.data_ptr(), G, C, kH, kW, orders, _stream(dw)),
           "finc_apply_grad_mask_f32")
    return dw


def logdet(w, B, H, W, G=4, orders=ORDERS_UNIT):
    w = _prep(w, "weight")
    _bind_device(w)
    C, kH, kW = int(w.shape[1]), int(w.shape[2]), int(w.shape[3])
    out = torch.empty(B, dtype=torch.float32, device=w.device)
    _check(load().finc_logdet_f32(w.data_ptr(), out.data_ptr(), B, G, C, H, W, kH, kW, orders, _stream(w)),
           "finc_logdet_f32")
    return out


def gaussian_logp(z, logdet=None, dz_scale=None, logp_out=None, dz_out=None):
    """logp[B] of a standard normal (+ logdet) and optionally dz = dz_scale * z."""
    z = _prep(z, "z")
    _bind_device(z)
    B = int(z.shape[0])
    D = z.numel() // max(B, 1)
    logp = torch.empty(B, dtype=torch.float32, device=z.device) if logp_out is None else logp_out
    dz = None
    if dz_scale is not None:
        dz = torch.empty_like(z) if dz_out is None else dz_out
    _check(load().finc_gaussian_logp_f32(z.data_ptr(), None if logdet is None else logdet.data_ptr(), logp.data_ptr(),
                                         None if dz is None else dz.data_ptr(), float(dz_scale or 0.0), B, D,
                                         _stream(z)), "finc_gaussian_logp_f32")
    return logp, dz


def prepared_weights_bytes(kind, B, G, C, H, W, kH, kW) -> int:
    """bytes of one unit's prepared table; 0 = shape not covered (do not use FLAG_PREPARED)"""
    return int(load().finc_prepared_weights_bytes(kind, B, G, C, H, W, kH, kW))


def prepare_weights(w_units, tables, kind, B, H, W, G=4, orders=ORDERS_UNIT):
    """w_units: [n_units, G*C, C, kH, kW] contiguous; tables: [n_units, bytes] uint8 -> filled in ONE launch"""
    w_units = _prep(w_units, "weights")
    _bind_device(w_units)
    n = int(w_units.shape[0])
    C, kH, kW = int(w_units.shape[2]), int(w_units.shape[3]), int(w_units.shape[4])
    _check(load().finc_prepare_weights_f32(w_units.data_ptr(), tables.data_ptr(), kind, n, w_units.stride(0), tables.stride(0),
                                           B, G, C, H, W, kH, kW, orders, _stream(w_units)), "finc_prepare_weights_f32")
    return tables


def adam_step_(param, grad, exp_avg, exp_avg_sq, step, lr=1e-3, betas=(0.9, 0.999), eps=1e-8):
    """in-place Adam on flat fp32 buffers; `step` is a 1-element float device tensor"""
    _bind_device(param)
    _check(load().finc_adam_step_f32(param.data_ptr(), grad.data_ptr(), exp_avg.data_ptr(), exp_avg_sq.data_ptr(),
                                     step.data_ptr(), lr, betas[0], betas[1], eps, param.numel(), _stream(param)),
           "finc_adam_step_f32", 2)
    return param


def allreduce_adam_(peer_grad_ptrs_dev, peer_signal_ptrs_dev, local, param, exp_avg, exp_avg_sq, step, rank, world,
                    lr=1e-3, betas=(0.9, 0.999), eps=1e-8, grad_scale=1.0):
    """fused NVLink peer-memory all-reduce(SUM) of the gradient buckets + Adam (finc_allreduce_adam_f32)"""
    _bind_device(param)
    _check(load().finc_allreduce_adam_f32(peer_grad_ptrs_dev, peer_signal_ptrs_dev, local.data_ptr(), param.data_ptr(),
                                          exp_avg.data_ptr(), exp_avg_sq.data_ptr(), step.data_ptr(), lr, betas[0],
                                          betas[1], eps, grad_scale, param.numel(), rank, world, _stream(param)),
           "finc_allreduce_adam_f32")
    return param


def squeeze(x, out=None):
    """[B,C,H,W] -> [B,4C,H/2,W/2], channel order 4c + 2dh + dw (layers/squeeze.py:5-13)"""
    x = _prep(x, "x")
    _bind_device(x)
    B, C, H, W = x.shape
    y = torch.empty((B, 4 * C, H // 2, W // 2), dtype=torch.float32, device=x.device) if out is None else out
    _check(load().finc_squeeze_f32(x.data_ptr(), y.data_ptr(), B, C, H, W, _stream(x)), "finc_squeeze_f32")
    return y


def unsqueeze(x, out=None):
    """[B,4C,H,W] -> [B,C,2H,2W] (layers/squeeze.py:16-24)"""
    x = _prep(x, "x")
    _bind_device(x)
    B, C4, H, W = x.shape
    y = torch.empty((B, C4 // 4, 2 * H, 2 * W), dtype=torch.float32, device=x.device) if out is None else out
    _check(load().finc_unsqueeze_f32(x.data_ptr(), y.data_ptr(), B, C4, H, W, _stream(x)), "finc_unsqueeze_f32")
    return y


def affine1x1(x, A, bias=None, out=None):
    """y[n,:,h,w] = A @ x[n,:,h,w] + bias: ActNorm followed by Conv1x1 (or their reverse / backward-data)
    as one per-pixel affine map (layers/actnorm.py:14-52, layers/conv1x1.py:18-43)"""
    x = _prep(x, "x")
    A = _prep(A, "A")
    _bind_device(x)
    B, C = x.shape[0], x.shape[1]
    HW = 1
    for d in x.shape[2:]:
        HW *= d
    if tuple(A.shape) != (C, C):
        raise FincNativeError(f"A must be [{C}, {C}], got {tuple(A.shape)}")
    if bias is not None:
        bias = _prep(bias, "bias")
        if bias.numel() != C:
            raise FincNativeError(f"bias must have {C} elements")
    y = torch.empty_like(x) if out is None else out
    _check(load().finc_affine1x1_f32(x.data_ptr(), A.data_ptr(), 0 if bias is None else bias.data_ptr(), y.data_ptr(),
                                     B, C, HW, _stream(x)), "finc_affine1x1_f32")
    return y


def affine1x1_backward_weight(dy, x, want_bias=True):
    """(dA [C,C], dbias [C] or None) of y = A x + b over all pixels (autograd of ActNorm + Conv1x1)"""
    dy = _prep(dy, "dy")
    x = _prep(x, "x")
    _bind_device(x)
    B, C = x.shape[0], x.shape[1]
    HW = 1
    for d in x.shape[2:]:
        HW *= d
    dA = torch.empty((C, C), dtype=torch.float32, device=x.device)
    db = torch.empty(C, dtype=torch.float32, device=x.device) if want_bias else None
    nbytes = load().finc_affine1x1_backward_weight_workspace_bytes(B, C, HW)
    ws = torch.empty(max(nbytes, 64), dtype=torch.uint8, device=x.device)
    _check(load().finc_affine1x1_backward_weight_f32(dy.data_ptr(), x.data_ptr(), dA.data_ptr(),
                                                     0 if db is None else db.data_ptr(), ws.data_ptr(), ws.numel(),
                                                     B, C, HW, _stream(x)), "finc_affine1x1_backward_weight_f32", 2)
    return dA, db


def slogdet_inverse(W):
    """(log|det W_i| [n], W_i^-1 [n, C, C]) of a batch of small matrices in one launch, no host sync"""
    W = _prep(W, "W")
    _bind_device(W)
    n, C = int(W.shape[0]), int(W.shape[-1])
    ld = torch.empty(n, dtype=torch.float32, device=W.device)
    Winv = torch.empty_like(W)
    _check(load().finc_slogdet_inverse_f32(W.data_ptr(), ld.data_ptr(), Winv.data_ptr(), n, C, _stream(W)),
           "finc_slogdet_inverse_f32")
    return ld, Winv


def preprocess(x, noise=None, alpha=1e-6, reverse=False, want_logdet=True):
    """dequantise + normalise + logit (and their log-determinants) in one kernel; reverse = sigmoid ... floor
    (fastflow_cifar_multi_gpu.py:162-186)"""
    x = _prep(x, "x")
    _bind_device(x)
    B = int(x.shape[0])
    D = x.numel() // max(B, 1)
    y = torch.empty_like(x)
    logdet = torch.empty(B, dtype=torch.float32, device=x.device) if (want_logdet and not reverse) else None
    if noise is not None:
        noise = _prep(noise, "noise")
    _check(load().finc_preprocess_f32(x.data_ptr(), None if noise is None else noise.data_ptr(), y.data_ptr(),
                                      None if logdet is None else logdet.data_ptr(), B, D, float(alpha), int(reverse),
                                      _stream(x)), "finc_preprocess_f32")
    return y, logdet


# ---------------------------------------------------------------------------------------------
# tensor-core path (tcgen05 / TMEM / TMA tensor maps)
# ---------------------------------------------------------------------------------------------
def _round_up(v, m):
    return (v + m - 1) // m * m


def tc_conv_prepare_weights(w, mode=0):
    """hi / lo TF32 split of an OIHW conv weight in the K-major layout of finc_tc_conv_nhwc_f32
    (mode 0 = as is, 1 = im2col form of a 3x3, 2 = transposed + flipped for backward-data)"""
    w = _prep(w, "weight")
    _bind_device(w)
    N, Cin, kh, kw = (int(v) for v in w.shape)
    taps = kh * kw
    nbytes = load().finc_tc_conv_weights_bytes(N, Cin, taps, mode)
    if nbytes == 0:
        raise FincNativeError(f"tc_conv_prepare_weights: unsupported weight shape {tuple(w.shape)}")
    out = torch.empty(nbytes // 4, dtype=torch.float32, device=w.device)
    _check(load().finc_tc_conv_prepare_weights_f32(w.data_ptr(), out.data_ptr(), N, Cin, taps, mode, _stream(w)),
           "finc_tc_conv_prepare_weights_f32")
    return out


def tc_conv_nhwc(x, wprep, bias, Npad, taps, relu=False, relu_mask=None, flags=0, out=None):
    """channels-last conv on the tensor cores: x [B,H,W,Cin_pad] -> y [B,H,W,Npad] (both padded to 32)"""
    x = _prep(x, "x")
    _bind_device(x)
    B, H, W, Cp = (int(v) for v in x.shape)
    y = torch.empty((B, H, W, Npad), dtype=torch.float32, device=x.device) if out is None else out
    _check(load().finc_tc_conv_nhwc_f32(x.data_ptr(), wprep.data_ptr(), bias.data_ptr(),
                                        None if relu_mask is None else relu_mask.data_ptr(), y.data_ptr(),
                                        B, H, W, Cp, Npad, taps, int(relu), flags, _stream(x)), "finc_tc_conv_nhwc_f32")
    return y


def tc_wgrad(P, Q, M=None, N=None, flags=0, out=None):
    """dW[m, n] = sum_p P[p, m] * Q[p, n] for channels-last activations P [..., ldP], Q [..., ldQ]"""
    P, Q = _prep(P, "P"), _prep(Q, "Q")
    _bind_device(P)
    ldP, ldQ = int(P.shape[-1]), int(Q.shape[-1])
    M = ldP if M is None else M
    N = ldQ if N is None else N
    npix = P.numel() // ldP
    nbytes = load().finc_tc_wgrad_workspace_bytes(npix, M, N)
    if nbytes == 0:
        raise FincNativeError(f"tc_wgrad: N={N} not covered (multiple of 64 needed)")
    ws = torch.empty(nbytes, dtype=torch.uint8, device=P.device)
    dW = torch.empty((M, N), dtype=torch.float32, device=P.device) if out is None else out
    _check(load().finc_tc_wgrad_f32(P.data_ptr(), Q.data_ptr(), dW.data_ptr(), ws.data_ptr(), ws.numel(), npix, M, N,
                                    ldP, ldQ, int(dW.stride(0)), flags, _stream(P)), "finc_tc_wgrad_f32", 2)
    return dW


def coupling_prepared_bytes(C, width, with_backward=False) -> int:
    """bytes of the prepared weight blob of one Coupling layer; 0 = not covered by the tensor-core path"""
    return int(load().finc_coupling_prepared_bytes(C, width, int(with_backward)))


def coupling_workspace_bytes(B, C, H, W, width) -> int:
    return int(load().finc_coupling_workspace_bytes(B, C, H, W, width))


def coupling_prepare(w1, b1, w2, b2, w3, b3, logs3, logscale_factor=3.0, out=None, with_backward=False):
    """weights of Coupling.net (layers/coupling.py:56-66) -> one prepared blob (uint8 tensor);
    with_backward adds the transposed weights the backward pass needs"""
    ts = [_prep(t, "coupling parameter") for t in (w1, b1, w2, b2, w3, b3, logs3)]
    _bind_device(ts[0])
    C, width = int(w3.shape[0]), int(w1.shape[0])
    nbytes = coupling_prepared_bytes(C, width, with_backward)
    if nbytes == 0:
        raise FincNativeError(f"coupling_prepare: C={C}, width={width} not covered by the tensor-core path")
    blob = out if (out is not None and out.numel() == nbytes) else torch.empty(nbytes, dtype=torch.uint8, device=ts[0].device)
    _check(load().finc_coupling_prepare_f32(*[t.data_ptr() for t in ts], float(logscale_factor), blob.data_ptr(),
                                            C, width, int(with_backward), _stream(ts[0])), "finc_coupling_prepare_f32",
           5 if with_backward else 4)
    return blob


_scratch = {}


def _shared_scratch(nbytes, device):
    """one transient scratch buffer per device, grown on demand (stream-ordered reuse)"""
    buf = _scratch.get(device)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(nbytes, dtype=torch.uint8, device=device)
        _scratch[device] = buf
    return buf


def coupling_backward(x, dy, dlogdet, blob, fwd_workspace, width, flags=0):
    """(dx, dw1, db1, dw2, db2, dw3, db3, dlogs3) of the coupling_apply call that filled `fwd_workspace` from input `x`;
    `blob` prepared with_backward.  flags | FLAG_COUPLING_REVERSE: that call was a reverse (reverse=True), and `dlogdet`
    is the gradient of its log-det."""
    x, dy = _prep(x, "x"), _prep(dy, "dy")
    _bind_device(x)
    B, C, H, W = (int(v) for v in x.shape)
    nbytes = int(load().finc_coupling_backward_workspace_bytes(B, C, H, W, width))
    if nbytes == 0:
        raise FincNativeError(f"coupling_backward: shape {tuple(x.shape)}, width {width} not covered")
    scratch = _shared_scratch(nbytes, x.device)
    f = dict(dtype=torch.float32, device=x.device)
    dx = torch.empty_like(x)
    dw1, db1 = torch.empty((width, C // 2, 3, 3), **f), torch.empty(width, **f)
    dw2, db2 = torch.empty((width, width, 1, 1), **f), torch.empty(width, **f)
    dw3, db3, dlogs3 = torch.empty((C, width, 3, 3), **f), torch.empty(C, **f), torch.empty(C, **f)
    if dlogdet is not None:
        dlogdet = _prep(dlogdet, "dlogdet")
    _check(load().finc_coupling_backward_f32(x.data_ptr(), dy.data_ptr(), None if dlogdet is None else dlogdet.data_ptr(),
                                             blob.data_ptr(), fwd_workspace.data_ptr(), scratch.data_ptr(), scratch.numel(),
                                             dx.data_ptr(), dw1.data_ptr(), db1.data_ptr(), dw2.data_ptr(), db2.data_ptr(),
                                             dw3.data_ptr(), db3.data_ptr(), dlogs3.data_ptr(), B, C, H, W, width, flags,
                                             _stream(x)), "finc_coupling_backward_f32", 24)
    return dx, dw1, db1, dw2, db2, dw3, db3, dlogs3


def coupling_apply(x, blob, width, reverse=False, want_logdet=None, logdet_out=None, flags=0, out=None, workspace=None):
    """Coupling.forward / .reverse (layers/coupling.py:85-99): y, logdet[B] or None.  The log-det is the direction's own
    (reverse: -sum log_s); by default it is computed for the forward and not for the reverse (want_logdet=True or
    `logdet_out` asks for it)."""
    x = _prep(x, "x")
    _bind_device(x)
    B, C, H, W = (int(v) for v in x.shape)
    y = torch.empty_like(x) if out is None else out
    nbytes = coupling_workspace_bytes(B, C, H, W, width)
    if nbytes == 0:
        raise FincNativeError(f"coupling_apply: shape {tuple(x.shape)}, width {width} not covered")
    ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device) if workspace is None else workspace
    logdet = None
    if want_logdet is None:
        want_logdet = not reverse
    if want_logdet or logdet_out is not None:
        logdet = torch.empty(B, dtype=torch.float32, device=x.device) if logdet_out is None else logdet_out
    _check(load().finc_coupling_apply_f32(x.data_ptr(), y.data_ptr(), None if logdet is None else logdet.data_ptr(),
                                          blob.data_ptr(), ws.data_ptr(), ws.numel(), B, C, H, W, width, int(reverse),
                                          flags, _stream(x)), "finc_coupling_apply_f32", 5)
    return y, logdet


def inverse_dense_bytes(G, C, H, W) -> int:
    """bytes of the dense-inverse table of one unit; 0 = shape not covered (n = C*H*W in [64, 1024], n % 64 == 0)"""
    return int(load().finc_inverse_dense_bytes(G, C, H, W))


def inverse_dense_prepare(w, H, W, G=4, orders=ORDERS_UNIT, out=None):
    """L^-1 of every group of a unit (hi / lo split, K-major), by running the wavefront inverse on the identity"""
    w = _prep(w, "weight")
    _bind_device(w)
    C, kH, kW = int(w.shape[1]), int(w.shape[2]), int(w.shape[3])
    nbytes = inverse_dense_bytes(G, C, H, W)
    if nbytes == 0:
        raise FincNativeError(f"inverse_dense_prepare: C={C}, H={H}, W={W} not covered")
    blob = torch.empty(nbytes, dtype=torch.uint8, device=w.device) if out is None else out
    scratch = _shared_scratch(int(load().finc_inverse_dense_scratch_bytes(G, C, H, W)), w.device)
    _check(load().finc_inverse_dense_prepare_f32(w.data_ptr(), blob.data_ptr(), scratch.data_ptr(), scratch.numel(),
                                                 G, C, H, W, kH, kW, orders, _stream(w)),
           "finc_inverse_dense_prepare_f32", 3)
    return blob


def inverse_dense(z, blob, G=4, flags=0, out=None):
    """x = L^-1 z as ONE block-diagonal tensor-core GEMM over all groups (same map as inverse(); fixed weights)"""
    z = _prep(z, "z")
    _bind_device(z)
    B, CT, H, W = (int(v) for v in z.shape)
    x = torch.empty_like(z) if out is None else out
    _check(load().finc_inverse_dense_f32(z.data_ptr(), blob.data_ptr(), x.data_ptr(), B, G, CT // G, H, W, flags,
                                         _stream(z)), "finc_inverse_dense_f32", G)
    return x


def chain_supported(G, C, H, W, ksize=(3, 3), with_affine=False) -> bool:
    return bool(load().finc_chain_supported(G, C, H, W, int(ksize[0]), int(ksize[1]), 1 if with_affine else 0))


def chain(x, w_units, out, G=4, orders=ORDERS_UNIT, A=None, bias=None, logdet_out=None, units=None, transpose=False,
          flags=0):
    """A chain of FInC units in ONE launch (C ABI: finc_chain_f32).

    x [B, G*C, H, W]; w_units [U, G*C, C, 3, 3] (contiguous); `units` = the unit indices in the order they are
    applied (an arithmetic sequence; default 0..U-1).  out [U, B, G*C, H, W]: unit u writes out[u]; or out
    [B, G*C, H, W]: only the result of the last unit is kept.  A [U, GC, GC] / bias [U, GC]: the affine map applied
    after each unit.  transpose=True: each unit's backward-data map.  logdet_out [B]: the chain's FInC logdet."""
    x = _prep(x, "x")
    w_units = _prep(w_units, "weights")
    _bind_device(x)
    U = int(w_units.shape[0])
    units = list(range(U)) if units is None else list(units)
    n = len(units)
    step = units[1] - units[0] if n > 1 else 1
    if (n > 1 and step == 0) or any(units[i + 1] - units[i] != step for i in range(n - 1)) or min(units) < 0 or max(units) >= U:
        raise FincNativeError("chain: `units` must be an arithmetic sequence inside [0, U)")
    B, CT, H, W = (int(v) for v in x.shape)
    C = CT // G
    if tuple(w_units.shape[1:]) != (CT, C, 3, 3):
        raise FincNativeError(f"chain: weights {tuple(w_units.shape)} do not match x {tuple(x.shape)} with G={G}")
    if out.dim() == 5:
        if tuple(out.shape) != (U, B, CT, H, W) or not out.is_contiguous():
            raise FincNativeError("chain: out must be a contiguous [U, B, G*C, H, W] tensor")
        y_stride = B * CT * H * W
    else:
        if tuple(out.shape) != tuple(x.shape) or not out.is_contiguous():
            raise FincNativeError("chain: out must be contiguous and shaped like x")
        y_stride = 0
    if (A is None) != (bias is None):
        raise FincNativeError("chain: A and bias come together")
    if A is not None:
        A, bias = _prep(A, "A"), _prep(bias, "bias")
        if tuple(A.shape) != (U, CT, CT) or tuple(bias.shape) != (U, CT):
            raise FincNativeError("chain: A must be [U, GC, GC] and bias [U, GC]")
    if transpose:
        flags |= FLAG_CHAIN_TRANSPOSE
    _check(load().finc_chain_f32(x.data_ptr(), w_units.data_ptr(), CT * C * 9, out.data_ptr(), y_stride,
                                 0 if A is None else A.data_ptr(), 0 if bias is None else bias.data_ptr(),
                                 0 if logdet_out is None else logdet_out.data_ptr(), B, G, C, H, W, 3, 3, orders,
                                 n, units[0], step, flags, _stream(x)), "finc_chain_f32")
    return out


def backward_weight_batched_workspace_bytes(B, G, C, H, W, kH, kW, n_units) -> int:
    return int(load().finc_backward_weight_batched_workspace_bytes(B, G, C, H, W, kH, kW, n_units))


def backward_weight_batched(dz_units, x_units, out_units, ksize, G=4, orders=ORDERS_UNIT, flags=0, workspace=None):
    """masked dW of U units in ONE launch: dz_units / x_units [U, B, G*C, H, W] (any uniform unit stride, each unit
    contiguous), out_units [U, G*C, C, kH, kW] (uniform unit stride).  C ABI: finc_backward_weight_batched_f32."""
    U, B, CT, H, W = (int(v) for v in dz_units.shape)
    C = CT // G
    for t in (dz_units, x_units):
        if t.dtype != torch.float32 or not t[0].is_contiguous() or tuple(t.shape) != (U, B, CT, H, W):
            raise FincNativeError("backward_weight_batched: [U, B, G*C, H, W] fp32 tensors with contiguous units expected")
    if tuple(out_units.shape) != (U, CT, C, int(ksize[0]), int(ksize[1])) or not out_units[0].is_contiguous():
        raise FincNativeError("backward_weight_batched: out must be [U, G*C, C, kH, kW] with contiguous units")
    _bind_device(dz_units)
    nbytes = int(load().finc_backward_weight_batched_workspace_bytes(B, G, C, H, W, int(ksize[0]), int(ksize[1]), U))
    if nbytes == 0:
        raise FincNativeError("backward_weight_batched: shape not covered", )
    if workspace is None:
        workspace = torch.zeros(nbytes, dtype=torch.uint8, device=dz_units.device)
    _check(load().finc_backward_weight_batched_f32(dz_units.data_ptr(), x_units.data_ptr(), out_units.data_ptr(),
                                                   workspace.data_ptr(), workspace.numel() * workspace.element_size(),
                                                   B, G, C, H, W, int(ksize[0]), int(ksize[1]), orders, flags, U,
                                                   dz_units.stride(0) if U > 1 else 0, x_units.stride(0) if U > 1 else 0,
                                                   out_units.stride(0) if U > 1 else 0, _stream(dz_units)),
           "finc_backward_weight_batched_f32")
    return out_units


def _inverse_level(z, tables, ksize, units, G, orders, out, what):
    """validated FincInverseLevel for one inverse chain (and its output tensor)"""
    units = list(units)
    n = len(units)
    step = units[1] - units[0] if n > 1 else 1
    if (n > 1 and step == 0) or any(units[i + 1] - units[i] != step for i in range(n - 1)) or min(units) < 0 \
            or max(units) >= tables.shape[0]:
        raise FincNativeError(f"{what}: `units` must be an arithmetic sequence of table rows")
    B, CT, H, W = (int(v) for v in z.shape)
    x = torch.empty_like(z) if out is None else out
    lv = FincInverseLevel(z.data_ptr(), tables.data_ptr(), tables.stride(0) * tables.element_size(), x.data_ptr(),
                          B, G, CT // G, H, W, int(ksize[0]), int(ksize[1]), orders, n, units[0], step)
    return lv, x


def inverse_chain(z, tables, ksize, units, G=4, orders=ORDERS_UNIT, out=None):
    """x = the inverse of the units `units` (an arithmetic sequence of rows of `tables`, applied in that order) in
    ONE launch; `tables` = [U, nbytes] FINC_PREP_INVERSE tables from prepare_weights.  Raises FincNativeError
    (rc FINC_E_UNSUPPORTED) when the shape is not covered -- callers fall back to one inverse() per unit."""
    z = _prep(z, "z")
    _bind_device(z)
    lv, x = _inverse_level(z, tables, ksize, units, G, orders, out, "inverse_chain")
    _check(load().finc_inverse_chain_f32(lv.z, lv.prepared, lv.prepared_stride_bytes, lv.x, lv.B, lv.G, lv.C, lv.H,
                                         lv.W, lv.kH, lv.kW, lv.orders, lv.n_units, lv.u_first, lv.u_step, _stream(z)),
           "finc_inverse_chain_f32")
    return x


def inverse_chain_multi(levels, G=4, orders=ORDERS_UNIT):
    """inverse_chain of several levels in ONE launch: `levels` = [(z, tables, ksize, units, out), ...] on one device
    and stream (out may be None).  Each result equals inverse_chain(z, tables, ksize, units, out=out) bit for bit.
    Raises FincNativeError (rc FINC_E_UNSUPPORTED) when the levels are not covered together -- callers fall back to
    one inverse_chain() per level.  Returns the outputs."""
    if not levels:
        raise FincNativeError("inverse_chain_multi: no levels")
    zs = [_prep(lv[0], "z") for lv in levels]
    if any(z.device != zs[0].device for z in zs):
        raise FincNativeError("inverse_chain_multi: all levels must be on one device")
    _bind_device(zs[0])
    arr = (FincInverseLevel * len(levels))()
    outs = []
    for i, (z, (_, tables, ksize, units, out)) in enumerate(zip(zs, levels)):
        arr[i], x = _inverse_level(z, tables, ksize, units, G, orders, out, "inverse_chain_multi")
        outs.append(x)
    _check(load().finc_inverse_chain_multi_f32(arr, len(levels), _stream(zs[0])), "finc_inverse_chain_multi_f32")
    return outs


def sm_count() -> int:
    return load().finc_sm_count()
