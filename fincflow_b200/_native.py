"""ctypes binding of libfincflow_b200.so (include/fincflow_b200.h) for torch tensors.

PyTorch is plumbing here: it owns device memory and streams; every kernel on the FInC hot
path is our own sm_100a code behind the C ABI.  There is NO CPU fallback: a missing
library or a non-CUDA tensor raises.

Every buffer the library writes (outputs, workspaces, prepared tables) is checked on the host before the call: device,
dtype, shape or size, layout.  A wrong buffer raises FincNativeError instead of becoming an out-of-bounds device write.
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


class FincNativeError(RuntimeError):
    pass


class FincInverseLevel(ctypes.Structure):
    """include/fincflow_b200.h: FincInverseLevel (the arguments of finc_inverse_chain_f32)"""
    _fields_ = [("z", ctypes.c_void_p), ("prepared", ctypes.c_void_p), ("prepared_stride_bytes", ctypes.c_size_t),
                ("x", ctypes.c_void_p)] + [(n, ctypes.c_int) for n in ("B", "G", "C", "H", "W", "kH", "kW")] + [
                ("orders", ctypes.c_uint), ("n_units", ctypes.c_int), ("u_first", ctypes.c_int), ("u_step", ctypes.c_int)]


_i, _u, _l, _f, _p, _sz = ctypes.c_int, ctypes.c_uint, ctypes.c_long, ctypes.c_float, ctypes.c_void_p, ctypes.c_size_t
_DIMS = [_i] * 7  # B, G, C, H, W, kH, kW
# name -> (restype, argtypes) of every function declared in include/fincflow_b200.h
_SIGNATURES = {
    "finc_abi_version": (_i, []),
    "finc_error_string": (ctypes.c_char_p, [_i]),
    "finc_set_device": (_i, [_i]),
    "finc_sm_count": (_i, []),
    "finc_forward_f32": (_i, [_p, _p, _p, _p, *_DIMS, _u, _u, _p]),
    "finc_backward_input_f32": (_i, [_p, _p, _p, *_DIMS, _u, _u, _p]),
    "finc_backward_weight_workspace_bytes": (_sz, _DIMS),
    "finc_backward_weight_f32": (_i, [_p, _p, _p, _p, _sz, *_DIMS, _u, _u, _p]),
    "finc_inverse_f32": (_i, [_p, _p, _p, *_DIMS, _u, _u, _p]),
    "finc_inverse_adjoint_f32": (_i, [_p, _p, _p, *_DIMS, _u, _u, _p]),
    "finc_apply_grad_mask_f32": (_i, [_p, _i, _i, _i, _i, _u, _p]),
    "finc_logdet_f32": (_i, [_p, _p, *_DIMS, _u, _p]),
    "finc_gaussian_logp_f32": (_i, [_p, _p, _p, _p, _f, _i, _l, _p]),
    "finc_adam_step_f32": (_i, [_p] * 5 + [_f] * 4 + [_l, _p]),
    "finc_allreduce_adam_f32": (_i, [_p] * 7 + [_f] * 5 + [_l, _i, _i, _p]),
    "finc_squeeze_f32": (_i, [_p, _p, _i, _i, _i, _i, _p]),
    "finc_unsqueeze_f32": (_i, [_p, _p, _i, _i, _i, _i, _p]),
    "finc_slogdet_inverse_f32": (_i, [_p, _p, _p, _i, _i, _p]),
    "finc_preprocess_f32": (_i, [_p, _p, _p, _p, _i, _l, _f, _i, _p]),
    "finc_affine1x1_f32": (_i, [_p, _p, _p, _p, _i, _i, _l, _p]),
    "finc_affine1x1_backward_weight_workspace_bytes": (_sz, [_i, _i, _l]),
    "finc_affine1x1_backward_weight_f32": (_i, [_p, _p, _p, _p, _p, _sz, _i, _i, _l, _p]),
    "finc_prepared_weights_bytes": (_sz, [_i, *_DIMS]),
    "finc_prepare_weights_f32": (_i, [_p, _p, _i, _i, _sz, _sz, *_DIMS, _u, _p]),
    "finc_tc_conv_weights_bytes": (_sz, [_i, _i, _i, _i]),
    "finc_tc_conv_prepare_weights_f32": (_i, [_p, _p, _i, _i, _i, _i, _p]),
    "finc_tc_conv_nhwc_f32": (_i, [_p] * 5 + [_i] * 7 + [_u, _p]),
    "finc_tc_wgrad_workspace_bytes": (_sz, [_l, _i, _i]),
    "finc_tc_wgrad_f32": (_i, [_p, _p, _p, _p, _sz, _l, _i, _i, _i, _i, _i, _u, _p]),
    "finc_coupling_prepared_bytes": (_sz, [_i, _i, _i]),
    "finc_coupling_workspace_bytes": (_sz, [_i] * 5),
    "finc_coupling_prepare_f32": (_i, [_p] * 7 + [_f, _p, _i, _i, _i, _p]),
    "finc_coupling_apply_f32": (_i, [_p] * 5 + [_sz] + [_i] * 6 + [_u, _p]),
    "finc_coupling_backward_workspace_bytes": (_sz, [_i] * 5),
    "finc_coupling_backward_f32": (_i, [_p] * 6 + [_sz] + [_p] * 8 + [_i] * 5 + [_u, _p]),
    "finc_inverse_dense_bytes": (_sz, [_i] * 4),
    "finc_inverse_dense_scratch_bytes": (_sz, [_i] * 4),
    "finc_inverse_dense_prepare_f32": (_i, [_p, _p, _p, _sz] + [_i] * 6 + [_u, _p]),
    "finc_inverse_dense_f32": (_i, [_p, _p, _p] + [_i] * 5 + [_u, _p]),
    "finc_backward_weight_batched_workspace_bytes": (_sz, [*_DIMS, _i]),
    "finc_backward_weight_batched_f32": (_i, [_p, _p, _p, _p, _sz, *_DIMS, _u, _u, _i, _l, _l, _l, _p]),
    "finc_inverse_chain_f32": (_i, [_p, _p, _sz, _p, *_DIMS, _u, _i, _i, _i, _p]),
    "finc_inverse_chain_multi_f32": (_i, [ctypes.POINTER(FincInverseLevel), _i, _p]),
    "finc_chain_supported": (_i, [_i] * 7),
    "finc_chain_f32": (_i, [_p, _p, _l, _p, _l, _p, _p, _p, *_DIMS, _u, _i, _i, _i, _u, _p]),
    "finc_debug_timestamps": (_i, [_p, _i]),
}
SYMBOLS = tuple(_SIGNATURES)

_lib = None
_tls = threading.local()
# kernels of ours enqueued through this module (bench.py's gpu_launches): each wrapper adds what its C entry point
# launches for the call's arguments (memset and copy nodes are not kernels).  One choice is the library's own and
# invisible here: whether the tiled kernel of finc_forward_f32 covers a shape depends on the device's shared memory
# and SM count (launch_conv_fast), so a forward with a log-det is counted as the tiled path's one fused launch
# unless FLAG_NAIVE forces the generic kernel plus the log-det kernel.
launch_count = 0


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
    for name, (restype, argtypes) in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = restype, argtypes
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
    """raise on an error code; on success count the call's kernel launches"""
    global launch_count
    if rc != 0:
        msg = load().finc_error_string(rc).decode()
        raise FincNativeError(f"{what} failed: {msg} (code {rc})")
    launch_count += launches


# ---- host checks of the tensors handed to the library ------------------------------------------------------------
def _input(t: torch.Tensor, name: str, device=None) -> torch.Tensor:
    """a float32 tensor the library reads, on `device` (any CUDA device when None); a contiguous copy if strided"""
    if not t.is_cuda:
        raise FincNativeError(f"{name} must be a CUDA tensor: fincflow_b200 has no CPU path")
    if device is not None and t.device != device:
        raise FincNativeError(f"{name} is on {t.device}, the call runs on {device}")
    if t.dtype != torch.float32:
        raise FincNativeError(f"{name} must be float32, got {t.dtype}")
    return t if t.is_contiguous() else t.contiguous()


def _output(t, name: str, device, shape, dtype=torch.float32, layout="contiguous") -> torch.Tensor:
    """`t`, a tensor the library writes (or reads laid out like one), checked against what the call writes: a CUDA
    tensor on `device` of this dtype and exact shape.  Layout: "contiguous"; "units" (each t[u] contiguous, the library
    takes the unit stride); "rows" (unit stride along the last dimension, the library takes the leading dimension).
    None: a new contiguous tensor."""
    if t is None:
        return torch.empty(shape, dtype=dtype, device=device)
    shape = tuple(int(v) for v in shape)
    if not t.is_cuda or t.device != device:
        raise FincNativeError(f"{name} must be a CUDA tensor on {device}, got one on {t.device}")
    if t.dtype != dtype:
        raise FincNativeError(f"{name} must be {dtype}, got {t.dtype}")
    if tuple(t.shape) != shape:
        raise FincNativeError(f"{name} must have shape {list(shape)}, got {list(t.shape)}")
    if t.numel() and not (t.stride(-1) == 1 if layout == "rows" else (t[0] if layout == "units" else t).is_contiguous()):
        raise FincNativeError(f"{name} must be dense ({layout}), got strides {list(t.stride())}")
    return t


def _bytes(t, name: str, device, nbytes: int, rows: int = 0, align: int = 1):
    """`t`, a uint8 buffer of at least `nbytes` bytes on `device` (a workspace, or a table); with `rows`, a stack of
    at least that many tables [n, >= nbytes] whose rows start `align`-byte aligned.  None: a new [nbytes] buffer."""
    if t is None:
        return torch.empty(int(nbytes), dtype=torch.uint8, device=device)
    if not t.is_cuda or t.device != device:
        raise FincNativeError(f"{name} must be a CUDA tensor on {device}, got one on {t.device}")
    if t.dtype != torch.uint8:
        raise FincNativeError(f"{name} must be uint8, got {t.dtype}")
    if t.dim() != (2 if rows else 1) or t.stride(-1) != 1 or t.shape[-1] < nbytes or (rows and t.shape[0] < rows):
        want = f"[>= {rows}, >= {nbytes}] with dense rows" if rows else f"[>= {nbytes}] contiguous"
        raise FincNativeError(f"{name} must be {want}, got {list(t.shape)} with strides {list(t.stride())}")
    if t.data_ptr() % align or (rows and t.stride(0) % align):
        raise FincNativeError(f"{name}: rows must start {align}-byte aligned")
    return t


def _table(t, name: str, device, kind: int, dims, rows: int = 0):
    """a prepared table (or a stack of them, one per unit) of `kind` for the FInC call of shape `dims` on `device`"""
    nbytes = prepared_weights_bytes(kind, *dims)
    if nbytes == 0 and dims[0] > 0:  # (B = 0 reads no table)
        raise FincNativeError(f"{name}: no prepared table covers the shape {dims} (use the raw weights)")
    return _bytes(t, name, device, nbytes, rows, 16)


def _dims(x: torch.Tensor, G: int, w=None, ksize=None):
    """(B, G, C, H, W, kH, kW) of a FInC call on x [B, G*C, H, W], with weights w [G*C, C, kH, kW] or a `ksize`"""
    B, CT, H, W = (int(v) for v in x.shape)
    if CT % G != 0:
        raise FincNativeError(f"channels {CT} not divisible by groups {G}")
    C = CT // G
    if w is not None:
        if w.dim() != 4 or tuple(w.shape[:2]) != (CT, C):
            raise FincNativeError(f"weight shape {tuple(w.shape)} does not match [G*C={CT}, C={C}, kH, kW]")
        ksize = w.shape[2:]
    return B, G, C, H, W, int(ksize[0]), int(ksize[1])


def _weights(x, w, G, flags, prepared, ksize, kind):
    """(dims, weights, flags) of forward / backward_input / inverse: the raw weights `w`, or a `prepared` table of
    `kind` built for this call's shape (with `ksize`; FLAG_PREPARED)"""
    if prepared is None:
        w = _input(w, "weight", x.device)
        return _dims(x, G, w=w), w, flags
    d = _dims(x, G, ksize=ksize)
    return d, _table(prepared, "prepared", x.device, kind, d), flags | FLAG_PREPARED


def _unit_sequence(units, n_rows: int, what: str):
    """(n, first, step) of `units`: a non-empty arithmetic sequence of indices in [0, n_rows)"""
    units = list(units)
    n = len(units)
    step = units[1] - units[0] if n > 1 else 1
    if n == 0 or step == 0 or any(b - a != step for a, b in zip(units, units[1:])) or min(units) < 0 \
            or max(units) >= n_rows:
        raise FincNativeError(f"{what}: `units` must be an arithmetic sequence inside [0, {n_rows})")
    return n, units[0], step


def _bind_device(t: torch.Tensor):
    """make the tensor's device the current CUDA device of this thread.  Checked against the runtime on every call
    (torch.cuda.current_device() is a cudaGetDevice): a cached value goes stale when torch switches devices
    (torch.cuda.set_device, leaving a `with torch.cuda.device(i)` block)."""
    dev = t.device.index
    if torch.cuda.current_device() != dev:
        _check(load().finc_set_device(dev), "finc_set_device", 0)


def _stream(t: torch.Tensor) -> int:
    return torch.cuda.current_stream(t.device).cuda_stream


def _numel(shape) -> int:
    n = 1
    for d in shape:
        n *= int(d)
    return n


# ---- FInC convolution ----------------------------------------------------------------------------------------------
def forward(x, w, G=4, orders=ORDERS_UNIT, want_logdet=True, flags=0, out=None, logdet_out=None, prepared=None,
            ksize=None):
    """z, logdet[B] (or None).  C ABI: finc_forward_f32.  With `logdet_out` and
    FLAG_LOGDET_ACCUMULATE the layer's logdet is added into a running [B] accumulator.
    `prepared` (a table from prepare_weights, with `ksize`) replaces `w`; no logdet then."""
    x = _input(x, "x")
    d, w, flags = _weights(x, w, G, flags, prepared, ksize, PREP_FORWARD)
    z = _output(out, "out", x.device, x.shape)
    logdet = None
    if want_logdet or logdet_out is not None:
        logdet = _output(logdet_out, "logdet_out", x.device, (d[0],))
    _bind_device(x)
    _check(load().finc_forward_f32(x.data_ptr(), w.data_ptr(), z.data_ptr(), None if logdet is None else logdet.data_ptr(),
                                   *d, orders, flags, _stream(x)), "finc_forward_f32",
           0 if d[0] == 0 else 2 if logdet is not None and flags & FLAG_NAIVE else 1)
    return z, logdet


def backward_input(dz, w, G=4, orders=ORDERS_UNIT, flags=0, out=None, prepared=None, ksize=None):
    dz = _input(dz, "dz")
    d, w, flags = _weights(dz, w, G, flags, prepared, ksize, PREP_BACKWARD_INPUT)
    dx = _output(out, "out", dz.device, dz.shape)
    _bind_device(dz)
    _check(load().finc_backward_input_f32(dz.data_ptr(), w.data_ptr(), dx.data_ptr(), *d, orders, flags,
                                          _stream(dz)), "finc_backward_input_f32", int(d[0] > 0))
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
    x = _input(x, "x")
    dz = _input(dz, "dz", x.device)
    d = _dims(x, G, ksize=ksize)
    B, _, C, _, _, kH, kW = d
    if dz.shape != x.shape:
        raise FincNativeError(f"dz {list(dz.shape)} must be shaped like x {list(x.shape)}")
    out = _output(out, "out", x.device, (G * C, C, kH, kW))
    nbytes = backward_weight_workspace_bytes(*d)
    if workspace is not None:
        flags |= FLAG_WORKSPACE_CLEAN  # caller-owned, zero-initialised once (see new_workspace): skips the memset node
    ws = _bytes(workspace, "workspace", x.device, max(nbytes, 16))
    _bind_device(x)
    _check(load().finc_backward_weight_f32(dz.data_ptr(), x.data_ptr(), out.data_ptr(), ws.data_ptr(), ws.numel(),
                                           *d, orders, flags, _stream(x)), "finc_backward_weight_f32")
    return out


def inverse(z, w, G=4, orders=ORDERS_UNIT, flags=0, out=None, prepared=None, ksize=None):
    z = _input(z, "z")
    d, w, flags = _weights(z, w, G, flags, prepared, ksize, PREP_INVERSE)
    x = _output(out, "out", z.device, z.shape)
    _bind_device(z)
    _check(load().finc_inverse_f32(z.data_ptr(), w.data_ptr(), x.data_ptr(), *d, orders, flags, _stream(z)),
           "finc_inverse_f32", int(d[0] > 0))
    return x


def inverse_adjoint(dx, w, G=4, orders=ORDERS_UNIT, flags=0, out=None):
    """dz = A^-T dx, the adjoint of inverse() (x = A^-1 z): <dx, inverse(z)> == <inverse_adjoint(dx), z>.
    `out` may be `dx` (in place).  C ABI: finc_inverse_adjoint_f32."""
    dx = _input(dx, "dx")
    w = _input(w, "weight", dx.device)
    d = _dims(dx, G, w=w)
    dz = _output(out, "out", dx.device, dx.shape)
    _bind_device(dx)
    _check(load().finc_inverse_adjoint_f32(dx.data_ptr(), w.data_ptr(), dz.data_ptr(), *d, orders, flags, _stream(dx)),
           "finc_inverse_adjoint_f32", int(d[0] > 0))
    return dz


def apply_grad_mask_(dw, G, orders):
    C, kH, kW = (int(v) for v in dw.shape[1:])
    dw = _output(dw, "dw", dw.device, (G * C, C, kH, kW))  # in place: must already be what the kernel writes
    _bind_device(dw)
    _check(load().finc_apply_grad_mask_f32(dw.data_ptr(), G, C, kH, kW, orders, _stream(dw)),
           "finc_apply_grad_mask_f32")
    return dw


def logdet(w, B, H, W, G=4, orders=ORDERS_UNIT):
    w = _input(w, "weight")
    _bind_device(w)
    C, kH, kW = int(w.shape[1]), int(w.shape[2]), int(w.shape[3])
    out = torch.empty(B, dtype=torch.float32, device=w.device)
    _check(load().finc_logdet_f32(w.data_ptr(), out.data_ptr(), B, G, C, H, W, kH, kW, orders, _stream(w)),
           "finc_logdet_f32", int(B > 0))
    return out


def gaussian_logp(z, logdet=None, dz_scale=None, logp_out=None, dz_out=None):
    """logp[B] of a standard normal (+ logdet) and optionally dz = dz_scale * z."""
    z = _input(z, "z")
    B = int(z.shape[0])
    D = z.numel() // max(B, 1)
    if logdet is not None:
        logdet = _input(logdet, "logdet", z.device)
    logp = _output(logp_out, "logp_out", z.device, (B,))
    dz = None if dz_scale is None else _output(dz_out, "dz_out", z.device, z.shape)
    _bind_device(z)
    _check(load().finc_gaussian_logp_f32(z.data_ptr(), None if logdet is None else logdet.data_ptr(), logp.data_ptr(),
                                         None if dz is None else dz.data_ptr(), float(dz_scale or 0.0), B, D,
                                         _stream(z)), "finc_gaussian_logp_f32", int(B > 0))
    return logp, dz


def prepared_weights_bytes(kind, B, G, C, H, W, kH, kW) -> int:
    """bytes of one unit's prepared table; 0 = shape not covered (do not use FLAG_PREPARED)"""
    return int(load().finc_prepared_weights_bytes(kind, B, G, C, H, W, kH, kW))


def prepare_weights(w_units, tables, kind, B, H, W, G=4, orders=ORDERS_UNIT):
    """w_units: [n_units, G*C, C, kH, kW] contiguous; tables: [n_units, bytes] uint8 -> filled in ONE launch"""
    w_units = _input(w_units, "weights")
    n, C, kH, kW = int(w_units.shape[0]), int(w_units.shape[2]), int(w_units.shape[3]), int(w_units.shape[4])
    if int(w_units.shape[1]) != G * C:
        raise FincNativeError(f"weights {list(w_units.shape)} must be [n_units, G*C, C, kH, kW] with G={G}")
    _table(tables, "tables", w_units.device, kind, (B, G, C, H, W, kH, kW), rows=n)
    _bind_device(w_units)
    _check(load().finc_prepare_weights_f32(w_units.data_ptr(), tables.data_ptr(), kind, n, w_units.stride(0),
                                           tables.stride(0), B, G, C, H, W, kH, kW, orders, _stream(w_units)),
           "finc_prepare_weights_f32")
    return tables


# ---- glue -----------------------------------------------------------------------------------------------------------
def adam_step_(param, grad, exp_avg, exp_avg_sq, step, lr=1e-3, betas=(0.9, 0.999), eps=1e-8):
    """in-place Adam on flat fp32 buffers; `step` is a 1-element float device tensor"""
    _bind_device(param)
    n = param.numel()
    _check(load().finc_adam_step_f32(param.data_ptr(), grad.data_ptr(), exp_avg.data_ptr(), exp_avg_sq.data_ptr(),
                                     step.data_ptr(), lr, betas[0], betas[1], eps, n, _stream(param)),
           "finc_adam_step_f32", 2 if n > 0 else 0)  # the update, then the step counter's tick
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
    x = _input(x, "x")
    B, C, H, W = x.shape
    y = _output(out, "out", x.device, (B, 4 * C, H // 2, W // 2))
    _bind_device(x)
    _check(load().finc_squeeze_f32(x.data_ptr(), y.data_ptr(), B, C, H, W, _stream(x)), "finc_squeeze_f32", int(B > 0))
    return y


def unsqueeze(x, out=None):
    """[B,4C,H,W] -> [B,C,2H,2W] (layers/squeeze.py:16-24)"""
    x = _input(x, "x")
    B, C4, H, W = x.shape
    y = _output(out, "out", x.device, (B, C4 // 4, 2 * H, 2 * W))
    _bind_device(x)
    _check(load().finc_unsqueeze_f32(x.data_ptr(), y.data_ptr(), B, C4, H, W, _stream(x)), "finc_unsqueeze_f32",
           int(B > 0))
    return y


def affine1x1(x, A, bias=None, out=None):
    """y[n,:,h,w] = A @ x[n,:,h,w] + bias: ActNorm followed by Conv1x1 (or their reverse / backward-data)
    as one per-pixel affine map (layers/actnorm.py:14-52, layers/conv1x1.py:18-43)"""
    x = _input(x, "x")
    A = _input(A, "A", x.device)
    B, C, HW = int(x.shape[0]), int(x.shape[1]), _numel(x.shape[2:])
    if tuple(A.shape) != (C, C):
        raise FincNativeError(f"A must be [{C}, {C}], got {tuple(A.shape)}")
    if bias is not None:
        bias = _input(bias, "bias", x.device)
        if bias.numel() != C:
            raise FincNativeError(f"bias must have {C} elements")
    y = _output(out, "out", x.device, x.shape)
    _bind_device(x)
    _check(load().finc_affine1x1_f32(x.data_ptr(), A.data_ptr(), 0 if bias is None else bias.data_ptr(), y.data_ptr(),
                                     B, C, HW, _stream(x)), "finc_affine1x1_f32", int(B > 0))
    return y


def affine1x1_backward_weight(dy, x, want_bias=True):
    """(dA [C,C], dbias [C] or None) of y = A x + b over all pixels (autograd of ActNorm + Conv1x1)"""
    x = _input(x, "x")
    dy = _input(dy, "dy", x.device)
    B, C, HW = int(x.shape[0]), int(x.shape[1]), _numel(x.shape[2:])
    dA = torch.empty((C, C), dtype=torch.float32, device=x.device)
    db = torch.empty(C, dtype=torch.float32, device=x.device) if want_bias else None
    nbytes = int(load().finc_affine1x1_backward_weight_workspace_bytes(B, C, HW))
    ws = torch.empty(max(nbytes, 64), dtype=torch.uint8, device=x.device)
    _bind_device(x)
    # B = 0: two memsets.  The generic kernel (one launch) keeps no partials: its workspace is the 16-float minimum;
    # the tiled path is the partial sums plus their reduction
    _check(load().finc_affine1x1_backward_weight_f32(dy.data_ptr(), x.data_ptr(), dA.data_ptr(),
                                                     0 if db is None else db.data_ptr(), ws.data_ptr(), ws.numel(),
                                                     B, C, HW, _stream(x)), "finc_affine1x1_backward_weight_f32",
           0 if B == 0 else 1 if nbytes <= 64 else 2)
    return dA, db


def slogdet_inverse(W):
    """(log|det W_i| [n], W_i^-1 [n, C, C]) of a batch of small matrices in one launch, no host sync"""
    W = _input(W, "W")
    _bind_device(W)
    n, C = int(W.shape[0]), int(W.shape[-1])
    ld = torch.empty(n, dtype=torch.float32, device=W.device)
    Winv = torch.empty_like(W)
    _check(load().finc_slogdet_inverse_f32(W.data_ptr(), ld.data_ptr(), Winv.data_ptr(), n, C, _stream(W)),
           "finc_slogdet_inverse_f32", int(n > 0))
    return ld, Winv


def preprocess(x, noise=None, alpha=1e-6, reverse=False, want_logdet=True):
    """dequantise + normalise + logit (and their log-determinants) in one kernel; reverse = sigmoid ... floor
    (fastflow_cifar_multi_gpu.py:162-186)"""
    x = _input(x, "x")
    _bind_device(x)
    B = int(x.shape[0])
    D = x.numel() // max(B, 1)
    y = torch.empty_like(x)
    logdet = torch.empty(B, dtype=torch.float32, device=x.device) if (want_logdet and not reverse) else None
    if noise is not None:
        noise = _input(noise, "noise", x.device)
    _check(load().finc_preprocess_f32(x.data_ptr(), None if noise is None else noise.data_ptr(), y.data_ptr(),
                                      None if logdet is None else logdet.data_ptr(), B, D, float(alpha), int(reverse),
                                      _stream(x)), "finc_preprocess_f32", int(B > 0))
    return y, logdet


# ---------------------------------------------------------------------------------------------
# tensor-core path (tcgen05 / TMEM / TMA tensor maps)
# ---------------------------------------------------------------------------------------------
def tc_conv_prepare_weights(w, mode=0):
    """hi / lo TF32 split of an OIHW conv weight in the K-major layout of finc_tc_conv_nhwc_f32
    (mode 0 = as is, 1 = im2col form of a 3x3, 2 = transposed + flipped for backward-data)"""
    w = _input(w, "weight")
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
    x = _input(x, "x")
    B, H, W, Cp = (int(v) for v in x.shape)
    y = _output(out, "out", x.device, (B, H, W, Npad))
    _bind_device(x)
    _check(load().finc_tc_conv_nhwc_f32(x.data_ptr(), wprep.data_ptr(), bias.data_ptr(),
                                        None if relu_mask is None else relu_mask.data_ptr(), y.data_ptr(),
                                        B, H, W, Cp, Npad, taps, int(relu), flags, _stream(x)), "finc_tc_conv_nhwc_f32")
    return y


def tc_wgrad(P, Q, M=None, N=None, flags=0, out=None):
    """dW[m, n] = sum_p P[p, m] * Q[p, n] for channels-last activations P [..., ldP], Q [..., ldQ]"""
    P = _input(P, "P")
    Q = _input(Q, "Q", P.device)
    ldP, ldQ = int(P.shape[-1]), int(Q.shape[-1])
    M = ldP if M is None else M
    N = ldQ if N is None else N
    npix = P.numel() // ldP
    nbytes = load().finc_tc_wgrad_workspace_bytes(npix, M, N)
    if nbytes == 0:
        raise FincNativeError(f"tc_wgrad: N={N} not covered (multiple of 64 needed)")
    dW = _output(out, "out", P.device, (M, N), layout="rows")
    ws = torch.empty(nbytes, dtype=torch.uint8, device=P.device)
    _bind_device(P)
    _check(load().finc_tc_wgrad_f32(P.data_ptr(), Q.data_ptr(), dW.data_ptr(), ws.data_ptr(), ws.numel(), npix, M, N,
                                    ldP, ldQ, int(dW.stride(0)), flags, _stream(P)), "finc_tc_wgrad_f32",
           2)  # the split-K GEMM, then the reduction of its slices
    return dW


def coupling_prepared_bytes(C, width, with_backward=False) -> int:
    """bytes of the prepared weight blob of one Coupling layer; 0 = not covered by the tensor-core path"""
    return int(load().finc_coupling_prepared_bytes(C, width, int(with_backward)))


def coupling_workspace_bytes(B, C, H, W, width) -> int:
    return int(load().finc_coupling_workspace_bytes(B, C, H, W, width))


def coupling_prepare(w1, b1, w2, b2, w3, b3, logs3, logscale_factor=3.0, out=None, with_backward=False):
    """weights of Coupling.net (layers/coupling.py:56-66) -> one prepared blob (uint8 tensor);
    with_backward adds the transposed weights the backward pass needs.  `out` is reused when it is a blob of the
    size this call writes, otherwise a new one is returned."""
    ts = [_input(w1, "coupling parameter")]
    ts += [_input(t, "coupling parameter", ts[0].device) for t in (b1, w2, b2, w3, b3, logs3)]
    dev = ts[0].device
    C, width = int(w3.shape[0]), int(w1.shape[0])
    nbytes = coupling_prepared_bytes(C, width, with_backward)
    if nbytes == 0:
        raise FincNativeError(f"coupling_prepare: C={C}, width={width} not covered by the tensor-core path")
    reuse = out is not None and out.device == dev and out.dtype == torch.uint8 and out.is_contiguous() \
        and out.numel() == nbytes
    blob = out if reuse else torch.empty(nbytes, dtype=torch.uint8, device=dev)
    _bind_device(ts[0])
    _check(load().finc_coupling_prepare_f32(*[t.data_ptr() for t in ts], float(logscale_factor), blob.data_ptr(),
                                            C, width, int(with_backward), _stream(ts[0])), "finc_coupling_prepare_f32",
           5 if with_backward else 4)  # three weight splits, the vectors, the transposed weights
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
    x = _input(x, "x")
    dy = _input(dy, "dy", x.device)
    if dlogdet is not None:
        dlogdet = _input(dlogdet, "dlogdet", x.device)
    B, C, H, W = (int(v) for v in x.shape)
    nbytes = int(load().finc_coupling_backward_workspace_bytes(B, C, H, W, width))
    if nbytes == 0:
        raise FincNativeError(f"coupling_backward: shape {tuple(x.shape)}, width {width} not covered")
    _bytes(fwd_workspace, "fwd_workspace", x.device, coupling_workspace_bytes(B, C, H, W, width))
    scratch = _shared_scratch(nbytes, x.device)
    f = dict(dtype=torch.float32, device=x.device)
    dx = torch.empty_like(x)
    dw1, db1 = torch.empty((width, C // 2, 3, 3), **f), torch.empty(width, **f)
    dw2, db2 = torch.empty((width, width, 1, 1), **f), torch.empty(width, **f)
    dw3, db3, dlogs3 = torch.empty((C, width, 3, 3), **f), torch.empty(C, **f), torch.empty(C, **f)
    _bind_device(x)
    # pointwise step, three (column sums: 2 launches, weight-gradient GEMM + slice reduction: 2, backward-data GEMM: 1)
    # rounds, the tap expansion, two weight unpacks, col2im: tc_api.cu finc_coupling_backward_f32
    _check(load().finc_coupling_backward_f32(x.data_ptr(), dy.data_ptr(), None if dlogdet is None else dlogdet.data_ptr(),
                                             blob.data_ptr(), fwd_workspace.data_ptr(), scratch.data_ptr(), scratch.numel(),
                                             dx.data_ptr(), dw1.data_ptr(), db1.data_ptr(), dw2.data_ptr(), db2.data_ptr(),
                                             dw3.data_ptr(), db3.data_ptr(), dlogs3.data_ptr(), B, C, H, W, width, flags,
                                             _stream(x)), "finc_coupling_backward_f32", 1 + 3 * 5 + 1 + 2 + 1)
    return dx, dw1, db1, dw2, db2, dw3, db3, dlogs3


def coupling_apply(x, blob, width, reverse=False, want_logdet=None, logdet_out=None, flags=0, out=None, workspace=None):
    """Coupling.forward / .reverse (layers/coupling.py:85-99): y, logdet[B] or None.  The log-det is the direction's own
    (reverse: -sum log_s); by default it is computed for the forward and not for the reverse (want_logdet=True or
    `logdet_out` asks for it).  `out` may be `x`."""
    x = _input(x, "x")
    B, C, H, W = (int(v) for v in x.shape)
    nbytes = coupling_workspace_bytes(B, C, H, W, width)
    if nbytes == 0:
        raise FincNativeError(f"coupling_apply: shape {tuple(x.shape)}, width {width} not covered")
    y = _output(out, "out", x.device, x.shape)
    ws = _bytes(workspace, "workspace", x.device, nbytes)
    if want_logdet is None:
        want_logdet = not reverse
    logdet = None
    if want_logdet or logdet_out is not None:
        logdet = _output(logdet_out, "logdet_out", x.device, (B,))
    _bind_device(x)
    # im2col, two 1x1-form convolutions, the nine-tap GEMM, the gather; the log-det's row reduction when asked for
    _check(load().finc_coupling_apply_f32(x.data_ptr(), y.data_ptr(), None if logdet is None else logdet.data_ptr(),
                                          blob.data_ptr(), ws.data_ptr(), ws.numel(), B, C, H, W, width, int(reverse),
                                          flags, _stream(x)), "finc_coupling_apply_f32", 5 + (logdet is not None))
    return y, logdet


def inverse_dense_bytes(G, C, H, W) -> int:
    """bytes of the dense-inverse table of one unit; 0 = shape not covered (n = C*H*W in [64, 1024], n % 64 == 0)"""
    return int(load().finc_inverse_dense_bytes(G, C, H, W))


def inverse_dense_prepare(w, H, W, G=4, orders=ORDERS_UNIT, out=None):
    """L^-1 of every group of a unit (hi / lo split, K-major), by running the wavefront inverse on the identity"""
    w = _input(w, "weight")
    C, kH, kW = int(w.shape[1]), int(w.shape[2]), int(w.shape[3])
    nbytes = inverse_dense_bytes(G, C, H, W)
    if nbytes == 0:
        raise FincNativeError(f"inverse_dense_prepare: C={C}, H={H}, W={W} not covered")
    blob = _bytes(out, "out", w.device, nbytes)
    _bind_device(w)
    scratch = _shared_scratch(int(load().finc_inverse_dense_scratch_bytes(G, C, H, W)), w.device)
    _check(load().finc_inverse_dense_prepare_f32(w.data_ptr(), blob.data_ptr(), scratch.data_ptr(), scratch.numel(),
                                                 G, C, H, W, kH, kW, orders, _stream(w)),
           "finc_inverse_dense_prepare_f32", 3)  # identity batch, its inverse, the table layout
    return blob


def inverse_dense(z, blob, G=4, flags=0, out=None):
    """x = L^-1 z as ONE block-diagonal tensor-core GEMM over all groups (same map as inverse(); fixed weights)"""
    z = _input(z, "z")
    B, G, C, H, W = _dims(z, G, ksize=(1, 1))[:5]  # (the dense table does not depend on the kernel size)
    nbytes = inverse_dense_bytes(G, C, H, W)
    if nbytes == 0:
        raise FincNativeError(f"inverse_dense: C={C}, H={H}, W={W} not covered")
    _bytes(blob, "blob", z.device, nbytes)
    x = _output(out, "out", z.device, z.shape)
    _bind_device(z)
    _check(load().finc_inverse_dense_f32(z.data_ptr(), blob.data_ptr(), x.data_ptr(), B, G, C, H, W, flags,
                                         _stream(z)), "finc_inverse_dense_f32", int(B > 0))
    return x


# ---- chains of FInC units --------------------------------------------------------------------------------------------
def chain_supported(G, C, H, W, ksize=(3, 3), with_affine=False) -> bool:
    return bool(load().finc_chain_supported(G, C, H, W, int(ksize[0]), int(ksize[1]), 1 if with_affine else 0))


def chain(x, w_units, out, G=4, orders=ORDERS_UNIT, A=None, bias=None, logdet_out=None, units=None, transpose=False,
          flags=0):
    """A chain of FInC units in ONE launch (C ABI: finc_chain_f32).

    x [B, G*C, H, W]; w_units [U, G*C, C, 3, 3] (contiguous); `units` = the unit indices in the order they are
    applied (an arithmetic sequence; default 0..U-1).  out [U, B, G*C, H, W] (each out[u] contiguous): unit u writes
    out[u]; or out [B, G*C, H, W]: only the result of the last unit is kept.  A [U, GC, GC] / bias [U, GC]: the affine
    map applied after each unit.  transpose=True: each unit's backward-data map.  logdet_out [B]: the chain's FInC
    logdet."""
    x = _input(x, "x")
    w_units = _input(w_units, "weights", x.device)
    U = int(w_units.shape[0])
    n, u_first, u_step = _unit_sequence(range(U) if units is None else units, U, "chain")
    B, _, C, H, W, _, _ = _dims(x, G, ksize=(3, 3))
    CT = G * C
    if tuple(w_units.shape[1:]) != (CT, C, 3, 3):
        raise FincNativeError(f"chain: weights {tuple(w_units.shape)} do not match x {tuple(x.shape)} with G={G}")
    if out is not None and out.dim() == 5:
        out = _output(out, "out", x.device, (U, B, CT, H, W), layout="units")
        y_stride = out.stride(0)
    else:
        out = _output(out, "out", x.device, x.shape)
        y_stride = 0
    if (A is None) != (bias is None):
        raise FincNativeError("chain: A and bias come together")
    if A is not None:
        A, bias = _input(A, "A", x.device), _input(bias, "bias", x.device)
        if tuple(A.shape) != (U, CT, CT) or tuple(bias.shape) != (U, CT):
            raise FincNativeError("chain: A must be [U, GC, GC] and bias [U, GC]")
    if logdet_out is not None:
        logdet_out = _output(logdet_out, "logdet_out", x.device, (B,))
    if transpose:
        flags |= FLAG_CHAIN_TRANSPOSE
    _bind_device(x)
    _check(load().finc_chain_f32(x.data_ptr(), w_units.data_ptr(), CT * C * 9, out.data_ptr(), y_stride,
                                 0 if A is None else A.data_ptr(), 0 if bias is None else bias.data_ptr(),
                                 0 if logdet_out is None else logdet_out.data_ptr(), B, G, C, H, W, 3, 3, orders,
                                 n, u_first, u_step, flags, _stream(x)), "finc_chain_f32", int(B > 0))
    return out


def backward_weight_batched_workspace_bytes(B, G, C, H, W, kH, kW, n_units) -> int:
    return int(load().finc_backward_weight_batched_workspace_bytes(B, G, C, H, W, kH, kW, n_units))


def backward_weight_batched(dz_units, x_units, out_units, ksize, G=4, orders=ORDERS_UNIT, flags=0, workspace=None):
    """masked dW of U units in ONE launch: dz_units / x_units [U, B, G*C, H, W] (any uniform unit stride, each unit
    contiguous), out_units [U, G*C, C, kH, kW] (uniform unit stride).  C ABI: finc_backward_weight_batched_f32."""
    if not dz_units.is_cuda:
        raise FincNativeError("dz_units must be a CUDA tensor: fincflow_b200 has no CPU path")
    dev = dz_units.device
    U = int(dz_units.shape[0])
    B, G, C, H, W, kH, kW = _dims(dz_units[0], G, ksize=ksize)
    for t, name in ((dz_units, "dz_units"), (x_units, "x_units")):  # read, but passed with their unit stride
        _output(t, name, dev, (U, B, G * C, H, W), layout="units")
    _output(out_units, "out_units", dev, (U, G * C, C, kH, kW), layout="units")
    nbytes = backward_weight_batched_workspace_bytes(B, G, C, H, W, kH, kW, U)
    if nbytes == 0:
        raise FincNativeError("backward_weight_batched: shape not covered")
    if workspace is None:
        workspace = torch.zeros(nbytes, dtype=torch.uint8, device=dev)
    _bytes(workspace, "workspace", dev, nbytes)
    _bind_device(dz_units)
    _check(load().finc_backward_weight_batched_f32(dz_units.data_ptr(), x_units.data_ptr(), out_units.data_ptr(),
                                                   workspace.data_ptr(), workspace.numel(),
                                                   B, G, C, H, W, kH, kW, orders, flags, U,
                                                   dz_units.stride(0) if U > 1 else 0, x_units.stride(0) if U > 1 else 0,
                                                   out_units.stride(0) if U > 1 else 0, _stream(dz_units)),
           "finc_backward_weight_batched_f32")
    return out_units


def _inverse_level(z, tables, ksize, units, G, orders, out, what):
    """validated FincInverseLevel for one inverse chain (and its output tensor)"""
    n, u_first, u_step = _unit_sequence(units, int(tables.shape[0]), what)
    d = _dims(z, G, ksize=ksize)
    _table(tables, "tables", z.device, PREP_INVERSE, d, rows=1)
    x = _output(out, "out", z.device, z.shape)
    lv = FincInverseLevel(z.data_ptr(), tables.data_ptr(), tables.stride(0), x.data_ptr(), *d, orders, n, u_first,
                          u_step)
    return lv, x


def inverse_chain(z, tables, ksize, units, G=4, orders=ORDERS_UNIT, out=None):
    """x = the inverse of the units `units` (an arithmetic sequence of rows of `tables`, applied in that order) in
    ONE launch; `tables` = [U, nbytes] FINC_PREP_INVERSE tables from prepare_weights.  Raises FincNativeError
    (rc FINC_E_UNSUPPORTED) when the shape is not covered -- callers fall back to one inverse() per unit."""
    z = _input(z, "z")
    lv, x = _inverse_level(z, tables, ksize, units, G, orders, out, "inverse_chain")
    _bind_device(z)
    _check(load().finc_inverse_chain_f32(lv.z, lv.prepared, lv.prepared_stride_bytes, lv.x, lv.B, lv.G, lv.C, lv.H,
                                         lv.W, lv.kH, lv.kW, lv.orders, lv.n_units, lv.u_first, lv.u_step, _stream(z)),
           "finc_inverse_chain_f32", int(lv.B > 0))
    return x


def inverse_chain_multi(levels, G=4, orders=ORDERS_UNIT):
    """inverse_chain of several levels in ONE launch: `levels` = [(z, tables, ksize, units, out), ...] on one device
    and stream (out may be None).  Each result equals inverse_chain(z, tables, ksize, units, out=out) bit for bit.
    Raises FincNativeError (rc FINC_E_UNSUPPORTED) when the levels are not covered together -- callers fall back to
    one inverse_chain() per level.  Returns the outputs."""
    if not levels:
        raise FincNativeError("inverse_chain_multi: no levels")
    zs = [_input(levels[0][0], "z")]
    zs += [_input(lv[0], "z", zs[0].device) for lv in levels[1:]]
    arr = (FincInverseLevel * len(levels))()
    outs = []
    for i, (z, (_, tables, ksize, units, out)) in enumerate(zip(zs, levels)):
        arr[i], x = _inverse_level(z, tables, ksize, units, G, orders, out, "inverse_chain_multi")
        outs.append(x)
    _bind_device(zs[0])
    _check(load().finc_inverse_chain_multi_f32(arr, len(levels), _stream(zs[0])), "finc_inverse_chain_multi_f32",
           int(any(lv.B > 0 for lv in arr)))
    return outs


def sm_count() -> int:
    return load().finc_sm_count()
