"""The reference's own CPU implementation of the hot path, for timing (TEST/BENCH INFRASTRUCTURE).

Used only by bench.py (`cpu_baseline` leg and `--impl reference`) and tests/.  It performs
exactly the library calls the reference performs on CPU tensors:

  forward   torch.chunk -> F.pad -> F.conv2d (bias-free) -> torch.cat     fastflow/fastflow.py:31-50,
                                                                         layers/conv.py:102-107
  backward  torch autograd (conv backward), then `grad * mask`            layers/conv.py:98-99,
                                                                         train/experiment.py:240-251
  inverse   per quadrant: flip -> float64 -> solve_parallel -> float32 -> flip   layers/conv.py:109-163,
            FastFlowUnit.reverse_level1 (fastflow.py:57-76); the solver is the reference's
            Cython `solve_parallel` compiled from its own .pyx into oracle/_ref (kind
            "reference"); if that file is absent the C restatement oracle/finc_oracle.c is
            used instead (kind "port").

The reference's shipped solver build has no OpenMP (1 thread).  To let the CPU arm use all
host cores, the batch is then sharded over a fork()ed process pool (each worker runs the
unmodified solver on its shard).  The C restatement used without that solver is OpenMP-parallel
itself and runs in the calling process.  `cores` reports the thread count.
"""
from __future__ import annotations

import math
import multiprocessing as mp
import os

import numpy as np
import torch
import torch.nn.functional as F

from . import build_ref
from . import finc_oracle as fo

ORDERS = ("TL", "TR", "BL", "BR")
_FLIP = {"TL": [], "TR": [3], "BL": [2], "BR": [2, 3]}
_solver = None


def solver_kind():
    return "reference" if build_ref.built_path() or os.path.exists(build_ref.REF_PYX) else "port"


def _get_solver():
    global _solver
    if _solver is None:
        _solver = build_ref.load() or False
    return _solver


def _pad(order, kH, kW):
    return {"TL": (kW - 1, 0, kH - 1, 0), "TR": (0, kW - 1, kH - 1, 0),
            "BL": (kW - 1, 0, 0, kH - 1), "BR": (0, kW - 1, 0, kH - 1)}[order]


def unit_forward(x, w4):
    """x [B,4Cq,H,W], w4 [4Cq,Cq,kH,kW] (stored orientation)"""
    kH, kW = w4.shape[2:]
    outs = []
    for xq, wq, order in zip(torch.chunk(x, 4, dim=1), torch.chunk(w4, 4, dim=0), ORDERS):
        outs.append(F.conv2d(F.pad(xq, _pad(order, kH, kW)), wq))
    return torch.cat(outs, dim=1)


def unit_mask(cq, ksize):
    return torch.from_numpy(np.concatenate([fo.grad_mask(cq, ksize, o) for o in ORDERS], 0))


def _solve_shard(args):
    z64, w64, ksize = args
    sol = _get_solver()
    if sol:
        return sol.solve_parallel(z64, w64, ksize)  # in place, returns its argument
    return fo.inverse(z64, w64, (0,), dtype=np.float64)


def unit_reverse(z, w4, pool=None, nshards=1):
    """FastFlowUnit.reverse_level1 on CPU tensors (flip to TL form, solve in f64, flip back)."""
    kH, kW = w4.shape[2:]
    jobs, meta = [], []
    for q, (zq, wq, order) in enumerate(zip(torch.chunk(z, 4, dim=1), torch.chunk(w4, 4, dim=0), ORDERS)):
        dims = _FLIP[order]
        zf = torch.flip(zq, dims) if dims else zq
        wf = torch.flip(wq, dims) if dims else wq
        z64 = np.asarray(zf.detach().numpy(), dtype=np.float64)
        w64 = np.ascontiguousarray(wf.detach().numpy(), dtype=np.float64)
        for shard in np.array_split(z64, min(nshards, z64.shape[0]), axis=0):
            jobs.append((np.ascontiguousarray(shard), w64, (kH, kW)))
            meta.append(q)
    res = pool.map(_solve_shard, jobs) if pool is not None else [_solve_shard(j) for j in jobs]
    outs = []
    for q, order in enumerate(ORDERS):
        y = torch.from_numpy(np.concatenate([r for r, m in zip(res, meta) if m == q], 0)).to(torch.float32)
        dims = _FLIP[order]
        outs.append(torch.flip(y, dims) if dims else y)
    return torch.cat(outs, dim=1)


class ReferenceCpuStack:
    """CPU twin of fincflow_b200.stack.FincStack + HotPathRunner (same step definition)."""

    def __init__(self, levels, batch, seed=0, lr=1e-3, threads=None):
        self.levels, self.B = levels, batch
        self.threads = threads or os.cpu_count() or 1
        torch.set_num_threads(self.threads)
        rng = np.random.default_rng(seed)
        self.weights, self.masks = [], []
        for lv in levels:
            ws = [torch.from_numpy(fo.init_unit_weight(lv.cq, lv.kernel_size, rng)).requires_grad_(True)
                  for _ in range(lv.n_units)]
            self.weights.append(ws)
            self.masks.append(unit_mask(lv.cq, lv.kernel_size))
        self.opt = torch.optim.Adam([w for ws in self.weights for w in ws], lr=lr)
        g = torch.Generator().manual_seed(seed)
        self.x = [torch.randn(batch, lv.channels, lv.height, lv.width, generator=g) for lv in levels]
        self.z = [torch.randn(batch, lv.channels, lv.height, lv.width, generator=g) for lv in levels]
        self.pool = None
        self.nshards = 1
        # the reference's solver runs on one thread, so the batch is sharded over forked workers; the C
        # restatement that stands in for it is OpenMP-parallel already, and forked workers that enter
        # OpenMP after the parent has used it crawl (20x slower per step on 8 cores) or stall
        if self.threads > 1 and _get_solver():
            self.nshards = min(self.threads, 32)
            self.pool = mp.get_context("fork").Pool(self.nshards)

    def close(self):
        if self.pool is not None:
            self.pool.terminate()
            self.pool = None

    def step(self):
        """same work as HotPathRunner.step: train step on x, then a sampling pass on z"""
        self.opt.zero_grad(set_to_none=True)
        logps = []
        for li, lv in enumerate(self.levels):
            h = self.x[li]
            for w in self.weights[li]:
                h = unit_forward(h, w)
            logdet = 0.0  # layers/conv.py:106
            logp = -0.5 * h.flatten(1).pow(2).sum(1) - 0.5 * lv.dim * math.log(2 * math.pi) + logdet
            logps.append(logp)
            (-logp.sum() / self.B).backward()
        for ws, m in zip(self.weights, self.masks):
            for w in ws:
                w.grad = w.grad * m  # PaddedConv2d.reset_gradients
        self.opt.step()
        samples = []
        with torch.no_grad():
            for li, lv in enumerate(self.levels):
                h = self.z[li]
                for w in reversed(self.weights[li]):
                    h = unit_reverse(h, w, self.pool, self.nshards)
                samples.append(h)
        return logps, samples


class ReferenceGpuStack:
    """The reference's own GPU path for the same step (bench.py `gpu_reference`, tests): forward /
    backward = torch.chunk -> F.pad -> F.conv2d -> torch.cat under autograd with TF32 off
    (fastflow/fastflow.py:31-50, layers/conv.py:102-107; the reference's CUDA 10.2 stack predates
    TF32), `grad * mask` (layers/conv.py:98-99), torch.optim.Adam, and sampling through
    FastFlowUnit.reverse_level2 (fastflow/fastflow.py:78-100) on the reference's CUDA extension
    compiled unmodified by oracle/build_ref_cuda.py: (H+W-1)*Cq launches + device syncs per unit
    (cinc_cuda_kernel_level2.cu:98-132)."""

    def __init__(self, levels, batch, device, seed=0, lr=1e-3):
        from . import build_ref_cuda

        self.ext = build_ref_cuda.load(2)
        if self.ext is None:
            raise RuntimeError("oracle/_ref/cinc_cuda_level2 was not built")
        self.levels, self.B, self.device = levels, batch, torch.device(device)
        rng = np.random.default_rng(seed)
        self.weights, self.masks = [], []
        for lv in levels:
            ws = [torch.from_numpy(fo.init_unit_weight(lv.cq, lv.kernel_size, rng)).to(self.device).requires_grad_(True)
                  for _ in range(lv.n_units)]
            self.weights.append(ws)
            self.masks.append(unit_mask(lv.cq, lv.kernel_size).to(self.device))
        self.opt = torch.optim.Adam([w for ws in self.weights for w in ws], lr=lr)
        g = torch.Generator(device=self.device).manual_seed(seed)
        self.x = [torch.randn(batch, lv.channels, lv.height, lv.width, generator=g, device=self.device) for lv in levels]
        self.z = [torch.randn(batch, lv.channels, lv.height, lv.width, generator=g, device=self.device) for lv in levels]

    def unit_reverse(self, z, w4):
        """fastflow/fastflow.py:78-100"""
        ks = [wq if not _FLIP[o] else torch.flip(wq, _FLIP[o]) for wq, o in zip(torch.chunk(w4, 4, dim=0), ORDERS)]
        kernel = torch.cat(ks, dim=0).contiguous()
        xs = [zq if not _FLIP[o] else torch.flip(zq, _FLIP[o]) for zq, o in zip(torch.chunk(z, 4, dim=1), ORDERS)]
        x = torch.cat(xs, dim=1).contiguous()
        y = torch.zeros_like(x).to(x.device)
        y = self.ext.inverse(x, kernel, y)[0]
        ys = [yq if not _FLIP[o] else torch.flip(yq, _FLIP[o]) for yq, o in zip(torch.chunk(y, 4, dim=1), ORDERS)]
        return torch.cat(ys, dim=1)

    def train_step(self):
        self.opt.zero_grad(set_to_none=True)
        for li, lv in enumerate(self.levels):
            h = self.x[li]
            for w in self.weights[li]:
                h = unit_forward(h, w)
            logp = -0.5 * h.flatten(1).pow(2).sum(1) - 0.5 * lv.dim * math.log(2 * math.pi)
            (-logp.sum() / self.B).backward()
        for ws, m in zip(self.weights, self.masks):
            for w in ws:
                w.grad = w.grad * m
        self.opt.step()

    def forward_only(self):
        with torch.no_grad():
            for li, lv in enumerate(self.levels):
                h = self.x[li]
                for w in self.weights[li]:
                    h = unit_forward(h, w)

    def sample(self):
        out = []
        with torch.no_grad():
            for li in range(len(self.levels)):
                h = self.z[li]
                for w in reversed(self.weights[li]):
                    h = self.unit_reverse(h, w.detach())
                out.append(h)
        return out
