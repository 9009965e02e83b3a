"""FincStack: a flow made of FastFlowUnits only (per level a chain of units + standard-normal
base), and HotPathRunner: its train step / sampling pass as CUDA graphs.

This is the reference's FlowSequential (fastflow/layers/flowsequential.py:21-44,89-115:
iterate layers, `logdet += layer_logdet`, `base.log_prob(z) + logdet`, reverse = iterate
reversed) restricted to the hot-path layer, i.e. the FInC-unit skeleton of the multi-scale
FastFlow models (fastflow/fastflow_cifar_multi_gpu.py:295-313: per level `block_size`
FastFlowSteps on [B, 4Cq, H, W]).  The Glow glue between the units (ActNorm, Conv1x1,
Coupling) is out of scope of the hot path (SURVEY.md section 8f).

B200-first choices:
  * all unit weights live in ONE flat parameter and all masked weight gradients in ONE flat
    bucket, written directly by the wgrad kernel -- the bucket is what NCCL all-reduces;
  * per-layer logdet is accumulated by the forward kernel's epilogue into one [B] vector;
  * a train step / sampling pass is a fixed launch sequence -> captured once per input slot
    in CUDA graphs (launch-bound: ~1 us of HBM traffic per unit at batch 256).
"""
from __future__ import annotations

import math
import os
from dataclasses import dataclass

import torch
import torch.nn as nn

from . import _native
from .layers.conv import ORDERS, init_finc_weight_
from .ops import finc_conv, finc_inverse


@dataclass(frozen=True)
class LevelSpec:
    channels: int   # 4*Cq
    height: int
    width: int
    n_units: int
    kernel_size: tuple = (3, 3)

    @property
    def cq(self):
        return self.channels // 4

    @property
    def unit_numel(self):
        return 4 * self.cq * self.cq * self.kernel_size[0] * self.kernel_size[1]

    @property
    def dim(self):
        return self.channels * self.height * self.width


# FInC-unit skeletons of the reference's model scripts (SURVEY.md section 8 shape table)
def cifar10_levels(n_units=16, k=3):
    """fastflow_cifar_multi_gpu.py:295-313 with n_blocks=3, block_size=16"""
    return [LevelSpec(12, 16, 16, n_units, (k, k)), LevelSpec(24, 8, 8, n_units, (k, k)),
            LevelSpec(48, 4, 4, n_units, (k, k))]


def mnist_levels(n_units=16, k=3):
    """fastflow_mnist_multi_gpu.py:299-314,414-416: n_blocks=2, block_size=16, ONE final step"""
    return [LevelSpec(4, 14, 14, n_units, (k, k)), LevelSpec(8, 7, 7, 1, (k, k))]


def imagenet32_levels(n_units=48, k=3):
    return cifar10_levels(n_units, k)


def imagenet64_levels(n_units=48, k=3):
    """fastflow_imagenet64_multi_gpu.py:299-314,424-426: 4 blocks x 48, ONE final step"""
    return [LevelSpec(12, 32, 32, n_units, (k, k)), LevelSpec(24, 16, 16, n_units, (k, k)),
            LevelSpec(48, 8, 8, n_units, (k, k)), LevelSpec(96, 4, 4, 1, (k, k))]


class FincStack(nn.Module):
    def __init__(self, levels):
        super().__init__()
        self.levels = list(levels)
        self.offsets = []
        off = 0
        for lv in self.levels:
            assert lv.channels % 4 == 0
            self.offsets.append([off + u * lv.unit_numel for u in range(lv.n_units)])
            off += lv.n_units * lv.unit_numel
        self.flat = nn.Parameter(torch.empty(off))
        self.reset_parameters()

    def reset_parameters(self):
        for li, lv in enumerate(self.levels):
            for u in range(lv.n_units):
                w = self.unit_weight(li, u).data
                for q, order in enumerate(ORDERS):
                    init_finc_weight_(w[q * lv.cq:(q + 1) * lv.cq], order)

    def unit_weight(self, li, u, flat=None):
        lv = self.levels[li]
        flat = self.flat if flat is None else flat
        o = self.offsets[li][u]
        return flat[o:o + lv.unit_numel].view(4 * lv.cq, lv.cq, *lv.kernel_size)

    # ---- autograd API (FlowSequential semantics, one level) --------------------------------
    def forward(self, x, level=0):
        """(z, logp[B]) = units of `level` applied in order, standard-normal base + logdet."""
        lv = self.levels[level]
        logdet = None
        for u in range(lv.n_units):
            x, ld = finc_conv(x, self.unit_weight(level, u), 4, _native.ORDERS_UNIT, True, True)
            logdet = ld if logdet is None else logdet + ld
        logp = -0.5 * x.flatten(1).pow(2).sum(1) - 0.5 * lv.dim * math.log(2 * math.pi) + logdet
        return x, logp

    def reverse(self, z, level=0):
        lv = self.levels[level]
        for u in reversed(range(lv.n_units)):
            z = finc_inverse(z, self.unit_weight(level, u))
        return z


def _carve(flat, shapes, align=64):
    """views of the given shapes into one flat fp32 buffer, each starting on a 256-byte boundary"""
    out, off = [], 0
    for shp in shapes:
        n = math.prod(shp)
        out.append(flat[off:off + n].view(shp))
        off += (n + align - 1) // align * align
    return out


def _carved_numel(shapes, align=64):
    return sum((math.prod(shp) + align - 1) // align * align for shp in shapes)


class _Slot:
    """static device buffers of one input slot (graphs replay on fixed addresses).

    Everything that crosses PCIe lives in two contiguous slabs per direction: `in_dev` / `in_host` hold the data
    batch of every level followed by the sampling latents of every level, `out_dev` / `out_host` the per-sample
    log-likelihoods followed by the generated samples -- a step is ONE host->device and ONE device->host copy
    (round 1 issued 3 + 6 small ones per step; at 8 ranks behind one host that cost 20 % of the end-to-end rate)."""

    def __init__(self, stack, B, device, pinned):
        f = dict(dtype=torch.float32, device=device)
        self.acts, self.logdet, self.logp, self.dzs, self.samp, self.zin = [], [], [], [], [], []
        self.x_host, self.z_host, self.logp_host, self.samp_host = [], [], [], []
        self.acts_blk, self.dzs_blk = [], []
        self.sample_out = {}
        self.ev_in, self.ev_computed, self.ev_out, self.ev_samp = (torch.cuda.Event() for _ in range(4))
        shapes = [(B, lv.channels, lv.height, lv.width) for lv in stack.levels]
        in_shapes = shapes + shapes                       # x of every level, then z of every level
        out_shapes = [(B,) for _ in shapes] + shapes      # logp of every level, then the samples
        self.n_x = _carved_numel(shapes)                  # the x part of the input slab (device_latents: only this is copied)
        self.in_dev = torch.zeros(_carved_numel(in_shapes), **f)
        self.out_dev = torch.zeros(_carved_numel(out_shapes), **f)
        in_views, out_views = _carve(self.in_dev, in_shapes), _carve(self.out_dev, out_shapes)
        L = len(shapes)
        for li, (lv, shp) in enumerate(zip(stack.levels, shapes)):
            # acts[u + 1] (output of unit u) and dzs[u] are slices of ONE tensor per level: the chain kernel writes
            # unit u's result at base + u * stride
            blk = torch.zeros((lv.n_units,) + shp, **f)
            self.acts_blk.append(blk)
            self.acts.append([in_views[li]] + [blk[u] for u in range(lv.n_units)])
            self.logdet.append(torch.zeros(B, **f))
            self.logp.append(out_views[li])
            dblk = torch.zeros((lv.n_units + 1,) + shp, **f)
            self.dzs_blk.append(dblk)
            self.dzs.append([dblk[u] for u in range(lv.n_units + 1)])  # dzs[u] = dL/d acts[u]
            self.zin.append(in_views[L + li])
            # the inverse chain ping-pongs between two buffers; the one its LAST unit writes is the slab view
            pp = [torch.zeros(shp, **f), torch.zeros(shp, **f)]
            pp[(lv.n_units - 1) % 2] = out_views[L + li]
            self.samp.append(pp)
        if pinned:
            self.in_host = torch.zeros(self.in_dev.numel(), dtype=torch.float32).pin_memory()
            self.out_host = torch.zeros(self.out_dev.numel(), dtype=torch.float32).pin_memory()
            hin, hout = _carve(self.in_host, in_shapes), _carve(self.out_host, out_shapes)
            self.x_host, self.z_host = hin[:L], hin[L:]
            self.logp_host, self.samp_host = hout[:L], hout[L:]


class HotPathRunner:
    """Train step (forward+logdet, base log-prob, backward dX + masked dW into the flat
    bucket, [all-reduce], Adam) and sampling pass (wavefront inverse chain) of a FincStack.

    The step order is the reference's Experiment.train_epoch (train/experiment.py:226-251):
    forward -> loss = -mean(logp) -> backward -> FInC gradient mask (here: inside the wgrad
    kernel) -> optimizer step; sampling is model.sample (train/experiment.py:327-337).
    """

    PHASES = ("forward_logdet", "backward", "optimizer", "inverse")
    # side streams for the mutually independent dW launches (swept 2/3/4/6/8 on B200: 6 is the knee)
    N_SIDE = int(os.environ.get("FINC_NSIDE", "6"))

    def __init__(self, stack: FincStack, batch: int, device, slots=1, lr=1e-3, host_io=False,
                 process_group=None, use_graphs=True, use_prepared=True, fused_collective=True,
                 device_latents=False, overlap_sampling=False, dense_inverse=False, level_parallel=False, chain=True,
                 batched_wgrad=True, multi_level_inverse=True):
        self.stack, self.B, self.device = stack, batch, torch.device(device)
        # chain: the forward pass of a level and its backward-data chain are ONE launch each (finc_chain_f32: the
        # image tiles stay in shared memory between units; all activations are still written) wherever the shape
        # is covered; bit-identical to the per-unit launches
        self.chain = [chain and _native.chain_supported(4, lv.cq, lv.height, lv.width, lv.kernel_size)
                      for lv in stack.levels]
        # dW of all units of a chained level in one launch (finc_backward_weight_batched_f32): own workspace per level
        self.wg_batched = []
        for lv, c in zip(stack.levels, self.chain):
            nb = _native.backward_weight_batched_workspace_bytes(batch, 4, lv.cq, lv.height, lv.width, *lv.kernel_size,
                                                                 lv.n_units - 1) if (c and batched_wgrad and lv.n_units > 2) else 0
            self.wg_batched.append(torch.zeros(nb, dtype=torch.uint8, device=self.device) if nb else None)
        self.inv_chain = [0] * len(stack.levels)   # units per inverse-chain launch: _probe_inverse_chain(), once the tables exist
        self._want_inv_chain = chain
        # multi_level_inverse: when every level's sampling chain is one whole launch, the chains of all levels run in
        # ONE launch (finc_inverse_chain_multi_f32; bit-identical): at small batches one level's chain leaves most
        # SMs idle, so the levels run side by side instead of one after another.  Set by _probe_inverse_chain().
        self._want_inv_multi = multi_level_inverse
        self.inv_multi = False
        # level_parallel: the levels of a FincStack have independent inputs, so their unit chains (forward,
        # dX, inverse) may run next to each other -- one stream per level, forked from and joined to the
        # current stream (inside a graph: parallel branches).  Batch-256 launches are latency-bound and do not
        # fill the GPU, so the chains overlap.  Off by default: per-phase launch durations stay clean.
        self.level_parallel = level_parallel and len(stack.levels) > 1
        self.level_streams = [torch.cuda.Stream(torch.device(device)) for _ in stack.levels] if self.level_parallel else None
        # dense_inverse: sampling with FIXED weights -- the deep, small levels (4x4 / 8x8 tiles, n = Cq*H*W <= 1024
        # unknowns per group) run x = L^-1 z as tensor-core GEMMs (finc_inverse_dense_f32); L^-1 is rebuilt by
        # prepare_dense() and NOT by the optimizer phase, so do not combine it with training steps
        self.dense_inverse = dense_inverse
        self.dense = {}
        self.pg = process_group
        self.world = 1 if process_group is None else torch.distributed.get_world_size(process_group)
        self.host_io, self.use_graphs = host_io, use_graphs
        # sampling latents z ~ N(0, I): drawn on the device inside the sampling graph, like the
        # reference's model.sample -> base_distribution.sample (train/experiment.py:327-337), instead of
        # travelling from the host
        self.device_latents = device_latents
        # overlap_sampling: the sampling pass (inverse phase) of step k runs on its own stream,
        # concurrently with the forward / backward phases of step k+1 -- both only READ the weights
        # produced by update k; update k+1 waits until that sampling pass has finished with the tables
        self.overlap_sampling = overlap_sampling
        self.samp_stream = torch.cuda.Stream(torch.device(device)) if overlap_sampling else None
        self._ev_samp_prev = None
        self.grad = torch.zeros_like(stack.flat.data)
        self.fused_collective = False
        if self.world > 1 and fused_collective:
            self._setup_peer_memory()
        stack.flat.grad = self.grad
        # Adam state for the flat parameter (one fused launch per step, finc_adam_step_f32)
        self.lr = lr
        self.exp_avg = torch.zeros_like(stack.flat.data)
        self.exp_avg_sq = torch.zeros_like(stack.flat.data)
        self.adam_step = torch.zeros(1, dtype=torch.float32, device=self.device)
        ws = 16
        for lv in stack.levels:
            ws = max(ws, _native.backward_weight_workspace_bytes(batch, 4, lv.cq, lv.height, lv.width,
                                                                 *lv.kernel_size))
        # the dW launches of different units are independent: fan them out over side streams
        # (one reduction workspace per stream: calls sharing a workspace must be stream-ordered)
        self.side = [torch.cuda.Stream(self.device) for _ in range(self.N_SIDE)]
        self.workspaces = [_native.new_workspace(ws, self.device) for _ in range(self.N_SIDE)]
        # prepared weight tables: one batched launch per (level, kind) after every weight update
        # instead of re-transposing the weights inside each of the 3*n_units launches
        self.tables = None
        if use_prepared:
            tabs = []
            for lv in stack.levels:
                nb = [_native.prepared_weights_bytes(kind, batch, 4, lv.cq, lv.height, lv.width, *lv.kernel_size)
                      for kind in (_native.PREP_FORWARD, _native.PREP_BACKWARD_INPUT, _native.PREP_INVERSE)]
                li = len(tabs)
                # a chained level stages the raw weights itself: only its inverse table is needed
                need = [k for k in range(3) if not (self.chain[li] and k != _native.PREP_INVERSE)]
                if min(nb[k] for k in need) == 0:
                    tabs.append(None)               # this level re-stages the raw weights in every launch
                    continue
                tabs.append([torch.empty((lv.n_units, nb[k]), dtype=torch.uint8, device=self.device) if k in need else None
                             for k in range(3)])
            self.tables = tabs
        self.slots = [_Slot(stack, batch, self.device, host_io) for _ in range(slots)]
        self.graphs = [None] * slots
        self.launches_per_step = None
        self.copy_graphs = [None] * slots
        self.copy_stream = torch.cuda.Stream(self.device) if host_io else None
        self.copy_out_stream = torch.cuda.Stream(self.device) if host_io else None

    def _setup_peer_memory(self):
        """Put the flat gradient bucket in symmetric (peer-mapped) memory so that the fused
        all-reduce + Adam kernel can read every rank's bucket over NVLink.  Any failure (no
        symmetric-memory support, no P2P) leaves the NCCL all-reduce path in place."""
        try:
            import torch.distributed._symmetric_memory as symm

            n = self.stack.flat.numel()
            bucket = symm.empty(n, dtype=torch.float32, device=self.device)
            handle = symm.rendezvous(bucket, self.pg.group_name)
            if handle.signal_pad_size < 2048:
                raise RuntimeError("signal pad too small")
            bucket.zero_()
            self.rank = torch.distributed.get_rank(self.pg)
            self.peer_grad = torch.tensor(list(handle.buffer_ptrs), dtype=torch.int64, device=self.device)
            # our flags live at byte 1024 of the pads, away from the slots torch's own barrier uses
            self.peer_signal = torch.tensor([p + 1024 for p in handle.signal_pad_ptrs], dtype=torch.int64,
                                            device=self.device)
            self.coll_local = torch.zeros(4, dtype=torch.int32, device=self.device)
            handle.barrier()  # pads and buckets are initialised everywhere before the first step
            self._symm = (bucket, handle)
            ok = True
        except Exception as e:  # pragma: no cover - depends on the machine
            self.fused_collective_error = repr(e)
            ok = False
        # every rank must take the same path: one rank falling back to NCCL while its peers spin in the
        # fused kernel would deadlock the job
        flag = torch.tensor([1 if ok else 0], dtype=torch.int32, device=self.device)
        torch.distributed.all_reduce(flag, op=torch.distributed.ReduceOp.MIN, group=self.pg)
        if int(flag.item()) == 1:
            self.grad = self._symm[0]
            self.fused_collective = True
        elif ok:
            self.fused_collective_error = "another rank could not set up peer memory"

    def _prepare_weights(self):
        """one batched launch per (level, kind); the launches are independent of each other, so they
        are fanned out over the side streams (fork / join on the current stream, graph-capturable)"""
        if self.tables is None:
            return
        st = self.stack
        main = torch.cuda.current_stream(self.device)
        fork = torch.cuda.Event()
        fork.record(main)
        k = 0
        for li, lv in enumerate(st.levels):
            if self.tables[li] is None:
                continue
            o = st.offsets[li][0]
            w_units = st.flat.detach()[o:o + lv.n_units * lv.unit_numel].view(lv.n_units, 4 * lv.cq, lv.cq, *lv.kernel_size)
            for kind in range(3):
                if self.chain[li] and kind != _native.PREP_INVERSE:
                    continue                        # the chain kernel stages the raw weights itself
                side = self.side[k % self.N_SIDE]
                if k < self.N_SIDE:
                    side.wait_event(fork)
                with torch.cuda.stream(side):
                    _native.prepare_weights(w_units, self.tables[li][kind], kind, self.B, lv.height, lv.width)
                k += 1
        for side in self.side[:min(k, self.N_SIDE)]:
            main.wait_stream(side)

    def prepare_dense(self, max_n=1024):
        """build the dense inverse tables (see dense_inverse) of the levels where the GEMM form is MEASURED faster
        than the wavefront kernel at this batch size (k=5 and the 4x4 levels: 2-5x; 8x8 at k=3: about even)"""
        self.dense = {}
        if not self.dense_inverse:
            return
        for li, lv in enumerate(self.stack.levels):
            n = lv.cq * lv.height * lv.width
            if n > max_n or _native.inverse_dense_bytes(4, lv.cq, lv.height, lv.width) == 0:
                continue
            w0 = self.stack.unit_weight(li, 0).detach().contiguous()
            blob = _native.inverse_dense_prepare(w0, lv.height, lv.width)
            z = torch.randn(self.B, 4 * lv.cq, lv.height, lv.width, device=self.device)
            out = torch.empty_like(z)
            times = []
            for fn in (lambda: _native.inverse(z, out=out, **self._w(li, 0, _native.PREP_INVERSE)), lambda: _native.inverse_dense(z, blob, out=out)):
                for _ in range(2):
                    fn()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(5):
                    fn()
                e1.record()
                e1.synchronize()
                times.append(e0.elapsed_time(e1))
            if times[1] < times[0]:
                self.dense[li] = [blob] + [_native.inverse_dense_prepare(self.stack.unit_weight(li, u).detach().contiguous(),
                                                                         lv.height, lv.width) for u in range(1, lv.n_units)]

    def _w(self, li, u, kind):
        """keyword arguments selecting the raw weights or the prepared table of unit (li, u)"""
        if self.tables is None or self.tables[li] is None:
            return dict(w=self.stack.unit_weight(li, u).detach())
        return dict(w=None, prepared=self.tables[li][kind][u], ksize=self.stack.levels[li].kernel_size)

    # ---- the four phases as plain launch sequences on the current stream ----------------------
    def _copy_in(self, s):
        """host -> device, ONE copy: this step's data batch (x) and sampling latents (z) of every level"""
        n = s.n_x if self.device_latents else s.in_dev.numel()
        s.in_dev[:n].copy_(s.in_host[:n], non_blocking=True)

    def _copy_out(self, s):
        """device -> host, ONE copy: per-sample log-likelihoods and the generated samples of every level"""
        s.out_host.copy_(s.out_dev, non_blocking=True)

    def _per_level(self, body):
        """run body(li, lv) for every level: in order on the current stream, or (level_parallel) each level on
        its own stream between a fork and a join on the current stream"""
        levels = list(enumerate(self.stack.levels))
        if not self.level_parallel:
            for li, lv in levels:
                body(li, lv)
            return
        main = torch.cuda.current_stream(self.device)
        fork = torch.cuda.Event()
        fork.record(main)
        for li, lv in levels:
            ls = self.level_streams[li]
            ls.wait_event(fork)
            with torch.cuda.stream(ls):
                body(li, lv)
        for ls in self.level_streams:
            main.wait_stream(ls)

    def _forward(self, s):
        self._per_level(lambda li, lv: self._forward_level(s, li, lv))

    def _units_w(self, li):
        lv, st = self.stack.levels[li], self.stack
        o = st.offsets[li][0]
        return st.flat.detach()[o:o + lv.n_units * lv.unit_numel].view(lv.n_units, 4 * lv.cq, lv.cq, *lv.kernel_size)

    def _forward_level(self, s, li, lv):
        if self.chain[li]:
            _native.chain(s.acts[li][0], self._units_w(li), s.acts_blk[li], logdet_out=s.logdet[li])
        else:
            for u in range(lv.n_units):
                flags = _native.FLAG_LOGDET_ACCUMULATE if u else 0
                _native.forward(s.acts[li][u], flags=flags, out=s.acts[li][u + 1], logdet_out=s.logdet[li],
                                **self._w(li, u, _native.PREP_FORWARD))
        # logp and dz = d(-mean_n logp)/dz = z / (B * world)
        _native.gaussian_logp(s.acts[li][lv.n_units], s.logdet[li], 1.0 / (self.B * self.world),
                              logp_out=s.logp[li], dz_out=s.dzs[li][lv.n_units])

    def _backward(self, s):
        """dX chain on the current stream; the masked dW of every unit -- written straight into
        the flat gradient bucket -- on side streams as soon as its dz exists.
        dzs[u] = dL/d acts[u]; the data gradient of unit 0 is never needed."""
        st = self.stack
        outer = torch.cuda.current_stream(self.device)
        used = set()                                # side streams that got work (only those can be joined)
        base = [0]
        for lv in st.levels:
            base.append(base[-1] + lv.n_units)

        def level(li, lv):
            main = torch.cuda.current_stream(self.device)
            k = base[li]
            if self.chain[li] and lv.n_units > 1:   # the whole dX chain first (one launch), then every dW at once
                _native.chain(s.dzs[li][lv.n_units], self._units_w(li), s.dzs_blk[li][:lv.n_units],
                              units=range(lv.n_units - 1, 0, -1), transpose=True)
                if self.wg_batched[li] is not None:
                    # dW of the units 1 .. U-1 in ONE launch (their x are slices of one tensor), unit 0 (x = the
                    # level's input) in a second one, on two side streams
                    U, o = lv.n_units, self.stack.offsets[li][0]
                    gw = self.grad[o:o + U * lv.unit_numel].view(U, 4 * lv.cq, lv.cq, *lv.kernel_size)
                    ready = torch.cuda.Event()
                    ready.record(main)
                    used.update(((2 * li) % self.N_SIDE, (2 * li + 1) % self.N_SIDE))
                    side = self.side[(2 * li) % self.N_SIDE]
                    side.wait_event(ready)
                    with torch.cuda.stream(side):
                        _native.backward_weight_batched(s.dzs_blk[li][2:U + 1], s.acts_blk[li][:U - 1], gw[1:],
                                                        lv.kernel_size, workspace=self.wg_batched[li])
                    side = self.side[(2 * li + 1) % self.N_SIDE]
                    side.wait_event(ready)
                    with torch.cuda.stream(side):
                        _native.backward_weight(s.dzs[li][1], s.acts[li][0], lv.kernel_size, out=gw[0],
                                                flags=_native.FLAG_QUARTER_GPU, workspace=self.workspaces[(2 * li + 1) % self.N_SIDE])
                    return
            ready = torch.cuda.Event()
            ready.record(main)                      # dzs[n] comes from the forward phase
            for u in reversed(range(lv.n_units)):
                side = self.side[k % self.N_SIDE]
                used.add(k % self.N_SIDE)
                side.wait_event(ready)
                with torch.cuda.stream(side):
                    _native.backward_weight(s.dzs[li][u + 1], s.acts[li][u], lv.kernel_size,
                                            out=st.unit_weight(li, u, self.grad), flags=_native.FLAG_QUARTER_GPU,
                                            workspace=self.workspaces[k % self.N_SIDE])
                k += 1
                if u > 0 and not self.chain[li]:
                    _native.backward_input(s.dzs[li][u + 1], out=s.dzs[li][u],
                                           **self._w(li, u, _native.PREP_BACKWARD_INPUT))
                    ready = torch.cuda.Event()
                    ready.record(main)

        self._per_level(level)
        for i in sorted(used):
            outer.wait_stream(self.side[i])

    def _optimizer(self, s):
        if self.fused_collective:
            # one kernel: cross-rank barrier, P2P reads of every rank's bucket over NVLink, Adam
            _native.allreduce_adam_(self.peer_grad.data_ptr(), self.peer_signal.data_ptr(), self.coll_local,
                                    self.stack.flat.data, self.exp_avg, self.exp_avg_sq, self.adam_step,
                                    self.rank, self.world, lr=self.lr)
            self._prepare_weights()
            return
        if self.world > 1:
            torch.distributed.all_reduce(self.grad, group=self.pg)  # NCCL over NVLink, training only
        _native.adam_step_(self.stack.flat.data, self.grad, self.exp_avg, self.exp_avg_sq, self.adam_step, lr=self.lr)
        self._prepare_weights()

    def _inverse(self, s):
        if self.inv_multi:
            if self.device_latents:
                for z in s.zin:
                    z.normal_()
            self._inverse_multi(s)
            return
        self._per_level(lambda li, lv: self._inverse_level(s, li, lv))

    def _inverse_multi(self, s):
        """the whole sampling chain of every level in one launch, into the buffer the per-level path ends in"""
        outs = _native.inverse_chain_multi([
            (s.zin[li], self.tables[li][_native.PREP_INVERSE], lv.kernel_size, range(lv.n_units - 1, -1, -1),
             s.samp[li][(lv.n_units - 1) % 2]) for li, lv in enumerate(self.stack.levels)])
        for li, x in enumerate(outs):
            s.sample_out[li] = x

    def _inverse_level(self, s, li, lv):
        if self.device_latents:
            s.zin[li].normal_()
        if self.inv_chain[li] and li not in self.dense:
            # the sampling chain of the level in sub-chains of `m` units (m = all of them when their tables fit shared
            # memory together): one launch each, tiles stay in shared memory, nothing written in between
            m, U = self.inv_chain[li], lv.n_units
            n_chunks = (U + m - 1) // m
            final = (U - 1) % 2                            # the buffer the per-unit path ends in (the out-slab view)
            src, cur, hi = s.zin[li], (final - (n_chunks - 1)) % 2, U - 1
            for _ in range(n_chunks):
                lo = max(hi - m + 1, 0)
                _native.inverse_chain(src, self.tables[li][_native.PREP_INVERSE], lv.kernel_size,
                                      range(hi, lo - 1, -1), out=s.samp[li][cur])
                src, cur, hi = s.samp[li][cur], cur ^ 1, lo - 1
            s.sample_out[li] = src
            return
        src, cur = s.zin[li], 0
        for u in reversed(range(lv.n_units)):
            if li in self.dense:
                _native.inverse_dense(src, self.dense[li][u], out=s.samp[li][cur])
            else:
                _native.inverse(src, out=s.samp[li][cur], **self._w(li, u, _native.PREP_INVERSE))
            src, cur = s.samp[li][cur], cur ^ 1
        s.sample_out[li] = src

    def _phase_fns(self):
        return (self._forward, self._backward, self._optimizer, self._inverse)

    # ---- graphs -------------------------------------------------------------------------------
    def prepare(self):
        """warm up eagerly (binds the device, sets kernel attributes), then capture one CUDA graph
        per (slot, phase).  The all-reduce stays outside graphs.

        Side-effect free for the model: the warm-up passes run every phase -- including the optimizer
        and, on several ranks, the gradient all-reduce -- on whatever the slot buffers hold (zeros
        unless the caller filled them), so the parameters and the Adam state (exp_avg, exp_avg_sq,
        step counter) are snapshotted before and restored after.  Slot buffers (activations,
        gradients, samples, host buffers) are scratch and ARE overwritten."""
        saved = [t.detach().clone() for t in (self.stack.flat.data, self.exp_avg, self.exp_avg_sq, self.adam_step)]
        try:
            self._prepare_warm_and_capture()
        finally:
            for dst, src in zip((self.stack.flat.data, self.exp_avg, self.exp_avg_sq, self.adam_step), saved):
                dst.copy_(src)
            self._prepare_weights()
            torch.cuda.synchronize(self.device)

    def _probe_inverse_chain(self):
        """per level: how many units one finc_inverse_chain_f32 launch solves (0 = the shape is not covered by the
        register-window kernel: one launch per unit).  All units when their tables fit shared memory together,
        otherwise the largest sub-chain that does."""
        self.inv_chain = [0] * len(self.stack.levels)
        if not self._want_inv_chain or self.tables is None:
            return
        s = self.slots[0]
        for li, lv in enumerate(self.stack.levels):
            U = lv.n_units
            if self.tables[li] is None:
                continue
            for m in sorted({U, (U + 1) // 2, (U + 2) // 3, (U + 3) // 4, 8, 4, 2}, reverse=True):
                if m < 2 or m > U:
                    continue
                try:
                    _native.inverse_chain(s.zin[li], self.tables[li][_native.PREP_INVERSE], lv.kernel_size,
                                          range(U - 1, U - 1 - m, -1), out=s.samp[li][(U - 1) % 2])
                    self.inv_chain[li] = m
                    break
                except _native.FincNativeError:
                    pass
        self.inv_multi = False
        if self._want_inv_multi and len(self.stack.levels) > 1 and not self.dense and \
                all(m == lv.n_units for m, lv in zip(self.inv_chain, self.stack.levels)):
            try:
                self._inverse_multi(s)
                self.inv_multi = True
            except _native.FincNativeError:
                pass

    def _prepare_warm_and_capture(self):
        self._prepare_weights()
        self.prepare_dense()
        self._probe_inverse_chain()
        for s in self.slots:
            if self.host_io:
                self._copy_in(s)
            for fn in self._phase_fns():
                fn(s)
            if self.host_io:
                self._copy_out(s)
        torch.cuda.synchronize(self.device)
        c0 = _native.launch_count
        for fn in self._phase_fns():
            fn(self.slots[0])
        self.launches_per_step = _native.launch_count - c0
        torch.cuda.synchronize(self.device)
        if not self.use_graphs:
            return
        for i, s in enumerate(self.slots):
            gs = []
            for name, fn in zip(self.PHASES, self._phase_fns()):
                if name == "optimizer" and self.world > 1 and not self.fused_collective:
                    gs.append(None)  # eager: NCCL all-reduce + Adam
                    continue
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    fn(s)
                gs.append(g)
            self.graphs[i] = gs
            if self.host_io:
                cg = {}
                for which, fn in (("in", self._copy_in), ("out", self._copy_out)):
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g):
                        fn(s)
                    cg[which] = g
                self.copy_graphs[i] = cg
        torch.cuda.synchronize(self.device)

    def run_phase(self, slot, phase_idx):
        s = self.slots[slot]
        g = self.graphs[slot][phase_idx] if self.graphs[slot] is not None else None
        if g is not None:
            g.replay()
        else:
            self._phase_fns()[phase_idx](s)

    def step(self, slot=0, events=None):
        """one full hot-path pass; `events` (len(PHASES)+1 torch.cuda.Event) get phase boundaries.

        With host_io the step is a three-stage pipeline over the slots: host->device copies of
        this step's inputs (copy-in stream), the four compute phases (current stream) and the
        device->host copies of its results (copy-out stream) are ordered by events per slot, so
        the copies of step k+1 / k-1 travel while step k computes.  Results of `slot` are valid on
        the host after `wait(slot)` (or `drain()`).

        With overlap_sampling the last phase (the sampling pass) runs on a second stream next to the
        forward / backward phases of the following step; phase events of that pass are recorded on its
        own stream, so phase durations overlap and no longer add up to the step time."""
        n = len(self.PHASES)
        s = self.slots[slot]
        main = torch.cuda.current_stream(self.device)
        if self.host_io:
            self.copy_stream.wait_event(s.ev_computed)   # previous use of this slot has read its inputs
            if self.overlap_sampling:
                self.copy_stream.wait_event(s.ev_samp)
            with torch.cuda.stream(self.copy_stream):
                self._replay_or_run(slot, "in", self._copy_in)
                s.ev_in.record(self.copy_stream)
            main.wait_event(s.ev_in)
            main.wait_event(s.ev_out)                    # previous results of this slot have left the device
        if not self.overlap_sampling:
            for p in range(n):
                if events is not None:
                    events[p].record()
                self.run_phase(slot, p)
            if events is not None:
                events[n].record()
        else:
            samp = self.samp_stream
            if self.host_io:
                main.wait_event(s.ev_samp)               # (slot reuse: its previous sampling pass is done)
            for p in range(n - 1):
                if events is not None:
                    events[p].record()
                if p == n - 2 and self._ev_samp_prev is not None:
                    main.wait_event(self._ev_samp_prev)  # the tables are rewritten by this phase
                self.run_phase(slot, p)
            ev_opt = torch.cuda.Event()
            ev_opt.record(main)
            samp.wait_event(ev_opt)
            with torch.cuda.stream(samp):
                if events is not None:
                    events[n - 1].record()
                self.run_phase(slot, n - 1)
                if events is not None:
                    events[n].record()
                s.ev_samp.record(samp)
            self._ev_samp_prev = s.ev_samp
        if self.host_io:
            s.ev_computed.record(main)
            self.copy_out_stream.wait_event(s.ev_computed)
            if self.overlap_sampling:
                self.copy_out_stream.wait_event(s.ev_samp)
            with torch.cuda.stream(self.copy_out_stream):
                self._replay_or_run(slot, "out", self._copy_out)
                s.ev_out.record(self.copy_out_stream)

    def _replay_or_run(self, slot, which, fn):
        g = self.copy_graphs[slot].get(which) if self.copy_graphs[slot] else None
        if g is not None:
            g.replay()
        else:
            fn(self.slots[slot])

    def wait(self, slot):
        """block the host until the results of the last step on `slot` are in its pinned buffers"""
        if self.host_io:
            self.slots[slot].ev_out.synchronize()

    def drain(self):
        """make the current stream wait for every outstanding host copy (so that an event recorded
        after drain() covers the whole pipeline)"""
        main = torch.cuda.current_stream(self.device)
        if self.overlap_sampling:
            main.wait_stream(self.samp_stream)
        if self.host_io:
            main.wait_stream(self.copy_stream)
            main.wait_stream(self.copy_out_stream)
