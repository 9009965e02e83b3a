#!/usr/bin/env python
"""bench.py -- FInC hot-path benchmark (driver contract in the task statement).

    python bench.py --gpus N --steps K --warmup W [--impl reference]

Workload (BASELINE.json configs[2], the config the metric's "1/2/4/8 B200" is quoted on):
the FInC-unit skeleton of the CIFAR-10-shaped FInCFlow -- 3 levels x 16 FastFlowUnits on
[256,12,16,16], [256,24,8,8], [256,48,4,4] (k=3), per-GPU batch 256 (weak scaling), fp32,
synthetic N(0,1) inputs, reference-initialised weights.  One step = one pass of the hot path
over one batch: forward+logdet (+standard-normal log-prob), backward dX, masked dW into the
flat gradient bucket, [NCCL all-reduce when N>1], Adam, then one inverse (sampling) pass.
metric = images/sec of that step (whole job, all GPUs).

  value  inputs resident in HBM; input/activation sets rotate over 3 slots (> L2 in total)
  e2e    the same step through the public API (HotPathRunner(host_io=True)): every step copies
         that step's data batch from pinned host memory and reads logp + samples back (the sampling
         latents are drawn on the device, as the reference's model.sample does)
  roofline  dominant kernel family: algorithmic bytes per launch / average launch duration,
         from CUDA events recorded at the phase boundaries inside the timed region
  cpu_baseline / --impl reference  the reference's own CPU path (torch CPU conv + autograd +
         its Cython wavefront solver from oracle/_ref) on the host cores, same step
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

PER_GPU_BATCH = 256
UNITS_PER_LEVEL = 16
KSIZE = 3
WORKLOAD = ("cifar10_finc_stack: FInC-unit skeleton of the CIFAR-10-shaped FInCFlow (BASELINE configs[2]): "
            "3 levels x 16 FastFlowUnits on [256,12,16,16],[256,24,8,8],[256,48,4,4], k=3; "
            "step = fwd+logdet+base logp, bwd dX, masked dW, Adam, inverse sampling pass")


def levels():
    from fincflow_b200.stack import cifar10_levels

    return cifar10_levels(UNITS_PER_LEVEL, KSIZE)


def extra_workload_specs(world):
    """the other configurations the metric names (BASELINE.json configs[0,1,3,4] + configs[2] with the
    GLOBAL batch fixed): name -> (levels, per-GPU batch, scaling, phases to run)"""
    from fincflow_b200.stack import LevelSpec, cifar10_levels, imagenet32_levels, imagenet64_levels, mnist_levels

    allp = ("forward_logdet", "backward", "optimizer", "inverse")
    return {
        "cfg1_single_layer": dict(levels=[LevelSpec(4, 14, 14, 1, (3, 3))], batch=64, scaling="weak", phases=allp,
                                  what="one FastFlowUnit(4) on the squeezed 1x28x28 MNIST shape, batch 64 per GPU"),
        "cfg2_mnist": dict(levels=mnist_levels(), batch=128, scaling="weak", phases=allp,
                           what="MNIST flow skeleton: 16 units [4,14,14] + 1 unit [8,7,7], batch 128 per GPU"),
        "cfg3_strong": dict(levels=cifar10_levels(UNITS_PER_LEVEL, KSIZE), batch=max(PER_GPU_BATCH // world, 1),
                            scaling="strong", phases=allp,
                            what="the headline workload with the GLOBAL batch fixed at 256 (256 / N per GPU)"),
        "cfg4_imagenet32": dict(levels=imagenet32_levels(), batch=512, scaling="weak", phases=allp,
                                what="ImageNet32 flow skeleton: 3 levels x 48 units, batch 512 per GPU"),
        "cfg5_imagenet64_k3": dict(levels=imagenet64_levels(48, 3), batch=max(1024 // world, 1), scaling="strong",
                                   phases=("inverse",), dense=True,
                                   what="ImageNet64 flow skeleton k=3 (48,48,48,1 units), SAMPLING only, 1024 images sharded by batch"),
        "cfg5_imagenet64_k5": dict(levels=imagenet64_levels(48, 5), batch=max(1024 // world, 1), scaling="strong",
                                   phases=("inverse",), dense=True,
                                   what="ImageNet64 flow skeleton k=5, SAMPLING only, 1024 images sharded by batch"),
    }


def run_extra_workloads(torch, dev, world, rank, pg, K, names=None):
    """phase times of the other named configurations through the same HotPathRunner (CUDA graphs, one
    slot); multi-GPU: every rank runs its shard, times are the max over ranks"""
    from fincflow_b200.stack import FincStack, HotPathRunner

    out = []
    K = max(3, min(K, 20))
    for name, spec in extra_workload_specs(world).items():
        if names is not None and name not in names:
            continue
        try:
            torch.manual_seed(0)
            stack = FincStack(spec["levels"]).to(dev)
            B = spec["batch"]
            runner = HotPathRunner(stack, B, dev, slots=1, process_group=pg if "optimizer" in spec["phases"] else None,
                                   dense_inverse=spec.get("dense", False))
            g = torch.Generator(device=dev).manual_seed(4000 + rank)
            for li in range(len(spec["levels"])):
                runner.slots[0].acts[li][0].normal_(generator=g)
                runner.slots[0].zin[li].normal_(generator=g)
            runner.prepare()
            idx = [HotPathRunner.PHASES.index(p) for p in spec["phases"]]
            for _ in range(3):
                for p in idx:
                    runner.run_phase(0, p)
            if world > 1:
                torch.distributed.barrier()
            torch.cuda.synchronize(dev)
            evs = [[torch.cuda.Event(enable_timing=True) for _ in range(len(idx) + 1)] for _ in range(K)]
            for i in range(K):
                for j, p in enumerate(idx):
                    evs[i][j].record()
                    runner.run_phase(0, p)
                evs[i][len(idx)].record()
            torch.cuda.synchronize(dev)
            tot = evs[0][0].elapsed_time(evs[K - 1][len(idx)]) / K
            ph = [sum(evs[i][j].elapsed_time(evs[i][j + 1]) for i in range(K)) / K for j in range(len(idx))]
            t = torch.tensor([tot] + ph, device=dev, dtype=torch.float64)
            if world > 1:
                torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
            tot, ph = float(t[0]), [float(v) for v in t[1:]]
            pm = dict(zip(spec["phases"], ph))
            gb = B * world
            elems = sum(lv.n_units * B * lv.dim for lv in spec["levels"])
            ips = {}
            if "forward_logdet" in pm:
                ips["forward_logdet"] = round(gb / (pm["forward_logdet"] * 1e-3))
                ips["train_step"] = round(gb / ((pm["forward_logdet"] + pm["backward"] + pm["optimizer"]) * 1e-3))
            if "inverse" in pm:
                ips["inverse_sampling"] = round(gb / (pm["inverse"] * 1e-3))
            peak, _ = measured_peak()
            out.append({"name": name, "what": spec["what"], "per_gpu_batch": B, "global_batch": gb,
                        "scaling": spec["scaling"], "steps": K, "ms_per_step": round(tot, 4),
                        "phases_ms": {k: round(v, 4) for k, v in pm.items()}, "images_per_s": ips,
                        "dense_inverse_levels": sorted(runner.dense), "inverse_chain_units_per_launch": list(runner.inv_chain),
                        "frac_of_hbm_peak": {k: round(8 * elems * (1.5 if k == "backward" else 1.0) / (v * 1e-3) / 1e9 / peak, 4)
                                             for k, v in pm.items() if k != "optimizer"}})
            del runner, stack
            torch.cuda.empty_cache()
        except Exception as e:  # never fail the bench line over an extra workload
            out.append({"name": name, "error": repr(e)})
    return out


def fused_vs_nccl_check(torch, dev, rank, pg):
    """N > 1: three training steps of a small stack through the fused NVLink all-reduce + Adam kernel and through
    NCCL all-reduce + Adam from identical states: max |parameter difference| between the two paths (fp32 summation
    order differs: <= 1e-5) -- the driver-visible form of tests/multirank_check.py"""
    from fincflow_b200.stack import FincStack, HotPathRunner, LevelSpec

    try:
        lv = [LevelSpec(12, 8, 8, 3, (3, 3)), LevelSpec(24, 4, 4, 2, (3, 3))]
        res = {}
        for fused in (True, False):
            torch.manual_seed(0)
            stack = FincStack(lv).to(dev)
            runner = HotPathRunner(stack, 8, dev, slots=1, lr=1e-2, process_group=pg, fused_collective=fused)
            if fused and not runner.fused_collective:
                return {"skipped": getattr(runner, "fused_collective_error", "no peer memory")}
            g = torch.Generator(device=dev).manual_seed(100 + rank)
            for li in range(len(lv)):
                runner.slots[0].acts[li][0].normal_(generator=g)
                runner.slots[0].zin[li].normal_(generator=g)
            runner.prepare()          # side-effect free: parameters and Adam state are restored
            for _ in range(3):
                runner.step(0)
            torch.cuda.synchronize(dev)
            res[fused] = stack.flat.detach().clone()
            del runner
        d = (res[True] - res[False]).abs().max().reshape(1).double()
        torch.distributed.all_reduce(d, op=torch.distributed.ReduceOp.MAX)
        return {"max_abs_param_diff": float(d.item()), "steps": 3}
    except Exception as e:
        return {"error": repr(e)}


def gpu_reference_detail(torch, dev, ours_phase_ms):
    """the REFERENCE's own GPU path on the same box, same step: F.pad + conv2d fwd / autograd bwd with TF32
    off + `grad * mask` + Adam, and FastFlowUnit.reverse_level2 on the reference's CUDA extension (compiled
    unmodified into oracle/_ref by oracle/build_ref_cuda.py)"""
    try:
        from oracle.reference_path import ReferenceGpuStack

        old = torch.backends.cudnn.allow_tf32
        torch.backends.cudnn.allow_tf32 = False
        ref = ReferenceGpuStack(levels(), PER_GPU_BATCH, dev)

        def timed(fn, n):
            fn()
            torch.cuda.synchronize(dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(n):
                fn()
            e1.record()
            e1.synchronize()
            return e0.elapsed_time(e1) / n

        fwd = timed(ref.forward_only, 5)
        train = timed(ref.train_step, 5)
        samp = timed(ref.sample, 2)
        torch.backends.cudnn.allow_tf32 = old
        ours_train = ours_phase_ms["forward_logdet"] + ours_phase_ms["backward"] + ours_phase_ms["optimizer"]
        B = PER_GPU_BATCH
        return {"what": "reference GPU path (PyTorch/cuDNN fp32 with TF32 off + its cinc_cuda_level2 extension), same workload, 1 GPU",
                "forward_ms": round(fwd, 3), "train_step_ms": round(train, 3), "sample_ms": round(samp, 3),
                "images_per_s": {"forward_logdet": round(B / fwd * 1e3), "train_step": round(B / train * 1e3),
                                 "inverse_sampling": round(B / samp * 1e3)},
                "speedup_ours": {"forward_logdet": round(fwd / ours_phase_ms["forward_logdet"], 1),
                                 "train_step": round(train / ours_train, 1),
                                 "inverse_sampling": round(samp / ours_phase_ms["inverse"], 1)}}
    except Exception as e:
        return {"error": repr(e)}


def measured_peak():
    try:
        with open(os.path.join(REPO, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md: 6.65 TB/s)"


# ------------------------------------------------------------------------------------------
# clocks sampled DURING the timed region
# ------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting", 0x100: "display_clock_setting"}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag, self.window = index, [], False, [None, None]
        self.max_mhz = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        while not self.stop_flag:
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.samples.append((time.perf_counter(), mhz, rs))
            except Exception:
                pass
            time.sleep(0.005)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        t0, t1 = self.window
        inside = [s for s in self.samples if t0 is not None and t0 <= s[0] <= t1]
        use = inside or self.samples[-5:]
        bits = 0
        for s in use:
            bits |= s[2]
        reasons = sorted({name for bit, name in self.REASONS.items() if bits & bit})
        return {"sm_mhz": statistics.median(s[1] for s in use), "sm_max_mhz": self.max_mhz,
                "reasons": reasons, "samples": len(inside)}


# ------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the reference's CPU path on the host cores
# ------------------------------------------------------------------------------------------
def run_reference_cpu(steps, warmup, max_seconds=None):
    from oracle.reference_path import ReferenceCpuStack, solver_kind

    ref = ReferenceCpuStack(levels(), PER_GPU_BATCH, seed=0)
    try:
        for _ in range(warmup):
            ref.step()
        times = []
        t_start = time.perf_counter()
        for _ in range(steps):
            t0 = time.perf_counter()
            ref.step()
            times.append(time.perf_counter() - t0)
            if max_seconds is not None and time.perf_counter() - t_start > max_seconds:
                break
    finally:
        ref.close()
    total = sum(times)
    return {
        "value": PER_GPU_BATCH * len(times) / total, "unit": "images/s", "cores": ref.threads,
        "kind": solver_kind(),
        "sample": f"{len(times)} full steps of the same workload at batch {PER_GPU_BATCH} "
                  f"(torch CPU conv/autograd on {ref.threads} threads; inverse = "
                  + (f"reference Cython solver, batch sharded over {ref.nshards} forked workers)" if solver_kind() == "reference"
                     else "oracle C restatement of the reference solver, OpenMP)"),
        "steps": len(times), "ms_per_step": 1e3 * total / len(times),
    }


def base_config(world):
    """the keys both arms print identically (the driver compares `config` between the arms)"""
    return {"workload": WORKLOAD, "per_gpu_batch": PER_GPU_BATCH, "global_batch": PER_GPU_BATCH * world,
            "units_per_level": UNITS_PER_LEVEL, "kernel_size": KSIZE}


def reference_config(world):
    return base_config(world)


def main_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    # a step of the reference's CPU path takes ~0.6 s on the pool's hosts: bound the whole run to a few minutes
    r = run_reference_cpu(args.steps, max(args.warmup, 3), max_seconds=180.0)
    line = {
        "impl": "reference", "metric": "images/sec fwd+logdet, train step, and inverse sampling", "value": r["value"],
        "unit": "images/s", "n_gpus": args.gpus, "steps": args.steps, "steps_measured": r["steps"], "warmup": max(args.warmup, 3),
        "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": reference_config(args.gpus),
        "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": r["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)
    return 0


# ------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------
def dump_outputs(out_dir, runner, slot):
    """write what the last timed step returned, as float32 .npy files (about 12 MB for the headline workload):
    per level the latents z and per-sample log-likelihoods of the training batch and the samples of the sampling
    pass, and the FInC weights after that step's Adam update.  The inputs are seeded, so two builds of the
    project run with the same arguments can be compared file by file."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    s = runner.slots[slot]
    arrays = {"weights": runner.stack.flat}
    for li, lv in enumerate(runner.stack.levels):
        arrays[f"level{li}_z"] = s.acts[li][lv.n_units]
        arrays[f"level{li}_logp"] = s.logp[li]
        arrays[f"level{li}_samples"] = s.sample_out[li]
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


def algorithmic_bytes(phase, lv, B):
    """SURVEY.md 8(d): fp32, per FastFlowUnit on [B,C,H,W]: forward / backward-input / inverse
    read one tensor and write one (8 B/element); backward-weight reads two (8 B/element,
    dW itself negligible)."""
    return 8 * B * lv.channels * lv.height * lv.width


def fp32_peak():
    """measured FFMA throughput (tools/ffma_peak.cu, recorded in profiles/measured_fp32.json)"""
    try:
        with open(os.path.join(REPO, "profiles", "measured_fp32.json")) as f:
            return float(json.load(f)["fp32_ffma_tflops"])
    except Exception:
        return 74.4  # nominal: 148 SMs x 128 lanes x 2 x 1.965 GHz


def kernel_detail(torch, _native, dev, peak):
    """each kernel family alone at the three level shapes: batch 256 (the workload) and a
    batch large enough to stream from HBM; per-launch time of a CUDA graph of 8 launches.  The roofline
    time of a launch is max(algorithmic bytes / HBM peak, flops / fp32 FFMA peak): Cq = 3 is
    HBM-bound (6.75 flop/B), Cq >= 6 is bound by the fp32 pipe (SURVEY.md 8d)."""
    from fincflow_b200.fastflow import FastFlowUnit

    ffma = fp32_peak()

    flush = torch.empty(160 * 1024 * 1024 // 4, device=dev)
    out = []
    for (CT, H, W) in ((12, 16, 16), (24, 8, 8), (48, 4, 4)):
        for B in (PER_GPU_BATCH, 16384):
            unit = FastFlowUnit(CT, CT, (KSIZE, KSIZE)).to(dev)
            w = unit.weight.detach()
            x = torch.randn(B, CT, H, W, device=dev)
            dz = torch.randn_like(x)
            y = torch.empty_like(x)
            dw = torch.empty_like(w)
            ws = _native.new_workspace(_native.backward_weight_workspace_bytes(B, 4, CT // 4, H, W, KSIZE, KSIZE), dev)
            A1 = torch.linalg.qr(torch.randn(CT, CT, device=dev))[0].contiguous()
            b1 = torch.randn(CT, device=dev)
            # prepared weight tables, as in the step (one table per kind, built once per weight update)
            tabs = {}
            for kind in (_native.PREP_FORWARD, _native.PREP_BACKWARD_INPUT, _native.PREP_INVERSE):
                nb = _native.prepared_weights_bytes(kind, B, 4, CT // 4, H, W, KSIZE, KSIZE)
                tabs[kind] = torch.empty((1, nb), dtype=torch.uint8, device=dev)
                _native.prepare_weights(w[None], tabs[kind], kind, B, H, W)
            kk = (KSIZE, KSIZE)
            fns = {
                "affine1x1 (8f.1: ActNorm+Conv1x1 glue, HBM-bound)": lambda: _native.affine1x1(x, A1, b1, out=y),
                "forward_logdet": lambda: _native.forward(x, None, out=y, want_logdet=False,
                                                          prepared=tabs[_native.PREP_FORWARD][0], ksize=kk),
                "backward_input": lambda: _native.backward_input(dz, None, out=y,
                                                                 prepared=tabs[_native.PREP_BACKWARD_INPUT][0], ksize=kk),
                "backward_weight": lambda: _native.backward_weight(dz, x, kk, out=dw, workspace=ws),
                "inverse": lambda: _native.inverse(x, None, out=y, prepared=tabs[_native.PREP_INVERSE][0], ksize=kk),
            }
            nbytes = 8 * x.numel()
            flops = 2.0 * B * H * W * CT * (CT // 4) * KSIZE * KSIZE
            t_roof_us = max(nbytes / peak / 1e3, flops / ffma / 1e6)
            bound = "hbm" if nbytes / peak / 1e3 >= flops / ffma / 1e6 else "fp32"
            units_of = {}
            if B == PER_GPU_BATCH:   # the round-2 launches of the step: all 16 units of a level per launch
                U = UNITS_PER_LEVEL
                wU = torch.stack([FastFlowUnit(CT, CT, (KSIZE, KSIZE)).weight.detach() for _ in range(U)]).to(dev).contiguous()
                actsU = torch.empty(U, B, CT, H, W, device=dev)
                dzU = torch.randn(U + 1, B, CT, H, W, device=dev)
                dwU = torch.empty_like(wU)
                tabU = torch.empty((U, tabs[_native.PREP_INVERSE].shape[1]), dtype=torch.uint8, device=dev)
                _native.prepare_weights(wU, tabU, _native.PREP_INVERSE, B, H, W)
                wsU = torch.zeros(_native.backward_weight_batched_workspace_bytes(B, 4, CT // 4, H, W, KSIZE, KSIZE, U - 1),
                                  dtype=torch.uint8, device=dev)
                fns.update({
                    "forward chain (16 units / launch, all activations written)": lambda: _native.chain(x, wU, actsU),
                    "backward-data chain (15 units / launch)": lambda: _native.chain(dzU[U], wU, dzU[:U], units=range(U - 1, 0, -1), transpose=True),
                    "backward_weight batched (15 units / launch)": lambda: _native.backward_weight_batched(dzU[2:], actsU[:U - 1], dwU[1:], kk, workspace=wsU),
                    "inverse chain (16 units / launch, in place in shared memory)": lambda: _native.inverse_chain(x, tabU, kk, range(U - 1, -1, -1), out=y),
                })
                units_of = {"forward chain": U, "backward-data chain": U - 1, "backward_weight batched": U - 1, "inverse chain": U}
            for name, fn in fns.items():
                mult = next((v for k, v in units_of.items() if name.startswith(k)), 1)
                if name.startswith("affine1x1"):
                    k_flops, k_roof, k_bound = 2.0 * B * H * W * CT * CT, None, "hbm"
                    k_roof = max(nbytes / peak / 1e3, k_flops / ffma / 1e6)
                else:
                    k_flops, k_roof, k_bound = flops * mult, t_roof_us * mult, bound
                # a CUDA graph of CHAIN launches (what the step replays), L2 flushed before each replay;
                # at batch 256 the launches of a chain find their operands in L2, as inside the step
                CHAIN = 8
                side = torch.cuda.Stream(dev)
                with torch.cuda.stream(side):
                    for _ in range(2):
                        fn()
                torch.cuda.synchronize(dev)
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    for _ in range(CHAIN):
                        fn()
                ts = []
                for _ in range(5):
                    flush.zero_()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    g.replay()
                    e1.record()
                    e1.synchronize()
                    ts.append(e0.elapsed_time(e1) / CHAIN)
                del g
                us = 1e3 * statistics.median(ts)
                out.append({"kernel": name, "shape": [B, CT, H, W], "units_per_launch": mult, "us": round(us, 2),
                            "us_per_unit": round(us / mult, 2),
                            "GBps": round(mult * nbytes / us / 1e3, 1), "frac_of_hbm_peak": round(mult * nbytes / us / 1e3 / peak, 3),
                            "TFLOPs": round(k_flops / us / 1e6, 2), "bound": k_bound,
                            "frac_of_roofline": round(k_roof / us, 3), "images_per_s": round(B / us * 1e6)})
            del x, dz, y
    return out


def tensor_roofline(torch, dev):
    """the Coupling network's GEMMs (tcgen05 3xTF32, igemm_kernel) alone: TFLOP/s of TF32 MMAs issued (3 per fp32
    product) against the tensor-core peak.  kind::tf32 runs at half the bf16 rate, so peak = MEASURED_PEAKS.json's
    cuBLAS bf16 figure / 2 (burst for single launches; the sustained one for back-to-back phases: both kinds of run
    sit at the 1000 W power cap)."""
    from fincflow_b200 import _native

    try:
        with open(os.path.join(REPO, "MEASURED_PEAKS.json")) as f:
            mp = json.load(f)
        peak_burst, peak_sust, src = mp["bf16_tflops"] / 2, mp.get("bf16_tflops_sustained", mp["bf16_tflops"]) / 2, \
            "measured (MEASURED_PEAKS.json bf16_tflops / 2: kind::tf32 MMAs run at half the bf16 rate)"
    except Exception:
        peak_burst = peak_sust = 2250.0 / 2
        src = "fallback (B200_PROFILING.md: 2.25 PFLOP/s dense bf16, / 2 for tf32)"
    res = []
    for taps, name in ((1, "1x1 512->512 (coupling conv2)"), (9, "3x3 512->512 (long-K case)")):
        Bc, H, W, Cin, N = PER_GPU_BATCH, 16, 16, 512, 512
        k = 3 if taps == 9 else 1
        x = torch.randn(Bc, H, W, Cin, device=dev)
        w = torch.randn(N, Cin, k, k, device=dev) / (Cin * taps) ** 0.5
        wp = _native.tc_conv_prepare_weights(w, 0)
        bias = torch.zeros(N, device=dev)
        y = _native.tc_conv_nhwc(x, wp, bias, N, taps, relu=True)
        for _ in range(3):
            _native.tc_conv_nhwc(x, wp, bias, N, taps, relu=True, out=y)
        torch.cuda.synchronize(dev)
        n = 10 if taps == 1 else 4
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            _native.tc_conv_nhwc(x, wp, bias, N, taps, relu=True, out=y)
        e1.record()
        e1.synchronize()
        us = e0.elapsed_time(e1) / n * 1e3
        mma_tflops = 3 * 2.0 * Bc * H * W * Cin * taps * N / us / 1e6
        res.append({"gemm": name, "pixels": Bc * H * W, "us": round(us, 1), "fp32_equivalent_tflops": round(mma_tflops / 3, 1),
                    "achieved": round(mma_tflops, 1), "frac": round(mma_tflops / peak_burst, 3)})
        del x, y, w, wp
    return {"bound": "tensor", "unit": "TFLOP/s of TF32 MMAs (3 per fp32-accurate product)", "peak": round(peak_burst, 1),
            "peak_sustained": round(peak_sust, 1), "peak_source": src, "kernel": "finc::tc::igemm_kernel<128, 3, ...>", "gemms": res}


def whole_flow_detail(torch, dev, world=1, rank=0, pg=None):
    """cfg3_full_flow: the COMPLETE CIFAR-10-shaped FInCFlow (3 blocks x 16 steps, coupling width 512) with every
    layer on our kernels -- FInC units, fused ActNorm+Conv1x1, tensor-core Coupling (3xTF32, fp32 parity), fused
    preprocessing -- batch 256 per GPU: data-parallel train step through fincflow_b200.train.FlowTrainer
    (bucketed NCCL all-reduce overlapped with backward, Adam), exact log-likelihood evaluation, model.sample."""
    from fincflow_b200 import flows
    from fincflow_b200.train import FlowTrainer

    torch.manual_seed(0)
    B = PER_GPU_BATCH
    m = flows.fastflow_cifar10(actnorm=True).to(dev)
    trainer = FlowTrainer(m, lr=1e-3, process_group=pg, use_graph=os.environ.get("FINC_TRAINER_GRAPH", "1") == "1")
    g = torch.Generator(device=dev).manual_seed(7000 + rank)
    x = torch.randint(0, 256, (B, 3, 32, 32), device=dev, generator=g).float()

    def train():
        trainer.step(x)

    def evaluate():
        with torch.no_grad():
            m(x)

    def sample():
        with torch.no_grad():
            m.sample(B)

    out = {"model": "fincflow_b200.flows.fastflow_cifar10(actnorm=True): 3 blocks x 16 FastFlowSteps, coupling width 512, "
                    f"batch {B} per GPU, random init, synthetic uint8 images; all layers on our kernels "
                    "(Coupling: tcgen05 3xTF32 GEMMs, fp32 parity)",
           "n_params": sum(p.numel() for p in m.parameters()), "per_gpu_batch": B, "global_batch": B * world}
    out["train_step_execution"] = ("whole step (forward, backward" + (", bucketed NCCL all-reduces launched from the autograd hooks" if world > 1 else "")
                                   + ", Adam) replayed as ONE CUDA graph") if trainer.use_graph else \
        "eager; bucketed NCCL all-reduce launched from autograd hooks, overlapped with backward"
    for name, fn, n in (("train_step", train, 6), ("eval_loglik", evaluate, 5), ("sample", sample, 5)):
        for _ in range(5 if name == "train_step" else 2):
            fn()
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        e1.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) / n], device=dev, dtype=torch.float64)
        if world > 1:
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        ms = float(t.item())
        out[name + "_ms"] = round(ms, 2)
        out[name + "_images_per_s"] = round(B * world / ms * 1e3, 1)
    # the same evaluation / sampling as CUDA graphs (flows.InferenceSession): no host launch overhead
    try:
        sess = flows.InferenceSession(m)
        for name, fn in (("eval_loglik_graph", lambda: sess.log_prob(x)), ("sample_graph", lambda: sess.sample(B))):
            for _ in range(2):
                fn()
            torch.cuda.synchronize(dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(10):
                fn()
            e1.record()
            e1.synchronize()
            ms = e0.elapsed_time(e1) / 10
            out[name + "_ms"] = round(ms, 2)
            out[name + "_images_per_s"] = round(B * world / ms * 1e3, 1)
        del sess
        m.train()
    except Exception as e:
        out["graph_error"] = repr(e)
    try:   # the GEMM the step is made of, against the measured tensor-core peak
        out["tensor_roofline"] = tensor_roofline(torch, dev)
    except Exception as e:
        out["tensor_roofline"] = {"error": repr(e)}
    out["replica_param_maxdiff"] = trainer.replica_max_diff()
    trainer.close()   # the step graph holds NCCL work: it must go before the process group does
    out["round1_same_model_pytorch_glue"] = {"train_step_ms": 90.9, "sample_ms": 35.1,
                                             "note": "BENCH_r01: coupling networks through PyTorch/cuDNN (TF32)"}
    del m, trainer
    torch.cuda.empty_cache()
    return out


def main_ours(args):
    import torch

    from fincflow_b200 import _native
    from fincflow_b200.stack import FincStack, HotPathRunner

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback in the product path)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    pg = None
    host_cpus = None
    if world > 1:
        import torch.distributed as dist

        from fincflow_b200.distributed import bind_host_cores

        host_cpus = bind_host_cores(local, int(os.environ.get("LOCAL_WORLD_SIZE", world)))
        dist.init_process_group("nccl", device_id=dev)
        pg = dist.group.WORLD
    K, Wm = args.steps, max(args.warmup, 3)
    B = PER_GPU_BATCH
    lvls = levels()
    peak, peak_src = measured_peak()

    torch.manual_seed(0)  # same weights on every rank
    stack = FincStack(lvls).to(dev)
    NSLOT = 3
    runner = HotPathRunner(stack, B, dev, slots=NSLOT, process_group=pg)
    chain_flags = list(runner.chain)
    inv_chain_flags = None   # known after prepare()
    g = torch.Generator(device=dev).manual_seed(1000 + rank)  # different data per rank
    for s in runner.slots:
        for li in range(len(lvls)):
            s.acts[li][0].normal_(generator=g)
            s.zin[li].normal_(generator=g)
    runner.prepare()
    inv_chain_flags = list(runner.inv_chain)

    sampler = ClockSampler(local)
    sampler.start()

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize(dev)

    nph = len(runner.PHASES)
    for i in range(Wm):
        runner.step(i % NSLOT)
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(nph + 1)] for _ in range(K)]
    barrier()
    sampler.window[0] = time.perf_counter()
    for i in range(K):
        runner.step(i % NSLOT, evs[i])
    barrier()
    sampler.window[1] = time.perf_counter()
    elapsed_ms = evs[0][0].elapsed_time(evs[K - 1][nph])
    phase_ms = [sum(evs[i][p].elapsed_time(evs[i][p + 1]) for i in range(K)) / K for p in range(nph)]
    if world > 1:
        t = torch.tensor([elapsed_ms], device=dev, dtype=torch.float64)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        elapsed_ms = float(t.item())
    value = B * world * K / (elapsed_ms * 1e-3)
    if args.dump_outputs and rank == 0:   # before the runs below update the weights further
        dump_outputs(args.dump_outputs, runner, (K - 1) % NSLOT)

    # ---- the same K steps with the sampling pass on its own stream (reported next to `value`) ------
    overlap = None
    if not args.no_overlap:
        ov = HotPathRunner(stack, B, dev, slots=NSLOT, process_group=pg, overlap_sampling=True, level_parallel=True)
        for s_src, s_dst in zip(runner.slots, ov.slots):
            for li in range(len(lvls)):
                s_dst.acts[li][0].copy_(s_src.acts[li][0])
                s_dst.zin[li].copy_(s_src.zin[li])
        ov.prepare()
        for i in range(Wm):
            ov.step(i % NSLOT)
        ov.drain()
        barrier()
        o0, o1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        o0.record()
        for i in range(K):
            ov.step(i % NSLOT)
        ov.drain()
        o1.record()
        barrier()
        ov_ms = o0.elapsed_time(o1)
        if world > 1:
            t = torch.tensor([ov_ms], device=dev, dtype=torch.float64)
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
            ov_ms = float(t.item())
        overlap = {"value": round(B * world * K / (ov_ms * 1e-3), 1), "unit": "images/s", "ms_per_step": round(ov_ms / K, 4),
                   "api": "HotPathRunner(overlap_sampling=True, level_parallel=True).step",
                   "note": "same K steps, but the sampling pass of step k runs on a second stream next to the forward / "
                           "backward phases of step k+1 (both only read the weights of update k; update k+1 waits for it), and the "
                           "three levels of the stack -- independent inputs by construction -- run on one stream each inside a phase. "
                           "Not the headline: the timed region above keeps the phases serial so that per-phase and "
                           "per-launch durations stay clean"}
        del ov

    # ---- e2e: same step through the public API with HOST buffers --------------------------------
    del runner
    torch.cuda.empty_cache()
    ESLOT = 3  # copy-in / compute / copy-out of consecutive steps overlap (HotPathRunner.step)
    e2e_runner = HotPathRunner(stack, B, dev, slots=ESLOT, host_io=True, process_group=pg, device_latents=True)
    cpu_gen = torch.Generator().manual_seed(2000 + rank)
    for s in e2e_runner.slots:
        for li in range(len(lvls)):
            s.x_host[li].normal_(generator=cpu_gen)
    e2e_runner.prepare()
    for i in range(Wm):
        e2e_runner.step(i % ESLOT)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    t_host0 = time.perf_counter()
    for i in range(K):
        e2e_runner.step(i % ESLOT)
    host_ms_per_step = 1e3 * (time.perf_counter() - t_host0) / K   # CPU time to ENQUEUE a step (must stay below ms_per_step)
    e2e_runner.drain()  # the timed region ends when the last results have reached the host buffers
    e1.record()
    barrier()
    e2e_ms = e0.elapsed_time(e1)
    logp_last = float(e2e_runner.slots[(K - 1) % ESLOT].logp_host[0].mean())
    if world > 1:
        t = torch.tensor([e2e_ms], device=dev, dtype=torch.float64)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        e2e_ms = float(t.item())
    e2e_value = B * world * K / (e2e_ms * 1e-3)
    # counted from the slabs HotPathRunner.step copies: ONE host->device copy (the data batch x of every level; the
    # sampling latents are drawn on the device, like the reference's model.sample) and ONE device->host copy
    # (logp + samples of every level) per step
    slot0 = e2e_runner.slots[0]
    h2d = 4 * slot0.n_x
    d2h = 4 * slot0.out_dev.numel()
    launches = e2e_runner.launches_per_step
    fused_flag = getattr(e2e_runner, "fused_collective", False)
    crossrank = None
    if world > 1:
        # replicas must stay bit-identical: max over ranks of |flat - flat of rank 0|
        ref_w = stack.flat.detach().clone()
        torch.distributed.broadcast(ref_w, src=0)
        dmax = (stack.flat.detach() - ref_w).abs().max().reshape(1).double()
        torch.distributed.all_reduce(dmax, op=torch.distributed.ReduceOp.MAX)
        crossrank = float(dmax.item())
    fused_vs_nccl = fused_vs_nccl_check(torch, dev, rank, pg) if world > 1 else None
    e2e_runner_keep = e2e_runner
    del e2e_runner
    sampler.stop_flag = True
    sampler.join(timeout=1.0)
    clocks = sampler.summary()

    # ---- roofline of the longest phase ------------------------------------------------------------------
    # algorithmic bytes (SURVEY.md 8d): forward / inverse 8 B per element and unit, backward 12 (read dz, read x,
    # write dx).  forward and inverse are serial chains of one kernel family, so phase time / launches is a clean
    # per-launch duration; the backward phase overlaps the dX chain with the dW launches on side streams, so its
    # `avg_launch_us` is phase time / launches (an SM-time share, not a serial duration).
    n_units = sum(lv.n_units for lv in lvls)
    elems = sum(lv.n_units * B * lv.dim for lv in lvls)
    n_chain = sum(chain_flags)                                  # levels whose forward / dX chains are ONE launch each
    n_conv_fwd = sum(lv.n_units for lv, c in zip(lvls, chain_flags) if not c) + n_chain
    n_conv_bwd = sum(lv.n_units - 1 for lv, c in zip(lvls, chain_flags) if not c) + n_chain
    conv_name = "finc::chain::chain_kernel (all units of a level in one launch)" if n_chain else "finc::conv::conv_cta_kernel"
    phase_info = {
        "forward_logdet": (conv_name + " (forward) + gaussian_logp", n_conv_fwd + len(lvls),
                           8 * elems + sum(8 * B * lv.dim for lv in lvls)),
        "backward": (conv_name + " (dX) + finc::wgrad_kernel (dW), overlapped", n_conv_bwd + n_units, 12 * elems),
        "inverse": ("finc::rw::inverse_rw_kernel" + (" (all units of a level in one launch, solved in place in shared memory)" if any(inv_chain_flags) else ""),
                    sum(-(-lv.n_units // c) if c else lv.n_units for lv, c in zip(lvls, inv_chain_flags)), 8 * elems),
    }
    pm = dict(zip(HotPathRunner.PHASES, phase_ms))
    dom = max(phase_info, key=lambda p: pm[p])
    kname, nlaunch, bytes_phase = phase_info[dom]
    avg_us = 1e3 * pm[dom] / nlaunch
    achieved = bytes_phase / nlaunch / avg_us / 1e3  # GB/s
    traffic = None
    try:
        with open(os.path.join(REPO, "profiles", "ncu_traffic.json")) as f:
            traffic = json.load(f).get(dom)
    except Exception:
        pass
    roofline = {"bound": "hbm", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
                "frac": round(achieved / peak, 4), "traffic": traffic, "kernel": kname, "phase": dom,
                "launches_per_step": nlaunch, "avg_launch_us": round(avg_us, 3),
                "algorithmic_bytes_per_launch": bytes_phase // nlaunch, "peak_source": peak_src,
                "all_phases": {p: {"ms": round(pm[p], 4), "frac": round(phase_info[p][2] / (pm[p] * 1e-3) / 1e9 / peak, 4)}
                               for p in phase_info},
                "note": "algorithmic bytes count every unit (SURVEY 8d: 8 B per element and unit, 12 for backward) although a "
                        "chain launch keeps the 16 units of a level in shared memory and touches DRAM for one tensor "
                        "(`traffic`); batch-256 work is bound by dependent wavefront latency (inverse: 16 units x 31 steps per "
                        "tile) and instruction issue (forward / dX chains), not by HBM: see `kernels` for the per-unit "
                        "kernels streaming from HBM at batch 16384"}

    extras = None
    whole = None
    if not args.no_extra:
        del e2e_runner_keep
        torch.cuda.empty_cache()
        extras = run_extra_workloads(torch, dev, world, rank, pg, K)
        try:   # every rank takes part (data-parallel trainer); context only: never fail the bench line over it
            whole = whole_flow_detail(torch, dev, world, rank, pg)
        except Exception as e:
            whole = {"error": repr(e)}

    line = None
    if rank == 0:
        detail = kernel_detail(torch, _native, dev, peak) if (world == 1 and not args.no_detail) else None
        gpu_ref = gpu_reference_detail(torch, dev, pm) if (world == 1 and not args.no_detail) else None
        cpu = None
        if world == 1 and not args.no_cpu:
            r = run_reference_cpu(steps=6, warmup=1, max_seconds=25.0)
            cpu = {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")}
        line = {
            "metric": "images/sec fwd+logdet, train step, and inverse sampling", "value": round(value, 1),
            "unit": "images/s", "n_gpus": world, "steps": K, "warmup": Wm, "ms_per_step": round(elapsed_ms / K, 4),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": base_config(world),
            "config_detail": {"parallelism": f"dp{world} (batch sharded; train step: " + ("fused NVLink peer-memory all-reduce + Adam kernel" if fused_flag else "NCCL all-reduce of the flat FInC gradient bucket") + "; sampling without collective)",
                       "l2": f"{NSLOT} rotating input/activation sets (~{NSLOT * 0.2:.1f} GB total, > 126 MB L2); "
                             "intermediates of a step stay L2-resident as in a real flow",
                       "execution": "one CUDA graph per phase (forward: one chain launch per level -- all 16 units, tiles stay in shared memory, every activation still written; backward: one dX chain launch per level, then two dW launches per level -- units 1-15 batched, unit 0 -- on side streams; optimizer; inverse: one in-place chain launch per level); kernels launched with programmatic dependent launch"},
            "phases_ms": {k: round(v, 4) for k, v in pm.items()},
            "phase_images_per_s": {
                "forward_logdet": round(B * world / (pm["forward_logdet"] * 1e-3)),
                "train_step": round(B * world / ((pm["forward_logdet"] + pm["backward"] + pm["optimizer"]) * 1e-3)),
                "inverse_sampling": round(B * world / (pm["inverse"] * 1e-3))},
            "e2e": {"value": round(e2e_value, 1), "unit": "images/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": round(e2e_ms / K, 4), "api": "fincflow_b200.stack.HotPathRunner(host_io=True).step",
                    "copies_per_step": {"h2d": 1, "d2h": 1},
                    "host_enqueue_ms_per_step": round(host_ms_per_step, 4), "host_cpus": host_cpus,
                    "check_mean_logp_level0": logp_last},
            "gpu_launches": launches * K,
            "gpu_launches_per_step": launches,
            "roofline": roofline,
            "cpu_baseline": cpu,
            "clocks": clocks,
            "crossrank_param_maxdiff": crossrank,
            "fused_vs_nccl_maxdiff": fused_vs_nccl,
            "extra_workloads": extras,
            "gpu_reference": gpu_ref,
            "overlapped_sampling": overlap, "kernels": detail, "cfg3_full_flow": whole,
        }
        emit(line)
    if world > 1:
        # teardown must never hold the job: the line is out; if communicator teardown stalls, leave after 30 s
        import threading

        sys.stdout.flush()
        t = threading.Timer(30.0, lambda: os._exit(0))
        t.daemon = True
        t.start()
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()
        t.cancel()
    return 0


_REAL_STDOUT = None


def emit(line):
    """the ONE JSON line goes to the real stdout; everything else any library prints during
    the run (NCCL's version banner, warnings) was diverted to stderr by main()"""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)  # C-level stdout of this process (and of forked workers) -> stderr
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-overlap", action="store_true", help="skip the overlapped-sampling measurement")
    ap.add_argument("--no-detail", action="store_true", help="skip the per-kernel detail table")
    ap.add_argument("--no-extra", action="store_true", help="skip the other named configurations (extra_workloads)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of our timed path: it does not apply to --impl reference")
    if args.impl == "reference":
        return main_reference(args)
    return main_ours(args)


if __name__ == "__main__":
    sys.exit(main())
