"""Time the differentiable coupling reverse and FastFlow.sample_with_log_prob on the CIFAR-10 flow
(fastflow_cifar10(actnorm=True), width 512), tensor-core kernels against PyTorch / cuDNN fp32.

    python tools/coupling_reverse_grad_time.py [--batch 256] [--rounds 5] [--out DIR] [--profile]

Arms, each with Coupling.tensor_core = True ("tc") and False ("cudnn", fp32: set_fp32_parity(True)), alternated
inside every round of one process:
  * coupling_l<i>: one coupling's reverse_and_logdet + backward of (y * r).sum() + logdet.sum() (gradients of the input
    and the seven parameters) at the three level shapes [B, 12, 16, 16], [B, 24, 8, 8], [B, 48, 4, 4];
  * sample_with_log_prob: x, log_q = model.sample_with_log_prob(zs) + backward of (x * r).sum() + log_q.sum() (gradients
    of the latents and every parameter);
and the yardstick log_prob_train: an eager model.log_prob(x) forward + backward of its sum (tensor-core couplings),
which runs the same GEMMs.  Every timing is CUDA events around `iters` eager repetitions after a warm-up; the report is
the per-repetition median over `rounds` rounds and the spread (max - min), in ms, with the GPU's name, power limit and
max SM clock read in the same run.  --profile adds a torch.profiler kernel summary of one tensor-core sample + backward
(run after the timings, so it does not disturb them).  Prints one JSON object (and writes it to DIR with --out).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from fincflow_b200 import flows  # noqa: E402

LEVELS = [(12, 16, 16), (24, 8, 8), (48, 4, 4)]


def _randomise_last_convs(model):
    """Conv2dZero starts at zero in the reference; give the couplings a non-trivial scale and shift"""
    with torch.no_grad():
        for m in model.modules():
            if isinstance(m, flows.Coupling):
                m.net[4].weight.normal_(0, 0.02)
                m.net[4].bias.normal_(0, 0.1)
                m.net[4].logs.normal_(0, 0.1)


def _time_ms(fn, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / iters


def _with_tc(tc, fn):
    def run():
        flows.Coupling.tensor_core = tc
        try:
            fn()
        finally:
            flows.Coupling.tensor_core = True
    return run


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--coupling-iters", type=int, default=20)
    ap.add_argument("--flow-iters", type=int, default=3)
    ap.add_argument("--out", default=None)
    ap.add_argument("--profile", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("coupling_reverse_grad_time.py needs a CUDA device")
    flows.set_fp32_parity(True)
    dev = torch.device("cuda", 0)
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    B = args.batch
    torch.manual_seed(0)

    arms = {}   # name -> (fn, iters)
    for i, (C, H, W) in enumerate(LEVELS):
        cp = flows.Coupling((C, H, W), width=512).to(dev)
        _randomise_last_convs(cp)
        x = torch.randn(B, C, H, W, device=dev, requires_grad=True)
        r = torch.randn(B, C, H, W, device=dev)
        wanted = [x] + list(cp.parameters())

        def coupling_step(cp=cp, x=x, r=r, wanted=wanted):
            y, ld = cp.reverse_and_logdet(x)
            torch.autograd.grad((y * r).sum() + ld.sum(), wanted)

        for tc in (True, False):
            arms[f"coupling_l{i}_{'tc' if tc else 'cudnn'}"] = (_with_tc(tc, coupling_step), args.coupling_iters)

    model = flows.fastflow_cifar10(actnorm=True).to(dev)
    img = torch.randint(0, 256, (B, 3, 32, 32), device=dev).float()
    with torch.no_grad():
        zs, _ = model(img)                       # initialises ActNorm
    _randomise_last_convs(model)
    lat = [torch.randn_like(z).requires_grad_() for z in zs]
    r_img = torch.randn(B, 3, 32, 32, device=dev)
    params = list(model.parameters())

    def sample_step():
        x, log_q = model.sample_with_log_prob(zs=lat)
        torch.autograd.grad((x * r_img).sum() + log_q.sum(), params + lat)

    def log_prob_step():
        torch.autograd.grad(model.log_prob(img).sum(), params)

    arms["sample_with_log_prob_tc"] = (_with_tc(True, sample_step), args.flow_iters)
    arms["sample_with_log_prob_cudnn"] = (_with_tc(False, sample_step), args.flow_iters)
    arms["log_prob_train_tc"] = (_with_tc(True, log_prob_step), args.flow_iters)

    for fn, _ in arms.values():          # warm-up: module loads, cuDNN algorithm choice, allocator
        fn()
        fn()
    torch.cuda.synchronize()
    times = {name: [] for name in arms}
    for _ in range(args.rounds):
        for name, (fn, iters) in arms.items():
            times[name].append(_time_ms(fn, iters))
    res = {name: {"median_ms": round(statistics.median(v), 3), "spread_ms": round(max(v) - min(v), 3)}
           for name, v in times.items()}
    med = {name: v["median_ms"] for name, v in res.items()}
    ratios = {f"coupling_l{i}_cudnn_over_tc": round(med[f"coupling_l{i}_cudnn"] / med[f"coupling_l{i}_tc"], 2)
              for i in range(len(LEVELS))}
    ratios["sample_cudnn_over_tc"] = round(med["sample_with_log_prob_cudnn"] / med["sample_with_log_prob_tc"], 2)
    ratios["sample_tc_over_log_prob_train"] = round(med["sample_with_log_prob_tc"] / med["log_prob_train_tc"], 3)
    out = {"gpu": gpu, "batch": B, "rounds": args.rounds, "iters": {n: it for n, (_, it) in arms.items()},
           "times": res, "ratios": ratios}
    if args.profile:
        from torch.profiler import ProfilerActivity, profile

        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            arms["sample_with_log_prob_tc"][0]()
            torch.cuda.synchronize()
        table = prof.key_averages().table(sort_by="cuda_time_total", row_limit=30, max_name_column_width=90)
        out["profile_sample_tc"] = table
        print(table)
    print(json.dumps(out))
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "coupling_reverse_grad_time.json"), "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
