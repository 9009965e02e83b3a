"""A/B of HotPathRunner(multi_level_inverse=...) on the headline workload (cifar10_levels(16, 3), batch 256).

    python tools/inverse_multi_ab.py [--rounds 5] [--steps 50] [--out DIR]

Two runners on the same stack and inputs, one per setting; their CUDA graphs are replayed in alternation, `rounds`
times each, and every round reports the inverse phase and the whole step (CUDA events, `steps` steps per round):
median and spread (max - min) per setting.  Then the single launch is compared with itself run for one level at a
time (same plan per level), which shows whether hosting all three kernel bodies on one SM costs time.  Prints one
JSON object (and writes it to DIR/inverse_multi_ab.json with --out).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from fincflow_b200 import _native  # noqa: E402
from fincflow_b200.stack import FincStack, HotPathRunner, cifar10_levels  # noqa: E402


def _time(fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / n


def _summary(v):
    return {"median_ms": round(statistics.median(v), 4), "spread_ms": round(max(v) - min(v), 4),
            "runs_ms": [round(x, 4) for x in v]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    torch.manual_seed(0)
    levels = cifar10_levels(16, 3)
    stack = FincStack(levels).to(dev)
    runners = {}
    for multi in (False, True):
        r = HotPathRunner(stack, args.batch, dev, slots=1, multi_level_inverse=multi)
        g = torch.Generator(device=dev).manual_seed(1000)
        for li in range(len(levels)):
            r.slots[0].acts[li][0].normal_(generator=g)
            r.slots[0].zin[li].normal_(generator=g)
        r.prepare()
        assert r.inv_multi == multi, "the multi-level inverse was not accepted"
        runners[multi] = r
    inv = HotPathRunner.PHASES.index("inverse")
    res = {m: {"inverse": [], "step": [], "phases": []} for m in runners}
    for _ in range(3):
        for r in runners.values():
            r.step(0)
    torch.cuda.synchronize()
    for _ in range(args.rounds):
        for m, r in runners.items():
            res[m]["inverse"].append(_time(lambda: r.run_phase(0, inv), args.steps))
            res[m]["step"].append(_time(lambda: r.step(0), args.steps))
            ph = []
            for p in range(len(HotPathRunner.PHASES)):
                ph.append(_time(lambda: r.run_phase(0, p), args.steps))
            res[m]["phases"].append(ph)
    out = {"gpu": gpu, "batch": args.batch, "rounds": args.rounds, "steps_per_round": args.steps,
           "launches_per_step": {str(m): r.launches_per_step for m, r in runners.items()}}
    for m in runners:
        key = "multi_level_inverse" if m else "per_level_inverse"
        out[key] = {"inverse_phase": _summary(res[m]["inverse"]), "step": _summary(res[m]["step"]),
                    "phases_median_ms": {name: round(statistics.median(ph[p] for ph in res[m]["phases"]), 4)
                                         for p, name in enumerate(HotPathRunner.PHASES)}}
    # the single launch for all levels against the same launch for one level at a time
    r, s = runners[True], runners[True].slots[0]
    lv_args = [(s.zin[li], r.tables[li][_native.PREP_INVERSE], lv.kernel_size, range(lv.n_units - 1, -1, -1),
                s.samp[li][(lv.n_units - 1) % 2]) for li, lv in enumerate(levels)]
    n = 4 * args.steps
    alone = [_time(lambda: _native.inverse_chain_multi([a]), n) for a in lv_args]
    together = _time(lambda: _native.inverse_chain_multi(lv_args), n)
    per_level = [_time(lambda: _native.inverse_chain(*a[:4], out=a[4]), n) for a in lv_args]
    reversed_order = _time(lambda: _native.inverse_chain_multi(lv_args[::-1]), n)
    out["launch_ms"] = {"all_levels_one_launch": round(together, 4), "levels_in_reverse_order": round(reversed_order, 4),
                        "one_level_in_multi_launch": [round(v, 4) for v in alone],
                        "one_level_inverse_chain": [round(v, 4) for v in per_level]}
    print(json.dumps(out))
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "inverse_multi_ab.json"), "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
