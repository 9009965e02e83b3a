"""Time the FInC inverse (finc_inverse_f32) against its adjoint (finc_inverse_adjoint_f32), and one unit's whole
reverse backward (adjoint + negated weight gradient), on the shapes of the flows.

    python tools/inverse_adjoint_time.py [--rounds 5] [--launches 200] [--out DIR]

Each kernel is captured as a CUDA graph of `launches` back-to-back launches (so host overhead is not timed) and the
graphs of the two kernels are replayed in alternation, `rounds` times each (CUDA events).  The launches of a graph
rotate over enough distinct input / output buffers that together they exceed twice the 126 MB L2: every launch reads
its input from HBM, as in a sampling pass.  Reports per-launch median and spread (max - min) in microseconds, the
ratio adjoint / inverse, and the GPU's name, power limit and max SM clock.  Prints one JSON object (and writes it to
DIR/inverse_adjoint_time.json with --out).
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
from fincflow_b200.fastflow import FastFlowUnit  # noqa: E402

L2_BYTES = 126 * 2 ** 20
SHAPES = [  # (B, G*C, H, W, k): the CIFAR-10 levels at two batch sizes, one 5x5 level, one generic-kernel shape
    (256, 12, 16, 16, 3), (256, 24, 8, 8, 3), (256, 48, 4, 4, 3),
    (16384, 12, 16, 16, 3), (16384, 24, 8, 8, 3), (16384, 48, 4, 4, 3),
    (256, 24, 8, 8, 5),
    (2048, 48, 4, 4, 3),  # C = 12, P = 1, one tile per stack: the adjoint reads its corner weights from shared memory
    (256, 96, 4, 4, 3),   # C = 24 per group (ImageNet64's last level): the inverse's shared-memory wavefront kernel,
                          # the adjoint's generic kernel
]


def _graph(fn, n):
    fn(0)   # warm-up: module load, function attributes
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for i in range(n):
            fn(i)
    return g


def _replay_us(g, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    g.replay()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) * 1e3 / n


def _summary(v):
    return {"median_us": round(statistics.median(v), 2), "spread_us": round(max(v) - min(v), 2)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("inverse_adjoint_time.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    rows = []
    for B, CT, H, W, k in SHAPES:
        torch.manual_seed(B + CT + k)
        w = FastFlowUnit(CT, CT, (k, k)).weight.detach().to(dev)
        nbytes = 2 * B * CT * H * W * 4
        nbuf = max(1, min(args.launches, -(-2 * L2_BYTES // nbytes)))
        src = [torch.randn(B, CT, H, W, device=dev) for _ in range(nbuf)]
        dst = [torch.empty(B, CT, H, W, device=dev) for _ in range(nbuf)]
        dw = torch.empty_like(w)
        ws = _native.new_workspace(_native.backward_weight_workspace_bytes(B, 4, CT // 4, H, W, k, k), dev)

        def inverse(i):
            _native.inverse(src[i % nbuf], w, out=dst[i % nbuf])

        def adjoint(i):
            _native.inverse_adjoint(src[i % nbuf], w, out=dst[i % nbuf])

        def unit_backward(i):   # dz = A^-T dx, dW = -wgrad(dz, x): what FincInverseFunction.backward launches
            _native.inverse_adjoint(src[i % nbuf], w, out=dst[i % nbuf])
            _native.backward_weight(dst[i % nbuf], src[(i + 1) % nbuf], (k, k), flags=_native.FLAG_NEGATE, out=dw,
                                    workspace=ws)

        n = args.launches
        graphs = {"inverse": _graph(inverse, n), "adjoint": _graph(adjoint, n), "unit_backward": _graph(unit_backward, n)}
        times = {name: [] for name in graphs}
        for name, g in graphs.items():
            _replay_us(g, n)
        for _ in range(args.rounds):
            for name, g in graphs.items():
                times[name].append(_replay_us(g, n))
        row = {"shape": [B, CT, H, W, k], "buffers": nbuf}
        row.update({name: _summary(v) for name, v in times.items()})
        row["adjoint_over_inverse"] = round(row["adjoint"]["median_us"] / row["inverse"]["median_us"], 3)
        rows.append(row)
        print(json.dumps(row), flush=True)
        del graphs, src, dst
        torch.cuda.empty_cache()
    out = {"gpu": gpu, "rounds": args.rounds, "launches_per_graph": args.launches,
           "l2": "inputs rotate over buffers totalling >= 2x L2 (126 MB)", "rows": rows}
    print(json.dumps(out))
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "inverse_adjoint_time.json"), "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
