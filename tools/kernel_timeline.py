"""FINC_DEBUG_TS=1 python tools/kernel_timeline.py -- per-CTA phase timestamps of the tiled kernels
(debug aid; see finc_debug_timestamps in include/fincflow_b200.h)."""
import os, sys
os.environ["FINC_DEBUG_TS"] = "1"
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from fincflow_b200 import _native
from fincflow_b200.fastflow import FastFlowUnit

lib = _native.load()
dev = torch.device("cuda:0")
B = int(sys.argv[1]) if len(sys.argv) > 1 else 256
NAMES = {"forward": ["entry", "weights staged", "first chunk landed", "chunk computed"],
         "inverse": ["entry", "weights staged", "first item landed", "first item solved", "exit"],
         "backward_weight": ["entry", "first chunk landed", "sweeps done", "CTA reduced", "ticket taken", "last CTA done"]}
for (CT, H, W) in ((12, 16, 16), (24, 8, 8), (48, 4, 4)):
    unit = FastFlowUnit(CT, CT, (3, 3)).to(dev); w = unit.weight.detach()
    x = torch.randn(B, CT, H, W, device=dev); dz = torch.randn_like(x); y = torch.empty_like(x); dw = torch.empty_like(w)
    ws = _native.new_workspace(_native.backward_weight_workspace_bytes(B, 4, CT // 4, H, W, 3, 3), dev)
    fns = {"forward": lambda: _native.forward(x, w, out=y, want_logdet=False),
           "inverse": lambda: _native.inverse(x, w, out=y),
           "backward_weight": lambda: _native.backward_weight(dz, x, (3, 3), out=dw, workspace=ws, flags=int(os.environ.get("FINC_TL_DWFLAGS", "0")))}
    for name, fn in fns.items():
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        scratch = np.zeros(8192, dtype=np.uint64)
        lib.finc_debug_timestamps(scratch.ctypes.data, scratch.size)  # also clears the device marks
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record(); torch.cuda.synchronize()
        buf = np.zeros(1024 * 8, dtype=np.uint64)
        lib.finc_debug_timestamps(buf.ctypes.data, buf.size)
        ts = buf.reshape(1024, 8).astype(np.int64)
        n = len(NAMES[name])
        live = ts[:, 0] > 0
        t = ts[live][:, :n]
        t0 = t[:, 0].min()
        rel = (t - t0) / 1e3
        print(f"{name:16s} [{B},{CT},{H},{W}] ctas={live.sum()} event={e0.elapsed_time(e1)*1e3:.1f}us")
        for j, nm in enumerate(NAMES[name]):
            col = rel[:, j][t[:, j] > 0]
            if len(col):
                print(f"     {nm:22s} min {col.min():7.2f}  median {np.median(col):7.2f}  max {col.max():7.2f} us  (n={len(col)})")
        ts[:] = 0
