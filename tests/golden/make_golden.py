"""Generate golden fixtures by running the REFERENCE's own Python code (needs a reference checkout).

    python tests/golden/make_golden.py          # writes tests/golden/finc_golden_<part>.npz

The reference (a checkout of aditya-v-kallappa/FInCFlow named by FINCFLOW_REFERENCE) is a set of scripts
that import relative to ``fastflow/`` as CWD.  We import its ``layers.conv.PaddedConv2d``
and ``fastflow.FastFlowUnit`` unmodified through these shims (SURVEY.md section 8c):

  1. ``sys.path.insert(0, $FINCFLOW_REFERENCE/fastflow)``
  2. stub ``matplotlib`` (imported by utils/solve_mc.py:3)
  3. ``utils.fastflow_inverse.solve_parallel_mc`` -> the reference's .pyx compiled from
     its own source by oracle/build_ref.py (shipped .so files are cp37/cp39)
  4. ``torch.utils.cpp_extension.load`` -> stub (fastflow.py:9-10 JIT-builds the CUDA
     extension at import; there is no GPU here, so unit reverses use the reference's
     ``reverse_level1`` = four Cython solves, fastflow.py:57-76)

What is recorded per case (fp32 tensors, TF32 irrelevant on CPU):
  x, w (stored orientation, cat of the groups), z = forward(x), logdet (python float),
  dz, dx, dw_raw (autograd), dw_masked (after reset_gradients), zs ~ N(0,1),
  x_from_zs = reverse(zs), x_rt = reverse(z).
plus the integer known-answer inputs of cuda/cinc_cuda/test_cuda_kernel.py and
fastflow/test_examples.py (SURVEY.md appendix E) solved by the reference solver.
"""
from __future__ import annotations

import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
REFERENCE = os.environ.get("FINCFLOW_REFERENCE", "")
REF = os.path.join(REFERENCE, "fastflow")
PART_BYTES = 950_000  # every stored file stays under 1 MB
sys.path.insert(0, REPO)


def import_reference():
    from oracle import build_ref

    if not REFERENCE or not os.path.isdir(REF):
        sys.exit("set FINCFLOW_REFERENCE to a checkout of aditya-v-kallappa/FInCFlow "
                 f"(no directory {REF!r})")
    sys.path.insert(0, REF)
    mpl = types.ModuleType("matplotlib")
    mpl.use = lambda *a, **k: None
    mpl.pyplot = types.ModuleType("matplotlib.pyplot")
    mpl.colors = types.ModuleType("matplotlib.colors")
    sys.modules.update({"matplotlib": mpl, "matplotlib.pyplot": mpl.pyplot,
                        "matplotlib.colors": mpl.colors})
    solver = build_ref.load()
    assert solver is not None, "reference Cython solver did not build"
    import utils  # noqa: F401  (reference package, namespace for the next line)
    pkg = types.ModuleType("utils.fastflow_inverse")
    pkg.__path__ = []
    sys.modules["utils.fastflow_inverse"] = pkg
    sys.modules["utils.fastflow_inverse.solve_parallel_mc"] = solver
    import torch.utils.cpp_extension as cppext

    cppext.load = lambda *a, **k: types.SimpleNamespace(inverse=None)
    from layers.conv import PaddedConv2d  # noqa: E402
    from fastflow import FastFlowUnit  # noqa: E402

    return PaddedConv2d, FastFlowUnit, solver


def run_layer(layer, weights, x, dz, zs, reverse):
    x = x.clone().requires_grad_(True)
    z, logdet = layer(x)
    assert isinstance(logdet, float) and logdet == 0.0  # conv.py:106
    z.backward(dz)
    dw_raw = [w.grad.clone() for w in weights]
    for m in layer.modules():
        if hasattr(m, "reset_gradients"):
            m.reset_gradients()  # conv.py:98-99 via train/experiment.py:16-18
    dw_masked = [w.grad.clone() for w in weights]
    with torch.no_grad():
        x_rt = reverse(z.detach())
        x_zs = reverse(zs)
    return dict(
        x=x.detach(), w=torch.cat([w.detach() for w in weights], 0), z=z.detach(), dz=dz,
        dx=x.grad, dw_raw=torch.cat(dw_raw, 0), dw_masked=torch.cat(dw_masked, 0), zs=zs,
        x_from_zs=x_zs, x_rt=x_rt)


def main():
    PaddedConv2d, FastFlowUnit, solver = import_reference()
    torch.manual_seed(1234)
    torch.set_num_threads(1)
    out = {}
    index = []

    # ---- FastFlowUnit cases: (Cq, H, W, k, B) -------------------------------------
    unit_cases = [
        (1, 14, 14, (3, 3), 2), (2, 7, 7, (3, 3), 2),                       # MNIST levels
        (3, 16, 16, (3, 3), 2), (6, 8, 8, (3, 3), 2), (12, 4, 4, (3, 3), 2),  # CIFAR / IN32
        (3, 32, 32, (3, 3), 1), (6, 16, 16, (3, 3), 1), (12, 8, 8, (3, 3), 1),
        (24, 4, 4, (3, 3), 1),                                              # ImageNet64
        (3, 16, 16, (5, 5), 1), (6, 8, 8, (5, 5), 1), (12, 4, 4, (5, 5), 1),
        (24, 4, 4, (5, 5), 1),
        (1, 4, 4, (2, 2), 3), (2, 5, 9, (2, 3), 2), (3, 8, 8, (3, 2), 2), (5, 6, 6, (3, 3), 2),
    ]
    for (Cq, H, W, k, B) in unit_cases:
        unit = FastFlowUnit(4 * Cq, 4 * Cq, k)
        weights = [unit.conv_tl.conv.weight, unit.conv_tr.conv.weight,
                   unit.conv_bl.conv.weight, unit.conv_br.conv.weight]
        if Cq >= 3:  # "trained-like": break the pristine init a little (keeps the invariant)
            with torch.no_grad():
                for c in (unit.conv_tl, unit.conv_tr, unit.conv_bl, unit.conv_br):
                    c.conv.weight += 0.02 * torch.randn_like(c.conv.weight) * c.mask
        x = torch.randn(B, 4 * Cq, H, W)
        dz = torch.randn(B, 4 * Cq, H, W)
        zs = torch.randn(B, 4 * Cq, H, W)
        rec = run_layer(unit, weights, x, dz, zs, unit.reverse_level1)
        name = f"unit_C{Cq}_H{H}_W{W}_k{k[0]}x{k[1]}_B{B}"
        index.append(name)
        for key, val in rec.items():
            out[f"{name}/{key}"] = val.numpy().astype(np.float32)
        out[f"{name}/orders"] = np.array([0, 1, 2, 3], dtype=np.int32)

    # ---- single PaddedConv2d cases (incl. BASELINE config 1: C=4, 14x14, k=3) ------
    conv_cases = [(4, 14, 14, (3, 3), 2, o) for o in ("TL", "TR", "BL", "BR")]
    conv_cases += [(3, 6, 6, (3, 3), 2, "TR"), (1, 5, 5, (2, 2), 2, "BL"),
                   (3, 5, 9, (3, 3), 2, "BR"), (10, 7, 7, (3, 3), 1, "TL"),
                   (2, 6, 6, (5, 5), 2, "BR")]
    code = {"TL": 0, "TR": 1, "BL": 2, "BR": 3}
    for (C, H, W, k, B, order) in conv_cases:
        conv = PaddedConv2d(C, C, k, order=order)
        x = torch.randn(B, C, H, W)
        dz = torch.randn(B, C, H, W)
        zs = torch.randn(B, C, H, W)
        rec = run_layer(conv, [conv.conv.weight], x, dz, zs, lambda t: conv.reverse(t)[0])
        name = f"conv_{order}_C{C}_H{H}_W{W}_k{k[0]}x{k[1]}_B{B}"
        index.append(name)
        for key, val in rec.items():
            out[f"{name}/{key}"] = val.numpy().astype(np.float32)
        out[f"{name}/orders"] = np.array([code[order]], dtype=np.int32)
        out[f"{name}/mask"] = conv.mask.numpy().astype(np.float32)

    # ---- integer known-answer inputs (SURVEY.md appendix E) ------------------------
    grid4 = [[1, 2, 3, 4], [5, 6, 7, 8], [9, 10, 11, 12], [13, 14, 15, 16]]
    kats = [
        ("kat_2x2_corner_only", [grid4], [[0, 0], [0, 1]]),          # test_cuda_kernel.py:3-13
        ("kat_2x2_diag", [grid4], [[1, 0], [0, 1]]),                 # :16-26
        ("kat_2x2_batch2", [[[1, 2, 3], [5, 6, 7], [9, 10, 11]],
                            [[12, 13, 14], [15, 16, 17], [18, 19, 20]]], [[0, 0], [0, 1]]),  # :29-42
        ("kat_3x3_identity", [grid4], [[1, 0, 0], [0, 1, 0], [0, 0, 1]]),  # :45-56
    ]
    for name, inp, ker in kats:
        z = np.asarray(inp, dtype=np.float64)[:, None]          # [m,1,n,n]
        w = np.asarray(ker, dtype=np.float64)[None, None]       # [1,1,k,k] TL form
        y = solver.solve_parallel(z.copy(), w, w.shape[2:])
        # the reference's own consistency check, cuda/cinc_cuda/util.py:36
        k = w.shape[-1]
        back = torch.nn.functional.conv2d(
            torch.nn.functional.pad(torch.from_numpy(y), (k - 1, 0, k - 1, 0)), torch.from_numpy(w))
        assert (back.numpy() - z).__abs__().sum() == 0
        index.append(name)
        out[f"{name}/zs"] = z.astype(np.float32)
        out[f"{name}/w"] = w.astype(np.float32)
        out[f"{name}/x_from_zs"] = y.astype(np.float32)
        out[f"{name}/orders"] = np.array([0], dtype=np.int32)

    # fastflow/test_examples.py:54-73 (TR) and :6-25 (BL), through PaddedConv2d itself
    for name, order, wst in (("kat_TR_test_examples", "TR", [[0, 2], [1, 0]]),
                             ("kat_BL_test_examples", "BL", [[0, 1], [1, 0]])):
        conv = PaddedConv2d(1, 1, (2, 2), order=order)
        with torch.no_grad():
            conv.conv.weight.copy_(torch.tensor(wst, dtype=torch.float32)[None, None])
        x = torch.tensor([[1, 2, 3], [4, 5, 6], [7, 8, 9]], dtype=torch.float32)[None, None]
        with torch.no_grad():
            z, _ = conv(x)
            xr = conv.reverse(z)[0]
        assert torch.equal(xr, x)
        index.append(name)
        out[f"{name}/x"] = x.numpy()
        out[f"{name}/w"] = conv.conv.weight.detach().numpy()
        out[f"{name}/z"] = z.numpy()
        out[f"{name}/zs"] = z.numpy()
        out[f"{name}/x_from_zs"] = xr.numpy()
        out[f"{name}/orders"] = np.array([code[order]], dtype=np.int32)

    for path in save_parts(out, index, os.path.join(HERE, "finc_golden")):
        print(f"wrote {path}: {os.path.getsize(path) / 1e6:.2f} MB")


def save_parts(out, index, stem):
    """np.savez_compressed of whole cases, in order, into stem_0.npz, stem_1.npz, ... of at most PART_BYTES
    each; every part carries the names of its cases in `__index__`"""
    import io

    def packed(names):
        arrays = {k: v for k, v in out.items() if k.split("/")[0] in names}
        buf = io.BytesIO()
        np.savez_compressed(buf, __index__=np.array(names), **arrays)
        return buf.getvalue()

    parts, cur = [], []
    for name in index:
        if cur and len(packed(cur + [name])) > PART_BYTES:
            parts.append(cur)
            cur = []
        cur.append(name)
    parts.append(cur)
    paths = []
    for i, names in enumerate(parts):
        data = packed(names)
        assert len(data) <= PART_BYTES, (names, len(data))
        paths.append(f"{stem}_{i}.npz")
        with open(paths[-1], "wb") as f:
            f.write(data)
    return paths


if __name__ == "__main__":
    main()
