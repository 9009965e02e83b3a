"""The differentiable tensor-core coupling reverse and the log-density of FastFlow samples (run on the B200 box:
`pytest -m gpu`).

  * finc_coupling_backward_f32 with FINC_FLAG_COUPLING_REVERSE (the backward of finc_coupling_apply_f32 with
    reverse = 1) against float64 PyTorch autograd of the reverse formulas, on every supported N3pad;
  * the reverse log-det -sum log_s of finc_coupling_apply_f32 and FINC_FLAG_LOGDET_ACCUMULATE;
  * Coupling.reverse records a graph exactly when the PyTorch formulas would, with the same bits either way;
  * FastFlow.sample_with_log_prob: log q(x) equals model.log_prob(x), and its gradients equal a PyTorch reference
    flow's; a differentiable sample + backward runs only the library's kernels and PyTorch's own elementwise ones.
"""
import itertools
import json
import os
import re
import subprocess
import sys

import pytest
import torch

from conftest import rel_err
from test_gpu_inverse_grad import ORDERS, ref_inverse

pytestmark = pytest.mark.gpu

GRAD_TOL = 2e-5     # the bound of test_coupling_native_backward_matches_pytorch_autograd
LD_TOL = 1e-5


@pytest.fixture
def fp32_convs():
    """PyTorch's convolutions and matmuls in true fp32 (cuDNN / cuBLAS would otherwise use TF32 products)"""
    old = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def npy(t):
    return t.detach().double().cpu().numpy()


def coupling(C, H, W, width, seed=0):
    from fincflow_b200.flows import Coupling

    torch.manual_seed(seed)
    cp = Coupling((C, H, W), width=width).cuda()
    with torch.no_grad():  # the last conv is zero-initialised in the reference: give it something to do
        cp.net[4].weight.normal_(0, 0.02)
        cp.net[4].bias.normal_(0, 0.1)
        cp.net[4].logs.normal_(0, 0.1)
    return cp


class FixedMask(torch.nn.Module):
    """a ReLU whose decisions are given: h * mask"""

    def __init__(self, mask):
        super().__init__()
        self.mask = mask

    def forward(self, h):
        return h * self.mask


def kernel_relu_masks(cp, x):
    """the ReLU decisions of the tensor-core reverse of x: where its hidden activations, kept channels-last in the
    workspace of finc_coupling_apply_f32 (im2col patches [np, K1pad], then h1 [np, width], then h2 [np, width]), are
    positive"""
    from fincflow_b200 import _native

    B, C, H, W = x.shape
    n, w, k1 = B * H * W, cp.width, (9 * (C // 2) + 63) // 64 * 64
    ws = torch.empty(_native.coupling_workspace_bytes(B, C, H, W, w), dtype=torch.uint8, device=x.device)
    with torch.no_grad():
        _native.coupling_apply(x, cp.prepared(), w, reverse=True, flags=cp._flags(), workspace=ws)
    f = ws.view(torch.float32)
    h1, h2 = (f[n * (k1 + i * w):n * (k1 + (i + 1) * w)].view(B, H, W, w).permute(0, 3, 1, 2) for i in (0, 1))
    return (h1 > 0).double(), (h2 > 0).double()


def float64_copy(cp, x=None):
    """the layer in float64 (the PyTorch formulas).  Given x, its ReLUs take the decisions the tensor-core reverse
    of x takes: a pre-activation within rounding of 0 would otherwise switch a whole term of a gradient on or off
    between the two (at width 512 about one of the B*H*W*2*width activations does)."""
    from fincflow_b200.flows import Coupling

    cpd = Coupling((cp.n_channels, 1, 1), width=cp.width).cuda().double()
    cpd.load_state_dict({k: v.double() for k, v in cp.state_dict().items()})
    if x is not None:
        m1, m2 = kernel_relu_masks(cp, x)
        cpd.net[1], cpd.net[3] = FixedMask(m1), FixedMask(m2)
    return cpd


def reverse_grads(cp, x, gy, gl):
    """(y, ld, [dx, 7 parameter gradients]) of (y * gy).sum() + (ld * gl).sum() through cp.reverse_and_logdet
    (cp.reverse when gl is None)"""
    xi = x.detach().clone().requires_grad_()
    if gl is None:
        y, ld = cp.reverse(xi), None
        loss = (y * gy).sum()
    else:
        y, ld = cp.reverse_and_logdet(xi)
        loss = (y * gy).sum() + (ld * gl).sum()
    grads = torch.autograd.grad(loss, [xi] + list(cp.parameters()))
    return y, ld, grads


# B, C, H, W, width: N3pad = 16, 32, 48, 64, 96; widths 128, 256, 512; B = 1 and odd
NATIVE_CASES = [(1, 12, 16, 16, 128), (3, 24, 8, 8, 256), (5, 48, 4, 4, 512), (1, 64, 4, 4, 128), (3, 96, 4, 4, 256),
                (7, 12, 8, 8, 512)]


@pytest.mark.parametrize("with_dlogdet", [True, False], ids=["dlogdet", "no_dlogdet"])
@pytest.mark.parametrize("case", NATIVE_CASES, ids=lambda c: "B{}_C{}_{}x{}_w{}".format(*c))
def test_native_reverse_backward(case, with_dlogdet):
    from fincflow_b200 import _native

    B, C, H, W, width = case
    assert _native.coupling_prepared_bytes(C, width, True) > 0
    cp = coupling(C, H, W, width, seed=B + C)
    x = torch.randn(B, C, H, W, device="cuda")
    gy = torch.randn_like(x)
    gl = torch.randn(B, device="cuda") if with_dlogdet else None
    y, ld, got = reverse_grads(cp, x, gy, gl)
    assert y.grad_fn is not None
    _, _, want = reverse_grads(float64_copy(cp, x), x.double(), gy.double(), None if gl is None else gl.double())
    names = ["dx"] + [n for n, _ in cp.named_parameters()]
    for name, a, b in zip(names, got, want):
        assert a.shape == b.shape, name
        assert rel_err(npy(a), npy(b)) <= GRAD_TOL, (name, rel_err(npy(a), npy(b)))
    # deterministic backward
    _, _, again = reverse_grads(cp, x, gy, gl)
    for name, a, b in zip(names, got, again):
        assert torch.equal(a, b), name
    # the same output bits with a graph, in grad mode without one, and under no_grad
    with torch.no_grad():
        y0, ld0 = cp.reverse_and_logdet(x)
    cp.requires_grad_(False)
    y1, ld1 = cp.reverse_and_logdet(x)
    assert y1.grad_fn is None and ld1.grad_fn is None
    assert torch.equal(y, y0) and torch.equal(y1, y0) and torch.equal(ld1, ld0)
    if ld is not None:
        assert torch.equal(ld, ld0)


@pytest.mark.parametrize("case", NATIVE_CASES, ids=lambda c: "B{}_C{}_{}x{}_w{}".format(*c))
def test_reverse_logdet(case):
    from fincflow_b200 import _native

    B, C, H, W, width = case
    cp = coupling(C, H, W, width, seed=2 * B + C)
    y = torch.randn(B, C, H, W, device="cuda")
    with torch.no_grad():
        x, ld = cp.reverse_and_logdet(y)
        _, _, log_s, _ = float64_copy(cp)._st(y.double())
        assert rel_err(npy(ld), npy(-log_s.flatten(1).sum(1))) <= LD_TOL
        _, ld_fwd = cp(x)                                       # forward log-det at the reconstructed input
        assert rel_err(npy(ld), npy(-ld_fwd)) <= LD_TOL
        blob = cp.prepared()
        assert _native.coupling_apply(y, blob, width, reverse=True)[1] is None      # the default: no log-det
        xr, fresh = _native.coupling_apply(y, blob, width, reverse=True, want_logdet=True)
        assert torch.equal(xr, x) and torch.equal(fresh, ld)
        old = torch.randn(B, device="cuda")
        acc = old.clone()
        _native.coupling_apply(y, blob, width, reverse=True, logdet_out=acc, flags=_native.FLAG_LOGDET_ACCUMULATE)
        assert torch.equal(acc, old + fresh)


def test_recording_rules():
    """whether the result carries a graph is what the PyTorch formulas give, in every combination of grad mode,
    input requiring grad and parameters requiring grad; the values are the native path's bits under no_grad"""
    from fincflow_b200.flows import Coupling

    cp = coupling(12, 8, 8, 128, seed=3)
    x0 = torch.randn(3, 12, 8, 8, device="cuda")
    with torch.no_grad():
        y_ng, ld_ng = cp.reverse_and_logdet(x0)
    for grad_on, x_rg, p_rg in itertools.product([True, False], repeat=3):
        cp.requires_grad_(p_rg)
        x = x0.clone().requires_grad_(x_rg)
        got = {}
        for tc in (True, False):
            Coupling.tensor_core = tc
            try:
                with torch.set_grad_enabled(grad_on):
                    got[tc] = (cp.reverse(x), *cp.reverse_and_logdet(x))
            finally:
                Coupling.tensor_core = True
        what = (grad_on, x_rg, p_rg)
        assert [t.requires_grad for t in got[True]] == [t.requires_grad for t in got[False]], what
        assert [t.grad_fn is None for t in got[True]] == [t.grad_fn is None for t in got[False]], what
        assert torch.equal(got[True][0], y_ng) and torch.equal(got[True][1], y_ng), what
        assert torch.equal(got[True][2], ld_ng), what


@pytest.mark.parametrize("width", [32, 64])
def test_fallback_backward_widths(fp32_convs, width):
    """widths the native backward does not cover: the native forward, the PyTorch-recompute backward"""
    from fincflow_b200 import _native

    assert _native.coupling_prepared_bytes(12, width) > 0 and _native.coupling_prepared_bytes(12, width, True) == 0
    cp = coupling(12, 8, 8, width, seed=width)
    x = torch.randn(5, 12, 8, 8, device="cuda")
    gy, gl = torch.randn_like(x), torch.randn(5, device="cuda")
    y, ld, got = reverse_grads(cp, x, gy, gl)
    with torch.no_grad():
        y0, ld0 = cp.reverse_and_logdet(x)
    assert torch.equal(y, y0) and torch.equal(ld, ld0)
    _, _, want = reverse_grads(float64_copy(cp), x.double(), gy.double(), gl.double())
    for a, b in zip(got, want):
        assert rel_err(npy(a), npy(b)) <= 1e-5


def test_tf32_single_pass():
    cp = coupling(24, 8, 8, 256, seed=5)
    cp.precision = "tf32"
    x = torch.randn(4, 24, 8, 8, device="cuda")
    gy, gl = torch.randn_like(x), torch.randn(4, device="cuda")
    _, _, got = reverse_grads(cp, x, gy, gl)
    _, _, want = reverse_grads(float64_copy(cp, x), x.double(), gy.double(), gl.double())
    errs = [rel_err(npy(a), npy(b)) for a, b in zip(got, want)]
    assert max(errs) <= 2e-3, errs
    assert min(errs) > 1e-7, errs        # the single pass ran (3xTF32 is at ~1e-7)


# ---- whole flow ---------------------------------------------------------------------------------------------------
FLOWS = {
    "mnist": dict(n_blocks=2, block_size=2, image_size=(1, 28, 28), final_steps=1),
    "cifar": dict(n_blocks=3, block_size=2, image_size=(3, 32, 32)),
}


def flow(kind, B, width=128, seed=10):
    """an initialised flow (ActNorm from a first batch, the zero-initialised last coupling convs randomised) and
    latents shaped like its forward's"""
    from fincflow_b200 import flows

    torch.manual_seed(seed)
    model = flows.FastFlow(width=width, actnorm=True, **FLOWS[kind]).cuda()
    C, H, W = FLOWS[kind]["image_size"]
    x = torch.randint(0, 256, (B, C, H, W), device="cuda").float()
    with torch.no_grad():
        zs, _ = model(x)
        for m in model.modules():
            if isinstance(m, flows.Coupling):
                m.net[4].weight.normal_(0, 0.02)
                m.net[4].bias.normal_(0, 0.1)
                m.net[4].logs.normal_(0, 0.1)
    return model, [torch.randn_like(z) for z in zs]


@pytest.mark.parametrize("kind", FLOWS)
def test_log_q_is_the_model_log_prob(kind):
    model, zs = flow(kind, 3)
    with torch.no_grad():
        x, log_q = model.sample_with_log_prob(zs=zs)
        assert torch.equal(x, model.reverse(zs=zs, quantize=False))
        model.preprocess.layers[0].fixed_noise = torch.zeros_like(x)
        log_p = model.log_prob(x)
    assert log_q.shape == (3,)
    assert rel_err(npy(log_q), npy(log_p)) <= 1e-4, (npy(log_q), npy(log_p))
    with torch.no_grad():         # latents drawn inside: the split-prior ones are part of log q too
        torch.manual_seed(1)
        x1, log_q1 = model.sample_with_log_prob(n_samples=2)
        model.preprocess.layers[0].fixed_noise = torch.zeros_like(x1)
        log_p1 = model.log_prob(x1)
    assert rel_err(npy(log_q1), npy(log_p1)) <= 1e-4


@pytest.mark.parametrize("kind", FLOWS)
def test_sample_with_log_prob_grad_whole_flow(fp32_convs, monkeypatch, kind):
    """gradients of (x * r).sum() + (log_q * v).sum() in the latents and every parameter against the PyTorch
    reference flow (FInC inverse: the float64 fixed-point solve; ActNorm / Conv1x1 unfused: torch.inverse, slogdet,
    F.conv2d; Coupling: the PyTorch formulas); none is None or zero"""
    import fincflow_b200.fastflow as ffmod
    from fincflow_b200 import flows

    model, zs = flow(kind, 2)
    params = list(model.parameters())
    outs = {}
    for name in ("ours", "ref"):
        if name == "ref":
            monkeypatch.setattr(ffmod, "finc_inverse",     # (FastFlowUnit.reverse: G = 4, the unit's orders)
                                lambda z, w, G=4, orders=None, dense=None: ref_inverse(
                                    z.double(), w.double(), ORDERS).float())
            monkeypatch.setattr(flows.GlowStep, "fused", False)
            monkeypatch.setattr(flows.Coupling, "tensor_core", False)
        lat = [z.clone().requires_grad_() for z in zs]
        x, log_q = model.sample_with_log_prob(zs=lat)
        g = torch.Generator(device="cuda").manual_seed(11)
        r = torch.randn(x.shape, device="cuda", generator=g)
        v = torch.randn(log_q.shape, device="cuda", generator=g)
        outs[name] = (x, log_q, torch.autograd.grad((x * r).sum() + (log_q * v).sum(), params + lat))
    x, log_q, ours = outs["ours"]
    xr, log_qr, ref = outs["ref"]
    assert rel_err(npy(x), npy(xr)) <= 1e-4 and rel_err(npy(log_q), npy(log_qr)) <= 1e-4
    for (pname, _), a, b in zip(list(model.named_parameters()) + [(f"zs[{i}]", None) for i in range(len(zs))],
                                ours, ref):
        assert a is not None and b is not None, pname
        assert float(a.abs().max()) > 0, pname
        assert rel_err(npy(a), npy(b)) <= 1e-4, (pname, rel_err(npy(a), npy(b)))


def _base_name(name):
    """`finc::tc::coupling_gather_kernel` of `void finc::tc::coupling_gather_kernel(float const*, ...)`"""
    name = name.replace("(anonymous namespace)", "{anon}")
    if name.startswith("void "):
        name = name[5:]
    return re.split(r"[<(]", name, maxsplit=1)[0].strip()


def profiled_sample_kernels():
    """names of the CUDA kernels a differentiable sample + log-density + backward (CIFAR-shaped flow, width 128: the
    native coupling backward) launches, and whether every latent and parameter got a gradient"""
    from torch.profiler import ProfilerActivity, profile

    model, zs = flow("cifar", 4)
    lat = [z.clone().requires_grad_() for z in zs]
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        x, log_q = model.sample_with_log_prob(zs=lat)
        r = torch.randn_like(x)
        ((x * r).sum() + log_q.sum()).backward()
        torch.cuda.synchronize()
    kernels = sorted({e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA
                      and not e.name.startswith(("Memcpy", "Memset"))})
    grads = all(z.grad is not None for z in lat) and all(p.grad is not None for p in model.parameters())
    return {"kernels": kernels, "all_grads": grads}


def test_sample_with_log_prob_runs_only_library_kernels():
    """a differentiable sample + log-density + backward launches the library's kernels (its symbol table) and
    PyTorch's own at::native kernels only: no cuDNN, cuBLAS or cuSOLVER.

    The profile runs in a process of its own.  Its thousands of activity records would otherwise go through the CUPTI
    activity buffers of the test session, and the census tests of test_gpu_kernel_variants.py / test_gpu_tc_variants.py
    depend on the record of a lone kernel not being lost at an activity-buffer boundary."""
    from fincflow_b200 import _native

    here = os.path.dirname(os.path.abspath(__file__))
    code = ("import json, sys; sys.path[:0] = {!r}; import test_gpu_coupling_reverse as t; "
            "print(json.dumps(t.profiled_sample_kernels()))").format([os.path.dirname(here), here])
    run = subprocess.run([sys.executable, *(["-s"] if sys.flags.no_user_site else []), "-c", code],
                         cwd=os.path.dirname(here), capture_output=True, text=True, timeout=900)
    assert run.returncode == 0, run.stderr[-4000:]
    res = json.loads(run.stdout.strip().splitlines()[-1])
    syms = subprocess.run(["nm", "-C", "--defined-only", _native.LIB_PATH], capture_output=True, text=True,
                          check=True).stdout
    ours = {_base_name(line.split(" ", 2)[2]) for line in syms.splitlines() if line.count(" ") >= 2}
    kernels = res["kernels"]
    foreign = [k for k in kernels if "at::native::" not in k and _base_name(k) not in ours]
    assert not foreign, foreign
    mine = {_base_name(k) for k in kernels} & ours
    for k in ("finc::tc::coupling_bwd_pointwise_kernel", "finc::tc::coupling_gather_kernel",
              "finc::tc::rowsum_reduce_kernel"):
        assert k in mine, (k, sorted(mine))
    assert res["all_grads"]
