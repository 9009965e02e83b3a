"""GPU tests of the multi-scale flow assembly (fincflow_b200/flows.py) against a fixture produced
by the reference's own FastFlow model code (tests/golden/make_golden_flow.py), and of the
squeeze kernels (SURVEY.md section 8 row a12)."""
import os

import numpy as np
import pytest
import torch

from conftest import REPO, rel_err

pytestmark = pytest.mark.gpu

# the glue convolutions are PyTorch/cuDNN: full fp32 like the reference's CUDA 10.2 stack
# (modern PyTorch defaults cuDNN convs to TF32, ~5e-4 relative; SURVEY.md appendix D.10)
torch.backends.cudnn.allow_tf32 = False
torch.backends.cuda.matmul.allow_tf32 = False


def _ref_space_to_depth(x):  # the formula of layers/squeeze.py:5-13
    xs = x.size()
    x = x.view(xs[0], xs[1], xs[2] // 2, 2, xs[3] // 2, 2).permute((0, 1, 3, 5, 2, 4)).contiguous()
    return x.view(xs[0], xs[1] * 4, xs[2] // 2, xs[3] // 2)


@pytest.mark.parametrize("shape", [(3, 3, 32, 32), (5, 1, 28, 28), (2, 12, 16, 16), (1, 6, 2, 2), (256, 3, 32, 32),
                                   (64, 12, 64, 64),            # 1.6M float2 items: more than the grid's 148 * 32 * 256
                                   (3, 5, 30, 30), (2, 3, 6, 10)])   # odd H/2 and W/2
def test_squeeze_kernels_bit_exact(shape):
    from fincflow_b200 import _native

    x = torch.randn(*shape, device="cuda")
    y = _native.squeeze(x)
    assert torch.equal(y, _ref_space_to_depth(x))
    assert torch.equal(_native.unsqueeze(y), x)
    assert _native.squeeze(torch.empty(0, 3, 4, 4, device="cuda")).shape == (0, 12, 2, 2)


def test_whole_flow_matches_reference_model():
    from fincflow_b200.flows import FastFlow, clear_grad

    g = np.load(os.path.join(REPO, "tests", "golden", "flow_golden.npz"))
    model = FastFlow(n_blocks=3, block_size=2, image_size=(3, 16, 16), actnorm=True, width=16).cuda()
    sd = {k[3:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("sd/")}
    res = model.load_state_dict(sd, strict=False)
    assert res.missing_keys == []
    assert set(res.unexpected_keys) <= {"preprocess.layers.0.distribution.empty"}
    model.preprocess.layers[0].fixed_noise = torch.from_numpy(g["noise"]).cuda()
    x = torch.from_numpy(g["x"]).cuda()
    zs, logp = model(x)
    assert len(zs) == 3 and [tuple(z.shape[1:]) for z in zs] == [(6, 8, 8), (12, 4, 4), (48, 2, 2)]
    for i, z in enumerate(zs):
        assert rel_err(z.detach().cpu().numpy(), g[f"zs/{i}"]) <= 1e-4, i
    assert rel_err(logp.detach().cpu().numpy(), g["logp"]) <= 1e-5
    # training-step gradients of the FInC weights (mask applied inside the wgrad kernel)
    (-logp.sum() / x.shape[0]).backward()
    model.apply(clear_grad)
    own = {n: p.grad for n, p in model.named_parameters() if n.endswith("fastflow_unit.weight")}
    assert len(own) == 6
    for name, grad in own.items():
        prefix = name[:-len("weight")]
        want = np.concatenate([g[f"grad/{prefix}conv_{q}.conv.weight"] for q in ("tl", "tr", "bl", "br")], 0)
        assert rel_err(grad.cpu().numpy(), want) <= 1e-4, name
        assert np.array_equal(grad.cpu().numpy() == 0, want == 0)
    # exact reconstruction through the wavefront inverse kernels (pixels are integers)
    with torch.no_grad():
        x_rec = model.reverse(n_samples=x.shape[0], zs=[z.detach() for z in zs])
    assert torch.equal(x_rec, x)
    assert np.array_equal(x_rec.cpu().numpy(), g["x_rec"])


def test_builders_and_sampling_shapes():
    from fincflow_b200 import flows

    torch.manual_seed(0)
    m = flows.FastFlow(n_blocks=2, block_size=2, image_size=(1, 28, 28), final_steps=1, width=16).cuda()
    x = torch.randint(0, 256, (8, 1, 28, 28), device="cuda").float()
    zs, logp = m(x)
    assert [tuple(z.shape[1:]) for z in zs] == [(2, 14, 14), (8, 7, 7)] and logp.shape == (8,)
    assert torch.isfinite(logp).all()
    with torch.no_grad():
        s, _ = m.sample(5)
        assert s.shape == (5, 1, 28, 28)
        rec = m.reconstruct_exact(x)  # floor(x + u + err): u within err of 0/1 may flip a pixel by one
        assert (rec - x).abs().max().item() <= 1 and (rec != x).float().mean().item() < 1e-3
    m64 = flows.FastFlow(n_blocks=4, block_size=1, image_size=(3, 64, 64), final_steps=1, kernel_size=(5, 5),
                         width=16).cuda()
    xb = torch.randint(0, 256, (2, 3, 64, 64), device="cuda").float()
    with torch.no_grad():
        zs, logp = m64(xb)
        assert tuple(zs[-1].shape[1:]) == (96, 4, 4)
        rec = m64.reverse(n_samples=2, zs=zs)
        assert (rec - xb).abs().max().item() <= 1 and (rec != xb).float().mean().item() < 1e-3


@pytest.mark.parametrize("shape", [(5, 12, 16, 16), (7, 24, 8, 8), (9, 48, 4, 4), (3, 96, 4, 4), (6, 4, 14, 14), (5, 8, 7, 7),
                                   (4, 16, 5, 6), (3, 32, 3, 3), (2, 10, 5, 5), (256, 12, 16, 16), (1, 24, 16, 16)],
                         ids=lambda s: "B{}C{}_{}x{}".format(*s))
def test_affine1x1_is_actnorm_then_conv1x1(shape):
    """finc_affine1x1_f32 == the reference's ActNorm followed by Conv1x1 (layers/actnorm.py:14-52,
    layers/conv1x1.py:18-43), its reverse and its backward-data pass; fp64 formulas as the oracle"""
    from fincflow_b200 import _native

    B, C, H, W = shape
    gen = torch.Generator().manual_seed(C * 100 + H)
    x = torch.randn(B, C, H, W, generator=gen, dtype=torch.float64)
    Wm = torch.linalg.qr(torch.randn(C, C, generator=gen, dtype=torch.float64))[0] + 0.05 * torch.randn(C, C, generator=gen, dtype=torch.float64)
    t = torch.randn(C, generator=gen, dtype=torch.float64)
    ls = 0.3 * torch.randn(C, generator=gen, dtype=torch.float64)
    want = torch.einsum("oi,nihw->nohw", Wm, (x - t.view(1, C, 1, 1)) * torch.exp(-ls).view(1, C, 1, 1))
    A = Wm * torch.exp(-ls).unsqueeze(0)
    b = -(A @ t)
    xd = x.float().cuda()
    y = _native.affine1x1(xd, A.float().cuda(), b.float().cuda())
    assert rel_err(y.cpu().numpy(), want.numpy()) <= 1e-5
    # no bias == plain Conv1x1; A^T == its backward-data pass
    y0 = _native.affine1x1(xd, Wm.float().cuda())
    assert rel_err(y0.cpu().numpy(), torch.einsum("oi,nihw->nohw", Wm, x).numpy()) <= 1e-5
    yt = _native.affine1x1(xd, Wm.t().contiguous().float().cuda())
    assert rel_err(yt.cpu().numpy(), torch.einsum("io,nihw->nohw", Wm, x).numpy()) <= 1e-5
    # reverse: A^-1 with bias = translation
    Ainv = torch.exp(ls).unsqueeze(1) * torch.linalg.inv(Wm)
    back = _native.affine1x1(y, Ainv.float().cuda(), t.float().cuda())
    assert (back.cpu().double() - x).abs().max().item() <= 1e-4
    # unaligned view (odd float offset): the kernel falls back to narrower vectors
    buf = torch.zeros(xd.numel() + 1, device="cuda")
    xv = buf[1:].view_as(xd)
    xv.copy_(xd)
    assert torch.equal(_native.affine1x1(xv, A.float().cuda(), b.float().cuda()), y) or \
        rel_err(_native.affine1x1(xv, A.float().cuda(), b.float().cuda()).cpu().numpy(), want.numpy()) <= 1e-5


@pytest.mark.parametrize("actnorm", [False, True])
def test_fused_glow_step_equals_layerwise(actnorm):
    """GlowStep with ActNorm+Conv1x1 on the fused kernel == the layer-by-layer PyTorch path:
    values, log-determinant, every parameter gradient, reverse"""
    from fincflow_b200.flows import GlowStep

    torch.manual_seed(3)
    size = (12, 8, 8)
    step = GlowStep(size, actnorm=actnorm, width=16).cuda()
    for p in step.glow_step.coupling.parameters():   # zero-initialised last conv would hide the path
        p.data.normal_(0, 0.05)
    x = torch.randn(6, *size, device="cuda") * 1.7 + 0.3
    if actnorm:
        step.fused = False
        step(x)                                       # data-dependent init
        step.glow_step.actnorm.log_scale.data.add_(0.1 * torch.randn(12, device="cuda"))
    res = {}
    for fused in (False, True):
        step.fused = fused
        step.zero_grad()
        xi = x.clone().requires_grad_(True)
        y, ld = step(xi)
        (y.pow(2).sum() + (ld.sum() if torch.is_tensor(ld) else ld)).backward()
        res[fused] = (y.detach(), torch.as_tensor(ld).detach().expand(6).clone(), xi.grad.clone(),
                      {n: p.grad.clone() for n, p in step.named_parameters() if p.grad is not None})
        with torch.no_grad():
            assert (step.reverse(y.detach()) - x).abs().max().item() <= 1e-4
    (y0, l0, g0, p0), (y1, l1, g1, p1) = res[False], res[True]
    assert rel_err(y1.cpu().numpy(), y0.cpu().numpy()) <= 1e-5
    assert rel_err(l1.cpu().numpy(), l0.cpu().numpy()) <= 1e-5
    assert rel_err(g1.cpu().numpy(), g0.cpu().numpy()) <= 1e-5
    assert p0.keys() == p1.keys()
    for n in p0:
        assert rel_err(p1[n].cpu().numpy(), p0[n].cpu().numpy()) <= 2e-5, n


@pytest.mark.parametrize("shape", [(256, 12, 16, 16), (37, 24, 8, 8), (300, 48, 4, 4), (9, 96, 4, 4), (64, 4, 14, 14), (33, 8, 7, 7),
                                   (5, 10, 5, 5), (1, 12, 2, 2), (3000, 12, 16, 16)],
                         ids=lambda s: "B{}C{}_{}x{}".format(*s))
def test_affine1x1_backward_weight(shape):
    """dA = sum dy x^T, db = sum dy (finc_affine1x1_backward_weight_f32) vs fp64; deterministic"""
    from fincflow_b200 import _native

    B, C, H, W = shape
    gen = torch.Generator().manual_seed(B + C)
    x = torch.randn(B, C, H, W, generator=gen)
    dy = torch.randn(B, C, H, W, generator=gen)
    want_A = torch.einsum("nop,nip->oi", dy.double().flatten(2), x.double().flatten(2))
    want_b = dy.double().sum(dim=(0, 2, 3))
    dA, db = _native.affine1x1_backward_weight(dy.cuda(), x.cuda())
    scale = float(want_A.abs().max())
    assert (dA.cpu().double() - want_A).abs().max().item() <= 2e-5 * max(scale, (B * H * W) ** 0.5)
    assert (db.cpu().double() - want_b).abs().max().item() <= 2e-5 * max(float(want_b.abs().max()), (B * H * W) ** 0.5)
    dA2, db2 = _native.affine1x1_backward_weight(dy.cuda(), x.cuda())
    assert torch.equal(dA, dA2) and torch.equal(db, db2)
    dA3, none = _native.affine1x1_backward_weight(dy.cuda(), x.cuda(), want_bias=False)
    assert none is None and torch.equal(dA, dA3)


def test_fused_preprocess_matches_the_four_layers():
    """finc_preprocess_f32 == Dequantization -> Normalization(0,256) -> Normalization(-a, 1/(1-2a)) -> Logit
    with the summed log-determinants (fastflow_cifar_multi_gpu.py:162-186), and its reverse"""
    from fincflow_b200.flows import Preprocess

    torch.manual_seed(4)
    pre = Preprocess((3, 32, 32)).cuda()
    x = torch.randint(0, 256, (37, 3, 32, 32), device="cuda").float()
    pre.layers[0].fixed_noise = torch.rand_like(x)
    y, ld = pre(x)
    Preprocess.fused = False
    try:
        y_ref, ld_ref = pre(x)
        x_back_ref = pre.reverse(y_ref)
    finally:
        Preprocess.fused = True
    assert rel_err(y.cpu().numpy(), y_ref.cpu().numpy()) <= 1e-6
    assert rel_err(ld.cpu().numpy(), ld_ref.cpu().numpy()) <= 1e-6
    with torch.no_grad():
        x_back = pre.reverse(y)
    # floor(x + u + rounding): a noise value within rounding of 0 or 1 may flip a pixel by one level
    for back in (x_back, x_back_ref):
        assert (back - x).abs().max().item() <= 1 and (back != x).float().mean().item() < 1e-3
    assert (x_back != x_back_ref).float().mean().item() < 1e-3


@pytest.mark.parametrize("tag", ["cfg2", "cfg3"])
def test_full_depth_flows_match_the_reference_model(tag):
    """BASELINE configs[1] (MNIST 1x28x28 flow, exact log-likelihood / bits per dimension) and configs[2]
    (CIFAR-10-shaped flow, 3 blocks x 16 steps) at FULL depth and coupling width 512, against outputs of the
    reference's own model code (tests/golden/make_golden_flow_full.py; parameters = tests/golden/param_fill.py).
    Every layer runs on our kernels here: FInC units, fused ActNorm+Conv1x1, the tensor-core coupling, fused
    preprocessing, closed-form priors."""
    import math
    import sys

    sys.path.insert(0, os.path.join(REPO, "tests", "golden"))
    from param_fill import filled_state_dict

    from fincflow_b200 import flows

    g = np.load(os.path.join(REPO, "tests", "golden", "flow_full_golden.npz"))
    if tag == "cfg2":
        model, seed = flows.fastflow_mnist(actnorm=True), 21
    else:
        model, seed = flows.fastflow_cifar10(actnorm=True), 22
    res = model.load_state_dict(filled_state_dict(model, seed), strict=False)
    assert all(k.startswith("preprocess.") for k in res.missing_keys), res.missing_keys
    model = model.cuda().eval()
    x = torch.from_numpy(g[f"{tag}/x"]).cuda()
    model.preprocess.layers[0].fixed_noise = torch.from_numpy(g[f"{tag}/noise"]).cuda()
    with torch.no_grad():
        zs, logp = model(x)
        bpd = -model.log_prob(x, bits_per_pixel=True)
        x_rec = model.reverse(n_samples=x.shape[0], zs=zs)
    n = 0
    while f"{tag}/zs/{n}" in g.files:
        n += 1
    assert len(zs) == n
    # latents and log-likelihood <= 1e-5 (cfg2: 17 flow steps) / 2e-5 (cfg3: 48 steps deep; PyTorch's own fp32
    # GPU path differs from the CPU reference by 2e-6 .. 6e-6 on these latents)
    tol_z, tol_l = (1e-5, 1e-5) if tag == "cfg2" else (2e-5, 2e-5)
    for i, z in enumerate(zs):
        assert rel_err(z.cpu().numpy(), g[f"{tag}/zs/{i}"]) <= tol_z, (tag, i, rel_err(z.cpu().numpy(), g[f"{tag}/zs/{i}"]))
    assert rel_err(logp.cpu().numpy(), g[f"{tag}/logp"]) <= tol_l
    assert rel_err(bpd.cpu().numpy(), g[f"{tag}/bpd"]) <= tol_l
    assert (x_rec - x).abs().max().item() <= 1 and (x_rec != x).float().mean().item() < 1e-3


def test_inference_session_graphs_match_eager():
    """flows.InferenceSession (CUDA graphs of forward / sample) returns what the eager calls return"""
    from fincflow_b200 import flows

    torch.manual_seed(3)
    m = flows.FastFlow(n_blocks=3, block_size=2, image_size=(3, 16, 16), actnorm=True, width=128).cuda()
    x = torch.randint(0, 256, (8, 3, 16, 16), device="cuda").float()
    m.preprocess.layers[0].fixed_noise = torch.rand_like(x)
    with torch.no_grad():
        m(x)                                        # data-dependent ActNorm init
        zs, logp = m(x)
    sess = flows.InferenceSession(m)
    for _ in range(2):                              # capture, then replay
        zs_g, logp_g = sess.log_prob(x)
        assert torch.equal(logp_g, logp) and all(torch.equal(a, b) for a, b in zip(zs_g, zs))
    x2 = torch.randint(0, 256, (8, 3, 16, 16), device="cuda").float()
    with torch.no_grad():
        _, logp2 = m(x2)
    assert torch.equal(sess.log_prob(x2)[1], logp2)
    s1 = sess.sample(4).clone()
    s2 = sess.sample(4)
    assert s1.shape == (4, 3, 16, 16) and not torch.equal(s1, s2)     # fresh latents on every replay
    assert float(s2.min()) >= 0 and float(s2.max()) <= 255


@pytest.mark.parametrize("C", [4, 12, 24, 48, 96])
def test_batched_slogdet_inverse_kernel(C):
    """finc_slogdet_inverse_f32 against torch.linalg (fp64), and the autograd of the batched log-determinant"""
    from fincflow_b200 import _native
    from fincflow_b200.flows import _SlogdetFn

    torch.manual_seed(C)
    W = torch.linalg.qr(torch.randn(7, C, C, device="cuda"))[0] + 0.05 * torch.randn(7, C, C, device="cuda")
    ld, Winv = _native.slogdet_inverse(W.contiguous())
    ref_ld = torch.linalg.slogdet(W.double())[1]
    ref_inv = torch.linalg.inv(W.double())
    assert float((ld.double() - ref_ld).abs().max()) <= 1e-5 * max(1.0, float(ref_ld.abs().max()))
    assert rel_err(Winv.cpu().numpy(), ref_inv.cpu().numpy()) <= 1e-5
    Wg = W.clone().requires_grad_(True)
    g = torch.randn(7, device="cuda")
    (_SlogdetFn.apply(Wg) * g).sum().backward()
    Wd = W.double().requires_grad_(True)
    (torch.linalg.slogdet(Wd)[1] * g.double()).sum().backward()
    assert rel_err(Wg.grad.cpu().numpy(), Wd.grad.cpu().numpy()) <= 1e-5


def test_flow_trainer_graph_step_equals_eager_step():
    """FlowTrainer(use_graph=True): the CUDA-graph replay of the whole train step follows the eager trajectory"""
    from fincflow_b200 import flows
    from fincflow_b200.train import FlowTrainer

    def run(use_graph):
        torch.manual_seed(5)
        m = flows.FastFlow(n_blocks=2, block_size=2, image_size=(3, 16, 16), actnorm=True, width=128).cuda()
        tr = FlowTrainer(m, lr=1e-3, use_graph=use_graph, graph_warmup=2)
        g = torch.Generator(device="cuda").manual_seed(9)
        losses = []
        m.preprocess.layers[0].fixed_noise = torch.full((8, 3, 16, 16), 0.5, device="cuda")   # ONE tensor: the graph reads it in place
        for i in range(6):
            x = torch.randint(0, 256, (8, 3, 16, 16), device="cuda", generator=g).float()
            losses.append(float(tr.step(x)))
        return losses, [p.detach().clone() for p in m.parameters()], tr

    l_e, p_e, _ = run(False)
    l_g, p_g, tr = run(True)
    assert tr._graph is not None
    # the capturing call replays the graph once, so every call is exactly one optimizer step: same trajectory
    assert np.allclose(l_e, l_g, rtol=1e-4)
    for a, b in zip(p_g, p_e):
        assert rel_err(a.cpu().numpy(), b.detach().cpu().numpy()) <= 1e-4


@pytest.mark.parametrize("actnorm", [True, False])
def test_fastflowstep_fused_eval_equals_layer_by_layer(actnorm):
    """FastFlowStep under no_grad: FastFlowUnit + [ActNorm +] Conv1x1 in ONE finc_chain_f32 launch, then the
    coupling layer -- same values and log-determinants as the three separate layers"""
    from fincflow_b200 import _native, flows

    torch.manual_seed(11)
    for size, B in (((3, 32, 32), 64), ((6, 16, 16), 33), ((12, 8, 8), 256)):
        step = flows.FastFlowStep((size[0] * 4, size[1] // 2, size[2] // 2), actnorm=actnorm, width=64).cuda()
        x = torch.randn(B, size[0] * 4, size[1] // 2, size[2] // 2, device="cuda")
        with torch.no_grad():
            step(x)                                   # ActNorm data-dependent init (un-fused once)
            for p in step.parameters():
                p.add_(0.05 * torch.randn_like(p))
            step(x)                                   # rebuilds the cached glue constants for the new parameters
            n0 = _native.launch_count
            y, ld = step(x)
            fused_launches = _native.launch_count - n0
            flows.FastFlowStep.fused = False
            try:
                n0 = _native.launch_count
                y_ref, ld_ref = step(x)
                ref_launches = _native.launch_count - n0
            finally:
                flows.FastFlowStep.fused = True
        assert fused_launches == ref_launches - 1
        assert rel_err(y.cpu().numpy(), y_ref.cpu().numpy()) <= 2e-6
        with torch.no_grad():   # a view the chain kernel cannot take (not 16-byte aligned): the layer-by-layer path runs
            flat = torch.randn(x.numel() + 1, device="cuda")
            xv = flat[1:].view_as(x)
            xv.copy_(x)
            y2, ld2 = step(xv)
        assert rel_err(y2.cpu().numpy(), y_ref.cpu().numpy()) <= 2e-6 and rel_err(ld2.cpu().numpy(), ld_ref.cpu().numpy()) <= 1e-6
        assert rel_err(ld.cpu().numpy(), ld_ref.cpu().numpy()) <= 1e-6


def test_flat_adam_matches_torch_adam_and_caches_see_graph_updates():
    """FlowTrainer's one-launch Adam over the flattened parameters follows torch.optim.Adam, and an evaluation after
    CUDA-graph training steps sees the trained weights (version counters are bumped after every replay: the layers'
    prepared-weight caches are keyed on them)"""
    from fincflow_b200 import flows
    from fincflow_b200.train import FlowTrainer

    def run(**kw):
        torch.manual_seed(5)
        m = flows.FastFlow(n_blocks=2, block_size=2, image_size=(3, 16, 16), actnorm=True, width=128).cuda()
        tr = FlowTrainer(m, lr=1e-3, **kw)
        m.preprocess.layers[0].fixed_noise = torch.full((8, 3, 16, 16), 0.5, device="cuda")
        g = torch.Generator(device="cuda").manual_seed(9)
        xs = [torch.randint(0, 256, (8, 3, 16, 16), device="cuda", generator=g).float() for _ in range(6)]
        losses = [float(tr.step(x)) for x in xs]
        m.eval()
        with torch.no_grad():
            _, logp = m(xs[0])
        return losses, [p.detach().clone() for p in m.parameters()], logp.clone(), tr

    l_t, p_t, lp_t, tr_t = run(flat_adam=False)
    l_f, p_f, lp_f, tr_f = run(flat_adam=True)
    # the same training with the coupling layers on PyTorch's own convolutions (fp32): an implementation whose
    # weight caches survive an optimizer step (torch's fused Adam does not bump `_version`) fails here at step 2
    flows.Coupling.tensor_core = False
    try:
        l_ref = run(flat_adam=False)[0]
    finally:
        flows.Coupling.tensor_core = True
    # (the stale-cache bug showed as 7e-4 at the second step; fp32 round-off between the two coupling implementations
    # is ~1e-5 there and grows slowly with the number of updates)
    assert np.allclose(l_t[:3], l_ref[:3], rtol=1e-4) and np.allclose(l_f[:3], l_ref[:3], rtol=1e-4), (l_t, l_f, l_ref)
    assert np.allclose(l_t, l_ref, rtol=2e-3) and np.allclose(l_f, l_ref, rtol=2e-3), (l_t, l_f, l_ref)
    l_g, p_g, lp_g, tr_g = run(flat_adam=True, use_graph=True, graph_warmup=2)
    assert type(tr_t.optimizer).__name__ == "Adam" and type(tr_f.optimizer).__name__ == "FlatAdam"
    assert tr_g._graph is not None
    assert np.allclose(l_t, l_f, rtol=1e-4) and np.allclose(l_f, l_g, rtol=1e-4)
    for a, b, c in zip(p_t, p_f, p_g):
        assert rel_err(b.cpu().numpy(), a.cpu().numpy()) <= 1e-3     # two Adam implementations, six updates
        assert rel_err(c.cpu().numpy(), b.cpu().numpy()) <= 1e-4     # the same kernels, eager vs graph
    # evaluation after training: the graph run must not evaluate with weights cached before its last updates
    assert rel_err(lp_f.cpu().numpy(), lp_t.cpu().numpy()) <= 1e-4
    assert rel_err(lp_g.cpu().numpy(), lp_f.cpu().numpy()) <= 1e-4
    sd = tr_f.optimizer.state_dict()
    tr_g.optimizer.load_state_dict(sd)
    assert torch.equal(tr_g.optimizer.exp_avg, tr_f.optimizer.exp_avg) and float(tr_g.optimizer.step_t) == 6.0
