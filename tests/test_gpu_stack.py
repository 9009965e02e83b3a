"""GPU tests of the FInC stack runner (train step + sampling as CUDA graphs) against the
autograd path and the CPU oracle / reference-path twin."""
import math

import numpy as np
import pytest
import torch

from conftest import rel_err
from oracle import finc_oracle as fo

pytestmark = pytest.mark.gpu


def _small_levels():
    from fincflow_b200.stack import LevelSpec

    return [LevelSpec(12, 8, 8, 3, (3, 3)), LevelSpec(24, 4, 4, 2, (3, 3)), LevelSpec(8, 7, 7, 1, (3, 3))]


@pytest.mark.parametrize("use_graphs", [False, True])
def test_runner_matches_autograd_and_oracle(use_graphs):
    from fincflow_b200.stack import FincStack, HotPathRunner

    torch.manual_seed(0)
    B = 10
    lv = _small_levels()
    stack = FincStack(lv).cuda()
    w0 = stack.flat.detach().clone()
    runner = HotPathRunner(stack, B, "cuda", slots=2, lr=0.0, use_graphs=use_graphs)  # lr 0: weights stay fixed
    for s in runner.slots:
        for li in range(len(lv)):
            s.acts[li][0].normal_()
            s.zin[li].normal_()
    runner.prepare()
    runner.step(1)
    torch.cuda.synchronize()
    assert torch.equal(stack.flat.detach(), w0)
    s = runner.slots[1]
    # autograd twin
    ref = FincStack(lv).cuda()
    ref.flat.data.copy_(w0)
    loss = 0
    for li in range(len(lv)):
        z, logp = ref(s.acts[li][0], level=li)
        assert rel_err(s.logp[li].cpu().numpy(), logp.detach().cpu().numpy()) <= 1e-5
        loss = loss - logp.sum() / B
        assert torch.equal(z.detach(), s.acts[li][lv[li].n_units])
        # oracle: logp of the chain
        h = s.acts[li][0].cpu().numpy()
        for u in range(lv[li].n_units):
            h = fo.forward(h, ref.unit_weight(li, u).detach().cpu().numpy())
        want = -0.5 * (h.reshape(B, -1) ** 2).sum(1) - 0.5 * lv[li].dim * math.log(2 * math.pi)
        assert rel_err(s.logp[li].cpu().numpy(), want) <= 1e-5
    loss.backward()
    assert rel_err(runner.grad.cpu().numpy(), ref.flat.grad.cpu().numpy()) <= 1e-5
    # masked entries of the bucket are exactly zero
    g0 = stack.unit_weight(0, 0, runner.grad).cpu().numpy()
    assert np.array_equal(g0 == 0, fo.apply_grad_mask(np.ones_like(g0)) == 0)
    # sampling pass == reverse chain == oracle inverse chain
    for li in range(len(lv)):
        x = ref.reverse(s.zin[li], level=li)
        assert torch.equal(x, s.sample_out[li])
        h = s.zin[li].cpu().numpy()
        for u in reversed(range(lv[li].n_units)):
            h = fo.inverse(h, ref.unit_weight(li, u).detach().cpu().numpy())
        assert rel_err(x.cpu().numpy(), h) <= 1e-5


def test_host_io_step_and_adam_update():
    from fincflow_b200.stack import FincStack, HotPathRunner

    torch.manual_seed(1)
    B = 6
    lv = _small_levels()
    stack = FincStack(lv).cuda()
    w0 = stack.flat.detach().clone()
    runner = HotPathRunner(stack, B, "cuda", slots=1, lr=1e-3, host_io=True)
    s = runner.slots[0]
    for li in range(len(lv)):
        s.x_host[li].normal_()
        s.z_host[li].normal_()
    runner.prepare()
    w1 = stack.flat.detach().clone()
    # prepare() warms every phase up (optimizer included) but must leave the model untouched
    assert torch.equal(w1, w0)
    assert float(runner.adam_step) == 0.0 and not runner.exp_avg.any() and not runner.exp_avg_sq.any()
    runner.step(0)
    torch.cuda.synchronize()
    w2 = stack.flat.detach()
    assert not torch.equal(w1, w2) and float(runner.adam_step) == 1.0
    # the FInC invariant survives Adam because masked gradients are exactly zero
    for li in range(len(lv)):
        for u in range(lv[li].n_units):
            a, b = stack.unit_weight(li, u, w0).cpu().numpy(), stack.unit_weight(li, u).detach().cpu().numpy()
            frozen = fo.apply_grad_mask(np.ones_like(a)) == 0
            assert np.array_equal(a[frozen], b[frozen])
    # host results: logp finite, samples invert to the host z through the UPDATED weights
    for li in range(len(lv)):
        assert torch.isfinite(s.logp_host[li]).all()
        h = s.samp_host[li].cuda()
        for u in range(lv[li].n_units):
            h, _ = __import__("fincflow_b200")._native.forward(h, stack.unit_weight(li, u).detach(), want_logdet=False)
        assert (h.cpu() - s.z_host[li]).abs().max().item() <= 1e-4


def test_host_io_pipeline_over_slots():
    """copy-in / compute / copy-out of consecutive steps overlap; every slot still gets the
    results of ITS inputs (lr = 0 keeps the weights fixed so each step has a closed-form answer)"""
    from fincflow_b200.stack import FincStack, HotPathRunner

    torch.manual_seed(2)
    B, NS = 5, 3
    lv = _small_levels()
    stack = FincStack(lv).cuda()
    runner = HotPathRunner(stack, B, "cuda", slots=NS, lr=0.0, host_io=True)
    for s in runner.slots:
        for li in range(len(lv)):
            s.x_host[li].normal_()
            s.z_host[li].normal_()
    runner.prepare()
    for rounds in range(3):
        for k in range(NS):
            # fresh inputs for the slot: its previous results must have landed before we overwrite
            runner.wait(k)
            for li in range(len(lv)):
                runner.slots[k].x_host[li].normal_()
                runner.slots[k].z_host[li].normal_()
            runner.step(k)
    runner.drain()
    torch.cuda.synchronize()
    with torch.no_grad():
        for s in runner.slots:
            for li in range(len(lv)):
                z, logp = stack.forward(s.x_host[li].cuda(), li)
                assert (logp.cpu() - s.logp_host[li]).abs().max().item() <= 1e-5 * max(1.0, logp.abs().max().item())
                x = stack.reverse(s.z_host[li].cuda(), li)
                assert rel_err(x.cpu().numpy(), s.samp_host[li].numpy()) <= 1e-5


def test_device_latents_sampling():
    """device_latents=True: z ~ N(0, I) is drawn inside the sampling graph (reference: model.sample ->
    base_distribution.sample on the device); the samples invert the latents that were drawn"""
    from fincflow_b200.stack import FincStack, HotPathRunner

    torch.manual_seed(4)
    B = 64
    lv = _small_levels()
    stack = FincStack(lv).cuda()
    runner = HotPathRunner(stack, B, "cuda", slots=1, lr=0.0, host_io=True, device_latents=True)
    s = runner.slots[0]
    for li in range(len(lv)):
        s.x_host[li].normal_()
    runner.prepare()
    drawn = []
    for _ in range(2):
        runner.step(0)
        runner.drain()
        torch.cuda.synchronize()
        drawn.append([z.clone() for z in s.zin])
        with torch.no_grad():
            for li in range(len(lv)):
                z, _ = stack.forward(s.samp_host[li].cuda(), li)
                assert rel_err(z.cpu().numpy(), s.zin[li].cpu().numpy()) <= 1e-5
                assert abs(float(s.zin[li].mean())) < 0.05 and abs(float(s.zin[li].std()) - 1.0) < 0.05
    assert not torch.equal(drawn[0][0], drawn[1][0])   # a fresh draw per replay


@pytest.mark.parametrize("host_io", [False, True])
def test_overlapped_sampling_matches_serial(host_io):
    """overlap_sampling=True (sampling pass of step k on its own stream, next to the train phases of
    step k+1) produces exactly what the serial schedule produces: same weights after every update,
    same log-likelihoods, same samples"""
    from fincflow_b200.stack import FincStack, HotPathRunner

    B, NS, STEPS = 6, 3, 7
    lv = _small_levels()
    outs = []
    for overlap in (False, True):
        torch.manual_seed(11)
        stack = FincStack(lv).cuda()
        runner = HotPathRunner(stack, B, "cuda", slots=NS, lr=1e-2, host_io=host_io, overlap_sampling=overlap)
        gen = torch.Generator(device="cuda").manual_seed(5)
        cgen = torch.Generator().manual_seed(5)
        for s in runner.slots:
            for li in range(len(lv)):
                if host_io:
                    s.x_host[li].normal_(generator=cgen)
                    s.z_host[li].normal_(generator=cgen)
                else:
                    s.acts[li][0].normal_(generator=gen)
                    s.zin[li].normal_(generator=gen)
        runner.prepare()
        w_after_prepare = stack.flat.detach().clone()
        rec = []
        for k in range(STEPS):
            runner.step(k % NS)
        runner.drain()
        torch.cuda.synchronize()
        for s in runner.slots:
            for li in range(len(lv)):
                rec.append((s.logp_host[li].clone() if host_io else s.logp[li].clone().cpu(),
                            s.samp_host[li].clone() if host_io else s.sample_out[li].clone().cpu()))
        outs.append((w_after_prepare, stack.flat.detach().clone(), rec))
    (w0a, w1a, ra), (w0b, w1b, rb) = outs
    assert torch.equal(w0a, w0b) and torch.equal(w1a, w1b)
    assert not torch.equal(w0a, w1a)
    for (la, sa), (lb, sb) in zip(ra, rb):
        assert torch.equal(la, lb) and torch.equal(sa, sb)


def test_reference_cpu_path_twin_agrees():
    """bench.py's reference arm computes the same step as the GPU runner"""
    from fincflow_b200.stack import FincStack, HotPathRunner, LevelSpec
    from oracle.reference_path import ReferenceCpuStack

    lv = [LevelSpec(12, 8, 8, 2, (3, 3)), LevelSpec(24, 4, 4, 2, (3, 3))]
    B = 4
    ref = ReferenceCpuStack(lv, B, seed=5, lr=0.0, threads=1)
    stack = FincStack(lv).cuda()
    with torch.no_grad():
        for li in range(len(lv)):
            for u in range(lv[li].n_units):
                stack.unit_weight(li, u).copy_(ref.weights[li][u].detach())
    runner = HotPathRunner(stack, B, "cuda", slots=1, lr=0.0, use_graphs=False)
    s = runner.slots[0]
    for li in range(len(lv)):
        s.acts[li][0].copy_(ref.x[li])
        s.zin[li].copy_(ref.z[li])
    runner.prepare()
    logps, samples = ref.step()
    torch.cuda.synchronize()
    for li in range(len(lv)):
        assert rel_err(s.logp[li].cpu().numpy(), logps[li].detach().numpy()) <= 1e-5
        assert rel_err(s.sample_out[li].cpu().numpy(), samples[li].numpy()) <= 1e-5
        for u in range(lv[li].n_units):
            assert rel_err(stack.unit_weight(li, u, runner.grad).cpu().numpy(),
                           ref.weights[li][u].grad.numpy()) <= 1e-5


def test_fused_adam_matches_torch():
    from fincflow_b200 import _native

    torch.manual_seed(0)
    for n in (10007, 1000003):   # 1000003 > SMs * 8 * 256: the grid-stride loop runs more than one pass
        p0 = torch.randn(n, device="cuda")
        ref = p0.clone().requires_grad_(True)
        opt = torch.optim.Adam([ref], lr=1e-3)
        p, m, v, step = p0.clone(), torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda"), torch.zeros(1, device="cuda")
        for it in range(5):
            g = torch.randn(n, device="cuda")
            ref.grad = g.clone()
            opt.step()
            _native.adam_step_(p, g, m, v, step, lr=1e-3)
        assert step.item() == 5.0
        assert torch.allclose(p, ref.detach(), rtol=1e-5, atol=1e-6)


def _run_steps(levels, B, n_steps, **kw):
    from fincflow_b200.stack import FincStack, HotPathRunner

    torch.manual_seed(0)
    stack = FincStack(levels).cuda()
    r = HotPathRunner(stack, B, torch.device("cuda"), slots=1, lr=1e-2, **kw)
    g = torch.Generator(device="cuda").manual_seed(5)
    for li in range(len(levels)):
        r.slots[0].acts[li][0].normal_(generator=g)
        r.slots[0].zin[li].normal_(generator=g)
    r.prepare()
    for _ in range(n_steps):
        r.step(0)
    torch.cuda.synchronize()
    s = r.slots[0]
    return (stack.flat.detach().clone(), [t.clone() for t in s.logp], [s.sample_out[k].clone() for k in sorted(s.sample_out)], r)


@pytest.mark.gpu
def test_runner_execution_options_agree():
    """chain kernels / batched dW / level-parallel streams / per-unit launches: the same training trajectory and the
    same samples (chains are bit-identical; the batched dW sums its batch slices in another fixed order)"""
    from fincflow_b200.stack import LevelSpec

    levels = [LevelSpec(12, 16, 16, 5, (3, 3)), LevelSpec(24, 8, 8, 4, (3, 3)), LevelSpec(48, 4, 4, 3, (3, 3))]
    ref = _run_steps(levels, 64, 3, chain=False)
    # 12 forward + 3 base log-prob + 9 dX + 12 dW + 12 inverse + 2 Adam + 9 weight-table launches
    assert ref[3].launches_per_step == 12 + 3 + 9 + 12 + 12 + 2 + 9
    for kw in (dict(chain=True, batched_wgrad=False), dict(chain=True), dict(chain=True, level_parallel=True)):
        got = _run_steps(levels, 64, 3, **kw)
        assert all(got[3].chain) and all(got[3].inv_chain)
        assert got[3].launches_per_step < ref[3].launches_per_step
        exact = not kw.get("batched_wgrad", True)
        if exact:
            assert torch.equal(got[0], ref[0])
            assert all(torch.equal(a, b) for a, b in zip(got[1], ref[1]))
            assert all(torch.equal(a, b) for a, b in zip(got[2], ref[2]))
        else:
            assert rel_err(got[0].cpu().numpy(), ref[0].cpu().numpy()) <= 1e-5
            for a, b in zip(got[1] + got[2], ref[1] + ref[2]):
                assert rel_err(a.cpu().numpy(), b.cpu().numpy()) <= 1e-4


@pytest.mark.gpu
def test_runner_dense_inverse_sampling_matches_wavefront():
    from fincflow_b200.stack import HotPathRunner, LevelSpec

    levels = [LevelSpec(48, 8, 8, 3, (5, 5)), LevelSpec(96, 4, 4, 2, (5, 5))]
    a = _run_steps(levels, 512, 0)
    b = _run_steps(levels, 512, 0, dense_inverse=True)
    assert len(b[3].dense) >= 1                       # at least one level measured faster as a GEMM
    for r in (a[3], b[3]):
        r.run_phase(0, HotPathRunner.PHASES.index("inverse"))
    torch.cuda.synchronize()
    for li in range(len(levels)):
        xa, xb = a[3].slots[0].sample_out[li], b[3].slots[0].sample_out[li]
        assert rel_err(xb.cpu().numpy(), xa.cpu().numpy()) <= 1e-5
