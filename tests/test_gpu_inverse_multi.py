"""finc_inverse_chain_multi_f32 (the sampling chains of several levels in one launch) against the per-level
finc_inverse_chain_f32 launches it replaces, and HotPathRunner(multi_level_inverse=True) against the per-level path."""
import pytest
import torch

pytestmark = pytest.mark.gpu

CIFAR = [(12, 16, 16), (24, 8, 8), (48, 4, 4)]   # cifar10_levels at k = 3: C = 4*Cq, H, W


def _level(B, C, H, W, U, seed):
    from fincflow_b200 import _native
    from fincflow_b200.fastflow import FastFlowUnit

    torch.manual_seed(seed)
    w = torch.stack([FastFlowUnit(C, C, (3, 3)).weight.detach() for _ in range(U)]).cuda().contiguous()
    nb = _native.prepared_weights_bytes(_native.PREP_INVERSE, B, 4, C // 4, H, W, 3, 3)
    assert nb > 0
    tables = torch.empty((U, nb), dtype=torch.uint8, device="cuda")
    _native.prepare_weights(w, tables, _native.PREP_INVERSE, B, H, W)
    return torch.randn(B, C, H, W, device="cuda"), tables


def _check_against_per_level(levels):
    from fincflow_b200 import _native

    outs = _native.inverse_chain_multi([(z, t, (3, 3), units, torch.full_like(z, float("nan")))
                                        for z, t, units in levels])
    for (z, t, units), x in zip(levels, outs):
        assert torch.equal(x, _native.inverse_chain(z, t, (3, 3), units))


@pytest.mark.parametrize("B", [256, 37, 5, 1])
def test_cifar_levels_match_per_level_chains(B):
    U = 16
    levels = []
    for i, (C, H, W) in enumerate(CIFAR):
        z, t = _level(B, C, H, W, U, B + i)
        levels.append((z, t, range(U - 1, -1, -1)))
    _check_against_per_level(levels)


@pytest.mark.parametrize("li", range(3))
def test_one_level_alone(li):
    C, H, W = CIFAR[li]
    z, t = _level(256, C, H, W, 16, li)
    _check_against_per_level([(z, t, range(15, -1, -1))])


def test_sub_chains_and_mixed_batches():
    """two-unit sub-chains (range(1, -1, -1)), another level order, and levels of different batch sizes"""
    levels = []
    for i, ((C, H, W), B) in enumerate(zip(reversed(CIFAR), (64, 256, 7))):
        z, t = _level(B, C, H, W, 4, 100 + i)
        levels.append((z, t, range(1, -1, -1)))
    _check_against_per_level(levels)


def test_unsupported_mixes_raise():
    from fincflow_b200 import _native

    z0, t0 = _level(256, 12, 16, 16, 16, 0)
    z24, t24 = _level(16, 96, 4, 4, 2, 1)               # C = 24 per group: no register-window kernel
    with pytest.raises(_native.FincNativeError):
        _native.inverse_chain_multi([(z0, t0, (3, 3), range(15, -1, -1), None), (z24, t24, (3, 3), range(2), None)])
    z48, t48 = _level(256, 48, 4, 4, 48, 2)             # 48 units of 5.3 KB tables per group: too large
    with pytest.raises(_native.FincNativeError):
        _native.inverse_chain_multi([(z0, t0, (3, 3), range(15, -1, -1), None), (z48, t48, (3, 3), range(47, -1, -1), None)])
    with pytest.raises(_native.FincNativeError):
        _native.inverse_chain_multi([])


def _run(B, n_steps, **kw):
    from fincflow_b200.stack import FincStack, HotPathRunner, cifar10_levels

    torch.manual_seed(0)
    stack = FincStack(cifar10_levels(16, 3)).cuda()
    r = HotPathRunner(stack, B, torch.device("cuda"), slots=1, lr=1e-2, **kw)
    g = torch.Generator(device="cuda").manual_seed(5)
    for li in range(3):
        r.slots[0].acts[li][0].normal_(generator=g)
        r.slots[0].zin[li].normal_(generator=g)
    r.prepare()
    samples = []
    for _ in range(n_steps):   # Adam and the table refresh between the sampling passes
        r.step(0)
        if kw.get("overlap_sampling"):
            r.drain()
        samples.append([r.slots[0].sample_out[li].clone() for li in range(3)])
    torch.cuda.synchronize()
    return stack.flat.detach().clone(), samples, r


@pytest.mark.parametrize("kw", [dict(), dict(use_graphs=False), dict(level_parallel=True),
                                dict(overlap_sampling=True, level_parallel=True)])
def test_runner_multi_level_inverse_is_bit_identical(kw):
    ref = _run(64, 3, multi_level_inverse=False, **kw)
    got = _run(64, 3, multi_level_inverse=True, **kw)
    assert not ref[2].inv_multi and got[2].inv_multi
    assert got[2].launches_per_step == ref[2].launches_per_step - 2
    assert torch.equal(got[0], ref[0])
    for a, b in zip(got[1], ref[1]):
        assert all(torch.equal(x, y) for x, y in zip(a, b))


def test_runner_device_latents_multi_level_inverse():
    """device_latents: the latents are drawn before the single launch, in the order of the per-level path"""
    outs = []
    for multi in (False, True):
        outs.append(_run(32, 2, multi_level_inverse=multi, device_latents=True))
    assert outs[1][2].inv_multi
    for a, b in zip(outs[0][1], outs[1][1]):
        assert all(torch.equal(x, y) for x, y in zip(a, b))
