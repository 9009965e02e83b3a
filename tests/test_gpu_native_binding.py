"""The host side of the C ABI binding (fincflow_b200/_native.py).

Rejection: every wrapper that takes an output, a workspace or a prepared table refuses a wrong one with
FincNativeError before it calls the library.  These cases run with the library replaced by a recording stub: only the
host-only size queries (finc_*_bytes) reach the real library, and no other call may be recorded.  So a check that
regresses fails the test without handing a kernel a bad buffer.

Launch counts: for every wrapper and each argument combination that changes the count, the number of library kernels
torch.profiler sees equals the increase of `_native.launch_count` (bench.py's gpu_launches, HotPathRunner's
launches_per_step).  allreduce_adam_ is left out: its kernel spin-waits on peer ranks (tests/multirank_check.py).
"""
import pytest
import torch

from test_gpu_glue_variants import GLUE_FAMILIES
from test_gpu_kernel_variants import FAMILIES, kernels_in
from test_gpu_tc_variants import TC_FAMILIES

pytestmark = pytest.mark.gpu

LIBRARY_FAMILIES = {**{"finc_" + k: v for k, v in FAMILIES.items()}, **{"tc_" + k: v for k, v in TC_FAMILIES.items()},
                    **GLUE_FAMILIES}
B, G, C, H, W, K = 2, 4, 3, 8, 8, 3          # a FastFlowUnit of 12 channels on 8x8 images
CT = G * C


def nat():
    from fincflow_b200 import _native

    _native.load()
    return _native


def unit_weight(seed=0, ch=CT, k=K):
    from fincflow_b200.fastflow import FastFlowUnit

    torch.manual_seed(seed)
    return FastFlowUnit(ch, ch, (k, k)).weight.detach().cuda().contiguous()


def tables(kind, n=1, c=C, h=H, w=W, k=K, b=B):
    """prepared tables [n, bytes] of `kind` for a unit of 4 groups of `c` channels"""
    n_ = nat()
    nb = n_.prepared_weights_bytes(kind, b, G, c, h, w, k, k)
    assert nb > 0
    t = torch.empty((n, nb), dtype=torch.uint8, device="cuda")
    n_.prepare_weights(torch.stack([unit_weight(u, G * c, k) for u in range(n)]), t, kind, b, h, w)
    return t


# ---- rejection, with the library replaced by a recording stub -----------------------------------------------------
class _Recorder:
    def __init__(self, lib):
        self.lib, self.calls = lib, []

    def __getattr__(self, name):
        if name.endswith("_bytes"):
            return getattr(self.lib, name)

        def record(*args):
            self.calls.append(name)
            return 0
        return record


def bad_outputs(shape, dtype=torch.float32):
    """tensors a call writing a contiguous `shape` of `dtype` must refuse"""
    wrong = torch.float64 if dtype == torch.float32 else torch.float32
    bigger = list(shape[:-1]) + [2 * shape[-1]]
    return {"shape": torch.empty(list(shape[:-1]) + [shape[-1] + 1], dtype=dtype, device="cuda"),
            "dtype": torch.empty(shape, dtype=wrong, device="cuda"),
            "cpu": torch.empty(shape, dtype=dtype),
            "strided": torch.empty(bigger, dtype=dtype, device="cuda")[..., ::2]}


def bad_buffers(nbytes):
    """uint8 workspaces / tables a call needing `nbytes` must refuse"""
    return {"short": torch.empty(nbytes - 1, dtype=torch.uint8, device="cuda"),
            "dtype": torch.empty(nbytes, dtype=torch.float32, device="cuda"),
            "cpu": torch.empty(nbytes, dtype=torch.uint8),
            "strided": torch.empty(2 * nbytes, dtype=torch.uint8, device="cuda")[::2]}


def bad_tables(kind, n=1):
    """tables a FInC call of kind `kind` on [B, CT, H, W] (unit rows 0 .. n-1) must refuse"""
    n_ = nat()
    good = tables(kind, n)
    other = n_.PREP_FORWARD if kind == n_.PREP_INVERSE else n_.PREP_INVERSE
    small_kind = tables(other, n) if n_.prepared_weights_bytes(other, B, G, C, H, W, K, K) < good.shape[1] else None
    cases = {"row_short": good[:, :-16].contiguous(),
             "other_shape": tables(kind, n, c=2),                   # 4 groups of 2 channels: a smaller table
             "misaligned": torch.empty(good.numel() + 16, dtype=torch.uint8, device="cuda")[8:8 + good.numel()].view(
                 good.shape),
             "cpu": good.cpu(),
             "dtype": torch.empty(good.shape, dtype=torch.float32, device="cuda")}
    if small_kind is not None:
        cases["other_kind"] = small_kind
    if n > 1:
        cases["rows_short"] = good[:n - 1]
    return cases


def _rejections():
    """(id, call) of every bad output, workspace and table of every wrapper that takes one"""
    import fincflow_b200.compat as compat

    n_ = nat()
    x = torch.randn(B, CT, H, W, device="cuda")
    w = unit_weight()
    cases = []

    def add(what, bad, fn):
        cases.extend((f"{what}-{k}", lambda t=t: fn(t)) for k, t in bad.items())

    # the FInC convolution and its inverse
    add("forward.out", bad_outputs(x.shape), lambda t: n_.forward(x, w, out=t))
    add("forward.logdet_out", bad_outputs((B,)), lambda t: n_.forward(x, w, logdet_out=t))
    add("backward_input.out", bad_outputs(x.shape), lambda t: n_.backward_input(x, w, out=t))
    add("backward_weight.out", bad_outputs(w.shape), lambda t: n_.backward_weight(x, x, (K, K), out=t))
    ws_need = n_.backward_weight_workspace_bytes(B, G, C, H, W, K, K)
    add("backward_weight.workspace", bad_buffers(ws_need), lambda t: n_.backward_weight(x, x, (K, K), workspace=t))
    add("inverse.out", bad_outputs(x.shape), lambda t: n_.inverse(x, w, out=t))
    add("inverse_adjoint.out", bad_outputs(x.shape), lambda t: n_.inverse_adjoint(x, w, out=t))
    add("apply_grad_mask_.dw", {k: v for k, v in bad_outputs(w.shape).items() if k != "shape"},
        lambda t: n_.apply_grad_mask_(t, G, n_.ORDERS_UNIT))
    add("apply_grad_mask_.dw", {"groups": torch.empty((CT - C,) + tuple(w.shape[1:]), device="cuda")},
        lambda t: n_.apply_grad_mask_(t, G, n_.ORDERS_UNIT))
    for fn, kind in ((n_.forward, n_.PREP_FORWARD), (n_.backward_input, n_.PREP_BACKWARD_INPUT),
                     (n_.inverse, n_.PREP_INVERSE)):
        add(f"{fn.__name__}.prepared", {k: t[0] for k, t in bad_tables(kind).items()},
            lambda t, fn=fn: fn(x, None, prepared=t, ksize=(K, K)))
    add("prepare_weights.tables", bad_tables(n_.PREP_INVERSE, 2),
        lambda t: n_.prepare_weights(torch.stack([w, w]), t, n_.PREP_INVERSE, B, H, W))
    add("compat.level2.output", bad_outputs(x.shape), lambda t: compat.cinc_cuda_level2.inverse(x, w, t))
    add("compat.level1.output", bad_outputs((B, C, H, W)),
        lambda t: compat.cinc_cuda_level1.inverse(x[:, :C].contiguous(), w[:C], t))
    # chains
    U = 2
    wu = torch.stack([w, unit_weight(1)])
    add("chain.out", bad_outputs(x.shape), lambda t: n_.chain(x, wu, t))
    add("chain.out5", {k: v for k, v in bad_outputs((U, B, CT, H, W)).items() if k != "strided"},
        lambda t: n_.chain(x, wu, t))
    add("chain.out5", {"unit_strided": torch.empty(U, B, CT, H, 2 * W, device="cuda")[..., ::2]},
        lambda t: n_.chain(x, wu, t))
    add("chain.logdet_out", bad_outputs((B,)), lambda t: n_.chain(x, wu, torch.empty_like(x), logdet_out=t))
    xs = torch.randn(U, B, CT, H, W, device="cuda")
    bw = torch.empty(U, CT, C, K, K, device="cuda")
    add("backward_weight_batched.out_units", {k: v for k, v in bad_outputs(bw.shape).items() if k != "strided"},
        lambda t: n_.backward_weight_batched(xs, xs, t, (K, K)))
    add("backward_weight_batched.out_units", {"unit_strided": torch.empty(U, CT, C, K, 2 * K, device="cuda")[..., ::2]},
        lambda t: n_.backward_weight_batched(xs, xs, t, (K, K)))
    add("backward_weight_batched.dz_units", {"cpu": xs.cpu(), "dtype": xs.double(), "shape": xs[:, :, :C]},
        lambda t: n_.backward_weight_batched(t, xs, bw, (K, K)))
    bnb = n_.backward_weight_batched_workspace_bytes(B, G, C, H, W, K, K, U)
    add("backward_weight_batched.workspace", bad_buffers(bnb),
        lambda t: n_.backward_weight_batched(xs, xs, bw, (K, K), workspace=t))
    good = tables(n_.PREP_INVERSE, 2)
    add("inverse_chain.out", bad_outputs(x.shape), lambda t: n_.inverse_chain(x, good, (K, K), range(1, -1, -1), out=t))
    add("inverse_chain.tables", bad_tables(n_.PREP_INVERSE, 2),
        lambda t: n_.inverse_chain(x, t, (K, K), range(1, -1, -1)))
    add("inverse_chain_multi.out", bad_outputs(x.shape),
        lambda t: n_.inverse_chain_multi([(x, good, (K, K), range(2), None), (x, good, (K, K), range(2), t)]))
    add("inverse_chain_multi.tables", bad_tables(n_.PREP_INVERSE, 2),
        lambda t: n_.inverse_chain_multi([(x, good, (K, K), range(2), None), (x, t, (K, K), range(2), None)]))
    # glue
    add("gaussian_logp.logp_out", bad_outputs((B,)), lambda t: n_.gaussian_logp(x, logp_out=t))
    add("gaussian_logp.dz_out", bad_outputs(x.shape), lambda t: n_.gaussian_logp(x, dz_scale=0.5, dz_out=t))
    add("squeeze.out", bad_outputs((B, 4 * CT, H // 2, W // 2)), lambda t: n_.squeeze(x, out=t))
    add("unsqueeze.out", bad_outputs((B, CT // 4, 2 * H, 2 * W)), lambda t: n_.unsqueeze(x, out=t))
    A = torch.randn(CT, CT, device="cuda")
    add("affine1x1.out", bad_outputs(x.shape), lambda t: n_.affine1x1(x, A, out=t))
    # tensor-core path
    xn = torch.randn(B, H, W, 32, device="cuda")
    wp = torch.empty(n_.load().finc_tc_conv_weights_bytes(32, 32, 1, 0) // 4, device="cuda")
    bias = torch.zeros(32, device="cuda")
    add("tc_conv_nhwc.out", bad_outputs((B, H, W, 32)), lambda t: n_.tc_conv_nhwc(xn, wp, bias, 32, 1, out=t))
    P = torch.randn(256, 64, device="cuda")
    add("tc_wgrad.out", {k: v for k, v in bad_outputs((64, 64)).items() if k != "strided"},
        lambda t: n_.tc_wgrad(P, P, out=t))
    add("tc_wgrad.out", {"column_strided": torch.empty(64, 128, device="cuda")[:, ::2]}, lambda t: n_.tc_wgrad(P, P, out=t))
    Cc, width = 12, 128
    xc = torch.randn(B, Cc, H, W, device="cuda")
    blob = torch.empty(n_.coupling_prepared_bytes(Cc, width, True), dtype=torch.uint8, device="cuda")
    cws = n_.coupling_workspace_bytes(B, Cc, H, W, width)
    add("coupling_apply.out", bad_outputs(xc.shape), lambda t: n_.coupling_apply(xc, blob, width, out=t))
    add("coupling_apply.logdet_out", bad_outputs((B,)), lambda t: n_.coupling_apply(xc, blob, width, logdet_out=t))
    add("coupling_apply.workspace", bad_buffers(cws), lambda t: n_.coupling_apply(xc, blob, width, workspace=t))
    add("coupling_backward.fwd_workspace", bad_buffers(cws),
        lambda t: n_.coupling_backward(xc, xc, None, blob, t, width))
    zd = torch.randn(B, 16, 4, 4, device="cuda")
    dnb = n_.inverse_dense_bytes(G, 4, 4, 4)
    w16 = unit_weight(0, 16)
    add("inverse_dense_prepare.out", bad_buffers(dnb), lambda t: n_.inverse_dense_prepare(w16, 4, 4, out=t))
    dblob = torch.empty(dnb, dtype=torch.uint8, device="cuda")
    add("inverse_dense.out", bad_outputs(zd.shape), lambda t: n_.inverse_dense(zd, dblob, out=t))
    add("inverse_dense.blob", bad_buffers(dnb), lambda t: n_.inverse_dense(zd, t))
    return cases


def test_bad_buffers_are_refused_before_the_library_is_called(monkeypatch):
    n_ = nat()
    cases = _rejections()   # (building the valid tables runs kernels: before the stub goes in)
    rec = _Recorder(n_.load())
    monkeypatch.setattr(n_, "_lib", rec)
    accepted = []
    for what, call in cases:
        try:
            call()
            accepted.append(what)
        except n_.FincNativeError:
            pass
        except Exception as e:   # refused, but not by the binding's checks
            accepted.append(f"{what} ({type(e).__name__})")
    assert not accepted, f"not refused with FincNativeError: {accepted}"
    assert not rec.calls, f"library calls despite a bad buffer: {rec.calls}"
    print(f"\n[binding] {len(cases)} bad buffers refused on the host")


def test_stub_records_a_valid_call(monkeypatch):
    """the recorder sees the calls a valid buffer leads to (so an empty record above means something)"""
    n_ = nat()
    x = torch.randn(B, CT, H, W, device="cuda")
    w = unit_weight()
    t = tables(n_.PREP_INVERSE)
    rec = _Recorder(n_.load())
    monkeypatch.setattr(n_, "_lib", rec)
    n_.forward(x, w, out=torch.empty_like(x))
    n_.inverse(x, None, prepared=t[0], ksize=(K, K))
    assert rec.calls == ["finc_forward_f32", "finc_inverse_f32"]


# ---- launch counts ------------------------------------------------------------------------------------------------
def library_launches(fn):
    """(kernels of the library that ran in fn(), the increase of _native.launch_count)"""
    from torch.profiler import ProfilerActivity, profile

    n_ = nat()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        torch.zeros(1, device="cuda").add_(1)   # (see test_gpu_kernel_variants.launched)
        torch.cuda.synchronize()
        c0 = n_.launch_count
        fn()
        torch.cuda.synchronize()
        counted = n_.launch_count - c0
    ran = sum(e.count for e in prof.key_averages()
              if e.device_type == torch.autograd.DeviceType.CUDA and kernels_in([e.key], LIBRARY_FAMILIES))
    return ran, counted


def _recipes():
    n_ = nat()
    x = torch.randn(B, CT, H, W, device="cuda")
    x0 = x[:0]
    w = unit_weight()
    ld = torch.zeros(B, device="cuda")
    r = {
        "forward": lambda: n_.forward(x, w),
        "forward.no_logdet": lambda: n_.forward(x, w, want_logdet=False),
        "forward.naive": lambda: n_.forward(x, w, flags=n_.FLAG_NAIVE),
        "forward.naive_no_logdet": lambda: n_.forward(x, w, want_logdet=False, flags=n_.FLAG_NAIVE),
        "forward.logdet_out": lambda: n_.forward(x, w, logdet_out=ld, flags=n_.FLAG_LOGDET_ACCUMULATE),
        "forward.prepared": lambda t=tables(n_.PREP_FORWARD): n_.forward(x, None, prepared=t[0], ksize=(K, K)),
        "forward.B0": lambda: n_.forward(x0, w),
        "backward_input": lambda: n_.backward_input(x, w),
        "backward_input.naive": lambda: n_.backward_input(x, w, flags=n_.FLAG_NAIVE),
        "backward_input.prepared": lambda t=tables(n_.PREP_BACKWARD_INPUT): n_.backward_input(
            x, None, prepared=t[0], ksize=(K, K)),
        "backward_weight": lambda: n_.backward_weight(x, x, (K, K)),
        "backward_weight.workspace": lambda ws=n_.new_workspace(n_.backward_weight_workspace_bytes(
            B, G, C, H, W, K, K), "cuda"): n_.backward_weight(x, x, (K, K), workspace=ws),
        "backward_weight.naive": lambda: n_.backward_weight(x, x, (K, K), flags=n_.FLAG_NAIVE),
        "backward_weight.B0": lambda: n_.backward_weight(x0, x0, (K, K)),
        "inverse": lambda: n_.inverse(x, w),
        "inverse.naive": lambda: n_.inverse(x, w, flags=n_.FLAG_NAIVE),
        "inverse.generic_tiled": lambda: n_.inverse(x, w, flags=n_.FLAG_GENERIC_TILED),
        "inverse.prepared": lambda t=tables(n_.PREP_INVERSE): n_.inverse(x, None, prepared=t[0], ksize=(K, K)),
        "inverse.B0": lambda: n_.inverse(x0, w),
        "inverse_adjoint": lambda: n_.inverse_adjoint(x, w),
        "apply_grad_mask_": lambda: n_.apply_grad_mask_(w.clone(), G, n_.ORDERS_UNIT),
        "logdet": lambda: n_.logdet(w, B, H, W),
        "gaussian_logp": lambda: n_.gaussian_logp(x, ld),
        "gaussian_logp.dz": lambda: n_.gaussian_logp(x, None, dz_scale=0.5),
        "prepare_weights": lambda: tables(n_.PREP_FORWARD, 2),
        "adam_step_": lambda p=torch.zeros(1000, device="cuda"), s=torch.zeros(1, device="cuda"): n_.adam_step_(
            p, torch.ones_like(p), torch.zeros_like(p), torch.zeros_like(p), s),
        "squeeze": lambda: n_.squeeze(x),
        "unsqueeze": lambda: n_.unsqueeze(x),
        "affine1x1": lambda: n_.affine1x1(x, torch.eye(CT, device="cuda"), torch.zeros(CT, device="cuda")),
        "affine1x1_backward_weight.tiled": lambda x16=torch.randn(B, 16, 8, 8, device="cuda"):
            n_.affine1x1_backward_weight(x16, x16),
        "affine1x1_backward_weight.generic": lambda x6=torch.randn(B, 6, 8, 8, device="cuda"):
            n_.affine1x1_backward_weight(x6, x6),
        "affine1x1_backward_weight.B0": lambda: n_.affine1x1_backward_weight(x0, x0),
        "slogdet_inverse": lambda: n_.slogdet_inverse(torch.eye(CT, device="cuda").expand(3, CT, CT).contiguous()),
        "preprocess": lambda: n_.preprocess(torch.full((B, 3, 8, 8), 100.0, device="cuda")),
        "preprocess.reverse": lambda: n_.preprocess(x, reverse=True),
    }
    # tensor-core path
    Cc, width = 12, 128
    torch.manual_seed(1)
    ps = [torch.randn(width, Cc // 2, 3, 3), torch.randn(width), torch.randn(width, width, 1, 1), torch.randn(width),
          torch.zeros(Cc, width, 3, 3), torch.zeros(Cc), torch.zeros(Cc)]
    ps = [0.05 * p.cuda() for p in ps]
    blob = n_.coupling_prepare(*ps, with_backward=True)
    xc = torch.randn(B, Cc, H, W, device="cuda")
    fws = torch.empty(n_.coupling_workspace_bytes(B, Cc, H, W, width), dtype=torch.uint8, device="cuda")
    n_.coupling_apply(xc, blob, width, workspace=fws)
    xn = torch.randn(B, H, W, 32, device="cuda")
    wp = n_.tc_conv_prepare_weights(torch.randn(32, 32, 1, 1, device="cuda"))
    zd = torch.randn(B, 16, 4, 4, device="cuda")
    w16 = unit_weight(0, 16)
    dblob = n_.inverse_dense_prepare(w16, 4, 4)
    r.update({
        "tc_conv_prepare_weights": lambda: n_.tc_conv_prepare_weights(torch.randn(32, 32, 1, 1, device="cuda")),
        "tc_conv_nhwc": lambda: n_.tc_conv_nhwc(xn, wp, torch.zeros(32, device="cuda"), 32, 1),
        "tc_wgrad": lambda: n_.tc_wgrad(xn.view(-1, 32), torch.randn(B * H * W, 64, device="cuda")),
        "coupling_prepare": lambda: n_.coupling_prepare(*ps),
        "coupling_prepare.with_backward": lambda: n_.coupling_prepare(*ps, with_backward=True),
        "coupling_apply": lambda: n_.coupling_apply(xc, blob, width),
        "coupling_apply.reverse": lambda: n_.coupling_apply(xc, blob, width, reverse=True),
        "coupling_apply.reverse_logdet": lambda: n_.coupling_apply(xc, blob, width, reverse=True, want_logdet=True),
        "coupling_apply.no_logdet": lambda: n_.coupling_apply(xc, blob, width, want_logdet=False),
        "coupling_backward": lambda: n_.coupling_backward(xc, torch.randn_like(xc), torch.ones(B, device="cuda"), blob,
                                                          fws, width),
        "coupling_backward.reverse": lambda: n_.coupling_backward(xc, torch.randn_like(xc), None, blob, fws, width,
                                                                  flags=n_.FLAG_COUPLING_REVERSE),
        "inverse_dense_prepare": lambda: n_.inverse_dense_prepare(w16, 4, 4),
        "inverse_dense": lambda: n_.inverse_dense(zd, dblob),
    })
    # chains (the inverse chains on the levels of test_gpu_inverse_multi, which the register-window kernel covers)
    from test_gpu_inverse_multi import CIFAR, _level

    U = 3
    wu = torch.stack([unit_weight(u) for u in range(U)])
    xs = torch.randn(U, B, CT, H, W, device="cuda")
    levels = [_level(8, *shape, 2, i) for i, shape in enumerate(CIFAR)]
    r.update({
        "chain": lambda: n_.chain(x, wu, torch.empty(U, B, CT, H, W, device="cuda")),
        "chain.last": lambda: n_.chain(x, wu, torch.empty_like(x), logdet_out=torch.zeros(B, device="cuda")),
        "chain.transpose": lambda: n_.chain(x, wu, torch.empty(U, B, CT, H, W, device="cuda"), units=range(U - 1, 0, -1),
                                            transpose=True),
        "backward_weight_batched": lambda: n_.backward_weight_batched(xs, xs, torch.empty(U, CT, C, K, K, device="cuda"),
                                                                      (K, K)),
        "inverse_chain": lambda: n_.inverse_chain(*levels[0], (3, 3), range(1, -1, -1)),
        "inverse_chain_multi": lambda: n_.inverse_chain_multi([(z, t, (3, 3), range(1, -1, -1), None) for z, t in levels]),
    })
    return r


def test_launch_count_matches_the_kernels_that_ran():
    recipes = _recipes()
    wrong = {}
    for name, fn in recipes.items():
        fn()   # warm: module loads, kernel attributes
        ran, counted = library_launches(fn)
        if ran != counted:
            wrong[name] = (ran, counted)
    assert not wrong, f"(kernels that ran, launch_count increase): {wrong}"
    n_ = nat()
    covered = {name.split(".")[0] for name in recipes}
    public = {k for k, v in vars(n_).items() if callable(v) and getattr(v, "__module__", "") == n_.__name__
              and not k.startswith("_") and not isinstance(v, type)}
    queries = {k for k in public if k.endswith("_bytes")} | {"load", "pack_orders", "chain_supported", "sm_count",
                                                            "new_workspace", "allreduce_adam_"}
    assert public - queries - covered == set()
