"""GPU tests of the fused qkv + window-attention forward (csrc/winattn_tc_qkv_fwd.cuh, torch.ops.mmn_b200.winattn_qkv_fwd).

Its exact reference is the unfused path on the same bf16 inputs: the tensor-core projection (linear_fwd, same K = 96
fp32 accumulation, fp32 bias, one bf16 rounding) followed by winattn_fwd.  The module tests compare against the fp64
oracle at the tolerances of test_gpu_parity.py.
"""
import math

import pytest
import torch

from oracle import ref_nd as R

pytestmark = pytest.mark.gpu

BF16_TOL = 2e-2


@pytest.fixture(scope="module")
def mm():
    from multimodal_neuroimage_b200 import _lib, ops  # noqa: F401
    from multimodal_neuroimage_b200.modules import swin_v2_module as v2
    from multimodal_neuroimage_b200.modules import swinfusion_module as fu
    _lib.load()

    class NS:
        pass
    ns = NS()
    ns.lib, ns.ops, ns.v2, ns.fu = _lib, ops, v2, fu
    return ns


def rel_err(got, want):
    got, want = got.detach().double().cpu(), want.detach().double().cpu()
    return float((got - want).abs().max() / want.abs().max().clamp_min(1e-30))


GEOS = {  # batch, grid, window, shift
    "cfg2_b1": (1, (32, 32, 32), (4, 4, 4), (2, 2, 2)),
    "cfg2_b3": (3, (32, 32, 32), (4, 4, 4), (2, 2, 2)),
    "all_classes_odd_counts": (1, (16, 16, 16), (4, 4, 4), (2, 2, 2)),   # 27, 9, 9, 9, 3, 3, 3, 1 windows per class
    "shift0": (2, (8, 8, 12), (4, 4, 4), (0, 0, 0)),
    "2d": (2, (16, 16), (8, 8), (4, 4)),
}
VARIANTS = ["cosine_qv_bias", "scaled_full_bias", "scaled_no_bias"]


def _inputs(mm, geo, variant, seed=0):
    B, grid, window, shift = GEOS[geo]
    C, nH = 96, 3
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(B, *grid, C, generator=g, device="cuda").bfloat16()
    w = (torch.randn(3 * C, C, generator=g, device="cuda") * C ** -0.5).bfloat16()
    if variant == "cosine_qv_bias":        # SwinV2: cat(q_bias, 0, v_bias)
        b = torch.randn(3 * C, generator=g, device="cuda") * 0.3
        b[C:2 * C] = 0
    elif variant == "scaled_full_bias":    # SwinFusion: nn.Linear bias
        b = torch.randn(3 * C, generator=g, device="cuda") * 0.3
    else:
        b = None
    cos = variant.startswith("cosine")
    bias = torch.randn(nH, 64, 64, generator=g, device="cuda")
    hs = torch.rand(nH, generator=g, device="cuda") * 10 + 1 if cos else None
    score = mm.lib.SCORE_COSINE if cos else mm.lib.SCORE_SCALED
    mk = mm.lib.MASK_SHIFT if any(shift) else mm.lib.MASK_NONE
    geo_args = (list(grid), list(window), list(shift), nH, score, mk, 1.0 if cos else 32 ** -0.5)
    return x, w, b, bias, hs, geo_args


def _unfused(mm, x, w, b, bias, hs, geo_args):
    a = torch.ops.mmn_b200.linear_fwd(x.view(-1, x.shape[-1]), w, b, mm.lib.ACT_NONE, False)[0].view(*x.shape[:-1], -1)
    out, lse = torch.ops.mmn_b200.winattn_fwd(a, None, bias, hs, None, *geo_args, 0.0, 0, 0, mm.lib.PATH_AUTO)
    return a, out, lse


def _fused(x, w, b, bias, hs, geo_args, path=0):
    return torch.ops.mmn_b200.winattn_qkv_fwd(x, w, b, bias, hs, None, *geo_args, path)


def _ulps(a, b):
    """bf16 ulp distance of two same-sign-or-zero tensors (bit patterns as integers)"""
    ia, ib = a.view(torch.int16).int(), b.view(torch.int16).int()
    return (ia - ib).abs()


@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("geo", list(GEOS))
def test_fused_equals_unfused(mm, geo, variant):
    x, w, b, bias, hs, geo_args = _inputs(mm, geo, variant)
    assert mm.ops.winattn_qkv_path_name(tuple(x.shape), x.dtype, *geo_args[:6]) == "tcgen05-fused"
    a, out_u, lse_u = _unfused(mm, x, w, b, bias, hs, geo_args)
    qkv, out, lse = _fused(x, w, b, bias, hs, geo_args)
    torch.cuda.synchronize()
    # qkv: the same K = 96 tcgen05 accumulation and fp32 bias as linear_fwd, rounded once
    assert qkv.shape == a.shape
    assert int(_ulps(qkv, a).max()) <= 1, f"qkv differs by {int(_ulps(qkv, a).max())} bf16 ulp"
    # out / lse against winattn_fwd on the fused kernel's own qkv
    out_r, lse_r = torch.ops.mmn_b200.winattn_fwd(qkv, None, bias, hs, None, *geo_args, 0.0, 0, 0, mm.lib.PATH_AUTO)
    tol = out_r.float().abs() * 2 ** -8 + 1e-6
    assert bool(((out.float() - out_r.float()).abs() <= tol).all()), f"out max diff {float((out.float() - out_r.float()).abs().max())}"
    nWB = lse.shape[1]
    assert torch.allclose(lse[0], lse_r[0], rtol=1e-5, atol=1e-5)
    rec, rec_r = lse[1:].reshape(nWB, 3, 3, 64), lse_r[1:].reshape(nWB, 3, 3, 64)
    k = slice(0, 3) if variant.startswith("cosine") else slice(2, 3)       # 1/|q|, 1/|k| only for cosine
    assert torch.allclose(rec[:, :, k], rec_r[:, :, k], rtol=1e-5, atol=1e-6)
    # and, transitively, against the unfused output (identical qkv makes this exact too)
    if torch.equal(qkv, a):
        assert torch.equal(out, out_u)
    assert rel_err(out, out_u) < 1e-2


def _sd64_grad(module):
    names = {n for n, _ in module.named_parameters()}
    sd = {}
    for k, v in module.state_dict().items():
        t = (v.detach().double() if v.is_floating_point() else v.detach()).cpu()
        if k in names:
            t.requires_grad_(True)
        sd[k] = t
    return sd


def _randomise(module, seed):
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for name, p in module.named_parameters():
            if "norm" in name and name.endswith("weight"):
                p.copy_(torch.empty(p.shape).uniform_(0.5, 1.5, generator=g))
            elif name.endswith("relative_position_bias_table"):
                p.copy_(torch.empty(p.shape).normal_(0, 1.0, generator=g))
            elif name.endswith("bias"):
                p.copy_(torch.empty(p.shape).normal_(0, 0.3, generator=g))


class _Spy:
    """counts the C calls of the window-attention forward paths; `qkv_linear` = linear_fwd calls with 3C outputs"""

    def __init__(self, mm, monkeypatch):
        lib = mm.lib.load()
        self.calls = {"mmn_winattn_qkv_fwd": 0, "mmn_winattn_fwd": 0, "qkv_linear": 0}
        for name in ("mmn_winattn_qkv_fwd", "mmn_winattn_fwd", "mmn_linear_fwd"):
            real = getattr(lib, name)

            def f(*a, _name=name, _real=real):
                if _name == "mmn_linear_fwd":
                    if a[9] == 3 * a[8]:
                        self.calls["qkv_linear"] += 1
                else:
                    self.calls[_name] += 1
                return _real(*a)
            monkeypatch.setattr(lib, name, f)


def _v2_block(mm, C=96, nH=3, attn_drop=0.0):
    blk = mm.v2.SwinTransformerBlock(C, (8, 8, 8), nH, window_size=4, shift_size=2, attn_drop=attn_drop)
    _randomise(blk, 11)
    with torch.no_grad():   # trained SwinV2 logit scales (see test_gpu_parity.test_swinv2_block_3d)
        blk.attn.logit_scale.copy_(torch.linspace(0.0, math.log(20.0), nH).view(nH, 1, 1))
    return blk


@pytest.mark.parametrize("kind", ["swinv2_cosine", "swinfusion_scaled"])
def test_module_against_fp64_oracle(mm, kind, monkeypatch):
    """The block on the fused path against the same block on the two-kernel path (its exact reference: the same bf16 qkv,
    so only sums done with float atomics may differ) and against the fp64 oracle.  Every input is seeded here, so the
    check does not depend on which tests ran before.  A bf16 module's gradients of parameters that enter through a long
    cancelling sum (the cosine logit scale: up to 4 % of fp64 on either path, from the bf16 rounding of x, W and q/k) are
    held to the two-kernel path's own fp64 error where that exceeds the parity tolerance."""
    grid, C, nH, B = (8, 8, 8), 96, 3, 2
    torch.manual_seed(0)
    if kind == "swinv2_cosine":
        blk = _v2_block(mm)
        ref = lambda x, p: R.swin_v2_block(x, p, grid, 4, 2, nH)
    else:
        blk = mm.fu.SwinTransformerBlock_fusion(C, grid, nH, window_size=4, shift_size=2)
        _randomise(blk, 12)
        ref = lambda x, p: R.fusion_block(x, p, grid, grid, 4, 2, nH)
    x = torch.randn(B, math.prod(grid), C, generator=torch.Generator().manual_seed(5))
    sd = _sd64_grad(blk)
    xo = x.double().requires_grad_(True)
    want = ref(xo, sd)
    cot = torch.randn(want.shape, generator=torch.Generator().manual_seed(6))
    pnames = [n for n, _ in blk.named_parameters()]
    gw = torch.autograd.grad((want * cot.double()).sum(), [xo] + [sd[n] for n in pnames], allow_unused=True)
    blk = blk.cuda()
    spy = _Spy(mm, monkeypatch)
    real_path = mm.ops.winattn_qkv_path_name

    def run(fused_path):
        monkeypatch.setattr(mm.ops, "winattn_qkv_path_name", real_path if fused_path else (lambda *a, **k: "off"))
        before = dict(spy.calls)
        xc = x.cuda().requires_grad_(True)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            got = blk(xc, grid) if kind == "swinfusion_scaled" else blk(xc)
        calls = {k: spy.calls[k] - before[k] for k in spy.calls}
        assert calls == ({"mmn_winattn_qkv_fwd": 1, "mmn_winattn_fwd": 0, "qkv_linear": 0} if fused_path else
                         {"mmn_winattn_qkv_fwd": 0, "mmn_winattn_fwd": 1, "qkv_linear": 1}), calls
        return [got] + list(torch.autograd.grad((got.float() * cot.cuda()).sum(), [xc] + list(blk.parameters()), allow_unused=True))
    fused, two_kernel = run(True), run(False)
    names = ["out", "dx"] + pnames
    for n, f, u, w in zip(names, fused, two_kernel, [want] + list(gw)):
        if w is None or float(w.detach().abs().max()) == 0.0:
            continue
        assert f is not None and u is not None, n
        assert rel_err(f, u) < 1e-5, f"{n}: fused and two-kernel paths differ"
        tol = BF16_TOL if n == "out" else BF16_TOL * 1.5
        if n in ("out", "dx"):
            assert rel_err(f, w) < tol, n
        else:
            assert rel_err(f, w) < max(tol, rel_err(u, w) + 1e-5), n


def test_other_shapes_keep_the_two_kernel_path(mm, monkeypatch):
    grid = (8, 8, 8)
    spy = _Spy(mm, monkeypatch)

    def run(blk, dtype, *args):
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=dtype == torch.bfloat16):
            return blk(*args)

    x96 = torch.randn(2, math.prod(grid), 96, device="cuda")
    cases = {
        "cross-attention": lambda: run(mm.fu.Cross_SwinTransformerBlock(96, grid, 3, window_size=4, shift_size=2).cuda(),
                                       torch.bfloat16, x96, x96.clone(), grid),
        "C = 192": lambda: run(_v2_block(mm, C=192, nH=6).cuda(), torch.bfloat16, torch.randn(2, math.prod(grid), 192, device="cuda")),
        "fp32": lambda: run(_v2_block(mm).cuda(), torch.float32, x96),
        "dropout": lambda: run(_v2_block(mm, attn_drop=0.1).cuda().train(), torch.bfloat16, x96),
    }
    for name, fn in cases.items():
        before = dict(spy.calls)
        fn()
        assert spy.calls["mmn_winattn_qkv_fwd"] == before["mmn_winattn_qkv_fwd"], name
        assert spy.calls["mmn_winattn_fwd"] > before["mmn_winattn_fwd"], name
    # and the cfg2 shape takes the fused kernel
    before = dict(spy.calls)
    run(_v2_block(mm).cuda(), torch.bfloat16, x96)
    assert spy.calls["mmn_winattn_qkv_fwd"] == before["mmn_winattn_qkv_fwd"] + 1
    assert spy.calls["mmn_winattn_fwd"] == before["mmn_winattn_fwd"] and spy.calls["qkv_linear"] == before["qkv_linear"]


def test_graph_replay_and_concurrent_streams(mm):
    # module forward + backward captured in a CUDA graph replays to the eager result
    blk = _v2_block(mm).cuda()
    grid = (8, 8, 8)
    x = torch.randn(2, math.prod(grid), 96, device="cuda", requires_grad=True)
    dy = torch.randn(2, math.prod(grid), 96, device="cuda")

    def step():
        with torch.autocast("cuda", dtype=torch.bfloat16):
            y = blk(x)
        y.backward(dy)
        return y
    y_e = step().detach().clone()
    gx_e = x.grad.clone()
    gp_e = [p.grad.clone() for p in blk.parameters()]
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for p in blk.parameters():
            p.grad = None
        x.grad = None
        step()
    torch.cuda.current_stream().wait_stream(side)
    for p in blk.parameters():
        p.grad = None
    x.grad = None
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        y_s = step()
    for _ in range(2):
        x.grad.zero_()
        for p in blk.parameters():
            p.grad.zero_()
        graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(y_s, y_e)
    assert rel_err(x.grad, gx_e) < 1e-2
    for p, g in zip(blk.parameters(), gp_e):
        assert rel_err(p.grad, g) < 1e-2
    # two launches on two streams at once give the serial results bit for bit
    ins = [_inputs(mm, "all_classes_odd_counts", "cosine_qv_bias", seed=s) for s in (1, 2)]
    want = [_fused(*a) for a in ins]
    torch.cuda.synchronize()
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    for s in streams:
        s.wait_stream(torch.cuda.current_stream())
    got = [None, None]
    for _ in range(5):
        for k in (0, 1):
            with torch.cuda.stream(streams[k]):
                got[k] = _fused(*ins[k])
    torch.cuda.synchronize()
    for k in (0, 1):
        for t_got, t_want in zip(got[k], want[k]):
            assert torch.equal(t_got, t_want)


def test_deterministic_step_is_bit_repeatable(mm):
    blk = _v2_block(mm).cuda()
    grid = (8, 8, 8)
    x0 = torch.randn(2, math.prod(grid), 96, device="cuda")
    dy = torch.randn(2, math.prod(grid), 96, device="cuda")
    prev = torch.are_deterministic_algorithms_enabled()
    prev_warn = torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True, warn_only=True)
    try:
        runs = []
        for _ in range(2):
            for p in blk.parameters():
                p.grad = None
            x = x0.clone().requires_grad_(True)
            with torch.autocast("cuda", dtype=torch.bfloat16):
                y = blk(x)
            y.backward(dy)
            runs.append([y.detach().clone(), x.grad.clone()] + [p.grad.clone() for p in blk.parameters()])
        for a, b in zip(*runs):
            assert torch.equal(a, b)
    finally:
        torch.use_deterministic_algorithms(prev, warn_only=prev_warn)
