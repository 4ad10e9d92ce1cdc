"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle and the golden
fixtures produced by the unmodified reference.

Tolerances (BASELINE.json north_star): fp32 path 1e-5 relative, bf16 path 2e-2 relative,
where "relative" is max|got - want| / max|want| over the tensor (a gradient that the
reference leaves exactly zero must come out below 1e-6 absolute).
"""
import math

import numpy as np
import pytest
import torch

from oracle import ref_nd as R

pytestmark = pytest.mark.gpu

FP32_TOL = 1e-5
BF16_TOL = 2e-2


@pytest.fixture(scope="module")
def mm():
    from multimodal_neuroimage_b200 import _lib, ops  # noqa: F401
    from multimodal_neuroimage_b200.modules import crossmodal_transformer as cm
    from multimodal_neuroimage_b200.modules import multihead_attention as mh
    from multimodal_neuroimage_b200.modules import swin_v2_module as v2
    from multimodal_neuroimage_b200.modules import swinfusion_module as fu
    _lib.load()
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False

    class NS:
        pass
    ns = NS()
    ns.lib, ns.ops, ns.cm, ns.mh, ns.v2, ns.fu = _lib, ops, cm, mh, v2, fu
    return ns


def rel_err(got, want):
    got, want = got.detach().double().cpu(), want.detach().double().cpu()
    assert got.shape == want.shape, (got.shape, want.shape)
    assert torch.isfinite(got).all()
    scale = want.abs().max().item()
    err = (got - want).abs().max().item()
    return err / scale if scale > 0 else err * 1e1     # zero reference: absolute, 1e-6 -> 1e-5


def check(got, want, tol, what=""):
    e = rel_err(got, want)
    assert e <= tol, f"{what}: relative error {e:.3e} > {tol:.1e}"


# ------------------------------------------------------------------------------------------
# 1. Core op vs oracle: every geometry / variant / mask mode, fp32 and bf16, fwd + bwd
# ------------------------------------------------------------------------------------------
CORE_CASES = [
    # grid, window, shift, nH, d, cosine, mask ("none" | "shift" | "tensor"), batch
    ((12, 12), (6, 6), (3, 3), 3, 4, True, "shift", 2),          # reference default stage 1 (d=4, N=36)
    ((12, 12), (6, 6), (0, 0), 6, 2, False, "none", 2),          # fusion default (d=2)
    ((6, 6), (3, 3), (1, 1), 12, 4, True, "shift", 1),           # N=9
    ((8, 16), (4, 4), (2, 2), 2, 16, False, "shift", 2),
    ((16, 16), (8, 8), (4, 4), 3, 32, True, "shift", 2),         # 2-D N=64 d=32
    ((8, 8, 8), (4, 4, 4), (2, 2, 2), 3, 32, True, "shift", 2),  # cfg2 geometry, small grid
    ((8, 8, 8), (4, 4, 4), (0, 0, 0), 3, 32, False, "none", 1),
    ((4, 8, 12), (2, 4, 4), (1, 2, 2), 2, 8, True, "shift", 1),  # anisotropic 3-D
    ((8, 8, 4), (4, 4, 4), (2, 2, 0), 2, 32, False, "shift", 1), # one axis unshifted
    ((36,), (36,), (0,), 3, 4, True, "tensor", 8),               # pre-windowed call with a (nW,N,N) mask
    ((64,), (64,), (0,), 2, 32, False, "tensor", 6),
    ((16, 16), (8, 8), (4, 4), 1, 64, True, "shift", 1),         # d=64
    ((8, 8, 8), (8, 8, 8), (0, 0, 0), 2, 16, False, "none", 1),  # N=512 (key chunking)
    ((14, 14), (7, 7), (3, 3), 2, 7, False, "shift", 1),         # odd head_dim, N=49
    # class-sorted item schedule of the tensor-core path (tc_sched.cuh): all eight wrap classes, odd class
    # counts (single-window items), class changes inside a CTA's item range
    ((12, 12, 12), (4, 4, 4), (2, 2, 2), 3, 32, True, "shift", 1),
    ((12, 8, 16), (4, 4, 4), (2, 2, 2), 2, 32, False, "shift", 3),
    ((16, 16, 16), (4, 4, 4), (2, 2, 2), 3, 32, True, "shift", 2),
    ((24, 40), (8, 8), (4, 4), 3, 32, True, "shift", 3),         # 2-D, odd batch
    ((8, 8, 16), (4, 4, 4), (2, 2, 2), 6, 32, True, "shift", 1), # cfg5 stage-1 head count (C = 192)
]


def _core_inputs(case, dtype, cross, seed=0):
    grid, window, shift, nH, d, cosine, mask_mode, B = case
    g = torch.Generator().manual_seed(seed)
    C = nH * d
    N = math.prod(window)
    if cross:
        a = torch.randn(B, *grid, C, generator=g)
        b = torch.randn(B, *grid, 2 * C, generator=g)
    else:
        a = torch.randn(B, *grid, 3 * C, generator=g)
        b = None
    bias = torch.randn(nH, N, N, generator=g)
    hs = torch.rand(nH, generator=g) * 20 + 0.5 if cosine else None
    mask = None
    if mask_mode == "tensor":
        nW = 2 if B % 2 == 0 else 1
        reg = torch.randint(0, 3, (nW, N), generator=g).float()
        dm = reg.unsqueeze(1) - reg.unsqueeze(2)
        mask = dm.masked_fill(dm != 0, -100.0).masked_fill(dm == 0, 0.0)
    dout = torch.randn(B, *grid, C, generator=g)
    if dtype == torch.bfloat16:       # identical bf16-representable inputs on both sides
        a, dout = a.bfloat16().float(), dout.bfloat16().float()
        b = b.bfloat16().float() if b is not None else None
    return a, b, bias, hs, mask, dout


def _oracle_core(case, a, b, bias, hs, mask, dout, keep=None):
    grid, window, shift, nH, d, cosine, mask_mode, B = case
    C = nH * d
    dd = torch.float64
    a = a.to(dd).requires_grad_(True)
    b = b.to(dd).requires_grad_(True) if b is not None else None
    bias = bias.to(dd).requires_grad_(True)
    hs = hs.to(dd).requires_grad_(True) if hs is not None else None
    if b is None:
        q, k, v = a[..., :C], a[..., C:2 * C], a[..., 2 * C:]
    else:
        q, k, v = a, b[..., :C], b[..., C:]
    m = mask.to(dd) if mask is not None else None
    if mask_mode == "shift":
        m = R.shift_mask_nd(grid, window, shift, dd)
    out, lse = R.window_attention_core(q, k, v, grid, window, shift, nH, cosine=cosine, scale=d ** -0.5,
                                       head_scale=hs, bias=bias, mask=m, keep=keep)
    wrt = [t for t in (a, b, bias, hs) if t is not None]
    grads = torch.autograd.grad((out * dout.to(dd)).sum(), wrt)
    it = iter(grads)
    return out, lse, next(it), (next(it) if b is not None else None), next(it), (next(it) if hs is not None else None)


def _run_core(mm, case, dtype, cross, path):
    grid, window, shift, nH, d, cosine, mask_mode, B = case
    a, b, bias, hs, mask, dout = _core_inputs(case, dtype, cross)
    want = _oracle_core(case, a, b, bias, hs, mask, dout)
    dev = "cuda"
    ac = a.to(dev, dtype).requires_grad_(True)
    bc = b.to(dev, dtype).requires_grad_(True) if b is not None else None
    biasc = bias.to(dev).requires_grad_(True)
    hsc = hs.to(dev).requires_grad_(True) if hs is not None else None
    maskc = mask.to(dev) if mask is not None else None
    kind = {"none": mm.lib.MASK_NONE, "shift": mm.lib.MASK_SHIFT, "tensor": mm.lib.MASK_TENSOR}[mask_mode]
    out, lse = torch.ops.mmn_b200.winattn_fwd(ac, bc, biasc, hsc, maskc, list(grid), list(window), list(shift), nH,
                                              mm.lib.SCORE_COSINE if cosine else mm.lib.SCORE_SCALED, kind, d ** -0.5,
                                              0.0, 0, 0, path)
    wrt = [t for t in (ac, bc, biasc, hsc) if t is not None]
    grads = torch.autograd.grad((out.float() * dout.to(dev)).sum(), wrt)
    it = iter(grads)
    # lse is (4, B*nW, nH, N): slab 0 = log-sum-exp; slabs 1-3 = per-window records kept by the tcgen05 forward for its backward
    got = (out, lse[0], next(it), (next(it) if bc is not None else None), next(it), (next(it) if hsc is not None else None))
    tol = FP32_TOL if dtype == torch.float32 else BF16_TOL
    names = ["out", "lse", "d_a", "d_b", "d_bias", "d_head_scale"]
    for n, g_, w_ in zip(names, got, want):
        if w_ is None:
            continue
        check(g_, w_, tol, f"{n} {case} {dtype} cross={cross}")


@pytest.mark.parametrize("case", CORE_CASES, ids=lambda c: f"g{'x'.join(map(str, c[0]))}_w{'x'.join(map(str, c[1]))}_s{'x'.join(map(str, c[2]))}_h{c[3]}d{c[4]}_{'cos' if c[5] else 'dot'}_{c[6]}")
@pytest.mark.parametrize("cross", [False, True], ids=["self", "cross"])
def test_winattn_core_fp32_generic(mm, case, cross):
    _run_core(mm, case, torch.float32, cross, mm.lib.PATH_GENERIC)


@pytest.mark.parametrize("case", [CORE_CASES[0], CORE_CASES[4], CORE_CASES[5], CORE_CASES[9]],
                         ids=["d4", "2d_n64", "3d_n64", "prewindowed"])
def test_winattn_core_bf16_generic(mm, case):
    _run_core(mm, case, torch.bfloat16, False, mm.lib.PATH_GENERIC)


TC_CASES = [c for c in CORE_CASES if math.prod(c[1]) == 64 and c[4] == 32]


@pytest.mark.parametrize("case", TC_CASES, ids=lambda c: f"g{'x'.join(map(str, c[0]))}_s{'x'.join(map(str, c[2]))}_{'cos' if c[5] else 'dot'}_{c[6]}")
@pytest.mark.parametrize("cross", [False, True], ids=["self", "cross"])
def test_winattn_core_bf16_tcgen05(mm, case, cross):
    grid, window, shift, nH, d, cosine, mask_mode, B = case
    a, b, *_ = _core_inputs(case, torch.bfloat16, cross)
    kind = {"none": mm.lib.MASK_NONE, "shift": mm.lib.MASK_SHIFT, "tensor": mm.lib.MASK_TENSOR}[mask_mode]
    name = mm.ops.winattn_path_name(a.cuda().bfloat16(), None if b is None else b.cuda().bfloat16(), grid, window, shift,
                                    nH, mm.lib.SCORE_COSINE if cosine else mm.lib.SCORE_SCALED, kind)
    assert name == "tcgen05", f"tuned shape fell back to {name}"
    _run_core(mm, case, torch.bfloat16, cross, mm.lib.PATH_AUTO)


# ------------------------------------------------------------------------------------------
# 2. Golden fixtures (unmodified reference, fp32): modules end to end, outputs + all grads
# ------------------------------------------------------------------------------------------
def _golden_module_case(G, case, module, call, in_names, tol=FP32_TOL):
    module.load_state_dict(G.group(f"{case}/sd/"), strict=True)
    module = module.cuda().eval()
    ins = {k: v.cuda().requires_grad_(k in in_names) for k, v in G.group(f"{case}/in/").items()}
    outs = call(module, ins)
    outs = outs if isinstance(outs, (tuple, list)) else (outs,)
    n_out = len(G.keys(f"{case}/out/"))
    loss = 0
    for i in range(n_out):
        if outs[i] is None:
            continue
        check(outs[i], G.t(f"{case}/out/{i}"), tol, f"{case} out{i}")
        if i in G.arr(f"{case}/loss_outs").tolist():
            loss = loss + (outs[i] * G.t(f"{case}/cot/{i}").cuda()).sum()
    module.zero_grad()
    loss.backward()
    for k in in_names:
        check(ins[k].grad, G.t(f"{case}/gin/{k}"), tol * 5, f"{case} d{k}")
    params = dict(module.named_parameters())
    for k, ref in G.group(f"{case}/gsd/").items():
        g = params[k].grad
        if g is None:
            assert float(ref.abs().max()) == 0.0, k
        else:
            check(g, ref, tol * 5, f"{case} d{k}")


def test_golden_swinv2(mm, golden):
    G = golden("swinv2")
    for case in ("wa_c12", "wa_c96", "wa_c48_nomask"):
        C, nH, w0, w1 = G.arr(f"{case}/cfg").tolist()
        _golden_module_case(G, case, mm.v2.WindowAttention(C, (w0, w1), nH), lambda m, i: m(i["x"], i.get("mask")), ["x"])
    for case in ("blk_shift", "blk_noshift", "blk_clamp", "blk_rect"):
        C, nH, H, W, ws, s = G.arr(f"{case}/cfg").tolist()
        _golden_module_case(G, case, mm.v2.SwinTransformerBlock(C, (H, W), nH, window_size=ws, shift_size=s),
                            lambda m, i: m(i["x"]), ["x"])


def test_golden_swinfusion(mm, golden):
    G = golden("swinfusion")
    for c in ("wa_c12", "wa_c64"):
        C, nH, w0, w1 = G.arr(f"self_{c}/cfg").tolist()
        _golden_module_case(G, "self_" + c, mm.fu.WindowAttention_fusion(C, (w0, w1), nH), lambda m, i: m(i["x"], i["mask"]), ["x"])
        _golden_module_case(G, "cross_" + c, mm.fu.Cross_WindowAttention(C, (w0, w1), nH),
                            lambda m, i: m(i["x"], i["y"], i["mask"]), ["x", "y"])
    for c in ("blk_shift", "blk_xsize", "blk_noshift"):
        C, nH, r0, r1, x0, x1, ws, s = G.arr(f"self_{c}/cfg").tolist()
        _golden_module_case(G, "self_" + c, mm.fu.SwinTransformerBlock_fusion(C, (r0, r1), nH, window_size=ws, shift_size=s),
                            lambda m, i: m(i["x"], (x0, x1)), ["x"])
        _golden_module_case(G, "cross_" + c, mm.fu.Cross_SwinTransformerBlock(C, (r0, r1), nH, window_size=ws, shift_size=s),
                            lambda m, i: m(i["x"], i["y"], (x0, x1)), ["x", "y"])


def test_golden_crossmodal(mm, golden):
    G = golden("crossmodal")
    for case in ("mha_self_d7", "mha_cross_d7", "mha_cross_TneS", "mha_self_d14_nomask"):
        E, nH, T, S, B, has_mask = G.arr(f"{case}/cfg").tolist()
        names = ["q"] if "self" in case else ["q", "k", "v"]

        def call(m, i):
            mask = mm.cm.buffered_future_mask(torch.zeros(T, 1, 1, device="cuda"), torch.zeros(S, 1, 1, device="cuda")) if has_mask else None
            q = i["q"]
            k, v = (q, q) if "k" not in i else (i["k"], i["v"])
            return m(q, k, v, attn_mask=mask)
        _golden_module_case(G, case, mm.mh.MultiheadAttention(E, nH), call, names)
    for case in ("enc_self", "enc_cross", "enc_cross_nomask"):
        E, nH, L, T, B, use_mask, cross = G.arr(f"{case}/cfg").tolist()
        names = ["x"] if case == "enc_self" else ["x", "xk", "xv"]
        _golden_module_case(G, case, mm.cm.TransformerEncoder(E, nH, L, attn_mask=bool(use_mask)),
                            lambda m, i: m(i["x"], i.get("xk"), i.get("xv")), names)


def test_mha_dense_mask_equals_generated_mask(mm):
    """An explicit (T,S) tensor mask and the in-kernel future mask must agree bit for bit."""
    T, S, B, E, nH = 33, 41, 2, 24, 4
    g = torch.Generator().manual_seed(3)
    q, k, v = (torch.randn(n, B, E, generator=g).cuda() for n in (T, S, S))
    dense = R.future_mask(T, S).cuda()
    a = torch.ops.mmn_b200.mha_fwd(q, k, v, dense, nH, mm.lib.MASK_TENSOR, 0, 0.4, 0.0, 0, 0)
    b = torch.ops.mmn_b200.mha_fwd(q, k, v, None, nH, mm.lib.MASK_FUTURE, 1 + abs(S - T), 0.4, 0.0, 0, 0)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


# ------------------------------------------------------------------------------------------
# 3. 3-D modules (our generalisation) vs the n-D oracle, fp32 and bf16 autocast
# ------------------------------------------------------------------------------------------
def _sd64(module):
    return {k: (v.detach().double() if v.is_floating_point() else v.detach()).cpu() for k, v in module.state_dict().items()}


def _randomise(module, seed):
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for name, p in module.named_parameters():
            if "norm" in name and name.endswith("weight"):
                p.copy_(torch.empty(p.shape).uniform_(0.5, 1.5, generator=g))
            elif name.endswith("relative_position_bias_table"):
                p.copy_(torch.empty(p.shape).normal_(0, 1.0, generator=g))
            elif name.endswith("logit_scale"):
                p.copy_(torch.empty(p.shape).uniform_(0.0, math.log(200.0), generator=g))
            elif name.endswith("bias"):
                p.copy_(torch.empty(p.shape).normal_(0, 0.3, generator=g))


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
def test_swinv2_block_3d(mm, dtype):
    grid, C, nH, B = (8, 8, 8), 96, 3, 2
    blk = mm.v2.SwinTransformerBlock(C, grid, nH, window_size=4, shift_size=2)
    _randomise(blk, 11)
    if dtype == torch.bfloat16:
        # logit scales of trained SwinV2 models (init ln 10).  Near the clamp (g = 100) a 16-bit q / k operand moves a logit by
        # ~0.1 whatever computes it (tools/debug_fp16.py), so a whole-block bf16 comparison there measures the operand
        # rounding, not the kernels; the clamp range is covered by the fp32 variant of this test.
        with torch.no_grad():
            blk.attn.logit_scale.copy_(torch.tensor([1.0, 10.0, 20.0]).log().view(3, 1, 1))
    x = torch.randn(B, math.prod(grid), C, generator=torch.Generator().manual_seed(5))
    xo = x.double().requires_grad_(True)
    want = R.swin_v2_block(xo, _sd64(blk), grid, 4, 2, nH)
    cot = torch.randn(want.shape, generator=torch.Generator().manual_seed(6))
    gx_want, = torch.autograd.grad((want * cot.double()).sum(), xo)
    blk = blk.cuda()
    xc = x.cuda().requires_grad_(True)
    with torch.autocast("cuda", dtype=torch.bfloat16, enabled=dtype == torch.bfloat16):
        got = blk(xc)
    gx_got, = torch.autograd.grad((got.float() * cot.cuda()).sum(), xc)
    tol = FP32_TOL if dtype == torch.float32 else BF16_TOL
    check(got, want, tol, "block3d out")
    check(gx_got, gx_want, tol * (5 if dtype == torch.float32 else 1.5), "block3d dx")


def test_cross_block_3d_fp32(mm):
    grid, C, nH, B = (4, 8, 8), 32, 2, 1
    blk = mm.fu.Cross_SwinTransformerBlock(C, grid, nH, window_size=4, shift_size=2)
    _randomise(blk, 12)
    g = torch.Generator().manual_seed(7)
    x, y = torch.randn(B, math.prod(grid), C, generator=g), torch.randn(B, math.prod(grid), C, generator=g)
    xo, yo = x.double().requires_grad_(True), y.double().requires_grad_(True)
    wx, wy = R.cross_block(xo, yo, _sd64(blk), grid, grid, 4, 2, nH)
    gx_w, gy_w = torch.autograd.grad(wx.sum() + 2 * wy.sum(), (xo, yo))
    blk = blk.cuda()
    xc, yc = x.cuda().requires_grad_(True), y.cuda().requires_grad_(True)
    ox, oy = blk(xc, yc, grid)
    gx, gy = torch.autograd.grad(ox.sum() + 2 * oy.sum(), (xc, yc))
    for got, want, n in ((ox, wx, "x"), (oy, wy, "y"), (gx, gx_w, "dx"), (gy, gy_w, "dy")):
        check(got, want, FP32_TOL * 5, "cross3d " + n)


# ------------------------------------------------------------------------------------------
# 4. Size-independent properties at BASELINE cfg2 size (oracle too slow there)
# ------------------------------------------------------------------------------------------
def test_full_size_properties(mm):
    """cfg2: (B,32,32,32,96), 4x4x4 windows, shift 2, 3 heads x 32, bf16."""
    B, grid, window, shift, nH, d = 2, (32, 32, 32), (4, 4, 4), (2, 2, 2), 3, 32
    C, N = nH * d, 64
    g = torch.Generator(device="cuda").manual_seed(0)
    qkv = torch.randn(B, *grid, 3 * C, generator=g, device="cuda", dtype=torch.bfloat16)
    bias = torch.randn(nH, N, N, generator=g, device="cuda")
    hs = torch.rand(nH, generator=g, device="cuda") * 10 + 1
    args = (list(grid), list(window), list(shift), nH, mm.lib.SCORE_COSINE, mm.lib.MASK_SHIFT, 1.0, 0.0, 0, 0)
    out, lse = torch.ops.mmn_b200.winattn_fwd(qkv, None, bias, hs, None, *args, mm.lib.PATH_AUTO)
    # (a) probabilities sum to one: V == 1 everywhere -> out == 1
    ones = qkv.clone()
    ones[..., 2 * C:] = 1.0
    o1, _ = torch.ops.mmn_b200.winattn_fwd(ones, None, bias, hs, None, *args, mm.lib.PATH_AUTO)
    assert (o1.float() - 1).abs().max().item() < 1e-2
    # (b) translation equivariance: rolling the volume by one window pitch (4) on every axis
    #     along with the batch of windows is a symmetry of the op only where no mask region
    #     boundary moves -- instead use the exact symmetry: out(roll(x, w)) on the UNSHIFTED,
    #     unmasked op equals roll(out(x), w).
    a0 = (list(grid), list(window), [0, 0, 0], nH, mm.lib.SCORE_COSINE, mm.lib.MASK_NONE, 1.0, 0.0, 0, 0)
    o_a, _ = torch.ops.mmn_b200.winattn_fwd(qkv, None, bias, hs, None, *a0, mm.lib.PATH_AUTO)
    rolled = torch.roll(qkv, (4, 8, 12), (1, 2, 3))
    o_b, _ = torch.ops.mmn_b200.winattn_fwd(rolled, None, bias, hs, None, *a0, mm.lib.PATH_AUTO)
    assert torch.equal(torch.roll(o_a, (4, 8, 12), (1, 2, 3)), o_b)
    # (c) shifted op == unshifted op on the rolled volume with the explicit mask tensor
    mask = R.shift_mask_nd(grid, window, shift).cuda()
    xr = torch.roll(qkv, (-2, -2, -2), (1, 2, 3))
    xw = R.window_partition_nd(xr, window).reshape(-1, N, 3 * C)
    o_w, _ = torch.ops.mmn_b200.winattn_fwd(xw, None, bias, hs, mask, [N], [N], [0], nH, mm.lib.SCORE_COSINE,
                                            mm.lib.MASK_TENSOR, 1.0, 0.0, 0, 0, mm.lib.PATH_GENERIC)
    o_w = torch.roll(R.window_reverse_nd(o_w.reshape(-1, *window, C), window, grid), (2, 2, 2), (1, 2, 3))
    assert rel_err(out, o_w) < BF16_TOL
    # (d) both code paths agree at full size
    o_g, lse_g = torch.ops.mmn_b200.winattn_fwd(qkv, None, bias, hs, None, *args, mm.lib.PATH_GENERIC)
    assert rel_err(out, o_g) < BF16_TOL and rel_err(lse[0], lse_g[0]) < 1e-2
    # (e) batch independence (the sharding property of SURVEY.md 8e): sample 1 alone == sample 1 of the batch
    o_s, _ = torch.ops.mmn_b200.winattn_fwd(qkv[1:2].contiguous(), None, bias, hs, None, *args, mm.lib.PATH_AUTO)
    assert torch.equal(o_s, out[1:2])


def test_full_size_backward_properties(mm):
    """cfg2 size, backward: tcgen05 gradients == generic-path gradients (all of them), column sums of the
    packed gradient == the kernel's dcolsum, and batch independence of the input gradient."""
    B, grid, window, shift, nH, d = 2, (32, 32, 32), (4, 4, 4), (2, 2, 2), 3, 32
    C, N = nH * d, 64
    g = torch.Generator(device="cuda").manual_seed(1)
    qkv = torch.randn(B, *grid, 3 * C, generator=g, device="cuda", dtype=torch.bfloat16)
    dout = torch.randn(B, *grid, C, generator=g, device="cuda", dtype=torch.bfloat16)
    bias = torch.randn(nH, N, N, generator=g, device="cuda")
    hs = torch.rand(nH, generator=g, device="cuda") * 10 + 1
    args = (list(grid), list(window), list(shift), nH, mm.lib.SCORE_COSINE, mm.lib.MASK_SHIFT, 1.0, 0.0, 0, 0)
    res = {}
    for name, path in (("tc", mm.lib.PATH_AUTO), ("gen", mm.lib.PATH_GENERIC)):
        out, lse = torch.ops.mmn_b200.winattn_fwd(qkv, None, bias, hs, None, *args, path)
        res[name] = torch.ops.mmn_b200.winattn_bwd(dout, qkv, None, bias, hs, None, out, lse, *args, path, True)
    for i, n in ((0, "dqkv"), (2, "dbias"), (3, "dhead_scale"), (4, "dcolsum")):
        assert rel_err(res["tc"][i], res["gen"][i]) < BF16_TOL, n
    dqkv, dcs = res["tc"][0], res["tc"][4]
    assert rel_err(dcs.reshape(-1), dqkv.float().sum((0, 1, 2, 3))) < 1e-2
    out, lse = torch.ops.mmn_b200.winattn_fwd(qkv[1:2].contiguous(), None, bias, hs, None, *args, mm.lib.PATH_AUTO)
    one = torch.ops.mmn_b200.winattn_bwd(dout[1:2].contiguous(), qkv[1:2].contiguous(), None, bias, hs, None, out, lse, *args,
                                         mm.lib.PATH_AUTO, True)
    assert torch.equal(one[0], dqkv[1:2])


def test_dynamic_schedule_streams_and_slot_reuse(mm):
    """The tcgen05 kernels hand out work through self-resetting device counters, one slot per launch out of a pool of
    128 (tc_sched.cuh: ClassQueue, winattn_tc_fwd.cuh: work_slot).  (a) Launches on two streams at the same time use
    different slots: results equal the serial ones.  (b) More launches than slots: a slot is re-armed by the last
    CTA of the launch that used it, so launch 300 is as good as launch 1.  (c) A captured CUDA graph replays correctly
    (its slot is baked into the kernel parameters)."""
    grid, window, shift, nH, d = (16, 16, 16), (4, 4, 4), (2, 2, 2), 3, 32
    C, N = nH * d, 64
    g = torch.Generator(device="cuda").manual_seed(1)
    args = (list(grid), list(window), list(shift), nH, mm.lib.SCORE_COSINE, mm.lib.MASK_SHIFT, 1.0, 0.0, 0, 0, mm.lib.PATH_AUTO)
    bias = torch.randn(nH, N, N, generator=g, device="cuda")
    hs = torch.rand(nH, generator=g, device="cuda") * 10 + 1
    xs = [torch.randn(B, *grid, 3 * C, generator=g, device="cuda", dtype=torch.bfloat16) for B in (3, 5)]
    dys = [torch.randn(x.shape[0], *grid, C, generator=g, device="cuda", dtype=torch.bfloat16) for x in xs]
    assert mm.ops.winattn_path_name(xs[0], None, grid, window, shift, nH, mm.lib.SCORE_COSINE, mm.lib.MASK_SHIFT) == "tcgen05"

    def run(x, dy):
        out, lse = torch.ops.mmn_b200.winattn_fwd(x, None, bias, hs, None, *args)
        dx = torch.ops.mmn_b200.winattn_bwd(dy, x, None, bias, hs, None, out, lse, *args, True)[0]
        return out, dx

    want = [run(x, dy) for x, dy in zip(xs, dys)]
    torch.cuda.synchronize()
    # (a) two streams, interleaved
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    got = [None, None]
    for _ in range(10):
        for k in (0, 1):
            with torch.cuda.stream(streams[k]):
                got[k] = run(xs[k], dys[k])
    torch.cuda.synchronize()
    for k in (0, 1):
        assert torch.equal(got[k][0], want[k][0]), "forward differs when two streams run it concurrently"
        assert rel_err(got[k][1], want[k][1]) < 1e-2
    # (b) slot pool wrap-around
    for _ in range(300):
        out, _ = torch.ops.mmn_b200.winattn_fwd(xs[0], None, bias, hs, None, *args)
    assert torch.equal(out, want[0][0])
    # (c) graph replay
    static_x = xs[1].clone()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        g_out, g_dx = run(static_x, dys[1])
    for _ in range(3):
        graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(g_out, want[1][0]) and rel_err(g_dx, want[1][1]) < 1e-2


@pytest.mark.parametrize("rows,n_out", [(128, 96), (1000, 288), (4096 + 37, 192), (70000, 288), (300, 96)])
def test_linear_bwd_fused(mm, rows, n_out):
    """Fused projection backward (linbwd_tc.cu): dx, dw, db of y = x W^T + b against fp64 on the same bf16 operands;
    row counts that are not a multiple of the 128-token tile exercise the TMA out-of-bounds fill / clipping."""
    n_in = 96
    g = torch.Generator().manual_seed(rows + n_out)
    dy = torch.randn(rows, n_out, generator=g).bfloat16()
    x = torch.randn(rows, n_in, generator=g).bfloat16()
    w = (torch.randn(n_out, n_in, generator=g) * n_in ** -0.5).bfloat16()
    assert mm.ops.linear_bwd_supported(dy.cuda(), x.cuda(), w.cuda())
    dx, dw, db = torch.ops.mmn_b200.linear_bwd(dy.cuda(), x.cuda(), w.cuda())
    dyd, xd, wd = dy.double(), x.double(), w.double()
    check(dx, dyd @ wd, BF16_TOL, "linear_bwd dx")
    check(dw, dyd.t() @ xd, 2e-3, "linear_bwd dw")        # fp32 accumulation of bf16 products
    check(db, dyd.sum(0), 2e-3, "linear_bwd db")
    # strided operands: dy as a channel slice of a wider tensor
    wide = torch.randn(rows, n_out + 64, generator=g).bfloat16().cuda()
    dx2, dw2, db2 = torch.ops.mmn_b200.linear_bwd(wide[:, 32:32 + n_out] if False else wide[:, :n_out], x.cuda(), w.cuda())
    check(dw2, wide[:, :n_out].double().cpu().t() @ xd, 2e-3, "linear_bwd dw (strided dy)")


@pytest.mark.parametrize("window,nH", [((4, 4, 4), 3), ((8, 8), 6), ((6, 6), 12), ((4, 4, 4), 24)])
def test_cpb_bias_fused(mm, window, nH):
    """cpb_bias.cu against the reference formulation 16*sigmoid(cpb_mlp(table))[index] (swin_v2_module.py:158-162) in
    fp64, forward and all three parameter gradients."""
    from multimodal_neuroimage_b200 import geometry
    g = torch.Generator().manual_seed(nH)
    n = len(window)
    coords = geometry.cpb_coords_table(window).reshape(-1, n).float()
    index = geometry.relative_position_index(window).reshape(-1)
    w1 = torch.randn(512, n, generator=g) * 0.7
    b1 = torch.randn(512, generator=g) * 0.3
    w2 = torch.randn(nH, 512, generator=g) * 0.1
    cot = torch.randn(nH, index.numel(), generator=g)
    pd = [t.double().requires_grad_(True) for t in (w1, b1, w2)]
    tab = torch.relu(coords.double() @ pd[0].t() + pd[1]) @ pd[2].t()
    want = (16 * torch.sigmoid(tab))[index].t()
    gw = torch.autograd.grad((want * cot.double()).sum(), pd)
    pc = [t.cuda().requires_grad_(True) for t in (w1, b1, w2)]
    assert mm.ops.cpb_bias_supported(coords.cuda(), pc[0], pc[2])
    got, _ = torch.ops.mmn_b200.cpb_bias_fwd(coords.cuda(), pc[0], pc[1], pc[2], index.cuda())
    gg = torch.autograd.grad((got * cot.cuda()).sum(), pc)
    check(got, want, FP32_TOL, "cpb bias")
    for a, b, nm in zip(gg, gw, ("dw1", "db1", "dw2")):
        check(a, b, FP32_TOL * 2, "cpb " + nm)


def test_dropout_statistics_and_backward_consistency(mm):
    """p > 0: keep-rate ~ 1-p, E[out] ~ no-dropout out, and fwd/bwd regenerate the same mask
    (checked by linearity: with probabilities frozen, out is linear in v)."""
    T, B, E, nH, p = 64, 4, 32, 4, 0.25
    g = torch.Generator().manual_seed(9)
    q, k = (torch.randn(T, B, E, generator=g).cuda() for _ in range(2))
    v = torch.randn(T, B, E, generator=g).cuda().requires_grad_(True)
    out, lse = torch.ops.mmn_b200.mha_fwd(q, k, v, None, nH, 0, 0, 0.35, p, 123, 7)
    avg = torch.ops.mmn_b200.mha_avg_weights(q, k, None, lse, nH, 0, 0, 0.35, p, 123, 7)
    avg0 = torch.ops.mmn_b200.mha_avg_weights(q, k, None, lse, nH, 0, 0, 0.35, 0.0, 0, 0)
    kept = (avg > 0).float().mean().item()          # a (b,i,j) survives unless all heads drop it
    assert abs(avg.sum(-1).mean().item() - 1.0) < 0.05 and kept > 0.9
    assert torch.allclose(avg0.sum(-1), torch.ones_like(avg0.sum(-1)), atol=1e-4)
    cot = torch.randn(out.shape, generator=g).cuda()
    gv, = torch.autograd.grad((out * cot).sum(), v)
    # out = P_drop v  =>  <cot, out> = <P_drop^T cot, v> ; check with a second v
    v2 = torch.randn(T, B, E, generator=g).cuda()
    out2, _ = torch.ops.mmn_b200.mha_fwd(q, k, v2, None, nH, 0, 0, 0.35, p, 123, 7)
    lhs = (out2 * cot).sum().item()
    rhs = (gv * v2).sum().item()
    assert abs(lhs - rhs) <= 1e-3 * max(1.0, abs(lhs))
