"""Deterministic mode: under torch.use_deterministic_algorithms(True) every gradient the library produces is the same bit
for bit from run to run (repeated calls, a backward racing another one on a second stream, CUDA-graph replay), matches the
default mode to fp32 rounding, and matches the fp64 oracle; with the flag off the default kernels run exactly as before."""
import ctypes
import math
import os
import subprocess
import sys

import pytest
import torch

from test_gpu_parity import BF16_TOL, CORE_CASES, FP32_TOL, _core_inputs, _oracle_core, check, mm, rel_err  # noqa: F401

pytestmark = pytest.mark.gpu


@pytest.fixture
def det():
    """Turns the process-wide flag on for one test and restores it afterwards."""
    prev, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True)
    yield
    torch.use_deterministic_algorithms(prev, warn_only=warn)


def _flag(on):
    torch.use_deterministic_algorithms(on)


def _same(runs, what):
    for r in runs[1:]:
        for i, (a, b) in enumerate(zip(runs[0], r)):
            assert torch.equal(a, b), f"{what}: output {i} differs between runs"


def _repeat(fn, what, n=5, graph=True):
    """fn() -> tuple of tensors: n calls, one while another call runs on a second stream, one CUDA-graph replay."""
    runs = [tuple(t.clone() for t in fn()) for _ in range(n)]
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        other = fn()
    runs.append(tuple(t.clone() for t in fn()))
    torch.cuda.current_stream().wait_stream(side)
    runs.append(tuple(t.clone() for t in other))
    if graph:
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            fn()
        torch.cuda.current_stream().wait_stream(s)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            out = fn()
        g.replay()
        torch.cuda.synchronize()
        runs.append(tuple(t.clone() for t in out))
    torch.cuda.synchronize()
    _same(runs, what)
    return runs[0]


# ------------------------------------------------------------------------------------------
# window attention backward: tensor-core and generic paths
# ------------------------------------------------------------------------------------------
def _win_setup(mm, case, dtype, cross, path):
    grid, window, shift, nH, d, cosine, mask_mode, B = case
    a, b, bias, hs, mask, dout = _core_inputs(case, dtype, cross)
    dev = "cuda"
    ac = a.to(dev, dtype)
    bc = b.to(dev, dtype) if b is not None else None
    kind = {"none": mm.lib.MASK_NONE, "shift": mm.lib.MASK_SHIFT, "tensor": mm.lib.MASK_TENSOR}[mask_mode]
    cfg = (list(grid), list(window), list(shift), nH, mm.lib.SCORE_COSINE if cosine else mm.lib.SCORE_SCALED, kind, d ** -0.5,
           0.0, 0, 0, path)
    biasc, hsc = bias.to(dev), (hs.to(dev) if hs is not None else None)
    maskc = mask.to(dev) if mask is not None else None
    out, lse = torch.ops.mmn_b200.winattn_fwd(ac, bc, biasc, hsc, maskc, *cfg)
    doc = dout.to(dev, dtype)

    def bwd():
        da, db, dbias, dhs, dcs = torch.ops.mmn_b200.winattn_bwd(doc, ac, bc, biasc, hsc, maskc, out, lse, *cfg, True)
        return tuple(t for t in (da, db, dbias, dhs, dcs) if t.numel())
    return (a, b, bias, hs, mask, dout), bwd


def _check_win(mm, case, dtype, cross, path, oracle=True):
    inputs, bwd = _win_setup(mm, case, dtype, cross, path)
    _flag(False)
    ref = tuple(t.clone() for t in bwd())
    _flag(True)
    got = _repeat(bwd, f"winattn bwd {case} cross={cross}")
    n_tok = 2 if cross else 1
    for i, (g, r) in enumerate(zip(got, ref)):
        if i < n_tok:
            assert torch.equal(g, r), "dq / dk / dv must not depend on the mode"
        elif i == len(got) - 1 and dtype != torch.float32 and path == mm.lib.PATH_GENERIC:
            # generic bf16: the deterministic dcolsum sums the bf16-rounded dq / dk / dv, the default their fp32 values
            check(g, r, BF16_TOL, "deterministic vs default dcolsum")
        else:
            check(g, r, FP32_TOL if dtype == torch.float32 else 1e-5, f"deterministic vs default, output {i}")
    C = case[3] * case[4]
    tok = torch.cat([t.reshape(-1, t.shape[-1]) for t in got[:n_tok]], dim=-1).double().sum(0)    # dq | dk | dv column sums
    check(got[-1].reshape(-1), tok, 1e-5 if dtype == torch.float32 else 1e-4, "dcolsum vs the column sums of dq, dk, dv")
    if oracle:
        want = _oracle_core(case, *inputs)
        tol = FP32_TOL if dtype == torch.float32 else BF16_TOL
        wants = [w for w in want[2:] if w is not None]
        for g, w in zip(got[:len(wants)], wants):
            check(g, w, tol, "deterministic vs fp64 oracle")
    assert got[-1].shape == (3, C)


TC_DET_CASES = [CORE_CASES[14], CORE_CASES[15], CORE_CASES[16],              # all eight wrap classes, cosine / scaled
                ((32, 32, 32), (4, 4, 4), (2, 2, 2), 3, 32, True, "shift", 1)] + \
               [((8, 8, 8), (4, 4, 4), (2, 2, 2), h, 32, True, "shift", 1) for h in (6, 12, 24, 48)]     # cfg5 head counts


@pytest.mark.parametrize("case", TC_DET_CASES, ids=lambda c: f"g{'x'.join(map(str, c[0]))}_h{c[3]}_{'cos' if c[5] else 'dot'}_b{c[7]}")
@pytest.mark.parametrize("cross", [False, True], ids=["self", "cross"])
def test_winattn_bwd_tcgen05_deterministic(mm, det, case, cross):
    a, b, *_ = _core_inputs(case, torch.bfloat16, cross)
    grid, window, shift, nH = case[:4]
    name = mm.ops.winattn_path_name(a.cuda().bfloat16(), None if b is None else b.cuda().bfloat16(), grid, window, shift, nH,
                                    mm.lib.SCORE_COSINE if case[5] else mm.lib.SCORE_SCALED, mm.lib.MASK_SHIFT)
    assert name == "tcgen05"
    _check_win(mm, case, torch.bfloat16, cross, mm.lib.PATH_AUTO, oracle=nH <= 12)


GEN_DET_CASES = [CORE_CASES[0], CORE_CASES[1], CORE_CASES[2], CORE_CASES[5], CORE_CASES[7], CORE_CASES[9]]


@pytest.mark.parametrize("case", GEN_DET_CASES, ids=lambda c: f"g{'x'.join(map(str, c[0]))}_w{'x'.join(map(str, c[1]))}_h{c[3]}d{c[4]}_{c[6]}")
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
def test_winattn_bwd_generic_deterministic(mm, det, case, dtype):
    _check_win(mm, case, dtype, False, mm.lib.PATH_GENERIC)


# ------------------------------------------------------------------------------------------
# LayerNorm, column sums, projection bias, bias tables
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cols", [96, 768, 1536, 98])
@pytest.mark.parametrize("mode", [0, 1], ids=["pre", "post"])
def test_layernorm_bwd_deterministic(mm, det, cols, mode):
    g = torch.Generator().manual_seed(cols + mode)
    rows = 20000
    x = torch.randn(rows, cols, generator=g).cuda()
    r = torch.randn(rows, cols, generator=g).cuda()
    gamma, beta = (torch.randn(cols, generator=g) * 0.5 + 1).cuda(), torch.randn(cols, generator=g).cuda()
    gs, gn = torch.randn(rows, cols, generator=g).cuda(), torch.randn(rows, cols, generator=g).cuda()
    _, _, mean, rstd = torch.ops.mmn_b200.layernorm_fwd(r, x, gamma, beta, 1e-5, mode, True, mm.lib.DT_F32)
    xn = (x + r) if mode == 0 else x

    def bwd():
        return torch.ops.mmn_b200.layernorm_bwd(gs, gn, xn, gamma, mean, rstd, mode, mm.lib.DT_F32, mm.lib.DT_F32, True)
    _flag(False)
    ref = bwd()
    _flag(True)
    got = _repeat(bwd, f"layernorm bwd cols={cols}")
    for a, b in zip(got[:2], ref[:2]):
        assert torch.equal(a, b)
    xd = xn.double()
    xhat = (xd - xd.mean(1, keepdim=True)) / torch.sqrt(xd.var(1, unbiased=False, keepdim=True) + 1e-5)
    u = gn.double() if mode == 0 else gs.double() + gn.double()
    check(got[2], (u * xhat).sum(0), 1e-4, "dgamma")
    check(got[3], u.sum(0), 1e-4, "dbeta")
    check(got[2], ref[2], 1e-5, "dgamma vs default")


@pytest.mark.parametrize("cols", [8, 96, 392, 2048])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
def test_colsum_deterministic(mm, det, cols, dtype):
    x = torch.randn(50000, cols + 8, generator=torch.Generator().manual_seed(cols)).to(dtype).cuda()[:, :cols]
    got, = _repeat(lambda: (torch.ops.mmn_b200.colsum(x),), f"colsum {cols}")
    check(got, x.double().sum(0), 1e-5, "colsum")


def test_linear_bwd_general_and_fused_deterministic(mm, det):
    g = torch.Generator().manual_seed(7)
    for rows, n_in, n_out in ((3000, 64, 160), (3000, 96, 288)):        # dgrad + wgrad + column sums; the fused single pass
        x = torch.randn(rows, n_in, generator=g).bfloat16().cuda()
        w = (torch.randn(n_out, n_in, generator=g) * 0.1).bfloat16().cuda()
        dy = torch.randn(rows, n_out, generator=g).bfloat16().cuda()
        dx, dw, db = _repeat(lambda: torch.ops.mmn_b200.linear_bwd(dy, x, w), f"linear_bwd {n_in}->{n_out}")
        check(db, dy.double().sum(0), 1e-5, "db")
        check(dw, dy.double().t() @ x.double(), 1e-4, "dw")


@pytest.mark.parametrize("window,nH", [((4, 4, 4), 3), ((7, 7), 4), ((4, 4, 2), 48)], ids=["3d_w4", "2d_w7", "3d_442_48h"])
def test_table_bias_bwd_deterministic(mm, det, window, nH):
    from multimodal_neuroimage_b200 import geometry
    N, T = math.prod(window), math.prod(2 * w - 1 for w in window)
    index = geometry.relative_position_index(window).view(-1).cuda()
    cot = torch.randn(nH, N * N, generator=torch.Generator().manual_seed(N)).cuda()
    got, = _repeat(lambda: (torch.ops.mmn_b200.table_bias_bwd(cot, index, T),), "table bias bwd")
    want = torch.zeros(T, nH, dtype=torch.float64).index_add_(0, index.cpu(), cot.double().cpu().t())
    check(got, want, FP32_TOL, "table bias backward")


@pytest.mark.parametrize("window,nH", [((4, 4, 4), 3), ((8, 8), 6), ((16, 16), 6), ((7, 7, 7), 3), ((24, 24), 4)])
def test_cpb_bias_bwd_deterministic(mm, det, window, nH):
    from multimodal_neuroimage_b200 import geometry
    g = torch.Generator().manual_seed(nH + window[0])
    n = len(window)
    coords = geometry.cpb_coords_table(window).reshape(-1, n).float().cuda()
    index = geometry.relative_position_index(window).reshape(-1).cuda()
    w1, b1, w2 = (torch.randn(512, n, generator=g) * 0.7).cuda(), (torch.randn(512, generator=g) * 0.3).cuda(), \
        (torch.randn(nH, 512, generator=g) * 0.1).cuda()
    cot = torch.randn(nH, index.numel(), generator=g).cuda()
    _, tab16 = torch.ops.mmn_b200.cpb_bias_fwd(coords, w1, b1, w2, index)
    got = _repeat(lambda: torch.ops.mmn_b200.cpb_bias_bwd(cot, coords, w1, b1, w2, index, tab16), "cpb bias bwd")
    pd = [t.double().cpu().requires_grad_(True) for t in (w1, b1, w2)]
    tab = torch.relu(coords.double().cpu() @ pd[0].t() + pd[1]) @ pd[2].t()
    want = torch.autograd.grad(((16 * torch.sigmoid(tab))[index.cpu()].t() * cot.double().cpu()).sum(), pd)
    for a, b, nm in zip(got, want, ("dw1", "db1", "dw2")):
        check(a, b, 5e-5, "cpb " + nm)


def test_inverse_index_guard(mm, det):
    """An inverse that does not cover the index (offsets[T] != NN) poisons the table gradient instead of returning sums."""
    from multimodal_neuroimage_b200 import geometry
    index = geometry.relative_position_index((4, 4)).view(-1).cuda()
    T = 49
    perm, offsets = geometry.inverse_index(index, T)
    offsets = offsets.clone()
    offsets[-1] -= 1
    dtab = torch.empty(T, 2, device="cuda")
    lib = mm.lib.load()
    dbias = torch.randn(2, index.numel(), device="cuda")
    mm.lib.check(lib.mmn_table_bias_bwd(mm.ops._ptr(dbias), mm.ops._ptr(index), mm.ops._ptr(perm), mm.ops._ptr(offsets), T, 2,
                                        index.numel(), mm.ops._ptr(dtab), 0, mm.ops._stream(dbias)), "table_bias_bwd")
    assert torch.isnan(dtab).all()


def test_gather_rows_index_add_deterministic(mm, det):
    """_GatherRows (the CPB fallback when the fused kernel does not apply) scatters with index_add_, which PyTorch runs
    deterministically under the flag."""
    from multimodal_neuroimage_b200 import geometry
    index = geometry.relative_position_index((6, 6, 6)).view(-1).cuda()
    tab = torch.randn(11 ** 3, 3, device="cuda", requires_grad=True)
    cot = torch.randn(index.numel(), 3, device="cuda")
    _repeat(lambda: torch.autograd.grad((mm.v2._GatherRows.apply(tab, index) * cot).sum(), tab), "_GatherRows", graph=False)


def test_mha_bwd_is_deterministic(mm, det):
    """The MHA kernels use no atomics: the flag changes nothing and the gradients repeat bit for bit."""
    g = torch.Generator().manual_seed(1)
    q, k, v, do = (torch.randn(200, 2, 128, generator=g).bfloat16().cuda() for _ in range(4))
    out, lse = torch.ops.mmn_b200.mha_fwd(q, k, v, None, 4, mm.lib.MASK_NONE, 0, 32 ** -0.5, 0.0, 0, 0)
    _repeat(lambda: torch.ops.mmn_b200.mha_bwd(do, q, k, v, None, out, lse, 4, mm.lib.MASK_NONE, 0, 32 ** -0.5, 0.0, 0, 0), "mha bwd")


# ------------------------------------------------------------------------------------------
# selection: what reaches the C entry points
# ------------------------------------------------------------------------------------------
def test_selection_follows_the_flag(mm, monkeypatch):
    lib = mm.lib.load()
    seen = {}

    def spy(name, pick):
        real = getattr(lib, name)

        def f(*a):
            seen.setdefault(name, []).append(pick(a))
            return real(*a)
        monkeypatch.setattr(lib, name, f)

    spy("mmn_winattn_bwd", lambda a: ctypes.cast(a[0], ctypes.POINTER(mm.lib.WinAttnDesc)).contents.deterministic)
    spy("mmn_layernorm_bwd", lambda a: a[17])
    spy("mmn_colsum", lambda a: a[7])
    spy("mmn_linear_bwd", lambda a: a[17])
    spy("mmn_table_bias_bwd", lambda a: int(a[2] is not None))
    spy("mmn_cpb_bias_bwd", lambda a: int(a[5] is not None))
    from multimodal_neuroimage_b200 import geometry
    case = CORE_CASES[14]
    _, wbwd = _win_setup(mm, case, torch.bfloat16, False, mm.lib.PATH_AUTO)
    _, gbwd = _win_setup(mm, CORE_CASES[0], torch.float32, False, mm.lib.PATH_GENERIC)
    rows, cols = 4096, 96
    x, gn = torch.randn(rows, cols, device="cuda"), torch.randn(rows, cols, device="cuda")
    gamma = torch.ones(cols, device="cuda")
    _, _, mean, rstd = torch.ops.mmn_b200.layernorm_fwd(None, x, gamma, None, 1e-5, 0, False, mm.lib.DT_F32)
    dy = torch.randn(rows, 160, device="cuda").bfloat16()
    xb, w = torch.randn(rows, 64, device="cuda").bfloat16(), torch.randn(160, 64, device="cuda").bfloat16()
    index = geometry.relative_position_index((4, 4, 4)).view(-1).cuda()
    coords = geometry.cpb_coords_table((4, 4, 4)).reshape(-1, 3).float().cuda()
    w1, b1, w2 = torch.randn(512, 3, device="cuda"), torch.randn(512, device="cuda"), torch.randn(3, 512, device="cuda")
    _, tab16 = torch.ops.mmn_b200.cpb_bias_fwd(coords, w1, b1, w2, index)
    dbias = torch.randn(3, index.numel(), device="cuda")
    calls = [("tc", wbwd, 1), ("generic", gbwd, 2),
             ("ln", lambda: torch.ops.mmn_b200.layernorm_bwd(None, gn, x, gamma, mean, rstd, 0, -1, mm.lib.DT_F32, False), 1),
             ("colsum", lambda: torch.ops.mmn_b200.colsum(dy), 1),
             ("table", lambda: torch.ops.mmn_b200.table_bias_bwd(dbias, index, 343), 1),
             ("cpb", lambda: torch.ops.mmn_b200.cpb_bias_bwd(dbias, coords, w1, b1, w2, index, tab16), 2)]
    prev = torch.are_deterministic_algorithms_enabled()
    try:
        for on in (False, True):
            _flag(on)
            seen.clear()
            for name, fn, launches in calls:
                n0 = mm.lib.launch_count()
                fn()
                if not on:          # the default kernels, launched exactly as before deterministic mode existed
                    assert mm.lib.launch_count() - n0 == launches, name
            torch.ops.mmn_b200.linear_bwd(dy, xb, w)
            torch.cuda.synchronize()
            for name in ("mmn_winattn_bwd", "mmn_layernorm_bwd", "mmn_colsum", "mmn_linear_bwd", "mmn_table_bias_bwd", "mmn_cpb_bias_bwd"):
                assert seen.get(name) and all(v == int(on) for v in seen[name]), (on, name, seen.get(name))
    finally:
        _flag(prev)


def test_workspace_sizes_unchanged_with_the_flag_off(mm):
    lib = mm.lib.load()
    for case in (CORE_CASES[14], CORE_CASES[0]):
        grid, window, shift, nH, d = case[:5]
        a = torch.empty(case[7], *grid, 3 * nH * d, device="cuda", dtype=torch.bfloat16)
        desc, _ = mm.ops._win_desc(a, None, grid, window, shift, nH, 1, 1, 1, 1.0, 0.0, 0, 0, mm.lib.PATH_AUTO)
        n_lse = case[7] * math.prod(g // w for g, w in zip(grid, window)) * nH * math.prod(window)
        assert lib.mmn_winattn_bwd_workspace_bytes(ctypes.byref(desc)) == max(8 * n_lse, mm.lib.WINATTN_WORK_BYTES)
        desc.deterministic = 1
        assert lib.mmn_winattn_bwd_workspace_bytes(ctypes.byref(desc)) >= max(8 * n_lse, mm.lib.WINATTN_WORK_BYTES)
    assert lib.mmn_linear_bwd_workspace_bytes(5000, 64, 160, 0) <= lib.mmn_linear_bwd_workspace_bytes(5000, 64, 160, 1)


# ------------------------------------------------------------------------------------------
# whole training steps (subprocess: cuBLAS needs CUBLAS_WORKSPACE_CONFIG before it initialises)
# ------------------------------------------------------------------------------------------
_TRAIN_SCRIPT = r"""
import sys, torch
sys.path.insert(0, sys.argv[1])
from multimodal_neuroimage_b200 import train_step as TS, workloads as W
torch.use_deterministic_algorithms(True)
bce = torch.nn.functional.binary_cross_entropy_with_logits

def run(kind, use_graph):
    torch.manual_seed(0)
    if kind == "swinfusion":
        model = W.SwinFusion3D(img_size=32, Ex_depths=(2,), Fusion_depths=(2,), Re_depths=(2,))
        W.randomise_norms(model)
        model = model.cuda()
        A, B, y = W.synthetic_batch(2, 32, "cuda")
        ins = (A, B)
    else:
        model = W.FuncStructCross3D(img_size=32, fmri_layers=1, seq_len=48)
        W.randomise_norms(model)
        model = model.cuda()
        x_l, x_u, struct, y = W.synthetic_batch_cfg4(2, 32, "cuda", seq_len=48)
        ins = (x_l, x_u, struct)
    ts = TS.TrainStep(model, bce, ins, y, lr=1e-3, warmup=2, use_graph=use_graph)
    assert (ts.g_fb is not None) == use_graph
    losses = torch.stack([ts().detach().clone() for _ in range(4)])
    torch.cuda.synchronize()
    return losses, [p.detach().clone() for p in model.parameters()]

for kind in ("swinfusion", "cfg4"):
    for use_graph in (True, False):
        (l1, p1), (l2, p2) = run(kind, use_graph), run(kind, use_graph)
        assert torch.isfinite(l1).all() and l1[-1] < l1[0], (kind, l1)
        assert torch.equal(l1, l2), (kind, use_graph, l1, l2)
        assert len(p1) > 20 and all(torch.equal(a, b) for a, b in zip(p1, p2)), (kind, use_graph)
print("deterministic training steps OK")
"""


def test_training_steps_bit_identical():
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, CUBLAS_WORKSPACE_CONFIG=":4096:8")
    r = subprocess.run([sys.executable, "-c", _TRAIN_SCRIPT, root], env=env, capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0 and "OK" in r.stdout, r.stdout[-3000:] + r.stderr[-6000:]
