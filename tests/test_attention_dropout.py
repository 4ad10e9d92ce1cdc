"""Attention dropout against an exact host-side reference of its mask (oracle/philox.py, a transcription of
csrc/dropout_rng.cuh), and fresh masks on every CUDA-graph replay.

CPU: the Philox transcription reproduces Random123's known-answer vectors, the keep threshold is ceil(float32(p) * 2^24),
and a large oracle mask keeps 1 - thr / 2^24 of the probabilities.
GPU: every kernel that applies the mask -- generic and tensor-core multi-head attention, generic window attention, forward
and the transposed backward -- drops exactly the elements the oracle drops (read out bit for bit), outputs and gradients
match the fp64 oracle given that mask, the modules do the same with the stream they drew, and a captured CUDA graph draws
a new stream on every replay.
"""
import contextlib
import math

import numpy as np
import pytest
import torch

from oracle import philox as PH
from oracle import ref_nd as R
from test_deterministic import _repeat
from test_gpu_parity import BF16_TOL, CORE_CASES, FP32_TOL, _core_inputs, _oracle_core, check, rel_err

# seeds and offsets above 2^32: their high words only reach key.y
SEED = (0x5DEECE66D << 20) | 0x3B7
OFFSET = (0x2545F491 << 24) | 0x1F3
READOUT_P = [1e-7, 0.1, 0.5, 0.9]


# ------------------------------------------------------------------------------------------
# CPU: the reference itself
# ------------------------------------------------------------------------------------------
# Random123 kat_vectors, philox4x32-10
KAT = [((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
       ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
       ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
        (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1))]


@pytest.mark.parametrize("ctr,key,want", KAT, ids=["zeros", "ones", "pi"])
def test_philox_known_answer_vectors(ctr, key, want):
    assert tuple(int(w) for w in PH.philox4x32_10(ctr, key)) == want
    # vectorised: the same vector at every position of a batch
    batch = PH.philox4x32_10(np.tile(np.array(ctr, np.uint64), (5, 1)), np.array(key, np.uint64))
    assert (batch == np.array(want, np.uint32)).all()


@pytest.mark.parametrize("p,thr", [(0.1, 1677722), (0.3, 5033165), (0.5, 8388608), (1e-7, 2), (0.999, 16760439), (0.0, 0)])
def test_dropout_threshold(p, thr):
    assert PH.dropout_threshold(p) == thr


@pytest.mark.parametrize("p", [0.1, 0.5, 0.9])
def test_oracle_keep_rate_and_scale(p):
    m = PH.keep_table(p, SEED, OFFSET, 3, 300, 301)
    assert m.dtype == np.float32
    assert set(np.unique(m).tolist()) == {0.0, float(np.float32(1.0) / (np.float32(1.0) - np.float32(p)))}
    want = 1.0 - PH.dropout_threshold(p) / 2 ** 24
    rate = float((m > 0).mean())
    assert abs(rate - want) < 6 * math.sqrt(want * (1 - want) / m.size), (rate, want)
    # the element function agrees with the table, and every part of the stream matters
    idx = (np.array([0, 2, 1]), np.array([5, 299, 0]), np.array([7, 0, 300]))
    assert (PH.keep_scale(p, SEED, OFFSET, *idx) == m[idx]).all()
    for s, o in ((SEED ^ (1 << 40), OFFSET), (SEED ^ 1, OFFSET), (SEED, OFFSET ^ (1 << 40)), (SEED, OFFSET ^ 1)):
        assert (PH.keep_table(p, s, o, 3, 300, 301) != m).any()


# ------------------------------------------------------------------------------------------
# GPU fixtures and helpers
# ------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def mm():
    from multimodal_neuroimage_b200 import _lib, ops  # noqa: F401
    from multimodal_neuroimage_b200.modules import multihead_attention as mh
    from multimodal_neuroimage_b200.modules import swinfusion_module as fu
    _lib.load()
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False

    class NS:
        pass
    ns = NS()
    ns.lib, ns.ops, ns.mh, ns.fu = _lib, ops, mh, fu
    return ns


@pytest.fixture
def streams(mm, monkeypatch):
    """Records what every call of ops.next_dropout_stream returned."""
    rec = []
    orig = mm.ops.next_dropout_stream

    def spy(p, training, device):
        r = orig(p, training, device)
        rec.append(r)
        return r
    monkeypatch.setattr(mm.ops, "next_dropout_stream", spy)
    return rec


def _replay_stream(mm, monkeypatch, rec):
    """Make every module call use the recorded stream `rec` (as next_dropout_stream returned it)."""
    monkeypatch.setattr(mm.ops, "next_dropout_stream", lambda p, training, device: rec)


def _seed_offset(rec):
    """(seed, offset) of a stream next_dropout_stream returned: the device words when it drew them there."""
    rng = rec[3] if len(rec) > 3 else None
    return tuple(int(x) for x in rng.tolist()) if rng is not None else (rec[1], rec[2])


def _keep(p, seed, offset, items, nq, nk):
    return torch.from_numpy(PH.keep_table(p, seed, offset, items, nq, nk)).double()


def _rng(seed, offset):
    return torch.tensor([seed, offset], dtype=torch.int64, device="cuda")


@contextlib.contextmanager
def _deterministic():
    """torch.use_deterministic_algorithms(True) for the block: the window-attention backward then sums dbias, dhead_scale
    and dcolsum in a fixed order instead of with float atomics, so two runs can be compared bit for bit."""
    prev, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(prev, warn_only=warn)


def _mha_path(mm, T, S, B, nH, d, dtype, p, q):
    dsc = mm.lib.MhaDesc()
    dsc.tgt_len, dsc.src_len, dsc.batch, dsc.num_heads, dsc.head_dim = T, S, B, nH, d
    dsc.io_dtype = mm.lib.DT_BF16 if dtype == torch.bfloat16 else mm.lib.DT_F32
    dsc.dropout_p = p
    dsc.q_stride_t, dsc.q_stride_b = q.stride(0), q.stride(1)
    return mm.lib.load().mmn_mha_path(dsc).decode()


def _blocks(n, d):
    """Index blocks (positions, channels) of a one-hot readout: position blk * d + c in channel c."""
    for blk in range((n + d - 1) // d):
        pos = torch.arange(blk * d, min(n, blk * d + d))
        yield pos, pos - blk * d


# ------------------------------------------------------------------------------------------
# (a) the mask, bit for bit
# ------------------------------------------------------------------------------------------
# q = 0 makes every logit 0, so every kept probability is 1/S (nonzero) and every dropped one exactly 0; v one-hot over a
# block of keys (v[j, h*d + c] = 1 iff j = blk*d + c) puts P_ij keep_ij into out[i, h*d + c].  The backward: dout one-hot
# over a block of queries puts P_ij keep_ij of query i = blk*d + c into dv[j, h*d + c] (the dK / dV kernels regenerate the
# mask transposed).
MHA_READOUT = [("generic", torch.float32, 16), ("generic", torch.bfloat16, 16), ("tcgen05", torch.bfloat16, 32),
               ("tcgen05", torch.bfloat16, 64)]


@pytest.mark.gpu
@pytest.mark.parametrize("p", READOUT_P)
@pytest.mark.parametrize("path,dtype,d", MHA_READOUT, ids=["generic_fp32", "generic_bf16", "tcgen05_d32", "tcgen05_d64"])
def test_mha_mask_readout(mm, path, dtype, d, p):
    T, S, B, nH = 131, 257, 2, 3
    E, seed, off = nH * d, SEED + int(p * 1000), OFFSET
    q = torch.zeros(T, B, E, device="cuda", dtype=dtype)
    k = torch.randn(S, B, E, device="cuda").to(dtype)
    assert _mha_path(mm, T, S, B, nH, d, dtype, p, q) == path
    keep = PH.keep_table(p, seed, off, B * nH, T, S) != 0
    args = (mm.lib.MASK_NONE, 0, d ** -0.5, p)
    for n, (j, c) in enumerate(_blocks(S, d)):
        v = torch.zeros(S, B, nH, d, device="cuda", dtype=dtype)
        v[j, :, :, c] = 1
        v = v.view(S, B, E)
        # alternate the stream's form: ints, or device words read by the kernels
        stream = (seed, off) if n % 2 == 0 else (0, 0, _rng(seed, off))
        out, _ = torch.ops.mmn_b200.mha_fwd(q, k, v, None, nH, *args, *stream)
        got = (out.view(T, B, nH, d)[:, :, :, c] != 0).permute(1, 2, 0, 3).reshape(B * nH, T, len(c)).cpu().numpy()
        bad = got != keep[:, :, j.numpy()]
        assert not bad.any(), f"forward: {bad.sum()} elements of key block {n} disagree with the oracle mask"
    v = torch.randn(S, B, E, device="cuda").to(dtype)
    out, lse = torch.ops.mmn_b200.mha_fwd(q, k, v, None, nH, *args, seed, off)
    for n, (i, c) in enumerate(_blocks(T, d)):
        dout = torch.zeros(T, B, nH, d, device="cuda", dtype=dtype)
        dout[i, :, :, c] = 1
        stream = (seed, off) if n % 2 == 0 else (0, 0, _rng(seed, off))
        _, _, dv = torch.ops.mmn_b200.mha_bwd(dout.view(T, B, E), q, k, v, None, out, lse, nH, *args, *stream)
        got = (dv.view(S, B, nH, d)[:, :, :, c] != 0).permute(1, 2, 3, 0).reshape(B * nH, len(c), S).cpu().numpy()
        bad = got != keep[:, i.numpy(), :]
        assert not bad.any(), f"backward: {bad.sum()} elements of query block {n} disagree with the oracle mask"


WIN_READOUT = [((14, 14), (7, 7), (3, 3), 2, 8, 2), ((6, 6, 6), (3, 3, 3), (1, 2, 1), 3, 8, 2)]


def _windows(t, grid, window, shift, nH, d):
    """(B, *grid, C) -> (B*nW, N, nH, d) in the kernels' window order."""
    return R.window_partition_nd(R.cyclic_shift_nd(t, shift), window).reshape(-1, math.prod(window), nH, d)


def _unwindows(tw, grid, window, shift):
    C = tw.shape[2] * tw.shape[3]
    return R.cyclic_shift_nd(R.window_reverse_nd(tw.reshape(-1, *window, C), window, grid), shift, inverse=True)


@pytest.mark.gpu
@pytest.mark.parametrize("p", READOUT_P)
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
@pytest.mark.parametrize("geo", WIN_READOUT, ids=["2d", "3d"])
def test_winattn_mask_readout(mm, geo, dtype, p):
    grid, window, shift, nH, d, B = geo
    C, N, nW = nH * d, math.prod(window), math.prod(g // w for g, w in zip(grid, window))
    seed, off = SEED + int(p * 1000), OFFSET
    keep = PH.keep_table(p, seed, off, B * nW * nH, N, N) != 0
    qk = torch.cat([torch.zeros(B, *grid, C), torch.randn(B, *grid, C)], -1).to("cuda", dtype)
    cfg = (list(grid), list(window), list(shift), nH, mm.lib.SCORE_SCALED, mm.lib.MASK_NONE, d ** -0.5, p)
    for n, (j, c) in enumerate(_blocks(N, d)):
        vw = torch.zeros(B * nW, N, nH, d, device="cuda", dtype=dtype)
        vw[:, j, :, c] = 1
        a = torch.cat([qk, _unwindows(vw, grid, window, shift)], -1).contiguous()
        stream = (seed, off, mm.lib.PATH_AUTO) if n % 2 == 0 else (0, 0, mm.lib.PATH_AUTO, _rng(seed, off))
        out, _ = torch.ops.mmn_b200.winattn_fwd(a, None, None, None, None, *cfg, *stream)
        ow = _windows(out, grid, window, shift, nH, d)[:, :, :, c]                 # (B*nW, N, nH, len(c))
        got = (ow != 0).permute(0, 2, 1, 3).reshape(B * nW * nH, N, len(c)).cpu().numpy()
        bad = got != keep[:, :, j.numpy()]
        assert not bad.any(), f"forward: {bad.sum()} elements of key block {n} disagree with the oracle mask"
    a = torch.cat([qk, torch.randn(B, *grid, C).to("cuda", dtype)], -1).contiguous()
    out, lse = torch.ops.mmn_b200.winattn_fwd(a, None, None, None, None, *cfg, seed, off, mm.lib.PATH_AUTO)
    for n, (i, c) in enumerate(_blocks(N, d)):
        dw = torch.zeros(B * nW, N, nH, d, device="cuda", dtype=dtype)
        dw[:, i, :, c] = 1
        stream = (seed, off, mm.lib.PATH_AUTO) if n % 2 == 0 else (0, 0, mm.lib.PATH_AUTO, False, _rng(seed, off))
        da = torch.ops.mmn_b200.winattn_bwd(_unwindows(dw, grid, window, shift).contiguous(), a, None, None, None, None, out, lse,
                                            *cfg, *stream)[0]
        dvw = _windows(da[..., 2 * C:].contiguous(), grid, window, shift, nH, d)[:, :, :, c]    # (B*nW, N keys, nH, len(c))
        got = (dvw != 0).permute(0, 2, 3, 1).reshape(B * nW * nH, len(c), N).cpu().numpy()
        bad = got != keep[:, i.numpy(), :]
        assert not bad.any(), f"backward: {bad.sum()} elements of query block {n} disagree with the oracle mask"


# ------------------------------------------------------------------------------------------
# (b) numerics against fp64 with the oracle's mask
# ------------------------------------------------------------------------------------------
# cosine + shift (dhead_scale), scaled without a mask, the pre-windowed tensor mask, a tcgen05-shaped cfg2 geometry (runs
# generic with dropout), N = 512 (key chunking), d = 7
WIN_CASES = [CORE_CASES[0], CORE_CASES[1], CORE_CASES[9], CORE_CASES[5], CORE_CASES[12], CORE_CASES[13]]
WIN_IDS = ["cos_shift", "dot_none", "tensor_mask", "cfg2_cos_shift", "n512", "d7"]


def _win_items(case):
    grid, window, shift, nH, d, cosine, mask_mode, B = case
    return B * math.prod(g // w for g, w in zip(grid, window)) * nH, math.prod(window)


def _win_dropout_run(mm, case, dtype, cross, p, seed, off):
    """Kernel outputs (out, lse, da, db, dbias, dhead_scale, dcolsum) and their fp64 oracle values with the oracle mask."""
    grid, window, shift, nH, d, cosine, mask_mode, B = case
    a, b, bias, hs, mask, dout = _core_inputs(case, dtype, cross)
    items, N = _win_items(case)
    want = list(_oracle_core(case, a, b, bias, hs, mask, dout, keep=_keep(p, seed, off, items, N, N)))
    C = nH * d
    cs = want[2].reshape(-1, want[2].shape[-1]).sum(0)
    if b is not None:
        cs = torch.cat([cs, want[3].reshape(-1, want[3].shape[-1]).sum(0)])
    want.append(cs.view(3, C))
    kind = {"none": mm.lib.MASK_NONE, "shift": mm.lib.MASK_SHIFT, "tensor": mm.lib.MASK_TENSOR}[mask_mode]
    cfg = (list(grid), list(window), list(shift), nH, mm.lib.SCORE_COSINE if cosine else mm.lib.SCORE_SCALED, kind, d ** -0.5,
           p, seed, off, mm.lib.PATH_AUTO)
    ac, bc = a.to("cuda", dtype), (b.to("cuda", dtype) if b is not None else None)
    biasc, hsc = bias.cuda(), (hs.cuda() if hs is not None else None)
    maskc, doc = (mask.cuda() if mask is not None else None), dout.to("cuda", dtype)

    def run():
        out, lse = torch.ops.mmn_b200.winattn_fwd(ac, bc, biasc, hsc, maskc, *cfg)
        da, db, dbias, dhs, dcs = torch.ops.mmn_b200.winattn_bwd(doc, ac, bc, biasc, hsc, maskc, out, lse, *cfg, True)
        return out, lse[0], da, db, dbias, dhs, dcs
    return run, want


def _win_check(got, want, dtype, what):
    tol = FP32_TOL if dtype == torch.float32 else BF16_TOL
    for n, g_, w_ in zip(["out", "lse", "da", "db", "dbias", "dhead_scale"], got, want):
        if w_ is not None:
            check(g_, w_, tol, f"{what} {n}")
    check(got[6], want[6], tol * 10, f"{what} dcolsum")        # a column sum of ~1e3 gradient rows


@pytest.mark.gpu
@pytest.mark.parametrize("cross", [False, True], ids=["self", "cross"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
@pytest.mark.parametrize("case", WIN_CASES, ids=WIN_IDS)
def test_winattn_dropout_vs_oracle(mm, case, dtype, cross):
    run, want = _win_dropout_run(mm, case, dtype, cross, 0.3, SEED, OFFSET)
    _win_check(run(), want, dtype, f"{case} {dtype} cross={cross}")


@pytest.mark.gpu
@pytest.mark.parametrize("cross", [False, True], ids=["self", "cross"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
@pytest.mark.parametrize("case", WIN_CASES, ids=WIN_IDS)
def test_winattn_dropout_deterministic(mm, case, dtype, cross):
    """Under torch.use_deterministic_algorithms(True) (the fixed-order dbias / dhead_scale / dcolsum kernels): bit-repeatable
    and still the oracle's numbers."""
    run, want = _win_dropout_run(mm, case, dtype, cross, 0.5, SEED + 1, OFFSET)
    with _deterministic():
        got = _repeat(run, f"dropout {case} {dtype} cross={cross}")
    _win_check(got, want, dtype, f"deterministic {case} {dtype} cross={cross}")


def _mha_oracle(q, k, v, nH, scale, mask, keep):
    """fp64 core with the dropout mask: (out, lse, head-averaged dropped probabilities)."""
    T, B, E = q.shape
    S = k.shape[0]
    d = E // nH
    qh = (q * scale).reshape(T, B * nH, d).transpose(0, 1)
    kh = k.reshape(S, B * nH, d).transpose(0, 1)
    vh = v.reshape(S, B * nH, d).transpose(0, 1)
    s = qh @ kh.transpose(1, 2)
    if mask is not None:
        s = s + mask
    pd = torch.softmax(s, -1) * keep
    return (pd @ vh).transpose(0, 1).reshape(T, B, E), torch.logsumexp(s, -1), pd.view(B, nH, T, S).mean(1)


MHA_CASES = [  # path, dtype, d, nH, T, S, B, mask, packed
    ("generic", torch.float32, 16, 3, 131, 257, 2, "none", False),
    ("generic", torch.float32, 8, 2, 301, 301, 1, "future", True),
    ("generic", torch.float32, 16, 2, 130, 77, 2, "tensor", False),
    ("tcgen05", torch.bfloat16, 64, 2, 200, 333, 2, "none", False),
    ("tcgen05", torch.bfloat16, 32, 3, 300, 300, 2, "future", True),
    ("tcgen05", torch.bfloat16, 32, 2, 257, 130, 2, "tensor", False),
    ("tcgen05", torch.bfloat16, 64, 2, 129, 511, 1, "future", False)]


@pytest.mark.gpu
@pytest.mark.parametrize("p", [0.1, 0.5])
@pytest.mark.parametrize("case", MHA_CASES, ids=lambda c: f"{c[0]}_d{c[2]}_T{c[4]}_S{c[5]}_{c[7]}{'_packed' if c[8] else ''}")
def test_mha_dropout_vs_oracle(mm, case, p):
    path, dtype, d, nH, T, S, B, mask_kind, packed = case
    E, seed, off = d * nH, SEED + 7, OFFSET + int(p * 10)
    g = torch.Generator().manual_seed(T * 7 + S)
    if packed:
        qkv = torch.randn(T, B, 3 * E, generator=g).to(dtype)
        q, k, v = qkv.chunk(3, -1)
    else:
        q, k, v = (torch.randn(n, B, E, generator=g).to(dtype) for n in (T, S, S))
    cot = torch.randn(T, B, E, generator=g).to(dtype)
    diag = 1 + abs(S - T) if mask_kind == "future" else 0
    mask = None
    if mask_kind == "future":
        mask = R.future_mask(T, S, torch.float64)
    elif mask_kind == "tensor":
        mask = torch.randn(T, S, generator=g).double() * 2
        mask[torch.rand(T, S, generator=g) < 0.2] = float("-inf")
        mask[:, 0] = 0.0
    ins = [t.double().requires_grad_(True) for t in (q, k, v)]
    want, lse_w, avg_w = _mha_oracle(*ins, nH, d ** -0.5, mask, _keep(p, seed, off, B * nH, T, S))
    gw = torch.autograd.grad((want * cot.double()).sum(), ins)
    if packed:
        qkvc = qkv.cuda().requires_grad_(True)
        qc, kc, vc = qkvc.chunk(3, -1)
        leaves = [qkvc]
    else:
        qc, kc, vc = (t.cuda().requires_grad_(True) for t in (q, k, v))
        leaves = [qc, kc, vc]
    assert _mha_path(mm, T, S, B, nH, d, dtype, p, qc) == path
    kind = {"none": mm.lib.MASK_NONE, "future": mm.lib.MASK_FUTURE, "tensor": mm.lib.MASK_TENSOR}[mask_kind]
    mk = mask.float().cuda().contiguous() if mask_kind == "tensor" else None
    out, lse = torch.ops.mmn_b200.mha_fwd(qc, kc, vc, mk, nH, kind, diag, d ** -0.5, p, seed, off)
    gg = torch.autograd.grad((out.float() * cot.cuda().float()).sum(), leaves)
    if packed:
        gg = gg[0].chunk(3, -1)
    tol = FP32_TOL if dtype == torch.float32 else BF16_TOL
    check(out, want, tol, "out")
    check(lse.reshape(B * nH, T), lse_w, tol if dtype == torch.float32 else 1e-2, "lse")
    for a, b, n in zip(gg, gw, "qkv"):
        check(a, b, tol, "d" + n)
    avg = torch.ops.mmn_b200.mha_avg_weights(qc.detach(), kc.detach(), mk, lse, nH, kind, diag, d ** -0.5, p, seed, off)
    check(avg, avg_w, tol, "mha_avg_weights")


@pytest.mark.gpu
def test_device_stream_equals_int_stream(mm):
    """A device {seed, offset} gives bit for bit what the ints (seed, offset) give, on every kernel family."""
    rng = _rng(SEED, OFFSET)
    for dtype, d in ((torch.float32, 16), (torch.bfloat16, 64)):
        T, S, B, nH = 129, 200, 2, 2
        q, k, v = (torch.randn(n, B, nH * d, device="cuda").to(dtype).requires_grad_(True) for n in (T, S, S))
        cot = torch.randn(T, B, nH * d, device="cuda").to(dtype)
        res = []
        for stream in ((SEED, OFFSET), (0, 0, rng)):
            out, lse = torch.ops.mmn_b200.mha_fwd(q, k, v, None, nH, mm.lib.MASK_NONE, 0, d ** -0.5, 0.3, *stream)
            gs = torch.autograd.grad((out.float() * cot.float()).sum(), (q, k, v))
            avg = torch.ops.mmn_b200.mha_avg_weights(q.detach(), k.detach(), None, lse, nH, mm.lib.MASK_NONE, 0, d ** -0.5, 0.3,
                                                     *stream)
            res.append((out, lse, avg) + gs)
        for i, (x, y) in enumerate(zip(*res)):
            assert torch.equal(x, y), f"mha {dtype} output {i}"
    grid, window, shift, nH, d, cosine, mask_mode, B = CORE_CASES[5]
    a, b, bias, hs, mask, dout = _core_inputs(CORE_CASES[5], torch.bfloat16, True)
    ac, bc, doc = (t.to("cuda", torch.bfloat16) for t in (a, b, dout))
    biasc, hsc = bias.cuda(), hs.cuda()
    geo = (list(grid), list(window), list(shift), nH, mm.lib.SCORE_COSINE, mm.lib.MASK_SHIFT, d ** -0.5, 0.3)
    res = []
    for seed, off, rng_ in ((SEED, OFFSET, None), (0, 0, rng)):
        cfg = geo + (seed, off, mm.lib.PATH_AUTO)
        with _deterministic():
            out, lse = torch.ops.mmn_b200.winattn_fwd(ac, bc, biasc, hsc, None, *cfg, rng_)
            r = torch.ops.mmn_b200.winattn_bwd(doc, ac, bc, biasc, hsc, None, out, lse, *cfg, True, rng_)
        res.append((out, lse[0]) + tuple(r))
    for i, (x, y) in enumerate(zip(*res)):
        assert torch.equal(x, y), f"window attention output {i}"


# ------------------------------------------------------------------------------------------
# routing: window-attention dropout runs on the generic kernels
# ------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_winattn_dropout_routing(mm):
    case = CORE_CASES[5]                                      # cfg2 geometry: tcgen05 without dropout
    grid, window, shift, nH, d, cosine, mask_mode, B = case
    a, b, bias, hs, mask, dout = _core_inputs(case, torch.bfloat16, False)
    ac, doc = a.to("cuda", torch.bfloat16), dout.to("cuda", torch.bfloat16)
    geo = (list(grid), list(window), list(shift), nH, mm.lib.SCORE_COSINE, mm.lib.MASK_SHIFT)
    assert mm.ops.winattn_path_name(ac, None, *geo) == "tcgen05"
    assert mm.ops.winattn_path_name(ac, None, *geo, dropout_p=0.1) == "generic"
    res = {}
    for path in (mm.lib.PATH_AUTO, mm.lib.PATH_GENERIC):
        cfg = geo + (d ** -0.5, 0.1, SEED, OFFSET, path)
        with _deterministic():
            out, lse = torch.ops.mmn_b200.winattn_fwd(ac, None, bias.cuda(), hs.cuda(), None, *cfg)
            r = torch.ops.mmn_b200.winattn_bwd(doc, ac, None, bias.cuda(), hs.cuda(), None, out, lse, *cfg, True)
        res[path] = (out, lse[0], r[0], r[2], r[3], r[4])
    for i, (x, y) in enumerate(zip(res[mm.lib.PATH_AUTO], res[mm.lib.PATH_GENERIC])):
        assert torch.equal(x, y), f"AUTO with dropout differs from GENERIC in output {i}"
    with pytest.raises(RuntimeError, match="dropout"):
        torch.ops.mmn_b200.winattn_fwd(ac, None, bias.cuda(), hs.cuda(), None, *geo, d ** -0.5, 0.1, SEED, OFFSET,
                                       mm.lib.PATH_TCGEN05)


# ------------------------------------------------------------------------------------------
# (c) modules
# ------------------------------------------------------------------------------------------
def _sd64(module):
    return {k: (v.detach().double() if v.is_floating_point() else v.detach()).cpu() for k, v in module.state_dict().items()}


def _randomise(module, seed):
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for p in module.parameters():
            p.copy_(torch.randn(p.shape, generator=g) * 0.3)


@pytest.mark.gpu
def test_multihead_attention_module_dropout(mm, streams, monkeypatch):
    T, S, B, E, nH, p = 37, 45, 2, 48, 3, 0.3
    mod = mm.mh.MultiheadAttention(E, nH, attn_dropout=p)
    _randomise(mod, 1)
    sd = _sd64(mod)
    mod = mod.cuda().train()
    g = torch.Generator().manual_seed(2)
    x, y, cot = torch.randn(T, B, E, generator=g), torch.randn(S, B, E, generator=g), torch.randn(T, B, E, generator=g)
    xc, yc = x.cuda().requires_grad_(True), y.cuda().requires_grad_(True)
    out, w = mod(xc, yc, yc)
    params = [mod.in_proj_weight, mod.in_proj_bias, mod.out_proj.weight, mod.out_proj.bias]
    gg = torch.autograd.grad((out * cot.cuda()).sum(), [xc, yc] + params)
    assert len(streams) == 1 and streams[0][0] == p
    seed, off = _seed_offset(streams[0])
    leaves = [x.double().requires_grad_(True), y.double().requires_grad_(True)]
    sdl = {k: (v.requires_grad_(True) if v.is_floating_point() else v) for k, v in sd.items()}
    want, w_want = R.multihead_attention(leaves[0], leaves[1], leaves[1], sdl, nH, keep=_keep(p, seed, off, B * nH, T, S))
    gw = torch.autograd.grad((want * cot.double()).sum(),
                             leaves + [sdl["in_proj_weight"], sdl["in_proj_bias"], sdl["out_proj.weight"], sdl["out_proj.bias"]])
    check(out, want, FP32_TOL, "mha module out")
    check(w, w_want, FP32_TOL, "mha module weights")
    for a, b_, n in zip(gg, gw, ["x", "y", "in_proj_weight", "in_proj_bias", "out_proj.weight", "out_proj.bias"]):
        check(a, b_, FP32_TOL * 3, "mha module d" + n)
    # the same torch.manual_seed, the same result; another seed, another mask
    runs = []
    for s in (11, 11, 12):
        torch.manual_seed(s)
        runs.append(mod(xc, yc, yc)[0].detach())
    assert torch.equal(runs[0], runs[1]) and not torch.equal(runs[0], runs[2])
    # eval() drops nothing
    mod.eval()
    out_e, w_e = mod(xc, yc, yc)
    want_e, w_want_e = R.multihead_attention(x.double(), y.double(), y.double(), sd, nH)
    check(out_e, want_e, FP32_TOL, "mha module eval out")
    check(w_e, w_want_e, FP32_TOL, "mha module eval weights")


@pytest.mark.gpu
@pytest.mark.parametrize("grid,window,shift", [((12, 12), (6, 6), (3, 3)), ((8, 8, 8), (4, 4, 4), (2, 2, 2))], ids=["2d", "3d"])
def test_window_attention_module_dropout(mm, streams, grid, window, shift):
    C, nH, B, p = 24, 3, 2, 0.3
    mod = mm.fu.WindowAttention_fusion(C, window, nH, attn_drop=p)
    _randomise(mod, 3)
    sd = _sd64(mod)
    mod = mod.cuda().train()
    L = math.prod(grid)
    g = torch.Generator().manual_seed(4)
    x, cot = torch.randn(B, L, C, generator=g), torch.randn(B, L, C, generator=g)
    xc = x.cuda().requires_grad_(True)
    out = mod.forward_grid(xc, grid, shift)
    names = ["qkv.weight", "qkv.bias", "proj.weight", "proj.bias", "relative_position_bias_table"]
    pm = dict(mod.named_parameters())
    gg = torch.autograd.grad((out * cot.cuda()).sum(), [xc] + [pm[n] for n in names])
    assert len(streams) == 1
    seed, off = _seed_offset(streams[0])
    nW = math.prod(gi // w for gi, w in zip(grid, window))
    N = math.prod(window)
    xo = x.double().requires_grad_(True)
    sdl = {k: (v.requires_grad_(True) if v.is_floating_point() else v) for k, v in sd.items()}
    qkv = torch.nn.functional.linear(xo, sdl["qkv.weight"], sdl["qkv.bias"]).view(B, *grid, 3 * C)
    a, _ = R.window_attention_core(qkv[..., :C], qkv[..., C:2 * C], qkv[..., 2 * C:], grid, window, shift, nH, cosine=False,
                                   scale=(C // nH) ** -0.5, bias=R.table_bias(sdl, window),
                                   mask=R.shift_mask_nd(grid, window, shift, torch.float64),
                                   keep=_keep(p, seed, off, B * nW * nH, N, N))
    want = torch.nn.functional.linear(a.reshape(B, L, C), sdl["proj.weight"], sdl["proj.bias"])
    gw = torch.autograd.grad((want * cot.double()).sum(), [xo] + [sdl[n] for n in names])
    check(out, want, FP32_TOL, "window module out")
    for a_, b_, n in zip(gg, gw, ["x"] + names):
        check(a_, b_, FP32_TOL * 3, "window module d" + n)
    mod.eval()
    want_e = R.window_attention_core(*(t.detach() for t in (qkv[..., :C], qkv[..., C:2 * C], qkv[..., 2 * C:])), grid, window,
                                     shift, nH, cosine=False, scale=(C // nH) ** -0.5, bias=R.table_bias(sd, window),
                                     mask=R.shift_mask_nd(grid, window, shift, torch.float64))[0]
    want_e = torch.nn.functional.linear(want_e.reshape(B, L, C), sd["proj.weight"], sd["proj.bias"])
    check(mod.forward_grid(xc, grid, shift), want_e, FP32_TOL, "window module eval out")


@pytest.mark.gpu
def test_checkpointed_layer_matches_plain_layer_with_dropout(mm):
    """Activation checkpointing recomputes each block's forward in the backward: it must redraw the same dropout stream."""
    grid, C, nH = (8, 8), 24, 3
    layers = [mm.fu.BasicLayer_fusion(C, grid, 2, nH, 4, attn_drop=0.4, use_checkpoint=ck) for ck in (False, True)]
    _randomise(layers[0], 9)
    layers[1].load_state_dict(layers[0].state_dict())
    g = torch.Generator().manual_seed(10)
    x, cot = torch.randn(2, math.prod(grid), C, generator=g).cuda(), torch.randn(2, math.prod(grid), C, generator=g).cuda()
    res = []
    for layer in layers:
        layer = layer.cuda().train()
        xc = x.clone().requires_grad_(True)
        torch.manual_seed(21)
        out = layer(xc, grid)
        gs = torch.autograd.grad((out * cot).sum(), [xc] + list(layer.parameters()))
        res.append((out,) + gs)
    torch.manual_seed(22)
    other = layers[0](x, grid)
    assert rel_err(other, res[0][0]) > 1e-3                  # another seed: another mask
    check(res[1][0], res[0][0], FP32_TOL, "checkpointed vs plain out")
    for i, (a, b) in enumerate(zip(res[1][1:], res[0][1:])):
        check(a, b, FP32_TOL * 10, f"checkpointed vs plain, gradient {i}")


# ------------------------------------------------------------------------------------------
# (d) CUDA-graph replay draws a fresh mask
# ------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_graph_replay_draws_fresh_attention_dropout(mm, streams, monkeypatch):
    T, B, E, nH = 65, 2, 48, 3
    torch.manual_seed(0)
    mod = mm.mh.MultiheadAttention(E, nH, attn_dropout=0.5).cuda().train()
    params = list(mod.parameters())
    x = torch.randn(T, B, E, device="cuda")
    cot = torch.randn(T, B, E, device="cuda")

    def step():
        out, _ = mod(x, x, x, need_weights=False)
        (out * cot).sum().backward()
        return out

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            step()
    torch.cuda.current_stream().wait_stream(side)
    for p_ in params:
        p_.grad = None
    graph = torch.cuda.CUDAGraph()
    streams.clear()
    with torch.cuda.graph(graph):
        out = step()
    assert len(streams) == 1
    rec = streams[0]
    replays = []
    for _ in range(3):
        graph.replay()
        torch.cuda.synchronize()
        replays.append((tuple(t.clone() if torch.is_tensor(t) else t for t in rec), out.clone(),
                        [p_.grad.clone() for p_ in params]))
    for i in range(3):
        for j in range(i):
            assert not torch.equal(replays[i][1], replays[j][1]), f"replays {j} and {i} dropped the same attention probabilities"
    for rec_i, out_i, grads_i in replays:
        _replay_stream(mm, monkeypatch, rec_i)
        for p_ in params:
            p_.grad = None
        eager = step()
        check(out_i, eager, 1e-6, "replay vs eager out")
        for a, b in zip(grads_i, [p_.grad for p_ in params]):
            check(a, b, 1e-6, "replay vs eager grad")


class _AttnModel(torch.nn.Module):
    def __init__(self, mh, E, nH, p):
        super().__init__()
        self.attn = mh.MultiheadAttention(E, nH, attn_dropout=p)

    def forward(self, x):
        return self.attn(x, x, x, need_weights=False)[0]


@pytest.mark.gpu
@pytest.mark.parametrize("use_graph", [True, False], ids=["graph", "eager"])
def test_train_step_redraws_attention_dropout(mm, use_graph):
    """lr = 0 keeps the weights fixed: on a fixed batch only the dropout mask can change the loss from step to step."""
    from multimodal_neuroimage_b200 import train_step as TS
    torch.manual_seed(3)
    model = _AttnModel(mm.mh, 96, 3, 0.5).cuda().train()
    x, tgt = torch.randn(130, 4, 96, device="cuda"), torch.randn(130, 4, 96, device="cuda")
    step = TS.TrainStep(model, lambda out, t: ((out - t) ** 2).mean(), [x], tgt, lr=0.0, weight_decay=0.0, use_graph=use_graph)
    assert (step.g_fb is not None) == use_graph
    w0 = [p_.detach().clone() for p_ in model.parameters()]
    losses = [step().item() for _ in range(4)]
    assert len(set(losses)) == len(losses), f"steps repeated a dropout mask: losses {losses}"
    assert all(torch.equal(a, b) for a, b in zip(w0, model.parameters()))
