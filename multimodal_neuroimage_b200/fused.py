"""The window-attention MODULE as one autograd node: projection(s) -> fused shifted-window
attention kernel -> output projection, with a hand-written backward.

Why not leave it to autograd: F.linear's backward reduces its (tokens x channels) grad_output
over tokens to get the bias gradient with a generic reduction kernel -- 20 % of the step at
BASELINE cfg2.  Here the q/k/v bias gradients come out of the attention backward kernel for
free (column sums of dq, dk, dv, `dcolsum`), the output-projection bias gradient from a
memory-speed column-sum kernel, and nothing but the GEMMs (cuBLAS: plain library GEMMs) is left
to PyTorch.  Mirrors, for the self and the cross variant:
  reference swin_v2_module.py:147-176, swinfusion_module.py:121-143, 221-244.
"""
from __future__ import annotations

from typing import Optional

import torch
import torch.nn.functional as F

from . import _lib, ops  # noqa: F401  (ops registers torch.ops.mmn_b200.*)


def _mm_f32(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    """a @ b with fp32 output (weight gradients are accumulated over ~1e6 tokens)."""
    if a.dtype == torch.float32:
        return a @ b
    try:
        return torch.mm(a, b, out_dtype=torch.float32)
    except TypeError:
        return (a @ b).float()


def _project(x2: torch.Tensor, w: torch.Tensor, b) -> torch.Tensor:
    """x2 (rows, in) @ w^T + b.  bf16 with widths that are multiples of 32: the tensor-core projection kernel
    (csrc/gemm_tc.cu), bias added in fp32 in its epilogue; anything else (fp32 parity path, the reference's 12/24/48-wide
    stages): a plain library GEMM."""
    if ops.linear_supported(x2, w):
        return torch.ops.mmn_b200.linear_fwd(x2, w, None if b is None else b.float(), _lib.ACT_NONE, False)[0]
    return F.linear(x2, w, None if b is None else b.to(x2.dtype))


class WindowAttentionModuleFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, y, w_a, b_a, w_b, b_b, w_proj, b_proj, bias, head_scale, grid, window, shift, num_heads,
                score_kind, mask_kind, scale, dropout, path):
        """x (B, L, C) [queries; also keys/values when y is None]; y (B, L, C) or None.
        self:  w_a (3C, C), b_a (3C) | None;  w_b, b_b = None.
        cross: w_a (C, C) for q from x;  w_b (2C, C), b_b for kv from y."""
        odt = torch.get_autocast_dtype("cuda") if torch.is_autocast_enabled("cuda") else x.dtype
        cdt = torch.bfloat16 if odt == torch.float16 else odt     # fp16 autocast (trainer.py:378) runs as bf16 (ops.kernel_io)
        B, L, C = x.shape
        with torch.autocast("cuda", enabled=False):
            cast = lambda t: None if t is None else t.to(cdt)
            xc, yc = cast(x).reshape(B * L, C), (cast(y).reshape(B * L, C) if y is not None else None)
            castw = (lambda t: None if t is None else ops.weight_bf16(t)) if cdt == torch.bfloat16 else cast
            wa, wb, wp = castw(w_a), castw(w_b), castw(w_proj)       # biases stay in their own dtype: added in fp32
            p, seed, off, rng = dropout
            if y is None and cdt == torch.bfloat16 and xc.is_contiguous() and ops.winattn_qkv_path_name(
                    (B, *grid, C), cdt, grid, window, shift, num_heads, score_kind, mask_kind, p, path) == "tcgen05-fused":
                # one kernel: x read once, qkv written for the backward, the attention computed from it
                a, out, lse = torch.ops.mmn_b200.winattn_qkv_fwd(
                    xc.view(B, *grid, C), wa.contiguous(), None if b_a is None else b_a.float().contiguous(), bias,
                    head_scale, None, list(grid), list(window), list(shift), num_heads, score_kind, mask_kind, scale, path)
                b = None
            else:
                a = _project(xc, wa, b_a).view(B, *grid, -1)
                b = _project(yc, wb, b_b).view(B, *grid, -1) if y is not None else None
                out, lse = torch.ops.mmn_b200.winattn_fwd(a, b, bias, head_scale, None, list(grid), list(window), list(shift),
                                                          num_heads, score_kind, mask_kind, scale, p, seed, off, path, rng)
            res = _project(out.view(B * L, C), wp, b_proj).view(B, L, C).to(odt)
        ctx.save_for_backward(xc, yc, a, b, out, lse, wa, wb, wp, bias, head_scale, rng)
        ctx.cfg = (list(grid), list(window), list(shift), num_heads, score_kind, mask_kind, scale, p, seed, off, path)
        ctx.meta = (x.dtype, None if y is None else y.dtype, w_a.dtype, None if b_a is None else b_a.dtype,
                    None if w_b is None else w_b.dtype, None if b_b is None else b_b.dtype, w_proj.dtype,
                    None if b_proj is None else b_proj.dtype, (B, L, C))
        return res

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, dres):
        xc, yc, a, b, out, lse, wa, wb, wp, bias, head_scale, rng = ctx.saved_tensors
        xdt, ydt, wadt, badt, wbdt, bbdt, wpdt, bpdt, (B, L, C) = ctx.meta
        with torch.autocast("cuda", enabled=False):
            dy = dres.to(xc.dtype).reshape(B * L, C)
            if not dy.is_contiguous():
                dy = dy.contiguous()
            out2 = out.view(B * L, C)
            if ops.linear_bwd_supported(dy, out2, wp):
                # one pass over dy: dout = dy Wp, dWp = dy^T out, dbp = colsum(dy)  (libmmn_b200: linbwd_tc.cu)
                dout2, d_wp, d_bp = torch.ops.mmn_b200.linear_bwd(dy, out2, wp)
                dout = dout2.view(out.shape)
                d_wp = d_wp.to(wpdt)
                d_bp = d_bp.to(bpdt) if bpdt is not None else None
            else:
                d_bp = None
                if bpdt is not None:      # the column-sum kernel moves 8 columns per thread; odd widths are the reference's tiny stages
                    d_bp = (torch.ops.mmn_b200.colsum(dy) if C % 8 == 0 and C <= 2048 else dy.float().sum(0)).to(bpdt)
                d_wp = _mm_f32(dy.t(), out2).to(wpdt)
                dout = (dy @ wp).view(out.shape)
            da, db, dbias, dhs, dcs = torch.ops.mmn_b200.winattn_bwd(dout, a, b, bias, head_scale, None, out, lse, *ctx.cfg,
                                                                     True, rng)
            da2 = da.view(B * L, -1)
            if ops.linear_bwd_supported(da2, xc, wa):
                dx, d_wa, _ = torch.ops.mmn_b200.linear_bwd(da2, xc, wa)
                dx, d_wa = dx.view(B, L, C).to(xdt), d_wa.to(wadt)
            else:
                d_wa = _mm_f32(da2.t(), xc).to(wadt)
                dx = (da2 @ wa).view(B, L, C).to(xdt)
            if b is None:
                d_ba = dcs.reshape(-1).to(badt) if badt is not None else None
                d_y = d_wb = d_bb = None
            else:
                db2 = db.view(B * L, -1)
                d_ba = dcs[0].to(badt) if badt is not None else None
                d_bb = dcs[1:].reshape(-1).to(bbdt) if bbdt is not None else None
                if ops.linear_bwd_supported(db2, yc, wb):
                    d_y, d_wb, _ = torch.ops.mmn_b200.linear_bwd(db2, yc, wb)
                    d_y, d_wb = d_y.view(B, L, C).to(ydt), d_wb.to(wbdt)
                else:
                    d_wb = _mm_f32(db2.t(), yc).to(wbdt)
                    d_y = (db2 @ wb).view(B, L, C).to(ydt)
        return (dx, d_y, d_wa, d_ba, d_wb, d_bb, d_wp, d_bp, dbias if bias is not None else None,
                dhs if head_scale is not None else None) + (None,) * 9


def window_attention_module(x: torch.Tensor, y: Optional[torch.Tensor], w_a, b_a, w_b, b_b, w_proj, b_proj, bias, head_scale,
                            grid, window, shift, num_heads: int, score_kind: int, mask_kind: int, scale: float,
                            dropout=(0.0, 0, 0, None), path: int = 0) -> torch.Tensor:
    """dropout: (p, seed, offset, rng) as ops.next_dropout_stream returns it."""
    return WindowAttentionModuleFn.apply(x, y, w_a, b_a, w_b, b_b, w_proj, b_proj, bias, head_scale, tuple(grid), tuple(window),
                                         tuple(shift), num_heads, score_kind, mask_kind, float(scale), dropout, path)


class MlpFn(torch.autograd.Function):
    """fc1 -> activation -> fc2 (swin_v2_module.py:27-31, swinfusion_module.py:25-29, crossmodal_transformer.py:158-160) as
    two tensor-core GEMMs with the bias + activation in the first one's epilogue, and a three-GEMM-pass backward:
        dpre = (dy W2) o act'(pre)      dgrad of fc2; act'(pre) was written by fc1's forward epilogue next to act(pre)
        dW2  = dy^T h, db2              wgrad of fc2
        dx, dW1, db1                    backward of fc1 (one fused pass for in = 96)
    PyTorch runs this as 2 GEMMs + 1 elementwise kernel forward and 4 GEMMs + 3 elementwise/reduction kernels backward."""

    @staticmethod
    def forward(ctx, x, w1, b1, w2, b2, act):
        x2 = x.reshape(-1, x.shape[-1])
        w1c, w2c = ops.weight_bf16(w1), ops.weight_bf16(w2)
        h, dact = torch.ops.mmn_b200.linear_fwd(x2, w1c, None if b1 is None else b1.float(), act, True)   # act(pre), act'(pre)
        y, _ = torch.ops.mmn_b200.linear_fwd(h, w2c, None if b2 is None else b2.float(), _lib.ACT_NONE, False)
        ctx.save_for_backward(x2, dact, h, w1c, w2c)
        ctx.meta = (x.shape, w1.dtype, None if b1 is None else b1.dtype, w2.dtype, None if b2 is None else b2.dtype, act,
                    x.requires_grad)
        return y.view(*x.shape[:-1], w2.shape[0])

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, dy):
        x2, dact, h, w1c, w2c = ctx.saved_tensors
        shape, w1dt, b1dt, w2dt, b2dt, act, need_dx = ctx.meta
        dy2 = dy.reshape(-1, dy.shape[-1]).to(torch.bfloat16)
        if not dy2.is_contiguous():
            dy2 = dy2.contiguous()
        dpre, dw2, db2 = torch.ops.mmn_b200.linear_bwd(dy2, h, w2c, dact, act, True, True)
        dx, dw1, db1 = torch.ops.mmn_b200.linear_bwd(dpre, x2, w1c, None, 0, need_dx, True)
        return (dx.view(shape) if need_dx else None, dw1.to(w1dt), db1.to(b1dt) if b1dt is not None else None, dw2.to(w2dt),
                db2.to(b2dt) if b2dt is not None else None, None)


def mlp(x: torch.Tensor, fc1: torch.nn.Linear, fc2: torch.nn.Linear, act: str, drop: float = 0.0, training: bool = False,
        drop_out=None):
    """The Mlp of a block.  Fused path: CUDA, bf16 activations (autocast), widths multiples of 32, no dropout in
    between; otherwise the reference's own sequence of F.linear / activation / dropout.  `drop` follows the activation,
    `drop_out` (default: the same p, as in the Swin Mlp) follows fc2."""
    drop_out = drop if drop_out is None else drop_out
    cdt = torch.get_autocast_dtype("cuda") if torch.is_autocast_enabled("cuda") else x.dtype
    odt = cdt
    if cdt == torch.float16:
        cdt = torch.bfloat16
    widths_ok = all(d % 32 == 0 for d in (fc1.in_features, fc1.out_features, fc2.out_features))
    if x.is_cuda and cdt == torch.bfloat16 and widths_ok and x.numel() > 0 and not (training and (drop > 0.0 or drop_out > 0.0)):
        with torch.autocast("cuda", enabled=False):
            xc = x.to(torch.bfloat16)
            if not xc.is_contiguous():
                xc = xc.contiguous()
            return MlpFn.apply(xc, fc1.weight, fc1.bias, fc2.weight, fc2.bias, ops._ACT[act]).to(odt)
    h = fc1(x)
    h = F.gelu(h) if act == "gelu" else F.relu(h)
    h = F.dropout(h, drop, training)
    return F.dropout(fc2(h), drop_out, training)


# ------------------------------------------------------------------------------------------
# LayerNorm + residual add (csrc/layernorm.cu) -- the glue between the attention and Mlp calls of a block
# ------------------------------------------------------------------------------------------
def _ln_ok(x: torch.Tensor, ln) -> bool:
    return (isinstance(ln, torch.nn.LayerNorm) and ln.weight is not None and len(ln.normalized_shape) == 1
            and ops.layernorm_supported(x, x.shape[-1]) and ln.normalized_shape[0] == x.shape[-1])


def _act_dtype(x: torch.Tensor):
    """dtype of activations handed to the next GEMM: the autocast dtype (fp16 runs as bf16, ops.kernel_io), else x's own."""
    if torch.is_autocast_enabled("cuda"):
        dt = torch.get_autocast_dtype("cuda")
        return torch.bfloat16 if dt == torch.float16 else dt
    return x.dtype


def layer_norm(x: torch.Tensor, ln, out_dtype=None) -> torch.Tensor:
    """ln(x), emitted directly in the dtype the consumer wants (bf16 under autocast: no separate cast kernel)."""
    if not _ln_ok(x, ln):
        return ln(x)
    out_dtype = out_dtype or _act_dtype(x)
    with torch.autocast("cuda", enabled=False):
        return ops.AddLayerNormFn.apply(x, None, ln.weight, ln.bias, ln.eps, _lib.LN_PRE, out_dtype)[1]


def add_layer_norm(resid: torch.Tensor, delta: torch.Tensor, ln, out_dtype=None):
    """Pre-norm blocks: (s, ln(s)) with s = resid + delta, one pass (swinfusion_module.py:377-378,535-539)."""
    if not _ln_ok(resid, ln) or delta.dtype not in (torch.float32, torch.bfloat16) or delta.shape != resid.shape:
        s = resid + delta
        return s, ln(s)
    out_dtype = out_dtype or _act_dtype(resid)
    with torch.autocast("cuda", enabled=False):
        return ops.AddLayerNormFn.apply(resid, delta, ln.weight, ln.bias, ln.eps, _lib.LN_PRE, out_dtype)


def post_norm_add(resid: torch.Tensor, delta: torch.Tensor, ln, copy_dtype=None):
    """SwinV2 res-post-norm: s = resid + ln(delta) in one pass (swin_v2_module.py:299,302).  Returns (s, s cast to
    `copy_dtype`) -- the copy is what the next GEMM reads; None skips it."""
    if not _ln_ok(resid, ln) or delta.dtype not in (torch.float32, torch.bfloat16) or delta.shape != resid.shape:
        s = resid + ln(delta)
        return s, (s.to(copy_dtype) if copy_dtype is not None else None)
    with torch.autocast("cuda", enabled=False):
        return ops.AddLayerNormFn.apply(resid, delta, ln.weight, ln.bias, ln.eps, _lib.LN_POST, copy_dtype)


# ------------------------------------------------------------------------------------------
# Independent branches on two streams
# ------------------------------------------------------------------------------------------
PARALLEL_BRANCHES = False      # opt-in (bench / TrainStep switch it on): same arithmetic, two CUDA streams
_side_streams = {}


def parallel(fn_a, fn_b, ref: torch.Tensor, inputs_b=()):
    """(fn_a(), fn_b()) for two branches that do not depend on each other -- the two modalities' intra-modal groups
    (swinfusion_module.py:916-917; model.py's Ex_A / Ex_B stages).  With PARALLEL_BRANCHES on CUDA, fn_b is issued on a
    side stream forked from and joined back to the current one, so its kernels fill the SMs that fn_a's persistent
    kernels leave idle in their ramp-up and tail (at cfg3 a launch is 20-60 us of work: ~40 % of it is ramp and tail,
    tools/bench_blocks.py).  Autograd replays each branch's backward on the stream its forward ran on, and a CUDA-graph
    capture records the fork / join as parallel branches of the graph.  `inputs_b`: the tensors fn_b reads that were
    produced on the current stream -- the caching allocator is told that the side stream uses them too (and, below, that
    the current stream uses fn_b's results), so neither pool hands their memory out again while the other stream may still
    be reading it."""
    if not (PARALLEL_BRANCHES and ref.is_cuda):
        return fn_a(), fn_b()
    cur = torch.cuda.current_stream(ref.device)
    side = _side_streams.get(ref.device.index)
    if side is None:
        side = _side_streams[ref.device.index] = torch.cuda.Stream(ref.device)
    side.wait_stream(cur)
    for t in inputs_b:
        if isinstance(t, torch.Tensor):
            t.record_stream(side)
    with torch.cuda.stream(side):
        b = fn_b()
    a = fn_a()
    cur.wait_stream(side)
    for t in (b if isinstance(b, (tuple, list)) else (b,)):
        if isinstance(t, torch.Tensor):
            t.record_stream(cur)           # allocated from the side stream's pool, consumed on the current stream
    return a, b
