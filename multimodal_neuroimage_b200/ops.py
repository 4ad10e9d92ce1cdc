"""torch.library custom ops over the C ABI (include/mmn_b200.h).

PyTorch is plumbing here: it owns device memory and streams and records the autograd
graph; the arithmetic happens in libmmn_b200.so.  Ops:

  mmn_b200::winattn_fwd / winattn_bwd   fused shift + window gather + attention + scatter
  mmn_b200::mha_fwd / mha_bwd           (T,B,E) multi-head attention core
  mmn_b200::mha_avg_weights             head-averaged probabilities

Under `torch.use_deterministic_algorithms(True)` the backward ops select the library's deterministic kernels (fixed-order
reductions instead of float atomics), as PyTorch's own ops do; the flag is read when the op runs, so a CUDA graph
captured with it on replays them.

Window attention takes its q/k/v in one of two packings so that the backward can write one
packed gradient tensor (no slice-backward copies):
  a = qkv (..., 3C), b = None            self attention   (swin_v2 / swinfusion self)
  a = q   (..., C),  b = kv (..., 2C)    cross attention  (swinfusion Cross_WindowAttention)
All tensors are in the un-windowed, un-shifted (B, *grid, channels) order.
"""
from __future__ import annotations

import ctypes as C
import functools
from typing import List, Optional, Tuple

import torch

from . import _lib, geometry
from ._lib import MhaDesc, WinAttnDesc

Tensor = torch.Tensor

_DT = {torch.float32: _lib.DT_F32, torch.bfloat16: _lib.DT_BF16}


def kernel_io(t: Optional[Tensor]) -> Optional[Tensor]:
    """Activation dtype the kernels run in.  The kernels take float32 and bfloat16; float16 -- what the reference
    trainer's `torch.cuda.amp.autocast()` produces (trainer.py:378, `--amp` default on, main.py:88) -- goes through them
    as bfloat16 (same 16-bit traffic, fp32 softmax / accumulation inside; the caller casts the result back)."""
    return t.to(torch.bfloat16) if t is not None and t.dtype == torch.float16 else t


# ------------------------------------------------------------------------------------------
# bf16 copies of the master weights
# ------------------------------------------------------------------------------------------
# Every projection casts its fp32 master weight to bf16 on the way in: one tiny kernel per weight and step (276 of them in
# the cfg3 step, ~2.5 us each even inside a CUDA graph).  A training loop that owns the optimizer step can keep the copies
# alive instead and refresh them all with one multi-tensor copy after the step (train_step.TrainStep does).  A copy is
# used only while the weight's version counter is the one seen at the last refresh: load_state_dict, .to(), or any other
# in-place update from outside invalidates it by construction and the cast happens as before.
# (Writes through `w.data` have their own version counter and are NOT seen: refresh() after them, as TrainStep does after
# broadcasting the initial weights.)
_BF16_SHADOWS = {}


def weight_bf16(w: Tensor) -> Tensor:
    """w as bfloat16: w itself, its registered up-to-date copy, or a fresh cast."""
    if w.dtype == torch.bfloat16:
        return w
    hit = _BF16_SHADOWS.get(id(w))
    if hit is not None and hit[0]() is w and hit[2] == w._version:
        return hit[1]
    return w.to(torch.bfloat16)


class Bf16Shadows:
    """bf16 copies of the (>= 2-D, fp32) parameters in `params`, served by `weight_bf16`.  Call refresh() after every
    update of the parameters (inside a CUDA-graph capture of the optimizer step it is captured with it)."""

    def __init__(self, params):
        import weakref
        self._ref = weakref.ref
        self.src = [p for p in params if p.dtype == torch.float32 and p.dim() >= 2]
        self.dst = [torch.empty_like(p, dtype=torch.bfloat16) for p in self.src]
        self.refresh()

    def refresh(self):
        if not self.src:
            return
        with torch.no_grad():
            torch._foreach_copy_(self.dst, self.src)
        for p, d in zip(self.src, self.dst):
            key = id(p)
            # the entry (and the copy it holds) goes when the weight does
            _BF16_SHADOWS[key] = (self._ref(p, lambda _r, key=key: _BF16_SHADOWS.pop(key, None)), d, p._version)

    def close(self):
        for p in self.src:
            hit = _BF16_SHADOWS.get(id(p))
            if hit is not None and hit[0]() is p:
                del _BF16_SHADOWS[id(p)]
        self.src, self.dst = [], []


def _require_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("multimodal_neuroimage_b200 ops run on CUDA tensors only (there is no CPU path); "
                               f"got a tensor on {t.device}")


def _ptr(t: Optional[Tensor], elem_offset: int = 0):
    if t is None:
        return None
    return C.c_void_p(t.data_ptr() + elem_offset * t.element_size())


def _row_stride(t: Tensor) -> int:
    """Element stride between consecutive tokens of a (..., channels) tensor whose leading
    dims collapse to one uniform stride (true for contiguous tensors and channel slices)."""
    if t.stride(-1) != 1:
        raise RuntimeError("channel dimension must be contiguous")
    rs = t.stride(-2)
    exp = rs
    for i in range(t.dim() - 2, -1, -1):
        if t.shape[i] != 1 and t.stride(i) != exp:
            raise RuntimeError(f"token rows are not uniformly strided: shape {tuple(t.shape)} strides {t.stride()}")
        exp *= t.shape[i]
    return rs


def _stream(t: Tensor):
    return C.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)


def _deterministic() -> bool:
    return torch.are_deterministic_algorithms_enabled()


def _workspace(nbytes: int, like: Tensor) -> Tensor:
    return torch.empty((nbytes + 3) // 4, dtype=torch.float32, device=like.device)


# Inverse of a bias-table index (geometry.inverse_index) for the deterministic table-gradient gather, per index tensor.  The
# entry keeps the index alive, so its address cannot be reused by another index while the entry exists; an in-place write
# to the index bumps its version and misses.  Inverses built during graph capture are not cached (their values only exist
# once the graph replays).
_INVERSE = {}


def _inverse_index(index: Tensor, T: int) -> Tuple[Tensor, Tensor]:
    key = (index.device, index.data_ptr(), index.numel(), index._version, T)
    hit = _INVERSE.get(key)
    if hit is not None:
        return hit[1], hit[2]
    perm, offsets = geometry.inverse_index(index.reshape(-1), T)
    if not torch.cuda.is_current_stream_capturing():
        _INVERSE[key] = (index, perm, offsets)
    return perm, offsets


# Optional live kernel timing (bench.py): when KERNEL_EVENTS is a dict, every C call is
# bracketed by CUDA events recorded on the launching stream and appended under its name.
KERNEL_EVENTS = None


class _timed:
    def __init__(self, name, t):
        self.name, self.t = name, t

    def __enter__(self):
        if KERNEL_EVENTS is not None:
            self.e0 = torch.cuda.Event(enable_timing=True)
            self.e1 = torch.cuda.Event(enable_timing=True)
            self.e0.record(torch.cuda.current_stream(self.t.device))

    def __exit__(self, *exc):
        if KERNEL_EVENTS is not None:
            self.e1.record(torch.cuda.current_stream(self.t.device))
            KERNEL_EVENTS.setdefault(self.name, []).append((self.e0, self.e1))
        return False


def _rng_ptr(rng: Optional[Tensor], like: Tensor) -> Optional[int]:
    """Device address of a dropout stream {seed, offset} (next_dropout_stream), or None."""
    if rng is None:
        return None
    if rng.dtype != torch.int64 or rng.numel() != 2 or not rng.is_contiguous() or rng.device != like.device:
        raise RuntimeError("rng must be a contiguous (2,) int64 tensor {seed, offset} on the attention's device")
    return rng.data_ptr()


def _win_desc(a: Tensor, b: Optional[Tensor], grid, window, shift, num_heads, score_kind, mask_kind, mask_windows,
              scale, dropout_p, seed, offset, path, rng=None) -> Tuple[WinAttnDesc, int]:
    n = len(grid)
    if a.dtype not in _DT:
        raise RuntimeError(f"unsupported dtype {a.dtype}: the window-attention kernels take float32 or bfloat16")
    Cc = a.shape[-1] // 3 if b is None else a.shape[-1]
    if Cc % num_heads:
        raise RuntimeError("channels not divisible by heads")
    d = WinAttnDesc()
    d.ndim, d.batch = n, a.shape[0]
    for i in range(n):
        d.grid[i], d.window[i], d.shift[i] = int(grid[i]), int(window[i]), int(shift[i])
    d.num_heads, d.head_dim = num_heads, Cc // num_heads
    d.score_kind, d.mask_kind, d.mask_windows = score_kind, mask_kind, mask_windows
    d.io_dtype, d.path = _DT[a.dtype], path
    d.scale, d.dropout_p, d.seed, d.offset = scale, dropout_p, seed, offset
    d.rng = _rng_ptr(rng, a)
    return d, Cc


@torch.library.custom_op("mmn_b200::winattn_fwd", mutates_args=())
def winattn_fwd(a: Tensor, b: Optional[Tensor], bias: Optional[Tensor], head_scale: Optional[Tensor],
                mask: Optional[Tensor], grid: List[int], window: List[int], shift: List[int], num_heads: int,
                score_kind: int, mask_kind: int, scale: float, dropout_p: float, seed: int, offset: int,
                path: int, rng: Optional[Tensor] = None) -> Tuple[Tensor, Tensor]:
    """rng: None, or a device {seed, offset} (next_dropout_stream) that replaces seed / offset."""
    _require_cuda(a, b, bias, head_scale, mask)
    lib = _lib.load()
    d, Cc = _win_desc(a, b, grid, window, shift, num_heads, score_kind, mask_kind,
                      mask.shape[0] if mask is not None else 0, scale, dropout_p, seed, offset, path, rng)
    if tuple(a.shape[1:-1]) != tuple(grid):
        raise RuntimeError(f"tensor grid {tuple(a.shape[1:-1])} != geometry {tuple(grid)}")
    out = torch.empty(*a.shape[:-1], Cc, dtype=a.dtype, device=a.device)
    N = 1
    nW = 1
    for g, w in zip(grid, window):
        N *= w
        nW *= g // w
    # four slabs.  [0]: log-sum-exp (B*nW, nH, N) by window position.  [1:4]: one record per window and head,
    # (B*nW, nH, 3, N) = 1/max(||q||,eps) | 1/max(||k||,eps) | log2-domain lse in the kernel's tile row order, written
    # by the tensor-core forward kernel for its backward kernel; the generic kernels use slab 0 only.
    lse = torch.empty(4, a.shape[0] * nW, num_heads, N, dtype=torch.float32, device=a.device)
    if b is None:
        q, k, v = _ptr(a), _ptr(a, Cc), _ptr(a, 2 * Cc)
        d.q_row_stride = d.k_row_stride = d.v_row_stride = _row_stride(a)
    else:
        q, k, v = _ptr(a), _ptr(b), _ptr(b, Cc)
        d.q_row_stride = _row_stride(a)
        d.k_row_stride = d.v_row_stride = _row_stride(b)
    d.o_row_stride = Cc
    for t in (bias, head_scale, mask):
        if t is not None and (t.dtype != torch.float32 or not t.is_contiguous()):
            raise RuntimeError("bias / head_scale / mask must be contiguous float32")
    work = torch.empty(_lib.WINATTN_WORK_BYTES, dtype=torch.uint8, device=a.device)   # this launch's work-queue counters
    with _timed("winattn_fwd", a):
        _lib.check(lib.mmn_winattn_fwd(C.byref(d), q, k, v, _ptr(bias), _ptr(head_scale), _ptr(mask), _ptr(out),
                                       _ptr(lse), _ptr(work), a.device.index, _stream(a)), "mmn_winattn_fwd")
    return out, lse


@winattn_fwd.register_fake
def _(a, b, bias, head_scale, mask, grid, window, shift, num_heads, score_kind, mask_kind, scale, dropout_p, seed,
      offset, path, rng=None):
    Cc = a.shape[-1] // 3 if b is None else a.shape[-1]
    N = nW = 1
    for g, w in zip(grid, window):
        N *= w
        nW *= g // w
    return a.new_empty(*a.shape[:-1], Cc), a.new_empty(4, a.shape[0] * nW, num_heads, N, dtype=torch.float32)


@torch.library.custom_op("mmn_b200::winattn_qkv_fwd", mutates_args=())
def winattn_qkv_fwd(x: Tensor, w: Tensor, b: Optional[Tensor], bias: Optional[Tensor], head_scale: Optional[Tensor],
                    mask: Optional[Tensor], grid: List[int], window: List[int], shift: List[int], num_heads: int,
                    score_kind: int, mask_kind: int, scale: float, path: int) -> Tuple[Tensor, Tensor, Tensor]:
    """Self-attention forward with the qkv projection fused in (csrc/winattn_tc_qkv_fwd.cuh).  x (B, *grid, C) bf16,
    w (3C, C) bf16, b (3C) fp32 or None.  Returns (qkv, out, lse): qkv = x w^T + b in bf16, the packed (B, *grid, 3C)
    tensor winattn_bwd takes as `a`; out and lse as winattn_fwd computes them from that qkv.  Only shapes for which
    winattn_qkv_path_name says "tcgen05-fused"."""
    _require_cuda(x, w, b, bias, head_scale, mask)
    Cc = x.shape[-1]
    if x.dtype != torch.bfloat16 or w.dtype != torch.bfloat16 or not x.is_contiguous() or not w.is_contiguous() \
            or tuple(w.shape) != (3 * Cc, Cc):
        raise RuntimeError("winattn_qkv_fwd expects contiguous bf16 x (..., C) and w (3C, C)")
    if b is not None and (b.dtype != torch.float32 or not b.is_contiguous() or b.numel() != 3 * Cc):
        raise RuntimeError("winattn_qkv_fwd takes its qkv bias as a contiguous float32 (3C) tensor")
    if tuple(x.shape[1:-1]) != tuple(grid):
        raise RuntimeError(f"tensor grid {tuple(x.shape[1:-1])} != geometry {tuple(grid)}")
    for t in (bias, head_scale, mask):
        if t is not None and (t.dtype != torch.float32 or not t.is_contiguous()):
            raise RuntimeError("bias / head_scale / mask must be contiguous float32")
    qkv = torch.empty(*x.shape[:-1], 3 * Cc, dtype=x.dtype, device=x.device)
    d, _ = _win_desc(qkv, None, grid, window, shift, num_heads, score_kind, mask_kind,
                     mask.shape[0] if mask is not None else 0, scale, 0.0, 0, 0, path)
    d.q_row_stride = d.k_row_stride = d.v_row_stride = 3 * Cc
    d.o_row_stride = Cc
    out = torch.empty_like(x)
    N = nW = 1
    for g, w_ in zip(grid, window):
        N *= w_
        nW *= g // w_
    lse = torch.empty(4, x.shape[0] * nW, num_heads, N, dtype=torch.float32, device=x.device)   # as winattn_fwd
    work = torch.empty(_lib.WINATTN_WORK_BYTES, dtype=torch.uint8, device=x.device)
    with _timed("winattn_qkv_fwd", x):
        _lib.check(_lib.load().mmn_winattn_qkv_fwd(C.byref(d), _ptr(x), _ptr(w), _ptr(b), _ptr(bias), _ptr(head_scale),
                                                   _ptr(mask), _ptr(qkv), _ptr(out), _ptr(lse), _ptr(work), x.device.index,
                                                   _stream(x)), "mmn_winattn_qkv_fwd")
    return qkv, out, lse


@winattn_qkv_fwd.register_fake
def _(x, w, b, bias, head_scale, mask, grid, window, shift, num_heads, score_kind, mask_kind, scale, path):
    N = nW = 1
    for g, w_ in zip(grid, window):
        N *= w_
        nW *= g // w_
    return (x.new_empty(*x.shape[:-1], 3 * x.shape[-1]), x.new_empty(x.shape),
            x.new_empty(4, x.shape[0] * nW, num_heads, N, dtype=torch.float32))


@torch.library.custom_op("mmn_b200::winattn_bwd", mutates_args=())
def winattn_bwd(dout: Tensor, a: Tensor, b: Optional[Tensor], bias: Optional[Tensor], head_scale: Optional[Tensor],
                mask: Optional[Tensor], out: Tensor, lse: Tensor, grid: List[int], window: List[int], shift: List[int],
                num_heads: int, score_kind: int, mask_kind: int, scale: float, dropout_p: float, seed: int,
                offset: int, path: int, want_colsum: bool = False,
                rng: Optional[Tensor] = None) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor]:
    """Returns (da, db, dbias, dhead_scale, dcolsum); unused ones are empty tensors.  dcolsum (3, C) fp32 =
    column sums over all tokens of dq, dk, dv, i.e. the bias gradients of the q/k/v projections.  rng: the forward's."""
    _require_cuda(dout, a, b, bias, head_scale, mask, out, lse)
    lib = _lib.load()
    d, Cc = _win_desc(a, b, grid, window, shift, num_heads, score_kind, mask_kind,
                      mask.shape[0] if mask is not None else 0, scale, dropout_p, seed, offset, path, rng)
    dout = dout.contiguous()
    da = torch.empty(a.shape, dtype=a.dtype, device=a.device)
    db = torch.empty(b.shape, dtype=b.dtype, device=b.device) if b is not None else a.new_empty(0)
    if b is None:
        q, k, v = _ptr(a), _ptr(a, Cc), _ptr(a, 2 * Cc)
        dq, dk, dv = _ptr(da), _ptr(da, Cc), _ptr(da, 2 * Cc)
        d.q_row_stride = d.k_row_stride = d.v_row_stride = _row_stride(a)
        d.dq_row_stride = d.dk_row_stride = d.dv_row_stride = 3 * Cc
    else:
        q, k, v = _ptr(a), _ptr(b), _ptr(b, Cc)
        dq, dk, dv = _ptr(da), _ptr(db), _ptr(db, Cc)
        d.q_row_stride = _row_stride(a)
        d.k_row_stride = d.v_row_stride = _row_stride(b)
        d.dq_row_stride = Cc
        d.dk_row_stride = d.dv_row_stride = 2 * Cc
    d.o_row_stride = _row_stride(out)
    d.do_row_stride = Cc
    d.deterministic = int(_deterministic())
    dbias = torch.zeros_like(bias) if bias is not None else a.new_empty(0, dtype=torch.float32)
    dhs = torch.zeros_like(head_scale) if head_scale is not None else a.new_empty(0, dtype=torch.float32)
    ws = _workspace(lib.mmn_winattn_bwd_workspace_bytes(C.byref(d)), lse)
    dcs = torch.zeros(3, Cc, dtype=torch.float32, device=a.device) if want_colsum else a.new_empty(0, dtype=torch.float32)
    with _timed("winattn_bwd", a):
        _lib.check(lib.mmn_winattn_bwd(C.byref(d), q, k, v, _ptr(bias), _ptr(head_scale), _ptr(mask), _ptr(out), _ptr(lse),
                                       _ptr(dout), dq, dk, dv, _ptr(dbias) if bias is not None else None,
                                       _ptr(dhs) if head_scale is not None else None, _ptr(dcs) if want_colsum else None,
                                       _ptr(ws), a.device.index, _stream(a)), "mmn_winattn_bwd")
    return da, db, dbias, dhs, dcs


@winattn_bwd.register_fake
def _(dout, a, b, bias, head_scale, mask, out, lse, grid, window, shift, num_heads, score_kind, mask_kind, scale,
      dropout_p, seed, offset, path, want_colsum=False, rng=None):
    Cc = a.shape[-1] // 3 if b is None else a.shape[-1]
    return (torch.empty_like(a), torch.empty_like(b) if b is not None else a.new_empty(0),
            torch.empty_like(bias) if bias is not None else a.new_empty(0, dtype=torch.float32),
            torch.empty_like(head_scale) if head_scale is not None else a.new_empty(0, dtype=torch.float32),
            a.new_empty((3, Cc) if want_colsum else (0,), dtype=torch.float32))


def _winattn_setup(ctx, inputs, output):
    (a, b, bias, head_scale, mask, grid, window, shift, num_heads, score_kind, mask_kind, scale, dropout_p, seed,
     offset, path, rng) = inputs
    out, lse = output
    ctx.save_for_backward(a, b, bias, head_scale, mask, out, lse, rng)
    ctx.cfg = (grid, window, shift, num_heads, score_kind, mask_kind, scale, dropout_p, seed, offset, path)


def _winattn_backward(ctx, dout, dlse):
    a, b, bias, head_scale, mask, out, lse, rng = ctx.saved_tensors
    da, db, dbias, dhs, _ = torch.ops.mmn_b200.winattn_bwd(dout, a, b, bias, head_scale, mask, out, lse, *ctx.cfg, False, rng)
    return (da, db if b is not None else None, dbias if bias is not None else None,
            dhs if head_scale is not None else None, None) + (None,) * 12


torch.library.register_autograd("mmn_b200::winattn_fwd", _winattn_backward, setup_context=_winattn_setup)


# ------------------------------------------------------------------------------------------
# multi-head attention
# ------------------------------------------------------------------------------------------
def _tb_strides(t: Tensor) -> Tuple[int, int]:
    if t.dim() != 3 or t.stride(2) != 1:
        raise RuntimeError("expected a (len, batch, embed) tensor with contiguous embed dimension")
    return t.stride(0), t.stride(1)


def _mha_desc(q, k, num_heads, mask_kind, mask_diag, scale, dropout_p, seed, offset, rng=None) -> MhaDesc:
    if q.dtype not in _DT:
        raise RuntimeError(f"unsupported dtype {q.dtype}: the attention kernels take float32 or bfloat16")
    d = MhaDesc()
    d.tgt_len, d.batch, E = q.shape
    d.src_len = k.shape[0]
    if E % num_heads:
        raise RuntimeError("embed_dim not divisible by heads")
    d.num_heads, d.head_dim = num_heads, E // num_heads
    d.mask_kind, d.mask_diagonal = mask_kind, mask_diag
    d.io_dtype, d.path = _DT[q.dtype], _lib.PATH_AUTO
    d.scale, d.dropout_p, d.seed, d.offset = scale, dropout_p, seed, offset
    d.rng = _rng_ptr(rng, q)
    return d


@torch.library.custom_op("mmn_b200::mha_fwd", mutates_args=())
def mha_fwd(q: Tensor, k: Tensor, v: Tensor, mask: Optional[Tensor], num_heads: int, mask_kind: int, mask_diag: int,
            scale: float, dropout_p: float, seed: int, offset: int, rng: Optional[Tensor] = None) -> Tuple[Tensor, Tensor]:
    """rng: None, or a device {seed, offset} (next_dropout_stream) that replaces seed / offset."""
    _require_cuda(q, k, v, mask)
    lib = _lib.load()
    d = _mha_desc(q, k, num_heads, mask_kind, mask_diag, scale, dropout_p, seed, offset, rng)
    out = torch.empty(q.shape, dtype=q.dtype, device=q.device)
    lse = torch.empty(q.shape[1] * num_heads, q.shape[0], dtype=torch.float32, device=q.device)
    d.q_stride_t, d.q_stride_b = _tb_strides(q)
    d.k_stride_t, d.k_stride_b = _tb_strides(k)
    d.v_stride_t, d.v_stride_b = _tb_strides(v)
    d.o_stride_t, d.o_stride_b = _tb_strides(out)
    if mask is not None and (mask.dtype != torch.float32 or not mask.is_contiguous()):
        raise RuntimeError("attn_mask must be contiguous float32")
    with _timed("mha_fwd", q):
        _lib.check(lib.mmn_mha_fwd(C.byref(d), _ptr(q), _ptr(k), _ptr(v), _ptr(mask), _ptr(out), _ptr(lse), q.device.index,
                                   _stream(q)), "mmn_mha_fwd")
    return out, lse


@mha_fwd.register_fake
def _(q, k, v, mask, num_heads, mask_kind, mask_diag, scale, dropout_p, seed, offset, rng=None):
    return torch.empty_like(q, memory_format=torch.contiguous_format), q.new_empty(q.shape[1] * num_heads, q.shape[0],
                                                                                    dtype=torch.float32)


@torch.library.custom_op("mmn_b200::mha_bwd", mutates_args=())
def mha_bwd(dout: Tensor, q: Tensor, k: Tensor, v: Tensor, mask: Optional[Tensor], out: Tensor, lse: Tensor,
            num_heads: int, mask_kind: int, mask_diag: int, scale: float, dropout_p: float, seed: int,
            offset: int, rng: Optional[Tensor] = None) -> Tuple[Tensor, Tensor, Tensor]:
    _require_cuda(dout, q, k, v, mask, out, lse)
    lib = _lib.load()
    d = _mha_desc(q, k, num_heads, mask_kind, mask_diag, scale, dropout_p, seed, offset, rng)
    dout = dout.contiguous()
    dq = torch.empty(q.shape, dtype=q.dtype, device=q.device)
    dk = torch.empty(k.shape, dtype=k.dtype, device=k.device)
    dv = torch.empty(v.shape, dtype=v.dtype, device=v.device)
    d.q_stride_t, d.q_stride_b = _tb_strides(q)
    d.k_stride_t, d.k_stride_b = _tb_strides(k)
    d.v_stride_t, d.v_stride_b = _tb_strides(v)
    d.o_stride_t, d.o_stride_b = _tb_strides(out)
    d.do_stride_t, d.do_stride_b = _tb_strides(dout)
    d.dq_stride_t, d.dq_stride_b = _tb_strides(dq)
    d.dk_stride_t, d.dk_stride_b = _tb_strides(dk)
    d.dv_stride_t, d.dv_stride_b = _tb_strides(dv)
    ws = lse.new_empty(2 * lse.shape[0] * ((lse.shape[1] + 127) // 128 * 128))      # row data per query, padded to whole tiles
    with _timed("mha_bwd", q):
        _lib.check(lib.mmn_mha_bwd(C.byref(d), _ptr(q), _ptr(k), _ptr(v), _ptr(mask), _ptr(out), _ptr(lse), _ptr(dout),
                                   _ptr(dq), _ptr(dk), _ptr(dv), _ptr(ws), q.device.index, _stream(q)), "mmn_mha_bwd")
    return dq, dk, dv


@mha_bwd.register_fake
def _(dout, q, k, v, mask, out, lse, num_heads, mask_kind, mask_diag, scale, dropout_p, seed, offset, rng=None):
    c = torch.contiguous_format
    return torch.empty_like(q, memory_format=c), torch.empty_like(k, memory_format=c), torch.empty_like(v, memory_format=c)


def _mha_setup(ctx, inputs, output):
    q, k, v, mask, num_heads, mask_kind, mask_diag, scale, dropout_p, seed, offset, rng = inputs
    out, lse = output
    ctx.save_for_backward(q, k, v, mask, out, lse, rng)
    ctx.cfg = (num_heads, mask_kind, mask_diag, scale, dropout_p, seed, offset)


def _mha_backward(ctx, dout, dlse):
    q, k, v, mask, out, lse, rng = ctx.saved_tensors
    dq, dk, dv = torch.ops.mmn_b200.mha_bwd(dout, q, k, v, mask, out, lse, *ctx.cfg, rng)
    return (dq, dk, dv, None) + (None,) * 8


torch.library.register_autograd("mmn_b200::mha_fwd", _mha_backward, setup_context=_mha_setup)


@torch.library.custom_op("mmn_b200::mha_avg_weights", mutates_args=())
def mha_avg_weights(q: Tensor, k: Tensor, mask: Optional[Tensor], lse: Tensor, num_heads: int, mask_kind: int,
                    mask_diag: int, scale: float, dropout_p: float, seed: int, offset: int,
                    rng: Optional[Tensor] = None) -> Tensor:
    _require_cuda(q, k, mask, lse)
    lib = _lib.load()
    d = _mha_desc(q, k, num_heads, mask_kind, mask_diag, scale, dropout_p, seed, offset, rng)
    d.q_stride_t, d.q_stride_b = _tb_strides(q)
    d.k_stride_t, d.k_stride_b = _tb_strides(k)
    avg = torch.empty(q.shape[1], q.shape[0], k.shape[0], dtype=torch.float32, device=q.device)
    _lib.check(lib.mmn_mha_avg_weights(C.byref(d), _ptr(q), _ptr(k), _ptr(mask), _ptr(lse), _ptr(avg), q.device.index,
                                       _stream(q)), "mmn_mha_avg_weights")
    return avg


@mha_avg_weights.register_fake
def _(q, k, mask, lse, num_heads, mask_kind, mask_diag, scale, dropout_p, seed, offset, rng=None):
    return q.new_empty(q.shape[1], q.shape[0], k.shape[0], dtype=torch.float32)


@torch.library.custom_op("mmn_b200::colsum", mutates_args=())
def colsum(x: Tensor) -> Tensor:
    """(rows, cols) -> (cols,) fp32 column sums (a projection's bias gradient) at memory speed."""
    _require_cuda(x)
    if x.dim() != 2 or x.stride(1) != 1 or x.dtype not in _DT:
        raise RuntimeError("colsum expects a 2-D float32/bfloat16 tensor with contiguous columns")
    out = torch.zeros(x.shape[1], dtype=torch.float32, device=x.device)
    lib, det = _lib.load(), _deterministic()
    ws = _workspace(lib.mmn_colsum_workspace_bytes(x.shape[0], x.shape[1]), x) if det else None
    with _timed("colsum", x):
        _lib.check(lib.mmn_colsum(_ptr(x), _DT[x.dtype], x.shape[0], x.shape[1], x.stride(0), _ptr(out), _ptr(ws), int(det),
                                  x.device.index, _stream(x)), "mmn_colsum")
    return out


@colsum.register_fake
def _(x):
    return x.new_empty(x.shape[1], dtype=torch.float32)


@torch.library.custom_op("mmn_b200::table_bias_fwd", mutates_args=())
def table_bias_fwd(table: Tensor, index: Tensor) -> Tensor:
    """(T, nH) fp32 table, (NN,) int64 index -> (nH, NN) bias = table[index].T in one launch (swinfusion_module.py:127-130)."""
    _require_cuda(table, index)
    if table.dim() != 2 or table.dtype != torch.float32 or not table.is_contiguous() or index.dtype != torch.int64 or \
            not index.is_contiguous():
        raise RuntimeError("table_bias_fwd expects a contiguous fp32 (T, heads) table and a contiguous int64 index")
    T, nH, NN = table.shape[0], table.shape[1], index.numel()
    bias = torch.empty(nH, NN, dtype=torch.float32, device=table.device)
    _lib.check(_lib.load().mmn_table_bias_fwd(_ptr(table), _ptr(index), T, nH, NN, _ptr(bias), table.device.index, _stream(table)),
               "mmn_table_bias_fwd")
    return bias


@table_bias_fwd.register_fake
def _(table, index):
    return table.new_empty(table.shape[1], index.numel())


@torch.library.custom_op("mmn_b200::table_bias_bwd", mutates_args=())
def table_bias_bwd(dbias: Tensor, index: Tensor, table_rows: int) -> Tensor:
    _require_cuda(dbias, index)
    dbias = dbias.contiguous()
    nH, NN = dbias.shape[0], index.numel()
    dtable = torch.empty(table_rows, nH, dtype=torch.float32, device=dbias.device)
    perm, offsets = _inverse_index(index, table_rows) if _deterministic() else (None, None)
    _lib.check(_lib.load().mmn_table_bias_bwd(_ptr(dbias), _ptr(index), _ptr(perm), _ptr(offsets), table_rows, nH, NN, _ptr(dtable),
                                             dbias.device.index, _stream(dbias)), "mmn_table_bias_bwd")
    return dtable


@table_bias_bwd.register_fake
def _(dbias, index, table_rows):
    return dbias.new_empty(table_rows, dbias.shape[0])


def _table_bias_setup(ctx, inputs, output):
    table, index = inputs
    ctx.save_for_backward(index)
    ctx.rows = table.shape[0]


def _table_bias_backward(ctx, dbias):
    index, = ctx.saved_tensors
    return torch.ops.mmn_b200.table_bias_bwd(dbias.float().reshape(dbias.shape[0], -1), index, ctx.rows), None


torch.library.register_autograd("mmn_b200::table_bias_fwd", _table_bias_backward, setup_context=_table_bias_setup)


def cpb_bias_supported(coords: Tensor, w1: Tensor, w2: Tensor) -> bool:
    """True when the fused continuous-position-bias kernels take these operands (fp32 CUDA, <= 3 coordinates,
    <= 64 heads, table x heads <= 12288)."""
    ok = coords.is_cuda and all(t.dtype == torch.float32 for t in (coords, w1, w2))
    T = coords.numel() // coords.shape[-1]
    # backward kernel's dynamic shared memory (csrc/cpb_bias.cu: cpb_bwd_smem_bytes): (11 T + 4096) floats <= 227 KB
    return bool(ok and coords.shape[-1] <= 3 and w2.shape[0] <= 64 and T * w2.shape[0] <= 12288 and (11 * T + 4100) * 4 <= 227 * 1024)


@torch.library.custom_op("mmn_b200::cpb_bias_fwd", mutates_args=())
def cpb_bias_fwd(coords: Tensor, w1: Tensor, b1: Tensor, w2: Tensor, index: Tensor) -> Tuple[Tensor, Tensor]:
    """coords (T, n), w1 (J, n), b1 (J), w2 (nH, J), index (NN) int64 -> bias (nH, NN), tab16 (T, nH)."""
    _require_cuda(coords, w1, b1, w2, index)
    T, n_in, J, nH, NN = coords.shape[0], coords.shape[1], w1.shape[0], w2.shape[0], index.numel()
    tab16 = torch.empty(T, nH, dtype=torch.float32, device=coords.device)
    bias = torch.empty(nH, NN, dtype=torch.float32, device=coords.device)
    _lib.check(_lib.load().mmn_cpb_bias_fwd(_ptr(coords), _ptr(w1), _ptr(b1), _ptr(w2), _ptr(index), T, n_in, J, nH, NN,
                                           _ptr(tab16), _ptr(bias), coords.device.index, _stream(coords)), "mmn_cpb_bias_fwd")
    return bias, tab16


@cpb_bias_fwd.register_fake
def _(coords, w1, b1, w2, index):
    return (coords.new_empty(w2.shape[0], index.numel()), coords.new_empty(coords.shape[0], w2.shape[0]))


@torch.library.custom_op("mmn_b200::cpb_bias_bwd", mutates_args=())
def cpb_bias_bwd(dbias: Tensor, coords: Tensor, w1: Tensor, b1: Tensor, w2: Tensor, index: Tensor,
                 tab16: Tensor) -> Tuple[Tensor, Tensor, Tensor]:
    _require_cuda(dbias, coords, w1, b1, w2, index, tab16)
    T, n_in, J, nH, NN = coords.shape[0], coords.shape[1], w1.shape[0], w2.shape[0], index.numel()
    dbias = dbias.contiguous()
    dw1, db1, dw2 = torch.empty_like(w1), torch.empty_like(b1), torch.empty_like(w2)
    scratch = torch.empty(T, nH, dtype=torch.float32, device=coords.device)
    perm, offsets = _inverse_index(index, T) if _deterministic() else (None, None)
    _lib.check(_lib.load().mmn_cpb_bias_bwd(_ptr(coords), _ptr(w1), _ptr(b1), _ptr(w2), _ptr(index), _ptr(perm), _ptr(offsets),
                                           _ptr(tab16), _ptr(dbias),
                                           T, n_in, J, nH, NN, _ptr(scratch), _ptr(dw1), _ptr(db1), _ptr(dw2),
                                           coords.device.index, _stream(coords)), "mmn_cpb_bias_bwd")
    return dw1, db1, dw2


@cpb_bias_bwd.register_fake
def _(dbias, coords, w1, b1, w2, index, tab16):
    return torch.empty_like(w1), torch.empty_like(b1), torch.empty_like(w2)


def _cpb_setup(ctx, inputs, output):
    coords, w1, b1, w2, index = inputs
    ctx.save_for_backward(coords, w1, b1, w2, index, output[1])


def _cpb_backward(ctx, dbias, _dtab16):
    coords, w1, b1, w2, index, tab16 = ctx.saved_tensors
    dw1, db1, dw2 = torch.ops.mmn_b200.cpb_bias_bwd(dbias, coords, w1, b1, w2, index, tab16)
    return None, dw1, db1, dw2, None


cpb_bias_fwd.register_autograd(_cpb_backward, setup_context=_cpb_setup)


_ACT = {"none": _lib.ACT_NONE, "relu": _lib.ACT_RELU, "gelu": _lib.ACT_GELU}


def _rows2d(t: Tensor) -> bool:
    return t.dim() == 2 and t.stride(1) == 1 and t.is_cuda and t.dtype == torch.bfloat16


def linear_supported(x: Tensor, w: Tensor) -> bool:
    """True when the tensor-core projection kernels take these operands: bf16 CUDA, x (rows, in) with contiguous columns,
    w (out, in) contiguous, in and out multiples of 32."""
    if not (_rows2d(x) and w.is_cuda and w.dtype == torch.bfloat16 and w.dim() == 2 and w.is_contiguous()) or x.shape[0] < 1:
        return False
    return bool(_lib.load().mmn_linear_supported(_lib.DT_BF16, x.shape[0], x.shape[1], w.shape[0], x.stride(0), w.shape[0]))


@torch.library.custom_op("mmn_b200::linear_fwd", mutates_args=())
def linear_fwd(x: Tensor, w: Tensor, bias: Optional[Tensor], act: int, want_pre: bool) -> Tuple[Tensor, Tensor]:
    """y = act(x w^T + bias) on the tensor cores; returns (y, dact) where dact = act'(x w^T + bias), the activation's derivative
    at the pre-activation (what the backward multiplies with) when `want_pre`, else an empty tensor."""
    _require_cuda(x, w, bias)
    if not _rows2d(x) or w.dtype != torch.bfloat16 or not w.is_contiguous():
        raise RuntimeError("linear_fwd expects bf16 x (rows, in) with contiguous columns and a contiguous bf16 weight")
    if bias is not None and (bias.dtype != torch.float32 or not bias.is_contiguous()):
        raise RuntimeError("linear_fwd takes its bias in float32")
    rows, n_in, n_out = x.shape[0], x.shape[1], w.shape[0]
    y = torch.empty(rows, n_out, dtype=x.dtype, device=x.device)
    pre = torch.empty(rows, n_out, dtype=x.dtype, device=x.device) if want_pre else x.new_empty(0)
    with _timed("linear_fwd", x):
        _lib.check(_lib.load().mmn_linear_fwd(_ptr(x), _ptr(w), _ptr(bias), _ptr(y), _ptr(pre) if want_pre else None, act,
                                              _lib.DT_BF16, rows, n_in, n_out, x.stride(0), n_out, x.device.index, _stream(x)),
                   "mmn_linear_fwd")
    return y, pre


@linear_fwd.register_fake
def _(x, w, bias, act, want_pre):
    return x.new_empty(x.shape[0], w.shape[0]), (x.new_empty(x.shape[0], w.shape[0]) if want_pre else x.new_empty(0))


def linear_bwd_supported(dy: Tensor, x: Tensor, w: Tensor) -> bool:
    """True when the tensor-core projection backward takes these operands (bf16, in and out multiples of 32)."""
    if not (_rows2d(dy) and _rows2d(x) and w.is_cuda and w.dtype == torch.bfloat16 and w.is_contiguous()) or dy.shape[0] < 1:
        return False
    return bool(_lib.load().mmn_linear_bwd_supported(_lib.DT_BF16, dy.shape[0], x.shape[1], dy.shape[1], dy.stride(0),
                                                     x.stride(0), x.shape[1]))


@torch.library.custom_op("mmn_b200::linear_bwd", mutates_args=())
def linear_bwd(dy: Tensor, x: Tensor, w: Tensor, act_aux: Optional[Tensor] = None, act: int = 0, want_dx: bool = True,
               want_dw: bool = True) -> Tuple[Tensor, Tensor, Tensor]:
    """Backward of y = x w^T + b: returns (dx bf16 (rows, in), dw fp32 (out, in), db fp32 (out)).  With `act_aux` (the
    act'(pre) that linear_fwd wrote for the layer whose activation produced x) dx is additionally multiplied by it in the
    kernel's epilogue, i.e. it is the gradient w.r.t. that pre-activation.  in = 96 runs as one fused pass over dy and x,
    other widths as dgrad + wgrad."""
    _require_cuda(dy, x, w, act_aux)
    lib = _lib.load()
    rows, n_out, n_in = dy.shape[0], dy.shape[1], x.shape[1]
    dx = torch.empty(rows, n_in, dtype=dy.dtype, device=dy.device) if want_dx else dy.new_empty(0)
    dw = torch.empty(n_out, n_in, dtype=torch.float32, device=dy.device) if want_dw else dy.new_empty(0, dtype=torch.float32)
    db = torch.empty(n_out, dtype=torch.float32, device=dy.device) if want_dw else dy.new_empty(0, dtype=torch.float32)
    det = _deterministic()
    ws = torch.empty(lib.mmn_linear_bwd_workspace_bytes(rows, n_in, n_out, int(det)), dtype=torch.uint8, device=dy.device)
    if act_aux is not None and (not _rows2d(act_aux) or act_aux.shape != (rows, n_in)):
        raise RuntimeError("act_aux must be a bf16 (rows, in) tensor with contiguous columns")
    with _timed("linear_bwd", dy):
        _lib.check(lib.mmn_linear_bwd(_ptr(dy), _ptr(x), _ptr(w), _ptr(dx) if want_dx else None, _ptr(dw) if want_dw else None,
                                      _ptr(db) if want_dw else None, _ptr(ws), _ptr(act_aux),
                                      act_aux.stride(0) if act_aux is not None else 0, act if act_aux is not None else 0,
                                      _DT[dy.dtype], rows, n_in, n_out, dy.stride(0), x.stride(0), n_in, int(det), dy.device.index,
                                      _stream(dy)), "mmn_linear_bwd")
    return dx, dw, db


@linear_bwd.register_fake
def _(dy, x, w, act_aux=None, act=0, want_dx=True, want_dw=True):
    f32 = dict(dtype=torch.float32)
    return (dy.new_empty(dy.shape[0], x.shape[1]) if want_dx else dy.new_empty(0),
            dy.new_empty(dy.shape[1], x.shape[1], **f32) if want_dw else dy.new_empty(0, **f32),
            dy.new_empty(dy.shape[1], **f32) if want_dw else dy.new_empty(0, **f32))


class LinearFn(torch.autograd.Function):
    """y = act(x w^T + b) with the tensor-core forward and backward above; x (..., in) bf16, w / b master weights of any
    float dtype (cast to bf16 / fp32 here, gradients returned in their dtypes)."""

    @staticmethod
    def forward(ctx, x, w, b, act):
        x2 = x.reshape(-1, x.shape[-1])
        wc = weight_bf16(w)
        y, pre = torch.ops.mmn_b200.linear_fwd(x2, wc, None if b is None else b.float(), act, act != _lib.ACT_NONE)
        ctx.save_for_backward(x2, wc, pre)
        ctx.meta = (x.shape, w.dtype, None if b is None else b.dtype, act, x.requires_grad)
        return y.view(*x.shape[:-1], w.shape[0])

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, dy):
        x2, wc, pre = ctx.saved_tensors
        shape, wdt, bdt, act, need_dx = ctx.meta
        dy2 = dy.reshape(-1, dy.shape[-1]).to(torch.bfloat16)
        if act != _lib.ACT_NONE:                       # through the activation: dy o act'(pre), then the plain projection backward
            dy2 = dy2 * pre
        dx, dw, db = torch.ops.mmn_b200.linear_bwd(dy2.contiguous(), x2, wc, None, 0, need_dx, True)
        return (dx.view(shape) if need_dx else None, dw.to(wdt), db.to(bdt) if bdt is not None else None, None)


def linear(x: Tensor, w: Tensor, b: Optional[Tensor] = None, act: str = "none") -> Tensor:
    """Drop-in for F.linear (+ activation) on CUDA bf16 activations whose widths are multiples of 32; anything else falls
    to F.linear (a plain library GEMM: the reference's own 12/24/48/84-wide layers)."""
    x2 = x.reshape(-1, x.shape[-1]) if x.dim() != 2 else x
    if x.is_cuda and x.dtype == torch.bfloat16 and x.numel() > 0 and w.shape[1] % 32 == 0 and w.shape[0] % 32 == 0 and \
            x2.stride(-1) == 1 and x2.stride(0) % 8 == 0 and x2.data_ptr() % 16 == 0:
        return LinearFn.apply(x, w, b, _ACT[act])
    y = torch.nn.functional.linear(x, w.to(x.dtype), None if b is None else b.to(x.dtype))
    return y if act == "none" else (torch.relu(y) if act == "relu" else torch.nn.functional.gelu(y))


# ------------------------------------------------------------------------------------------
# LayerNorm fused with the residual add (csrc/layernorm.cu)
# ------------------------------------------------------------------------------------------
_DTC = {torch.float32: _lib.DT_F32, torch.bfloat16: _lib.DT_BF16}
_DTC_INV = {_lib.DT_F32: torch.float32, _lib.DT_BF16: torch.bfloat16}


@functools.lru_cache(maxsize=None)
def _layernorm_width_supported(cols: int) -> bool:
    return bool(_lib.load().mmn_layernorm_supported(cols))


def layernorm_supported(x: Tensor, cols: int) -> bool:
    return bool(x.is_cuda and x.dtype in _DTC and x.numel() > 0 and _layernorm_width_supported(cols))


@torch.library.custom_op("mmn_b200::layernorm_fwd", mutates_args=())
def layernorm_fwd(resid: Optional[Tensor], delta: Optional[Tensor], gamma: Tensor, beta: Optional[Tensor], eps: float, mode: int,
                  want_sum: bool, norm_dt: int) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    """mode 0 (pre-norm): s = resid + delta, out_norm = LN(s);  mode 1 (post-norm): s = resid + LN(delta), out_norm = s.
    Returns (out_sum [dtype of resid, or delta's], out_norm [norm_dt: -1 none, else MMN_DT_*], mean, rstd); rows = all
    leading dims.  Skipped outputs are empty tensors."""
    _require_cuda(resid, delta, gamma, beta)
    ref = resid if resid is not None else delta
    cols = ref.shape[-1]
    rows = ref.numel() // cols
    for t in (resid, delta):
        if t is not None and (not t.is_contiguous() or t.dtype not in _DTC or t.shape != ref.shape):
            raise RuntimeError("layernorm_fwd expects contiguous float32/bfloat16 tensors of one shape")
    if gamma.dtype != torch.float32 or (beta is not None and beta.dtype != torch.float32):
        raise RuntimeError("layernorm_fwd takes gamma / beta in float32")
    out_sum = torch.empty_like(ref) if want_sum else ref.new_empty(0)
    out_norm = torch.empty(ref.shape, dtype=_DTC_INV[norm_dt], device=ref.device) if norm_dt >= 0 else ref.new_empty(0)
    mean = torch.empty(rows, dtype=torch.float32, device=ref.device)
    rstd = torch.empty(rows, dtype=torch.float32, device=ref.device)
    dt = lambda t: _DTC[t.dtype] if t is not None else 0
    with _timed("layernorm_fwd", ref):
        _lib.check(_lib.load().mmn_layernorm_fwd(_ptr(resid), dt(resid), _ptr(delta), dt(delta), _ptr(gamma), _ptr(beta), eps, mode,
                                                 _ptr(out_sum) if want_sum else None, _DTC[ref.dtype],
                                                 _ptr(out_norm) if norm_dt >= 0 else None, max(norm_dt, 0), _ptr(mean), _ptr(rstd),
                                                 rows, cols, ref.device.index, _stream(ref)), "mmn_layernorm_fwd")
    return out_sum, out_norm, mean, rstd


@layernorm_fwd.register_fake
def _(resid, delta, gamma, beta, eps, mode, want_sum, norm_dt):
    ref = resid if resid is not None else delta
    rows = ref.numel() // ref.shape[-1]
    return (torch.empty_like(ref) if want_sum else ref.new_empty(0),
            ref.new_empty(ref.shape, dtype=_DTC_INV[norm_dt]) if norm_dt >= 0 else ref.new_empty(0),
            ref.new_empty(rows, dtype=torch.float32), ref.new_empty(rows, dtype=torch.float32))


@torch.library.custom_op("mmn_b200::layernorm_bwd", mutates_args=())
def layernorm_bwd(g_sum: Optional[Tensor], g_norm: Optional[Tensor], x: Tensor, gamma: Tensor, mean: Tensor, rstd: Tensor, mode: int,
                  resid_dt: int, delta_dt: int, want_beta: bool) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    """Returns (d_resid [resid_dt, -1: skipped], d_delta [delta_dt, -1: skipped], dgamma, dbeta)."""
    _require_cuda(g_sum, g_norm, x, gamma, mean, rstd)
    cols = x.shape[-1]
    rows = x.numel() // cols
    g_sum = g_sum.contiguous() if g_sum is not None else None
    g_norm = g_norm.contiguous() if g_norm is not None else None
    mk = lambda code: torch.empty(x.shape, dtype=_DTC_INV[code], device=x.device) if code >= 0 else x.new_empty(0)
    d_resid, d_delta = mk(resid_dt), mk(delta_dt)
    dgamma = torch.zeros(cols, dtype=torch.float32, device=x.device)
    dbeta = torch.zeros(cols, dtype=torch.float32, device=x.device) if want_beta else x.new_empty(0, dtype=torch.float32)
    dt = lambda t: _DTC[t.dtype] if t is not None else 0
    lib, det = _lib.load(), _deterministic()
    ws = _workspace(lib.mmn_layernorm_bwd_workspace_bytes(rows, cols), x) if det else None
    with _timed("layernorm_bwd", x):
        _lib.check(lib.mmn_layernorm_bwd(_ptr(g_sum), dt(g_sum), _ptr(g_norm), dt(g_norm), _ptr(x), _DTC[x.dtype], _ptr(gamma),
                                                 _ptr(mean), _ptr(rstd), mode, _ptr(d_resid) if resid_dt >= 0 else None, max(resid_dt, 0),
                                                 _ptr(d_delta) if delta_dt >= 0 else None, max(delta_dt, 0), _ptr(dgamma),
                                                 _ptr(dbeta) if want_beta else None, _ptr(ws), int(det), rows, cols, x.device.index,
                                                 _stream(x)),
                   "mmn_layernorm_bwd")
    return d_resid, d_delta, dgamma, dbeta


@layernorm_bwd.register_fake
def _(g_sum, g_norm, x, gamma, mean, rstd, mode, resid_dt, delta_dt, want_beta):
    mk = lambda code: x.new_empty(x.shape, dtype=_DTC_INV[code]) if code >= 0 else x.new_empty(0)
    return (mk(resid_dt), mk(delta_dt), x.new_empty(x.shape[-1], dtype=torch.float32),
            x.new_empty(x.shape[-1] if want_beta else 0, dtype=torch.float32))


class AddLayerNormFn(torch.autograd.Function):
    """(resid, delta, gamma, beta) -> (out_sum, out_norm) in one kernel each way; see layernorm_fwd for the two modes."""

    @staticmethod
    def forward(ctx, resid, delta, gamma, beta, eps, mode, norm_dtype):
        ref = resid if resid is not None else delta
        want_sum = resid is not None and delta is not None
        g32 = gamma.float()
        b32 = beta.float() if beta is not None else None
        rc = resid.contiguous() if resid is not None else None
        dc = delta.contiguous() if delta is not None else None
        out_sum, out_norm, mean, rstd = torch.ops.mmn_b200.layernorm_fwd(rc, dc, g32, b32, eps, mode, want_sum,
                                                                         _DTC[norm_dtype] if norm_dtype is not None else -1)
        x = (out_sum if want_sum else (rc if rc is not None else dc)) if mode == _lib.LN_PRE else dc
        ctx.save_for_backward(x, g32, mean, rstd)
        ctx.meta = (mode, None if resid is None else resid.dtype, None if delta is None else delta.dtype, gamma.dtype,
                    None if beta is None else beta.dtype, want_sum, norm_dtype is not None)
        ctx.set_materialize_grads(False)
        return (out_sum if want_sum else None), (out_norm if norm_dtype is not None else None)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g_sum, g_norm):
        x, g32, mean, rstd = ctx.saved_tensors
        mode, rdt, ddt, gdt, bdt, had_sum, had_norm = ctx.meta
        g_sum = g_sum if had_sum else None
        g_norm = g_norm if had_norm else None
        if g_sum is None and g_norm is None:
            return (None,) * 7
        need_r = rdt is not None and ctx.needs_input_grad[0]
        need_d = ddt is not None and ctx.needs_input_grad[1]
        d_resid, d_delta, dgamma, dbeta = torch.ops.mmn_b200.layernorm_bwd(
            g_sum, g_norm, x, g32, mean, rstd, mode,
            _DTC[rdt] if need_r else -1, _DTC[ddt] if need_d else -1, bdt is not None)
        return (d_resid if need_r else None, d_delta if need_d else None, dgamma.to(gdt), dbeta.to(bdt) if bdt is not None else None,
                None, None, None)


def next_dropout_stream(p: float, training: bool, device) -> Tuple[float, int, int, Optional[Tensor]]:
    """(p, seed, offset, rng) for one attention call, the last four arguments of the attention ops.  rng is a (2,) int64
    {seed, offset} drawn on `device` from its CUDA generator, so `torch.manual_seed` controls it and a CUDA graph that
    captured this call draws a fresh one on every replay; the kernels read it when they run (seed and offset are then 0).
    Outside training, or with p = 0: (0.0, 0, 0, None)."""
    if not training or p <= 0.0:
        return 0.0, 0, 0, None
    return float(p), 0, 0, torch.randint(0, 2 ** 62, (2,), dtype=torch.int64, device=device)


def winattn_qkv_path_name(x_shape, dtype, grid, window, shift, num_heads, score_kind, mask_kind, dropout_p: float = 0.0,
                          path: int = _lib.PATH_AUTO) -> str:
    """"tcgen05-fused" when winattn_qkv_fwd takes a self-attention call on x of this shape and dtype, else the reason it
    does not (the call then runs the projection and winattn_fwd separately)."""
    a = torch.empty(*x_shape[:-1], 3 * x_shape[-1], dtype=dtype, device="meta")
    d, Cc = _win_desc(a, None, grid, window, shift, num_heads, score_kind, mask_kind, 1, 1.0, dropout_p, 0, 0, path)
    d.q_row_stride = d.k_row_stride = d.v_row_stride = 3 * Cc
    d.o_row_stride = Cc
    return _lib.load().mmn_winattn_qkv_path(C.byref(d), int(x_shape[-1])).decode()


def winattn_path_name(a: Tensor, b: Optional[Tensor], grid, window, shift, num_heads, score_kind, mask_kind,
                      dropout_p: float = 0.0) -> str:
    d, _ = _win_desc(a, b, grid, window, shift, num_heads, score_kind, mask_kind, 1, 1.0, dropout_p, 0, 0, _lib.PATH_AUTO)
    return _lib.load().mmn_winattn_path(C.byref(d)).decode()
