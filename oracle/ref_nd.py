"""CPU oracle for the attention hot path -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` /
``--impl reference`` legs may import this module; the product path
(``multimodal_neuroimage_b200``) never does and has no CPU fallback.

What it is: a functional restatement (plain ``torch`` on CPU, any float dtype, fp64 for
tight checks) of the reference algorithms, generalised from the reference's 2-D windows
to n spatial dims (n in {1,2,3}).  The arithmetic is the reference's own (``F.linear``,
``@``, ``F.normalize``, ``softmax``); only the control structure differs: parameters are
passed as a flat ``dict`` with the reference's ``state_dict`` keys, so a reference
``state_dict`` can be fed in unchanged.

Parity pin: ``tests/test_oracle_golden.py`` checks every function here against the
fixtures under ``tests/golden/`` which were produced by importing and running the
UNMODIFIED reference modules (``tests/golden/make_golden.py``, 2-D -- the reference has
no 3-D code, SURVEY.md F1).  The n=3 instantiation is *our* specification (SURVEY.md
section 8a "3D generalisation"); it is pinned only through the n=2 equality of the same
code path, and DESIGN.md says so.

Reference citations are relative to /root/reference.
"""
from __future__ import annotations

import math
from typing import Dict, Optional, Sequence, Tuple

import torch
import torch.nn.functional as F

Tensor = torch.Tensor


def _tup(v, n: int) -> Tuple[int, ...]:
    if isinstance(v, (tuple, list)):
        assert len(v) == n, (v, n)
        return tuple(int(a) for a in v)
    return (int(v),) * n


# ----------------------------------------------------------------------------------------
# a1 / a2: window partition and reverse        modules/swin_v2_module.py:35-62,
#                                               modules/swinfusion_module.py:33-62
# ----------------------------------------------------------------------------------------
def window_partition_nd(x: Tensor, window: Sequence[int]) -> Tensor:
    """(B, *grid, C) -> (B*nW, *window, C); window id is row-major over the window grid,
    in-window position row-major over the window (swin_v2_module.py:43-45)."""
    n = x.dim() - 2
    window = _tup(window, n)
    B, C = x.shape[0], x.shape[-1]
    grid = x.shape[1:-1]
    split = []
    for g, w in zip(grid, window):
        assert g % w == 0, (grid, window)
        split += [g // w, w]
    x = x.reshape(B, *split, C)
    outer = [1 + 2 * i for i in range(n)]
    inner = [2 + 2 * i for i in range(n)]
    x = x.permute(0, *outer, *inner, 1 + 2 * n).contiguous()
    return x.reshape(-1, *window, C)


def window_reverse_nd(windows: Tensor, window: Sequence[int], grid: Sequence[int]) -> Tensor:
    """Inverse of :func:`window_partition_nd` (swin_v2_module.py:59-61)."""
    n = len(grid)
    window = _tup(window, n)
    counts = [g // w for g, w in zip(grid, window)]
    nW = int(math.prod(counts))
    B = windows.shape[0] // nW
    x = windows.reshape(B, *counts, *window, -1)
    perm = [0]
    for i in range(n):
        perm += [1 + i, 1 + n + i]
    x = x.permute(*perm, 1 + 2 * n).contiguous()
    return x.reshape(B, *grid, -1)


# ----------------------------------------------------------------------------------------
# a3: cyclic shift                               swin_v2_module.py:277-280,294-297
# ----------------------------------------------------------------------------------------
def cyclic_shift_nd(x: Tensor, shift: Sequence[int], inverse: bool = False) -> Tensor:
    n = x.dim() - 2
    shift = _tup(shift, n)
    if not any(shift):
        return x
    sgn = 1 if inverse else -1
    return torch.roll(x, shifts=tuple(sgn * s for s in shift), dims=tuple(range(1, n + 1)))


def effective_window(grid: Sequence[int], window: int, shift: int) -> Tuple[int, int]:
    """`if min(input_resolution) <= window_size: shift = 0; window = min(res)`
    (swin_v2_module.py:226-229; swinfusion_module.py:294-297,429-432)."""
    if min(grid) <= window:
        return min(grid), 0
    return window, shift


# ----------------------------------------------------------------------------------------
# a4: shift mask                                 swin_v2_module.py:244-266,
#                                                swinfusion_module.py:317-338,461-482
# ----------------------------------------------------------------------------------------
def shift_region_ids_nd(grid: Sequence[int], window: Sequence[int], shift: Sequence[int]) -> Tensor:
    """Region id image (*grid) int64 in the SHIFTED frame.  Per axis the three slices
    are [0,-w) [-w,-s) [-s,None) and `cnt` runs with the first axis outermost
    (swin_v2_module.py:247-258).  An axis with shift 0 contributes a single region, which
    is what python slicing with -0 does NOT do in the reference (slice(-w,-0) is empty and
    slice(-0,None) is everything) -- but the reference only builds masks when shift>0 and
    always shifts every axis by the same amount, so that case never occurs there."""
    n = len(grid)
    window, shift = _tup(window, n), _tup(shift, n)
    img = torch.zeros(tuple(grid), dtype=torch.int64)
    per_axis = []
    for g, w, s in zip(grid, window, shift):
        if s > 0:
            per_axis.append([slice(0, g - w), slice(g - w, g - s), slice(g - s, g)])
        else:
            per_axis.append([slice(0, g)])
    cnt = 0

    def rec(axis, idx):
        nonlocal cnt
        if axis == n:
            img[tuple(idx)] = cnt
            cnt += 1
            return
        for sl in per_axis[axis]:
            rec(axis + 1, idx + [sl])

    rec(0, [])
    return img


def shift_mask_nd(grid: Sequence[int], window: Sequence[int], shift: Sequence[int],
                  dtype=torch.float32) -> Optional[Tensor]:
    """(nW, N, N) additive mask with values {0, -100} (swin_v2_module.py:259-262)."""
    n = len(grid)
    window, shift = _tup(window, n), _tup(shift, n)
    if not any(shift):
        return None
    ids = shift_region_ids_nd(grid, window, shift).to(dtype)
    mw = window_partition_nd(ids.reshape(1, *grid, 1), window).reshape(-1, int(math.prod(window)))
    diff = mw.unsqueeze(1) - mw.unsqueeze(2)
    return diff.masked_fill(diff != 0, -100.0).masked_fill(diff == 0, 0.0)


# ----------------------------------------------------------------------------------------
# a5: relative position index and CPB coordinate table   swin_v2_module.py:95-124,
#                                                        swinfusion_module.py:92-103
# ----------------------------------------------------------------------------------------
def relative_position_index_nd(window: Sequence[int]) -> Tensor:
    """(N, N) int64.  2-D: (dh+wh-1)*(2ww-1) + (dw+ww-1) (swin_v2_module.py:113-122)."""
    window = tuple(int(w) for w in window)
    coords = torch.stack(torch.meshgrid([torch.arange(w) for w in window], indexing="ij"))
    flat = coords.flatten(1)                                   # n, N
    rel = flat[:, :, None] - flat[:, None, :]                  # n, N, N
    idx = torch.zeros(rel.shape[1:], dtype=torch.int64)
    for a, w in enumerate(window):
        idx = idx * (2 * w - 1) + (rel[a] + w - 1)
    return idx


def cpb_coords_table_nd(window: Sequence[int], pretrained_window: Optional[Sequence[int]] = None) -> Tensor:
    """(1, 2w0-1, ..., n) fp32 log-spaced coordinates (swin_v2_module.py:96-110)."""
    window = tuple(int(w) for w in window)
    n = len(window)
    axes = [torch.arange(-(w - 1), w, dtype=torch.float32) for w in window]
    table = torch.stack(torch.meshgrid(axes, indexing="ij")).permute(*range(1, n + 1), 0).contiguous().unsqueeze(0)
    use_pre = pretrained_window is not None and pretrained_window[0] > 0
    for a in range(n):
        den = (pretrained_window[a] - 1) if use_pre else (window[a] - 1)
        table[..., a] /= den
    table *= 8
    return torch.sign(table) * torch.log2(torch.abs(table) + 1.0) / math.log2(8)


# ----------------------------------------------------------------------------------------
# a6: SwinV2 cosine window attention             swin_v2_module.py:138-178
# ----------------------------------------------------------------------------------------
def cpb_bias(p: Dict[str, Tensor], window: Sequence[int], num_heads: int) -> Tensor:
    """16*sigmoid(cpb_mlp(table))[index] -> (nH, N, N) (swin_v2_module.py:158-162)."""
    N = int(math.prod(window))
    t = p["relative_coords_table"]
    h = F.relu(F.linear(t, p["cpb_mlp.0.weight"], p["cpb_mlp.0.bias"]))
    tab = F.linear(h, p["cpb_mlp.2.weight"]).view(-1, num_heads)
    b = tab[p["relative_position_index"].view(-1)].view(N, N, -1).permute(2, 0, 1).contiguous()
    return 16 * torch.sigmoid(b)


def _softmax_with_mask(attn: Tensor, mask: Optional[Tensor], num_heads: int) -> Tensor:
    """swin_v2_module.py:165-171: mask (nW,N,N) broadcast over batch and heads."""
    if mask is not None:
        B_, _, N, M = attn.shape
        nW = mask.shape[0]
        attn = attn.view(B_ // nW, nW, num_heads, N, M) + mask.unsqueeze(1).unsqueeze(0)
        attn = attn.view(-1, num_heads, N, M)
    return attn.softmax(dim=-1)


def window_attention_cosine(x: Tensor, p: Dict[str, Tensor], window: Sequence[int], num_heads: int,
                            mask: Optional[Tensor] = None) -> Tensor:
    """x (B_, N, C) -> (B_, N, C); p holds WindowAttention's state_dict keys."""
    B_, N, C = x.shape
    qkv_bias = None
    if p.get("q_bias") is not None:
        qkv_bias = torch.cat((p["q_bias"], torch.zeros_like(p["v_bias"]), p["v_bias"]))   # :147
    qkv = F.linear(x, p["qkv.weight"], qkv_bias).reshape(B_, N, 3, num_heads, -1).permute(2, 0, 3, 1, 4)
    q, k, v = qkv[0], qkv[1], qkv[2]
    attn = F.normalize(q, dim=-1) @ F.normalize(k, dim=-1).transpose(-2, -1)               # :153
    logit_scale = torch.clamp(p["logit_scale"], max=math.log(1.0 / 0.01)).exp()             # :154-155
    attn = attn * logit_scale
    attn = attn + cpb_bias(p, window, num_heads).unsqueeze(0)                               # :158-163
    attn = _softmax_with_mask(attn, mask, num_heads)
    out = (attn @ v).transpose(1, 2).reshape(B_, N, C)
    return F.linear(out, p["proj.weight"], p["proj.bias"])


# ----------------------------------------------------------------------------------------
# a8 / a9: SwinFusion scaled-dot window attention, self and cross
#                                                swinfusion_module.py:114-145, 213-246
# ----------------------------------------------------------------------------------------
def table_bias(p: Dict[str, Tensor], window: Sequence[int]) -> Tensor:
    N = int(math.prod(window))
    b = p["relative_position_bias_table"][p["relative_position_index"].view(-1)].view(N, N, -1)
    return b.permute(2, 0, 1).contiguous()


def window_attention_scaled(x: Tensor, p: Dict[str, Tensor], window: Sequence[int], num_heads: int,
                            mask: Optional[Tensor] = None, y: Optional[Tensor] = None,
                            qk_scale: Optional[float] = None) -> Tensor:
    """Self (y None: keys qkv.*) or cross (y given: keys q.*, kv.*) window attention."""
    B_, N, C = x.shape
    d = C // num_heads
    scale = qk_scale or d ** -0.5
    if y is None:
        qkv = F.linear(x, p["qkv.weight"], p.get("qkv.bias")).reshape(B_, N, 3, num_heads, d).permute(2, 0, 3, 1, 4)
        q, k, v = qkv[0], qkv[1], qkv[2]
    else:
        q = F.linear(x, p["q.weight"], p.get("q.bias")).reshape(B_, N, 1, num_heads, d).permute(2, 0, 3, 1, 4)[0]
        kv = F.linear(y, p["kv.weight"], p.get("kv.bias")).reshape(B_, N, 2, num_heads, d).permute(2, 0, 3, 1, 4)
        k, v = kv[0], kv[1]
    q = q * scale                                                                            # :124 / :225
    attn = q @ k.transpose(-2, -1)
    attn = attn + table_bias(p, window).unsqueeze(0)
    attn = _softmax_with_mask(attn, mask, num_heads)
    out = (attn @ v).transpose(1, 2).reshape(B_, N, C)
    return F.linear(out, p["proj.weight"], p["proj.bias"])


# ----------------------------------------------------------------------------------------
# a7 / a10: blocks
# ----------------------------------------------------------------------------------------
def _sub(p: Dict[str, Tensor], prefix: str) -> Dict[str, Tensor]:
    L = len(prefix)
    return {k[L:]: v for k, v in p.items() if k.startswith(prefix)}


def _ln(x, p, name):
    return F.layer_norm(x, (x.shape[-1],), p[name + ".weight"], p[name + ".bias"], 1e-5)


def _mlp(x, p, name):
    """fc1 -> GELU -> fc2 (swin_v2_module.py:26-32; swinfusion_module.py:24-30)."""
    return F.linear(F.gelu(F.linear(x, p[name + ".fc1.weight"], p[name + ".fc1.bias"])),
                    p[name + ".fc2.weight"], p[name + ".fc2.bias"])


def _windowed(x: Tensor, grid, window, shift, fn):
    """roll -> partition -> fn(windows) -> reverse -> roll back (swin_v2_module.py:274-297)."""
    B, L, C = x.shape
    n = len(grid)
    xs = cyclic_shift_nd(x.view(B, *grid, C), shift)
    xw = window_partition_nd(xs, window).view(-1, int(math.prod(window)), C)
    return xw, (lambda aw: cyclic_shift_nd(
        window_reverse_nd(aw.view(-1, *window, C), window, grid), shift, inverse=True).reshape(B, L, C))


def swin_v2_block(x: Tensor, p: Dict[str, Tensor], grid: Sequence[int], window: int, shift: int,
                  num_heads: int) -> Tensor:
    """Post-norm SwinV2 block, no drop-path (swin_v2_module.py:268-304)."""
    n = len(grid)
    window, shift = effective_window(grid, window, shift)
    w, s = _tup(window, n), _tup(shift, n)
    mask = shift_mask_nd(grid, w, s, x.dtype) if shift > 0 else None
    xw, back = _windowed(x, grid, w, s, None)
    a = back(window_attention_cosine(xw, _sub(p, "attn."), w, num_heads, mask))
    x = x + _ln(a, p, "norm1")
    return x + _ln(_mlp(x, p, "mlp"), p, "norm2")


def fusion_block(x: Tensor, p: Dict[str, Tensor], x_size: Sequence[int], input_resolution: Sequence[int],
                 window: int, shift: int, num_heads: int) -> Tensor:
    """Pre-norm self block (swinfusion_module.py:340-380).  The window/shift clamp uses
    `input_resolution` (ctor, :294-297) while the mask uses `x_size` (:360-363)."""
    n = len(x_size)
    window, shift = effective_window(input_resolution, window, shift)
    w, s = _tup(window, n), _tup(shift, n)
    mask = shift_mask_nd(x_size, w, s, x.dtype) if shift > 0 else None
    xw, back = _windowed(_ln(x, p, "norm1"), x_size, w, s, None)
    x = x + back(window_attention_scaled(xw, _sub(p, "attn."), w, num_heads, mask))
    return x + _mlp(_ln(x, p, "norm2"), p, "mlp")


def cross_block(x: Tensor, y: Tensor, p: Dict[str, Tensor], x_size: Sequence[int],
                input_resolution: Sequence[int], window: int, shift: int,
                num_heads: int) -> Tuple[Tensor, Tensor]:
    """Pre-norm cross-modal block (swinfusion_module.py:484-540)."""
    n = len(x_size)
    window, shift = effective_window(input_resolution, window, shift)
    w, s = _tup(window, n), _tup(shift, n)
    mask = shift_mask_nd(x_size, w, s, x.dtype) if shift > 0 else None
    xw, back_x = _windowed(_ln(x, p, "norm1_A"), x_size, w, s, None)
    yw, back_y = _windowed(_ln(y, p, "norm1_B"), x_size, w, s, None)
    ax = back_x(window_attention_scaled(xw, _sub(p, "attn_A."), w, num_heads, mask, y=yw))
    ay = back_y(window_attention_scaled(yw, _sub(p, "attn_B."), w, num_heads, mask, y=xw))
    x = x + ax
    x = x + _mlp(_ln(x, p, "norm2_A"), p, "mlp_A")
    y = y + ay
    y = y + _mlp(_ln(y, p, "norm2_B"), p, "mlp_B")
    return x, y


# ----------------------------------------------------------------------------------------
# a12: fairseq-style multi-head attention        modules/multihead_attention.py:51-134
# ----------------------------------------------------------------------------------------
def multihead_attention(query: Tensor, key: Tensor, value: Tensor, p: Dict[str, Tensor], num_heads: int,
                        attn_mask: Optional[Tensor] = None, keep: Optional[Tensor] = None) -> Tuple[Tensor, Tensor]:
    """(T,B,E),(S,B,E),(S,B,E) -> ((T,B,E), head-averaged weights (B,T,S)); eval mode, or with `keep` (B*nH, T, S)
    (oracle/philox.py: 0 or 1/(1-p)) the training-mode attention dropout (:123), which both outputs see.
    The three projection branches of the reference (:69-84) are numerically the same
    slicing of in_proj_weight, so one code path restates all of them."""
    T, B, E = query.shape
    d = E // num_heads
    W, b = p["in_proj_weight"], p.get("in_proj_bias")
    sl = lambda t, a, z: None if t is None else t[a:z]
    q = F.linear(query, W[:E], sl(b, 0, E)) * d ** -0.5                                     # :85
    k = F.linear(key, W[E:2 * E], sl(b, E, 2 * E))
    v = F.linear(value, W[2 * E:], sl(b, 2 * E, 3 * E))
    q = q.contiguous().view(T, B * num_heads, d).transpose(0, 1)
    k = k.contiguous().view(-1, B * num_heads, d).transpose(0, 1)
    v = v.contiguous().view(-1, B * num_heads, d).transpose(0, 1)
    S = k.size(1)
    w = torch.bmm(q, k.transpose(1, 2))
    if attn_mask is not None:
        w = w + attn_mask.unsqueeze(0)                                                      # :112-118
    w = F.softmax(w.float(), dim=-1).type_as(w)                                             # :120
    if keep is not None:
        w = w * keep.to(w.dtype)                                                            # :123
    a = torch.bmm(w, v).transpose(0, 1).contiguous().view(T, B, E)
    a = F.linear(a, p["out_proj.weight"], p.get("out_proj.bias"))
    return a, w.view(B, num_heads, T, S).sum(dim=1) / num_heads


# ----------------------------------------------------------------------------------------
# a14: future mask                               modules/crossmodal_transformer.py:174-186
# ----------------------------------------------------------------------------------------
def future_mask(T: int, S: Optional[int] = None, dtype=torch.float32) -> Tensor:
    S = T if S is None else S
    m = torch.triu(torch.full((T, S), float("-inf"), dtype=torch.float32), 1 + abs(S - T))
    return m.to(dtype)


# ----------------------------------------------------------------------------------------
# a16: sinusoidal positions                      modules/position_embedding.py:8-27,41-75
# ----------------------------------------------------------------------------------------
def sinusoidal_table(num: int, dim: int, padding_idx: int = 0) -> Tensor:
    half = dim // 2
    f = torch.exp(torch.arange(half, dtype=torch.float) * -(math.log(10000) / (half - 1)))
    e = torch.arange(num, dtype=torch.float).unsqueeze(1) * f.unsqueeze(0)
    e = torch.cat([torch.sin(e), torch.cos(e)], dim=1).view(num, -1)
    if dim % 2 == 1:
        e = torch.cat([e, torch.zeros(num, 1)], dim=1)
    e[padding_idx, :] = 0
    return e


def token_positions(tokens: Tensor, padding_idx: int = 0) -> Tensor:
    """(B,T) float 'tokens' -> int64 positions: t+1 where token != padding_idx else the
    token value itself cast to long, i.e. 0 (position_embedding.py:21-27, left_pad=0)."""
    Bsz, T = tokens.shape
    rng = torch.arange(padding_idx + 1, padding_idx + 1 + T).to(tokens.dtype).expand(Bsz, T)
    return torch.where(tokens.ne(padding_idx), rng, tokens).long()


def sinusoidal_positions(tokens: Tensor, dim: int) -> Tensor:
    """(B,T) -> (B,T,dim), detached (position_embedding.py:62-75)."""
    Bsz, T = tokens.shape
    tab = sinusoidal_table(1 + T, dim).to(tokens.dtype)
    return tab.index_select(0, token_positions(tokens).flatten()).view(Bsz, T, -1).detach()


# ----------------------------------------------------------------------------------------
# a13 / a15: encoder layer and encoder           modules/crossmodal_transformer.py:49-90,133-165
# ----------------------------------------------------------------------------------------
def encoder_layer(x: Tensor, p: Dict[str, Tensor], num_heads: int, use_mask: bool,
                  x_k: Optional[Tensor] = None, x_v: Optional[Tensor] = None) -> Tensor:
    res = x
    x = _ln(x, p, "layer_norms.0")
    mask = future_mask(x.shape[0], None if x_k is None else x_k.shape[0], x.dtype) if use_mask else None
    if x_k is None and x_v is None:
        a, _ = multihead_attention(x, x, x, _sub(p, "self_attn."), num_heads, mask)
    else:
        a, _ = multihead_attention(x, _ln(x_k, p, "layer_norms.0"), _ln(x_v, p, "layer_norms.0"),
                                   _sub(p, "self_attn."), num_heads, mask)                  # :150-152
    x = res + a
    res = x
    x = _ln(x, p, "layer_norms.1")
    x = F.linear(F.relu(F.linear(x, p["fc1.weight"], p["fc1.bias"])), p["fc2.weight"], p["fc2.bias"])
    return res + x


def transformer_encoder(x_in: Tensor, p: Dict[str, Tensor], num_heads: int, num_layers: int, use_mask: bool,
                        x_in_k: Optional[Tensor] = None, x_in_v: Optional[Tensor] = None) -> Tensor:
    E = x_in.shape[-1]
    emb = lambda t: math.sqrt(E) * t + sinusoidal_positions(t.transpose(0, 1)[:, :, 0], E).transpose(0, 1)
    x = emb(x_in)
    cross = x_in_k is not None and x_in_v is not None
    if cross:
        x_k, x_v = emb(x_in_k), emb(x_in_v)
    for i in range(num_layers):
        lp = _sub(p, f"layers.{i}.")
        x = encoder_layer(x, lp, num_heads, use_mask, x_k, x_v) if cross else encoder_layer(x, lp, num_heads, use_mask)
    return _ln(x, p, "layer_norm")


# ----------------------------------------------------------------------------------------
# Core-only attention (what the CUDA kernels compute between the projections): used by the
# GPU parity tests to check the kernels in isolation on already-projected q,k,v.
# ----------------------------------------------------------------------------------------
def window_attention_core(q: Tensor, k: Tensor, v: Tensor, grid: Sequence[int], window: Sequence[int],
                          shift: Sequence[int], num_heads: int, *, cosine: bool, scale: float = 1.0,
                          head_scale: Optional[Tensor] = None, bias: Optional[Tensor] = None,
                          mask: Optional[Tensor] = None, keep: Optional[Tensor] = None) -> Tuple[Tensor, Tensor]:
    """q,k,v: (B, *grid, C) un-windowed.  Returns (out (B,*grid,C), lse (B*nW, nH, N)).
    Same maths as a6/a8 between `qkv = linear(x)` and `proj`, with the roll/partition/
    reverse/roll-back of the block around it.  keep: attention dropout, (B*nW*nH, N, N) factors 0 or 1/(1-p)
    (oracle/philox.py) that multiply the probabilities before `@ v`; lse is unaffected."""
    B, C = q.shape[0], q.shape[-1]
    n = len(grid)
    window, shift = _tup(window, n), _tup(shift, n)
    N = int(math.prod(window))
    d = C // num_heads

    def win(t):
        tw = window_partition_nd(cyclic_shift_nd(t, shift), window).view(-1, N, num_heads, d)
        return tw.permute(0, 2, 1, 3)

    qw, kw, vw = win(q), win(k), win(v)
    if cosine:
        attn = F.normalize(qw, dim=-1) @ F.normalize(kw, dim=-1).transpose(-2, -1)
        attn = attn * head_scale.view(1, num_heads, 1, 1)
    else:
        attn = (qw * scale) @ kw.transpose(-2, -1)
    if bias is not None:
        attn = attn + bias.unsqueeze(0)
    if mask is not None:
        nW = mask.shape[0]
        attn = (attn.view(-1, nW, num_heads, N, N) + mask.unsqueeze(1).unsqueeze(0)).view(-1, num_heads, N, N)
    lse = torch.logsumexp(attn, dim=-1)
    probs = attn.softmax(-1)
    if keep is not None:
        probs = probs * keep.to(probs.dtype).view(-1, num_heads, N, N)
    out = (probs @ vw).transpose(1, 2).reshape(-1, *window, C)
    out = cyclic_shift_nd(window_reverse_nd(out, window, grid), shift, inverse=True)
    return out, lse
