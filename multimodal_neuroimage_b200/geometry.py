"""Integer index maps of the window-attention hot path, n-D (n in {1,2,3}), in closed form.

Host-side only (built once per module, on the CPU, as the reference does in its
constructors); the CUDA kernels evaluate the same closed forms per thread and never read
these tensors, except for `state_dict` compatibility buffers (`attn_mask`,
`relative_position_index`, `relative_coords_table`).  Bit-exactness against the reference
is asserted in tests/ (through the oracle and the golden fixtures).

Closed forms (SURVEY.md 8a; reference: modules/swin_v2_module.py:35-62,95-124,244-266):
  window id      n = sum_a (c_a // w_a) * prod_{b>a} nW_b          (row-major over windows)
  in-window pos  p = sum_a (c_a %  w_a) * prod_{b>a} w_b
  shifted gather window n, pos p  <-  source coordinate ((i_a*w_a + a_a + s_a) mod L_a)_a
  region id      per axis 0 if v < L-w, 1 if v < L-s, else 2 (v in the shifted frame),
                 combined row-major with 3 slots per shifted axis; mask = 0 if equal else -100
  rel-pos index  sum_a (delta_a + w_a - 1) * prod_{b>a} (2 w_b - 1)
"""
from __future__ import annotations

import math
from typing import Optional, Sequence, Tuple

import torch


def as_tuple(v, n: int) -> Tuple[int, ...]:
    if isinstance(v, (tuple, list)):
        if len(v) != n:
            raise ValueError(f"expected {n} values, got {v}")
        return tuple(int(x) for x in v)
    return (int(v),) * n


def clamp_window(resolution: Sequence[int], window: int, shift: int) -> Tuple[int, int]:
    """A stage no larger than the window is attended whole and never shifted
    (swin_v2_module.py:226-229; swinfusion_module.py:294-297,429-432)."""
    if min(resolution) <= window:
        return int(min(resolution)), 0
    return int(window), int(shift)


def _axis_coords(grid: Sequence[int]) -> torch.Tensor:
    """(n, prod(grid)) int64 coordinates of every token in row-major order."""
    axes = [torch.arange(g, dtype=torch.int64) for g in grid]
    mesh = torch.meshgrid(*axes, indexing="ij")
    return torch.stack([m.reshape(-1) for m in mesh])


def window_gather_map(grid: Sequence[int], window: Sequence[int], shift: Sequence[int]) -> torch.Tensor:
    """(nW, N) int64: flat source-token index (un-shifted frame) of each (window, position)."""
    n = len(grid)
    window, shift = as_tuple(window, n), as_tuple(shift, n)
    counts = [g // w for g, w in zip(grid, window)]
    wi = _axis_coords(counts)            # n, nW
    ai = _axis_coords(window)            # n, N
    flat = torch.zeros(wi.shape[1], ai.shape[1], dtype=torch.int64)
    for a in range(n):
        c = (wi[a][:, None] * window[a] + ai[a][None, :] + shift[a]) % grid[a]
        flat = flat * grid[a] + c
    return flat


def shift_region_ids(grid: Sequence[int], window: Sequence[int], shift: Sequence[int]) -> torch.Tensor:
    """(nW, N) int64 region id of every (window, position) of the shifted frame."""
    n = len(grid)
    window, shift = as_tuple(window, n), as_tuple(shift, n)
    counts = [g // w for g, w in zip(grid, window)]
    wi, ai = _axis_coords(counts), _axis_coords(window)
    rid = torch.zeros(wi.shape[1], ai.shape[1], dtype=torch.int64)
    for a in range(n):
        v = wi[a][:, None] * window[a] + ai[a][None, :]
        if shift[a] > 0:
            r = (v >= grid[a] - window[a]).long() + (v >= grid[a] - shift[a]).long()
            rid = rid * 3 + r
    return rid


def shift_attention_mask(grid: Sequence[int], window: Sequence[int], shift: Sequence[int],
                         dtype=torch.float32) -> Optional[torch.Tensor]:
    """(nW, N, N) additive {0,-100} mask, or None when nothing is shifted."""
    n = len(grid)
    if not any(as_tuple(shift, n)):
        return None
    rid = shift_region_ids(grid, window, shift)
    same = rid[:, :, None] == rid[:, None, :]
    mask = torch.full(same.shape, -100.0, dtype=dtype)
    mask[same] = 0.0
    return mask


def relative_position_index(window: Sequence[int]) -> torch.Tensor:
    """(N, N) int64 index into the (prod(2w-1))-entry bias table."""
    window = tuple(int(w) for w in window)
    ai = _axis_coords(window)
    idx = torch.zeros(ai.shape[1], ai.shape[1], dtype=torch.int64)
    for a, w in enumerate(window):
        idx = idx * (2 * w - 1) + (ai[a][:, None] - ai[a][None, :] + (w - 1))
    return idx


def inverse_index(index: torch.Tensor, table_rows: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """Inverse of a (NN,) bias-table index in CSR form, on the index's device: (perm, offsets) int32 with perm = the entries
    e sorted by (index[e], e) and offsets (table_rows + 1) the start of each table entry's run, offsets[-1] = NN.  What the
    deterministic table-gradient gather walks (csrc/cpb_bias.cu: each entry sums its dbias values in increasing e)."""
    index = index.reshape(-1)
    srt, perm = torch.sort(index, stable=True)
    offsets = torch.searchsorted(srt, torch.arange(table_rows + 1, dtype=index.dtype, device=index.device))
    return perm.to(torch.int32), offsets.to(torch.int32)


def cpb_coords_table(window: Sequence[int], pretrained_window: Optional[Sequence[int]] = None) -> torch.Tensor:
    """(1, 2w_0-1, ..., n) fp32: sign(x)*log2(|x|+1)/log2(8) of 8*delta/(w-1)."""
    window = tuple(int(w) for w in window)
    n = len(window)
    pre = None
    if pretrained_window is not None and int(pretrained_window[0]) > 0:
        pre = tuple(int(p) for p in pretrained_window)
    cols = []
    for a, w in enumerate(window):
        rel = torch.arange(-(w - 1), w, dtype=torch.float32)
        rel = rel / float((pre[a] if pre else w) - 1)
        shape = [1] * n
        shape[a] = 2 * w - 1
        cols.append(rel.view(shape).expand([2 * x - 1 for x in window]))
    table = torch.stack(cols, dim=-1).unsqueeze(0).contiguous()
    table = table * 8
    return torch.sign(table) * torch.log2(torch.abs(table) + 1.0) / math.log2(8)


def future_mask_diagonal(tgt_len: int, src_len: int) -> int:
    """Entries with j - i >= this are -inf (crossmodal_transformer.py:183)."""
    return 1 + abs(int(src_len) - int(tgt_len))


def future_mask(tgt_len: int, src_len: Optional[int] = None, dtype=torch.float32, device=None) -> torch.Tensor:
    src_len = tgt_len if src_len is None else src_len
    i = torch.arange(tgt_len, device=device)[:, None]
    j = torch.arange(src_len, device=device)[None, :]
    m = torch.zeros(tgt_len, src_len, dtype=dtype, device=device)
    return m.masked_fill(j - i >= future_mask_diagonal(tgt_len, src_len), float("-inf"))


def shard_range(total: int, world_size: int, rank: int) -> Tuple[int, int]:
    """Contiguous [lo, hi) slice of `total` independent units for `rank` (batch sharding:
    the only partitioning the path has, SURVEY.md 8e).  Remainders go to the low ranks."""
    base, rem = divmod(int(total), int(world_size))
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)
