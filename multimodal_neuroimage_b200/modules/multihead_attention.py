"""Drop-in replacement for the reference's modules/multihead_attention.py
(fairseq-derived MultiheadAttention), with the attention core -- q*scaling, QK^T, additive
mask, fp32 softmax, dropout, PV -- in one CUDA kernel call (torch.ops.mmn_b200.mha_fwd).

Same constructor arguments, forward signature and state_dict keys (`in_proj_weight`,
`in_proj_bias`, `out_proj.*`, optional `bias_k`/`bias_v`).  Differences, all documented in
DESIGN.md: the (B*nH, T, S) score tensor is never materialised; the head-averaged weights
the reference returns (multihead_attention.py:131-133) are produced by a second small
kernel only when `need_weights` is true (default, for API compatibility) and are detached;
a causal mask produced by `buffered_future_mask` is recognised by identity and generated
inside the kernel from indices instead of being read from memory.
"""
from __future__ import annotations

import torch
import torch.nn.functional as F
from torch import nn
from torch.nn import Parameter

from .. import _lib, geometry, ops


_future_masks = {}


def cached_future_mask(tgt_len: int, src_len: int, device) -> torch.Tensor:
    """Dense (T,S) {0,-inf} future mask, built once per (T, S, device) ON the device (the
    reference rebuilds it on the CPU and copies it for every layer of every forward)."""
    key = (int(tgt_len), int(src_len), str(device))
    m = _future_masks.get(key)
    if m is None:
        m = geometry.future_mask(tgt_len, src_len, dtype=torch.float32, device=device)
        _future_masks[key] = m
    return m


def future_mask_diagonal_of(mask):
    """If `mask` IS one of the cached future masks return its diagonal (so the kernel can
    regenerate the pattern from indices instead of reading the tensor), else None."""
    if mask is None or mask.dim() != 2:
        return None
    key = (mask.shape[0], mask.shape[1], str(mask.device))
    return geometry.future_mask_diagonal(mask.shape[0], mask.shape[1]) if _future_masks.get(key) is mask else None


class _SplitRows(torch.autograd.Function):
    """t -> row blocks t[0:s0], t[s0:s0+s1], ... (views), with the gradient assembled by ONE torch.cat.  Autograd's own
    slicing gives every block a SliceBackward -- a zero fill of the full tensor, a device-to-device memcpy into the slice and
    an add of the partial gradients -- and inside a CUDA graph each of those memcpy nodes costs ~8 us of dependency latency
    between kernel nodes (tools/find_memcpy.py: 48 of them per cfg4 training step, all from the in-projection slices)."""

    @staticmethod
    def forward(ctx, t, *sizes):
        ctx.sizes = sizes
        ctx.set_materialize_grads(False)
        ctx.like = (t.shape[1:], t.dtype, t.device)
        return tuple(t.split(list(sizes), dim=0))

    @staticmethod
    def backward(ctx, *grads):
        shape, dtype, device = ctx.like
        parts = [g if g is not None else torch.zeros((n,) + tuple(shape), dtype=dtype, device=device)
                 for g, n in zip(grads, ctx.sizes)]
        return (torch.cat(parts, dim=0),) + (None,) * len(ctx.sizes)


class MultiheadAttention(nn.Module):
    def __init__(self, embed_dim, num_heads_mult, attn_dropout=0., bias=True, add_bias_kv=False, add_zero_attn=False):
        super().__init__()
        self.embed_dim = embed_dim
        self.num_heads_mult = num_heads_mult
        self.attn_dropout = attn_dropout
        self.head_dim = embed_dim // num_heads_mult
        assert self.head_dim * num_heads_mult == self.embed_dim, "embed_dim must be divisible by num_heads_mult"
        self.scaling = self.head_dim ** -0.5
        self.in_proj_weight = Parameter(torch.Tensor(3 * embed_dim, embed_dim))
        self.register_parameter('in_proj_bias', None)
        if bias:
            self.in_proj_bias = Parameter(torch.Tensor(3 * embed_dim))
        self.out_proj = nn.Linear(embed_dim, embed_dim, bias=bias)
        if add_bias_kv:
            self.bias_k = Parameter(torch.Tensor(1, 1, embed_dim))
            self.bias_v = Parameter(torch.Tensor(1, 1, embed_dim))
        else:
            self.bias_k = self.bias_v = None
        self.add_zero_attn = add_zero_attn
        self.need_weights = True
        self.reset_parameters()

    def reset_parameters(self):
        nn.init.xavier_uniform_(self.in_proj_weight)
        nn.init.xavier_uniform_(self.out_proj.weight)
        if self.in_proj_bias is not None:
            nn.init.constant_(self.in_proj_bias, 0.)
            nn.init.constant_(self.out_proj.bias, 0.)
        if self.bias_k is not None:
            nn.init.xavier_normal_(self.bias_k)
        if self.bias_v is not None:
            nn.init.xavier_normal_(self.bias_v)

    def forward(self, query, key, value, attn_mask=None, need_weights=None):
        """query (T,B,E), key/value (S,B,E) -> (attn (T,B,E), head-averaged weights (B,T,S) | None)."""
        tgt_len, bsz, embed_dim = query.size()
        assert embed_dim == self.embed_dim
        assert key.size() == value.size()
        # Projection branches as in the reference (multihead_attention.py:59-84): identical
        # tensors share one GEMM; the results are the same slices of in_proj_weight.
        # Head dims the tensor-core kernels do not take (the reference's own 7 and 14: embed 84 / 168, 12 heads) run on them
        # all the same when the projections compute in 16 bits anyway (autocast): each head is padded to 32 (or 64) channels
        # by zero ROWS in the in-projection weights -- q, k, v come out of the GEMM already padded, 64-byte aligned per head --
        # and zero COLUMNS in the out-projection weight.  Zero channels change neither q.k nor the output; the gradient
        # reaches the true weights through the pad.  (fp32 calls keep the exact generic kernels.)
        pad = self._padded_head_dim(query)
        E = self.embed_dim
        if query is key and key is value or (query.data_ptr() == key.data_ptr() == value.data_ptr()):
            q, k, v = self._project(query, self.in_proj_weight, self.in_proj_bias, pad).chunk(3, dim=-1)
        elif key is value or key.data_ptr() == value.data_ptr():
            (wq, wkv), (bq, bkv) = self._split_in_proj(E, 2 * E)
            q = self._project(query, wq, bq, pad)
            k, v = self._project(key, wkv, bkv, pad).chunk(2, dim=-1)
        else:
            (wq, wk, wv), (bq, bk, bv) = self._split_in_proj(E, E, E)
            q = self._project(query, wq, bq, pad)
            k = self._project(key, wk, bk, pad)
            v = self._project(value, wv, bv, pad)

        diagonal = future_mask_diagonal_of(attn_mask)
        if self.bias_k is not None:
            k = torch.cat([k, self._pad_heads(self.bias_k, pad).to(k.dtype).repeat(1, bsz, 1)])
            v = torch.cat([v, self._pad_heads(self.bias_v, pad).to(v.dtype).repeat(1, bsz, 1)])
            if attn_mask is not None:
                attn_mask = torch.cat([attn_mask, attn_mask.new_zeros(attn_mask.size(0), 1)], dim=1)
                diagonal = None
        if self.add_zero_attn:
            k = torch.cat([k, k.new_zeros((1,) + k.size()[1:])], dim=0)
            v = torch.cat([v, v.new_zeros((1,) + v.size()[1:])], dim=0)
            if attn_mask is not None:
                attn_mask = torch.cat([attn_mask, attn_mask.new_zeros(attn_mask.size(0), 1)], dim=1)
                diagonal = None

        if attn_mask is None:
            kind, diag, mask = _lib.MASK_NONE, 0, None
        elif diagonal is not None:
            kind, diag, mask = _lib.MASK_FUTURE, diagonal, None
        else:
            kind, diag = _lib.MASK_TENSOR, 0
            mask = attn_mask.to(device=q.device, dtype=torch.float32).contiguous()

        p, seed, off, rng = ops.next_dropout_stream(self.attn_dropout, self.training, q.device)
        io = q.dtype                                   # float16 under the reference trainer's autocast: kernels run it as bf16
        q, k, v = ops.kernel_io(q), ops.kernel_io(k), ops.kernel_io(v)
        attn, lse = torch.ops.mmn_b200.mha_fwd(q, k, v, mask, self.num_heads_mult, kind, diag, float(self.scaling),
                                               p, seed, off, rng)
        if pad:
            w_out = F.pad(self.out_proj.weight.view(E, self.num_heads_mult, self.head_dim), (0, pad - self.head_dim))
            attn = F.linear(attn.to(io), w_out.reshape(E, self.num_heads_mult * pad), self.out_proj.bias)
        else:
            attn = self.out_proj(attn.to(io))
        need = self.need_weights if need_weights is None else need_weights
        weights = None
        if need:
            with torch.no_grad():
                weights = torch.ops.mmn_b200.mha_avg_weights(q.detach(), k.detach(), mask, lse, self.num_heads_mult, kind,
                                                             diag, float(self.scaling), p, seed, off, rng).to(attn.dtype)
        return attn, weights

    def in_proj_qkv(self, query):
        return self._in_proj(query).chunk(3, dim=-1)

    def in_proj_kv(self, key):
        return self._in_proj(key, start=self.embed_dim).chunk(2, dim=-1)

    def in_proj_q(self, query, **kwargs):
        return self._in_proj(query, end=self.embed_dim, **kwargs)

    def in_proj_k(self, key):
        return self._in_proj(key, start=self.embed_dim, end=2 * self.embed_dim)

    def in_proj_v(self, value):
        return self._in_proj(value, start=2 * self.embed_dim)

    def _padded_head_dim(self, query):
        """0, or the head dim (32 / 64) the tensor-core kernels run this module at: CUDA, 16-bit projections, head_dim that
        is not 32 / 64 itself and fits."""
        d = self.head_dim
        if not query.is_cuda or d in (32, 64) or d > 64:
            return 0
        dt = torch.get_autocast_dtype("cuda") if torch.is_autocast_enabled("cuda") else query.dtype
        if dt not in (torch.bfloat16, torch.float16):
            return 0
        return 32 if d < 32 else 64

    def _pad_heads(self, t, pad):
        """(..., heads * head_dim) -> (..., heads * pad) with zero channels at the end of every head."""
        if not pad:
            return t
        lead = t.shape[:-1]
        return F.pad(t.reshape(*lead, self.num_heads_mult, self.head_dim), (0, pad - self.head_dim)).reshape(*lead, self.num_heads_mult * pad)

    def _split_in_proj(self, *sizes):
        """Row blocks of in_proj_weight / in_proj_bias whose gradients come back through one torch.cat (_SplitRows)."""
        w = _SplitRows.apply(self.in_proj_weight, *sizes)
        b = _SplitRows.apply(self.in_proj_bias, *sizes) if self.in_proj_bias is not None else (None,) * len(sizes)
        return w, b

    def _in_proj(self, input, start=0, end=None, pad=0, **kwargs):
        weight = kwargs.get('weight', self.in_proj_weight)
        bias = kwargs.get('bias', self.in_proj_bias)
        weight = weight[start:end, :]
        if bias is not None:
            bias = bias[start:end]
        return self._project(input, weight, bias, pad)

    def _project(self, input, weight, bias, pad=0):
        """F.linear with the rows of `weight` / `bias` (whole heads) zero-padded per head to `pad` channels (0: as they are)."""
        if pad:                                       # zero rows after every head's head_dim rows: the output is head-padded
            nb = weight.shape[0] // self.embed_dim
            weight = F.pad(weight.view(nb * self.num_heads_mult, self.head_dim, -1), (0, 0, 0, pad - self.head_dim))
            weight = weight.reshape(nb * self.num_heads_mult * pad, -1)
            if bias is not None:
                bias = self._pad_heads(bias.view(nb, -1), pad).reshape(-1)
        return F.linear(input, weight, bias)
