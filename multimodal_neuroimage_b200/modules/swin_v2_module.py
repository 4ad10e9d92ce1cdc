"""Drop-in replacements for the classes of the reference's modules/swin_v2_module.py,
backed by the fused CUDA window-attention op and generalised from 2-D to n-D windows.

Same class names, constructor arguments, forward signatures and state_dict keys/shapes as
the reference (SURVEY.md 8b), so `model.py` builds them unchanged and reference `.pth`
files load.  What differs is where the work happens: `SwinTransformerBlock.forward` never
rolls, partitions or reverses anything in PyTorch -- it hands the un-windowed (B,*grid,3C)
qkv tensor to `torch.ops.mmn_b200.winattn_fwd`, which gathers the shifted windows, applies
cosine attention with the continuous-position bias and the shift mask (generated in the
kernel) and scatters the result back in place.  The reference's per-forward host->device
scalar copy (swin_v2_module.py:154) is gone: the clamp constant is a Python float.
"""
from __future__ import annotations

import math
from typing import Optional, Sequence

import numpy as np  # noqa: F401  (star-exported: the reference's model.py takes `np` from here, model.py:15)
import torch
import torch.nn as nn
import torch.nn.functional as F
import torch.utils.checkpoint as checkpoint
from torch.nn.init import trunc_normal_  # noqa: F401  (the reference re-exports timm's; model.py:625,680,1085 call it)

from .. import _lib, fused, geometry, ops

_LOGIT_MAX = math.log(1.0 / 0.01)


def to_ntuple(x, n=2):
    return geometry.as_tuple(x, n)


def to_2tuple(x):
    return geometry.as_tuple(x, 2)


class DropPath(nn.Module):
    """Stochastic depth per sample (the reference takes this from timm)."""

    def __init__(self, drop_prob: float = 0.0):
        super().__init__()
        self.drop_prob = float(drop_prob)

    def forward(self, x):
        if self.drop_prob == 0.0 or not self.training:
            return x
        keep = 1.0 - self.drop_prob
        shape = (x.shape[0],) + (1,) * (x.dim() - 1)
        return x * x.new_empty(shape).bernoulli_(keep).div_(keep)


class Mlp(nn.Module):
    """fc1 -> act -> drop -> fc2 -> drop (swin_v2_module.py:16-32)."""

    def __init__(self, in_features, hidden_features=None, out_features=None, act_layer=nn.GELU, drop=0.):
        super().__init__()
        out_features = out_features or in_features
        hidden_features = hidden_features or in_features
        self.fc1 = nn.Linear(in_features, hidden_features)
        self.act = act_layer()
        self.fc2 = nn.Linear(hidden_features, out_features)
        self.drop = nn.Dropout(drop)

    def forward(self, x):
        if isinstance(self.act, nn.GELU) and getattr(self.act, "approximate", "none") == "none":
            # two tensor-core GEMMs, bias + GELU in the first one's epilogue (fused.MlpFn); plain F.linear off the fast path
            return fused.mlp(x, self.fc1, self.fc2, "gelu", self.drop.p, self.training)
        return self.drop(self.fc2(self.drop(self.act(self.fc1(x)))))


def window_partition(x, window_size):
    """(B, *grid, C) -> (B*nW, *window, C).  Kept for API compatibility (star-exported by
    the reference, swin_v2_module.py:35-46); the blocks below never call it."""
    n = x.dim() - 2
    ws = to_ntuple(window_size, n)
    idx = geometry.window_gather_map(x.shape[1:-1], ws, (0,) * n).to(x.device)
    flat = x.reshape(x.shape[0], -1, x.shape[-1])
    return flat[:, idx.reshape(-1)].reshape(-1, *ws, x.shape[-1])


def window_reverse(windows, window_size, *grid):
    """(B*nW, *window, C) -> (B, *grid, C) (swin_v2_module.py:49-62)."""
    n = len(grid)
    ws = to_ntuple(window_size, n)
    idx = geometry.window_gather_map(grid, ws, (0,) * n).reshape(-1).to(windows.device)
    L = idx.numel()
    B = windows.shape[0] * math.prod(ws) // L
    flat = windows.reshape(B, L, -1)
    out = torch.empty_like(flat)
    out[:, idx] = flat
    return out.reshape(B, *grid, -1)


class _GatherRows(torch.autograd.Function):
    """table[index] for a (T, H) table and a fixed int64 index; backward = index_add_."""

    @staticmethod
    def forward(ctx, table, index):
        ctx.save_for_backward(index)
        ctx.rows = table.shape[0]
        return table.index_select(0, index)

    @staticmethod
    def backward(ctx, grad):
        index, = ctx.saved_tensors
        out = torch.zeros(ctx.rows, grad.shape[1], dtype=grad.dtype, device=grad.device)
        return out.index_add_(0, index, grad), None


class WindowAttention(nn.Module):
    """SwinV2 window attention: cosine similarity with a clamped learnable per-head logit
    scale and a log-spaced continuous relative position bias (swin_v2_module.py:65-195).
    `window_size` may have 2 or 3 entries."""

    def __init__(self, dim, window_size, num_heads_swin, qkv_bias=True, attn_drop=0., proj_drop=0.,
                 pretrained_window_size=[0, 0]):
        super().__init__()
        self.dim = dim
        self.window_size = tuple(int(w) for w in window_size)
        n = len(self.window_size)
        pws = pretrained_window_size
        if isinstance(pws, (list, tuple)):
            pws = tuple(int(p) for p in pws) if len(pws) == n else (int(pws[0]),) * n
        else:
            pws = (int(pws),) * n
        self.pretrained_window_size = pws
        self.num_heads_swin = num_heads_swin
        self.logit_scale = nn.Parameter(torch.log(10 * torch.ones((num_heads_swin, 1, 1))), requires_grad=True)
        self.cpb_mlp = nn.Sequential(nn.Linear(n, 512, bias=True), nn.ReLU(inplace=True),
                                     nn.Linear(512, num_heads_swin, bias=False))
        self.register_buffer("relative_coords_table",
                             geometry.cpb_coords_table(self.window_size, self.pretrained_window_size))
        self.register_buffer("relative_position_index", geometry.relative_position_index(self.window_size))
        self.qkv = nn.Linear(dim, dim * 3, bias=False)
        if qkv_bias:
            self.q_bias = nn.Parameter(torch.zeros(dim))
            self.v_bias = nn.Parameter(torch.zeros(dim))
        else:
            self.q_bias = None
            self.v_bias = None
        self.attn_drop = nn.Dropout(attn_drop)
        self.proj = nn.Linear(dim, dim)
        self.proj_drop = nn.Dropout(proj_drop)
        self.softmax = nn.Softmax(dim=-1)
        self.kernel_path = _lib.PATH_AUTO

    # -- pieces that stay in PyTorch: tiny, and they need autograd through learnable tables --
    def position_bias(self) -> torch.Tensor:
        """(nH, N, N) fp32 = 16*sigmoid(cpb_mlp(table))[index] (swin_v2_module.py:158-162).  The reference re-runs the
        MLP in every forward of every block; outside training (eval mode, or no gradient wanted) the table is a constant
        of the weights and is cached -- keyed on the weights' in-place version counters, so an optimizer step,
        `load_state_dict` or `.to()` invalidates it by construction."""
        params = (self.cpb_mlp[0].weight, self.cpb_mlp[0].bias, self.cpb_mlp[2].weight)
        cacheable = not (torch.is_grad_enabled() and any(p.requires_grad for p in params))
        if cacheable:
            key = tuple((p.data_ptr(), p._version) for p in params)
            hit = getattr(self, "_bias_cache", None)
            if hit is not None and hit[0] == key:
                return hit[1]
            with torch.no_grad():
                b = self._position_bias()
            self._bias_cache = (key, b)
            return b
        return self._position_bias()

    def _position_bias(self) -> torch.Tensor:
        N = math.prod(self.window_size)
        with torch.autocast(device_type="cuda", enabled=False):
            coords = self.relative_coords_table.float().reshape(-1, self.relative_coords_table.shape[-1])
            lin1, lin2 = self.cpb_mlp[0], self.cpb_mlp[2]
            if lin2.bias is None and ops.cpb_bias_supported(coords, lin1.weight, lin2.weight):
                # libmmn_b200 cpb_bias.cu: MLP + 16 sigmoid + gather in two launches, hand-written backward
                b, _ = torch.ops.mmn_b200.cpb_bias_fwd(coords, lin1.weight, lin1.bias, lin2.weight,
                                                       self.relative_position_index.view(-1))
                return b.view(-1, N, N)
            tab = self.cpb_mlp(self.relative_coords_table.float()).view(-1, self.num_heads_swin)
            # 16*sigmoid commutes with the gather: apply it on the (2w-1)^n-entry table, not on N*N entries, and
            # scatter the gradient back with one index_add_ instead of autograd's sort-based index backward
            b = _GatherRows.apply(16 * torch.sigmoid(tab), self.relative_position_index.view(-1))
            return b.view(N, N, -1).permute(2, 0, 1).contiguous().float()

    def head_scale(self) -> torch.Tensor:
        """(nH,) fp32 = exp(min(logit_scale, ln 100)) (swin_v2_module.py:154-155)."""
        return torch.clamp(self.logit_scale.float(), max=_LOGIT_MAX).exp().reshape(-1)

    def _qkv(self, x):
        bias = None
        if self.q_bias is not None:
            bias = torch.cat((self.q_bias, torch.zeros_like(self.v_bias, requires_grad=False), self.v_bias))
        return F.linear(x, self.qkv.weight, bias)

    def _core(self, qkv, grid, window, shift, mask_kind, mask):
        p, seed, off, rng = ops.next_dropout_stream(self.attn_drop.p, self.training, qkv.device)
        out, _ = torch.ops.mmn_b200.winattn_fwd(ops.kernel_io(qkv), None, self.position_bias(), self.head_scale(), mask,
                                                list(grid), list(window), list(shift), self.num_heads_swin,
                                                _lib.SCORE_COSINE, mask_kind, 1.0, p, seed, off, self.kernel_path, rng)
        return out.to(qkv.dtype)

    def forward(self, x, mask=None):
        """x: (num_windows*B, N, C) already partitioned; mask: (nW, N, N) additive or None."""
        B_, N, C = x.shape
        qkv = self._qkv(x)
        if mask is not None:
            mask = mask.to(device=x.device, dtype=torch.float32).contiguous()
        out = self._core(qkv, (N,), (N,), (0,), _lib.MASK_TENSOR if mask is not None else _lib.MASK_NONE, mask)
        return self.proj_drop(self.proj(out))

    def forward_grid(self, x, grid, shift):
        """x: (B, prod(grid), C) in the natural token order; the cyclic shift, the window
        gather/scatter and the shift mask all happen inside the kernel."""
        shifted = any(int(s) > 0 for s in shift)
        bias = None
        if self.q_bias is not None:
            bias = torch.cat((self.q_bias, torch.zeros_like(self.v_bias, requires_grad=False), self.v_bias))
        y = fused.window_attention_module(x, None, self.qkv.weight, bias, None, None, self.proj.weight, self.proj.bias,
                                          self.position_bias(), self.head_scale(), grid, self.window_size, shift,
                                          self.num_heads_swin, _lib.SCORE_COSINE,
                                          _lib.MASK_SHIFT if shifted else _lib.MASK_NONE, 1.0,
                                          ops.next_dropout_stream(self.attn_drop.p, self.training, x.device), self.kernel_path)
        return self.proj_drop(y)

    def extra_repr(self) -> str:
        return (f"dim={self.dim}, window_size={self.window_size}, "
                f"pretrained_window_size={self.pretrained_window_size}, num_heads_swin={self.num_heads_swin}")

    def flops(self, N):
        d = self.dim // self.num_heads_swin
        return N * self.dim * 3 * self.dim + 2 * self.num_heads_swin * N * d * N + N * self.dim * self.dim


class SwinTransformerBlock(nn.Module):
    """Post-norm SwinV2 block (swin_v2_module.py:198-322).  `input_resolution` may have 2
    or 3 entries; `window_size` / `shift_size` are ints applied to every axis."""

    def __init__(self, dim, input_resolution, num_heads_swin, window_size=4, shift_size=0, mlp_ratio=4., qkv_bias=True,
                 drop=0., attn_drop=0., drop_path=0., act_layer=nn.GELU, norm_layer=nn.LayerNorm,
                 pretrained_window_size=0):
        super().__init__()
        self.dim = dim
        self.input_resolution = tuple(int(r) for r in input_resolution)
        self.num_heads_swin = num_heads_swin
        self.mlp_ratio = mlp_ratio
        self.window_size, self.shift_size = geometry.clamp_window(self.input_resolution, window_size, shift_size)
        assert 0 <= self.shift_size < self.window_size, "shift_size must in 0-window_size"
        n = len(self.input_resolution)
        self.norm1 = norm_layer(dim)
        self.attn = WindowAttention(dim, window_size=to_ntuple(self.window_size, n), num_heads_swin=num_heads_swin,
                                    qkv_bias=qkv_bias, attn_drop=attn_drop, proj_drop=drop,
                                    pretrained_window_size=to_ntuple(pretrained_window_size, n))
        self.drop_path = DropPath(drop_path) if drop_path > 0. else nn.Identity()
        self.norm2 = norm_layer(dim)
        self.mlp = Mlp(in_features=dim, hidden_features=int(dim * mlp_ratio), act_layer=act_layer, drop=drop)
        # state_dict compatibility only: the kernel derives the same mask from the geometry.
        mask = None
        if self.shift_size > 0:
            mask = geometry.shift_attention_mask(self.input_resolution, to_ntuple(self.window_size, n),
                                                 to_ntuple(self.shift_size, n))
        self.register_buffer("attn_mask", mask)

    def forward(self, x):
        B, L, C = x.shape
        assert L == math.prod(self.input_resolution), "input feature has wrong size"
        n = len(self.input_resolution)
        a = self.attn.forward_grid(x, self.input_resolution, to_ntuple(self.shift_size, n))
        if isinstance(self.drop_path, nn.Identity) or not self.training:
            # x + norm(branch) in one pass each (csrc/layernorm.cu); the second output is x already cast for the Mlp's GEMM
            cd = fused._act_dtype(x)
            x, xc = fused.post_norm_add(x, a, self.norm1, cd if x.is_cuda and cd != x.dtype else None)
            m = self.mlp(xc if xc is not None else x)
            return fused.post_norm_add(x, m, self.norm2)[0]
        x = x + self.drop_path(self.norm1(a))
        return x + self.drop_path(self.norm2(self.mlp(x)))

    def extra_repr(self) -> str:
        return (f"dim={self.dim}, input_resolution={self.input_resolution}, num_heads_swin={self.num_heads_swin}, "
                f"window_size={self.window_size}, shift_size={self.shift_size}, mlp_ratio={self.mlp_ratio}")

    def flops(self):
        L = math.prod(self.input_resolution)
        N = self.window_size ** len(self.input_resolution)
        return 2 * self.dim * L + (L / N) * self.attn.flops(N) + 2 * L * self.dim * self.dim * self.mlp_ratio


class PatchMerging(nn.Module):
    """2x downsample per axis: concatenate the 2^n neighbours, Linear(2^n C -> 2C), norm
    (swin_v2_module.py:325-373; neighbour order there is (0,0),(1,0),(0,1),(1,1))."""

    def __init__(self, input_resolution, dim, norm_layer=nn.LayerNorm):
        super().__init__()
        self.input_resolution = tuple(int(r) for r in input_resolution)
        self.dim = dim
        n = len(self.input_resolution)
        self.reduction = nn.Linear((2 ** n) * dim, 2 * dim, bias=False)
        self.norm = norm_layer(2 * dim)

    def forward(self, x):
        B, L, C = x.shape
        res = self.input_resolution
        n = len(res)
        assert L == math.prod(res), "input feature has wrong size"
        assert all(r % 2 == 0 for r in res), f"x size {res} are not even."
        x = x.view(B, *res, C)
        parts = []
        for code in range(2 ** n):
            # first axis varies fastest, as in the reference's x0..x3 ordering
            sl = [slice(None)] + [slice((code >> a) & 1, None, 2) for a in range(n)] + [slice(None)]
            parts.append(x[tuple(sl)])
        x = torch.cat(parts, -1).view(B, -1, (2 ** n) * C)
        return self.norm(self.reduction(x))

    def extra_repr(self) -> str:
        return f"input_resolution={self.input_resolution}, dim={self.dim}"

    def flops(self):
        L = math.prod(self.input_resolution)
        n = len(self.input_resolution)
        return (L // 2 ** n) * (2 ** n) * self.dim * 2 * self.dim + L * self.dim // 2


class BasicLayer(nn.Module):
    """One stage: `depth` blocks alternating shift 0 / window//2, optional downsample
    (swin_v2_module.py:376-451)."""

    def __init__(self, dim, input_resolution, depth, num_heads_swin, window_size, mlp_ratio=4., qkv_bias=True, drop=0.,
                 attn_drop=0., drop_path=0., norm_layer=nn.LayerNorm, downsample=None, use_checkpoint=False,
                 pretrained_window_size=0):
        super().__init__()
        self.dim = dim
        self.input_resolution = input_resolution
        self.depth = depth
        self.use_checkpoint = use_checkpoint
        self.blocks = nn.ModuleList([
            SwinTransformerBlock(dim=dim, input_resolution=input_resolution, num_heads_swin=num_heads_swin,
                                 window_size=window_size, shift_size=0 if (i % 2 == 0) else window_size // 2,
                                 mlp_ratio=mlp_ratio, qkv_bias=qkv_bias, drop=drop, attn_drop=attn_drop,
                                 drop_path=drop_path[i] if isinstance(drop_path, list) else drop_path,
                                 norm_layer=norm_layer, pretrained_window_size=pretrained_window_size)
            for i in range(depth)])
        self.downsample = downsample(input_resolution, dim=dim, norm_layer=norm_layer) if downsample is not None else None

    def forward(self, x):
        for blk in self.blocks:
            x = checkpoint.checkpoint(blk, x, use_reentrant=False) if self.use_checkpoint else blk(x)
        if self.downsample is not None:
            x = self.downsample(x)
        return x

    def extra_repr(self) -> str:
        return f"dim={self.dim}, input_resolution={self.input_resolution}, depth={self.depth}"

    def flops(self):
        f = sum(blk.flops() for blk in self.blocks)
        return f + (self.downsample.flops() if self.downsample is not None else 0)

    def _init_respostnorm(self):
        for blk in self.blocks:
            for norm in (blk.norm1, blk.norm2):
                nn.init.constant_(norm.bias, 0)
                nn.init.constant_(norm.weight, 0)


class PatchEmbed(nn.Module):
    """Strided-conv patch embedding (swin_v2_module.py:454-499): (B,C,H,W) -> (B, Ph*Pw, E)."""

    def __init__(self, img_size_w=1, img_size_h=84, patch_size=4, in_chans=1, embed_dim=96, norm_layer=None):
        super().__init__()
        patch_size = to_2tuple(patch_size)
        if img_size_w // patch_size[1] == 0:
            patches_resolution = [img_size_h // patch_size[0], img_size_w]
        else:
            patches_resolution = [img_size_h // patch_size[0], img_size_w // patch_size[1]]
        self.img_size_h = img_size_h
        self.img_size_w = img_size_w
        self.patch_size = patch_size
        self.patches_resolution = patches_resolution
        self.num_patches = patches_resolution[0] * patches_resolution[1]
        self.in_chans = in_chans
        self.embed_dim = embed_dim
        self.proj = nn.Conv2d(in_chans, embed_dim, kernel_size=patch_size, stride=patch_size)
        self.norm = norm_layer(embed_dim) if norm_layer is not None else None

    def forward(self, x):
        B, C, H, W = x.shape
        assert H == self.img_size_h and W == self.img_size_w, \
            f"Input image size ({H}*{W}) doesn't match model ({self.img_size_h}*{self.img_size_w})."
        x = self.proj(x).flatten(2).transpose(1, 2)
        return fused.layer_norm(x, self.norm, out_dtype=torch.float32) if self.norm is not None else x

    def flops(self):
        Ho, Wo = self.patches_resolution
        f = Ho * Wo * self.embed_dim * self.in_chans * (self.patch_size[0] * self.patch_size[1])
        return f + (Ho * Wo * self.embed_dim if self.norm is not None else 0)


class PatchEmbed3D(nn.Module):
    """3-D counterpart used by the volumetric configurations (our extension, SURVEY.md F1):
    (B, C, D, H, W) -> (B, Pd*Ph*Pw, E) with a strided Conv3d."""

    def __init__(self, img_size=96, patch_size=4, in_chans=1, embed_dim=96, norm_layer=None):
        super().__init__()
        self.img_size = to_ntuple(img_size, 3)
        self.patch_size = to_ntuple(patch_size, 3)
        self.patches_resolution = [s // p for s, p in zip(self.img_size, self.patch_size)]
        self.num_patches = math.prod(self.patches_resolution)
        self.in_chans, self.embed_dim = in_chans, embed_dim
        self.proj = nn.Conv3d(in_chans, embed_dim, kernel_size=self.patch_size, stride=self.patch_size)
        self.norm = norm_layer(embed_dim) if norm_layer is not None else None

    def forward(self, x):
        assert tuple(x.shape[2:]) == self.img_size, f"Input volume {tuple(x.shape[2:])} doesn't match {self.img_size}"
        x = self._embed(x)
        return fused.layer_norm(x, self.norm, out_dtype=torch.float32) if self.norm is not None else x

    def _embed(self, x):
        """The strided convolution as what it is -- a projection of non-overlapping patches: one gather of the patches
        into rows (cast to the compute dtype on the way), then the tensor-core projection kernel with the conv weight
        viewed as (E, C p^3).  cuDNN runs the same convolution as layout conversions + an implicit GEMM, four times the
        GPU time at the cfg3 / cfg5 sizes (tools/profile_step.py)."""
        B, C = x.shape[:2]
        p, g = self.patch_size, self.patches_resolution
        K = C * p[0] * p[1] * p[2]
        dt = torch.get_autocast_dtype("cuda") if torch.is_autocast_enabled("cuda") else x.dtype
        dt = torch.bfloat16 if dt == torch.float16 else dt
        if not (x.is_cuda and dt == torch.bfloat16 and K % 32 == 0 and self.embed_dim % 32 == 0):
            return self.proj(x).flatten(2).transpose(1, 2)
        rows = torch.empty(B, g[0], g[1], g[2], C, p[0], p[1], p[2], device=x.device, dtype=dt)
        rows.copy_(x.view(B, C, g[0], p[0], g[1], p[1], g[2], p[2]).permute(0, 2, 4, 6, 1, 3, 5, 7))
        with torch.autocast("cuda", enabled=False):
            y = ops.linear(rows.view(-1, K), self.proj.weight.view(self.embed_dim, K), self.proj.bias)
        return y.view(B, self.num_patches, self.embed_dim)
