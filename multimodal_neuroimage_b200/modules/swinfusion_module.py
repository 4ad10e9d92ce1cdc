"""Drop-in replacements for the classes of the reference's modules/swinfusion_module.py:
Swin-V1-style window attention (q * head_dim^-0.5, learned relative_position_bias_table)
in self- and cross-modal form, the pre-norm blocks around them and the RSTB / CRSTB
residual groups -- backed by the fused CUDA window-attention op, n-D windows.

Same class names, constructor arguments, forward signatures and state_dict keys as the
reference (SURVEY.md 8b).  The blocks hand un-windowed tensors to the kernel; the shift
mask is generated in-kernel from `x_size`, so the reference's per-call CPU mask rebuild +
H2D copy when `x_size != input_resolution` (swinfusion_module.py:360-363,511-516) is gone.
"""
from __future__ import annotations

import math

import torch
import torch.nn as nn
import torch.nn.functional as F  # noqa: F401  (star-exported like the reference's)
import torch.utils.checkpoint as checkpoint
from torch.nn.init import trunc_normal_  # noqa: F401  (model.py:1229,1374 call it through the star import)

from .. import _lib, fused, geometry, ops
from .swin_v2_module import DropPath, _GatherRows, to_2tuple, to_ntuple, window_partition, window_reverse

window_partition_fusion = window_partition


def window_reverse_fusion(windows, window_size, *grid):
    return window_reverse(windows, window_size, *grid)


class Mlp_fusion(nn.Module):
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
            return fused.mlp(x, self.fc1, self.fc2, "gelu", self.drop.p, self.training)      # swinfusion_module.py:25-29
        return self.drop(self.fc2(self.drop(self.act(self.fc1(x)))))


class _TableBiasAttention(nn.Module):
    """Shared pieces of the two scaled-dot window attentions: the learned bias table, its
    index buffer, dropout bookkeeping and the call into the kernel."""

    def _init_common(self, dim, window_size, num_heads, qk_scale, attn_drop, proj_drop):
        self.dim = dim
        self.window_size = tuple(int(w) for w in window_size)
        self.num_heads = num_heads
        head_dim = dim // num_heads
        self.scale = qk_scale or head_dim ** -0.5
        entries = math.prod(2 * w - 1 for w in self.window_size)
        self.relative_position_bias_table = nn.Parameter(torch.zeros(entries, num_heads))
        self.register_buffer("relative_position_index", geometry.relative_position_index(self.window_size))
        self.kernel_path = _lib.PATH_AUTO

    def position_bias(self) -> torch.Tensor:
        """(nH, N, N) fp32 = table[index] (swinfusion_module.py:127-130)."""
        N = math.prod(self.window_size)
        table, index = self.relative_position_bias_table, self.relative_position_index.view(-1)
        if table.is_cuda and table.dtype == torch.float32 and table.is_contiguous() and index.is_contiguous():
            # libmmn_b200 cpb_bias.cu: gather + head-major layout in one launch, scatter-add backward in one
            return torch.ops.mmn_b200.table_bias_fwd(table, index).view(-1, N, N)
        b = _GatherRows.apply(table.float(), index)
        return b.view(N, N, -1).permute(2, 0, 1).contiguous()

    def _core(self, a, b, grid, window, shift, mask_kind, mask):
        p, seed, off, rng = ops.next_dropout_stream(self.attn_drop.p, self.training, a.device)
        out, _ = torch.ops.mmn_b200.winattn_fwd(ops.kernel_io(a), ops.kernel_io(b), self.position_bias(), None, mask,
                                                list(grid), list(window), list(shift), self.num_heads, _lib.SCORE_SCALED,
                                                mask_kind, float(self.scale), p, seed, off, self.kernel_path, rng)
        return out.to(a.dtype)

    @staticmethod
    def _mask_args(mask, device):
        if mask is None:
            return _lib.MASK_NONE, None
        return _lib.MASK_TENSOR, mask.to(device=device, dtype=torch.float32).contiguous()

    def extra_repr(self) -> str:
        return f"dim={self.dim}, window_size={self.window_size}, num_heads={self.num_heads}"

    def flops(self, N):
        d = self.dim // self.num_heads
        return N * self.dim * 3 * self.dim + 2 * self.num_heads * N * d * N + N * self.dim * self.dim


class WindowAttention_fusion(_TableBiasAttention):
    """Self window attention (swinfusion_module.py:65-161)."""

    def __init__(self, dim, window_size, num_heads, qkv_bias=True, qk_scale=None, attn_drop=0., proj_drop=0.):
        super().__init__()
        self._init_common(dim, window_size, num_heads, qk_scale, attn_drop, proj_drop)
        self.qkv = nn.Linear(dim, dim * 3, bias=qkv_bias)
        self.attn_drop = nn.Dropout(attn_drop)
        self.proj = nn.Linear(dim, dim)
        self.proj_drop = nn.Dropout(proj_drop)
        nn.init.trunc_normal_(self.relative_position_bias_table, std=.02)
        self.softmax = nn.Softmax(dim=-1)

    def forward(self, x, mask=None):
        B_, N, C = x.shape
        kind, mask = self._mask_args(mask, x.device)
        out = self._core(self.qkv(x), None, (N,), (N,), (0,), kind, mask)
        return self.proj_drop(self.proj(out))

    def forward_grid(self, x, grid, shift):
        shifted = any(int(s) > 0 for s in shift)
        y = fused.window_attention_module(x, None, self.qkv.weight, self.qkv.bias, None, None, self.proj.weight,
                                          self.proj.bias, self.position_bias(), None, grid, self.window_size, shift,
                                          self.num_heads, _lib.SCORE_SCALED, _lib.MASK_SHIFT if shifted else _lib.MASK_NONE,
                                          float(self.scale), ops.next_dropout_stream(self.attn_drop.p, self.training, x.device),
                                          self.kernel_path)
        return self.proj_drop(y)


class Cross_WindowAttention(_TableBiasAttention):
    """Cross-modal window attention: queries from x, keys/values from y
    (swinfusion_module.py:163-262)."""

    def __init__(self, dim, window_size, num_heads, qkv_bias=True, qk_scale=None, attn_drop=0., proj_drop=0.):
        super().__init__()
        self._init_common(dim, window_size, num_heads, qk_scale, attn_drop, proj_drop)
        self.q = nn.Linear(dim, dim, bias=qkv_bias)
        self.kv = nn.Linear(dim, dim * 2, bias=qkv_bias)
        self.attn_drop = nn.Dropout(attn_drop)
        self.proj = nn.Linear(dim, dim)
        self.proj_drop = nn.Dropout(proj_drop)
        nn.init.trunc_normal_(self.relative_position_bias_table, std=.02)
        self.softmax = nn.Softmax(dim=-1)

    def forward(self, x, y, mask=None):
        B_, N, C = x.shape
        kind, mask = self._mask_args(mask, x.device)
        out = self._core(self.q(x), self.kv(y), (N,), (N,), (0,), kind, mask)
        return self.proj_drop(self.proj(out))

    def forward_grid(self, x, y, grid, shift):
        shifted = any(int(s) > 0 for s in shift)
        out = fused.window_attention_module(x, y, self.q.weight, self.q.bias, self.kv.weight, self.kv.bias, self.proj.weight,
                                            self.proj.bias, self.position_bias(), None, grid, self.window_size, shift,
                                            self.num_heads, _lib.SCORE_SCALED,
                                            _lib.MASK_SHIFT if shifted else _lib.MASK_NONE, float(self.scale),
                                            ops.next_dropout_stream(self.attn_drop.p, self.training, x.device),
                                            self.kernel_path)
        return self.proj_drop(out)


class _FusionBlockBase(nn.Module):
    def _init_geometry(self, dim, input_resolution, num_heads, window_size, shift_size, mlp_ratio):
        self.dim = dim
        self.input_resolution = tuple(int(r) for r in input_resolution)
        self.num_heads = num_heads
        self.mlp_ratio = mlp_ratio
        self.window_size, self.shift_size = geometry.clamp_window(self.input_resolution, window_size, shift_size)
        assert 0 <= self.shift_size < self.window_size, "shift_size must in 0-window_size"

    def calculate_mask(self, x_size):
        """(nW, N, N) {0,-100} mask of the shifted frame for an arbitrary x_size
        (swinfusion_module.py:317-338).  API compatibility; the kernel does not read it."""
        n = len(x_size)
        return geometry.shift_attention_mask(tuple(x_size), to_ntuple(self.window_size, n), to_ntuple(self.shift_size, n))

    def _register_mask(self):
        mask = self.calculate_mask(self.input_resolution) if self.shift_size > 0 else None
        self.register_buffer("attn_mask", mask)

    def extra_repr(self) -> str:
        return (f"dim={self.dim}, input_resolution={self.input_resolution}, num_heads={self.num_heads}, "
                f"window_size={self.window_size}, shift_size={self.shift_size}, mlp_ratio={self.mlp_ratio}")

    def _flops(self, attn):
        L = math.prod(self.input_resolution)
        N = self.window_size ** len(self.input_resolution)
        return 2 * self.dim * L + (L / N) * attn.flops(N) + 2 * L * self.dim * self.dim * self.mlp_ratio


class SwinTransformerBlock_fusion(_FusionBlockBase):
    """Pre-norm self block; forward(x, x_size) (swinfusion_module.py:265-398)."""

    def __init__(self, dim, input_resolution, num_heads, window_size=7, shift_size=0, mlp_ratio=4., qkv_bias=True,
                 qk_scale=None, drop=0., attn_drop=0., drop_path=0., act_layer=nn.GELU, norm_layer=nn.LayerNorm):
        super().__init__()
        self._init_geometry(dim, input_resolution, num_heads, window_size, shift_size, mlp_ratio)
        n = len(self.input_resolution)
        self.norm1 = norm_layer(dim)
        self.attn = WindowAttention_fusion(dim, window_size=to_ntuple(self.window_size, n), num_heads=num_heads,
                                           qkv_bias=qkv_bias, qk_scale=qk_scale, attn_drop=attn_drop, proj_drop=drop)
        self.drop_path = DropPath(drop_path) if drop_path > 0. else nn.Identity()
        self.norm2 = norm_layer(dim)
        self.mlp = Mlp_fusion(in_features=dim, hidden_features=int(dim * mlp_ratio), act_layer=act_layer, drop=drop)
        self._register_mask()

    def forward_deferred(self, x, delta, x_size):
        """The block on the stream `x + delta` (delta None: just x), returning (x', delta') with the block's output
        = x' + delta'.  The residual add that closes a block is left to the LayerNorm kernel that opens the next one
        (BasicLayer_fusion chains blocks this way), so a block is two add+LayerNorm passes and no separate add -- forward
        and backward (each intermediate stream feeds exactly one kernel: autograd has nothing to accumulate)."""
        n = len(x_size)
        if delta is None:
            h = fused.layer_norm(x, self.norm1)
        else:
            x, h = fused.add_layer_norm(x, delta, self.norm1)
        a = self.attn.forward_grid(h, tuple(x_size), to_ntuple(self.shift_size, n))
        x, h = fused.add_layer_norm(x, self.drop_path(a), self.norm2)          # x + a and norm2 of it in one pass
        return x, self.drop_path(self.mlp(h))

    def forward(self, x, x_size):
        x, d = self.forward_deferred(x, None, x_size)
        return x + d

    def flops(self):
        return self._flops(self.attn)


class Cross_SwinTransformerBlock(_FusionBlockBase):
    """Pre-norm cross-modal block; forward(x, y, x_size) -> (x, y): stream A attends to B
    and B to A with separate weights (swinfusion_module.py:400-558)."""

    def __init__(self, dim, input_resolution, num_heads, window_size=7, shift_size=0, mlp_ratio=4., qkv_bias=True,
                 qk_scale=None, drop=0., attn_drop=0., drop_path=0., act_layer=nn.GELU, norm_layer=nn.LayerNorm):
        super().__init__()
        self._init_geometry(dim, input_resolution, num_heads, window_size, shift_size, mlp_ratio)
        n = len(self.input_resolution)
        self.norm1_A = norm_layer(dim)
        self.norm1_B = norm_layer(dim)
        kw = dict(window_size=to_ntuple(self.window_size, n), num_heads=num_heads, qkv_bias=qkv_bias, qk_scale=qk_scale,
                  attn_drop=attn_drop, proj_drop=drop)
        self.attn_A = Cross_WindowAttention(dim, **kw)
        self.attn_B = Cross_WindowAttention(dim, **kw)
        self.drop_path_A = DropPath(drop_path) if drop_path > 0. else nn.Identity()
        self.drop_path_B = DropPath(drop_path) if drop_path > 0. else nn.Identity()
        self.norm2_A = norm_layer(dim)
        self.norm2_B = norm_layer(dim)
        hidden = int(dim * mlp_ratio)
        self.mlp_A = Mlp_fusion(in_features=dim, hidden_features=hidden, act_layer=act_layer, drop=drop)
        self.mlp_B = Mlp_fusion(in_features=dim, hidden_features=hidden, act_layer=act_layer, drop=drop)
        self._register_mask()

    def forward_deferred(self, x, dx, y, dy, x_size):
        """As SwinTransformerBlock_fusion.forward_deferred, for the two streams x + dx and y + dy."""
        n = len(x_size)
        grid, shift = tuple(x_size), to_ntuple(self.shift_size, n)

        def open_stream(t, dt, ln):                       # the stream's pending add + norm1
            return (t, fused.layer_norm(t, ln)) if dt is None else fused.add_layer_norm(t, dt, ln)

        def side(t, tn, on, attn, drop_path, norm2, mlp):  # one modality: attends to the other's normalised stream
            a = attn.forward_grid(tn, on, grid, shift)
            t, h = fused.add_layer_norm(t, drop_path(a), norm2)
            return t, drop_path(mlp(h))

        # the two modalities only meet in the attention calls (each reads both normalised streams): everything else of the
        # two sides is independent, so fused.parallel may run them on two streams
        (x, xn), (y, yn) = fused.parallel(lambda: open_stream(x, dx, self.norm1_A), lambda: open_stream(y, dy, self.norm1_B), x, (y, dy))
        (x, dxo), (y, dyo) = fused.parallel(lambda: side(x, xn, yn, self.attn_A, self.drop_path_A, self.norm2_A, self.mlp_A),
                                            lambda: side(y, yn, xn, self.attn_B, self.drop_path_B, self.norm2_B, self.mlp_B),
                                            x, (y, yn, xn))
        return x, dxo, y, dyo

    def forward(self, x, y, x_size):
        x, dx, y, dy = self.forward_deferred(x, None, y, None, x_size)
        return x + dx, y + dy

    def flops(self):
        return self._flops(self.attn_A)


class PatchMerging_fusion(nn.Module):
    """norm(2^n C) then Linear(2^n C -> 2C) (swinfusion_module.py:560-605: note the norm is
    BEFORE the reduction here, unlike SwinV2's PatchMerging)."""

    def __init__(self, input_resolution, dim, norm_layer=nn.LayerNorm):
        super().__init__()
        self.input_resolution = tuple(int(r) for r in input_resolution)
        self.dim = dim
        n = len(self.input_resolution)
        self.reduction = nn.Linear((2 ** n) * dim, 2 * dim, bias=False)
        self.norm = norm_layer((2 ** n) * dim)

    def forward(self, x):
        B, L, C = x.shape
        res = self.input_resolution
        n = len(res)
        assert L == math.prod(res), "input feature has wrong size"
        assert all(r % 2 == 0 for r in res), f"x size {res} are not even."
        x = x.view(B, *res, C)
        parts = []
        for code in range(2 ** n):
            sl = [slice(None)] + [slice((code >> a) & 1, None, 2) for a in range(n)] + [slice(None)]
            parts.append(x[tuple(sl)])
        x = torch.cat(parts, -1).view(B, -1, (2 ** n) * C)
        return self.reduction(self.norm(x))

    def extra_repr(self) -> str:
        return f"input_resolution={self.input_resolution}, dim={self.dim}"

    def flops(self):
        L = math.prod(self.input_resolution)
        n = len(self.input_resolution)
        return L * self.dim + (L // 2 ** n) * (2 ** n) * self.dim * 2 * self.dim


class BasicLayer_fusion(nn.Module):
    """`depth` self blocks alternating shift 0 / window//2 (swinfusion_module.py:609-676)."""

    def __init__(self, dim, input_resolution, depth, num_heads, window_size, mlp_ratio=4., qkv_bias=True, qk_scale=None,
                 drop=0., attn_drop=0., drop_path=0., norm_layer=nn.LayerNorm, downsample=None, use_checkpoint=False):
        super().__init__()
        self.dim = dim
        self.input_resolution = input_resolution
        self.depth = depth
        self.use_checkpoint = use_checkpoint
        self.blocks = nn.ModuleList([
            SwinTransformerBlock_fusion(dim=dim, input_resolution=input_resolution, num_heads=num_heads,
                                        window_size=window_size, shift_size=0 if (i % 2 == 0) else window_size // 2,
                                        mlp_ratio=mlp_ratio, qkv_bias=qkv_bias, qk_scale=qk_scale, drop=drop,
                                        attn_drop=attn_drop,
                                        drop_path=drop_path[i] if isinstance(drop_path, list) else drop_path,
                                        norm_layer=norm_layer)
            for i in range(depth)])
        self.downsample = downsample(input_resolution, dim=dim, norm_layer=norm_layer) if downsample is not None else None

    def forward(self, x, x_size):
        if self.use_checkpoint:
            for blk in self.blocks:
                x = checkpoint.checkpoint(blk, x, x_size, use_reentrant=False)
        else:
            delta = None                      # the stream is x + delta: each block's closing add rides on the next LayerNorm
            for blk in self.blocks:
                x, delta = blk.forward_deferred(x, delta, x_size)
            if delta is not None:
                x = x + delta
        if self.downsample is not None:
            x = self.downsample(x)
        return x

    def extra_repr(self) -> str:
        return f"dim={self.dim}, input_resolution={self.input_resolution}, depth={self.depth}"

    def flops(self):
        f = sum(blk.flops() for blk in self.blocks)
        return f + (self.downsample.flops() if self.downsample is not None else 0)


class Cross_BasicLayer(nn.Module):
    """`depth` cross-modal blocks (swinfusion_module.py:678-747)."""

    def __init__(self, dim, input_resolution, depth, num_heads, window_size, mlp_ratio=4., qkv_bias=True, qk_scale=None,
                 drop=0., attn_drop=0., drop_path=0., norm_layer=nn.LayerNorm, downsample=None, use_checkpoint=False):
        super().__init__()
        self.dim = dim
        self.input_resolution = input_resolution
        self.depth = depth
        self.use_checkpoint = use_checkpoint
        self.blocks = nn.ModuleList([
            Cross_SwinTransformerBlock(dim=dim, input_resolution=input_resolution, num_heads=num_heads,
                                       window_size=window_size, shift_size=0 if (i % 2 == 0) else window_size // 2,
                                       mlp_ratio=mlp_ratio, qkv_bias=qkv_bias, qk_scale=qk_scale, drop=drop,
                                       attn_drop=attn_drop,
                                       drop_path=drop_path[i] if isinstance(drop_path, list) else drop_path,
                                       norm_layer=norm_layer)
            for i in range(depth)])
        self.downsample = downsample(input_resolution, dim=dim, norm_layer=norm_layer) if downsample is not None else None

    def forward(self, x, y, x_size):
        if self.use_checkpoint:
            for blk in self.blocks:
                x, y = checkpoint.checkpoint(blk, x, y, x_size, use_reentrant=False)
        else:
            dx = dy = None
            for blk in self.blocks:
                x, dx, y, dy = blk.forward_deferred(x, dx, y, dy, x_size)
            if dx is not None:
                x, y = x + dx, y + dy
        if self.downsample is not None:
            x = self.downsample(x)
            y = self.downsample(y)
        return x, y

    def extra_repr(self) -> str:
        return f"dim={self.dim}, input_resolution={self.input_resolution}, depth={self.depth}"

    def flops(self):
        f = sum(blk.flops() for blk in self.blocks)
        return f + (self.downsample.flops() if self.downsample is not None else 0)


def _resi_conv(dim, resi_connection, n):
    """The convolution the reference declares in RSTB/CRSTB but never calls in forward
    (swinfusion_module.py:813,924-925 are commented out); kept so state_dicts match."""
    conv = nn.Conv2d if n == 2 else nn.Conv3d
    if resi_connection == '1conv':
        return conv(dim, dim, 3, 1, 1)
    if resi_connection == '3conv':
        return nn.Sequential(conv(dim, dim // 4, 3, 1, 1), nn.LeakyReLU(negative_slope=0.2, inplace=True),
                             conv(dim // 4, dim // 4, 1, 1, 0), nn.LeakyReLU(negative_slope=0.2, inplace=True),
                             conv(dim // 4, dim, 3, 1, 1))
    raise ValueError(f"unknown resi_connection {resi_connection!r}")


class RSTB(nn.Module):
    """Residual Swin Transformer Block: residual_group(x) + x (swinfusion_module.py:750-824)."""

    def __init__(self, dim, input_resolution, depth, num_heads, window_size, mlp_ratio=4., qkv_bias=True, qk_scale=None,
                 drop=0., attn_drop=0., drop_path=0., norm_layer=nn.LayerNorm, downsample=None, use_checkpoint=False,
                 img_size=224, patch_size=4, resi_connection='1conv'):
        super().__init__()
        self.dim = dim
        self.input_resolution = input_resolution
        self.residual_group = BasicLayer_fusion(dim=dim, input_resolution=input_resolution, depth=depth,
                                                num_heads=num_heads, window_size=window_size, mlp_ratio=mlp_ratio,
                                                qkv_bias=qkv_bias, qk_scale=qk_scale, drop=drop, attn_drop=attn_drop,
                                                drop_path=drop_path, norm_layer=norm_layer, downsample=downsample,
                                                use_checkpoint=use_checkpoint)
        self.conv = _resi_conv(dim, resi_connection, len(input_resolution))
        self.patch_embed = PatchEmbed_fusion(img_size=img_size, patch_size=patch_size, in_chans=0, embed_dim=dim,
                                             norm_layer=None)
        self.patch_unembed = PatchUnEmbed(img_size=img_size, patch_size=patch_size, in_chans=0, embed_dim=dim,
                                          norm_layer=None)

    def forward(self, x, x_size):
        return self.residual_group(x, x_size) + x

    def flops(self):
        L = math.prod(self.input_resolution)
        return self.residual_group.flops() + L * self.dim * self.dim * 9 + self.patch_embed.flops()


class CRSTB(nn.Module):
    """Intra-modal groups A and B, then the cross-modal group, each with a residual
    (swinfusion_module.py:826-939)."""

    def __init__(self, dim, input_resolution, depth, num_heads, window_size, mlp_ratio=4., qkv_bias=True, qk_scale=None,
                 drop=0., attn_drop=0., drop_path=0., norm_layer=nn.LayerNorm, downsample=None, use_checkpoint=False,
                 img_size=224, patch_size=4, resi_connection='1conv'):
        super().__init__()
        self.dim = dim
        self.input_resolution = input_resolution
        kw = dict(dim=dim, input_resolution=input_resolution, depth=depth, num_heads=num_heads, window_size=window_size,
                  mlp_ratio=mlp_ratio, qkv_bias=qkv_bias, qk_scale=qk_scale, drop=drop, attn_drop=attn_drop,
                  drop_path=drop_path, norm_layer=norm_layer, downsample=downsample, use_checkpoint=use_checkpoint)
        self.residual_group = Cross_BasicLayer(**kw)
        self.residual_group_A = BasicLayer_fusion(**kw)
        self.residual_group_B = BasicLayer_fusion(**kw)
        n = len(input_resolution)
        self.conv_A = _resi_conv(dim, resi_connection, n)
        self.conv_B = _resi_conv(dim, resi_connection, n)
        self.patch_embed = PatchEmbed_fusion(img_size=img_size, patch_size=patch_size, in_chans=0, embed_dim=dim,
                                             norm_layer=None)
        self.patch_unembed = PatchUnEmbed(img_size=img_size, patch_size=patch_size, in_chans=0, embed_dim=dim,
                                          norm_layer=None)

    def forward(self, x, y, x_size):
        # the two intra-modal groups are independent: fused.parallel may run them on two streams
        x, y = fused.parallel(lambda: self.residual_group_A(x, x_size) + x, lambda: self.residual_group_B(y, x_size) + y, x, (y,))
        x1, y1 = x, y
        x, y = self.residual_group(x1, y1, x_size)
        return x + x1, y + y1

    def flops(self):
        L = math.prod(self.input_resolution)
        return (self.residual_group_A.flops() + self.residual_group_B.flops() + L * self.dim * self.dim * 9
                + self.patch_embed.flops())


class PatchEmbed_fusion(nn.Module):
    """(B, C, *spatial) -> (B, L, C), optional norm (swinfusion_module.py:941-981)."""

    def __init__(self, img_size=224, patch_size=4, in_chans=3, embed_dim=96, norm_layer=None):
        super().__init__()
        img_size = to_2tuple(img_size) if not isinstance(img_size, (list, tuple)) else tuple(img_size)
        patch_size = to_ntuple(patch_size, len(img_size))
        self.img_size = img_size
        self.patch_size = patch_size
        self.patches_resolution = [i // p for i, p in zip(img_size, patch_size)]
        self.num_patches = math.prod(self.patches_resolution)
        self.in_chans = in_chans
        self.embed_dim = embed_dim
        self.norm = norm_layer(embed_dim) if norm_layer is not None else None

    def forward(self, x):
        x = x.flatten(2).transpose(1, 2)
        return self.norm(x) if self.norm is not None else x

    def flops(self):
        return math.prod(self.img_size) * self.embed_dim if self.norm is not None else 0


class PatchUnEmbed(nn.Module):
    """(B, L, C) -> (B, C, *x_size) (swinfusion_module.py:984-1015)."""

    def __init__(self, img_size=224, patch_size=4, in_chans=3, embed_dim=96, norm_layer=None):
        super().__init__()
        img_size = to_2tuple(img_size) if not isinstance(img_size, (list, tuple)) else tuple(img_size)
        patch_size = to_ntuple(patch_size, len(img_size))
        self.img_size = img_size
        self.patch_size = patch_size
        self.patches_resolution = [i // p for i, p in zip(img_size, patch_size)]
        self.num_patches = math.prod(self.patches_resolution)
        self.in_chans = in_chans
        self.embed_dim = embed_dim

    def forward(self, x, x_size):
        B, L, C = x.shape
        return x.transpose(1, 2).reshape(B, self.embed_dim, *x_size)

    def flops(self):
        return 0


class Upsample(nn.Sequential):
    """Conv + PixelShuffle upsampler (swinfusion_module.py:1018-1040; `model.SwinFusion` builds it for
    `upsampler='pixelshuffle'`, model.py:1348).  scale = 2^k: k x (Conv2d(f, 4f, 3) + PixelShuffle(2)); scale = 3: one
    Conv2d(f, 9f, 3) + PixelShuffle(3)."""

    def __init__(self, scale, num_feat):
        layers = []
        if scale >= 1 and scale & (scale - 1) == 0:
            for _ in range(scale.bit_length() - 1):
                layers += [nn.Conv2d(num_feat, 4 * num_feat, 3, 1, 1), nn.PixelShuffle(2)]
        elif scale == 3:
            layers += [nn.Conv2d(num_feat, 9 * num_feat, 3, 1, 1), nn.PixelShuffle(3)]
        else:
            raise ValueError(f'scale {scale} is not supported. Supported scales: 2^n and 3.')
        super().__init__(*layers)


class UpsampleOneStep(nn.Sequential):
    """One Conv2d(f, scale^2 * out, 3) + PixelShuffle(scale) (swinfusion_module.py:1043-1061; model.py:1352)."""

    def __init__(self, scale, num_feat, num_out_ch, input_resolution=None):
        self.num_feat = num_feat
        self.input_resolution = input_resolution
        super().__init__(nn.Conv2d(num_feat, (scale ** 2) * num_out_ch, 3, 1, 1), nn.PixelShuffle(scale))

    def flops(self):
        H, W = self.input_resolution
        return H * W * self.num_feat * 3 * 9
