"""Generate the golden fixtures in this directory by importing and running the UNMODIFIED
reference modules (read-only) on seeded synthetic inputs.

Run on a CPU with a checkout of the reference:   MMN_REFERENCE=<dir> python tests/golden/make_golden.py
The fixtures (*.npz) are committed, so nothing at test time reads the reference.
Harness-side shims only (SURVEY.md 8c): a `timm` stub on
sys.path and a CPU `Tensor.get_device` patch for swin_v2_module.py:154.  Gotchas honoured:
LayerNorm weights randomised (F10), bias tables scaled up, logit_scale values on both sides
of the ln(100) clamp, k != v tensors for the 3-projection MHA branch, a shifted block whose
windows wrap in every axis, and x_size != input_resolution for the fusion blocks.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.environ.get("MMN_REFERENCE", "")
if not (REF and os.path.isdir(os.path.join(REF, "modules"))):
    sys.exit("set MMN_REFERENCE to a checkout of the reference (the directory holding model.py and modules/)")
sys.path.insert(0, os.path.join(HERE, "_shims"))
sys.path.insert(1, REF)

_orig_get_device = torch.Tensor.get_device
torch.Tensor.get_device = lambda self: (self.device if not self.is_cuda else _orig_get_device(self))

from modules import swin_v2_module as v2            # noqa: E402
from modules import swinfusion_module as fu         # noqa: E402
from modules import crossmodal_transformer as cm    # noqa: E402
from modules import multihead_attention as mha      # noqa: E402
from modules import position_embedding as pe        # noqa: E402


def npy(t):
    return t.detach().cpu().numpy()


def randomise(module, gen):
    """Module default init, then the perturbations SURVEY.md 8c/8d prescribe."""
    with torch.no_grad():
        for name, p in module.named_parameters():
            if "norm" in name and name.endswith("weight"):
                p.copy_(torch.empty_like(p).uniform_(0.5, 1.5, generator=gen))
            elif "norm" in name and name.endswith("bias"):
                p.copy_(torch.empty_like(p).normal_(0, 0.2, generator=gen))
            elif name.endswith("relative_position_bias_table"):
                p.copy_(torch.empty_like(p).normal_(0, 1.0, generator=gen))
            elif name.endswith("logit_scale"):
                p.copy_(torch.empty_like(p).uniform_(0.0, float(np.log(200.0)), generator=gen))
            elif name.endswith("bias") or name.endswith("q_bias") or name.endswith("v_bias"):
                p.copy_(torch.empty_like(p).normal_(0, 0.3, generator=gen))


def record(out, case, module, inputs, outputs, grads_wrt, loss_outs=None):
    """Store state_dict, inputs, outputs and d(sum(outputs * cot))/d(inputs, params)."""
    for k, v in module.state_dict().items():
        out[f"{case}/sd/{k}"] = npy(v)
    for k, v in inputs.items():
        out[f"{case}/in/{k}"] = npy(v)
    outs = outputs if isinstance(outputs, (tuple, list)) else (outputs,)
    gen = torch.Generator().manual_seed(1234)
    loss = 0
    for i, o in enumerate(outs):
        cot = torch.randn(o.shape, generator=gen, dtype=o.dtype)
        out[f"{case}/out/{i}"] = npy(o)
        out[f"{case}/cot/{i}"] = npy(cot)
        if loss_outs is None or i in loss_outs:
            loss = loss + (o * cot).sum()
    out[f"{case}/loss_outs"] = np.array(list(range(len(outs))) if loss_outs is None else list(loss_outs), np.int64)
    module.zero_grad()
    loss.backward()
    for k, v in grads_wrt.items():
        out[f"{case}/gin/{k}"] = npy(v.grad)
    for k, p in module.named_parameters():
        if p.grad is not None:
            out[f"{case}/gsd/{k}"] = npy(p.grad)


def index_maps():
    out = {}
    # a1/a2/a3: composite gather map = partition(roll(arange)) for several geometries
    for (H, W, ws, s) in [(12, 12, 6, 3), (12, 12, 6, 0), (8, 16, 4, 2), (6, 6, 3, 1), (16, 8, 8, 4)]:
        ids = torch.arange(H * W, dtype=torch.float32).view(1, H, W, 1)
        rolled = torch.roll(ids, shifts=(-s, -s), dims=(1, 2)) if s > 0 else ids
        win = v2.window_partition(rolled, ws)
        out[f"gather/{H}x{W}_w{ws}_s{s}"] = npy(win.view(-1, ws * ws)).astype(np.int64)
        back = v2.window_reverse(win, ws, H, W)
        back = torch.roll(back, shifts=(s, s), dims=(1, 2)) if s > 0 else back
        assert torch.equal(back, ids)
        winf = fu.window_partition_fusion(rolled, ws)
        assert torch.equal(win, winf)
    # a4: masks from the block constructors (SwinV2 and both fusion blocks)
    for (H, W, ws, s) in [(12, 12, 6, 3), (8, 16, 4, 2), (6, 6, 3, 1), (16, 8, 8, 4), (4, 4, 6, 3)]:
        blk = v2.SwinTransformerBlock(12, (H, W), 3, window_size=ws, shift_size=s)
        key = f"{H}x{W}_w{ws}_s{s}"
        out[f"mask_v2/{key}"] = npy(blk.attn_mask) if blk.attn_mask is not None else np.zeros((0,), np.float32)
        out[f"mask_v2_eff/{key}"] = np.array([blk.window_size, blk.shift_size], np.int64)
        fb = fu.SwinTransformerBlock_fusion(12, (H, W), 3, window_size=ws, shift_size=s)
        out[f"mask_fusion/{key}"] = npy(fb.attn_mask) if fb.attn_mask is not None else np.zeros((0,), np.float32)
        cb = fu.Cross_SwinTransformerBlock(12, (H, W), 3, window_size=ws, shift_size=s)
        out[f"mask_cross/{key}"] = npy(cb.attn_mask) if cb.attn_mask is not None else np.zeros((0,), np.float32)
    fb = fu.SwinTransformerBlock_fusion(12, (12, 12), 3, window_size=6, shift_size=3)
    out["mask_fusion_xsize/18x24_w6_s3"] = npy(fb.calculate_mask((18, 24)))
    # a5: relative position index / coords table
    for ws in [(3, 3), (6, 6), (4, 8), (8, 8)]:
        wa = v2.WindowAttention(12, ws, 3)
        out[f"rpi/{ws[0]}x{ws[1]}"] = npy(wa.relative_position_index)
        out[f"coords/{ws[0]}x{ws[1]}"] = npy(wa.relative_coords_table)
        wf = fu.WindowAttention_fusion(12, ws, 3)
        assert torch.equal(wf.relative_position_index, wa.relative_position_index)
    wa = v2.WindowAttention(12, (6, 6), 3, pretrained_window_size=[4, 4])
    out["coords_pretrained4/6x6"] = npy(wa.relative_coords_table)
    # a14: future masks
    for (T, S) in [(5, 5), (4, 2), (2, 4), (7, 9), (368, 368)]:
        m = cm.buffered_future_mask(torch.zeros(T, 1, 1), torch.zeros(S, 1, 1))
        out[f"future/{T}x{S}"] = np.isinf(npy(m)).astype(np.uint8)
        assert ((npy(m) == 0) | np.isneginf(npy(m))).all()
    # a16: positions + table
    gen = torch.Generator().manual_seed(7)
    tok = torch.randn(3, 11, generator=gen)
    tok[0, 2] = 0.0
    tok[2, 10] = 0.0
    out["pos/tokens"] = npy(tok)
    out["pos/positions"] = npy(pe.make_positions(tok, 0, 0))
    for dim in (28, 7):
        emb = pe.SinusoidalPositionalEmbedding(dim)
        out[f"pos/emb{dim}"] = npy(emb(tok))
    return out


def swinv2():
    out = {}
    gen = torch.Generator().manual_seed(0)
    # WindowAttention alone: reference-default-like (C=12, 3 heads, d=4, ws 6) with a random {0,-100} mask
    for case, (C, nH, ws, nW, B) in {"wa_c12": (12, 3, (6, 6), 4, 2), "wa_c96": (96, 3, (8, 8), 2, 1),
                                      "wa_c48_nomask": (48, 12, (3, 3), 1, 3)}.items():
        m = v2.WindowAttention(C, ws, nH)
        randomise(m, gen)
        N = ws[0] * ws[1]
        x = torch.randn(B * nW, N, C, generator=gen, requires_grad=True)
        mask = None
        if "nomask" not in case:
            reg = torch.randint(0, 3, (nW, N), generator=gen).float()
            d = reg.unsqueeze(1) - reg.unsqueeze(2)
            mask = d.masked_fill(d != 0, -100.0).masked_fill(d == 0, 0.0)
        y = m(x, mask)
        ins = {"x": x}
        if mask is not None:
            ins["mask"] = mask
        record(out, case, m, ins, y, {"x": x})
        out[f"{case}/cfg"] = np.array([C, nH, ws[0], ws[1]], np.int64)
    # Blocks: shifted, windows wrap in both axes; and the min(res)<=ws clamp
    for case, (C, nH, res, ws, s, B) in {"blk_shift": (24, 6, (12, 12), 6, 3, 2), "blk_noshift": (12, 3, (8, 16), 4, 0, 1),
                                          "blk_clamp": (48, 12, (3, 3), 6, 3, 2), "blk_rect": (32, 2, (8, 16), 4, 2, 2)}.items():
        m = v2.SwinTransformerBlock(C, res, nH, window_size=ws, shift_size=s)
        randomise(m, gen)
        x = torch.randn(B, res[0] * res[1], C, generator=gen, requires_grad=True)
        y = m(x)
        record(out, case, m, {"x": x}, y, {"x": x})
        out[f"{case}/cfg"] = np.array([C, nH, res[0], res[1], ws, s], np.int64)
    return out


def swinfusion():
    out = {}
    gen = torch.Generator().manual_seed(1)
    for case, (C, nH, ws, nW, B) in {"wa_c12": (12, 6, (6, 6), 4, 2), "wa_c64": (64, 2, (8, 8), 2, 1)}.items():
        N = ws[0] * ws[1]
        reg = torch.randint(0, 3, (nW, N), generator=gen).float()
        d = reg.unsqueeze(1) - reg.unsqueeze(2)
        mask = d.masked_fill(d != 0, -100.0).masked_fill(d == 0, 0.0)
        m = fu.WindowAttention_fusion(C, ws, nH)
        randomise(m, gen)
        x = torch.randn(B * nW, N, C, generator=gen, requires_grad=True)
        record(out, f"self_{case}", m, {"x": x, "mask": mask}, m(x, mask), {"x": x})
        out[f"self_{case}/cfg"] = np.array([C, nH, ws[0], ws[1]], np.int64)
        m = fu.Cross_WindowAttention(C, ws, nH)
        randomise(m, gen)
        x = torch.randn(B * nW, N, C, generator=gen, requires_grad=True)
        y = torch.randn(B * nW, N, C, generator=gen, requires_grad=True)
        record(out, f"cross_{case}", m, {"x": x, "y": y, "mask": mask}, m(x, y, mask), {"x": x, "y": y})
        out[f"cross_{case}/cfg"] = np.array([C, nH, ws[0], ws[1]], np.int64)
    # blocks; x_size == input_resolution and != (mask recompute path, :360-363, :511-516)
    for case, (C, nH, res, xs, ws, s, B) in {"blk_shift": (12, 6, (12, 12), (12, 12), 6, 3, 2),
                                              "blk_xsize": (12, 3, (12, 12), (18, 24), 6, 3, 1),
                                              "blk_noshift": (16, 2, (8, 8), (8, 8), 4, 0, 2)}.items():
        m = fu.SwinTransformerBlock_fusion(C, res, nH, window_size=ws, shift_size=s)
        randomise(m, gen)
        x = torch.randn(B, xs[0] * xs[1], C, generator=gen, requires_grad=True)
        record(out, f"self_{case}", m, {"x": x}, m(x, xs), {"x": x})
        out[f"self_{case}/cfg"] = np.array([C, nH, res[0], res[1], xs[0], xs[1], ws, s], np.int64)
        m = fu.Cross_SwinTransformerBlock(C, res, nH, window_size=ws, shift_size=s)
        randomise(m, gen)
        x = torch.randn(B, xs[0] * xs[1], C, generator=gen, requires_grad=True)
        y = torch.randn(B, xs[0] * xs[1], C, generator=gen, requires_grad=True)
        record(out, f"cross_{case}", m, {"x": x, "y": y}, m(x, y, xs), {"x": x, "y": y})
        out[f"cross_{case}/cfg"] = np.array([C, nH, res[0], res[1], xs[0], xs[1], ws, s], np.int64)
    return out


def crossmodal():
    out = {}
    gen = torch.Generator().manual_seed(2)
    # MultiheadAttention: self (qkv same tensor), cross with k != v, T != S, head_dim 7 and 14
    for case, (E, nH, T, S, B, kind) in {"mha_self_d7": (28, 4, 24, 24, 2, "self"), "mha_cross_d7": (84, 12, 40, 40, 2, "cross"),
                                          "mha_cross_TneS": (56, 4, 9, 13, 3, "cross"), "mha_self_d14_nomask": (56, 4, 16, 16, 1, "self")}.items():
        m = mha.MultiheadAttention(E, nH).eval()
        randomise(m, gen)
        q = torch.randn(T, B, E, generator=gen, requires_grad=True)
        mask = None if "nomask" in case else cm.buffered_future_mask(torch.zeros(T, 1, 1), torch.zeros(S, 1, 1))
        if kind == "self":
            a, w = m(q, q, q, attn_mask=mask)
            ins, gw = {"q": q}, {"q": q}
        else:
            k = torch.randn(S, B, E, generator=gen, requires_grad=True)
            v = torch.randn(S, B, E, generator=gen, requires_grad=True)
            a, w = m(q, k, v, attn_mask=mask)
            ins, gw = {"q": q, "k": k, "v": v}, {"q": q, "k": k, "v": v}
        # the head-averaged weights (output 1) are returned but every caller discards them
        # (crossmodal_transformer.py:148,152): gradients are taken through output 0 only
        record(out, case, m, ins, (a, w), gw, loss_outs=(0,))
        out[f"{case}/cfg"] = np.array([E, nH, T, S, B, int(mask is not None)], np.int64)
    # Encoder: self and cross streams, mask on/off; a zero in channel 0 exercises the padding position
    for case, (E, nH, L, T, B, use_mask, cross) in {"enc_self": (28, 4, 2, 20, 2, True, False), "enc_cross": (84, 12, 2, 16, 2, True, True),
                                                     "enc_cross_nomask": (28, 4, 1, 12, 1, False, True)}.items():
        m = cm.TransformerEncoder(E, nH, L, attn_mask=use_mask).eval()
        randomise(m, gen)
        x = torch.randn(T, B, E, generator=gen)
        x[3, 0, 0] = 0.0
        x.requires_grad_(True)
        if cross:
            xk = torch.randn(T, B, E, generator=gen, requires_grad=True)
            xv = torch.randn(T, B, E, generator=gen, requires_grad=True)
            y = m(x, xk, xv)
            ins, gw = {"x": x, "xk": xk, "xv": xv}, {"x": x, "xk": xk, "xv": xv}
        else:
            y = m(x)
            ins, gw = {"x": x}, {"x": x}
        record(out, case, m, ins, y, gw)
        out[f"{case}/cfg"] = np.array([E, nH, L, T, B, int(use_mask), int(cross)], np.int64)
    return out


if __name__ == "__main__":
    torch.manual_seed(0)
    torch.set_num_threads(1)            # fixed reduction order
    for name, fn in [("index_maps", index_maps), ("swinv2", swinv2), ("swinfusion", swinfusion), ("crossmodal", crossmodal)]:
        data = fn()
        path = os.path.join(HERE, name + ".npz")
        np.savez_compressed(path, **data)
        print(f"{name}: {len(data)} arrays, {os.path.getsize(path) / 1024:.0f} KiB")
