"""Time the fused qkv + window-attention forward (winattn_qkv_fwd) against the two kernels it replaces (linear_fwd for the
qkv projection, then winattn_fwd) at the cfg2 shape: CUDA events around bursts of launches, median of N bursts, tensors
far larger than L2.  Prints the fused kernel's rate on its algorithmic bytes (x in; qkv, o, lse and records out) and that
rate as a share of HBM bandwidth (the 7.7 TB/s data-sheet figure, or --hbm-gbs).
Usage: python tools/time_qkv_fwd.py [--batch 32] [--iters 30] [--burst 10] [--hbm-gbs 7700]"""
import argparse
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from multimodal_neuroimage_b200 import _lib, ops  # noqa: E402,F401

ap = argparse.ArgumentParser()
ap.add_argument("--batch", type=int, default=32)
ap.add_argument("--iters", type=int, default=30)
ap.add_argument("--burst", type=int, default=10)
ap.add_argument("--hbm-gbs", type=float, default=7700.0)
args = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("time_qkv_fwd.py needs a CUDA device")

B = args.batch
grid, nH, d, N = (32, 32, 32), 3, 32, 64
C = nH * d
torch.manual_seed(0)
x = torch.randn(B, *grid, C, device="cuda", dtype=torch.bfloat16)
w = (torch.randn(3 * C, C, device="cuda") * C ** -0.5).bfloat16()
b = torch.randn(3 * C, device="cuda") * 0.3
bias = torch.randn(nH, N, N, device="cuda")
hs = torch.rand(nH, device="cuda") * 10 + 1
geo = (list(grid), [4, 4, 4], [2, 2, 2], nH, _lib.SCORE_COSINE, _lib.MASK_SHIFT, 1.0)
assert ops.winattn_qkv_path_name(tuple(x.shape), x.dtype, *geo[:6]) == "tcgen05-fused"


def fused():
    return torch.ops.mmn_b200.winattn_qkv_fwd(x, w, b, bias, hs, None, *geo, _lib.PATH_AUTO)


def unfused():
    a = torch.ops.mmn_b200.linear_fwd(x.view(-1, C), w, b, _lib.ACT_NONE, False)[0].view(B, *grid, 3 * C)
    return torch.ops.mmn_b200.winattn_fwd(a, None, bias, hs, None, *geo, 0.0, 0, 0, _lib.PATH_AUTO)


def timeit(fn):
    for _ in range(20):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(args.iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.burst):
            fn()
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1) / args.burst)
    ts.sort()
    return ts[len(ts) // 2], ts[0]


windows = B * (32 ** 3 // N)
# per window: x (64 x C bf16) in; qkv (64 x 3C bf16), o (64 x C bf16), lse and records (4 x nH x 64 fp32) out
bytes_fused = windows * (N * C * 2 + N * 3 * C * 2 + N * C * 2 + 4 * nH * N * 4)
res = {}
for name, fn in (("fused", fused), ("unfused", unfused), ("fused", fused), ("unfused", unfused)):
    med, mn = timeit(fn)
    res.setdefault(name, []).append((med, mn))
f_med = min(m for m, _ in res["fused"])
u_med = min(m for m, _ in res["unfused"])
gbs = bytes_fused / (f_med * 1e-3) / 1e9
print(f"B={B}: fused {f_med * 1e3:.1f} us  linear_fwd + winattn_fwd {u_med * 1e3:.1f} us  (saves {(u_med - f_med) * 1e3:.1f} us, "
      f"{u_med / f_med:.2f}x)")
print(f"fused: {bytes_fused / 1e9:.3f} GB algorithmic -> {gbs:.0f} GB/s = {gbs / args.hbm_gbs:.2f} of {args.hbm_gbs:.0f} GB/s")
print("runs (median, min ms):", res)
