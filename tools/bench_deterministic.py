"""What deterministic mode (torch.use_deterministic_algorithms(True)) costs, measured with the flag off and on alternately in
one process:
  core   the tensor-core window-attention backward alone at cfg2, batch 32 (CUDA events over bursts of 10 launches)
  cfg2   the graph-replayed SwinV2 window-attention module step (forward + backward) at cfg2, batch 32
  cfg3   the graph-replayed cfg3 TrainStep (bench.py's nested training line)
Writes a JSON record with the GPU name and power limit.  CUBLAS_WORKSPACE_CONFIG=:4096:8 is set for both modes (PyTorch
requires it for cuBLAS under the flag; the workloads' small layers still use cuBLAS).
Usage: python tools/bench_deterministic.py [--out profiles/det_overhead.json] [--rounds 3]"""
import argparse
import json
import os
import subprocess
import sys

os.environ.setdefault("CUBLAS_WORKSPACE_CONFIG", ":4096:8")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from multimodal_neuroimage_b200 import _lib, ops  # noqa: E402,F401
from multimodal_neuroimage_b200.modules import swin_v2_module as v2  # noqa: E402

GRID, WIN, SHIFT, NH, D, B = (32, 32, 32), (4, 4, 4), (2, 2, 2), 3, 32, 32


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def events(fn, iters, burst=10):
    """median ms per call over `iters` bursts of `burst` back-to-back calls"""
    for _ in range(5):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(burst):
            fn()
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1) / burst)
    ts.sort()
    return ts[len(ts) // 2]


def graphed(step):
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(3):
            step()
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        step()
    return g.replay


def core_setup():
    C = NH * D
    torch.manual_seed(0)
    qkv = torch.randn(B, *GRID, 3 * C, device="cuda", dtype=torch.bfloat16)
    dout = torch.randn(B, *GRID, C, device="cuda", dtype=torch.bfloat16)
    bias = torch.randn(NH, 64, 64, device="cuda")
    hs = torch.rand(NH, device="cuda") * 10 + 1
    cfg = (list(GRID), list(WIN), list(SHIFT), NH, _lib.SCORE_COSINE, _lib.MASK_SHIFT, 1.0, 0.0, 0, 0, _lib.PATH_AUTO)
    out, lse = torch.ops.mmn_b200.winattn_fwd(qkv, None, bias, hs, None, *cfg)
    return lambda: torch.ops.mmn_b200.winattn_bwd(dout, qkv, None, bias, hs, None, out, lse, *cfg, True)


def module_setup():
    torch.manual_seed(0)
    attn = v2.WindowAttention(NH * D, WIN, NH).cuda()
    x = torch.randn(B, GRID[0] * GRID[1] * GRID[2], NH * D, device="cuda", dtype=torch.bfloat16, requires_grad=True)
    dy = torch.randn_like(x)
    params = [p for p in attn.parameters() if p.requires_grad]

    def step():
        with torch.autocast("cuda", dtype=torch.bfloat16):
            y = attn.forward_grid(x, GRID, SHIFT)
        torch.autograd.grad(y, [x] + params, dy)
    return step


def cfg3_step(steps, warmup):
    import bench
    return bench.run_train_workload("cfg3", torch.device("cuda", 0), 0, 1, steps, warmup)["ms_per_step"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "det_overhead.json"))
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--iters", type=int, default=20)
    args = ap.parse_args()
    res = {"gpu": gpu_info(), "cublas_workspace_config": os.environ["CUBLAS_WORKSPACE_CONFIG"], "rounds": []}
    core = core_setup()
    module = module_setup()
    for r in range(args.rounds):
        row = {}
        for on in (False, True):
            torch.use_deterministic_algorithms(on)
            tag = "on" if on else "off"
            row[f"core_bwd_ms_{tag}"] = events(core, args.iters)
            row[f"cfg2_module_step_ms_{tag}"] = events(graphed(module), args.iters)
            torch.cuda.synchronize()
            row[f"cfg3_step_ms_{tag}"] = cfg3_step(20, 3)
            torch.cuda.empty_cache()
        torch.use_deterministic_algorithms(False)
        print(json.dumps(row), flush=True)
        res["rounds"].append(row)
    summary = {}
    for k in ("core_bwd_ms", "cfg2_module_step_ms", "cfg3_step_ms"):
        off = sorted(x[f"{k}_off"] for x in res["rounds"])[len(res["rounds"]) // 2]
        on = sorted(x[f"{k}_on"] for x in res["rounds"])[len(res["rounds"]) // 2]
        summary[k] = {"off": off, "on": on, "overhead_pct": 100.0 * (on - off) / off}
    res["median"] = summary
    print(json.dumps(summary, indent=1))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
