"""ctypes binding of libmmn_b200.so (C ABI: include/mmn_b200.h) and its in-tree build.

The library is the product; there is no Python/CPU fallback.  `load()` raises if the
shared object is missing and every op raises if the C call returns an error.
"""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess
import threading

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG_DIR)
CSRC = os.path.join(PKG_DIR, "csrc")
# MMN_LIB=<path>: load another build of the library (A/B timing of kernel variants on one GPU box)
LIB_PATH = os.environ.get("MMN_LIB") or os.path.join(PKG_DIR, "libmmn_b200.so")
# translation unit -> headers it depends on (besides include/mmn_b200.h)
SOURCES = {"mmn_abi.cu": ["generic_launch.h", "attn_generic.cuh", "winattn_tc.h", "dropout_rng.cuh", "zero_fill.h"],
           "generic_launch.cu": ["generic_launch.h", "attn_generic.cuh", "dropout_rng.cuh", "zero_fill.h"],
           "winattn_tc.cu": ["winattn_tc.h", "winattn_tc_fwd.cuh", "winattn_tc_bwd.cuh", "winattn_tc_qkv_fwd.cuh", "tc_window.cuh", "tc_sched.cuh", "tc_common.cuh",
                             "zero_fill.h"],
           "linbwd_tc.cu": ["winattn_tc.h", "tc_window.cuh", "tc_common.cuh"],
           "gemm_tc.cu": ["winattn_tc.h", "tc_window.cuh", "tc_common.cuh"],
           "mha_tc.cu": ["winattn_tc.h", "tc_window.cuh", "tc_common.cuh", "dropout_rng.cuh"],
           "layernorm.cu": ["generic_launch.h", "attn_generic.cuh", "dropout_rng.cuh"],
           "cpb_bias.cu": ["generic_launch.h", "attn_generic.cuh", "dropout_rng.cuh", "zero_fill.h"]}
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC"]
# MMN_BUILD_TRACE=1 compiles the per-phase clock tracing into the tensor-core kernels (tools/trace_*.py);
# production builds leave it out (it costs ~8 % of the softmax warps' instructions).
if os.environ.get("MMN_BUILD_TRACE"):
    NVCC_FLAGS.append("-DMMN_TC_TRACING")
# MMN_NVCC_DEFINES="-DMMN_DEBUG_WAIT ...": extra nvcc defines for debugging builds (forces a rebuild)
NVCC_FLAGS += os.environ.get("MMN_NVCC_DEFINES", "").split()

# enums of include/mmn_b200.h
DT_F32, DT_BF16 = 0, 1
SCORE_SCALED, SCORE_COSINE = 0, 1
MASK_NONE, MASK_SHIFT, MASK_TENSOR, MASK_FUTURE = 0, 1, 2, 3
PATH_AUTO, PATH_GENERIC, PATH_TCGEN05 = 0, 1, 2
ACT_NONE, ACT_RELU, ACT_GELU = 0, 1, 2
LN_PRE, LN_POST = 0, 1
ABI_VERSION = 7
WINATTN_WORK_BYTES = 2048

EXPORTS = ["mmn_abi_version", "mmn_last_error", "mmn_winattn_path", "mmn_mha_path", "mmn_launch_count",
           "mmn_winattn_fwd", "mmn_winattn_qkv_path", "mmn_winattn_qkv_fwd", "mmn_winattn_bwd", "mmn_winattn_bwd_workspace_bytes", "mmn_mha_fwd", "mmn_mha_bwd", "mmn_mha_avg_weights",
           "mmn_colsum", "mmn_colsum_workspace_bytes", "mmn_layernorm_bwd_workspace_bytes",
           "mmn_linear_supported", "mmn_linear_fwd", "mmn_linear_bwd", "mmn_linear_bwd_supported", "mmn_linear_bwd_workspace_bytes",
           "mmn_cpb_bias_fwd", "mmn_cpb_bias_bwd", "mmn_table_bias_fwd", "mmn_table_bias_bwd", "mmn_layernorm_supported", "mmn_layernorm_fwd", "mmn_layernorm_bwd"]


class WinAttnDesc(C.Structure):
    _fields_ = [("ndim", C.c_int32), ("batch", C.c_int32),
                ("grid", C.c_int32 * 3), ("window", C.c_int32 * 3), ("shift", C.c_int32 * 3),
                ("num_heads", C.c_int32), ("head_dim", C.c_int32),
                ("score_kind", C.c_int32), ("mask_kind", C.c_int32), ("mask_windows", C.c_int32),
                ("io_dtype", C.c_int32), ("path", C.c_int32),
                ("scale", C.c_float), ("dropout_p", C.c_float),
                ("seed", C.c_uint64), ("offset", C.c_uint64),
                ("q_row_stride", C.c_int64), ("k_row_stride", C.c_int64), ("v_row_stride", C.c_int64),
                ("o_row_stride", C.c_int64), ("do_row_stride", C.c_int64), ("dq_row_stride", C.c_int64),
                ("dk_row_stride", C.c_int64), ("dv_row_stride", C.c_int64), ("deterministic", C.c_int32),
                ("rng", C.c_void_p)]


class MhaDesc(C.Structure):
    _fields_ = [("tgt_len", C.c_int32), ("src_len", C.c_int32), ("batch", C.c_int32),
                ("num_heads", C.c_int32), ("head_dim", C.c_int32),
                ("mask_kind", C.c_int32), ("mask_diagonal", C.c_int32),
                ("io_dtype", C.c_int32), ("path", C.c_int32),
                ("scale", C.c_float), ("dropout_p", C.c_float),
                ("seed", C.c_uint64), ("offset", C.c_uint64)] + \
               [(f"{t}_stride_{a}", C.c_int64) for t in ("q", "k", "v", "o", "do", "dq", "dk", "dv") for a in ("t", "b")] + \
               [("rng", C.c_void_p)]


def _stamp(files) -> float:
    return max(os.path.getmtime(f) for f in files if os.path.exists(f))


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile csrc/*.cu for sm_100a (one object per translation unit, rebuilt only when it
    or one of its headers changed) and link PKG_DIR/libmmn_b200.so.  nvcc cross-compiles
    without a GPU."""
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found: cannot build libmmn_b200.so")
    objdir = os.path.join(PKG_DIR, "build")
    os.makedirs(objdir, exist_ok=True)
    header = os.path.join(ROOT, "include", "mmn_b200.h")
    objs, procs = [], []
    for src, deps in SOURCES.items():
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        objs.append(obj)
        stamp = _stamp([os.path.join(CSRC, src), header] + [os.path.join(CSRC, d) for d in deps])
        if force or os.environ.get("MMN_BUILD_TRACE") or os.environ.get("MMN_NVCC_DEFINES") or not os.path.exists(obj) or os.path.getmtime(obj) < stamp:
            cmd = [nvcc] + NVCC_FLAGS + ["-c", os.path.join(CSRC, src), "-o", obj]
            if verbose:
                print(" ".join(cmd), flush=True)
            procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{out}")
    if procs or not os.path.exists(LIB_PATH) or os.path.getmtime(LIB_PATH) < _stamp(objs):
        cmd = [nvcc, "-shared", "-o", LIB_PATH + ".tmp"] + objs
        if verbose:
            print(" ".join(cmd), flush=True)
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError("link failed:\n" + res.stdout + res.stderr)
        os.replace(LIB_PATH + ".tmp", LIB_PATH)
    return LIB_PATH


_lock = threading.Lock()
_lib = None


def load() -> C.CDLL:
    """dlopen the library and type its entry points.  Raises loudly when it is absent."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                               "(multimodal_neuroimage_b200 has no CPU or PyTorch fallback)")
        lib = C.CDLL(LIB_PATH)
        vp, fp = C.c_void_p, C.c_void_p
        lib.mmn_abi_version.restype = C.c_int
        lib.mmn_last_error.restype = C.c_char_p
        lib.mmn_launch_count.restype = C.c_uint64
        lib.mmn_winattn_path.restype = C.c_char_p
        lib.mmn_winattn_path.argtypes = [C.POINTER(WinAttnDesc)]
        lib.mmn_mha_path.restype = C.c_char_p
        lib.mmn_mha_path.argtypes = [C.POINTER(MhaDesc)]
        lib.mmn_winattn_fwd.restype = C.c_int
        lib.mmn_winattn_fwd.argtypes = [C.POINTER(WinAttnDesc), vp, vp, vp, fp, fp, fp, vp, fp, vp, C.c_int, vp]
        lib.mmn_winattn_qkv_path.restype = C.c_char_p
        lib.mmn_winattn_qkv_path.argtypes = [C.POINTER(WinAttnDesc), C.c_int]
        lib.mmn_winattn_qkv_fwd.restype = C.c_int
        lib.mmn_winattn_qkv_fwd.argtypes = [C.POINTER(WinAttnDesc), vp, vp, fp, fp, fp, fp, vp, vp, fp, vp, C.c_int, vp]
        lib.mmn_winattn_bwd_workspace_bytes.restype = C.c_size_t
        lib.mmn_winattn_bwd_workspace_bytes.argtypes = [C.POINTER(WinAttnDesc)]
        lib.mmn_winattn_bwd.restype = C.c_int
        lib.mmn_winattn_bwd.argtypes = [C.POINTER(WinAttnDesc), vp, vp, vp, fp, fp, fp, vp, fp, vp, vp, vp, vp, fp, fp, fp, fp,
                                        C.c_int, vp]
        lib.mmn_mha_fwd.restype = C.c_int
        lib.mmn_mha_fwd.argtypes = [C.POINTER(MhaDesc), vp, vp, vp, fp, vp, fp, C.c_int, vp]
        lib.mmn_mha_bwd.restype = C.c_int
        lib.mmn_mha_bwd.argtypes = [C.POINTER(MhaDesc), vp, vp, vp, fp, vp, fp, vp, vp, vp, vp, fp, C.c_int, vp]
        lib.mmn_mha_avg_weights.restype = C.c_int
        lib.mmn_mha_avg_weights.argtypes = [C.POINTER(MhaDesc), vp, vp, fp, fp, fp, C.c_int, vp]
        lib.mmn_colsum.restype = C.c_int
        lib.mmn_colsum.argtypes = [vp, C.c_int, C.c_int64, C.c_int32, C.c_int64, fp, fp, C.c_int, C.c_int, vp]
        lib.mmn_colsum_workspace_bytes.restype = C.c_size_t
        lib.mmn_colsum_workspace_bytes.argtypes = [C.c_int64, C.c_int32]
        lib.mmn_cpb_bias_fwd.restype = C.c_int
        lib.mmn_cpb_bias_fwd.argtypes = [fp, fp, fp, fp, vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, fp, fp, C.c_int, vp]
        lib.mmn_table_bias_fwd.restype = C.c_int
        lib.mmn_table_bias_fwd.argtypes = [fp, vp, C.c_int32, C.c_int32, C.c_int32, fp, C.c_int, vp]
        lib.mmn_table_bias_bwd.restype = C.c_int
        lib.mmn_table_bias_bwd.argtypes = [fp, vp, vp, vp, C.c_int32, C.c_int32, C.c_int32, fp, C.c_int, vp]
        lib.mmn_cpb_bias_bwd.restype = C.c_int
        lib.mmn_cpb_bias_bwd.argtypes = [fp, fp, fp, fp, vp, vp, vp, fp, fp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                         fp, fp, fp, fp, C.c_int, vp]
        lib.mmn_linear_bwd_supported.restype = C.c_int
        lib.mmn_linear_bwd_supported.argtypes = [C.c_int, C.c_int64, C.c_int32, C.c_int32, C.c_int64, C.c_int64, C.c_int64]
        lib.mmn_linear_bwd_workspace_bytes.restype = C.c_size_t
        lib.mmn_linear_bwd_workspace_bytes.argtypes = [C.c_int64, C.c_int32, C.c_int32, C.c_int]
        lib.mmn_linear_bwd.restype = C.c_int
        lib.mmn_linear_bwd.argtypes = [vp, vp, vp, vp, fp, fp, vp, vp, C.c_int64, C.c_int, C.c_int, C.c_int64, C.c_int32, C.c_int32,
                                       C.c_int64, C.c_int64, C.c_int64, C.c_int, C.c_int, vp]
        lib.mmn_linear_supported.restype = C.c_int
        lib.mmn_linear_supported.argtypes = [C.c_int, C.c_int64, C.c_int32, C.c_int32, C.c_int64, C.c_int64]
        lib.mmn_linear_fwd.restype = C.c_int
        lib.mmn_linear_fwd.argtypes = [vp, vp, fp, vp, vp, C.c_int, C.c_int, C.c_int64, C.c_int32, C.c_int32, C.c_int64, C.c_int64,
                                       C.c_int, vp]
        lib.mmn_layernorm_supported.restype = C.c_int
        lib.mmn_layernorm_supported.argtypes = [C.c_int32]
        lib.mmn_layernorm_fwd.restype = C.c_int
        lib.mmn_layernorm_fwd.argtypes = [vp, C.c_int, vp, C.c_int, fp, fp, C.c_float, C.c_int, vp, C.c_int, vp, C.c_int, fp, fp,
                                          C.c_int64, C.c_int32, C.c_int, vp]
        lib.mmn_layernorm_bwd.restype = C.c_int
        lib.mmn_layernorm_bwd.argtypes = [vp, C.c_int, vp, C.c_int, vp, C.c_int, fp, fp, fp, C.c_int, vp, C.c_int, vp, C.c_int, fp, fp,
                                          fp, C.c_int, C.c_int64, C.c_int32, C.c_int, vp]
        lib.mmn_layernorm_bwd_workspace_bytes.restype = C.c_size_t
        lib.mmn_layernorm_bwd_workspace_bytes.argtypes = [C.c_int64, C.c_int32]
        if lib.mmn_abi_version() != ABI_VERSION:
            raise RuntimeError("libmmn_b200.so ABI version mismatch")
        _lib = lib
        return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().mmn_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"{what} failed (code {rc}): {msg}")


def launch_count() -> int:
    return int(load().mmn_launch_count())
