"""Host test of the fused qkv forward's shape query (mmn_winattn_qkv_path): which self-attention calls the fused kernel
takes and why it refuses the others.  No GPU needed: the query only reads the descriptor."""
import pytest
import torch


@pytest.fixture(scope="module")
def mm():
    from multimodal_neuroimage_b200 import _lib, ops
    _lib.load()

    class NS:
        pass
    ns = NS()
    ns.lib, ns.ops = _lib, ops
    return ns


def _path(mm, C=96, nH=3, grid=(32, 32, 32), window=(4, 4, 4), shift=(2, 2, 2), dtype=torch.bfloat16, p=0.0,
          mask_kind=None, path=None, B=2):
    lib = mm.lib
    mask_kind = (lib.MASK_SHIFT if any(shift) else lib.MASK_NONE) if mask_kind is None else mask_kind
    return mm.ops.winattn_qkv_path_name((B, *grid, C), dtype, grid, window, shift, nH, lib.SCORE_COSINE, mask_kind, p,
                                        lib.PATH_AUTO if path is None else path)


# without a driver the tensor-map encoder cannot be looked up; that check comes after every shape check
_ACCEPT = {"tcgen05-fused", "cuTensorMapEncodeTiled unavailable"}


def test_accepts_the_tcgen05_forward_shapes_at_c96(mm):
    assert _path(mm) in _ACCEPT                                              # cfg2
    assert _path(mm, grid=(16, 16, 16), B=1) in _ACCEPT                      # all eight wrap classes, odd counts
    assert _path(mm, shift=(0, 0, 0)) in _ACCEPT
    assert _path(mm, grid=(16, 16), window=(8, 8), shift=(4, 4)) in _ACCEPT  # 2-D
    assert _path(mm, path=mm.lib.PATH_TCGEN05) in _ACCEPT


def test_refusal_reasons(mm):
    assert _path(mm, C=192, nH=6) == "the fused qkv kernel is built for 3 heads of 32 channels (C = 96)"
    assert _path(mm, C=64, nH=2) == "the fused qkv kernel is built for 3 heads of 32 channels (C = 96)"
    assert _path(mm, C=96, nH=2) == "the fused qkv kernel is built for 3 heads of 32 channels (C = 96)"
    assert _path(mm, dtype=torch.float32) == "io dtype is not bf16"
    assert _path(mm, p=0.1) == "attention dropout is only implemented in the generic path"
    assert _path(mm, window=(2, 2, 2), shift=(1, 1, 1)) == "window does not hold 64 tokens"
    assert _path(mm, mask_kind=mm.lib.MASK_TENSOR) == "mask tensor together with a cyclic shift"
    assert _path(mm, path=mm.lib.PATH_GENERIC) == "generic path requested"
    assert _path(mm, grid=(30, 32, 32)) == "invalid"
