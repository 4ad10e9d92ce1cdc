"""geometry.inverse_index: the CSR inverse of a bias-table index that the deterministic table-gradient gather walks."""
import math

import pytest
import torch

from multimodal_neuroimage_b200 import geometry


@pytest.mark.parametrize("window", [(3, 3), (7, 7), (4, 4, 4), (2, 3, 4), (4, 4, 2)])
def test_inverse_index_is_the_sorted_csr_inverse(window):
    index = geometry.relative_position_index(window).view(-1)
    T = math.prod(2 * w - 1 for w in window)
    perm, offsets = geometry.inverse_index(index, T)
    assert perm.dtype == offsets.dtype == torch.int32 and offsets.shape == (T + 1,)
    assert offsets[0] == 0 and offsets[-1] == index.numel()
    for t in range(T):
        run = perm[offsets[t]:offsets[t + 1]].long()
        assert torch.equal(run, torch.nonzero(index == t).view(-1))      # every entry of t, in increasing e
    cot = torch.randn(3, index.numel(), dtype=torch.float64)
    gathered = torch.stack([cot[:, perm[offsets[t]:offsets[t + 1]].long()].sum(1) for t in range(T)])
    assert torch.allclose(gathered, torch.zeros(T, 3, dtype=torch.float64).index_add_(0, index, cot.t()))
