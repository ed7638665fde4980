"""CPU checks of the masked fit: the C ABI declares and binds both entry points with their arities, and the boundary
samples of the condition orders (boundary_sample_indices: first, second, second-to-last and last valid sample of
each row, torch ops only) match a Python loop on random masks, including rows with 0, 1 and 2 valid samples, with
every index in range."""
import os

import pytest
import torch

from beast_tokenizer_b200 import _lib
from beast_tokenizer_b200.beast_bspline_tokenizer import boundary_sample_indices

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_entry_points_declared_and_bound():
    header = open(os.path.join(ROOT, "include", "beast_b200.h")).read()
    for name in ("beast_fit_masked_f32", "beast_fit_masked_backward_f32"):
        assert f"int {name}(" in header
        assert name in _lib.exported_symbols()
    assert len(_lib._SIGNATURES["beast_fit_masked_f32"][1]) == 12
    assert len(_lib._SIGNATURES["beast_fit_masked_backward_f32"][1]) == 16
    # the unmasked pair keeps its signatures
    assert len(_lib._SIGNATURES["beast_fit_times_f32"][1]) == 9
    assert len(_lib._SIGNATURES["beast_fit_times_backward_f32"][1]) == 13


def loop_indices(row):
    valid = [t for t, v in enumerate(row) if v]
    return valid[0], valid[1], valid[-2], valid[-1]


@pytest.mark.parametrize("T", [1, 2, 3, 5, 50, 97])
def test_boundary_indices_match_python_loop(T):
    g = torch.Generator().manual_seed(T)
    B = 400
    p = torch.rand(B, 1, generator=g)                       # per-row density, from empty to full
    mask = torch.rand(B, T, generator=g) < p
    mask[0] = False                                         # 0 valid
    mask[1] = False
    mask[1, T // 2] = True                                  # 1 valid
    if T >= 2:
        mask[2] = False
        mask[2, 0] = mask[2, T - 1] = True                  # 2 valid, at the ends
    mask[3] = True                                          # all valid
    idx = boundary_sample_indices(mask)
    assert all(i.dtype == torch.int64 and i.shape == (B,) for i in idx)
    for i in idx:
        assert int(i.min()) >= 0 and int(i.max()) < T
    counts = mask.sum(1)
    for b in range(B):
        if int(counts[b]) >= 2:
            assert tuple(int(i[b]) for i in idx) == loop_indices(mask[b].tolist()), b
    full = [int(i[3]) for i in idx]
    assert full == [0, min(1, T - 1), max(T - 2, 0), T - 1]
    one = [int(i[1]) for i in idx]
    assert one[0] == one[3] == T // 2                       # the single valid sample is first and last


def test_boundary_indices_empty_batch():
    idx = boundary_sample_indices(torch.zeros(0, 7, dtype=torch.bool))
    assert all(i.shape == (0,) for i in idx)
