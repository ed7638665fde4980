"""CPU checks of the per-row-times fit: the C ABI declares and binds both entry points, and the kernel's local
Cox-de Boor triangle (spline_fit_times.cu: knot span by bisection, then only the p + 1 non-zero entries of each level,
same fp32 operations as deboor_basis) reproduces basis.bspline_basis bit for bit, including at knots, at the ends, for
clamped phases and with condition-order control points."""
import os

import numpy as np
import pytest
import torch

from beast_tokenizer_b200 import _lib, basis

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F32 = np.float32


def test_entry_points_declared_and_bound():
    header = open(os.path.join(ROOT, "include", "beast_b200.h")).read()
    for name in ("beast_fit_times_f32", "beast_fit_times_backward_f32"):
        assert f"int {name}(" in header
        assert name in _lib.exported_symbols()
    assert len(_lib._SIGNATURES["beast_fit_times_f32"][1]) == 9
    assert len(_lib._SIGNATURES["beast_fit_times_backward_f32"][1]) == 13


def knot_span(kn, lo, hi, u):
    while lo < hi:
        mid = (lo + hi + 1) >> 1
        if kn[mid] <= u:
            lo = mid
        else:
            hi = mid - 1
    return lo


def local_row(kn, nc, p, u):
    """(first column, p + 1 values) of the basis row at phase u, restated from fit_times_stage."""
    j = knot_span(kn, p, nc - 1, u)
    N = [F32(0)] * (p + 2)
    N[p] = F32(1)
    for k in range(1, p + 1):
        for i in range(j - k, j + 1):
            m = i - (j - p)
            d1 = F32(kn[i + k] - kn[i])
            d2 = F32(kn[i + k + 1] - kn[i + 1])
            t1 = F32(F32((u - kn[i]) / d1) * N[m]) if d1 != 0 else F32(0)
            t2 = F32(F32((kn[i + k + 1] - u) / d2) * N[m + 1]) if d2 != 0 else F32(0)
            N[m] = F32(t1 + t2) if (d1 != 0 and d2 != 0) else (t1 if d1 != 0 else t2)
    return j - p, N[:p + 1]


@pytest.mark.parametrize("nc,p", [(10, 4), (8, 3), (50, 0), (14, 4), (11, 3), (6, 1), (40, 4)])
def test_local_triangle_matches_full_recursion(nc, p):
    tau = float(torch.tensor(2 * np.pi, dtype=torch.float32))
    kn = basis.knot_vector(nc, p).numpy()
    g = torch.Generator().manual_seed(nc * 10 + p)
    t = torch.cat([torch.rand(400, generator=g) * 1.2 - 0.1,
                   torch.from_numpy(kn[p:nc + 1].astype(F32)) * tau,               # knots (as times)
                   torch.tensor([0.0, tau, -1.0, 2 * tau])]).to(torch.float32) * 1.0
    t[:400] *= tau
    full = basis.bspline_basis(t, tau, nc, p).numpy()
    u = basis.linear_phase(t, tau).numpy()
    for r in range(t.numel()):
        f, vals = local_row(kn, nc, p, u[r])
        row = np.zeros(nc + p + 1, F32)
        row[f:f + p + 1] = vals
        assert np.array_equal(row[:nc], full[r]), (r, float(u[r]))
        assert not np.any(full[r][:f]) and not np.any(full[r][f + p + 1:])
