"""CPU checks of the derivative tables (basis.bspline_basis_derivatives) and of the `orders` argument of the
derivative API: order 0 is the position basis bit for bit, orders 1 / 2 are the exact spline derivatives."""
import math

import numpy as np
import pytest
import torch
from scipy.interpolate import BSpline

from conftest import GOLDEN_CASES

TAU = 2 * math.pi
TAU32 = float(np.float32(TAU))

# (num_ctrlp, degree_p): the golden geometries, the condition-order geometries (num_basis + init + end columns),
# degree 1 and degree 0
GEOMETRIES = sorted({(c["num_basis"], c["degree_p"]) for c in GOLDEN_CASES.values()} |
                    {(10 + n, 4) for n in range(1, 5)} | {(8 + 3, 3), (6, 1), (9, 1), (10, 0)})


def grid(nc, p):
    """Samples at 0, tau, every knot (interior knots included), the tokenizer's own times and points outside."""
    from beast_tokenizer_b200.basis import knot_vector, make_times
    kn = knot_vector(nc, p)
    knots_t = (kn * torch.tensor(TAU32)).unique()
    return torch.cat([torch.tensor([0.0, TAU32, -1e-3, -2.0, TAU32 + 1e-3, TAU32 + 3.0]), knots_t,
                      make_times(TAU, 50), torch.linspace(-0.5, TAU + 0.5, 257)]).to(torch.float32)


def scipy_rows(times, nc, p, order):
    from beast_tokenizer_b200.basis import knot_vector
    kn = knot_vector(nc, p).double().numpy()
    t = times.numpy()
    raw = t / np.float32(TAU32)
    u = np.clip(raw.astype(np.float64), 0.0, 1.0)
    out = np.zeros((t.size, nc))
    if order <= p:
        for k in range(nc):
            e = np.zeros(nc)
            e[k] = 1.0
            spl = BSpline(kn, e, p)
            out[:, k] = (spl.derivative(order) if order else spl)(u) / TAU32 ** order
    if order:
        out[(raw < 0) | (raw > 1)] = 0.0
    return out


@pytest.mark.parametrize("nc,p", GEOMETRIES)
def test_order0_is_the_position_basis(nc, p):
    from beast_tokenizer_b200.basis import bspline_basis, bspline_basis_derivatives
    t = grid(nc, p)
    for max_order in (0, 1, 2):
        rows = bspline_basis_derivatives(t, TAU, nc, p, max_order)
        assert rows.shape == (max_order + 1, t.numel(), nc) and rows.dtype == torch.float32
        assert torch.equal(rows[0], bspline_basis(t, TAU, nc, p))
    # rows of a lower max_order are the leading rows of a higher one
    assert torch.equal(bspline_basis_derivatives(t, TAU, nc, p, 1), bspline_basis_derivatives(t, TAU, nc, p, 2)[:2])


@pytest.mark.parametrize("nc,p", GEOMETRIES)
def test_orders_1_2_match_scipy(nc, p):
    from beast_tokenizer_b200.basis import bspline_basis_derivatives
    t = grid(nc, p)
    rows = bspline_basis_derivatives(t, TAU, nc, p, 2).double().numpy()
    for order, tol in ((1, 5e-6), (2, 5e-6)):
        ref = scipy_rows(t, nc, p, order)
        scale = max(np.abs(ref).max(), 1e-30)
        assert np.abs(rows[order] - ref).max() <= tol * scale, (nc, p, order)
    raw = t.numpy() / np.float32(TAU32)
    outside = (raw < 0) | (raw > 1)
    assert outside.any() and not np.any(rows[1:, outside])                   # exactly 0 outside [0, tau]
    if p == 0:
        assert not np.any(rows[1:])
    if p == 1:
        assert not np.any(rows[2])


def test_boundary_derivatives_are_one_sided():
    """At t = 0 / t = tau the derivative of a clamped spline is the slope of its first / last control polygon leg."""
    from beast_tokenizer_b200.basis import bspline_basis_derivatives, knot_vector
    nc, p = 10, 4
    kn = knot_vector(nc, p).double()
    rows = bspline_basis_derivatives(torch.tensor([0.0, TAU32]), TAU, nc, p, 1).double()
    c = torch.linspace(-1.0, 2.0, nc, dtype=torch.float64) ** 2
    v0, v1 = (rows[1] @ c).tolist()
    assert v0 == pytest.approx(p / float(kn[p + 1] - kn[1]) * float(c[1] - c[0]) / TAU32, rel=1e-6)
    assert v1 == pytest.approx(p / float(kn[nc - 1 + p] - kn[nc - 1]) * float(c[-1] - c[-2]) / TAU32, rel=1e-6)


@pytest.mark.parametrize("bad", [(), [], (0, 0), (3,), (-1,), ("0",), (1.0,), (True,), None, 1, "012", (0, 1, 2, 0)])
def test_orders_validation(bad):
    from beast_tokenizer_b200 import BEASTBsplineTokenizer
    from beast_tokenizer_b200.basis import check_orders
    with pytest.raises(ValueError):
        check_orders(bad)
    tok = BEASTBsplineTokenizer(num_dof=7, device="cpu")
    toks = torch.zeros(2, 70, dtype=torch.long)
    with pytest.raises(ValueError):                     # checked before anything touches a device
        tok.reconstruct_traj_derivatives(toks, orders=bad)
    with pytest.raises(ValueError):
        tok.reconstruct_traj_continuous_derivatives(torch.zeros(2, 70), orders=bad)


def test_valid_orders_and_max_order():
    from beast_tokenizer_b200.basis import bspline_basis_derivatives, check_orders
    assert check_orders((2, 0)) == (2, 0) and check_orders([1]) == (1,)
    for bad in (-1, 3, True, 1.0):
        with pytest.raises(ValueError):
            bspline_basis_derivatives(torch.zeros(3), TAU, 10, 4, bad)
