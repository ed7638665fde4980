"""Host-side constants of one tokenizer: times, knots, basis Phi and the ridge projector P.

The reference rebuilds the basis (twice) and solves a [D*nb x D*nb] system per trajectory on
every encode (MP_lite_PyTorch/mp_pytorch/mp/uni_bspline.py:539-586).  Every trajectory shares
`self.times`, so all of that collapses to constants computed once here, on the CPU, with the
same fp32 torch operations the reference uses for times / phase / knots / basis (so Phi is
bit-identical to `mp.basis_gn.basis(times)`), and P = (Phi^T Phi + 1e-9 I)^-1 Phi^T in fp64.
"""
from dataclasses import dataclass
from typing import List, Optional

import torch


def make_times(duration: float, seq_len: int) -> torch.Tensor:
    """`self.times` (beast/beast_bspline_tokenizer.py:113 -> util_matrix.py:116, scalar branch)."""
    return torch.linspace(0, duration, seq_len)


def knot_vector(num_basis: int, degree_p: int) -> torch.Tensor:
    """Clamped uniform knots for `num_basis` control points (uni_bspline_basis.py:40-55; with
    init/end condition orders the caller passes num_ctrlp = num_basis + init + end)."""
    inner = num_basis + 1 - degree_p
    if inner < 1:
        raise ValueError(f"num_basis={num_basis} too small for degree_p={degree_p}")
    return torch.cat([torch.zeros(degree_p), torch.linspace(0, 1, inner), torch.ones(degree_p)]).to(torch.float32)


def linear_phase(times: torch.Tensor, tau: float) -> torch.Tensor:
    """clip((t - 0) / tau, 0, 1) with fp32 tau (linear_phase.py:22-23, phase_generator.py:41-42)."""
    t = times.to(torch.float32)
    tau_t = torch.tensor(tau, dtype=torch.float32)
    delay = torch.tensor(0.0, dtype=torch.float32)
    return torch.clip((t - delay) / tau_t, 0, 1)


def bspline_basis(times: torch.Tensor, tau: float, num_basis: int, degree_p: int) -> torch.Tensor:
    """Phi [..., T, num_basis], fp32.  Triangular (memoised) form of the Cox-de Boor recursion of
    uni_bspline_basis.py:82-113: each table entry is combined from the level below with exactly
    the reference's operations — ((u - k_i) / d1) * N[i] + ((k_{i+p+1} - u) / d2) * N[i+1], terms
    with a zero denominator dropped — so every value equals the recursive one bit for bit."""
    u = linear_phase(times, tau)
    kn = knot_vector(num_basis, degree_p)
    n0 = num_basis + degree_p
    level = []
    for i in range(n0):
        if i == num_basis - 1:
            inside = (u >= kn[i]) & (u <= kn[i + 1])       # last basis: closed on the right (:97-102)
        else:
            inside = (u >= kn[i]) & (u < kn[i + 1])
        level.append(inside.to(torch.float32))
    for p in range(1, degree_p + 1):
        nxt = []
        for i in range(n0 - p):
            d1 = kn[i + p] - kn[i]
            d2 = kn[i + p + 1] - kn[i + 1]
            t1 = None if d1 == 0 else (u - kn[i]) / d1 * level[i]
            t2 = None if d2 == 0 else (kn[i + p + 1] - u) / d2 * level[i + 1]
            if t1 is None and t2 is None:
                nxt.append(torch.zeros_like(u))
            elif t1 is None:
                nxt.append(t2)
            elif t2 is None:
                nxt.append(t1)
            else:
                nxt.append(t1 + t2)
        level = nxt
    return torch.stack(level[:num_basis], dim=-1).contiguous()


def check_orders(orders):
    """`orders` of the derivative API: a non-empty tuple / list of distinct ints from {0, 1, 2}."""
    if not isinstance(orders, (tuple, list)) or len(orders) == 0:
        raise ValueError(f"orders must be a non-empty tuple of distinct values from (0, 1, 2), got {orders!r}")
    for o in orders:
        if isinstance(o, bool) or not isinstance(o, int) or o not in (0, 1, 2):
            raise ValueError(f"orders must hold values from (0, 1, 2), got {orders!r}")
    if len(set(orders)) != len(orders):
        raise ValueError(f"orders must be distinct, got {orders!r}")
    return tuple(int(o) for o in orders)


def _deriv_step(level, kn, q, n_out):
    """d/du of the degree-q basis from the degree-(q-1) rows `level`: N'_i = q * (N_i / (k_{i+q} - k_i) -
    N_{i+1} / (k_{i+q+1} - k_{i+1})), terms with a zero denominator dropped.  One fp32 rounding per operation, in
    the order csrc/spline_deriv.cu (deboor_deriv) evaluates them."""
    out = []
    for i in range(n_out):
        d1 = kn[i + q] - kn[i]
        d2 = kn[i + q + 1] - kn[i + 1]
        a = None if d1 == 0 else level[i] / d1
        b = None if d2 == 0 else level[i + 1] / d2
        if a is None and b is None:
            v = torch.zeros_like(level[i])
        elif b is None:
            v = a
        elif a is None:
            v = -b
        else:
            v = a - b
        out.append(v * float(q))
    return out


def bspline_basis_derivatives(times: torch.Tensor, tau: float, num_basis: int, degree_p: int,
                              max_order: int) -> torch.Tensor:
    """[max_order + 1, T, num_basis] fp32: row o holds d^o/dt^o of the basis at `times` (o <= 2).

    Order 0 is `bspline_basis` bit for bit (same recursion, same operations).  Orders 1 / 2 are the derivative form
    of the same triangular recursion on the levels below the top one (`_deriv_step`), divided by tau once per order
    (t = u * tau).  Intervals are those of the basis: half-open, the last one closed, so an interior knot yields the
    right-hand derivative and t = 0 / t = tau the one-sided derivative from inside.  Outside [0, tau] the phase is
    clamped: the position is held and orders 1 / 2 are exactly 0.  csrc/spline_deriv.cu evaluates the same fp32
    operation sequence in-kernel, so these host rows and the device recursion agree bit for bit."""
    if isinstance(max_order, bool) or not isinstance(max_order, int) or max_order not in (0, 1, 2):
        raise ValueError(f"max_order must be 0, 1 or 2, got {max_order!r}")
    t = times.to(torch.float32)
    u = linear_phase(t, tau)
    tau_t = torch.tensor(tau, dtype=torch.float32)
    raw = (t - torch.tensor(0.0, dtype=torch.float32)) / tau_t
    outside = (raw < 0) | (raw > 1)
    kn = knot_vector(num_basis, degree_p)
    p = degree_p
    n0 = num_basis + p
    level = []
    for i in range(n0):
        if i == num_basis - 1:
            inside = (u >= kn[i]) & (u <= kn[i + 1])
        else:
            inside = (u >= kn[i]) & (u < kn[i + 1])
        level.append(inside.to(torch.float32))
    zero = torch.zeros_like(u)
    d1 = [zero] * num_basis
    d2 = [zero] * num_basis
    for q in range(1, p + 1):
        if q == p - 1 and max_order >= 2:            # level p-2 -> d/du of level p-1 -> d2/du2 of level p
            d2 = _deriv_step(_deriv_step(level, kn, p - 1, n0 - (p - 1)), kn, p, num_basis)
        if q == p and max_order >= 1:                # level p-1 -> d/du of level p
            d1 = _deriv_step(level, kn, p, num_basis)
        nxt = []
        for i in range(n0 - q):
            e1 = kn[i + q] - kn[i]
            e2 = kn[i + q + 1] - kn[i + 1]
            t1 = None if e1 == 0 else (u - kn[i]) / e1 * level[i]
            t2 = None if e2 == 0 else (kn[i + q + 1] - u) / e2 * level[i + 1]
            if t1 is None and t2 is None:
                nxt.append(torch.zeros_like(u))
            elif t1 is None:
                nxt.append(t2)
            elif t2 is None:
                nxt.append(t1)
            else:
                nxt.append(t1 + t2)
        level = nxt
    # degree 0: orders 1 / 2 stay exactly 0; degree 1: order 2 does
    rows = [torch.stack(level[:num_basis], dim=-1)]
    out = outside.unsqueeze(-1)
    if max_order >= 1:
        rows.append(torch.where(out, 0.0, torch.stack(d1, dim=-1) / tau_t))
    if max_order >= 2:
        rows.append(torch.where(out, 0.0, torch.stack(d2, dim=-1) / tau_t / tau_t))
    return torch.stack(rows).contiguous()


def ridge_projector(phi: torch.Tensor, reg: float = 1e-9) -> torch.Tensor:
    """P [nb, T] = (Phi^T Phi + reg I)^-1 Phi^T — the closed form of
    `solve(Phi_m^T Phi_m + 1e-9 I, Phi_m^T y)` (uni_bspline.py:564-586) for one DoF block, in fp64,
    rounded once to fp32."""
    f = phi.to(torch.float64)
    a = f.T @ f + reg * torch.eye(f.shape[1], dtype=torch.float64)
    return torch.linalg.solve(a, f.T).to(torch.float32).contiguous()


def ridge_projector64(phi: torch.Tensor, reg: float = 1e-9) -> torch.Tensor:
    f = phi.to(torch.float64)
    a = f.T @ f + reg * torch.eye(f.shape[1], dtype=torch.float64)
    return torch.linalg.solve(a, f.T)


def conditioned_projector(times: torch.Tensor, tau: float, phi_full: torch.Tensor, knots: torch.Tensor,
                          num_basis: int, degree_p: int, init_order: int, end_order: int) -> torch.Tensor:
    """Projector for init/end condition orders 1 and 2 (mp/uni_bspline.py:500-586).

    The reference pins the first `init_order` / last `end_order` control points to the boundary
    position and finite-difference velocity it reads off the trajectory itself
    (init_pos = y[0], init_vel = (y[1]-y[0])/dt, end_pos = y[-1] (- y[0]), end_vel =
    (y[-1]-y[-2])/dt; control points per uni_bspline_basis.py:192-274), subtracts their
    contribution (+ init_pos) from y and ridge-fits the remaining columns.  Every step is linear
    in y, so it is still w = P_eff . y with P_eff = P_learn (I - M): one [nb, T] table, fp64."""
    T = phi_full.shape[0]
    nc = num_basis + init_order + end_order
    f = phi_full.to(torch.float64)
    k = knots.to(torch.float64)
    t = times.to(torch.float64)
    tau64 = float(torch.tensor(tau, dtype=torch.float32))
    dt = float(t[1] - t[0])
    e = torch.eye(T, dtype=torch.float64)
    m = torch.zeros(T, T, dtype=torch.float64)
    if init_order != 0:
        m += torch.ones(T, 1, dtype=torch.float64) @ e[0:1]          # + init_pos on every sample
        if init_order == 2:                                           # ctrl 1 = init_vel*tau*dk/p (+0)
            dk = float(k[1 + degree_p] - k[1])
            m += f[:, 1:2] @ ((e[1:2] - e[0:1]) / dt * tau64 * dk / degree_p)
    if end_order != 0:
        end_pos = e[T - 1:T] - (e[0:1] if init_order != 0 else 0.0)  # relative when init_pos is pinned
        m += f[:, nc - 1:nc] @ end_pos
        if end_order == 2:
            dk = float(k[nc - 1 + degree_p] - k[nc - 1])
            end_vel = (e[T - 1:T] - e[T - 2:T - 1]) / dt
            m += f[:, nc - 2:nc - 1] @ (end_pos - end_vel * tau64 * dk / degree_p)
    p_learn = ridge_projector64(phi_full[:, init_order:nc - end_order])
    return (p_learn @ (e - m)).to(torch.float32).contiguous()


@dataclass
class SplineConstants:
    seq_len: int
    num_dof: int
    num_basis: int
    degree_p: int
    tau: float
    joint_indices: List[int]
    gripper_indices: List[int]
    times: torch.Tensor            # [T] fp32 (CPU)
    phi_joint: torch.Tensor        # [T, nb + init_order + end_order] (all control points)
    proj_joint: torch.Tensor       # [nb, T]
    knots_joint: torch.Tensor
    phi_grip: Optional[torch.Tensor]
    proj_grip: Optional[torch.Tensor]
    knots_grip: Optional[torch.Tensor]
    init_order: int = 0
    end_order: int = 0

    @property
    def slot_to_dof(self) -> List[int]:
        return list(self.joint_indices) + list(self.gripper_indices)


def build_constants(times: torch.Tensor, duration: float, num_basis: int, degree_p: int,
                    joint_indices, gripper_indices, init_order: int = 0, end_order: int = 0) -> SplineConstants:
    times = times.detach().to("cpu", torch.float32).reshape(-1).contiguous()
    nc = num_basis + init_order + end_order
    phi_j = bspline_basis(times, duration, nc, degree_p)
    knots_j = knot_vector(nc, degree_p)
    if init_order or end_order:
        proj_j = conditioned_projector(times, duration, phi_j, knots_j, num_basis, degree_p, init_order, end_order)
    else:
        proj_j = ridge_projector(phi_j)
    has_grip = len(gripper_indices) > 0
    phi_g = bspline_basis(times, duration, num_basis, 0) if has_grip else None
    return SplineConstants(
        seq_len=int(times.numel()), num_dof=len(joint_indices) + len(gripper_indices), num_basis=num_basis,
        degree_p=degree_p, tau=float(torch.tensor(duration, dtype=torch.float32)),
        joint_indices=list(joint_indices), gripper_indices=list(gripper_indices), times=times,
        phi_joint=phi_j, proj_joint=proj_j, knots_joint=knots_j,
        phi_grip=phi_g, proj_grip=ridge_projector(phi_g) if has_grip else None,
        knots_grip=knot_vector(num_basis, 0) if has_grip else None,
        init_order=init_order, end_order=end_order)
