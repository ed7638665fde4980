"""Gradients through the spline fit (encode_continuous backward): trajectory gradients against fp64 references on the
golden geometries and the condition orders, the adjoint identity, the tiled backward kernel against the generic one
bit for bit at multi-tile batch sizes with unaligned views and guard bands, edge semantics, no change without grad,
composition with the decode gradient, CUDA-graph capture and the C ABI's errors.
Run on the B200 box:  pytest -m gpu."""
import ctypes
import math

import numpy as np
import pytest
import torch

from conftest import GOLDEN_CASES, load_golden, rel_err

pytestmark = pytest.mark.gpu

TOL = 1e-5
COND_CFG = dict(num_dof=14, num_basis=10, seq_len=50, vocab_size=256, degree_p=4,
                gripper_zero_order=True, gripper_indices=[6, 13])
COND_ODD_CFG = dict(num_dof=5, num_basis=8, seq_len=33, vocab_size=1000, degree_p=3,
                    gripper_zero_order=True, gripper_indices=[0])
COND_CASES = [("cond_orders", o) for o in [(2, 0), (0, 2), (2, 2), (1, 1)]] + [("cond_odd", (2, 1))]
LOSS_KINDS = ("norm", "params", "both")
REPORT = {}


def _cfg(num_dof, num_basis=10, seq_len=50, degree_p=4, grippers=None):
    return dict(num_dof=num_dof, num_basis=num_basis, seq_len=seq_len, vocab_size=256, degree_p=degree_p,
                gripper_zero_order=bool(grippers), gripper_indices=grippers, llm_vocab_size=None)


# one geometry on each side of every dispatch boundary of the tiled kernel (see launch_restated)
SIZE_GEOMETRIES = {
    "shipped_d32_nb50_t10": GOLDEN_CASES["cli_default"],      # column sums of one term: projector through L1
    "cfg2_d14": GOLDEN_CASES["cfg2_d14"],                      # projector staged in shared memory, S = 64
    "d7_t1987": _cfg(7, seq_len=1987, grippers=[3]),           # projector beyond 32 KB: through L1
    "d57_t50": _cfg(57, grippers=[5, 56]),                     # staged, fewer trajectories per tile
}


def make_tok(cfg, g=None):
    from beast_tokenizer_b200 import BEASTBsplineTokenizer
    tok = BEASTBsplineTokenizer(device="cuda", **dict(cfg, llm_vocab_size=None))
    if g is not None:
        tok.w_min.copy_(torch.from_numpy(g["w_min_fit"]))
        tok.w_max.copy_(torch.from_numpy(g["w_max_fit"]))
    return tok


def cond_tok(case, orders):
    from beast_tokenizer_b200 import BEASTBsplineTokenizer
    io, eo = orders
    g = load_golden(case)
    cfg = COND_ODD_CFG if case == "cond_odd" else COND_CFG
    tok = BEASTBsplineTokenizer(device="cuda", init_cond_order=io, end_cond_order=eo, **cfg)
    tok.w_min.copy_(torch.from_numpy(g[f"o{io}{eo}_w_min"]))
    tok.w_max.copy_(torch.from_numpy(g[f"o{io}{eo}_w_max"]))
    return tok, g


def slots_of(tok):
    return list(tok.joint_indices) + list(tok.gripper_indices)


def chain64(tok, P_joint, P_grip, params, lo, hi, g_norm, g_params):
    """The dense fp64 adjoint: g_w [B, D, nb] from the loss gradients (mask / scale on the fp32 coefficients and
    bounds), then g_y [B, T, num_dof] = sum_k P[k, t] g_w[b, slot, k] with the joint or gripper projector [nb, T]."""
    B = params.shape[0]
    D, nb = tok.num_dof, tok.num_basis
    w = np.asarray(params, np.float32).reshape(B, D, nb)
    lo32 = np.asarray(lo, np.float32).reshape(D, nb)
    hi32 = np.asarray(hi, np.float32).reshape(D, nb)
    gw = np.zeros((B, D, nb))
    if g_norm is not None:
        scale = np.maximum(hi32.astype(np.float64) - lo32, 1e-8)
        mask = (w >= lo32) & (w <= hi32)
        gw += mask * (np.asarray(g_norm, np.float64).reshape(B, nb, D).transpose(0, 2, 1) * 2.0 / scale)
    if g_params is not None:
        gw += np.asarray(g_params, np.float64).reshape(B, D, nb)
    T = P_joint.shape[1]
    gy = np.zeros((B, T, D))
    nj = len(tok.joint_indices)
    for s, dof in enumerate(slots_of(tok)):
        P = P_joint if s < nj else P_grip
        gy[:, :, dof] = gw[:, s, :] @ np.asarray(P, np.float64)
    return gy


def independent_projectors(tok):
    """fp64 projectors rebuilt from the basis: the ridge solve, or conditioned_projector's fp64 product before its
    final rounding, restated."""
    from beast_tokenizer_b200 import basis
    c = tok._plan().consts
    io, eo = (c.init_order, c.end_order)
    nb, p = tok.num_basis, tok.degree_p
    nc = nb + io + eo
    times = c.times
    phi = basis.bspline_basis(times, tok.duration, nc, p)
    if io == 0 and eo == 0:
        Pj = basis.ridge_projector64(phi)
    else:
        T = phi.shape[0]
        f = phi.double()
        kn = basis.knot_vector(nc, p).double()
        t = times.double()
        tau = float(torch.tensor(tok.duration, dtype=torch.float32))
        dt = float(t[1] - t[0])
        e = torch.eye(T, dtype=torch.float64)
        m = torch.zeros(T, T, dtype=torch.float64)
        if io:
            m += torch.ones(T, 1, dtype=torch.float64) @ e[0:1]
            if io == 2:
                m += f[:, 1:2] @ ((e[1:2] - e[0:1]) / dt * tau * float(kn[1 + p] - kn[1]) / p)
        if eo:
            end_pos = e[T - 1:T] - (e[0:1] if io else 0.0)
            m += f[:, nc - 1:nc] @ end_pos
            if eo == 2:
                end_vel = (e[T - 1:T] - e[T - 2:T - 1]) / dt
                m += f[:, nc - 2:nc - 1] @ (end_pos - end_vel * tau * float(kn[nc - 1 + p] - kn[nc - 1]) / p)
        Pj = basis.ridge_projector64(phi[:, io:nc - eo]) @ (e - m)
    Pg = basis.ridge_projector64(basis.bspline_basis(times, tok.duration, nb, 0)) if tok.gripper_indices else None
    return Pj.numpy(), None if Pg is None else Pg.numpy()


def grad_of(tok, trajs, kind, seed, update_bounds=False):
    """x.grad of <normalised, Wn> + <params, Wp> (the terms of `kind`), with the forward's outputs and the bounds it
    normalised with."""
    x = trajs.clone().cuda().requires_grad_(True)
    norm, pd = tok.encode_continuous(x, update_bounds=update_bounds)
    lo, hi = tok.w_min.clone().cpu().numpy(), tok.w_max.clone().cpu().numpy()
    gen = torch.Generator(device="cuda").manual_seed(seed)
    wn = torch.randn(norm.shape, device="cuda", generator=gen) if kind in ("norm", "both") else None
    wp = torch.randn(norm.shape, device="cuda", generator=gen) if kind in ("params", "both") else None
    loss = 0.0
    if wn is not None:
        loss = loss + (norm * wn).sum()
    if wp is not None:
        loss = loss + (pd["params"] * wp).sum()
    loss.backward()
    c = lambda t: None if t is None else t.detach().cpu().numpy()
    return x.grad.cpu().numpy(), c(pd["params"]), lo, hi, c(wn), c(wp)


def check_against_fp64(tok, trajs, tag, seed):
    c = tok._plan().consts
    Pj32 = c.proj_joint.numpy()
    Pg32 = None if c.proj_grip is None else c.proj_grip.numpy()
    Pj64, Pg64 = independent_projectors(tok)
    for i, kind in enumerate(LOSS_KINDS):
        gx, params, lo, hi, wn, wp = grad_of(tok, trajs, kind, seed + i)
        for ref, P, Pg in (("tables", Pj32, Pg32), ("fp64", Pj64, Pg64)):
            want = chain64(tok, P, Pg, params, lo, hi, wn, wp)
            err = rel_err(gx, want)
            REPORT[(tag, kind, ref)] = err
            assert err <= TOL, (tag, kind, ref, err)


# ---------------------------------------------------------------- 1: against fp64
def test_grad_vs_fp64(golden_case):
    name, cfg, g = golden_case
    tok = make_tok(cfg, g)
    trajs = torch.from_numpy(g["trajs"])
    params = tok.compute_weights(trajs).cpu()
    lo, hi = tok.w_min.cpu(), tok.w_max.cpu()
    inside = ((params >= lo) & (params <= hi)).float().mean()
    assert 0.0 < inside < 1.0, (name, float(inside))         # the fit bounds clip some coefficients: both mask sides
    check_against_fp64(tok, trajs, name, 1)


@pytest.mark.parametrize("case,orders", COND_CASES)
def test_grad_vs_fp64_condition_orders(case, orders):
    tok, g = cond_tok(case, orders)
    trajs = torch.from_numpy(g["trajs"])
    check_against_fp64(tok, trajs, f"{case}{orders}", 2)
    # the boundary entries of params_dict: their gradients to the trajectories in closed form
    x = trajs.clone().cuda().requires_grad_(True)
    _, pd = tok.encode_continuous(x)
    keys = [k for k in ("init_pos", "init_vel", "end_pos", "end_vel") if pd[k] is not None]
    assert keys and all(pd[k].requires_grad for k in keys)
    gen = torch.Generator(device="cuda").manual_seed(9)
    ws = {k: torch.randn(pd[k].shape, device="cuda", generator=gen) for k in keys}
    sum((pd[k] * ws[k]).sum() for k in keys).backward()
    t = tok._plan().consts.times
    inv_dt = float(torch.tensor(1.0) / (t[1] - t[0]))
    want = np.zeros(x.shape)
    ji = list(tok.joint_indices)
    w = {k: v.double().cpu().numpy() for k, v in ws.items()}
    if "init_pos" in w:
        want[:, 0, ji] += w["init_pos"]
    if "init_vel" in w:
        want[:, 1, ji] += w["init_vel"] * inv_dt
        want[:, 0, ji] -= w["init_vel"] * inv_dt
    if "end_pos" in w:
        want[:, -1, ji] += w["end_pos"]                        # relative end_pos + y0: the y0 terms cancel
    if "end_vel" in w:
        want[:, -1, ji] += w["end_vel"] * inv_dt
        want[:, -2, ji] -= w["end_vel"] * inv_dt
    err = rel_err(x.grad.cpu().numpy(), want)
    REPORT[(f"{case}{orders}", "boundary", "closed form")] = err
    assert err <= 1e-6, (case, orders, err)
    # the state kept for later reconstructs holds no graph
    assert all(not v.requires_grad for v in tok._boundary.values() if isinstance(v, torch.Tensor))


# ---------------------------------------------------------------- 2: adjoint identity
@pytest.mark.parametrize("name", ["cfg1_d7", "cfg2_d14", "odd_d5", "cli_default"])
def test_adjoint_identity(name):
    cfg = GOLDEN_CASES[name]
    tok = make_tok(cfg)
    tok.w_min.fill_(-1e6)
    tok.w_max.fill_(1e6)                                       # mask all ones
    gen = torch.Generator(device="cuda").manual_seed(4)
    y = torch.randn(8, cfg["seq_len"], cfg["num_dof"], device="cuda", generator=gen).requires_grad_(True)
    _, pd = tok.encode_continuous(y)
    g = torch.randn(pd["params"].shape, device="cuda", generator=gen)
    (pd["params"] * g).sum().backward()
    lhs = float((pd["params"].detach().double() * g.double()).sum())
    rhs = float((y.detach().double() * y.grad.double()).sum())
    scale = float(pd["params"].detach().double().norm() * g.double().norm()
                  + y.detach().double().norm() * y.grad.double().norm())
    err = abs(lhs - rhs) / scale
    REPORT[(name, "params", "adjoint")] = err
    assert err <= 1e-6, (name, err)


# ---------------------------------------------------------------- 3 / 4: tiled == generic at multi-tile sizes
def launch_restated(tok, sms, optin):
    """launch_fit_grad_tiled's arithmetic: (S, grid, projector staged) or None when the generic kernel runs."""
    c = tok._plan().consts
    T, D, nb = c.seq_len, c.num_dof, c.num_basis
    nj = len(c.joint_indices)
    tabs = [(c.proj_joint, nj)] + ([(c.proj_grip, D - nj)] if c.proj_grip is not None else [])
    n_enc = sum(int((P != 0).any(1).sum()) * n for P, n in tabs)
    band_max = 0
    for P, _ in tabs:
        for t in range(T):
            nz = (P[:, t] != 0).nonzero().flatten()
            if nz.numel():
                band_max = max(band_max, int(nz[-1] - nz[0] + 1))
    p_bytes = 2 * T * (nb | 1) * 4
    p_smem = p_bytes <= 32 * 1024 and band_max > 2
    per = D * nb * 4
    extra = (3 * n_enc + 4 * T + D) * 4 + 16 + (p_bytes if p_smem else 0)
    budget = 108 * 1024
    if per + extra > budget:
        budget = optin
    if per + extra > budget:
        return None
    S = min(64, (budget - extra) // per)
    smem = S * per + extra
    per_sm = max(1, min(4, (220 * 1024) // (smem + 1024)))
    return S, sms * per_sm, p_smem


GUARD = 256


def _guarded(n, shift, fill):
    buf = torch.full((n + 2 * GUARD + shift,), fill, device="cuda")
    return buf, buf[GUARD + shift:GUARD + shift + n]


def _backward(tok, B, gn, gp, params, lo, hi, out):
    from beast_tokenizer_b200 import _lib
    plan = tok._plan()
    return plan._lib.beast_fit_backward_f32(plan.handle, B, _lib.ptr(gn), _lib.ptr(gp), _lib.ptr(params),
                                            _lib.ptr(lo), _lib.ptr(hi), _lib.ptr(out), _lib.stream_ptr(plan.device))


@pytest.mark.parametrize("name", list(SIZE_GEOMETRIES))
def test_tiled_equals_generic_at_size(name):
    from beast_tokenizer_b200 import _lib
    cfg = SIZE_GEOMETRIES[name]
    tok = make_tok(cfg)
    props = torch.cuda.get_device_properties(0)
    launch = launch_restated(tok, props.multi_processor_count, int(props.shared_memory_per_block_optin))
    assert launch is not None, name
    S, grid, p_smem = launch
    assert p_smem == (name in ("cfg2_d14", "d57_t50")), (name, p_smem)
    B = 3 * grid * S + S // 2 + 1                               # every CTA walks at least 3 tiles, ragged tail
    D, nb, T = cfg["num_dof"], cfg["num_basis"], cfg["seq_len"]
    n_in, n_out = B * D * nb, B * T * D
    gen = torch.Generator(device="cuda").manual_seed(7)
    lo = torch.rand(D * nb, device="cuda", generator=gen) * -2.0
    hi = lo + torch.rand(D * nb, device="cuda", generator=gen) * 4.0
    lo[:3] = hi[:3]                                             # degenerate columns
    ins = []
    for shift in (0, 1):                                        # aligned, then +4 B views of the three inputs
        bufs = [torch.empty(n_in + 4, device="cuda") for _ in range(3)]
        views = [b[shift:shift + n_in] for b in bufs]
        if shift == 0:
            for v in views:
                v.normal_(generator=gen)
            views[1].mul_(2.0)                                  # coefficients on both sides of the bounds
        else:
            for v, a in zip(views, ins[0][1]):
                v.copy_(a)
        ins.append((bufs, views))
    lib = _lib.load()
    for subset in (("n",), ("p",), ("n", "p")):
        res = {}
        for slow, shift in ((0, 0), (1, 0), (0, 1)):
            gn, params, gp = ins[shift][1]
            buf, out = _guarded(n_out, shift, float("nan"))
            prev = lib.beast_debug_disable_fast(slow)
            try:
                rc = _backward(tok, B, gn if "n" in subset else None, gp if "p" in subset else None,
                               params, lo, hi, out)
            finally:
                lib.beast_debug_disable_fast(prev)
            assert rc == 0, (name, rc)
            torch.cuda.synchronize()
            g = buf[:GUARD + shift], buf[GUARD + shift + n_out:]
            assert all(torch.isnan(x).all() for x in g), (name, subset, slow, shift, "store outside the window")
            assert not torch.isnan(out).any(), (name, subset, slow, shift)
            res[(slow, shift)] = out.clone()
            del buf, out
        assert torch.equal(res[(0, 0)], res[(1, 0)]), (name, subset, float((res[(0, 0)] - res[(1, 0)]).abs().max()))
        assert torch.equal(res[(0, 1)].view(torch.int32), res[(0, 0)].view(torch.int32)), (name, subset)
        del res
    del ins
    torch.cuda.empty_cache()


def test_public_api_unaligned_views():
    cfg = GOLDEN_CASES["cfg2_d14"]
    g = load_golden("cfg2_d14")
    tok = make_tok(cfg, g)
    x = torch.from_numpy(g["trajs"]).cuda()
    B = x.shape[0]
    base = torch.zeros(B * 50 * 14 + 1, device="cuda")
    base[1:].copy_(x.reshape(-1))
    grads = []
    for y in (x.clone().requires_grad_(True), base[1:].view(B, 50, 14).detach().requires_grad_(True)):
        norm, pd = tok.encode_continuous(y)
        gen = torch.Generator(device="cuda").manual_seed(3)
        w = torch.randn(B * 140 + 1, device="cuda", generator=gen)[1:].view(B, 140)   # +4 B gradient view
        (norm * w).sum().backward()
        grads.append(y.grad)
    assert torch.equal(grads[0], grads[1])


# ---------------------------------------------------------------- 5: edge semantics
def test_edge_semantics():
    from beast_tokenizer_b200 import _lib
    from beast_tokenizer_b200.utils import normalize_tensor
    cfg = GOLDEN_CASES["cfg2_d14"]
    g = load_golden("cfg2_d14")
    tok = make_tok(cfg)
    D, nb = 14, 10
    x = torch.from_numpy(g["trajs"][:8]).cuda()
    w = tok.compute_weights(x)                                  # [8, D*nb] '(d t)'
    # bounds: outside, inside and exactly at the bound (both sides), and degenerate columns
    lo, hi = w.min(0).values.clone(), w.max(0).values.clone()
    lo[0::4] = w[3, 0::4]                                       # row 3 at w_min, rows below it outside
    hi[1::4] = w[5, 1::4]                                       # row 5 at w_max
    lo[2::8] = w[2, 2::8]
    hi[2::8] = w[2, 2::8]                                       # degenerate: w_max == w_min == one row's value
    tok.w_min.copy_(lo)
    tok.w_max.copy_(hi)
    consts = tok._plan().consts
    # the degenerate columns get (g * 2) / 1e-8: a second pass without them, so that trajectory 2's other terms count
    degen = torch.zeros(D, nb, dtype=torch.bool, device="cuda")
    degen.view(-1)[2::8] = True
    gen = torch.Generator(device="cuda").manual_seed(1)
    wn0 = torch.randn(8, nb * D, device="cuda", generator=gen)
    for wn in (wn0, wn0 * ~degen.t().reshape(-1)):
        y = x.clone().requires_grad_(True)
        norm, pd = tok.encode_continuous(y)
        assert torch.equal(pd["params"].detach(), w)
        (norm * wn).sum().backward()
        # torch autograd through utils.normalize_tensor on the same fp32 coefficients, then the dense fp32-table chain
        c = w.clone().requires_grad_(True)
        nt = normalize_tensor(c, lo, hi).view(8, D, nb).transpose(1, 2).reshape(8, nb * D)
        (nt * wn).sum().backward()
        gw = c.grad.view(8, D, nb)
        at_bound = ((w == lo) | (w == hi)) & (wn.view(8, nb, D).transpose(1, 2).reshape(8, -1) != 0)
        assert at_bound.any() and (c.grad[at_bound] != 0).all()    # inclusive bounds: the full gradient
        assert ((w < lo) | (w > hi)).any() and (c.grad[(w < lo) | (w > hi)] == 0).all()
        gy = np.zeros(x.shape)
        for s, dof in enumerate(slots_of(tok)):
            P = (consts.proj_joint if s < len(tok.joint_indices) else consts.proj_grip).double().numpy()
            gy[:, :, dof] = gw[:, s, :].double().cpu().numpy() @ P
        # per trajectory: rows 3 / 5 hold coefficients exactly at w_min / w_max, row 2 the degenerate columns
        have = y.grad.double().cpu().numpy().reshape(8, -1)
        want = gy.reshape(8, -1)
        errs = np.abs(have - want).max(1) / np.maximum(np.abs(want).max(1), 1e-30)
        REPORT[("cfg2_d14", "bounds edge", "torch autograd")] = max(REPORT.get(("cfg2_d14", "bounds edge",
                                                                                  "torch autograd"), 0.0), errs.max())
        assert errs.max() <= TOL, errs
    # update_bounds=True, then another bounds update before backward: the snapshot of the call is used
    tok2 = make_tok(cfg, g)
    y2 = torch.from_numpy(g["trajs_ub"]).cuda().requires_grad_(True)
    norm2, pd2 = tok2.encode_continuous(y2, update_bounds=True)
    snap = tok2.w_min.clone().cpu().numpy(), tok2.w_max.clone().cpu().numpy()
    tok2.update_weights_bounds_per_batch(pd2["params"].detach() * 3.0)
    assert not np.array_equal(tok2.w_max.cpu().numpy(), snap[1])
    wn2 = torch.randn(norm2.shape, device="cuda", generator=gen)
    (norm2 * wn2).sum().backward()
    c2 = tok2._plan().consts
    want2 = chain64(tok2, c2.proj_joint.numpy(), c2.proj_grip.numpy(), pd2["params"].detach().cpu().numpy(),
                    *snap, wn2.cpu().numpy(), None)
    assert rel_err(y2.grad.cpu().numpy(), want2) <= TOL
    # extra trailing DoFs get 0; a CPU leaf receives the gradient through .to()
    xe = torch.cat([torch.from_numpy(g["trajs"][:4]), torch.randn(4, 50, 3)], dim=2).requires_grad_(True)
    norm3, _ = tok2.encode_continuous(xe)
    norm3.sum().backward()
    assert xe.grad.device.type == "cpu" and torch.all(xe.grad[..., D:] == 0) and xe.grad[..., :D].abs().sum() > 0
    # B = 0
    x0 = torch.zeros(0, 50, D, device="cuda", requires_grad=True)
    n0, p0 = tok2.encode_continuous(x0)
    (n0.sum() + p0["params"].sum()).backward()
    assert x0.grad.shape == (0, 50, D)
    # unused outputs: one output -> the other is NULL; neither -> no launch
    for use in ("norm", "params"):
        yy = x.clone().requires_grad_(True)
        nn_, pp = tok2.encode_continuous(yy)
        (nn_ if use == "norm" else pp["params"]).square().sum().backward()
        assert yy.grad.abs().sum() > 0
    yy = x.clone().requires_grad_(True)
    nn_, pp = tok2.encode_continuous(yy)
    n_before = _lib.launch_count()
    grads = torch.autograd.grad((nn_ * 0).sum() + (pp["params"] * 0).sum(), yy, allow_unused=True)
    assert _lib.launch_count() - n_before == 1                 # both used: one backward launch
    # double backward raises
    yy = x.clone().requires_grad_(True)
    nn_, _ = tok2.encode_continuous(yy)
    (gr,) = torch.autograd.grad(nn_.square().sum(), yy, create_graph=True)
    with pytest.raises(RuntimeError):
        gr.sum().backward()
    del grads


def test_unused_outputs_launch_nothing():
    from beast_tokenizer_b200 import _lib
    tok, g = cond_tok("cond_orders", (2, 2))
    y = torch.from_numpy(g["trajs"]).cuda().requires_grad_(True)
    _, pd = tok.encode_continuous(y)
    n0 = _lib.launch_count()
    pd["init_pos"].sum().backward()                            # only a boundary entry: the fit's node is not reached
    assert _lib.launch_count() == n0
    assert y.grad[:, 0, tok.joint_indices].eq(1).all()


class _DropGrad(torch.autograd.Function):
    """Identity whose backward passes no gradient: the node in front of it is reached with None for every output."""

    @staticmethod
    def forward(ctx, x):
        return x.clone()

    @staticmethod
    def backward(ctx, g):
        return None


def test_fit_node_without_gradients_launches_nothing():
    from beast_tokenizer_b200 import _lib
    tok = make_tok(GOLDEN_CASES["cfg2_d14"], load_golden("cfg2_d14"))
    y = torch.from_numpy(load_golden("cfg2_d14")["trajs"]).cuda().requires_grad_(True)
    norm, pd = tok.encode_continuous(y)
    loss = _DropGrad.apply(norm).sum() + _DropGrad.apply(pd["params"]).sum()
    n0 = _lib.launch_count()
    loss.backward()                                            # the fit's node runs with (None, None)
    torch.cuda.synchronize()
    assert _lib.launch_count() == n0
    assert y.grad is None


# ---------------------------------------------------------------- 6: no change without grad
def test_no_change_without_grad():
    from beast_tokenizer_b200 import _lib
    g = load_golden("cfg2_d14")
    for update_bounds in (False, True):
        outs = []
        for mode in ("parent", "no_req", "no_grad", "grad"):
            tok, _ = cond_tok("cond_orders", (2, 2))
            x = torch.from_numpy(g["trajs"]).cuda()
            n0 = _lib.launch_count()
            if mode == "parent":                              # the parent's call sequence
                with torch.no_grad():
                    _, params = tok._fit(x, want_tokens=False)
                    if update_bounds:
                        tok.update_weights_bounds_per_batch(params)
                    res = (tok._normalize(params), tok._params_dict(params))
            elif mode == "no_req":
                res = tok.encode_continuous(x, update_bounds=update_bounds)
            elif mode == "no_grad":
                with torch.no_grad():
                    res = tok.encode_continuous(x.clone().requires_grad_(True), update_bounds=update_bounds)
            else:
                res = tok.encode_continuous(x.clone().requires_grad_(True), update_bounds=update_bounds)
            n = _lib.launch_count() - n0
            norm, pd = res
            tensors = [norm] + [pd[k] for k in ("params", "init_pos", "init_vel", "end_pos", "end_vel")]
            if mode in ("no_req", "no_grad"):
                assert all(t.grad_fn is None and not t.requires_grad for t in tensors), mode
            if mode == "grad":
                assert all(t.requires_grad for t in tensors)
            assert all(not v.requires_grad for v in tok._boundary.values() if isinstance(v, torch.Tensor))
            outs.append((n, [t.detach() for t in tensors], tok.w_min.clone(), tok.w_max.clone()))
        for n, ts, lo, hi in outs[1:]:
            assert n == outs[0][0], (update_bounds, n, outs[0][0])
            for a, b in zip(ts, outs[0][1]):
                assert torch.equal(a.view(torch.int32), b.view(torch.int32))
            assert torch.equal(lo, outs[0][2]) and torch.equal(hi, outs[0][3])


# ---------------------------------------------------------------- 7: composition with the decode gradient
@pytest.mark.parametrize("name", ["cfg2_d14", "odd_d5"])
def test_projection_layer_composition(name):
    from scipy.interpolate import BSpline
    from beast_tokenizer_b200.basis import knot_vector
    cfg = GOLDEN_CASES[name]
    g = load_golden(name)
    tok = make_tok(cfg, g)
    y = torch.from_numpy(g["trajs"]).cuda().requires_grad_(True)
    norm, pd = tok.encode_continuous(y)
    pos, acc = tok.reconstruct_traj_continuous_derivatives(norm, orders=(0, 2))
    gen = torch.Generator(device="cuda").manual_seed(2)
    w0, w2 = (torch.randn(pos.shape, device="cuda", generator=gen) for _ in range(2))
    ((pos * w0).sum() + (acc * w2).sum()).backward()
    # dense fp64 chain: rows of the decode at the own times, the normalise / denormalise masks, the fit tables
    B, T, D = y.shape
    nb = cfg["num_basis"]
    c = tok._plan().consts
    tau = float(np.float32(2 * math.pi))
    u = np.clip(c.times.numpy().astype(np.float32) / np.float32(tau), 0, 1).astype(np.float64)
    spl = BSpline(knot_vector(nb, tok.degree_p).double().numpy(), np.eye(nb), tok.degree_p)
    rows = {0: spl(u), 2: spl.derivative(2)(u) / tau ** 2}
    grip = BSpline(knot_vector(nb, 0).double().numpy(), np.eye(nb), 0)(u)
    lo = tok.w_min.double().cpu().numpy().reshape(D, nb)
    hi = tok.w_max.double().cpu().numpy().reshape(D, nb)
    nrm = norm.detach().cpu().numpy().reshape(B, nb, D).transpose(0, 2, 1)
    gc = np.zeros((B, D, nb))
    nj = len(tok.joint_indices)
    for s, dof in enumerate(slots_of(tok)):
        if s < nj:
            gc[:, s] = w0.double().cpu().numpy()[:, :, dof] @ rows[0] + w2.double().cpu().numpy()[:, :, dof] @ rows[2]
        else:
            gc[:, s] = w0.double().cpu().numpy()[:, :, dof] @ grip
    g_norm = gc * 0.5 * (hi - lo) * ((nrm >= -1) & (nrm <= 1))   # denormalise, '(d t)'
    g_norm = g_norm.transpose(0, 2, 1).reshape(B, nb * D)
    want = chain64(tok, c.proj_joint.numpy(), None if c.proj_grip is None else c.proj_grip.numpy(),
                   pd["params"].detach().cpu().numpy(), lo.reshape(-1).astype(np.float32),
                   hi.reshape(-1).astype(np.float32), g_norm, None)
    err = rel_err(y.grad.cpu().numpy(), want)
    REPORT[(name, "composition", "composition fp64")] = err
    assert err <= TOL, (name, err)


# ---------------------------------------------------------------- 8: CUDA-graph capture of a training step
def test_graph_capture_training_step():
    cfg = GOLDEN_CASES["cfg2_d14"]
    g = load_golden("cfg2_d14")
    tok = make_tok(cfg, g)
    y = torch.from_numpy(g["trajs"]).cuda().requires_grad_(True)
    gen = torch.Generator(device="cuda").manual_seed(5)
    w0, w2 = (torch.randn(y.shape, device="cuda", generator=gen) for _ in range(2))

    def step():
        norm, _ = tok.encode_continuous(y)
        pos, acc = tok.reconstruct_traj_continuous_derivatives(norm, orders=(0, 2))
        ((pos - w0).square().mean() + 1e-3 * (acc * w2).square().mean()).backward()

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(3):
            y.grad = None
            step()
    torch.cuda.current_stream().wait_stream(s)
    eager = y.grad.clone()
    y.grad = None
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        step()
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(y.grad, eager) and eager.abs().sum() > 0


# ---------------------------------------------------------------- 9: C ABI errors
def test_c_abi_errors():
    from beast_tokenizer_b200 import _lib
    E_NULL, E_SHAPE, E_ALIGN = -1, -2, -3
    tok = make_tok(GOLDEN_CASES["cfg2_d14"])
    plan = tok._plan()
    lib = plan._lib
    B = 4
    buf = torch.zeros(B * 140 + 1, device="cuda")
    out = torch.zeros(B * 700 + 1, device="cuda")
    bnd = torch.zeros(141, device="cuda")
    G, O, W = _lib.ptr(buf), _lib.ptr(out), _lib.ptr(bnd)
    mis = ctypes.c_void_p(buf.data_ptr() + 2)
    st = _lib.stream_ptr(plan.device)

    def bw(h, b, gn, gp, par, lo, hi, o):
        return lib.beast_fit_backward_f32(h, b, gn, gp, par, lo, hi, o, st)

    assert bw(None, B, G, G, G, W, W, O) == E_NULL
    assert bw(plan.handle, B, None, None, G, W, W, O) == E_NULL            # no gradient at all
    assert bw(plan.handle, B, G, None, G, W, W, None) == E_NULL            # no output
    assert bw(plan.handle, B, G, None, None, W, W, O) == E_NULL            # grad_norm without params
    assert bw(plan.handle, B, G, None, G, None, W, O) == E_NULL            # ... or without bounds
    assert bw(plan.handle, B, G, None, G, W, None, O) == E_NULL
    assert bw(plan.handle, -1, G, None, G, W, W, O) == E_SHAPE
    assert bw(plan.handle, B, mis, None, G, W, W, O) == E_ALIGN
    assert bw(plan.handle, B, None, mis, None, None, None, O) == E_ALIGN
    assert bw(plan.handle, B, None, G, None, None, None, ctypes.c_void_p(out.data_ptr() + 1)) == E_ALIGN
    n0 = _lib.launch_count()
    assert bw(plan.handle, 0, G, None, G, W, W, O) == 0                    # B = 0: nothing launched
    assert _lib.launch_count() == n0
    assert bw(plan.handle, B, None, G, None, None, None, O) == 0           # grad_params alone needs no bounds
    torch.cuda.synchronize()


def test_zz_report():
    """Prints the observed normwise errors (pytest -s)."""
    groups = {}
    for key, v in REPORT.items():
        groups.setdefault(key[2], []).append(v)
    for kind, errs in sorted(groups.items()):
        print(f"{kind}: max normwise error {max(errs):.3e} over {len(errs)} gradients")
