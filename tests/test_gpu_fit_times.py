"""The spline fit on per-row times (encode / encode_continuous / compute_weights / update_weights_bounds with
times=[B, T]): coefficients against an fp64 ridge solve on the same fp32 basis rows and against the reference's fp32
per-row fit, tokens against the exact quantiser, consistency with the shared-grid path, invariance (rows, batch
sizes, views, guard bands), gradients against fp64 autograd, CUDA-graph capture, unchanged behaviour without times,
BPE pass-through and errors of the Python API and the C ABI.
Run on the B200 box:  pytest -m gpu."""
import ctypes
import math

import numpy as np
import pytest
import torch

from conftest import GOLDEN_CASES, load_golden, rel_err

pytestmark = pytest.mark.gpu

COND_CFG = dict(num_dof=14, num_basis=10, seq_len=50, vocab_size=256, degree_p=4,
                gripper_zero_order=True, gripper_indices=[6, 13])
COND_ODD_CFG = dict(num_dof=5, num_basis=8, seq_len=33, vocab_size=1000, degree_p=3,
                    gripper_zero_order=True, gripper_indices=[0])
COND_CASES = [("cond_orders", o) for o in [(2, 0), (0, 2), (2, 2), (1, 1)]] + [("cond_odd", (2, 1))]
TIME_KINDS = ("uniform", "jitter", "scaled", "other_t")


def make_tok(case, orders=(0, 0)):
    from beast_tokenizer_b200 import BEASTBsplineTokenizer
    io, eo = orders
    if case in GOLDEN_CASES:
        g = load_golden(case)
        tok = BEASTBsplineTokenizer(device="cuda", **dict(GOLDEN_CASES[case], llm_vocab_size=None))
        tok.w_min.copy_(torch.from_numpy(g["w_min_fit"]))
        tok.w_max.copy_(torch.from_numpy(g["w_max_fit"]))
        return tok
    g = load_golden(case)
    cfg = COND_ODD_CFG if case == "cond_odd" else COND_CFG
    tok = BEASTBsplineTokenizer(device="cuda", init_cond_order=io, end_cond_order=eo, **cfg)
    tok.w_min.copy_(torch.from_numpy(g[f"o{io}{eo}_w_min"]))
    tok.w_max.copy_(torch.from_numpy(g[f"o{io}{eo}_w_max"]))
    return tok


ALL_CASES = [(c, (0, 0)) for c in GOLDEN_CASES] + COND_CASES
CASE_IDS = [f"{c}-o{o[0]}{o[1]}" for c, o in ALL_CASES]


def make_times(tok, B, kind, seed, T=None):
    """[B, T] fp32 timestamps: the tokenizer's grid, jittered samples (sorted, first step kept positive), a grid over a
    per-row fraction of the duration, or a different sample count."""
    g = torch.Generator().manual_seed(seed)
    T = tok.times.numel() if T is None else T
    dur = float(tok.duration)
    if kind == "uniform":
        return tok.times.expand(B, -1).clone()
    if kind == "jitter":
        base = torch.linspace(0, dur, T).expand(B, -1)
        step = dur / max(T - 1, 1)
        t = base + 0.3 * step * (torch.rand(B, T, generator=g) - 0.5)
        t[:, 0], t[:, -1] = 0.0, dur
        return t.clamp(0, dur).sort(dim=1).values.contiguous()
    if kind == "scaled":
        span = 0.75 + 0.25 * torch.rand(B, 1, generator=g)
        return (torch.linspace(0, 1, T).view(1, T) * span * dur).contiguous()
    if kind == "other_t":
        return torch.linspace(0, dur, T + 13).expand(B, -1).clone()
    raise ValueError(kind)


def trajs_for(tok, times, seed):
    """Smooth trajectories sampled at each row's times (+ small noise), fp32 [B, T, D]."""
    g = torch.Generator().manual_seed(seed)
    B, T = times.shape
    D = tok.num_dof
    amp = 0.02 * torch.randn(B, 1, D, generator=g)
    freq = 3.0 * torch.rand(B, 1, D, generator=g)
    phase = 2 * math.pi * torch.rand(B, 1, D, generator=g)
    u = (times / float(tok.duration)).unsqueeze(-1)
    y = amp * torch.sin(2 * math.pi * freq * u + phase) + 0.002 * torch.randn(B, T, D, generator=g)
    return y.to(torch.float32).contiguous()


def ridge64(tok, x, times, bc=None, bias=None):
    """fp64 ridge solve of every row on the fp32 basis rows at its own times (basis.bspline_basis), after subtracting
    the pinned points and the bias; returns (params [B, D*nb] fp64, max cond of the joint Gram matrices per row)."""
    from beast_tokenizer_b200 import basis
    c = tok._plan().consts
    io, eo, nb, p = c.init_order, c.end_order, tok.num_basis, tok.degree_p
    nc = nb + io + eo
    B, T, _ = x.shape
    nj = len(tok.joint_indices)
    out = np.zeros((B, tok.num_dof, nb))
    conds = np.zeros(B)
    for b in range(B):
        phi = basis.bspline_basis(times[b], tok.duration, nc, p).double().numpy()
        free = phi[:, io:io + nb]
        G = free.T @ free + 1e-9 * np.eye(nb)
        sup = np.abs(free).sum(0) > 0          # a column without samples is decoupled (exactly 0 by construction)
        conds[b] = np.linalg.cond(G[np.ix_(sup, sup)])
        y = x[b].double().numpy()
        for s, dof in enumerate(tok.joint_indices):
            t = y[:, dof].copy()
            if bias is not None:
                t -= float(bias[b, s])
            if bc is not None:
                pin = np.concatenate([phi[:, :io], phi[:, io + nb:]], axis=1)
                t -= pin @ bc[b, s].double().numpy()
            out[b, s] = np.linalg.solve(G, free.T @ t)
        if tok.gripper_indices:
            phig = basis.bspline_basis(times[b], tok.duration, nb, 0).double().numpy()
            Gg = phig.T @ phig + 1e-9 * np.eye(nb)
            for s, dof in enumerate(tok.gripper_indices):
                out[b, nj + s] = np.linalg.solve(Gg, phig.T @ y[:, dof])
    return out.reshape(B, -1), conds


def rowwise(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return np.linalg.norm(a - b, axis=1) / np.maximum(np.linalg.norm(b, axis=1), 1e-30)


def oracle_rows(tok, x, times):
    """The reference's op sequence (fp32 per-row fit) row by row with times[b]."""
    from oracle import beast_oracle as O
    io, eo = tok.init_cond_order, tok.end_cond_order
    ws = []
    for b in range(x.shape[0]):
        xb, tb = x[b:b + 1].numpy(), times[b].numpy()
        if io or eo:
            w, _ = O.compute_weights_cond(xb, tb, tok.duration, tok.num_basis, tok.degree_p, tok.joint_indices,
                                          tok.gripper_indices, io, eo)
        else:
            w = O.compute_weights(xb, tb, tok.duration, tok.num_basis, tok.degree_p, tok.joint_indices,
                                  tok.gripper_indices)
        ws.append(w[0])
    return np.stack(ws)


# ------------------------------------------------------------------ accuracy
@pytest.mark.parametrize("case,orders", ALL_CASES, ids=CASE_IDS)
@pytest.mark.parametrize("kind", TIME_KINDS)
def test_coefficients_match_fp64_and_oracle(case, orders, kind):
    from oracle import beast_oracle as O
    tok = make_tok(case, orders)
    B = 24
    t = make_times(tok, B, kind, seed=11)
    x = trajs_for(tok, t, seed=12)
    tokens, pd = tok.encode(x, times=t)
    params = pd["params"].cpu()
    st = tok._boundary
    bc = None if st is None else st["bc"].cpu()
    bias = None if st is None or st["bias"] is None else st["bias"].cpu()
    ref, conds = ridge64(tok, x, t, bc, bias)
    ok = conds <= 1e6
    assert ok.any()
    err = rowwise(params.numpy(), ref)[ok]
    assert err.max() <= 1e-6, (err.max(), conds.max())
    lo, hi = tok.w_min.cpu().numpy(), tok.w_max.cpu().numpy()
    exact = O.tokens_from_params(params.numpy(), lo, hi, tok.vocab_size, tok.num_dof, tok.num_basis, 0)
    assert np.array_equal(tokens.cpu().numpy(), exact)
    # the reference's fp32 LU amplifies its rounding by cond(G): compared where that stays below the bar
    well = conds <= 1e3
    assert well.any()
    sel = torch.from_numpy(well)
    w_or = oracle_rows(tok, x[sel], t[sel])
    assert rel_err(params.numpy()[well], w_or) <= 1e-5
    t_or = O.tokens_from_params(w_or, lo, hi, tok.vocab_size, tok.num_dof, tok.num_basis, 0)
    mine = tokens.cpu().numpy()[well]
    assert np.abs(mine - t_or).max(initial=0) <= 1
    D, nb, vm1 = tok.num_dof, tok.num_basis, tok.vocab_size - 1
    for b, r in np.argwhere(mine != t_or):     # flips only within the coefficient tolerance of a bin edge
        k, s = divmod(int(r), D)
        col = s * nb + k
        scale = max(float(hi[col]) - float(lo[col]), 1e-8)
        v = (min(max(float(w_or[b, col]), lo[col]), hi[col]) - lo[col]) / scale * vm1
        assert abs(v - math.floor(v) - 0.5) * scale / vm1 <= 1e-5 * np.abs(w_or[b]).max()


# ------------------------------------------------------------------ consistency
@pytest.mark.parametrize("case,orders", ALL_CASES, ids=CASE_IDS)
def test_shared_times_reproduce_default_path(case, orders):
    tok = make_tok(case, orders)
    B = 40
    x = trajs_for(tok, make_times(tok, B, "uniform", 3), seed=4)
    tok_a, pd_a = tok.encode(x)
    st_a = tok._boundary
    tok_b, pd_b = tok.encode(x, times=tok.times.expand(B, -1))
    st_b = tok._boundary
    assert rowwise(pd_b["params"].cpu(), pd_a["params"].cpu()).max() <= 1e-6
    assert (tok_a != tok_b).sum().item() <= max(1, tok_a.numel() // 1000)
    assert (tok_a - tok_b).abs().max().item() <= 1
    if st_a is not None:
        for k in ("bc", "init_pos", "init_vel", "end_pos", "end_vel"):
            if st_a[k] is not None:
                assert torch.equal(st_a[k], st_b[k]), k


def test_permuted_samples_give_same_coefficients():
    tok = make_tok("cfg2_d14")
    B = 16
    t = make_times(tok, B, "jitter", 5)
    x = trajs_for(tok, t, 6)
    w = tok.compute_weights(x, times=t).cpu()
    perm = torch.stack([torch.randperm(t.shape[1], generator=torch.Generator().manual_seed(b)) for b in range(B)])
    tp = torch.gather(t, 1, perm)
    xp = torch.gather(x, 1, perm.unsqueeze(-1).expand(-1, -1, x.shape[2]))
    wp = tok.compute_weights(xp, times=tp).cpu()
    assert rowwise(wp, w).max() <= 1e-6


def test_empty_supports_are_exact_zeros():
    tok = make_tok("cfg2_d14")
    B = 8
    t = (torch.linspace(0, 0.28, 50) * float(tok.duration)).expand(B, -1).contiguous()
    x = trajs_for(tok, t, 7)
    w = tok.compute_weights(x, times=t).cpu().view(B, tok.num_dof, tok.num_basis)
    # joint basis k (degree 4, inner knots at multiples of 1/6) starts at knot k: 6..9 start beyond phase 0.28;
    # gripper intervals (width 0.1) 3..9 likewise
    assert torch.equal(w[:, :12, 6:], torch.zeros_like(w[:, :12, 6:]))
    assert torch.equal(w[:, 12:, 3:], torch.zeros_like(w[:, 12:, 3:]))
    assert (w[:, :12, :6] != 0).all() and (w[:, 12:, :3] != 0).all()


def test_round_trip_in_spline_space():
    tok = make_tok("cfg2_d14")
    tok.w_min.fill_(-1.0)
    tok.w_max.fill_(1.0)
    B = 32
    t = make_times(tok, B, "jitter", 8, T=64)
    g = torch.Generator().manual_seed(9)
    norm = (1.6 * torch.rand(B, tok.num_basis * tok.num_dof, generator=g) - 0.8).cuda()
    y = tok.reconstruct_traj_continuous(norm, times=t.cuda())
    enc, _ = tok.encode_continuous(y, times=t)
    y2 = tok.reconstruct_traj_continuous(enc, times=t.cuda())
    assert rel_err(y2.cpu().numpy(), y.cpu().numpy()) <= 1e-5
    assert rel_err(enc.cpu().numpy(), norm.cpu().numpy()) <= 1e-5


def test_update_weights_bounds_times():
    tok = make_tok("odd_d5")
    t = make_times(tok, 300, "scaled", 10)
    x = trajs_for(tok, t, 11)
    tok.update_weights_bounds(x, times=t)
    w = tok.compute_weights(x, times=t)
    assert torch.equal(tok.w_min.cuda(), w.min(0).values) and torch.equal(tok.w_max.cuda(), w.max(0).values)
    tok2 = make_tok("odd_d5")
    toks, _ = tok2.encode(x, update_bounds=True, times=t)
    assert torch.equal(toks, tok2._quantize(w))


# ------------------------------------------------------------------ invariance
def test_bit_invariance_rows_batches_repeats():
    tok = make_tok("cfg2_d14")
    props = torch.cuda.get_device_properties(0)
    B = 3 * props.multi_processor_count * 4 * 8 + 77      # every warp walks >= 3 rows, ragged tail
    t = make_times(tok, B, "jitter", 12)
    x = trajs_for(tok, t, 13)
    w = tok.compute_weights(x, times=t)
    assert torch.equal(w, tok.compute_weights(x, times=t))
    sub = torch.arange(B - 300, B)
    assert torch.equal(w[sub], tok.compute_weights(x[sub], times=t[sub]))
    rev = torch.arange(B - 1, -1, -1)
    assert torch.equal(w[rev], tok.compute_weights(x[rev], times=t[rev]))
    assert torch.equal(w[:5], tok.compute_weights(x[:5], times=t[:5]))


def _abi_fit(tok, x, t, out):
    plan = tok._plan()
    lib = plan._lib
    return lib.beast_fit_times_f32(plan.handle, ctypes.c_void_p(x.data_ptr()), x.shape[0], t.shape[1],
                                   ctypes.c_void_p(t.data_ptr()), None, None, ctypes.c_void_p(out.data_ptr()), None)


def test_unaligned_views_and_guard_bands():
    tok = make_tok("odd_d5")
    B, n = 333, tok.num_dof * tok.num_basis
    t = make_times(tok, B, "jitter", 14).cuda()
    x = trajs_for(tok, t.cpu(), 15).cuda()
    ref = torch.empty(B, n, device="cuda")
    assert _abi_fit(tok, x, t, ref) == 0
    # inputs and output at +4 B, sentinels on both sides of the output window
    xb = torch.empty(x.numel() + 1, device="cuda"); xb[1:] = x.reshape(-1)
    tb = torch.empty(t.numel() + 1, device="cuda"); tb[1:] = t.reshape(-1)
    ob = torch.full((B * n + 65,), 12345.0, device="cuda")
    xv, tv, ov = xb[1:].view(x.shape), tb[1:].view(t.shape), ob[1:1 + B * n].view(B, n)
    assert _abi_fit(tok, xv, tv, ov) == 0
    torch.cuda.synchronize()
    assert torch.equal(ov, ref)
    assert ob[0].item() == 12345.0 and (ob[1 + B * n:] == 12345.0).all()
    # public API on offset views
    assert torch.equal(tok.compute_weights(xv, times=tv), ref)


# ------------------------------------------------------------------ gradients
def dense64(tok, y, times, lo, hi, mask, gn, gp):
    """fp64 autograd chain: boundary state (per-row dt), pinned subtraction, ridge solve on the fp32 basis rows,
    normalisation with the forward's clamp mask -> <normalised, gn> + <params, gp>."""
    from beast_tokenizer_b200 import basis
    c = tok._plan().consts
    io, eo, nb, p = c.init_order, c.end_order, tok.num_basis, tok.degree_p
    nc = nb + io + eo
    B, T, D = y.shape
    nj = len(tok.joint_indices)
    kn = basis.knot_vector(nc, p).double()
    tau = float(torch.tensor(tok.duration, dtype=torch.float32))
    rows = []
    for b in range(B):
        phi = basis.bspline_basis(times[b], tok.duration, nc, p).double()
        free = phi[:, io:io + nb]
        G = free.T @ free + 1e-9 * torch.eye(nb, dtype=torch.float64)
        yj = y[b][:, tok.joint_indices]
        inv_dt = float(torch.tensor(1.0) / (times[b, 1] - times[b, 0]))     # the fp32 factor the forward uses
        tgt = yj
        if io or eo:
            parts = []
            y0, y1, ym2, ym1 = yj[0], yj[1], yj[-2], yj[-1]
            if io:
                parts.append(torch.zeros_like(y0))
                if io == 2:
                    parts.append((y1 - y0) * inv_dt * tau * float(kn[1 + p] - kn[1]) / p)
            if eo:
                end_pos = ym1 - y0 if io else ym1
                if eo == 2:
                    parts.append(end_pos - (ym1 - ym2) * inv_dt * tau * float(kn[nc - 1 + p] - kn[nc - 1]) / p)
                parts.append(end_pos)
            bc = torch.stack(parts, dim=-1)                       # [nj, nbc]
            pin = torch.cat([phi[:, :io], phi[:, io + nb:]], dim=1)
            tgt = yj - pin @ bc.T - (y0 if io else 0.0)
        wj = torch.linalg.solve(G, free.T @ tgt).T                # [nj, nb]
        ws = [wj]
        if tok.gripper_indices:
            phig = basis.bspline_basis(times[b], tok.duration, nb, 0).double()
            Gg = phig.T @ phig + 1e-9 * torch.eye(nb, dtype=torch.float64)
            ws.append(torch.linalg.solve(Gg, phig.T @ y[b][:, tok.gripper_indices]).T)
        rows.append(torch.cat(ws, 0).reshape(-1))
    w = torch.stack(rows)                                          # [B, D*nb] '(d t)'
    scale = torch.clamp(hi - lo, min=1e-8)
    norm = ((w - lo) / scale * 2 - 1) * mask
    norm_td = norm.view(B, D, nb).transpose(1, 2).reshape(B, -1)
    return (norm_td * gn).sum() + (w * gp).sum()


@pytest.mark.parametrize("case,orders", ALL_CASES, ids=CASE_IDS)
def test_gradients_against_fp64_autograd(case, orders):
    tok = make_tok(case, orders)
    B = 12
    t = make_times(tok, B, "jitter", 20)
    x = trajs_for(tok, t, 21)
    xr = x.cuda().requires_grad_(True)
    norm, pd = tok.encode_continuous(xr, times=t)
    assert norm.grad_fn is not None
    gen = torch.Generator().manual_seed(22)
    gn, gp = torch.randn(norm.shape, generator=gen), torch.randn(norm.shape, generator=gen)
    ((norm * gn.cuda()).sum() + (pd["params"] * gp.cuda()).sum()).backward()
    lo = tok.w_min.double().cpu()
    hi = tok.w_max.double().cpu()
    w32 = pd["params"].detach().cpu()
    mask = ((w32 >= tok.w_min.cpu()) & (w32 <= tok.w_max.cpu())).double()
    y64 = x.double().requires_grad_(True)
    dense64(tok, y64, t, lo, hi, mask, gn.double(), gp.double()).backward()
    assert rel_err(xr.grad.cpu().numpy(), y64.grad.numpy()) <= 1e-5
    # adjoint identity: the fit is linear in y (boundary state included)
    x2 = x.cuda().requires_grad_(True)
    _, pd2 = tok.encode_continuous(x2, times=t)
    wp = torch.randn(pd2["params"].shape, generator=gen).cuda()
    (pd2["params"] * wp).sum().backward()
    lhs = float((pd2["params"].detach().double() * wp.double()).sum())
    rhs = float((x2.grad.double() * x.cuda().double()).sum())
    assert abs(lhs - rhs) <= 1e-5 * max(abs(lhs), 1e-12)


def test_composition_with_decode_and_graph_capture():
    tok = make_tok("cfg2_d14")
    tok.w_min.fill_(-0.5)
    tok.w_max.fill_(0.5)
    B = 64
    t = make_times(tok, B, "jitter", 30).cuda()
    x = trajs_for(tok, t.cpu(), 31).cuda()
    xr = x.clone().requires_grad_(True)
    enc, _ = tok.encode_continuous(xr, times=t)
    rec = tok.reconstruct_traj_continuous(enc, times=t)
    r = torch.randn(rec.shape, device="cuda", generator=torch.Generator(device="cuda").manual_seed(32))
    (rec * r).sum().backward()
    g_eager = xr.grad.clone()
    # the projection y -> P y is symmetric in the (row-wise) least-squares sense only without the ridge term; here
    # check against an fp64 restatement via autograd of the dense chain
    from beast_tokenizer_b200 import basis
    y64 = x.double().cpu().requires_grad_(True)
    out = []
    for b in range(B):
        phi = basis.bspline_basis(t[b].cpu(), tok.duration, tok.num_basis, tok.degree_p).double()
        G = phi.T @ phi + 1e-9 * torch.eye(tok.num_basis, dtype=torch.float64)
        yj = y64[b][:, tok.joint_indices]
        wj = torch.linalg.solve(G, phi.T @ yj)
        phig = basis.bspline_basis(t[b].cpu(), tok.duration, tok.num_basis, 0).double()
        Gg = phig.T @ phig + 1e-9 * torch.eye(tok.num_basis, dtype=torch.float64)
        wg = torch.linalg.solve(Gg, phig.T @ y64[b][:, tok.gripper_indices])
        full = torch.zeros(t.shape[1], tok.num_dof, dtype=torch.float64)
        full = full.index_add(1, torch.tensor(tok.joint_indices), phi @ wj)
        full = full.index_add(1, torch.tensor(tok.gripper_indices), phig @ wg)
        out.append(full)
    (torch.stack(out) * r.double().cpu()).sum().backward()
    assert rel_err(g_eager.cpu().numpy(), y64.grad.numpy()) <= 1e-5
    # one captured training step (forward + backward) replays to the eager result
    xs = x.clone().requires_grad_(True)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            xs.grad = None
            e, _ = tok.encode_continuous(xs, times=t)
            (tok.reconstruct_traj_continuous(e, times=t) * r).sum().backward()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    xs.grad = None
    with torch.cuda.graph(graph):
        e, _ = tok.encode_continuous(xs, times=t)
        (tok.reconstruct_traj_continuous(e, times=t) * r).sum().backward()
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(xs.grad, g_eager)


def test_no_grad_fn_and_same_launches_without_grad():
    from beast_tokenizer_b200 import _lib
    tok = make_tok("cond_orders", (2, 2))
    t = make_times(tok, 20, "jitter", 40).cuda()
    x = trajs_for(tok, t.cpu(), 41).cuda()
    n0 = _lib.launch_count()
    a, pa = tok.encode_continuous(x, times=t)
    n1 = _lib.launch_count()
    xr = x.clone().requires_grad_(True)
    with torch.no_grad():
        b, pb = tok.encode_continuous(xr, times=t)
    n2 = _lib.launch_count()
    assert a.grad_fn is None and pa["params"].grad_fn is None and b.grad_fn is None
    assert n1 - n0 == n2 - n1 == 2                     # fit + normalise
    assert torch.equal(a, b)
    c, _ = tok.encode_continuous(xr, times=t)
    assert torch.equal(c.detach(), a)
    assert tok._boundary["bc"].grad_fn is None


def test_unused_outputs_and_empty_batch():
    tok = make_tok("cond_orders", (1, 1))
    x = torch.zeros(0, 50, 14, device="cuda", requires_grad=True)
    t = torch.zeros(0, 50, device="cuda")
    n, pd = tok.encode_continuous(x, times=t)
    assert n.shape == (0, 140)
    n.sum().backward()
    assert x.grad.shape == x.shape
    tokens, _ = tok.encode(x.detach(), times=t)
    assert tokens.shape == (0, 140)


# ------------------------------------------------------------------ unchanged behaviour / BPE
@pytest.mark.parametrize("case,orders", [("cfg2_d14", (0, 0)), ("cond_orders", (2, 2))])
def test_times_none_is_todays_path(case, orders):
    from beast_tokenizer_b200 import _lib
    tok = make_tok(case, orders)
    x = trajs_for(tok, make_times(tok, 50, "uniform", 50), 51).cuda()
    res = []
    lo, hi = tok.w_min.clone(), tok.w_max.clone()
    for kw in ({}, {"times": None}):
        tok.w_min.copy_(lo)                    # update_weights_bounds below moves them
        tok.w_max.copy_(hi)
        n0 = _lib.launch_count()
        outs = [tok.encode(x, **kw)[0], tok.compute_weights(x, **kw), tok.encode_continuous(x, **kw)[0]]
        tok.update_weights_bounds(x, **kw)
        outs.append(tok.w_min.clone())
        res.append((_lib.launch_count() - n0, outs))
    assert res[0][0] == res[1][0]
    for u, v in zip(res[0][1], res[1][1]):
        assert torch.equal(u, v)


def test_bpe_passes_times_through():
    from beast_tokenizer_b200 import BEASTBsplineBPETokenizer
    tok = make_tok("cfg2_d14")
    t = make_times(tok, 64, "scaled", 60)
    x = trajs_for(tok, t, 61)
    btok = BEASTBsplineBPETokenizer.from_beast(tok, bpe_vocab_size=300)
    btok.fit_from_trajectories([{"actions": trajs_for(tok, make_times(tok, 64, "uniform", 62), 63)}],
                               show_progress=False)
    ids, _ = btok.encode(x, times=t)
    mp, _ = btok.encode_to_mp_tokens(x, times=t)
    assert ids == btok._discrete_to_bpe(mp)
    flat, off, _ = btok.encode_csr(x, times=t)
    flat, off = flat.cpu().tolist(), off.cpu().tolist()
    assert [flat[off[i]:off[i + 1]] for i in range(len(ids))] == [list(r) for r in ids]


# ------------------------------------------------------------------ errors
def test_python_errors():
    tok = make_tok("cfg2_d14")
    x = torch.zeros(4, 50, 14)
    with pytest.raises(AssertionError):
        tok.encode(x, times=torch.zeros(50))
    with pytest.raises(AssertionError):
        tok.encode(x, times=torch.zeros(3, 50))
    with pytest.raises(AssertionError):
        tok.compute_weights(x, times=torch.zeros(4, 49))
    tc = make_tok("cond_orders", (1, 0))
    with pytest.raises(AssertionError):
        tc.encode(torch.zeros(4, 1, 14), times=torch.zeros(4, 1))
    w = tok.compute_weights(torch.zeros(4, 1, 14), times=torch.zeros(4, 1))   # T = 1 without conditions
    assert w.shape == (4, 140)
    from beast_tokenizer_b200 import BEASTBsplineTokenizer
    from beast_tokenizer_b200._lib import BeastB200Error
    big = BEASTBsplineTokenizer(num_dof=2, num_basis=316, seq_len=400, degree_p=4, device="cuda")
    with pytest.raises(BeastB200Error, match="unsupported"):
        big.compute_weights(torch.zeros(2, 400, 2), times=torch.zeros(2, 400))


def test_c_abi_errors():
    tok = make_tok("cond_orders", (2, 2))
    plan = tok._plan()
    lib = plan._lib
    vp = lambda t: ctypes.c_void_p(t.data_ptr())
    x = torch.zeros(2, 50, 14, device="cuda")
    t = torch.zeros(2, 50, device="cuda")
    out = torch.zeros(2, 140, device="cuda")
    bc = torch.zeros(2, 12, 4, device="cuda")
    assert lib.beast_fit_times_f32(None, vp(x), 2, 50, vp(t), vp(bc), None, vp(out), None) == -1
    assert lib.beast_fit_times_f32(plan.handle, vp(x), 2, 50, vp(t), None, None, vp(out), None) == -1
    assert lib.beast_fit_times_f32(plan.handle, None, 2, 50, vp(t), vp(bc), None, vp(out), None) == -1
    assert lib.beast_fit_times_f32(plan.handle, vp(x), -1, 50, vp(t), vp(bc), None, vp(out), None) == -2
    assert lib.beast_fit_times_f32(plan.handle, vp(x), 2, 1, vp(t), vp(bc), None, vp(out), None) == -2
    assert lib.beast_fit_times_f32(plan.handle, vp(x), 2, 0, vp(t), vp(bc), None, vp(out), None) == -2
    assert lib.beast_fit_times_f32(plan.handle, None, 0, 50, None, None, None, None, None) == 0
    mis = ctypes.c_void_p(out.data_ptr() + 2)
    assert lib.beast_fit_times_f32(plan.handle, vp(x), 2, 50, vp(t), vp(bc), None, mis, None) == -3
    g = torch.zeros(2, 50, 14, device="cuda")
    gp = torch.zeros(2, 140, device="cuda")
    bwd = lib.beast_fit_times_backward_f32
    assert bwd(plan.handle, 2, 50, vp(t), None, None, None, None, None, vp(g), vp(bc), None, None) == -1
    assert bwd(plan.handle, 2, 50, vp(t), vp(gp), None, None, None, None, vp(g), vp(bc), None, None) == -1
    assert bwd(plan.handle, 2, 50, vp(t), None, vp(gp), None, None, None, vp(g), None, None, None) == -1
    assert bwd(plan.handle, 2, 1, vp(t), None, vp(gp), None, None, None, vp(g), vp(bc), None, None) == -2
    assert bwd(plan.handle, 0, 50, None, None, vp(gp), None, None, None, None, None, None, None) == 0
    assert bwd(plan.handle, 2, 50, vp(t), None, vp(gp), None, None, None, vp(g), vp(bc), None, None) == 0
    torch.cuda.synchronize()
    from beast_tokenizer_b200 import BEASTBsplineTokenizer
    big = BEASTBsplineTokenizer(num_dof=2, num_basis=316, seq_len=400, degree_p=4, device="cuda")
    bp = big._plan()
    x2, t2, o2 = torch.zeros(1, 400, 2, device="cuda"), torch.zeros(1, 400, device="cuda"), torch.zeros(1, 632,
                                                                                                      device="cuda")
    assert bp._lib.beast_fit_times_f32(bp.handle, vp(x2), 1, 400, vp(t2), None, None, vp(o2), None) == -4
    assert bp._lib.beast_fit_times_backward_f32(bp.handle, 1, 400, vp(t2), None, vp(o2), None, None, None, vp(x2),
                                                None, None, None) == -4
