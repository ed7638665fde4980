"""The masked spline fit (encode / encode_continuous / compute_weights / update_weights_bounds with mask=[B, T]):
every row equals the per-row fit of its compacted row bit for bit, rows without a masked sample equal the unmasked
call bit for bit, accuracy against an fp64 ridge solve on the valid samples, padding garbage never reaches an output,
degenerate rows, tokens and bounds, gradients against fp64 autograd, invariance (rows, batch sizes, chunk-straddling
masks, views, guard bands, partial_only), CUDA-graph capture and the K1 / K3 overlap bookkeeping, BPE pass-through and
errors of the Python API and the C ABI.
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
ALL_CASES = [(c, (0, 0)) for c in GOLDEN_CASES] + COND_CASES
CASE_IDS = [f"{c}-o{o[0]}{o[1]}" for c, o in ALL_CASES]
MASK_KINDS = ("suffix", "prefix", "drops", "run", "all")


def make_tok(case, orders=(0, 0)):
    from beast_tokenizer_b200 import BEASTBsplineTokenizer
    io, eo = orders
    g = load_golden(case)
    if case in GOLDEN_CASES:
        tok = BEASTBsplineTokenizer(device="cuda", **dict(GOLDEN_CASES[case], llm_vocab_size=None))
        tok.w_min.copy_(torch.from_numpy(g["w_min_fit"]))
        tok.w_max.copy_(torch.from_numpy(g["w_max_fit"]))
        return tok
    cfg = COND_ODD_CFG if case == "cond_odd" else COND_CFG
    tok = BEASTBsplineTokenizer(device="cuda", init_cond_order=io, end_cond_order=eo, **cfg)
    tok.w_min.copy_(torch.from_numpy(g[f"o{io}{eo}_w_min"]))
    tok.w_max.copy_(torch.from_numpy(g[f"o{io}{eo}_w_max"]))
    return tok


def jitter_times(tok, B, seed, T=None):
    g = torch.Generator().manual_seed(seed)
    T = tok.times.numel() if T is None else T
    dur = float(tok.duration)
    step = dur / max(T - 1, 1)
    t = torch.linspace(0, dur, T).expand(B, -1) + 0.3 * step * (torch.rand(B, T, generator=g) - 0.5)
    t[:, 0], t[:, -1] = 0.0, dur
    return t.clamp(0, dur).sort(dim=1).values.contiguous()


def trajs_for(tok, times, seed):
    g = torch.Generator().manual_seed(seed)
    B, T = times.shape
    D = tok.num_dof
    amp = 0.02 * torch.randn(B, 1, D, generator=g)
    freq = 3.0 * torch.rand(B, 1, D, generator=g)
    phase = 2 * math.pi * torch.rand(B, 1, D, generator=g)
    u = (times / float(tok.duration)).unsqueeze(-1)
    y = amp * torch.sin(2 * math.pi * freq * u + phase) + 0.002 * torch.randn(B, T, D, generator=g)
    return y.to(torch.float32).contiguous()


def make_mask(kind, B, T, seed, full_every=0):
    """bool [B, T]: suffix padding of random length, a missing prefix, 10-30 % random drops, one valid run, or all
    valid.  Every row keeps at least max(2, T // 2) valid samples (a well-posed fit); with full_every = k every k-th
    row is all True."""
    g = torch.Generator().manual_seed(seed)
    ar = torch.arange(T).expand(B, T)
    keep = max(2, T // 2)
    if kind == "all":
        m = torch.ones(B, T, dtype=torch.bool)
    elif kind == "suffix":
        n = torch.randint(keep, T, (B, 1), generator=g)
        m = ar < n
    elif kind == "prefix":
        n = torch.randint(1, T - keep + 1, (B, 1), generator=g)
        m = ar >= n
    elif kind == "drops":
        rate = 0.1 + 0.2 * torch.rand(B, 1, generator=g)
        m = torch.rand(B, T, generator=g) >= rate
        m[:, :2] = True
    elif kind == "run":
        n = torch.randint(keep, T, (B, 1), generator=g)
        a = (torch.rand(B, 1, generator=g) * (T - n + 1)).long()
        m = (ar >= a) & (ar < a + n)
    else:
        raise ValueError(kind)
    if full_every:
        m[::full_every] = True
    return m.contiguous()


def compact(tok, x, times, mask, b):
    """(y [1, k, D], times [1, k]) of row b's valid samples (times None: the tokenizer's times)."""
    mb = mask[b].cpu()
    t = tok.times if times is None else times[b].cpu()
    return x[b:b + 1, mb.to(x.device)], t[mb].unsqueeze(0).contiguous()


def rowwise(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return np.linalg.norm(a - b, axis=1) / np.maximum(np.linalg.norm(b, axis=1), 1e-30)


def ridge64(tok, x, times, mask, bc=None, bias=None):
    """fp64 ridge solve of every row on the fp32 basis rows at its valid samples only (weights 0 / 1), after
    subtracting the pinned points and the bias; (params [B, D*nb], cond of each row's joint Gram matrix)."""
    from beast_tokenizer_b200 import basis
    c = tok._plan().consts
    io, eo, nb, p = c.init_order, c.end_order, tok.num_basis, tok.degree_p
    nc = nb + io + eo
    B = x.shape[0]
    nj = len(tok.joint_indices)
    out = np.zeros((B, tok.num_dof, nb))
    conds = np.zeros(B)
    for b in range(B):
        m = mask[b].cpu().numpy()
        tb = (tok.times if times is None else times[b].cpu())
        wgt = m.astype(np.float64)
        phi = basis.bspline_basis(tb, tok.duration, nc, p).double().numpy()
        free = phi[:, io:io + nb]
        G = free.T @ (wgt[:, None] * free) + 1e-9 * np.eye(nb)
        sup = np.abs(free[m]).sum(0) > 0
        conds[b] = np.linalg.cond(G[np.ix_(sup, sup)]) if sup.any() else np.inf
        y = np.where(m[:, None], x[b].double().cpu().numpy(), 0.0)
        for s, dof in enumerate(tok.joint_indices):
            t = y[:, dof].copy()
            if bias is not None:
                t -= float(bias[b, s])
            if bc is not None:
                pin = np.concatenate([phi[:, :io], phi[:, io + nb:]], axis=1)
                t -= pin @ bc[b, s].double().cpu().numpy()
            out[b, s] = np.linalg.solve(G, free.T @ (wgt * t))
        if tok.gripper_indices:
            phig = basis.bspline_basis(tb, tok.duration, nb, 0).double().numpy()
            Gg = phig.T @ (wgt[:, None] * phig) + 1e-9 * np.eye(nb)
            for s, dof in enumerate(tok.gripper_indices):
                out[b, nj + s] = np.linalg.solve(Gg, phig.T @ (wgt * y[:, dof]))
    return out.reshape(B, -1), conds


def state_of(tok):
    st = tok._boundary
    return None if st is None else {k: None if v is None else v.clone() for k, v in st.items()}


# ------------------------------------------------------------------ compaction identity and accuracy
@pytest.mark.parametrize("case,orders", ALL_CASES, ids=CASE_IDS)
@pytest.mark.parametrize("kind", MASK_KINDS)
@pytest.mark.parametrize("grid", ["shared", "per_row"])
def test_rows_equal_compacted_fit(case, orders, kind, grid):
    from oracle import beast_oracle as O
    tok = make_tok(case, orders)
    B = 12
    T = tok.times.numel()
    t = None if grid == "shared" else jitter_times(tok, B, 11)
    x = trajs_for(tok, tok.times.expand(B, -1) if t is None else t, 12).cuda()
    m = make_mask(kind, B, T, 13, full_every=4)
    tokens, pd = tok.encode(x, mask=m.cuda(), times=t)
    st = state_of(tok)
    params = pd["params"]
    # tokens are the exact quantiser of the returned coefficients
    lo, hi = tok.w_min.cpu().numpy(), tok.w_max.cpu().numpy()
    exact = O.tokens_from_params(params.cpu().numpy(), lo, hi, tok.vocab_size, tok.num_dof, tok.num_basis, 0)
    assert np.array_equal(tokens.cpu().numpy(), exact)
    assert torch.equal(tokens, tok._quantize(params))
    for b in range(B):
        if t is None and bool(m[b].all()):
            continue                                   # a full row on the shared grid is K1's result (tested below)
        xc, tc = compact(tok, x, t, m, b)
        w = tok.compute_weights(xc, times=tc)
        assert torch.equal(params[b:b + 1], w), b
        if st is not None:
            ref = tok._boundary
            for k in ("bc", "bias", "init_pos", "init_vel", "end_pos", "end_vel"):
                if st[k] is not None:
                    assert torch.equal(st[k][b:b + 1], ref[k]), (b, k)
            for k in ("init_pos", "init_vel", "end_pos", "end_vel"):
                if pd[k] is not None:
                    assert torch.equal(pd[k][b:b + 1], ref[k]), (b, k)
    # fp64 weighted ridge on the same fp32 basis rows
    bc = None if st is None else st["bc"].cpu()
    bias = None if st is None or st["bias"] is None else st["bias"].cpu()
    ref, conds = ridge64(tok, x.cpu(), t, m, bc, bias)
    ok = conds <= 1e6
    assert ok.any()
    err = rowwise(params.cpu().numpy(), ref)[ok]
    assert err.max() <= 1e-6, (err.max(), conds[ok].max())


@pytest.mark.parametrize("case,orders", [("cfg2_d14", (0, 0)), ("odd_d5", (0, 0)), ("cond_orders", (2, 2)),
                                         ("cond_odd", (2, 1))])
@pytest.mark.parametrize("grid", ["shared", "per_row"])
def test_full_rows_are_bit_identical_to_unmasked(case, orders, grid):
    tok = make_tok(case, orders)
    B = 40
    T = tok.times.numel()
    t = None if grid == "shared" else jitter_times(tok, B, 21).cuda()
    x = trajs_for(tok, tok.times.expand(B, -1) if t is None else t.cpu(), 22).cuda()
    m = make_mask("drops", B, T, 23, full_every=3).cuda()
    full = m.all(1)
    tk0, pd0 = tok.encode(x, times=t)
    st0 = state_of(tok)
    tk1, pd1 = tok.encode(x, times=t, mask=m)
    st1 = state_of(tok)
    assert torch.equal(tk0[full], tk1[full]) and torch.equal(pd0["params"][full], pd1["params"][full])
    assert not torch.equal(pd0["params"][~full], pd1["params"][~full])
    if st0 is not None:
        for k, v in st0.items():
            if v is not None:
                assert torch.equal(v[full], st1[k][full]), k
    # normalised and gradients
    gen = torch.Generator(device="cuda").manual_seed(24)
    gn = torch.randn(B, tok.num_dof * tok.num_basis, device="cuda", generator=gen)
    res = []
    for mk in (None, m):
        xr = x.clone().requires_grad_(True)
        norm, pd = tok.encode_continuous(xr, times=t, mask=mk)
        loss = (norm * gn).sum() + (pd["params"] * gn).sum()
        if pd["init_vel"] is not None:
            loss = loss + (pd["init_vel"] * 0.3).sum()
        if pd["end_pos"] is not None:
            loss = loss + (pd["end_pos"] * 0.7).sum()
        loss.backward()
        res.append((norm.detach(), xr.grad))
    assert torch.equal(res[0][0][full], res[1][0][full])
    assert torch.equal(res[0][1][full], res[1][1][full])
    # mask of ones: the whole call equals mask=None
    ones = torch.ones(B, T, dtype=torch.bool, device="cuda")
    tk2, pd2 = tok.encode(x, times=t, mask=ones)
    assert torch.equal(tk2, tk0) and torch.equal(pd2["params"], pd0["params"])
    w_ones = tok.compute_weights(x, times=t, mask=ones.to(torch.int32))
    assert torch.equal(w_ones, pd0["params"])
    n_ones, _ = tok.encode_continuous(x, times=t, mask=ones)
    assert torch.equal(n_ones, res[0][0])


# ------------------------------------------------------------------ garbage isolation and degenerate rows
@pytest.mark.parametrize("case,orders", [("cfg2_d14", (0, 0)), ("cond_orders", (2, 2)), ("cond_odd", (2, 1))])
@pytest.mark.parametrize("grid", ["shared", "per_row"])
@pytest.mark.parametrize("fill", [float("nan"), float("inf"), float("-inf"), 1e30])
def test_padding_garbage_never_reaches_outputs(case, orders, grid, fill):
    tok = make_tok(case, orders)
    B = 24
    T = tok.times.numel()
    t = None if grid == "shared" else jitter_times(tok, B, 31).cuda()
    x = trajs_for(tok, tok.times.expand(B, -1) if t is None else t.cpu(), 32).cuda()
    m = make_mask("suffix", B, T, 33, full_every=5).cuda()
    x0 = torch.where(m.unsqueeze(2), x, torch.zeros_like(x))
    xg = torch.where(m.unsqueeze(2), x, torch.full_like(x, fill))
    tg = None if t is None else torch.where(m, t, torch.full_like(t, fill))
    gen = torch.Generator(device="cuda").manual_seed(34)
    gw = torch.randn(B, tok.num_dof * tok.num_basis, device="cuda", generator=gen)
    outs = []
    for xi, ti in ((x0, t), (xg, tg)):
        tk, pd = tok.encode(xi, times=ti, mask=m)
        xr = xi.clone().requires_grad_(True)
        norm, pc = tok.encode_continuous(xr, times=ti, mask=m)
        loss = (norm * gw).sum() + (pc["params"] * gw).sum()
        if pc["init_pos"] is not None:
            loss = loss + pc["init_pos"].sum() + pc["init_vel"].sum()
        if pc["end_pos"] is not None:
            loss = loss + pc["end_pos"].sum()
        loss.backward()
        st = [v for v in (tok._boundary or {}).values() if v is not None]
        outs.append([tk, pd["params"], norm.detach(), xr.grad, *st])
    for a, b in zip(*outs):
        assert torch.equal(a, b)
        assert torch.isfinite(b.float()).all()
    assert torch.equal(outs[1][3][~m], torch.zeros_like(outs[1][3][~m]))


@pytest.mark.parametrize("grid", ["shared", "per_row"])
def test_rows_without_samples(grid):
    tok = make_tok("cfg2_d14")
    B, T = 9, 50
    t = None if grid == "shared" else jitter_times(tok, B, 41).cuda()
    x = trajs_for(tok, tok.times.expand(B, -1) if t is None else t.cpu(), 42).cuda()
    m = make_mask("drops", B, T, 43).cuda()
    m[3] = False
    w = tok.compute_weights(x, times=t, mask=m)
    assert torch.equal(w[3], torch.zeros_like(w[3]))
    keep = torch.arange(B, device="cuda") != 3
    assert torch.equal(w[keep], tok.compute_weights(x[keep], times=None if t is None else t[keep], mask=m[keep]))
    # condition orders: rows with 0 or 1 valid samples leave every other row bit-identical
    tc = make_tok("cond_orders", (2, 2))
    m2 = m.clone()
    m2[5] = False
    m2[5, 7] = True
    w_all = tc.compute_weights(x, times=t, mask=m2)
    st_all = state_of(tc)
    keep = (torch.arange(B, device="cuda") != 3) & (torch.arange(B, device="cuda") != 5)
    w_sub = tc.compute_weights(x[keep], times=None if t is None else t[keep], mask=m2[keep])
    st_sub = state_of(tc)
    assert torch.equal(w_all[keep], w_sub)
    for k, v in st_sub.items():
        if v is not None:
            assert torch.equal(st_all[k][keep], v), k


# ------------------------------------------------------------------ tokens and bounds
@pytest.mark.parametrize("grid", ["shared", "per_row"])
def test_tokens_and_bounds(grid):
    tok = make_tok("odd_d5")
    B, T = 300, tok.times.numel()
    t = None if grid == "shared" else jitter_times(tok, B, 51)
    x = trajs_for(tok, tok.times.expand(B, -1) if t is None else t, 52)
    m = make_mask("suffix", B, T, 53, full_every=2)
    tok.update_weights_bounds(x, times=t, mask=m)
    w = tok.compute_weights(x, times=t, mask=m)
    assert torch.equal(tok.w_min.cuda(), w.min(0).values) and torch.equal(tok.w_max.cuda(), w.max(0).values)
    tok2 = make_tok("odd_d5")
    toks, pd = tok2.encode(x, update_bounds=True, times=t, mask=m)
    assert torch.equal(pd["params"], w)
    assert torch.equal(toks, tok2._quantize(w))
    toks3, _ = tok2.encode(x, times=t, mask=m)
    assert torch.equal(toks3, tok2._quantize(w))


# ------------------------------------------------------------------ gradients
def dense64(tok, y, times, mask, lo, hi, clamp, gn, gp, gb):
    """fp64 autograd chain on each row's valid samples: boundary state (first two / last two valid samples, dt from
    the first two), pinned subtraction, ridge solve on the fp32 basis rows, normalisation with the forward's clamp
    mask -> <normalised, gn> + <params, gp> + sum of gb-weighted boundary entries."""
    from beast_tokenizer_b200 import basis
    c = tok._plan().consts
    io, eo, nb, p = c.init_order, c.end_order, tok.num_basis, tok.degree_p
    nc = nb + io + eo
    B, T, D = y.shape
    kn = basis.knot_vector(nc, p).double()
    tau = float(torch.tensor(tok.duration, dtype=torch.float32))
    rows, extra = [], 0.0
    for b in range(B):
        mb = mask[b]
        tb = (tok.times if times is None else times[b])[mb]
        yb = y[b][mb]
        phi = basis.bspline_basis(tb, tok.duration, nc, p).double()
        free = phi[:, io:io + nb]
        G = free.T @ free + 1e-9 * torch.eye(nb, dtype=torch.float64)
        yj = yb[:, tok.joint_indices]
        inv_dt = float(torch.tensor(1.0) / (tb[1] - tb[0]))
        tgt = yj
        if io or eo:
            parts = []
            y0, y1, ym2, ym1 = yj[0], yj[1], yj[-2], yj[-1]
            if io:
                parts.append(torch.zeros_like(y0))
                if io == 2:
                    parts.append((y1 - y0) * inv_dt * tau * float(kn[1 + p] - kn[1]) / p)
                extra = extra + (y0 * gb[0]).sum() + ((y1 - y0) * inv_dt * gb[1]).sum()
            if eo:
                end_pos = ym1 - y0 if io else ym1
                if eo == 2:
                    parts.append(end_pos - (ym1 - ym2) * inv_dt * tau * float(kn[nc - 1 + p] - kn[nc - 1]) / p)
                parts.append(end_pos)
                extra = extra + (ym1 * gb[2]).sum() + ((ym1 - ym2) * inv_dt * gb[3]).sum()
            bc = torch.stack(parts, dim=-1)
            pin = torch.cat([phi[:, :io], phi[:, io + nb:]], dim=1)
            tgt = yj - pin @ bc.T - (y0 if io else 0.0)
        wj = torch.linalg.solve(G, free.T @ tgt).T
        ws = [wj]
        if tok.gripper_indices:
            phig = basis.bspline_basis(tb, tok.duration, nb, 0).double()
            Gg = phig.T @ phig + 1e-9 * torch.eye(nb, dtype=torch.float64)
            ws.append(torch.linalg.solve(Gg, phig.T @ yb[:, tok.gripper_indices]).T)
        rows.append(torch.cat(ws, 0).reshape(-1))
    w = torch.stack(rows)
    scale = torch.clamp(hi - lo, min=1e-8)
    norm = ((w - lo) / scale * 2 - 1) * clamp
    norm_td = norm.view(B, D, nb).transpose(1, 2).reshape(B, -1)
    return (norm_td * gn).sum() + (w * gp).sum() + extra


@pytest.mark.parametrize("case,orders", ALL_CASES, ids=CASE_IDS)
@pytest.mark.parametrize("grid", ["shared", "per_row"])
@pytest.mark.parametrize("loss", ["normalised", "params", "both", "boundary"])
def test_gradients_against_fp64_autograd(case, orders, grid, loss):
    tok = make_tok(case, orders)
    B = 10
    T = tok.times.numel()
    t = None if grid == "shared" else jitter_times(tok, B, 61)
    x = trajs_for(tok, tok.times.expand(B, -1) if t is None else t, 62)
    m = make_mask("drops", B, T, 63, full_every=4)
    xr = x.cuda().requires_grad_(True)
    norm, pd = tok.encode_continuous(xr, times=t, mask=m.cuda())
    gen = torch.Generator().manual_seed(64)
    gn, gp = torch.randn(norm.shape, generator=gen), torch.randn(norm.shape, generator=gen)
    nj = len(tok.joint_indices)
    gb = torch.randn(4, nj, generator=gen)
    if loss == "normalised":
        gp = torch.zeros_like(gp)
    if loss == "params":
        gn = torch.zeros_like(gn)
    if loss != "boundary":
        gb = torch.zeros_like(gb)
    elif not tok._has_conditions:
        pytest.skip("no boundary entries without condition orders")
    total = (norm * gn.cuda()).sum() + (pd["params"] * gp.cuda()).sum()
    if pd["init_pos"] is not None:
        total = total + (pd["init_pos"] * gb[0].cuda()).sum() + (pd["init_vel"] * gb[1].cuda()).sum()
    if pd["end_pos"] is not None:
        total = total + (pd["end_pos"] * gb[2].cuda()).sum() + (pd["end_vel"] * gb[3].cuda()).sum()
    total.backward()
    g = xr.grad.cpu()
    assert torch.equal(g[~m], torch.zeros_like(g[~m]))
    lo, hi = tok.w_min.double().cpu(), tok.w_max.double().cpu()
    w32 = pd["params"].detach().cpu()
    clamp = ((w32 >= tok.w_min.cpu()) & (w32 <= tok.w_max.cpu())).double()
    y64 = x.double().requires_grad_(True)
    dense64(tok, y64, t, m, lo, hi, clamp, gn.double(), gp.double(), gb.double()).backward()
    assert rel_err(g.numpy(), y64.grad.numpy()) <= 1e-5
    if loss == "params":
        # adjoint identity: the masked fit is linear in y (boundary state included)
        lhs = float((pd["params"].detach().double().cpu() * gp.double()).sum())
        rhs = float((g.double() * x.double()).sum())
        scale = float(pd["params"].detach().double().norm() * gp.double().norm())
        assert abs(lhs - rhs) <= 1e-5 * scale


# ------------------------------------------------------------------ invariance
def _abi_masked(tok, x, t, stride, m, partial, out, bc=None, bias=None):
    plan = tok._plan()
    vp = lambda z: None if z is None else ctypes.c_void_p(z.data_ptr())
    return plan._lib.beast_fit_masked_f32(plan.handle, vp(x), x.shape[0], m.shape[1], vp(t), stride, vp(m), partial,
                                          vp(bc), vp(bias), vp(out), None)


def test_invariance_batch_sizes_and_positions():
    tok = make_tok("cfg2_d14")
    T = 50
    B = 65537
    for grid in ("shared", "per_row"):
        t = None if grid == "shared" else jitter_times(tok, B, 71).cuda()
        x = trajs_for(tok, tok.times.expand(B, -1) if t is None else t.cpu(), 72).cuda()
        m = make_mask("suffix", B, T, 73, full_every=3).cuda()
        w = tok.compute_weights(x, times=t, mask=m)
        assert torch.equal(w, tok.compute_weights(x, times=t, mask=m))
        for n in (1, 7, 33):
            for sel in (torch.arange(n), torch.arange(B - n, B), torch.randperm(B, generator=torch.Generator()
                                                                                 .manual_seed(n))[:n]):
                sel = sel.cuda()
                assert torch.equal(w[sel], tok.compute_weights(x[sel], times=None if t is None else t[sel],
                                                               mask=m[sel])), (grid, n)
        rev = torch.arange(B - 1, -1, -1, device="cuda")
        assert torch.equal(w[rev], tok.compute_weights(x[rev], times=None if t is None else t[rev], mask=m[rev]))


def test_long_rows_straddling_chunks():
    tok = make_tok("cfg2_d14")
    B, T = 16, 1987
    t = jitter_times(tok, B, 81, T=T)
    x = trajs_for(tok, t, 82).cuda()
    m = torch.ones(B, T, dtype=torch.bool)
    for b in range(B):                             # runs of drops that cross the 32-sample chunk boundaries
        for a in range(17 + b, T, 97 + 3 * b):
            m[b, a:a + 5 + b] = False
    m[0] = True
    m[1, 1960:] = False
    w = tok.compute_weights(x, times=t, mask=m)
    for b in range(B):
        xc, tc = compact(tok, x, t, m, b)
        assert torch.equal(w[b:b + 1], tok.compute_weights(xc, times=tc)), b
    ref, conds = ridge64(tok, x.cpu(), t, m)
    ok = conds <= 1e6
    assert ok.any() and rowwise(w.cpu().numpy(), ref)[ok].max() <= 1e-6


def test_shipped_shape():
    tok = make_tok("cli_default")
    B, T = 257, tok.times.numel()
    x = trajs_for(tok, tok.times.expand(B, -1), 91).cuda()
    for kind in ("suffix", "prefix", "drops"):
        m = make_mask(kind, B, T, 92, full_every=2).cuda()
        tk, pd = tok.encode(x, mask=m)
        full = m.all(1)
        tk0, pd0 = tok.encode(x)
        assert torch.equal(pd["params"][full], pd0["params"][full]) and torch.equal(tk[full], tk0[full])
        for b in (1, 3, 5, 255):
            if bool(m[b].all()):
                continue
            xc, tc = compact(tok, x, None, m, b)
            assert torch.equal(pd["params"][b:b + 1], tok.compute_weights(xc, times=tc)), (kind, b)


def test_unaligned_views_guard_bands_and_partial_only():
    tok = make_tok("odd_d5")
    B, n = 333, tok.num_dof * tok.num_basis
    T = tok.times.numel()
    t = jitter_times(tok, B, 101).cuda()
    x = trajs_for(tok, t.cpu(), 102).cuda()
    m = make_mask("drops", B, T, 103, full_every=3).cuda()
    mb = m.view(torch.uint8)
    ref = torch.empty(B, n, device="cuda")
    assert _abi_masked(tok, x, t, T, mb, 0, ref) == 0
    xb = torch.empty(x.numel() + 1, device="cuda"); xb[1:] = x.reshape(-1)
    tb = torch.empty(t.numel() + 1, device="cuda"); tb[1:] = t.reshape(-1)
    mbb = torch.empty(m.numel() + 3, device="cuda", dtype=torch.uint8); mbb[3:] = mb.reshape(-1)
    ob = torch.full((B * n + 65,), 12345.0, device="cuda")
    xv, tv, mv, ov = xb[1:].view(x.shape), tb[1:].view(t.shape), mbb[3:].view(m.shape), ob[1:1 + B * n].view(B, n)
    assert _abi_masked(tok, xv, tv, T, mv, 0, ov) == 0
    torch.cuda.synchronize()
    assert torch.equal(ov, ref)
    assert ob[0].item() == 12345.0 and (ob[1 + B * n:] == 12345.0).all()
    assert torch.equal(tok.compute_weights(xv, times=tv, mask=mv.view(torch.bool)), ref)
    # partial_only: full rows' output bytes stay untouched, partial rows equal the partial_only=0 result
    ob.fill_(12345.0)
    assert _abi_masked(tok, xv, tv, T, mv, 1, ov) == 0
    full = m.all(1)
    assert (ov[full] == 12345.0).all() and torch.equal(ov[~full], ref[~full])
    # backward, partial_only: untouched full rows in every output
    gp = torch.randn(B, n, device="cuda")
    g_ref = torch.empty(B, T, tok.num_dof, device="cuda")
    plan = tok._plan()
    vp = lambda z: None if z is None else ctypes.c_void_p(z.data_ptr())
    bwd = plan._lib.beast_fit_masked_backward_f32
    assert bwd(plan.handle, B, T, vp(t), T, vp(mb), 0, None, vp(gp), None, None, None, vp(g_ref), None, None,
               None) == 0
    g = torch.full((B, T, tok.num_dof), 777.0, device="cuda")
    assert bwd(plan.handle, B, T, vp(t), T, vp(mb), 1, None, vp(gp), None, None, None, vp(g), None, None, None) == 0
    torch.cuda.synchronize()
    assert (g[full] == 777.0).all() and torch.equal(g[~full], g_ref[~full])
    assert torch.equal(g_ref[~m], torch.zeros_like(g_ref[~m]))
    # stride 0: one grid for every row equals the same grid repeated per row
    grid = tok._plan().device_times()
    xs = trajs_for(tok, tok.times.expand(B, -1), 104).cuda()
    o0, o1 = torch.empty(B, n, device="cuda"), torch.empty(B, n, device="cuda")
    assert _abi_masked(tok, xs, grid, 0, mb, 0, o0) == 0
    assert _abi_masked(tok, xs, grid.expand(B, -1).contiguous(), T, mb, 0, o1) == 0
    torch.cuda.synchronize()
    assert torch.equal(o0, o1)


# ------------------------------------------------------------------ graph capture and overlap
@pytest.mark.parametrize("grid", ["shared", "per_row"])
def test_graph_capture(grid):
    tok = make_tok("cond_orders", (2, 2))
    B, T = 64, 50
    t = None if grid == "shared" else jitter_times(tok, B, 111).cuda()
    x = trajs_for(tok, tok.times.expand(B, -1) if t is None else t.cpu(), 112).cuda()
    m = make_mask("suffix", B, T, 113, full_every=3).cuda()
    r = torch.randn(B, tok.num_dof * tok.num_basis, device="cuda",
                    generator=torch.Generator(device="cuda").manual_seed(114))

    def step(xs):
        tk, pd = tok.encode(xs.detach(), mask=m, times=t)
        norm, pc = tok.encode_continuous(xs, mask=m, times=t)
        ((norm * r).sum() + pc["end_vel"].sum() + pc["init_vel"].sum()).backward()
        return tk, pd["params"], norm.detach()

    xs = x.clone().requires_grad_(True)
    eager = step(xs)
    g_eager = xs.grad.clone()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            xs.grad = None
            step(xs)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    xs.grad = None
    with torch.cuda.graph(graph):
        outs = step(xs)
    graph.replay()
    torch.cuda.synchronize()
    for a, b in zip(eager, outs):
        assert torch.equal(a, b)
    assert torch.equal(xs.grad, g_eager)


def test_no_overlap_across_the_masked_kernel():
    """A captured K1 -> masked fit -> K3 sequence: the K3 launch must not overlap across the masked launch (it is an
    ordinary launch); outputs equal those with every overlap forced off.  Without the masked launch, K3 overlaps K1."""
    from beast_tokenizer_b200 import BEASTBsplineTokenizer, _lib
    from beast_tokenizer_b200.synth import synth
    tok = BEASTBsplineTokenizer(num_dof=14, num_basis=10, seq_len=50, vocab_size=256, gripper_zero_order=True,
                                gripper_indices=[6, 13], device="cuda")
    B, T = 4096, 50
    dev = torch.device("cuda", torch.cuda.current_device())
    x = synth(B, T, 14, seed=5, device=dev)
    tok.update_weights_bounds(x)
    plan, lib, p = tok._plan(), tok._plan()._lib, _lib.ptr
    lo, hi = tok._bounds(dev)
    m = make_mask("suffix", B, T, 121, full_every=2).cuda().view(torch.uint8)
    grid = plan.device_times()
    toks_b = tok.encode(synth(B, T, 14, seed=6, device=dev))[0]
    params = torch.zeros(B, 140, device="cuda")
    out = torch.zeros(B, T, 14, device="cuda")

    toks_a = torch.zeros(B, 140, device="cuda", dtype=torch.int64)

    def ops(masked):
        _lib.check(lib.beast_encode_f32(plan.handle, p(x), B, p(lo), p(hi), 0, p(params), p(toks_a),
                                        _lib.stream_ptr(dev)), "encode")
        if masked:
            _lib.check(lib.beast_fit_masked_f32(plan.handle, p(x), B, T, p(grid), 0, p(m), 1, None, None, p(params),
                                                _lib.stream_ptr(dev)), "masked")
        _lib.check(lib.beast_decode_f32(plan.handle, p(toks_b), B, p(lo), p(hi), 0, None, p(out),
                                        _lib.stream_ptr(dev)), "decode")

    def captured(masked):
        params.zero_(); out.zero_()
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        n0 = _lib.overlap_count()
        with torch.cuda.graph(g):
            ops(masked)
        n = _lib.overlap_count() - n0
        params.zero_(); out.zero_()
        torch.cuda.synchronize()
        g.replay()
        torch.cuda.synchronize()
        return n, params.clone(), out.clone()

    ops(True)
    torch.cuda.synchronize()
    eager = (params.clone(), out.clone())
    n_plain, _, _ = captured(False)
    assert n_plain == 1                                  # the K1 / K3 pair does overlap without the masked launch
    n_masked, pm, om = captured(True)
    assert n_masked == 0
    prev = lib.beast_debug_force_wait(1)
    try:
        n_wait, pw, ow = captured(True)
    finally:
        lib.beast_debug_force_wait(prev)
    assert n_wait == 0
    for a, b, c in ((pm, pw, eager[0]), (om, ow, eager[1])):
        assert torch.equal(a, b) and torch.equal(a, c)


# ------------------------------------------------------------------ BPE, launches, errors
def test_bpe_passes_mask_through():
    from beast_tokenizer_b200 import BEASTBsplineBPETokenizer
    tok = make_tok("cfg2_d14")
    B, T = 64, 50
    x = trajs_for(tok, tok.times.expand(B, -1), 131)
    m = make_mask("suffix", B, T, 132, full_every=3)
    btok = BEASTBsplineBPETokenizer.from_beast(tok, bpe_vocab_size=300)
    btok.fit_from_trajectories([{"actions": trajs_for(tok, tok.times.expand(B, -1), 133)}], show_progress=False)
    ref, _ = tok.encode(x, mask=m)
    ids, _ = btok.encode(x, mask=m)
    assert ids == btok._discrete_to_bpe(ref)
    mp, _ = btok.encode_to_mp_tokens(x, mask=m)
    assert torch.equal(mp, ref)
    flat, off, _ = btok.encode_csr(x, mask=m)
    flat, off = flat.cpu().tolist(), off.cpu().tolist()
    assert [flat[off[i]:off[i + 1]] for i in range(len(ids))] == [list(r) for r in ids]


@pytest.mark.parametrize("case,orders", [("cfg2_d14", (0, 0)), ("cond_orders", (2, 2))])
def test_mask_none_keeps_launch_counts(case, orders):
    from beast_tokenizer_b200 import _lib
    tok = make_tok(case, orders)
    x = trajs_for(tok, tok.times.expand(50, -1), 141).cuda()
    t = jitter_times(tok, 50, 142).cuda()
    counts = []
    for kw in ({}, {"mask": None}):
        n0 = _lib.launch_count()
        tok.encode(x, **kw)
        tok.compute_weights(x, **kw)
        tok.encode_continuous(x, **kw)
        tok.encode(x, times=t, **kw)
        counts.append(_lib.launch_count() - n0)
    assert counts[0] == counts[1]
    m = torch.ones(50, 50, dtype=torch.bool, device="cuda")
    n0 = _lib.launch_count()
    tok.compute_weights(x)
    n_k1 = _lib.launch_count() - n0
    n0 = _lib.launch_count()
    tok.encode(x, mask=m)
    assert _lib.launch_count() - n0 == n_k1 + 2         # K1, masked (partial only), quantize


def test_python_errors():
    tok = make_tok("cfg2_d14")
    x = torch.zeros(4, 50, 14)
    with pytest.raises(AssertionError):
        tok.encode(x, mask=torch.ones(4, 49, dtype=torch.bool))
    with pytest.raises(AssertionError):
        tok.encode(x, mask=torch.ones(3, 50, dtype=torch.bool))
    with pytest.raises(AssertionError):
        tok.encode(x, mask=torch.ones(50, dtype=torch.bool))
    with pytest.raises(AssertionError):
        tok.encode(x, times=torch.zeros(4, 60), mask=torch.ones(4, 50, dtype=torch.bool))
    with pytest.raises(TypeError):
        tok.encode(x, mask=torch.ones(4, 50))
    with pytest.raises(TypeError):
        tok.compute_weights(x, mask=torch.ones(4, 50, dtype=torch.float16))
    w = tok.compute_weights(x, mask=torch.ones(4, 50, dtype=torch.int64))
    assert w.shape == (4, 140)


def test_c_abi_errors():
    tok = make_tok("cond_orders", (2, 2))
    plan = tok._plan()
    lib = plan._lib
    vp = lambda t: ctypes.c_void_p(t.data_ptr())
    x = torch.zeros(2, 50, 14, device="cuda")
    t = torch.zeros(2, 50, device="cuda")
    m = torch.ones(2, 50, device="cuda", dtype=torch.uint8)
    out = torch.zeros(2, 140, device="cuda")
    bc = torch.zeros(2, 12, 4, device="cuda")
    f = lib.beast_fit_masked_f32
    assert f(None, vp(x), 2, 50, vp(t), 50, vp(m), 0, vp(bc), None, vp(out), None) == -1
    assert f(plan.handle, vp(x), 2, 50, vp(t), 50, None, 0, vp(bc), None, vp(out), None) == -1
    assert f(plan.handle, vp(x), 2, 50, vp(t), 50, vp(m), 0, None, None, vp(out), None) == -1
    assert f(plan.handle, None, 2, 50, vp(t), 50, vp(m), 0, vp(bc), None, vp(out), None) == -1
    assert f(plan.handle, vp(x), 2, 50, None, 50, vp(m), 0, vp(bc), None, vp(out), None) == -1
    assert f(plan.handle, vp(x), 2, 50, vp(t), 49, vp(m), 0, vp(bc), None, vp(out), None) == -2
    assert f(plan.handle, vp(x), 2, 50, vp(t), 1, vp(m), 0, vp(bc), None, vp(out), None) == -2
    assert f(plan.handle, vp(x), -1, 50, vp(t), 50, vp(m), 0, vp(bc), None, vp(out), None) == -2
    assert f(plan.handle, vp(x), 2, 1, vp(t), 1, vp(m), 0, vp(bc), None, vp(out), None) == -2
    assert f(plan.handle, None, 0, 50, None, 50, None, 0, None, None, None, None) == 0
    mis = ctypes.c_void_p(out.data_ptr() + 2)
    assert f(plan.handle, vp(x), 2, 50, vp(t), 50, vp(m), 0, vp(bc), None, mis, None) == -3
    misx = ctypes.c_void_p(x.data_ptr() + 1)
    assert f(plan.handle, misx, 2, 50, vp(t), 0, vp(m), 1, vp(bc), None, vp(out), None) == -3
    g = torch.zeros(2, 50, 14, device="cuda")
    gp = torch.zeros(2, 140, device="cuda")
    bwd = lib.beast_fit_masked_backward_f32
    assert bwd(plan.handle, 2, 50, vp(t), 50, vp(m), 0, None, None, None, None, None, vp(g), vp(bc), None, None) == -1
    assert bwd(plan.handle, 2, 50, vp(t), 50, None, 0, None, vp(gp), None, None, None, vp(g), vp(bc), None,
               None) == -1
    assert bwd(plan.handle, 2, 50, vp(t), 50, vp(m), 0, vp(gp), None, None, None, None, vp(g), vp(bc), None,
               None) == -1
    assert bwd(plan.handle, 2, 50, vp(t), 50, vp(m), 0, None, vp(gp), None, None, None, vp(g), None, None, None) == -1
    assert bwd(plan.handle, 2, 50, vp(t), 7, vp(m), 0, None, vp(gp), None, None, None, vp(g), vp(bc), None,
               None) == -2
    assert bwd(plan.handle, 2, 1, vp(t), 1, vp(m), 0, None, vp(gp), None, None, None, vp(g), vp(bc), None,
               None) == -2
    assert bwd(plan.handle, 2, 50, vp(t), 50, vp(m), 0, None, mis, None, None, None, vp(g), vp(bc), None,
               None) == -3
    assert bwd(plan.handle, 0, 50, None, 50, None, 0, None, vp(gp), None, None, None, None, None, None, None) == 0
    assert bwd(plan.handle, 2, 50, vp(t), 0, vp(m), 1, None, vp(gp), None, None, None, vp(g), vp(bc), None,
               None) == 0
    torch.cuda.synchronize()
    from beast_tokenizer_b200 import BEASTBsplineTokenizer
    big = BEASTBsplineTokenizer(num_dof=2, num_basis=316, seq_len=400, degree_p=4, device="cuda")
    bp = big._plan()
    x2, t2, o2 = (torch.zeros(1, 400, 2, device="cuda"), torch.zeros(1, 400, device="cuda"),
                  torch.zeros(1, 632, device="cuda"))
    m2 = torch.ones(1, 400, device="cuda", dtype=torch.uint8)
    assert bp._lib.beast_fit_masked_f32(bp.handle, vp(x2), 1, 400, vp(t2), 400, vp(m2), 0, None, None, vp(o2),
                                        None) == -4
    assert bp._lib.beast_fit_masked_backward_f32(bp.handle, 1, 400, vp(t2), 400, vp(m2), 0, None, vp(o2), None, None,
                                                 None, vp(x2), None, None, None) == -4
