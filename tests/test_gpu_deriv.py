"""Derivatives of the decoded spline (reconstruct_traj_derivatives): order 0 against reconstruct_traj bit for bit,
orders 1 / 2 against scipy splines of the same coefficients in fp64, boundary velocities against the live reference's
numbers, and the tiled kernel against the generic one bit for bit.  Run on the B200 box:  pytest -m gpu."""
import math

import numpy as np
import pytest
import torch
from scipy.interpolate import BSpline

from conftest import GOLDEN_CASES, load_golden, rel_err

pytestmark = pytest.mark.gpu

TOL_VEL, TOL_ACC = 1e-5, 5e-5
TAU32 = float(np.float32(2 * math.pi))
COND_CFG = dict(num_dof=14, num_basis=10, seq_len=50, vocab_size=256, degree_p=4,
                gripper_zero_order=True, gripper_indices=[6, 13], llm_vocab_size=None)
COND_ODD_CFG = dict(num_dof=5, num_basis=8, seq_len=33, vocab_size=1000, degree_p=3,
                    gripper_zero_order=True, gripper_indices=[0])
COND_CASES = [("cond_orders", o) for o in [(2, 0), (0, 2), (2, 2), (1, 1)]] + [("cond_odd", (2, 1))]
REPORT = {}


def make_tok(cfg, g=None):
    from beast_tokenizer_b200 import BEASTBsplineTokenizer
    tok = BEASTBsplineTokenizer(device="cuda", **cfg)
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
    k = f"o{io}{eo}_"
    tok.w_min.copy_(torch.from_numpy(g[k + "w_min"]))
    tok.w_max.copy_(torch.from_numpy(g[k + "w_max"]))
    tok.encode(torch.from_numpy(g["trajs"]))                      # boundary state of this fit
    return tok, g, k


def shared_grid(tq, tok):
    """Tq samples including 0, tau, an interior knot and points outside [0, tau]."""
    from beast_tokenizer_b200.basis import knot_vector
    kn = knot_vector(tok.num_basis + tok.init_cond_order + tok.end_cond_order, tok.degree_p)
    special = [TAU32, 0.0, -0.25, TAU32 + 0.25, float(kn[tok.degree_p + 1]) * TAU32]
    t = torch.linspace(-0.5, TAU32 + 0.5, tq)
    n = min(tq, len(special))
    t[:n] = torch.tensor(special[:n])
    return t.to(torch.float32)


def oracle(tok, coeff, times, init_p=None):
    """fp64 scipy splines of the fp32 coefficients coeff [B, D*nb] '(d t)' at times [B, Tq] (or [Tq]):
    {order: [B, Tq, D]} for orders 1 and 2 (init_p substitution, pinned points of the last fit)."""
    from beast_tokenizer_b200.basis import knot_vector
    coeff = np.asarray(coeff, np.float64)
    B, D, nb, p = coeff.shape[0], tok.num_dof, tok.num_basis, tok.degree_p
    times = np.broadcast_to(np.asarray(times, np.float32), (B, np.asarray(times).shape[-1]))
    io, eo = (tok.init_cond_order, tok.end_cond_order) if tok._has_conditions else (0, 0)
    kn = knot_vector(nb + io + eo, p).double().numpy()
    bc = tok._boundary["bc"].double().cpu().numpy() if (io or eo) else None
    nj = len(tok.joint_indices)
    out = {o: np.zeros((B, times.shape[1], D)) for o in (1, 2)}
    for b in range(B):
        raw = times[b] / np.float32(TAU32)
        u = np.clip(raw.astype(np.float64), 0.0, 1.0)
        inside = (raw >= 0) & (raw <= 1)
        for s in range(nj):
            dof = tok.joint_indices[s]
            c = coeff[b, s * nb:(s + 1) * nb].copy()
            if init_p is not None:
                c[0] = init_p[b, dof]
            if bc is not None:
                c = np.concatenate([bc[b, s, :io], c, bc[b, s, io:]])
            spl = BSpline(kn, c, p)
            for o in (1, 2):
                if o <= p:
                    out[o][b, inside, dof] = spl.derivative(o)(u[inside]) / TAU32 ** o
    return out


def check_vs_oracle(tok, outs, coeff, times, init_p, tag):
    ref = oracle(tok, coeff, times, init_p)
    for o, tol in ((1, TOL_VEL), (2, TOL_ACC)):
        got = outs[o].cpu().numpy()
        if np.abs(ref[o]).max() == 0:
            assert not np.any(got), (tag, o)
            continue
        err = rel_err(got, ref[o])
        REPORT[(tag, o)] = err
        assert err <= tol, (tag, o, err)
    t = np.broadcast_to(np.asarray(times, np.float32), (coeff.shape[0], np.asarray(times).shape[-1]))
    raw = t / np.float32(TAU32)
    outside = (raw < 0) | (raw > 1)
    for o in (1, 2):
        got = outs[o].cpu().numpy()
        assert not np.any(got[outside]), (tag, o, "outside [0, tau]")
        assert not np.any(got[..., tok.gripper_indices]), (tag, o, "gripper slots")


def as_dict(res, orders=(0, 1, 2)):
    return dict(zip(orders, res))


# ---------------------------------------------------------------- 1, 2, 3: golden geometries
def test_order0_own_times_equals_reconstruct_traj(golden_case):
    name, cfg, g = golden_case
    tok = make_tok(cfg, g)
    toks = torch.from_numpy(g["tokens_fit"])                      # cfg2: LLM-offset tokens
    init_p = torch.from_numpy(g["init_p"])
    for kw in ({}, {"init_p": init_p}):
        pos, vel, acc = tok.reconstruct_traj_derivatives(toks, **kw)
        assert pos.dtype == torch.float32 and pos.shape == (toks.shape[0], cfg["seq_len"], cfg["num_dof"])
        assert torch.equal(pos, tok.reconstruct_traj(toks, **kw)), (name, kw.keys())
        (only,) = tok.reconstruct_traj_derivatives(toks, orders=(0,), **kw)
        assert torch.equal(only, pos)
        coeff = tok.decode(toks).cpu().numpy()
        check_vs_oracle(tok, {1: vel, 2: acc}, coeff, tok.times.numpy(),
                        init_p.numpy() if kw else None, f"{name}/own{'/init_p' if kw else ''}")


@pytest.mark.parametrize("tq", [1, 7, 200, 1000])
def test_shared_grid_equals_reconstruct_traj_and_oracle(golden_case, tq):
    name, cfg, g = golden_case
    tok = make_tok(cfg, g)
    toks = torch.from_numpy(g["tokens_fit"])
    B = toks.shape[0]
    grid = shared_grid(tq, tok)
    init_p = torch.from_numpy(g["init_p"])
    for kw in ({}, {"init_p": init_p}):
        res = as_dict(tok.reconstruct_traj_derivatives(toks, times=grid, **kw))
        assert res[0].shape == (B, tq, cfg["num_dof"])
        ref0 = tok.reconstruct_traj(toks, times=grid.expand(B, -1).contiguous(), **kw)
        assert torch.equal(res[0], ref0), (name, tq)
        check_vs_oracle(tok, res, tok.decode(toks).cpu().numpy(), grid.numpy(), init_p.numpy() if kw else None,
                        f"{name}/grid{tq}{'/init_p' if kw else ''}")
        if not kw:
            plain = res
    # orders in any order, any subset
    v, p = tok.reconstruct_traj_derivatives(toks, times=grid, orders=(1, 0))
    assert torch.equal(p, plain[0]) and torch.equal(v, plain[1])


def test_per_row_times_equal_reconstruct_traj_and_oracle(golden_case):
    name, cfg, g = golden_case
    tok = make_tok(cfg, g)
    toks = torch.from_numpy(g["tokens_fit"])
    B = toks.shape[0]
    rng = np.random.default_rng(5)
    tt = torch.from_numpy(rng.uniform(-0.3, TAU32 + 0.3, size=(B, 45)).astype(np.float32))
    tt[:, 0], tt[:, 1] = 0.0, TAU32
    cases = [tt] + ([torch.from_numpy(g["custom_times"])] if "custom_times" in g else [])
    for times in cases:
        res = as_dict(tok.reconstruct_traj_derivatives(toks, times=times))
        assert torch.equal(res[0], tok.reconstruct_traj(toks, times=times))
        check_vs_oracle(tok, res, tok.decode(toks).cpu().numpy(), times.numpy(), None, f"{name}/rows")


# ---------------------------------------------------------------- condition orders, 4: boundary velocities
@pytest.mark.parametrize("case,orders", COND_CASES)
def test_condition_orders(case, orders):
    tok, g, k = cond_tok(case, orders)
    io, eo = orders
    toks = torch.from_numpy(g[k + "tokens"])
    B = toks.shape[0]
    init_p = torch.from_numpy(g["init_p"])
    for kw in ({}, {"init_p": init_p}):
        pos, vel, acc = tok.reconstruct_traj_derivatives(toks, **kw)
        assert torch.equal(pos, tok.reconstruct_traj(toks, **kw))
        check_vs_oracle(tok, {1: vel, 2: acc}, tok.decode(toks).cpu().numpy(), tok.times.numpy(),
                        init_p.numpy() if kw else None, f"{case}{orders}/own")
    grid = shared_grid(200, tok)
    res = as_dict(tok.reconstruct_traj_derivatives(toks, times=grid))
    assert torch.equal(res[0], tok.reconstruct_traj(toks, times=grid.expand(B, -1).contiguous()))
    check_vs_oracle(tok, res, tok.decode(toks).cpu().numpy(), grid.numpy(), None, f"{case}{orders}/grid")
    tt = torch.from_numpy(g[k + "custom_times"])
    res = as_dict(tok.reconstruct_traj_derivatives(toks, times=tt))
    assert torch.equal(res[0], tok.reconstruct_traj(toks, times=tt))
    check_vs_oracle(tok, res, tok.decode(toks).cpu().numpy(), tt.numpy(), None, f"{case}{orders}/rows")
    # the pinned c0, c1 (c_{n-2}, c_{n-1}) fix the boundary slope to the fit's finite-difference velocity
    (vel,) = tok.reconstruct_traj_derivatives(toks, orders=(1,))
    ji = tok.joint_indices
    if io == 2:
        err = rel_err(vel[:, 0, ji].cpu().numpy(), g[k + "init_vel"])
        REPORT[(f"{case}{orders}", "init_vel")] = err
        assert err <= 1e-5
    if eo == 2:
        err = rel_err(vel[:, -1, ji].cpu().numpy(), g[k + "end_vel"])
        REPORT[(f"{case}{orders}", "end_vel")] = err
        assert err <= 1e-5


# ---------------------------------------------------------------- 5: tiled kernel == generic kernel
def _grid_call(tok, toks, grid, outs, init_p=None):
    from beast_tokenizer_b200 import _lib
    plan = tok._plan()
    gr = tok._grid(plan, grid, 2)
    lo, hi = tok._bounds(plan.device)
    off = tok._llm_vocab_offset() if tok.llm_vocab_size is not None else 0
    _lib.check(plan._lib.beast_decode_grid_f32(plan.handle, gr.handle, _lib.ptr(toks), None, toks.shape[0], _lib.ptr(lo),
                                               _lib.ptr(hi), off, _lib.ptr(init_p), None, None,
                                               *[_lib.ptr(o) for o in outs], _lib.stream_ptr(plan.device)),
               "beast_decode_grid_f32")


@pytest.mark.parametrize("name", ["cfg2_d14", "odd_d5", "cli_default"])
def test_tiled_equals_generic(name):
    from beast_tokenizer_b200 import _lib
    from beast_tokenizer_b200.synth import synth
    cfg = GOLDEN_CASES[name]
    g = load_golden(name)
    tok = make_tok(cfg, g)
    lib = _lib.load()
    T, D = cfg["seq_len"], cfg["num_dof"]
    sizes = (1, 3, 4097, 65536 + 5) if name == "cfg2_d14" else (1, 3, 4097)
    for B in sizes:
        x = synth(B, T, D, seed=B).cuda()
        toks, _ = tok.encode(x)
        ip = x[:, 0, :].contiguous()
        for grid in (tok.times, shared_grid(200, tok)):
            tq = grid.numel()
            n = B * tq * D
            res = {}
            for slow in (0, 1):
                prev = lib.beast_debug_disable_fast(slow)
                try:
                    full = tok.reconstruct_traj_derivatives(toks, times=grid, init_p=ip)
                    sub = tok.reconstruct_traj_derivatives(toks, times=grid, orders=(2, 0), init_p=ip)
                    # misaligned output views (4-byte aligned, not 16), one order left NULL
                    buf = [torch.full((n + 3,), float("nan"), device="cuda") for _ in range(2)]
                    views = [buf[0][1:n + 1], None, buf[1][3:n + 3]]
                    _grid_call(tok, toks, grid, views, ip)
                    torch.cuda.synchronize()
                    res[slow] = list(full) + list(sub) + [views[0].clone(), views[2].clone()]
                finally:
                    lib.beast_debug_disable_fast(prev)
            for i, (a, b) in enumerate(zip(res[0], res[1])):
                assert torch.equal(a, b), (name, B, tq, i, float((a.double() - b.double()).abs().max()))
            pos, acc = res[0][0], res[0][2]
            assert torch.equal(res[0][3], acc) and torch.equal(res[0][4], pos)
            assert torch.equal(res[0][5].view(B, tq, D), pos) and torch.equal(res[0][6].view(B, tq, D), acc)


# ---------------------------------------------------------------- 6: BPE subclass and continuous coefficients
def test_bpe_subclass_and_continuous():
    from beast_tokenizer_b200 import BEASTBsplineBPETokenizer, BEASTBsplineTokenizer
    from beast_tokenizer_b200.synth import synth
    cfg = dict(GOLDEN_CASES["cfg2_d14"], llm_vocab_size=None)
    tok = BEASTBsplineTokenizer(device="cuda", **cfg)
    x = synth(16 * 12 + 5, 50, 14, seed=9)
    tok.update_weights_bounds(x)
    btok = BEASTBsplineBPETokenizer.from_beast(tok, bpe_vocab_size=400)
    btok.fit_from_trajectories([{"actions": x}], show_progress=False)
    ids, _ = btok.encode(x)
    mp = btok.bpe_to_mp_tokens(ids)
    grid = shared_grid(120, tok)
    for kw in ({}, {"times": grid}, {"times": grid.expand(mp.shape[0], -1) * 0.5}):
        got = btok.reconstruct_traj_derivatives(ids, **kw)
        ref = BEASTBsplineTokenizer.reconstruct_traj_derivatives(btok, mp, **kw)
        assert len(got) == 3 and all(torch.equal(a, b) for a, b in zip(got, ref))
    assert torch.equal(btok.reconstruct_traj_derivatives(ids, orders=(0,))[0], btok.reconstruct_traj(ids))
    # continuous coefficients
    ct, pd = tok.encode_continuous(x)
    pos, vel, acc = tok.reconstruct_traj_continuous_derivatives(ct)
    assert torch.equal(pos, tok.reconstruct_traj_continuous(ct))
    tt = grid.expand(ct.shape[0], -1).contiguous()
    res = as_dict(tok.reconstruct_traj_continuous_derivatives(ct, times=tt))
    assert torch.equal(res[0], tok.reconstruct_traj_continuous(ct, times=tt))
    coeff = tok._denormalize_continuous(ct, tok._cuda()).cpu().numpy()
    check_vs_oracle(tok, res, coeff, tt.cpu().numpy(), None, "continuous/rows")
    res_g = as_dict(tok.reconstruct_traj_continuous_derivatives(ct, times=grid))
    assert all(torch.equal(res_g[o], res[o]) for o in (0, 1, 2))


# ---------------------------------------------------------------- 7: error paths
def test_error_paths():
    cfg = GOLDEN_CASES["cfg2_d14"]
    g = load_golden("cfg2_d14")
    tok = make_tok(cfg, g)
    toks = torch.from_numpy(g["tokens_fit"])
    B = toks.shape[0]
    for bad in (torch.zeros(B + 1, 5), torch.zeros(B, 5, 2)):
        with pytest.raises(AssertionError):
            tok.reconstruct_traj_derivatives(toks, times=bad)
    with pytest.raises(AssertionError):
        tok.reconstruct_traj(toks, times=torch.zeros(5))             # 1-D grids stay refused there
    with pytest.raises(ValueError):
        tok.reconstruct_traj_derivatives(toks, orders=(0, 3))
    empty = tok.reconstruct_traj_derivatives(toks[:0], times=torch.zeros(4))
    assert [e.shape for e in empty] == [(0, 4, 14)] * 3
    (e,) = tok.reconstruct_traj_derivatives(toks, times=torch.zeros(0), orders=(1,))
    assert e.shape == (B, 0, 14)
    from beast_tokenizer_b200 import BEASTBsplineTokenizer
    c = BEASTBsplineTokenizer(device="cuda", init_cond_order=2, end_cond_order=0, **COND_CFG)
    with pytest.raises(RuntimeError):
        c.reconstruct_traj_derivatives(toks)                        # no fit yet: no boundary state
    c.encode(torch.from_numpy(g["trajs"][:5]))
    with pytest.raises(RuntimeError):
        c.reconstruct_traj_derivatives(toks)                        # fitted for another batch size
    with pytest.raises(RuntimeError):
        c.reconstruct_traj_continuous_derivatives(torch.zeros(B, 140))


def test_zz_report():
    """Prints the observed normwise errors against the fp64 oracle (pytest -s)."""
    for o in (1, 2):
        errs = [v for (tag, oo), v in REPORT.items() if oo == o]
        if errs:
            print(f"order {o}: max normwise error {max(errs):.3e} over {len(errs)} tensors")
    for (tag, what), v in REPORT.items():
        if what in ("init_vel", "end_vel"):
            print(f"{tag} {what}: {v:.3e}")
