"""Gradients through the continuous spline decode (reconstruct_traj_continuous(_derivatives) backward): params.grad
and init_p.grad against an fp64 dense reference, the adjoint identity, the tiled backward kernel against the generic
one bit for bit, edge semantics, no change without grad, CUDA-graph capture and the C ABI's errors.
Run on the B200 box:  pytest -m gpu."""
import itertools
import math

import numpy as np
import pytest
import torch
from scipy.interpolate import BSpline

from conftest import GOLDEN_CASES, load_golden, rel_err

pytestmark = pytest.mark.gpu

TOL01, TOL2 = 1e-5, 5e-5
TAU32 = float(np.float32(2 * math.pi))
COND_CFG = dict(num_dof=14, num_basis=10, seq_len=50, vocab_size=256, degree_p=4,
                gripper_zero_order=True, gripper_indices=[6, 13], llm_vocab_size=None)
COND_ODD_CFG = dict(num_dof=5, num_basis=8, seq_len=33, vocab_size=1000, degree_p=3,
                    gripper_zero_order=True, gripper_indices=[0])
COND_CASES = [("cond_orders", o) for o in [(2, 0), (0, 2), (2, 2), (1, 1)]] + [("cond_odd", (2, 1))]
ORDER_SETS = [(0,), (1,), (2,), (0, 1, 2)]
REPORT = {}


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


def row_times(B, tq, seed):
    rng = np.random.default_rng(seed)
    tt = torch.from_numpy(rng.uniform(-0.3, TAU32 + 0.3, size=(B, tq)).astype(np.float32))
    tt[:, 0], tt[:, 1] = 0.0, TAU32
    return tt


def ref_rows(tok, times):
    """fp64 scipy design rows at times [B, Tq] (fp32): ({o: joint rows [B, Tq, nc]}, gripper rows [B, Tq, nb])."""
    from beast_tokenizer_b200.basis import knot_vector
    io, eo = (tok.init_cond_order, tok.end_cond_order) if tok._has_conditions else (0, 0)
    nb, p = tok.num_basis, tok.degree_p
    nc = nb + io + eo
    raw = np.asarray(times, np.float32) / np.float32(TAU32)
    u = np.clip(raw.astype(np.float64), 0.0, 1.0)
    inside = ((raw >= 0) & (raw <= 1))[..., None]
    spl = BSpline(knot_vector(nc, p).double().numpy(), np.eye(nc), p)
    rows = {0: spl(u)}
    for o in (1, 2):
        rows[o] = spl.derivative(o)(u) * inside / TAU32 ** o if o <= p else np.zeros(u.shape + (nc,))
    grip = BSpline(knot_vector(nb, 0).double().numpy(), np.eye(nb), 0)(u)
    return rows, grip, io


def ref_coeff_grad(tok, w, times, init_p_used):
    """Gradient of sum_o <w_o, x^(o)> to the de-normalised coefficients [B, D, nb] and to init_p [B, D] (fp64)."""
    rows, grip, io = ref_rows(tok, times)
    B = next(iter(w.values())).shape[0]
    D, nb, nj = tok.num_dof, tok.num_basis, len(tok.joint_indices)
    slots = list(tok.joint_indices) + list(tok.gripper_indices)
    gc = np.zeros((B, D, nb))
    for s, dof in enumerate(slots):
        for o, wo in w.items():
            if s < nj:
                gc[:, s] += np.einsum("btk,bt->bk", rows[o][..., io:io + nb], wo[..., dof])
            elif o == 0:
                gc[:, s] += np.einsum("btk,bt->bk", grip, wo[..., dof])
    gi = np.zeros((B, D))
    if init_p_used:
        for s in range(nj):
            gi[:, slots[s]] = gc[:, s, 0]
            gc[:, s, 0] = 0.0
    return gc, gi


def ref_param_grad(tok, x_norm, gc):
    """Chain the coefficient gradient [B, D, nb] through denormalising and the '(t d)' -> '(d t)' layout."""
    B, D, nb = gc.shape
    lo = tok.w_min.double().cpu().numpy().reshape(D, nb)
    hi = tok.w_max.double().cpu().numpy().reshape(D, nb)
    x_dt = np.asarray(x_norm, np.float32).reshape(B, nb, D).transpose(0, 2, 1)
    mask = (x_dt >= -1) & (x_dt <= 1)
    return (gc * 0.5 * (hi - lo) * mask).transpose(0, 2, 1).reshape(B, nb * D)


def run_grad(tok, x_norm, init_p, times, orders, w, derivatives=True):
    params = x_norm.clone().cuda().requires_grad_(True)
    ip = None if init_p is None else init_p.clone().cuda().requires_grad_(True)
    kw = {} if ip is None else {"init_p": ip}
    if derivatives:
        outs = tok.reconstruct_traj_continuous_derivatives(params, times=times, orders=orders, **kw)
    else:
        outs = (tok.reconstruct_traj_continuous(params, times=times, **kw),)
    loss = sum((out.double() * torch.from_numpy(w[o]).cuda()).sum() for o, out in zip(orders, outs))
    loss.backward()
    return params.grad.cpu().numpy(), None if ip is None else ip.grad.cpu().numpy()


def check_case(tok, tag, x_norm, init_p, times, times_bt, seed):
    rng = np.random.default_rng(seed)
    B, tq, D = x_norm.shape[0], times_bt.shape[1], tok.num_dof
    calls = [(o, True) for o in ORDER_SETS] + ([((0,), False)] if times is None or times.dim() == 2 else [])
    for orders, deriv in calls:
        w = {o: rng.standard_normal((B, tq, D)) for o in orders}
        gp, gi = run_grad(tok, x_norm, init_p, times, orders, w, deriv)
        gc, gi_ref = ref_coeff_grad(tok, w, times_bt, init_p is not None)
        gp_ref = ref_param_grad(tok, x_norm.numpy(), gc)
        tol = TOL2 if 2 in orders else TOL01
        key = (tag, orders, deriv)
        err = rel_err(gp, gp_ref)
        REPORT[key + ("params",)] = err
        assert err <= tol, (key, "params", err)
        if init_p is not None:
            err = rel_err(gi, gi_ref)
            REPORT[key + ("init_p",)] = err
            assert err <= tol, (key, "init_p", err)


# ---------------------------------------------------------------- 1: against fp64, golden geometries and condition orders
def test_grad_vs_fp64(golden_case):
    name, cfg, g = golden_case
    tok = make_tok(cfg, g)
    B, D, nb = g["init_p"].shape[0], cfg["num_dof"], cfg["num_basis"]
    rng = np.random.default_rng(11)
    x = torch.from_numpy(rng.uniform(-1, 1, size=(B, nb * D)).astype(np.float32))
    init_p = torch.from_numpy(g["init_p"])
    grid = shared_grid(200, tok)
    rows = row_times(B, 45, 3)
    own = tok.times.expand(B, -1).numpy()
    for ip in (None, init_p):
        sfx = "/init_p" if ip is not None else ""
        check_case(tok, f"{name}/own{sfx}", x, ip, None, own, 1)
        check_case(tok, f"{name}/grid{sfx}", x, ip, grid, grid.expand(B, -1).numpy(), 2)
        check_case(tok, f"{name}/rows{sfx}", x, ip, rows.cuda(), rows.numpy(), 3)


@pytest.mark.parametrize("case,orders", COND_CASES)
def test_grad_vs_fp64_condition_orders(case, orders):
    tok, g, k = cond_tok(case, orders)
    B, D, nb = g["trajs"].shape[0], tok.num_dof, tok.num_basis
    rng = np.random.default_rng(12)
    x = torch.from_numpy(rng.uniform(-1, 1, size=(B, nb * D)).astype(np.float32))
    init_p = torch.from_numpy(g["init_p"])
    tt = torch.from_numpy(g[k + "custom_times"])
    grid = shared_grid(200, tok)
    for ip in (None, init_p):
        sfx = "/init_p" if ip is not None else ""
        tag = f"{case}{orders}"
        check_case(tok, f"{tag}/own{sfx}", x, ip, None, tok.times.expand(B, -1).numpy(), 4)
        check_case(tok, f"{tag}/grid{sfx}", x, ip, grid, grid.expand(B, -1).numpy(), 5)
        check_case(tok, f"{tag}/rows{sfx}", x, ip, tt.cuda(), tt.numpy(), 6)


# ---------------------------------------------------------------- 2: adjoint identity through the C ABI
def _abi_forward_backward(tok, c, times, grads, gridded):
    """Forward (orders of the non-None grads) and backward through the C ABI on de-normalised coefficients c."""
    from beast_tokenizer_b200 import _lib
    plan = tok._plan()
    dev = plan.device
    B = c.shape[0]
    tq = times.shape[-1]
    outs = [torch.empty((B, tq, tok.num_dof), device=dev) if g is not None else None for g in grads]
    gp = torch.empty((B, tok.num_dof * tok.num_basis), device=dev)
    st = _lib.stream_ptr(dev)
    if gridded:
        gr = tok._grid(plan, times, 2)
        _lib.check(plan._lib.beast_decode_grid_f32(plan.handle, gr.handle, None, _lib.ptr(c), B, None, None, 0, None,
                                                   None, None, *[_lib.ptr(o) for o in outs], st), "fwd")
        _lib.check(plan._lib.beast_decode_grid_backward_f32(plan.handle, gr.handle, B, *[_lib.ptr(g) for g in grads],
                                                            0, _lib.ptr(gp), None, st), "bwd")
    else:
        tt = times.to(dev).contiguous()
        _lib.check(plan._lib.beast_decode_deriv_times_f32(plan.handle, None, _lib.ptr(c), B, None, None, 0, None,
                                                          _lib.ptr(tt), tq, None, None,
                                                          *[_lib.ptr(o) for o in outs], st), "fwd")
        _lib.check(plan._lib.beast_decode_deriv_times_backward_f32(plan.handle, B, _lib.ptr(tt), tq,
                                                                   *[_lib.ptr(g) for g in grads], 0, _lib.ptr(gp),
                                                                   None, st), "bwd")
    torch.cuda.synchronize()
    return outs, gp


@pytest.mark.parametrize("name", ["cfg1_d7", "cfg2_d14", "odd_d5", "cli_default"])
def test_adjoint_identity(name):
    cfg = GOLDEN_CASES[name]
    tok = make_tok(cfg, load_golden(name))
    B, D, nb = 8, cfg["num_dof"], cfg["num_basis"]
    gen = torch.Generator().manual_seed(3)
    c = torch.randn((B, D * nb), generator=gen).cuda()
    for times, gridded in ((shared_grid(200, tok), True), (row_times(B, 64, 7), False)):
        for orders in ORDER_SETS:
            grads = [torch.randn((B, times.shape[-1], D), generator=gen).cuda() if o in orders else None
                     for o in range(3)]
            outs, gp = _abi_forward_backward(tok, c, times, grads, gridded)
            lhs = sum(float((outs[o].double() * grads[o].double()).sum()) for o in orders)
            rhs = float((c.double() * gp.double()).sum())
            scale = sum(float(outs[o].double().norm() * grads[o].double().norm()) for o in orders)
            scale += float(c.double().norm() * gp.double().norm())
            err = abs(lhs - rhs) / max(scale, 1e-30)
            REPORT[(f"{name}/{'grid' if gridded else 'rows'}", orders, "adjoint")] = err
            assert err <= (TOL2 if 2 in orders else TOL01), (name, gridded, orders, err)


# ---------------------------------------------------------------- 3: tiled == generic, bit for bit
def _grid_backward(tok, gr, grads, init_p_used, B, with_init_p):
    from beast_tokenizer_b200 import _lib
    plan = tok._plan()
    dev = plan.device
    gp = torch.full((B, tok.num_dof * tok.num_basis), float("nan"), device=dev)
    gi = torch.full((B, tok.num_dof), float("nan"), device=dev) if with_init_p else None
    _lib.check(plan._lib.beast_decode_grid_backward_f32(plan.handle, gr.handle, B, *[_lib.ptr(g) for g in grads],
                                                        int(init_p_used), _lib.ptr(gp), _lib.ptr(gi),
                                                        _lib.stream_ptr(dev)), "beast_decode_grid_backward_f32")
    return gp, gi


@pytest.mark.parametrize("name", ["cfg2_d14", "odd_d5", "cli_default"])
def test_tiled_equals_generic(name):
    from beast_tokenizer_b200 import _lib
    cfg = GOLDEN_CASES[name]
    tok = make_tok(cfg, load_golden(name))
    lib = _lib.load()
    plan = tok._plan()
    D = cfg["num_dof"]
    sizes = (1, 3, 4097, 65541) if name == "cfg2_d14" else (1, 3, 4097)
    subsets = [s for r in (1, 2, 3) for s in itertools.combinations(range(3), r)]
    for B in sizes:
        for tq in ((37, 1000) if B <= 3 else (37, 200)):
            grid = shared_grid(tq, tok)
            gr = tok._grid(plan, grid, 2)
            n = B * tq * D
            gen = torch.Generator(device="cuda").manual_seed(B + tq)
            # gradients as misaligned views (4-byte aligned, not 16) of one buffer per order
            bufs = [torch.randn(n + 3, device="cuda", generator=gen) for _ in range(3)]
            views = [bufs[o][1 + o:1 + o + n].view(B, tq, D) for o in range(3)]
            for sub in subsets:
                grads = [views[o] if o in sub else None for o in range(3)]
                for init_p_used, with_ip in ((0, False), (1, False), (1, True)):
                    res = {}
                    for slow in (0, 1, 0):
                        prev = lib.beast_debug_disable_fast(slow)
                        try:
                            gp, gi = _grid_backward(tok, gr, grads, init_p_used, B, with_ip)
                            torch.cuda.synchronize()
                        finally:
                            lib.beast_debug_disable_fast(prev)
                        if slow in res:                        # two runs of the same call: the same bits
                            assert torch.equal(gp.view(torch.int32), res[slow][0].view(torch.int32)), (name, B, tq)
                        res[slow] = (gp, gi)
                    assert not torch.isnan(res[0][0]).any()
                    assert torch.equal(res[0][0], res[1][0]), (
                        name, B, tq, sub, init_p_used, float((res[0][0] - res[1][0]).abs().max()))
                    if with_ip:
                        assert not torch.isnan(res[0][1]).any()
                        assert torch.equal(res[0][1], res[1][1]), (name, B, tq, sub)
            del bufs, views
            torch.cuda.empty_cache()


# ---------------------------------------------------------------- 4: edge semantics
def test_edge_semantics():
    cfg = GOLDEN_CASES["cfg2_d14"]
    g = load_golden("cfg2_d14")
    tok = make_tok(cfg, g)
    B, D, nb = 6, cfg["num_dof"], cfg["num_basis"]
    rng = np.random.default_rng(4)
    x = rng.uniform(-1, 1, size=(B, nb * D)).astype(np.float32)
    x[0, :8] = [1.5, -1.5, 1.0, -1.0, 1.0000001, -1.0000001, 3.0, -7.0]
    xt = torch.from_numpy(x)
    # clamp rule: |params| > 1 -> exactly 0, params == +-1 -> the full gradient (fp64 reference uses the same mask)
    w = {0: rng.standard_normal((B, 50, D))}
    gp, _ = run_grad(tok, xt, None, None, (0,), w)
    gc, _ = ref_coeff_grad(tok, w, tok.times.expand(B, -1).numpy(), False)
    ref = ref_param_grad(tok, x, gc)
    assert np.all(gp[np.abs(x) > 1] == 0)
    at_one = np.abs(x) == 1
    assert np.all(gp[at_one] != 0) and rel_err(gp[at_one], ref[at_one]) <= TOL01
    # init_p: the replaced coefficient 0 gets 0, gripper and extra trailing init_p columns get 0
    init_p = torch.randn(B, D + 2).cuda().requires_grad_(True)
    params = torch.from_numpy(np.clip(x, -0.9, 0.9)).cuda().requires_grad_(True)
    for times in (None, shared_grid(77, tok), row_times(B, 31, 2).cuda()):
        params.grad, init_p.grad = None, None
        pos, vel, acc = tok.reconstruct_traj_continuous_derivatives(params, times=times, init_p=init_p)
        (pos.sum() + vel.square().sum() + acc.abs().sum()).backward()
        gpar = params.grad.view(B, nb, D)                 # '(t d)': [b, k, slot], joint slots first
        nj = len(tok.joint_indices)
        assert torch.all(gpar[:, 0, :nj] == 0) and torch.all(gpar[:, 1:, :nj] != 0)
        assert torch.all(init_p.grad[:, tok.gripper_indices] == 0)
        assert torch.all(init_p.grad[:, D:] == 0)
        assert torch.all(init_p.grad[:, tok.joint_indices] != 0)
        # grippers get nothing from orders 1 and 2
        params.grad = None
        vel, acc = tok.reconstruct_traj_continuous_derivatives(params, times=times, orders=(1, 2))
        (vel.sum() + acc.sum()).backward()
        assert torch.all(params.grad.view(B, nb, D)[:, :, nj:] == 0)
        assert params.grad.view(B, nb, D)[:, :, :nj].abs().sum() > 0
    # B = 0 and Tq = 0
    p0 = torch.zeros(0, nb * D, device="cuda", requires_grad=True)
    (pos,) = tok.reconstruct_traj_continuous_derivatives(p0, times=shared_grid(9, tok), orders=(0,))
    pos.sum().backward()
    assert p0.grad.shape == (0, nb * D)
    params.grad = None
    (vel,) = tok.reconstruct_traj_continuous_derivatives(params, times=torch.zeros(0), orders=(1,))
    assert vel.shape == (B, 0, D) and vel.requires_grad
    vel.sum().backward()
    assert params.grad is not None and torch.all(params.grad == 0)
    # double backward raises
    pos = tok.reconstruct_traj_continuous(params)
    (gr,) = torch.autograd.grad(pos.square().sum(), params, create_graph=True)
    with pytest.raises(RuntimeError):
        gr.sum().backward()
    # the BPE subclass inherits the differentiable methods
    from beast_tokenizer_b200 import BEASTBsplineBPETokenizer, BEASTBsplineTokenizer
    for m in ("reconstruct_traj_continuous", "reconstruct_traj_continuous_derivatives"):
        assert getattr(BEASTBsplineBPETokenizer, m) is getattr(BEASTBsplineTokenizer, m)


# ---------------------------------------------------------------- 5: nothing changes without grad
def test_no_change_without_grad():
    from beast_tokenizer_b200 import _lib
    cfg = GOLDEN_CASES["cfg2_d14"]
    g = load_golden("cfg2_d14")
    tok = make_tok(cfg, g)
    B, D, nb = 12, cfg["num_dof"], cfg["num_basis"]
    x = torch.rand(B, nb * D, device="cuda") * 2.2 - 1.1
    ip = torch.randn(B, D, device="cuda")
    grid = shared_grid(64, tok)
    rows = row_times(B, 20, 1).cuda()
    plan = tok._plan()
    dev = plan.device
    st = _lib.stream_ptr(dev)

    def parent(times, deriv):
        """The call sequence of the parent commit: denormalise, then one decode launch."""
        c = tok._denormalize_continuous(x, dev)
        if not deriv:
            tq = 0 if times is None else times.shape[1]
            out = torch.empty((B, 50 if times is None else tq, D), device=dev)
            _lib.check(plan._lib.beast_eval_f32(plan.handle, _lib.ptr(c), B, _lib.ptr(ip), _lib.ptr(times), tq,
                                                _lib.ptr(out), st), "eval")
            return (out,)
        outs = [torch.empty((B, times.shape[-1], D), device=dev) for _ in range(3)]
        if times.dim() == 1:
            gr = tok._grid(plan, times, 2)
            _lib.check(plan._lib.beast_decode_grid_f32(plan.handle, gr.handle, None, _lib.ptr(c), B, None, None, 0,
                                                       _lib.ptr(ip), None, None, *[_lib.ptr(o) for o in outs], st), "g")
        else:
            _lib.check(plan._lib.beast_decode_deriv_times_f32(plan.handle, None, _lib.ptr(c), B, None, None, 0,
                                                              _lib.ptr(ip), _lib.ptr(times), times.shape[1], None,
                                                              None, *[_lib.ptr(o) for o in outs], st), "t")
        return tuple(outs)

    cases = [(None, False), (rows, False), (grid, True), (rows, True)]
    for times, deriv in cases:
        with torch.no_grad():
            n0 = _lib.launch_count()
            ref = parent(times, deriv)
            n_ref = _lib.launch_count() - n0
        for req, ctx in ((False, torch.enable_grad), (True, torch.no_grad)):
            params = x.clone().requires_grad_(req)
            init_p = ip.clone().requires_grad_(req)
            with ctx():
                n0 = _lib.launch_count()
                if deriv:
                    got = tok.reconstruct_traj_continuous_derivatives(params, times=times, init_p=init_p)
                else:
                    got = (tok.reconstruct_traj_continuous(params, times=times, init_p=init_p),)
                n = _lib.launch_count() - n0
            assert n == n_ref, (times is None, deriv, req, n, n_ref)
            for a, b in zip(got, ref):
                assert not a.requires_grad and a.grad_fn is None
                assert torch.equal(a.view(torch.int32), b.view(torch.int32))
        # with grad: the same forward values, attached to the graph
        params = x.clone().requires_grad_(True)
        got = (tok.reconstruct_traj_continuous_derivatives(params, times=times, init_p=ip) if deriv
               else (tok.reconstruct_traj_continuous(params, times=times, init_p=ip),))
        for a, b in zip(got, ref):
            assert a.requires_grad and torch.equal(a.detach().view(torch.int32), b.view(torch.int32))


# ---------------------------------------------------------------- 6: CUDA-graph capture of a training step
@pytest.mark.parametrize("times_kind", ["own", "grid", "rows"])
def test_graph_capture_training_step(times_kind):
    cfg = GOLDEN_CASES["cfg2_d14"]
    tok = make_tok(cfg, load_golden("cfg2_d14"))
    B, D, nb = 64, cfg["num_dof"], cfg["num_basis"]
    times = {"own": None, "grid": shared_grid(120, tok), "rows": row_times(B, 40, 9).cuda()}[times_kind]
    gen = torch.Generator(device="cuda").manual_seed(5)
    x0 = torch.rand(B, nb * D, device="cuda", generator=gen) * 2 - 1
    ip = torch.randn(B, D, device="cuda", generator=gen)
    tq = 50 if times is None else times.shape[-1]
    w0, w2 = (torch.randn(B, tq, D, device="cuda", generator=gen) for _ in range(2))
    params = x0.clone().requires_grad_(True)
    init_p = ip.clone().requires_grad_(True)

    def step():
        pos, acc = tok.reconstruct_traj_continuous_derivatives(params, times=times, orders=(0, 2), init_p=init_p)
        ((pos - w0).square().mean() + 1e-3 * (acc * w2).square().mean()).backward()

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(3):
            params.grad, init_p.grad = None, None
            step()
    torch.cuda.current_stream().wait_stream(s)
    eager_p, eager_i = params.grad.clone(), init_p.grad.clone()
    params.grad, init_p.grad = None, None
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        step()
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(params.grad, eager_p) and torch.equal(init_p.grad, eager_i)
    assert eager_p.abs().sum() > 0


# ---------------------------------------------------------------- 7: C ABI errors
def test_c_abi_errors():
    from beast_tokenizer_b200 import _lib
    E_NULL, E_SHAPE, E_ALIGN = -1, -2, -3
    cfg = GOLDEN_CASES["cfg2_d14"]
    tok = make_tok(cfg)
    other = make_tok(GOLDEN_CASES["odd_d5"])
    plan, oplan = tok._plan(), other._plan()
    lib = plan._lib
    grid = shared_grid(20, tok)
    gr1 = tok._grid(plan, grid, 1)
    ogr = other._grid(oplan, shared_grid(20, other), 2)
    B, D, nb = 4, cfg["num_dof"], cfg["num_basis"]
    g = torch.zeros(B * 20 * D + 1, device="cuda")
    gp = torch.zeros(B * D * nb + 1, device="cuda")
    gi = torch.zeros(B * D, device="cuda")
    G, GP, GI = _lib.ptr(g), _lib.ptr(gp), _lib.ptr(gi)
    mis = C_void(g.data_ptr() + 2)
    st = _lib.stream_ptr(plan.device)

    def grid_bw(grid_h, g0, g1, g2, used, gparams, ginit, pl=plan):
        return lib.beast_decode_grid_backward_f32(pl.handle, grid_h, B, g0, g1, g2, used, gparams, ginit, st)

    def times_bw(times, tq, g0, g1, g2, used, gparams, ginit):
        return lib.beast_decode_deriv_times_backward_f32(plan.handle, B, times, tq, g0, g1, g2, used, gparams, ginit,
                                                         st)
    tt = torch.zeros(B * 20, device="cuda")
    T = _lib.ptr(tt)
    assert grid_bw(gr1.handle, G, None, None, 0, None, None) == E_NULL              # NULL grad_params
    assert times_bw(T, 20, G, None, None, 0, None, None) == E_NULL
    assert grid_bw(gr1.handle, None, None, None, 0, GP, None) == E_NULL             # every gradient NULL
    assert times_bw(T, 20, None, None, None, 0, GP, None) == E_NULL
    assert grid_bw(None, G, None, None, 0, GP, None) == E_NULL                      # no grid
    assert grid_bw(gr1.handle, mis, None, None, 0, GP, None) == E_ALIGN             # misaligned
    assert grid_bw(gr1.handle, G, None, None, 0, C_void(gp.data_ptr() + 1), None) == E_ALIGN
    assert times_bw(C_void(tt.data_ptr() + 2), 20, G, None, None, 0, GP, None) == E_ALIGN
    assert grid_bw(ogr.handle, G, None, None, 0, GP, None) == E_SHAPE               # a grid of another plan
    assert grid_bw(gr1.handle, None, None, G, 0, GP, None) == E_SHAPE               # order above max_order
    assert grid_bw(gr1.handle, G, None, None, 0, GP, GI) == E_SHAPE                 # grad_init_p without init_p
    assert times_bw(T, 20, G, None, None, 0, GP, GI) == E_SHAPE
    assert times_bw(T, -1, G, None, None, 0, GP, None) == E_SHAPE
    assert times_bw(None, 20, G, None, None, 0, GP, None) == E_NULL
    assert grid_bw(gr1.handle, G, G, None, 1, GP, GI) == 0
    torch.cuda.synchronize()


def C_void(addr):
    import ctypes
    return ctypes.c_void_p(addr)


def test_zz_report():
    """Prints the observed normwise errors (pytest -s)."""
    groups = {}
    for key, v in REPORT.items():
        kind = "adjoint" if key[-1] == "adjoint" else ("order2" if 2 in key[1] else "order01")
        groups.setdefault(kind, []).append(v)
    for kind, errs in sorted(groups.items()):
        print(f"{kind}: max normwise error {max(errs):.3e} over {len(errs)} gradients")
