"""Launch-boundary overlap of the bulk-copy K1 / K3 kernels.

A captured K1 / K3 launch may stream while the launch before it drains when that launch is the previous bulk-copy K1 /
K3 launch on the stream and the two touch disjoint memory.  Every case below runs the same C-ABI calls eagerly and
captured into a CUDA graph (replayed once, from the same initial buffer contents) and compares the outputs bit for bit;
the overlap count says which captured launches overlapped.  Eager launches never do.
"""

import pytest
import torch

pytestmark = pytest.mark.gpu

T, NB = 50, 10
B = 4096                    # 256 full tiles of 16 trajectories: only the bulk-copy kernels run


def bits(t):
    return t.view(torch.int32) if t.dtype == torch.float32 else t


class Tok:
    """One tokenizer's plan, bounds and C-ABI calls on the current stream."""

    def __init__(self, num_dof, gripper_indices, zero_order, seed):
        from beast_tokenizer_b200 import BEASTBsplineTokenizer, _lib
        from beast_tokenizer_b200.synth import synth
        self._lib, self.D = _lib, num_dof
        self.dev = torch.device("cuda", torch.cuda.current_device())
        self.tok = BEASTBsplineTokenizer(num_dof=num_dof, num_basis=NB, seq_len=T, vocab_size=256,
                                         gripper_zero_order=zero_order, gripper_indices=gripper_indices,
                                         device=str(self.dev), llm_vocab_size=32000)
        self.tok.update_weights_bounds(synth(2048, T, num_dof, seed=seed, device=self.dev))
        self.plan = self.tok._plan()
        self.lib = self.plan._lib
        self.lo, self.hi = self.tok._bounds(self.dev)
        self.offset = 32000 - 256

    def traj(self, n, seed):
        from beast_tokenizer_b200.synth import synth
        return synth(n, T, self.D, seed=seed, device=self.dev)

    def tokens(self, n):
        return torch.zeros((n, NB * self.D), device=self.dev, dtype=torch.int64)

    def params(self, n):
        return torch.zeros((n, NB * self.D), device=self.dev, dtype=torch.float32)

    def out(self, n):
        return torch.zeros((n, T, self.D), device=self.dev, dtype=torch.float32)

    def enc(self, x, toks, pars):
        L, p = self._lib, self._lib.ptr
        L.check(self.lib.beast_encode_f32(self.plan.handle, p(x), x.shape[0], p(self.lo), p(self.hi), self.offset,
                                          p(pars), p(toks), L.stream_ptr(self.dev)), "encode")

    def dec(self, toks, out):
        L, p = self._lib, self._lib.ptr
        L.check(self.lib.beast_decode_f32(self.plan.handle, p(toks), toks.shape[0], p(self.lo), p(self.hi), self.offset,
                                          None, p(out), L.stream_ptr(self.dev)), "decode")

    def bounds(self, x, lo, hi, ws):
        L, p = self._lib, self._lib.ptr
        L.check(self.lib.beast_fit_minmax_ws_f32(self.plan.handle, p(x), x.shape[0], p(lo), p(hi), 0, p(ws),
                                                 ws.numel() * 4, L.stream_ptr(self.dev)), "bounds")


@pytest.fixture(scope="module")
def tok():
    return Tok(14, [6, 13], True, seed=3)


def overlap_count():
    from beast_tokenizer_b200 import _lib
    return _lib.overlap_count()


def eager_vs_graph(reset, ops, outputs, expected_overlaps):
    """reset() puts every buffer into its initial state; ops() makes the calls.  Runs them eagerly, then captured
    and replayed; the outputs must agree bit for bit, and capturing must count `expected_overlaps`."""
    reset()
    n0 = overlap_count()
    ops()
    torch.cuda.synchronize()
    assert overlap_count() == n0, "an eager launch overlapped"
    eager = [o.clone() for o in outputs]
    reset()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    n0 = overlap_count()
    with torch.cuda.graph(g):
        ops()
    assert overlap_count() - n0 == expected_overlaps
    reset()
    torch.cuda.synchronize()
    g.replay()
    torch.cuda.synchronize()
    for e, o in zip(eager, outputs):
        assert torch.equal(bits(e), bits(o))
    return eager


def test_bench_rotating_step(tok):
    """The bench's step: encode of set j, decode of set j+2 (tokens written two steps earlier); every launch after
    the first overlaps.  With the overlap forced off nothing overlaps and the outputs are the same."""
    from beast_tokenizer_b200 import _lib
    R, K = 4, 6
    xs = [tok.traj(B, seed=20 + i) for i in range(R)]
    toks = [tok.tokens(B) for _ in range(R)]
    pars = [tok.params(B) for _ in range(R)]
    outs = [tok.out(B) for _ in range(R)]

    def reset():
        for i in range(R):
            pars[i].zero_()
            outs[i].zero_()
            tok.enc(xs[i], toks[i], pars[i])        # the tokens the first decodes read
            pars[i].zero_()

    def ops():
        for j in range(K):
            tok.enc(xs[j % R], toks[j % R], pars[j % R])
            tok.dec(toks[(j + 2) % R], outs[(j + 2) % R])

    ref = eager_vs_graph(reset, ops, toks + pars + outs, 2 * K - 1)
    prev = _lib.load().beast_debug_force_wait(1)
    try:
        again = eager_vs_graph(reset, ops, toks + pars + outs, 0)
    finally:
        _lib.load().beast_debug_force_wait(prev)
    for a, b in zip(ref, again):
        assert torch.equal(bits(a), bits(b))


def test_decode_of_the_tokens_just_encoded(tok):
    """Read after write: the decode reads the token buffer the encode before it writes."""
    x, toks, pars, out = tok.traj(B, seed=31), tok.tokens(B), tok.params(B), tok.out(B)

    def reset():
        for t in (toks, pars, out):
            t.zero_()

    eager_vs_graph(reset, lambda: (tok.enc(x, toks, pars), tok.dec(toks, out)), [toks, pars, out], 0)


def test_encode_of_the_trajectories_just_decoded(tok):
    """Read after write: the decode writes the trajectories the encode after it reads."""
    toks0 = tok.tokens(B)
    tok.enc(tok.traj(B, seed=32), toks0, tok.params(B))
    xbuf, toks, pars = tok.out(B), tok.tokens(B), tok.params(B)

    def reset():
        for t in (xbuf, toks, pars):
            t.zero_()

    eager_vs_graph(reset, lambda: (tok.dec(toks0, xbuf), tok.enc(xbuf, toks, pars)), [xbuf, toks, pars], 0)


def test_encode_overwriting_the_tokens_just_decoded(tok):
    """Write after read: the encode overwrites the tokens the decode before it reads."""
    x, toks, pars, out = tok.traj(B, seed=33), tok.tokens(B), tok.params(B), tok.out(B)
    toks_init = tok.tokens(B)
    tok.enc(tok.traj(B, seed=34), toks_init, tok.params(B))

    def reset():
        toks.copy_(toks_init)
        pars.zero_()
        out.zero_()

    eager_vs_graph(reset, lambda: (tok.dec(toks, out), tok.enc(x, toks, pars)), [toks, pars, out], 0)


@pytest.mark.parametrize("shift, expected", [(B // 2, 0), (B - 16, 0), (B, 1)])
def test_views_at_offsets(tok, shift, expected):
    """The encode writes rows [0, B) of a token buffer, the decode reads rows [shift, shift + B): partial overlaps
    conflict, the view that starts where the encode's rows end touches them only and overlaps."""
    x, pars = tok.traj(B, seed=35), tok.params(B)
    big, out = tok.tokens(2 * B), tok.out(B)
    big_init = tok.tokens(2 * B)
    tok.enc(tok.traj(2 * B, seed=36), big_init, tok.params(2 * B))

    def reset():
        big.copy_(big_init)
        pars.zero_()
        out.zero_()

    eager_vs_graph(reset, lambda: (tok.enc(x, big[:B], pars), tok.dec(big[shift:shift + B], out)), [big, pars, out],
                   expected)


def test_bounds_launches_sharing_a_workspace(tok):
    """Two update_weights_bounds launches (the single-launch reduction) on one workspace: write after write on the
    per-CTA partials and the ticket, so the second waits."""
    x1, x2 = tok.traj(B, seed=37), tok.traj(B, seed=38)
    ws = tok.plan.minmax_workspace()
    n = tok.D * NB
    lo1, hi1, lo2, hi2 = (torch.zeros(n, device=tok.dev) for _ in range(4))

    def reset():
        for t in (lo1, hi1, lo2, hi2):
            t.zero_()

    eager_vs_graph(reset, lambda: (tok.bounds(x1, lo1, hi1, ws), tok.bounds(x2, lo2, hi2, ws)), [lo1, hi1, lo2, hi2], 0)


def test_torch_op_between_two_launches(tok):
    """A foreign kernel captured between two encodes on disjoint buffers: the second is not adjacent to the first."""
    x1, x2 = tok.traj(B, seed=39), tok.traj(B, seed=40)
    t1, p1, t2, p2 = tok.tokens(B), tok.params(B), tok.tokens(B), tok.params(B)
    other = torch.zeros(1 << 20, device=tok.dev)

    def reset():
        for t in (t1, p1, t2, p2, other):
            t.zero_()

    def ops():
        tok.enc(x1, t1, p1)
        other.add_(1.0)
        tok.enc(x2, t2, p2)

    eager_vs_graph(reset, ops, [t1, p1, t2, p2, other], 0)


def test_two_plans_on_one_stream(tok):
    """Launches of two tokenizers (D = 14 and D = 7) alternate on one stream on disjoint buffers: each overlaps the
    one before it; the decode of A reads the tokens A encoded two launches earlier."""
    other = Tok(7, [6], False, seed=4)
    xa, xb = tok.traj(B, seed=41), other.traj(B, seed=42)
    ta, pa, oa = tok.tokens(B), tok.params(B), tok.out(B)
    tb, pb = other.tokens(B), other.params(B)

    def reset():
        for t in (ta, pa, oa, tb, pb):
            t.zero_()

    eager_vs_graph(reset, lambda: (tok.enc(xa, ta, pa), other.enc(xb, tb, pb), tok.dec(ta, oa)), [ta, pa, oa, tb, pb], 2)
