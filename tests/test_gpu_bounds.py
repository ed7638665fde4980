"""The weight-bound reductions against exact references: column min / max (beast_minmax_f32), the 1e-4 hysteresis
(beast_bounds_expand_f32), exact order statistics (beast_colselect_f32) and fit_parameters built on them, the public
bound updates on wide geometries, and the single-launch reduction fused into K1 (beast_fit_minmax_ws_f32).

Min, max and order statistics are exact operations, so every comparison is exact (torch.equal / np.array_equal).
Both compare numerically, so a -0 and a +0 count as equal: the sign of a zero result is not pinned (atomic_min_f32
folds -0 to +0, and np.sort / np.partition leave the order of -0 and +0 open).  Shapes the Python API cannot reach
are called through the C ABI.  NaN inputs are out of scope (the kernels use fminf / fmaxf).
"""
import ctypes as C
import json
import math
import os
import tempfile

import numpy as np
import pytest
import torch

from conftest import GOLDEN_CASES
from oracle import beast_oracle as O
from test_bounds_host import minmax_launch

pytestmark = pytest.mark.gpu

FMAX = float(np.finfo(np.float32).max)
INF = float("inf")


def _L():
    from beast_tokenizer_b200 import _lib as L
    return L, L.load()


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(int(seed))


def _bits(x_int32):
    return x_int32.to(torch.int32).view(torch.float32)


def make_tok(cfg):
    from beast_tokenizer_b200 import BEASTBsplineTokenizer
    return BEASTBsplineTokenizer(device="cuda", **cfg)


def _cfg(num_dof, num_basis, seq_len, grippers=None, degree_p=4, vocab_size=256, llm_vocab_size=None):
    return dict(num_dof=num_dof, num_basis=num_basis, seq_len=seq_len, vocab_size=vocab_size, degree_p=degree_p,
                gripper_zero_order=bool(grippers), gripper_indices=list(grippers or []), llm_vocab_size=llm_vocab_size)


def _offset(cfg):
    return 0 if cfg["llm_vocab_size"] is None else cfg["llm_vocab_size"] - cfg["vocab_size"]


# ---------------------------------------------------------------- (a) beast_minmax_f32
N_MINMAX_FAMILIES = 9


def minmax_data(rows, cols, shift):
    """[rows, cols] fp32 on the device; column c is drawn from family (c + shift) % 9:
    0 mixed signs; 1 all positive (the signed-int atomics); 2 all negative (the unsigned-int atomics); 3 constant;
    4 mixed with +-inf on some rows; 5 +-FLT_MAX among huge values; 6 subnormals and +-0 only; 7 the column's min
    (even c) or max (odd c) in the last row; 8 +-0 only."""
    g = _gen(rows * 7919 + cols * 31 + shift)
    u = torch.rand(rows, cols, generator=g, device="cuda")
    n = torch.randn(rows, cols, generator=g, device="cuda")
    sub = torch.randint(0, 1 << 23, (rows, cols), generator=g, device="cuda", dtype=torch.int32)
    sign = torch.where(n < 0, torch.tensor(-(1 << 31), dtype=torch.int32, device="cuda"),
                       torch.tensor(0, dtype=torch.int32, device="cuda"))
    c = torch.arange(cols, device="cuda")
    fam = ((c + shift) % N_MINMAX_FAMILIES)[None, :].expand(rows, cols)
    x = n.clone()
    x = torch.where(fam == 1, 1.0 + u, x)
    x = torch.where(fam == 2, -1.0 - u, x)
    x = torch.where(fam == 3, torch.full_like(x, 0.375), x)
    f4 = torch.where(u < 0.02, INF, torch.where(u > 0.98, -INF, n))
    x = torch.where(fam == 4, f4, x)
    f5 = torch.where(u < 0.05, FMAX, torch.where(u > 0.95, -FMAX, n * 1e37))
    x = torch.where(fam == 5, f5, x)
    x = torch.where(fam == 6, _bits(torch.bitwise_or(sub, sign)), x)
    if rows:
        last = torch.where(c % 2 == 0, -2.0, 2.0)
        f7 = u.clone()
        f7[-1] = last
        x = torch.where(fam == 7, f7, x)
    x = torch.where(fam == 8, _bits(sign), x)
    return x.contiguous()


def _minmax(x, rows, cols, lo, hi, acc):
    L, lib = _L()
    L.check(lib.beast_minmax_f32(L.ptr(x) if rows else None, rows, cols, L.ptr(lo), L.ptr(hi), acc,
                                 L.stream_ptr(lo.device)), "beast_minmax_f32")


def _start_bounds(x, rows, cols, mode):
    """Output buffers before the call: 'init' NaN garbage (accumulate = 0 must overwrite it); 'tight' bounds inside
    the data (a middle row, or +-1 with no rows); 'loose' bounds outside it on most columns (-FLT_MAX / +3e38, -inf,
    -0 / +0 mixed in)."""
    c = torch.arange(cols, device="cuda")
    if mode == "init":
        return torch.full((cols,), float("nan"), device="cuda"), torch.full((cols,), float("nan"), device="cuda")
    if mode == "tight":
        mid = x[rows // 2] if rows else torch.full((cols,), 1.0, device="cuda")
        lo = torch.where(torch.isinf(mid), 0.5, mid)
        return lo.clone(), torch.where(torch.isinf(mid), 0.25, mid).clone()
    lo = torch.where(c % 3 == 0, -FMAX, torch.where(c % 3 == 1, -INF, -0.0)).to(torch.float32)
    hi = torch.where(c % 3 == 0, 3e38, torch.where(c % 3 == 1, INF, 0.0)).to(torch.float32)
    return lo.contiguous(), hi.contiguous()


def _minmax_rows(cols, aligned, sms):
    L = minmax_launch(cols, aligned, 1, sms)
    cap = max(1, 4 * sms // L["chunks"])
    big = 10 ** 6 if cols * 10 ** 6 <= 1 << 28 else (1 << 28) // cols
    return sorted({0, 1, 31, 32, 33, 511, 512, 513, (cap - 1) * L["rpb"], cap * L["rpb"], cap * L["rpb"] + 1, big})


MINMAX_COLS = [1, 2, 3, 4, 5, 31, 140, 1023, 1024, 1025, 1050, 1600, 4096, 4097, 5120]


@pytest.mark.parametrize("cols", MINMAX_COLS)
def test_minmax_matches_torch(cols):
    """beast_minmax_f32 == x.amin(0) / x.amax(0) at every row count where the grid changes, aligned and through a
    view one float in (the scalar path), with accumulate = 0 and accumulate = 1 onto tighter and looser bounds; one
    init launch (accumulate = 0) plus one reduction launch (rows > 0) per call."""
    L, lib = _L()
    sms = _sms()
    shifts = range(N_MINMAX_FAMILIES) if cols < N_MINMAX_FAMILIES else (0,)
    for aligned in (True, False):
        for rows in _minmax_rows(cols, aligned, sms):
            for shift in (shifts if rows <= 4096 else (0,)):
                x = minmax_data(rows, cols, shift)
                if aligned:
                    xv = x
                else:
                    buf = torch.empty(rows * cols + 1, device="cuda")
                    xv = buf[1:].view(rows, cols)
                    xv.copy_(x)
                    assert rows == 0 or xv.data_ptr() % 16 == 4
                ref_lo = x.amin(0) if rows else torch.full((cols,), INF, device="cuda")
                ref_hi = x.amax(0) if rows else torch.full((cols,), -INF, device="cuda")
                for mode in ("init", "tight", "loose"):
                    lo, hi = _start_bounds(x, rows, cols, mode)
                    acc = 0 if mode == "init" else 1
                    lo0, hi0 = lo.clone(), hi.clone()
                    n0 = L.launch_count()
                    _minmax(xv, rows, cols, lo, hi, acc)
                    assert L.launch_count() - n0 == (1 - acc) + (1 if rows else 0), (rows, cols, mode)
                    want_lo = ref_lo if acc == 0 else torch.minimum(lo0, ref_lo)
                    want_hi = ref_hi if acc == 0 else torch.maximum(hi0, ref_hi)
                    where = (rows, cols, aligned, shift, mode)
                    assert torch.equal(lo, want_lo), ("min", where, (lo != want_lo).nonzero()[:4].flatten().tolist())
                    assert torch.equal(hi, want_hi), ("max", where, (hi != want_hi).nonzero()[:4].flatten().tolist())
                    if rows == 0 and acc:
                        assert torch.equal(lo.view(torch.int32), lo0.view(torch.int32))        # untouched, bit for bit
                        assert torch.equal(hi.view(torch.int32), hi0.view(torch.int32))
    torch.cuda.synchronize()


def _kernel_launches(fn):
    """(grid, block, shared memory) of every minmax_kernel launch in fn(), from a torch.profiler trace."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f)["traceEvents"]
    out = []
    for e in sorted((e for e in events if e.get("cat") == "kernel" and "minmax_kernel" in e.get("name", "")),
                    key=lambda e: e["ts"]):
        a = e["args"]
        out.append((tuple(a["grid"]), tuple(a["block"]), a.get("shared memory")))
    return out


def test_minmax_launch_configuration():
    """The launches the device records are the ones test_bounds_host.py restates: the 140-column shipped shape keeps
    its one-chunk grid, block and shared memory; wide rows are cut into chunks within the same block budget."""
    sms = _sms()
    cases = [(10 ** 6, 140, True), (10 ** 6, 140, False), (1000, 140, True), (4096, 1050, True), (4096, 1600, False),
             (20000, 4160, True), (20000, 5120, False)]
    data = {}
    for rows, cols, aligned in cases:
        x = minmax_data(rows, cols, 0)
        if not aligned:
            buf = torch.empty(rows * cols + 1, device="cuda")
            buf[1:].copy_(x.flatten())
            x = buf[1:].view(rows, cols)
        data[(rows, cols, aligned)] = x
    outs = {k: (torch.empty(k[1], device="cuda"), torch.empty(k[1], device="cuda")) for k in data}

    def run():
        for k, x in data.items():
            _minmax(x, k[0], k[1], *outs[k], 0)

    got = _kernel_launches(run)
    assert len(got) == len(cases), got
    for (rows, cols, aligned), (grid, block, smem) in zip(cases, got):
        want = minmax_launch(cols, aligned, rows, sms)
        assert grid == (want["grid"], 1, 1) and block == (want["block"], 1, 1), ((rows, cols, aligned), grid, block)
        if smem is not None:
            assert smem == want["smem"], ((rows, cols, aligned), smem, want["smem"])
    for k, x in data.items():
        assert torch.equal(outs[k][0], x.amin(0)) and torch.equal(outs[k][1], x.amax(0)), k


# ---------------------------------------------------------------- (b) beast_bounds_expand_f32
def expand_ref(w_min, w_max, bmin, bmax):
    """The reference's update (beast_bspline_tokenizer.py:384-389) in torch on the CPU, fp32: both masks are taken
    before either buffer is written."""
    w_min, w_max = w_min.cpu().clone(), w_max.cpu().clone()
    bmin, bmax = bmin.cpu(), bmax.cpu()
    smaller = bmin < w_min - 1e-4
    larger = bmax > w_max + 1e-4
    w_min[smaller] = bmin[smaller]
    w_max[larger] = bmax[larger]
    return w_min, w_max


@pytest.mark.parametrize("n", [1, 255, 256, 257, 10 ** 5])
def test_bounds_expand_at_the_ulp(n):
    """bmin at exactly fp32(w_min - 1e-4) and one ulp either side (and bmax at fp32(w_max + 1e-4) +- 1 ulp), over
    bounds of every magnitude, +-0 and +-inf, and +-inf batch extremes."""
    L, lib = _L()
    g = torch.Generator().manual_seed(n)
    base = torch.tensor([0.0, -0.0, 1e-4, -1e-4, 0.02, -0.02, 1.0, -1.0, 3.5e-3, 123.456, -7e4, 1e-30, 5e-5,
                         INF, -INF, FMAX, -FMAX], dtype=torch.float32)
    idx = torch.arange(n) % base.numel()
    w_min = torch.where(torch.arange(n) < base.numel(), base[idx], torch.randn(n, generator=g) * 10 ** (
        torch.randint(-6, 4, (n,), generator=g).float()))
    w_max = w_min + torch.rand(n, generator=g).abs()
    w_max = torch.where(torch.isnan(w_max), w_min, w_max)
    thr_lo = w_min - 1e-4                       # fp32, as the reference computes it
    thr_hi = w_max + 1e-4
    pick = torch.arange(n) % 5
    bmin = torch.stack([thr_lo, torch.nextafter(thr_lo, torch.tensor(-INF)), torch.nextafter(thr_lo, torch.tensor(INF)),
                        torch.full((n,), -INF), torch.full((n,), INF)])[(torch.arange(n) // 3) % 5, torch.arange(n)]
    bmax = torch.stack([thr_hi, torch.nextafter(thr_hi, torch.tensor(INF)), torch.nextafter(thr_hi, torch.tensor(-INF)),
                        torch.full((n,), INF), torch.full((n,), -INF)])[pick, torch.arange(n)]
    want_lo, want_hi = expand_ref(w_min, w_max, bmin, bmax)
    # the construction reaches both sides of both thresholds
    if n >= 15:
        finite = torch.isfinite(thr_lo)
        assert ((bmin == thr_lo) & finite & (want_lo == w_min)).any()
        assert ((bmin < thr_lo) & finite & (want_lo == bmin)).any()
        assert ((bmax > thr_hi) & torch.isfinite(thr_hi) & (want_hi == bmax)).any()
    # numpy's restatement (oracle) agrees with torch's
    lo_np = np.array(w_min.numpy(), copy=True)
    sm = bmin.numpy() < (w_min.numpy() - np.float32(1e-4)).astype(np.float32)
    lo_np[sm] = bmin.numpy()[sm]
    assert np.array_equal(lo_np, want_lo.numpy())
    d = {k: v.cuda() for k, v in dict(w_min=w_min, w_max=w_max, bmin=bmin, bmax=bmax).items()}
    L.check(lib.beast_bounds_expand_f32(L.ptr(d["bmin"]), L.ptr(d["bmax"]), L.ptr(d["w_min"]), L.ptr(d["w_max"]), n,
                                        1e-4, L.stream_ptr(d["w_min"].device)), "beast_bounds_expand_f32")
    assert torch.equal(d["w_min"].cpu(), want_lo), (d["w_min"].cpu() != want_lo).nonzero()[:4].flatten().tolist()
    assert torch.equal(d["w_max"].cpu(), want_hi), (d["w_max"].cpu() != want_hi).nonzero()[:4].flatten().tolist()
    # bmin / bmax untouched
    assert torch.equal(d["bmin"].cpu(), bmin) and torch.equal(d["bmax"].cpu(), bmax)


# ---------------------------------------------------------------- (c) beast_colselect_f32
N_SELECT_FAMILIES = 8


def select_data(rows, cols, shift, ks):
    """[rows, cols] fp32 on the device; column c is drawn from family (c + shift) % 8: 0 / 1 / 2 keys sharing their
    top 24 / 16 / 8 bits (1 + i ulp); 3 negatives sharing their top 16 key bits; 4 mixed signs with +-0, +-inf,
    subnormals and +-FLT_MAX; 5 / 6 two / three distinct values (gripper-like) whose tie run ends at k - 1, k or
    k + 1 for one of the ranks k asked for; 7 constant."""
    g = _gen(rows * 104729 + cols * 13 + shift)
    one = 0x3F800000
    c = torch.arange(cols, device="cuda")
    fam = ((c + shift) % N_SELECT_FAMILIES)[None, :].expand(rows, cols)
    r24 = torch.randint(0, 256, (rows, cols), generator=g, device="cuda", dtype=torch.int32)
    r16 = torch.randint(0, 1 << 16, (rows, cols), generator=g, device="cuda", dtype=torch.int32)
    r8 = torch.randint(0, 1 << 24, (rows, cols), generator=g, device="cuda", dtype=torch.int32)
    n = torch.randn(rows, cols, generator=g, device="cuda")
    u = torch.rand(rows, cols, generator=g, device="cuda")
    x = _bits(one + r24)
    x = torch.where(fam == 1, _bits(one + r16), x)
    x = torch.where(fam == 2, _bits(0x3F000000 + r8), x)
    x = torch.where(fam == 3, -_bits(one + r16), x)
    f4 = n.clone()
    f4 = torch.where(u < 0.05, _bits(r8 & 0x7FFFFF) * torch.sign(n), f4)          # subnormals (and +-0)
    f4 = torch.where((u >= 0.05) & (u < 0.08), torch.zeros_like(n) * torch.sign(n), f4)
    f4 = torch.where((u >= 0.08) & (u < 0.09), torch.where(n < 0, -INF, INF), f4)
    f4 = torch.where((u >= 0.09) & (u < 0.10), torch.where(n < 0, -FMAX, FMAX), f4)
    x = torch.where(fam == 4, f4, x)
    # ties: the first z_c rows (in a random order per column) hold the smallest value
    kk = torch.as_tensor([ks[i % len(ks)] for i in range(cols)], device="cuda")
    z = (kk + (c // N_SELECT_FAMILIES) % 3 - 1).clamp(0, rows)
    order = torch.rand(rows, cols, generator=g, device="cuda").argsort(0).argsort(0)      # a random rank per column
    below = order < z[None, :]
    x = torch.where(fam == 5, torch.where(below, 0.0, 1.0), x)
    x = torch.where(fam == 6, torch.where(below, -1.0, torch.where(order % 2 == 0, 0.0, 2.5)), x)
    x = torch.where(fam == 7, torch.full_like(x, -3.25), x)
    return x.contiguous()


def colselect(x, ks):
    L, lib = _L()
    rows, cols = x.shape
    nbytes = int(lib.beast_colselect_scratch_bytes(rows, cols, len(ks)))
    assert nbytes >= rows * cols * 4 and nbytes % 256 == 0
    scratch = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    out = torch.empty((len(ks), cols), device="cuda")
    arr = (C.c_int64 * len(ks))(*ks)
    n0 = L.launch_count()
    L.check(lib.beast_colselect_f32(L.ptr(x), rows, cols, arr, len(ks), L.ptr(out), L.ptr(scratch),
                                    L.stream_ptr(x.device)), "beast_colselect_f32")
    assert L.launch_count() - n0 == 2
    return out


def _ranks(rows, nk, seed):
    """nk ranks in [0, rows): 0 and rows - 1 first, then repeats and random ranks."""
    rng = np.random.default_rng(seed)
    base = [0, rows - 1, rows // 2, rows - 1, int(rng.integers(rows)), 0, int(rng.integers(rows)), rows // 3]
    return base[:nk]


SELECT_CASES = ([(r, c) for r in (1, 2, 31, 32, 33, 511, 512, 513) for c in (1, 31, 32, 33, 140, 1600)] +
                [(100003, 1), (100003, 33), (100003, 140), (2 ** 20 + 3, 1), (2 ** 20 + 3, 31)])


@pytest.mark.parametrize("rows, cols", SELECT_CASES)
def test_colselect_matches_np_sort(rows, cols):
    shifts = range(N_SELECT_FAMILIES) if cols < N_SELECT_FAMILIES else (0, 3)
    for i, shift in enumerate(shifts):
        nk = 1 + (rows + cols + i) % 8
        ks = _ranks(rows, nk, rows * 31 + cols + shift)
        x = select_data(rows, cols, shift, ks)
        got = colselect(x, ks).cpu().numpy()
        xh = x.cpu().numpy()
        want = np.partition(xh, sorted(set(ks)), axis=0)[ks]
        if not np.array_equal(got, want):
            bad = np.argwhere(got != want)[:4].tolist()
            raise AssertionError(f"rows={rows} cols={cols} shift={shift} ks={ks}: differs at (rank, col) {bad}")
        assert rows > 4096 or np.array_equal(want, np.sort(xh, axis=0)[ks])        # the reference itself


def test_colselect_all_eight_ranks_of_one_column():
    """nk = 8 with every rank of a 9-row column but one: the eight CTAs of a column each pick their own rank."""
    x = select_data(9, 40, 0, [0])
    ks = [8, 7, 6, 5, 3, 2, 1, 0]
    assert np.array_equal(colselect(x, ks).cpu().numpy(), np.sort(x.cpu().numpy(), axis=0)[ks])


# ---------------------------------------------------------------- (d) fit_parameters at training scale
class GripperLoader:
    """SyntheticLoader with the gripper DoFs snapped to {0, 1}: a handful of distinct coefficients, full of ties."""

    def __init__(self, inner, grippers, extra_rows=0):
        self.inner, self.grippers, self.extra_rows = inner, list(grippers), extra_rows

    def __iter__(self):
        from beast_tokenizer_b200.synth import synth
        for b in self.inner:
            yield {"actions": self._snap(b["actions"])}
        if self.extra_rows:
            x = synth(self.extra_rows, self.inner.seq_len, self.inner.num_dof, seed=987654)
            yield {"actions": self._snap(x)}

    def _snap(self, x):
        if self.grippers:
            x = x.clone()
            x[..., self.grippers] = (x[..., self.grippers] > 0).to(x.dtype)
        return x


def _quantile_ref(tok, loader):
    xs = torch.cat([b["actions"] for b in loader])
    ws = tok.compute_weights(xs).cpu().numpy()
    return ws, (np.quantile(ws, 0.01, 0).astype(np.float32), np.quantile(ws, 0.99, 0).astype(np.float32))


@pytest.mark.parametrize("name, grip, extra", [("cfg2_d14", False, 0), ("cli_default", False, 0),
                                               ("cfg2_d14", True, 0), ("cfg2_d14", True, 1), ("cli_default", False, 1)])
def test_fit_parameters_training_scale(name, grip, extra):
    """The reference training script's loader size (3 125 batches of 32): fit_parameters == np.quantile on the
    kernel's own coefficients.  grip: gripper DoFs in {0, 1}.  extra = 1: one more trajectory, n = 100 001 rows, where
    (n - 1) * fp32(q) is an exact integer for q = 0.01 and 0.99 (no interpolation; the next order statistic is read
    with weight 0)."""
    from beast_tokenizer_b200.synth import SyntheticLoader
    cfg = GOLDEN_CASES[name]
    tok = make_tok(cfg)
    inner = SyntheticLoader(3125, 32, cfg["seq_len"], cfg["num_dof"], seed0=4242)
    loader = GripperLoader(inner, cfg["gripper_indices"] if grip else [], extra)
    tok.fit_parameters(loader, verbose=False)
    ws, (lo, hi) = _quantile_ref(tok, loader)
    n = ws.shape[0]
    assert n == 100000 + extra
    if extra:
        for q in (0.01, 0.99):
            v = (n - 1) * np.float32(q)
            assert v.dtype == np.float32 and float(v).is_integer()
    if grip:
        D, nb = cfg["num_dof"], cfg["num_basis"]
        slot = len(tok.joint_indices)                   # the first gripper slot
        col = ws[:, slot * nb:(slot + 1) * nb]
        assert np.unique(col).size < n // 100           # ties, many of them
    assert np.array_equal(tok.w_min.cpu().numpy(), lo), np.argwhere(tok.w_min.cpu().numpy() != lo)[:4].tolist()
    assert np.array_equal(tok.w_max.cpu().numpy(), hi), np.argwhere(tok.w_max.cpu().numpy() != hi)[:4].tolist()


def test_column_quantiles_edges():
    """_column_quantiles at q = 0, 1 and 0.5 against np.quantile: one row, two rows, three rows, and 100 003 rows of
    select_data (ties, shared key bits, +-inf, +-0)."""
    tok = make_tok(GOLDEN_CASES["cfg1_d7"])
    for rows, cols in ((1, 5), (2, 7), (3, 70), (101, 70), (100003, 70)):
        x = select_data(rows, cols, 1, [rows // 2])
        if rows < 100:
            x = torch.where(torch.isinf(x), 0.5, x)       # a lerp between +-inf and a finite value is NaN on both sides
        xh = x.cpu().numpy()
        qs = (0.0, 1.0, 0.5, 0.01, 0.99)
        # two ranks per quantile, at most 8 ranks per beast_colselect_f32 call
        got = tok._column_quantiles(x, qs[:3]) + tok._column_quantiles(x, qs[3:])
        for q, g in zip(qs, got):
            want = np.quantile(xh, q, 0).astype(np.float32)
            g = g.numpy()
            same = (g == want) | (np.isnan(g) & np.isnan(want))
            assert same.all(), (rows, q, np.argwhere(~same)[:4].tolist())
        if rows == 1:
            for g in got:
                assert np.array_equal(g.numpy(), xh[0])


# ---------------------------------------------------------------- (e) wide geometries end to end
WIDE = {
    "d14_nb75": _cfg(14, 75, 100),                                   # 1 050 columns, not a multiple of 4
    "d64_nb65": _cfg(64, 65, 100),                                   # 4 160 columns, over 4 096
    "cli_default": GOLDEN_CASES["cli_default"],                      # 1 600 columns (a multiple of 4)
    "d14_nb75_grip_tied": _cfg(14, 75, 100, grippers=[6, 13], llm_vocab_size=32000),
}


@pytest.mark.parametrize("name", list(WIDE))
def test_wide_geometry_bound_updates(name):
    """update_weights_bounds_per_batch, encode(update_bounds=True), encode_continuous(update_bounds=True),
    update_weights_bounds(x) and update_weights_bounds(x, times=t) against the same operations in torch on
    compute_weights(x); also through a weights view one float in (the scalar column path)."""
    from beast_tokenizer_b200.synth import synth_device
    cfg = WIDE[name]
    D, nb, T = cfg["num_dof"], cfg["num_basis"], cfg["seq_len"]
    tok = make_tok(cfg)
    B = 1531
    x = synth_device(B, T, D, 77, "cuda")
    if cfg["gripper_indices"]:
        x[..., cfg["gripper_indices"]] = (x[..., cfg["gripper_indices"]] > 0).float()
    w = tok.compute_weights(x)
    bmin, bmax = w.amin(0), w.amax(0)

    def set_bounds(lo, hi):
        tok.w_min.copy_(lo)
        tok.w_max.copy_(hi)

    # starting bounds: the first third's min / max, with some columns exactly 1e-4 from the batch extreme
    lo0, hi0 = w[:B // 3].amin(0).clone(), w[:B // 3].amax(0).clone()
    cols = torch.arange(D * nb, device="cuda")
    lo0 = torch.where(cols % 7 == 0, bmin + 1e-4, lo0)
    hi0 = torch.where(cols % 7 == 1, bmax - 1e-4, hi0)
    want_lo, want_hi = (t.cuda() for t in expand_ref(lo0, hi0, bmin, bmax))
    assert not torch.equal(want_lo, lo0) and not torch.equal(want_lo, bmin)       # some columns move, some do not

    set_bounds(lo0, hi0)
    tok.update_weights_bounds_per_batch(w)
    assert torch.equal(tok.w_min, want_lo) and torch.equal(tok.w_max, want_hi), "update_weights_bounds_per_batch"

    flat = torch.empty(w.numel() + 1, device="cuda")
    wv = flat[1:].view_as(w)
    wv.copy_(w)
    assert wv.data_ptr() % 16 == 4
    set_bounds(lo0, hi0)
    tok.update_weights_bounds_per_batch(wv)
    assert torch.equal(tok.w_min, want_lo) and torch.equal(tok.w_max, want_hi), "per_batch on an offset view"

    set_bounds(lo0, hi0)
    tokens, pd = tok.encode(x, update_bounds=True)
    assert torch.equal(pd["params"], w)
    assert torch.equal(tok.w_min, want_lo) and torch.equal(tok.w_max, want_hi), "encode(update_bounds=True)"
    off = _offset(cfg)
    assert torch.equal(tokens, tok._quantize(w, off, (want_lo, want_hi)))
    ora = O.tokens_from_params(w.cpu().numpy(), want_lo.cpu().numpy(), want_hi.cpu().numpy(), cfg["vocab_size"], D, nb,
                               off)
    assert np.array_equal(tokens.cpu().numpy(), ora), "tokens != the exact quantiser under the expanded bounds"

    set_bounds(lo0, hi0)
    cont, pd = tok.encode_continuous(x, update_bounds=True)
    assert torch.equal(tok.w_min, want_lo) and torch.equal(tok.w_max, want_hi), "encode_continuous(update_bounds=True)"
    assert torch.equal(cont, tok._normalize(w))

    tok.update_weights_bounds(x)
    assert torch.equal(tok.w_min, bmin) and torch.equal(tok.w_max, bmax), "update_weights_bounds"

    g = torch.Generator().manual_seed(5)
    t = (tok.times[None, :] + 1e-3 * torch.rand(B, T, generator=g)).clamp(0, cfg.get("duration", 2 * math.pi))
    wt = tok.compute_weights(x, times=t)
    tok.update_weights_bounds(x, times=t)
    assert torch.equal(tok.w_min, wt.amin(0)) and torch.equal(tok.w_max, wt.amax(0)), "update_weights_bounds(times=)"


# ---------------------------------------------------------------- (f) the fused reduction
def _fit_minmax_ws(plan, x, B, lo, hi, acc, ws, ws_bytes, stream=None):
    L, lib = _L()
    st = C.c_void_p(stream.cuda_stream) if stream is not None else L.stream_ptr(x.device)
    wp = None if ws is None else C.c_void_p(ws if isinstance(ws, int) else ws.data_ptr())
    L.check(lib.beast_fit_minmax_ws_f32(plan.handle, L.ptr(x), B, L.ptr(lo), L.ptr(hi), acc, wp, ws_bytes, st),
            "beast_fit_minmax_ws_f32")


def test_fused_minmax_ticket_and_fallbacks():
    """cfg2_d14 (T = 50, nb = 10, tile S = 16): one workspace through a sequence of batch sizes that alternate between
    the ticket launch (B >= S) and initialisation + atomics (B < S), accumulate 0 and 1; every result equals torch's
    min / max of compute_weights, so a ticket left non-zero by one launch would show in the next.  A workspace one
    float short or 2 bytes off falls back (and is not written); no workspace at all is beast_fit_minmax_f32."""
    from beast_tokenizer_b200.synth import synth_device
    L, lib = _L()
    cfg = GOLDEN_CASES["cfg2_d14"]
    tok = make_tok(cfg)
    plan = tok._plan()
    sms = _sms()
    S = (7 * 32 // 14) & ~3
    assert S == 16
    Bmax = sms * S + 1
    x = synth_device(Bmax + 64, 50, 14, 31, "cuda")
    w = tok.compute_weights(x)
    n = 14 * 10
    need = int(lib.beast_fit_minmax_workspace_bytes(plan.handle))
    ws = torch.zeros(need // 4, device="cuda")
    sizes = [S - 1, S, S + 1, 5 * S, sms * S - 1, sms * S + 1]
    step = 0
    for rep in range(2):
        for B in sizes + sizes[::-1]:
            for acc in (0, 1):
                r0 = (step * 7) % 64                         # rows are 2 800 B: every start stays 16-byte aligned
                step += 1
                xs = x[r0:r0 + B]
                ref_lo, ref_hi = w[r0:r0 + B].amin(0), w[r0:r0 + B].amax(0)
                o = (step * 13) % (Bmax - 8)
                lo0, hi0 = w[o:o + 8].amin(0), w[o:o + 8].amax(0)                # other rows: tighter and looser
                lo = lo0.clone() if acc else torch.full((n,), float("nan"), device="cuda")
                hi = hi0.clone() if acc else torch.full((n,), float("nan"), device="cuda")
                _fit_minmax_ws(plan, xs, B, lo, hi, acc, ws, need)
                want_lo = torch.minimum(lo0, ref_lo) if acc else ref_lo
                want_hi = torch.maximum(hi0, ref_hi) if acc else ref_hi
                assert torch.equal(lo, want_lo) and torch.equal(hi, want_hi), (rep, B, acc)
    torch.cuda.synchronize()

    B = 5 * S + 3
    ref_lo, ref_hi = w[:B].amin(0), w[:B].amax(0)
    small = torch.zeros(need // 4, device="cuda")
    raw = torch.zeros(need // 4 + 4, device="cuda")
    for what, ptr, nbytes, buf in (("one float short", small, need - 4, small),
                                   ("2 bytes off", raw.data_ptr() + 2, need, raw), ("none", None, 0, None)):
        for acc in (0, 1):
            lo = w[B:B + 4].amin(0).clone() if acc else torch.empty(n, device="cuda")
            hi = w[B:B + 4].amax(0).clone() if acc else torch.empty(n, device="cuda")
            lo0, hi0 = lo.clone(), hi.clone()
            _fit_minmax_ws(plan, x, B, lo, hi, acc, ptr, nbytes)
            want_lo = torch.minimum(lo0, ref_lo) if acc else ref_lo
            want_hi = torch.maximum(hi0, ref_hi) if acc else ref_hi
            assert torch.equal(lo, want_lo) and torch.equal(hi, want_hi), (what, acc)
            if buf is not None:
                assert not bool(buf.any()), f"{what}: the workspace was written"
    for acc in (0, 1):
        lo = w[B:B + 4].amin(0).clone()
        hi = w[B:B + 4].amax(0).clone()
        lo0, hi0 = lo.clone(), hi.clone()
        L.check(lib.beast_fit_minmax_f32(plan.handle, L.ptr(x), B, L.ptr(lo), L.ptr(hi), acc, L.stream_ptr(x.device)),
                "beast_fit_minmax_f32")
        assert torch.equal(lo, torch.minimum(lo0, ref_lo) if acc else ref_lo)
        assert torch.equal(hi, torch.maximum(hi0, ref_hi) if acc else ref_hi)


def test_fused_minmax_two_streams():
    """Two streams, each with its own workspace, issue their calls back to back with no synchronisation between the
    streams; each stream's results equal its serial run on the default stream and torch's min / max."""
    from beast_tokenizer_b200.synth import synth_device
    _, lib = _L()
    cfg = GOLDEN_CASES["cfg2_d14"]
    tok = make_tok(cfg)
    plan = tok._plan()
    sms = _sms()
    S = 16
    x = synth_device(sms * S * 3, 50, 14, 32, "cuda")
    w = tok.compute_weights(x)
    n = 140
    need = int(lib.beast_fit_minmax_workspace_bytes(plan.handle))
    seqs = []
    for s in range(2):
        rng = np.random.default_rng(100 + s)
        seq = []
        for i in range(24):
            B = int(rng.choice([S - 1, S, S + 5, 7 * S, sms * S - 1, sms * S + 1, 2 * sms * S + 3]))
            r0 = int(rng.integers(0, x.shape[0] - B + 1))
            seq.append((r0, B, i % 2))
        seqs.append(seq)

    def starts(seq):
        return [(w[(r0 + 1) % 100:(r0 + 1) % 100 + 8].amin(0).clone(), w[(r0 + 1) % 100:(r0 + 1) % 100 + 8].amax(0).clone())
                for r0, _, _ in seq]

    def run(seq, outs, ws, stream):
        for (r0, B, acc), (lo, hi) in zip(seq, outs):
            _fit_minmax_ws(plan, x[r0:r0 + B], B, lo, hi, acc, ws, need, stream)

    serial = []
    ws0 = torch.zeros(need // 4, device="cuda")
    for seq in seqs:
        outs = starts(seq)
        run(seq, outs, ws0, None)
        serial.append(outs)
    torch.cuda.synchronize()
    conc = [starts(seq) for seq in seqs]
    wss = [torch.zeros(need // 4, device="cuda") for _ in seqs]
    streams = [torch.cuda.Stream() for _ in seqs]
    torch.cuda.synchronize()
    for i in range(len(seqs[0])):                       # interleaved on the host, concurrent on the device
        for s in range(2):
            run(seqs[s][i:i + 1], conc[s][i:i + 1], wss[s], streams[s])
    torch.cuda.synchronize()
    for s in range(2):
        start = starts(seqs[s])
        for i, ((r0, B, acc), (lo, hi), (slo, shi), (lo0, hi0)) in enumerate(zip(seqs[s], conc[s], serial[s], start)):
            ref_lo, ref_hi = w[r0:r0 + B].amin(0), w[r0:r0 + B].amax(0)
            want_lo = torch.minimum(lo0, ref_lo) if acc else ref_lo
            want_hi = torch.maximum(hi0, ref_hi) if acc else ref_hi
            assert torch.equal(slo, want_lo) and torch.equal(shi, want_hi), ("serial", s, i, B, acc)
            assert torch.equal(lo, slo) and torch.equal(hi, shi), ("concurrent", s, i, B, acc)
