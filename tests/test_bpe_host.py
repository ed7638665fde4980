"""CPU-only checks of the BPE host logic: file formats, alphabet construction, and the sharded
training protocol (world_size 2, gloo) with a numpy engine standing in for the GPU kernels."""
import json
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN, ROOT, load_golden
from oracle.bpe_oracle import OracleBPE, pretokenize


def test_model_files_round_trip(tmp_path):
    from beast_tokenizer_b200 import B200ByteLevelBPE, BEASTBsplineBPETokenizer
    for name in ("bpe_d14", "bpe_d14_small", "bpe_v1000"):
        src = os.path.join(GOLDEN, f"{name}_pretrained")
        tok = BEASTBsplineBPETokenizer.from_pretrained(src, device="cpu")
        out = tmp_path / name
        tok.save_pretrained(out)
        for f in ("beast_tokenizer_config.json", "bpe_tokenizer/vocab.json", "bpe_tokenizer/merges.txt",
                  "bpe_tokenizer/tokenizer.json"):
            assert open(os.path.join(src, f), encoding="utf-8").read() == open(out / f, encoding="utf-8").read(), f
        sd = tok.state_dict()
        assert sd["bpe"] == {"min_token": 0, "max_token": tok.vocab_size - 1, "vocab_size": tok.bpe_vocab_size,
                             "tokenizer_dir": "bpe_tokenizer"}
        m = tok.bpe_tokenizer
        assert m.get_vocab_size() == tok.bpe_vocab_size and m.token_to_id(m.id_to_token(300)) == 300
    with pytest.raises(ValueError):          # a base-tokenizer checkpoint is not a BPE checkpoint
        BEASTBsplineBPETokenizer.from_pretrained(os.path.join(GOLDEN, "cfg2_d14_pretrained"), device="cpu")
    from beast_tokenizer_b200 import BEASTBsplineTokenizer
    with pytest.raises(ValueError):
        BEASTBsplineTokenizer.from_pretrained(os.path.join(GOLDEN, "bpe_d14_pretrained"), device="cpu")
    with pytest.raises(FileNotFoundError):
        BEASTBsplineBPETokenizer.from_pretrained(tmp_path / "missing")


def test_ctor_errors_and_from_beast():
    from beast_tokenizer_b200 import BEASTBsplineBPETokenizer, BEASTBsplineTokenizer
    base = BEASTBsplineTokenizer(num_dof=7, device="cpu", llm_vocab_size=1000)
    base.w_min.fill_(-0.5)
    tok = BEASTBsplineBPETokenizer.from_beast(base, bpe_vocab_size=300)
    assert tok.bpe_vocab_size == 300 and tok.use_bpe and tok.llm_vocab_size == 1000
    assert torch.equal(tok.w_min, base.w_min) and tok.sequence_length == 70
    assert tok.get_config()["tokenizer_type"] == "beast_bspline_bpe"
    with pytest.raises(TypeError):
        BEASTBsplineBPETokenizer(7, base_tokenizer=base)
    with pytest.raises(TypeError):
        BEASTBsplineBPETokenizer(base_tokenizer=base, num_basis=3)
    with pytest.raises(TypeError):
        BEASTBsplineBPETokenizer(base_tokenizer=object())
    with pytest.raises(TypeError):
        BEASTBsplineBPETokenizer.from_beast(object())
    with pytest.raises(RuntimeError, match="has not been trained"):
        tok._require_bpe()
    from beast_tokenizer_b200 import FIGBPE
    with pytest.raises(RuntimeError):
        FIGBPE().get_state()
    with pytest.raises(ValueError):
        FIGBPE(show_progress=False).fit_from_sequences([[], []])


def test_alphabet_matches_oracle():
    from beast_tokenizer_b200.beast_bpe_trainer import build_alphabet
    rng = np.random.default_rng(0)
    for lo, hi in ((0, 256), (40, 91), (100, 230)):
        bins = rng.integers(lo, hi, (50, 40))
        o = OracleBPE.train(bins, 10)          # vocab_size below the alphabet: no merges, alphabet only
        seen = np.zeros(256, np.int32)
        for v in np.unique(bins - bins.min()):
            for b in chr(int(v)).encode("utf-8"):
                seen[b] = 1
        tokens, b2i = build_alphabet(int(bins.min()), int(bins.max()), seen)
        assert tokens == o.token_strings() and len(o.merges) == 0      # HF keeps the whole alphabet
        assert all((b2i[b] >= 0) == bool(seen[b]) or chr(b) in tokens for b in range(256))


# ---------------------------------------------------------------- sharded protocol on CPU (gloo)
class NumpyEngine:
    """Same interface as GpuBpeEngine, numpy on the CPU (test double for the orchestration)."""

    def __init__(self, bins, min_token, byte_to_id, V):
        self.V = V
        self.words = []
        for row in np.asarray(bins):
            cp = (row - min_token).astype(np.uint8)
            ws = pretokenize(cp)
            seq = []
            for c, w in zip(cp.tolist(), ws.tolist()):
                bs = chr(c).encode("utf-8")
                for j, b in enumerate(bs):
                    seq.append([int(byte_to_id[b]), bool(w) and j == 0])
            self.words.append(seq)
        self.hist = torch.zeros((V, V), dtype=torch.int32)
        for seq in self.words:
            for (x, _), (y, wy) in zip(seq[:-1], seq[1:]):
                if not wy:
                    self.hist[x, y] += 1
        self.delta = torch.zeros(4 * V, dtype=torch.int32)

    def argmax(self, n_active):
        h = self.hist[:n_active, :n_active]
        m = int(h.max())
        if m <= 0:
            return 0, -1, -1
        flat = int(torch.nonzero(h.reshape(-1) == m)[0])
        return m, flat // n_active, flat % n_active

    def merge(self, a, b, c):
        from collections import Counter
        V, d, net = self.V, self.delta, Counter()
        for seq in self.words:
            for (x, _), (y, wy) in zip(seq[:-1], seq[1:]):
                if not wy:
                    net[(x, y)] -= 1
            out, q = [], 0
            while q < len(seq):
                if q + 1 < len(seq) and seq[q][0] == a and seq[q + 1][0] == b and not seq[q + 1][1]:
                    out.append([c, seq[q][1]]); q += 2
                else:
                    out.append(seq[q]); q += 1
            seq[:] = out
            for (x, _), (y, wy) in zip(seq[:-1], seq[1:]):
                if not wy:
                    net[(x, y)] += 1
        for (x, y), n in net.items():
            if n == 0 or (x, y) == (a, b):
                continue
            if n < 0:
                if y == a: d[x] += n
                elif x == b: d[V + y] += n
                else: raise AssertionError(("lost pair outside column a / row b", x, y, n))
            else:
                if y == c: d[2 * V + x] += n
                elif x == c: d[3 * V + y] += n
                else: raise AssertionError(("gained pair outside column c / row c", x, y, n))

    def apply_delta(self, a, b, c):
        V, d = self.V, self.delta.clone()
        self.hist[:, a] += d[:V]; self.hist[b, :] += d[V:2 * V]; self.hist[:, c] += d[2 * V:3 * V]; self.hist[c, :] += d[3 * V:]
        self.hist[a, b] = 0
        self.delta.zero_()


def numpy_scan(bins, coll):
    bins = np.asarray(bins)
    lo = torch.tensor([int(bins.min())]); hi = torch.tensor([int(bins.max())])
    coll.reduce_(lo, "min"); coll.reduce_(hi, "max")
    mn, mx = int(lo), int(hi)
    seen = torch.zeros(256, dtype=torch.int32)
    for v in np.unique(bins - mn):
        for b in chr(int(v)).encode("utf-8"):
            seen[b] = 1
    coll.reduce_(seen, "max")
    return mn, mx, seen.numpy()


def _worker(rank, world, port, bins, vocab, q):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from beast_tokenizer_b200.beast_bpe_trainer import _Collective, train_bpe
    shard = bins[rank::world]
    tok, mn, mx = train_bpe(shard, vocab, 2, engine_factory=NumpyEngine, scan=numpy_scan, coll=_Collective())
    q.put((rank, tok.merges_txt(), tok.vocab_json(), mn, mx))
    dist.destroy_process_group()


def test_single_rank_protocol_matches_oracle():
    from beast_tokenizer_b200.beast_bpe_trainer import _Collective, train_bpe
    rng = np.random.default_rng(5)
    bins = rng.integers(30, 120, (60, 30))
    tok, mn, mx = train_bpe(bins, 260, 2, engine_factory=NumpyEngine, scan=numpy_scan, coll=_Collective(enabled=False))
    o = OracleBPE.train(bins, 260)
    assert tok.merges_txt() == o.merges_txt() and tok.vocab_json() == o.vocab_json()


def test_sharded_training_two_ranks_gloo():
    """Two processes, each with half of the sequences: min/max, seen bytes, histogram and per-merge
    deltas are all-reduced; both ranks end with the unsharded oracle's merges and vocabulary."""
    import torch.multiprocessing as mp
    rng = np.random.default_rng(11)
    bins = rng.integers(20, 140, (80, 24))
    bins[::2] += 60                                  # the two shards see different value ranges
    o = OracleBPE.train(bins, 300)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_worker, args=(r, 2, port, bins, 300, q)) for r in range(2)]
    for p in procs:
        p.start()
    results = [q.get(timeout=180) for _ in procs]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for _, merges_txt, vocab_json, mn, mx in results:
        assert merges_txt == o.merges_txt() and vocab_json == o.vocab_json()
        assert (mn, mx) == (int(bins.min()), int(bins.max()))


def test_ids_to_csr_accepts_every_container():
    """bpe_to_mp_tokens / reconstruct_traj take the ragged List[List[int]] that encode() returns, and also
    tuples, numpy rows, tensors, a single flat list: all must flatten to the same CSR (host logic, no GPU)."""
    from beast_tokenizer_b200.beast_bspline_bpe_tokenizer import BEASTBsplineBPETokenizer as T
    obj = T.__new__(T)
    rows = [[1, 2, 3], [4], [], [5, 6, 2047]]
    flat, off = T._ids_to_csr(obj, rows, "cpu")
    assert flat.dtype == torch.int32 and off.dtype == torch.int64
    assert flat.tolist() == [1, 2, 3, 4, 5, 6, 2047] and off.tolist() == [0, 3, 4, 4, 7]
    for variant in (tuple(tuple(r) for r in rows), [np.asarray(r, dtype=np.int64) for r in rows],
                    [torch.tensor(r, dtype=torch.long) for r in rows], [[np.int32(v) for v in r] for r in rows]):
        f2, o2 = T._ids_to_csr(obj, variant, "cpu")
        assert torch.equal(f2, flat) and torch.equal(o2, off)
    f3, o3 = T._ids_to_csr(obj, [7, 8, 9], "cpu")                     # one sequence given as a flat list
    assert f3.tolist() == [7, 8, 9] and o3.tolist() == [0, 3]
    f4, o4 = T._ids_to_csr(obj, torch.tensor([[1, 2], [3, 4]]), "cpu")
    assert f4.tolist() == [1, 2, 3, 4] and o4.tolist() == [0, 2, 4]
    with pytest.raises(ValueError):
        T._ids_to_csr(obj, [[2 ** 40]], "cpu")


def test_list_helpers_c_and_python_agree(monkeypatch):
    """CSR <-> List[List[int]] (the reference's return / argument type, beast_bspline_bpe_tokenizer.py:175-247):
    the CPython helper (csrc/pylists.c) and the pure-Python conversions must give the same lists / arrays,
    including empty rows, ids above the shared-int cache, negative ids and the int32 range error."""
    import beast_tokenizer_b200.beast_bspline_bpe_tokenizer as M
    rng = np.random.default_rng(11)
    lens = rng.integers(0, 40, 500)
    lens[[0, 7, 499]] = 0
    off = np.zeros(501, np.int64)
    np.cumsum(lens, out=off[1:])
    flat = rng.integers(0, 3000, int(off[-1])).astype(np.int32)
    flat[:4] = [-1, 2 ** 31 - 1, 1 << 20, (1 << 20) - 1]
    want = [flat[off[i]:off[i + 1]].tolist() for i in range(500)]
    cmod = M._pylists()
    assert cmod, "the in-tree CPython helper did not build / import"
    got = {}
    for name, mod in (("c", cmod), ("py", False)):
        monkeypatch.setattr(M, "_PYLISTS", mod)
        rows = M._split_rows(flat, off)
        assert rows == want and all(type(v) is int for r in rows for v in r), name
        f, o = M._flatten_rows(rows)
        assert f.dtype == np.int32 and o.dtype == np.int64
        assert np.array_equal(f, flat) and np.array_equal(o, off), name
        f, o = M._flatten_rows(tuple(tuple(r) for r in rows))
        assert np.array_equal(f, flat) and np.array_equal(o, off), name
        assert M._flatten_rows([np.arange(3)]) is None, name
        T = M.BEASTBsplineBPETokenizer                              # floats truncate like int() on either path
        f2, o2 = T._ids_to_csr(T.__new__(T), [[1, 2.5], [np.int64(7)]], "cpu")
        assert f2.tolist() == [1, 2, 7] and o2.tolist() == [0, 2, 3], name
        for bad in ([[2 ** 31]], [[-2 ** 31 - 1]], [[2 ** 80]]):
            with pytest.raises(ValueError):
                M._flatten_rows(bad)
        got[name] = rows
    assert got["c"] == got["py"]
    with pytest.raises(ValueError):
        cmod.split_rows(flat, off[:-3].copy())           # offsets that do not cover the ids
    bad_off = off.copy()
    bad_off[3] = off[-1] + 1
    with pytest.raises(ValueError):
        cmod.split_rows(flat, bad_off)


def test_match_resolution_by_function_composition():
    """The warp-per-sequence rewrite (csrc/bpe.cu: rewrite_sequence_warp) resolves the greedy left-to-right rule
    match[p] = cand[p] and not match[p-1] without a serial pass: every lane evaluates its 8-symbol chunk for both
    possible incoming values, the two results form a one-bit function, and an inclusive scan over function
    compositions gives each lane its true input.  Restated here lane by lane and compared with the serial rule."""
    rng = np.random.default_rng(5)

    def serial(cand):
        out, prev = [], 0
        for c in cand:
            prev = c & (prev ^ 1)
            out.append(prev)
        return out

    def run_chunk(bits, m_in):
        out, prev = [], m_in
        for c in bits:
            prev = c & (prev ^ 1)
            out.append(prev)
        return out

    for trial in range(400):
        n_lanes = 32
        p_run = rng.choice([0.05, 0.3, 0.7, 0.95])
        cand = (rng.random(n_lanes * 8) < p_run).astype(int).tolist()        # long runs exercise the (a, a) case
        chunks = [cand[8 * lane:8 * lane + 8] for lane in range(n_lanes)]
        f = []                                                               # bit x of f = chunk output for input x
        for ch in chunks:
            f.append(run_chunk(ch, 0)[-1] | (run_chunk(ch, 1)[-1] << 1))
        o = 1
        while o < n_lanes:                                                   # Hillis-Steele scan, F_l = f_l o F_{l-o}
            g = [f[lane - o] if lane >= o else None for lane in range(n_lanes)]
            f = [((f[lane] >> (g[lane] & 1)) & 1) | (((f[lane] >> ((g[lane] >> 1) & 1)) & 1) << 1)
                 if g[lane] is not None else f[lane] for lane in range(n_lanes)]
            o <<= 1
        m_in = [0] + [f[lane - 1] & 1 for lane in range(1, n_lanes)]
        got = [b for lane in range(n_lanes) for b in run_chunk(chunks[lane], m_in[lane])]
        assert got == serial(cand)


def test_parallel_utf8_decode_rules_match_the_state_machine():
    """The warp-per-sequence BPE decode (csrc/bpe.cu: bpe_decode_warp_kernel) classifies every byte on its own:
    a non-continuation byte starts a character (index = number of such bytes before it), a continuation byte
    must lie inside the span of the lead before it.  Restated here and compared with the sequential decoder and with
    Python's strict decoder (status 2 = invalid UTF-8 — overlong and surrogate forms included — or a character above
    U+FFFF, 3 = wrong length, character count) on random byte streams."""
    rng = np.random.default_rng(9)

    def lead_len(b):                                    # strict UTF-8: C0, C1 and F5..FF start nothing
        return 1 if b < 0x80 else 0 if b < 0xC2 else 2 if b < 0xE0 else 3 if b < 0xF0 else 4 if b < 0xF5 else 0

    def second_ok(lead, c):                             # overlong, surrogate and > U+10FFFF forms fail here
        lo = 0xA0 if lead == 0xE0 else 0x90 if lead == 0xF0 else 0x80
        hi = 0x9F if lead == 0xED else 0x8F if lead == 0xF4 else 0xBF
        return lo <= c <= hi

    def python_strict(bs, L):                           # Python's strict decoder + the kernels' status order
        try:
            cps = [ord(c) for c in bytes(bs).decode("utf-8")]
        except UnicodeDecodeError:
            return 2, None, None
        if any(c > 0xFFFF for c in cps):                # valid UTF-8, but no shifted bin
            return 2, None, None
        return (3 if len(cps) != L else 0), len(cps), cps[:L]

    def sequential(bs, L):
        status = cnt = pending = acc = lead = 0
        out = []
        for bt in bs:
            c = -1
            if pending:
                if not (second_ok(lead, bt) if lead else (bt & 0xC0) == 0x80):
                    return 2, cnt, out
                lead = 0
                acc = (acc << 6) | (bt & 0x3F)
                pending -= 1
                if pending == 0:
                    c = acc
            elif bt < 0x80:
                c = bt
            elif lead_len(bt) >= 2:
                pending = lead_len(bt) - 1
                acc = bt & (0x3F >> pending)
                lead = bt
            else:
                return 2, cnt, out
            if c >= 0:
                if c > 0xFFFF:
                    return 2, cnt, out
                if cnt < L:
                    out.append(c)
                cnt += 1
        if pending:
            return 2, cnt, out
        return (3 if cnt != L else 0), cnt, out

    def parallel(bs, L):
        B = len(bs)
        first_err, pend_end, n_start, out = None, False, 0, {}
        for i, b in enumerate(bs):                      # every i is an independent lane
            cont = (b & 0xC0) == 0x80
            err = None
            if not cont:
                n = lead_len(b)
                idx = sum(1 for j in range(i) if (bs[j] & 0xC0) != 0x80)
                if n == 0:
                    err = i
                else:
                    acc, complete = (b if n == 1 else b & (0x7F >> n)), True
                    for k in range(1, n):
                        if i + k >= B:
                            pend_end, complete = True, False
                            break
                        c = bs[i + k]
                        if not (second_ok(b, c) if k == 1 else (c & 0xC0) == 0x80):
                            err, complete = i + k, False
                            break
                        acc = (acc << 6) | (c & 0x3F)
                    if complete:
                        if acc > 0xFFFF:
                            err = i + n - 1
                        elif idx < L:
                            out[idx] = acc
                n_start += 1
            else:
                covered = False
                for k in range(1, min(3, i) + 1):
                    c = bs[i - k]
                    if (c & 0xC0) != 0x80:
                        covered = lead_len(c) > k
                        break
                if not covered:
                    err = i
            if err is not None and (first_err is None or err < first_err):
                first_err = err
        cnt = n_start - (1 if pend_end else 0)
        if first_err is not None:
            return 2, None, None
        if pend_end:
            return 2, None, None
        return (3 if cnt != L else 0), cnt, [out[i] for i in range(min(cnt, L))]

    pool = [0x41, 0x7A, 0xC3, 0xA9, 0x80, 0xBF, 0xE2, 0x82, 0xAC, 0xF0, 0x9F, 0x98, 0xF8, 0xFF, 0xC2,
            0xE0, 0xED, 0xA0, 0x90, 0x8F, 0xC0, 0xC1, 0xF4, 0xF5]
    fixed = [[0xE0, 0x80, 0x80], [0xED, 0xA0, 0x80], [0xC0, 0x80], [0xC1, 0xBF], [0xF0, 0x80, 0x80, 0x80],
             [0xF4, 0x90, 0x80, 0x80], [0xF5, 0x80], [0xE0, 0xA0, 0x80], [0xED, 0x9F, 0xBF], [0xEE, 0x80, 0x80],
             [0xF0, 0x90, 0x80, 0x80], [0x41, 0xE0], [0x41, 0xE0, 0x9F], [0x41, 0xED, 0xA0]]
    for bs in fixed:                                    # overlong / surrogate / out-of-range forms and their neighbours
        for L in range(4):
            want = python_strict(bs, L)
            for got in (sequential(bs, L), parallel(bs, L)):
                assert got[0] == want[0] and (want[0] == 2 or got[1:] == want[1:]), (bs, L, got, want)
    for trial in range(3000):
        if trial % 3 == 0:                              # valid text with a few mutations
            text = "".join(chr(int(v)) for v in rng.integers(1, 0x2FFF, int(rng.integers(0, 12))))
            bs = list(text.encode("utf-8"))
            if bs and trial % 6 == 0:
                bs[int(rng.integers(0, len(bs)))] = int(rng.choice(pool))
        else:
            bs = [int(v) for v in rng.choice(pool, int(rng.integers(0, 14)))]
        L = int(rng.integers(0, 8))
        s1, c1, o1 = sequential(bs, L)
        s2, c2, o2 = parallel(bs, L)
        s3, c3, o3 = python_strict(bs, L)
        assert s1 == s2 == s3, (bs, L, s1, s2, s3)
        if s1 in (0, 3):
            assert c1 == c2 == c3 and o1 == o2 == o3, (bs, L)


def test_token_character_table_matches_the_state_machine():
    """The decode kernel's fast path (csrc/bpe.cu: bpe_decode_warp_kernel) works per TOKEN from a precomputed table
    (bpe_model.token_char_entry): complete characters, leading continuation bytes, bytes the last character still
    needs.  Restated here lane by lane and compared with the sequential UTF-8 state machine on random token
    sequences: whenever the fast path accepts a sequence it must give the sequential decoder's characters; it must
    accept valid text cut into tokens at character boundaries, and text cut inside characters whenever the rest of a
    cut character lies in the next token (a character spread over three tokens takes the byte-level path)."""
    from beast_tokenizer_b200.bpe_model import token_char_entry
    rng = np.random.default_rng(13)

    def sequential(bs):                 # Python's strict decoder; characters above U+FFFF are no shifted bin
        try:
            out = [ord(c) for c in bytes(bs).decode("utf-8")]
        except UnicodeDecodeError:
            return None
        return None if any(c > 0xFFFF for c in out) else out

    def fast(tokens):
        ent = [token_char_entry(t) for t in tokens]
        if not ent:
            return []
        meta = [e[3] for e in ent]
        if any(m & 0x0C000080 for m in meta) or (meta[0] >> 5) & 3:     # slow, or a bare E0 / ED lead ends a token
            return None
        out = []
        for i, e in enumerate(ent):
            nst, need = meta[i] & 7, (meta[i] >> 3) & 3
            nmeta = meta[i + 1] if i + 1 < len(ent) else 0
            if need != (nmeta >> 5) & 3:
                return None
            cps = [e[0] & 0xffff, e[0] >> 16, e[1] & 0xffff, e[1] >> 16, e[2] & 0xffff, e[2] >> 16][:nst]
            if need:
                cps[-1] = (cps[-1] | ((nmeta >> 8) & 0x3ffff)) & 0xffff
            out += cps
        return out

    accepted = 0
    for trial in range(4000):
        if trial % 2 == 0:      # valid text (1-, 2-, 3-byte characters) cut at arbitrary byte positions
            text = "".join(chr(int(v)) for v in rng.choice([rng.integers(1, 128), rng.integers(128, 0x800), rng.integers(0x800, 0xD800)],
                                                              int(rng.integers(1, 30))))
            bs = text.encode("utf-8")
            cuts = sorted(set(rng.integers(1, len(bs), int(rng.integers(0, len(bs)))).tolist())) if len(bs) > 1 else []
            if trial % 4 == 0:      # cut at character boundaries only
                cuts = [c for c in cuts if (bs[c] & 0xC0) != 0x80]
            toks = [bs[a:b] for a, b in zip([0] + cuts, cuts + [len(bs)])]
            want = sequential(bs)
            got = fast(toks)
            assert want == [ord(c) for c in text]
            assert got is None or got == want, (toks, got, want)
            short = all(sum(1 for b in t if (b & 0xC0) != 0x80) <= 6 for t in toks)
            # a cut character is completed by the NEXT token alone unless that token is nothing but continuation bytes
            # and the character needs more
            chained = any(all((b & 0xC0) == 0x80 for b in t) and i + 1 < len(toks) and (toks[i + 1][0] & 0xC0) == 0x80
                          for i, t in enumerate(toks))
            # a token ending in a bare E0 / ED lead sends the sequence to the byte-level path (its next byte is restricted)
            bare_lead = any(t[-1] in (0xE0, 0xED) for t in toks[:-1])
            if short and not chained and not bare_lead:
                assert got == want, (toks, got, want)
                accepted += 1
        else:                   # garbage bytes: the fast path may refuse, but must never disagree
            pool = [0x41, 0x7A, 0xC3, 0xA9, 0x80, 0xBF, 0xE2, 0x82, 0xAC, 0xF0, 0x9F, 0x98, 0xF8, 0xFF, 0xC2,
                    0xE0, 0xED, 0xA0, 0x90, 0x8F, 0xC0, 0xC1, 0xF4, 0xF5]
            toks = [bytes(int(v) for v in rng.choice(pool, int(rng.integers(1, 5)))) for _ in range(int(rng.integers(1, 12)))]
            want = sequential(b"".join(toks))
            got = fast(toks)
            if got is not None:
                assert want == got, (toks, got, want)
    assert accepted > 1000
    # overlong and surrogate forms, whole or split after their lead: never accepted
    for toks in ([b"\xe0\x80\x80"], [b"\xe0", b"\x80\x80"], [b"\xe0\x80", b"\x80"], [b"\xed\xa0\x80"], [b"A\xed", b"\xa0\x80"],
                 [b"\xed", b"\xbf\xbf"], [b"\xc0\x80"], [b"\xc1", b"\xbf"]):
        assert fast(toks) is None, toks
    # the nearest valid forms are, unless split after their lead
    assert fast([b"\xed\x9f", b"\xbf"]) == [0xD7FF] and fast([b"\xe0\xa0", b"\x80A"]) == [0x800, 0x41]
    assert fast([b"\xed", b"\x9f\xbf"]) is None and fast([b"\xe0", b"\xa0\x80A"]) is None


def test_rank_order_batch_merging_equals_one_merge_at_a_time():
    """The cooperative long-word path of the encode kernel (csrc/bpe.cu: bpe_encode_warp_kernel, phase D) applies, per
    step, ALL occurrences of the lowest-rank pair present, left to right (overlapping candidates — runs of one symbol —
    alternate from the run's first position), instead of HF's 'lowest rank, leftmost first, one merge at a time'.
    The two are equal because a merge only creates pairs that involve the new token, whose rules were learned later
    (higher rank).  Restated here on random words and random merge tables that respect that property."""
    rng = np.random.default_rng(3)

    def one_at_a_time(word, rank, new_id):
        w = list(word)
        while True:
            best, bp = None, -1
            for q in range(len(w) - 1):
                r = rank.get((w[q], w[q + 1]))
                if r is not None and (best is None or r < best):
                    best, bp = r, q
            if best is None:
                return w
            w[bp:bp + 2] = [new_id[(w[bp], w[bp + 1])]]

    def batch_by_rank(word, rank, new_id):
        w = list(word)
        while True:
            ranks = [rank.get((w[q], w[q + 1])) for q in range(len(w) - 1)]
            present = [r for r in ranks if r is not None]
            if not present:
                return w
            best = min(present)
            cand = [r == best for r in ranks] + [False]
            # chunked run-parity resolution, as the kernel does it (32 positions per step, carry = last position matched)
            match, m_prev = [False] * len(w), False
            for q0 in range(0, len(w), 32):
                C = cand[q0:q0 + 32]
                for lane, c in enumerate(C):
                    zeros_below = [i for i in range(lane) if not C[i]]
                    run_start = zeros_below[-1] + 1 if zeros_below else 0
                    match[q0 + lane] = c and ((lane - run_start) + (int(m_prev) if run_start == 0 else 0)) % 2 == 0
                m_prev = match[min(q0 + 31, len(w) - 1)] if q0 + 32 <= len(w) else False
            out, q = [], 0
            while q < len(w):
                if match[q]:
                    out.append(new_id[(w[q], w[q + 1])]); q += 2
                else:
                    out.append(w[q]); q += 1
            w = out

    for trial in range(300):
        n_alpha = int(rng.integers(2, 6))
        rank, new_id, n_tok = {}, {}, n_alpha
        for r in range(int(rng.integers(1, 25))):       # every rule pairs EXISTING tokens: pairs of a new token rank later
            a, b = int(rng.integers(0, n_tok)), int(rng.integers(0, n_tok))
            if (a, b) in rank:
                continue
            rank[(a, b)] = r
            new_id[(a, b)] = n_tok
            n_tok += 1
        word = rng.integers(0, n_alpha, int(rng.integers(1, 150))).tolist()
        if trial % 3 == 0:                              # long runs of one symbol: the overlapping-candidate case
            word = ([0] * int(rng.integers(30, 100))) + word
        assert batch_by_rank(word, rank, new_id) == one_at_a_time(word, rank, new_id), (word, rank)


def _single_pass_word_starts(cp, cls):
    """CPU restatement of bpe_symbolize_kernel's one-pass pre-tokenizer (csrc/bpe.cu): constant work per codepoint,
    state = (class of the run being extended, inside a whitespace run of two or more, codepoints left of a
    contraction)."""
    n = len(cp)
    S = 3
    out = np.zeros(n, dtype=np.uint8)
    run_cls, skip, ws_run = -1, 0, False
    for p in range(n):
        c, k = int(cp[p]), int(cls[cp[p]])
        has1 = p + 1 < n
        c1 = int(cp[p + 1]) if has1 else 0
        k1 = int(cls[c1]) if has1 else -1
        if skip > 0:
            start = False
            skip -= 1
        elif k == S:
            next_s = k1 == S
            if not ws_run:
                start = True
                if next_s:
                    ws_run = True
                else:
                    run_cls = k1 if (has1 and c == 32) else -1
            elif next_s or not has1:
                start = False
            else:
                start, ws_run = True, False
                run_cls = k1 if c == 32 else -1
        elif k == run_cls:
            start = False
        else:
            start, run_cls = True, k
            if c == 39 and has1:
                c2 = int(cp[p + 2]) if p + 2 < n else 0
                cl = 0
                if chr(c1) in "stmd":
                    cl = 2
                elif (chr(c1), chr(c2)) in (("r", "e"), ("v", "e"), ("l", "l")):
                    cl = 3
                if cl:
                    skip, run_cls = cl - 1, -1
        out[p] = start
    return out


def test_single_pass_pretokenizer_equals_the_regex_walk():
    """The symboliser decides pre-token starts in one pass; the oracle walks the GPT-2 regex alternatives match by
    match (oracle/bpe_oracle.c, checked against the library in tests/test_bpe_oracle.py).  Same starts on random
    texts dense in blanks, apostrophes, contraction letters and class changes."""
    from oracle.bpe_oracle import unicode_classes
    cls = unicode_classes(0x3000)
    rng = np.random.default_rng(11)
    pools = [
        np.array([32, 32, 32, 9, 10, 39, 39, ord("s"), ord("t"), ord("r"), ord("e"), ord("l"), ord("v"), ord("m"), ord("d"),
                  ord("a"), ord("7"), ord("!"), 133, 160, 178], dtype=np.uint16),
        np.arange(0, 256, dtype=np.uint16),
        np.concatenate([np.arange(0, 700, dtype=np.uint16), np.array([0x2000, 0x2003, 0x2028, 0x1680], dtype=np.uint16)]),
    ]
    checked = 0
    for pool in pools:
        for _ in range(1500):
            n = int(rng.integers(0, 40))
            cp = pool[rng.integers(0, len(pool), size=n)]
            want = pretokenize(cp) if n else np.zeros(0, dtype=np.uint8)
            got = _single_pass_word_starts(cp, cls)
            if n:
                assert got[0] == 1
                want = want.copy()
                want[0] = 1                                  # the oracle may leave position 0 implicit
            np.testing.assert_array_equal(got, want, err_msg=str(cp.tolist()))
            checked += n
    assert checked > 50_000
