"""BPE apply kernels (csrc/bpe.cu) row by row against host references, at every launch geometry they take.

encode: bpe_encode_warp_kernel (lane-per-word and cooperative long-word paths) and bpe_encode_kernel (one thread per
sequence) against the C oracle's encode (SURVEY.md A.5); decode: bpe_decode_token_kernel<2|6>, bpe_decode_warp_kernel and
bpe_decode_kernel against Python's strict UTF-8 decoder over the token strings (A.6, the HF ByteLevel decoder).  The
tables come from the oracle's trainer, so no GPU trainer runs here.  The warp-per-sequence kernels are grid-capped and
stride over the rows: every case runs at least three passes of each such launch (a warp decodes or encodes a second
and third sequence with the shared memory of the first), at 8, 4, 2 and 1 warps per CTA, odd L and L not a multiple
of 32, with 1-, 2- and 3-byte UTF-8 symbols.  Run on the B200 box:  pytest -m gpu."""
import codecs
import ctypes as C

import numpy as np
import pytest
import torch

from oracle.bpe_oracle import OracleBPE

pytestmark = pytest.mark.gpu

OFFSET = 3                               # min_token: bins are codepoints + OFFSET


def apply_shape(kernel, L, max_shift):
    """(warps per CTA, CTA cap) the library launches kernel 0 = encode, 1 = decode per-token, 2 = decode byte-level with."""
    from beast_tokenizer_b200 import _lib
    w, c = C.c_int32(0), C.c_int64(0)
    _lib.check(_lib.load().bpe_apply_shape(kernel, L, max_shift, C.byref(w), C.byref(c)), "bpe_apply_shape")
    return w.value, c.value


def rows_for(passes_of, tail=37):
    """At least three full passes of every listed (warps, ctas) launch, plus a ragged tail."""
    return 3 * max(w * c for w, c in passes_of) + tail


# ------------------------------------------------------------------ models (trained by the oracle)
SETS = {
    # letters, digits, other, blanks, highest codepoint (the alphabet is chr(0 .. R))
    1: ("aaabbbcdeestlvrm", "0123", "!?-", " \t", 0x7F),
    2: ("aabbcst" + "".join(map(chr, range(0x3B1, 0x3B6))) + "àáâ", "01" + "٠١٢", "!-" + chr(0x7FF), "  " + chr(0xA0), 0x7FF),
    3: ("aabst" + "".join(map(chr, range(0x800, 0x808))) + "".join(map(chr, range(0x904, 0x90A))), "01", "!-", "  ", 0xA00),
    # 2-byte symbols below U+0100 where continuation bytes 0x80..0x8F never occur in training: their bins are dropped
    "drop": ("abcst" + "".join(map(chr, range(0x90, 0xA0))), "01", "!", " ", 0xBF),
}


CONTRACTIONS = ["s", "t", "m", "d", "re", "ve", "ll"]


def text_rows(kind, n, L, rng):
    """Rows of L codepoints cut from one stream of words: runs of one class (geometric lengths, some long), blanks,
    contractions."""
    pools = SETS[kind][:4]
    table = np.zeros((5, max(map(len, pools))), dtype=np.int64)
    for k, pool in enumerate(pools):
        table[k, :len(pool)] = [ord(c) for c in pool]
    sizes = np.array([len(p) for p in pools] + [1])
    contr = np.zeros((len(CONTRACTIONS), 3), dtype=np.int64)
    for i, c in enumerate(CONTRACTIONS):
        contr[i, :1 + len(c)] = [39] + [ord(x) for x in c]
    K = n * L // 3 + 64                                          # words: mean length above 3
    k = rng.choice(5, K, p=[0.5, 0.15, 0.1, 0.1, 0.15])
    ci = rng.integers(0, len(CONTRACTIONS), K)
    ln = np.where(k == 0, rng.geometric(0.12, K), rng.geometric(0.4, K))
    ln = np.where(k == 4, [1 + len(CONTRACTIONS[i]) for i in ci], ln)
    word = np.repeat(np.arange(K), ln)[:n * L]
    assert word.size == n * L
    pos = np.arange(word.size) - (np.cumsum(ln) - ln)[word]
    kw = k[word]
    pick = (rng.random(word.size) * sizes[kw]).astype(np.int64)
    cps = np.where(kw == 4, contr[ci[word], np.minimum(pos, 2)], table[np.minimum(kw, 3), pick])
    return cps.reshape(n, L)


_MODELS = {}


def model(kind, truncate_to_two_chars=False):
    """(oracle, device model, R).  truncate_to_two_chars: only the merges before the first token of three characters
    (the decode kernel's 8-byte table entries, slots = 2)."""
    key = (kind, truncate_to_two_chars)
    if key in _MODELS:
        return _MODELS[key]
    from beast_tokenizer_b200 import B200ByteLevelBPE
    rng = np.random.default_rng({1: 11, 2: 12, 3: 13, "drop": 14}[kind])
    R = SETS[kind][4]
    cps = text_rows(kind, 3000, 60, rng)
    cps[0, 0], cps[1, 0] = 0, R                                  # the whole range occurs
    if kind == "drop":
        assert not ((cps >= 0x80) & (cps < 0x90)).any()
    o = OracleBPE.train(cps + OFFSET, 300 if kind == 1 else R + 300)
    assert (o.min_token, o.max_token) == (OFFSET, OFFSET + R)
    if truncate_to_two_chars:
        toks = o.token_strings()
        n_chars = lambda t: sum(1 for b in token_bytes(t) if (b & 0xC0) != 0x80)
        k = next(i for i, (_, _, c) in enumerate(o.merges) if n_chars(toks[c]) > 2)
        n_vocab = int(o.merges[k, 2])                            # the first new token of 3 characters: ids below it stay
        o = OracleBPE(o.vocab_off[:n_vocab + 1], o.vocab_chars[:o.vocab_off[n_vocab]], o.merges[:k])
        o.min_token, o.max_token = OFFSET, OFFSET + R
    dm = B200ByteLevelBPE.from_vocab_merges(o.vocab_dict(), [tuple(m.split(" ")) for m in o.merges_lines()])
    _MODELS[key] = (o, dm, R)
    return _MODELS[key]


# ------------------------------------------------------------------ host decode reference
def _b2u():
    bs = list(range(33, 127)) + list(range(161, 173)) + list(range(174, 256))
    cs, n = bs[:], 0
    for b in range(256):
        if b not in bs:
            bs.append(b)
            cs.append(256 + n)
            n += 1
    return {chr(c): b for b, c in zip(bs, cs)}


U2B = _b2u()


def token_bytes(t):
    """HF ByteLevel decoder: a token maps char by char to bytes; one holding a character outside the map gives its UTF-8."""
    return bytes(U2B[c] for c in t) if all(c in U2B for c in t) else t.encode("utf-8")


def ref_decode(ids, L, tb):
    """(status, decoded length, codepoints) with the kernels' error order: the byte stream ends at the first id out of
    range; invalid UTF-8 before it -> 2 (so does a character above U+FFFF: no shifted bin), else the bad id -> 1, else a
    character cut off at the end -> 2, else a length != L -> 3."""
    bad = next((k for k, t in enumerate(ids) if not 0 <= t < len(tb)), len(ids))
    data = b"".join(tb[t] for t in ids[:bad])
    try:
        text, used = codecs.utf_8_decode(data, "strict", False)
    except UnicodeDecodeError:
        return 2, None, None
    cps = [ord(c) for c in text]
    if any(c > 0xFFFF for c in cps):
        return 2, None, None
    if bad < len(ids):
        return 1, None, None
    if used < len(data):
        return 2, None, None
    return (3 if len(cps) != L else 0), len(cps), cps


# ------------------------------------------------------------------ encode
def planted_rows(kind, L, rng):
    """Rows the kernels' boundaries live on: single-class words of kCoopWord - 1 .. + 1 (23..25), 32, 33, 64 symbols and
    whole-row words at several offsets; contractions straddling each lane's slice of P = ceil(L / 32) codepoints."""
    letters, digits, _, _, _ = SETS[kind]
    P = (L + 31) // 32
    rows = []
    for wl in (23, 24, 25, 32, 33, 64, L):
        for start in (0, 1, P - 1, L - wl):
            if wl > L or not 0 <= start <= L - wl:
                continue
            for pool in (letters, digits, letters[:1]):
                row = text_rows(kind, 1, L, rng)[0]
                row[start:start + wl] = [ord(pool[int(i)]) for i in rng.integers(0, len(pool), wl)]
                if start > 0:
                    row[start - 1] = 32
                if start + wl < L:
                    row[start + wl] = ord("!")
                rows.append(row)
    for c in ("s", "t", "re", "ll", "ve"):
        for shift in (-3, -2, -1, 0, 1):
            row = text_rows(kind, 1, L, rng)[0]
            for j in range(1, 32):
                q = j * P + shift
                if 1 <= q and q + len(c) < L:
                    row[q - 1] = ord(letters[0]) if j % 2 else 32
                    row[q:q + 1 + len(c)] = [39] + [ord(x) for x in c]
            rows.append(row)
    return np.stack(rows)


# (kind, L, warps per CTA the warp kernel must run with)
ENCODE_CASES = [(1, 140, 8), (1, 141, 8), (1, 3001, 4), (1, 5001, 2), (1, 7777, 1),
                (2, 141, 8), (2, 100, 8), (2, 1600, 4), (2, 3001, 2), (2, 4096, 1),
                (3, 97, 8), (3, 1201, 4), (3, 2047, 2), (3, 2730, 1),
                ("drop", 141, 8)]


def encode_rows(kind, L, n, rng, R):
    bins = np.concatenate([planted_rows(kind, L, rng), text_rows(kind, n, L, rng)])[:n]
    if kind == "drop":                                           # bins whose continuation byte has no symbol
        m = rng.random(bins.shape) < 0.05
        bins[m] = rng.integers(0x80, 0x90, int(m.sum()))
    bins = bins + OFFSET
    status = np.zeros(n, dtype=np.int32)
    for i in range(5, n, 97):                                    # out-of-range rows between good ones
        s = 1 + (i // 97) % 3
        pos = rng.choice(L, 2, replace=False)
        if s & 1:
            bins[i, pos[0]] = OFFSET - 1
        if s & 2:
            bins[i, pos[1]] = OFFSET + R + 1
        status[i] = s
    return bins, status


def check_encode(dm, o, bins, want_status, R):
    flat, offsets, status = dm.encode_bins(torch.from_numpy(bins).cuda(), OFFSET, OFFSET + R)
    torch.cuda.synchronize()
    flat, offsets, status = flat.cpu().numpy(), offsets.cpu().numpy(), status.cpu().numpy()
    assert np.array_equal(status, want_status), np.flatnonzero(status != want_status)[:10]
    good = np.flatnonzero(want_status == 0)
    ids, off = o.encode_batch(bins[good] - OFFSET)
    want_len = np.zeros(len(bins), dtype=np.int64)
    want_len[good] = np.diff(off)
    got_len = np.diff(offsets)
    bad = np.flatnonzero(got_len != want_len)
    assert bad.size == 0, f"{bad.size} rows differ in length, first {bad[:10]}"
    if not np.array_equal(flat, ids):
        first = int(np.argmax(flat != ids))
        row = int(np.searchsorted(offsets, first, side="right") - 1)
        pytest.fail(f"ids differ from row {row} on: got {flat[offsets[row]:offsets[row + 1]].tolist()[:40]}, "
                    f"want {o.encode(bins[row] - OFFSET)[:40]}")
    return flat, offsets


@pytest.mark.parametrize("kind,L,warps", ENCODE_CASES)
def test_encode_every_row_equals_the_oracle(kind, L, warps):
    o, dm, R = model(kind)
    w, ctas = apply_shape(0, L, R)
    assert w == warps
    n = rows_for([(w, ctas)])
    rng = np.random.default_rng(L * 7 + len(str(kind)))
    bins, status = encode_rows(kind, L, n, rng, R)
    assert len(bins) >= 3 * w * ctas                              # three passes of the persistent grid, at least
    check_encode(dm, o, bins, status, R)


@pytest.mark.parametrize("kind,L", [(1, 141), (2, 1600), (3, 2730), ("drop", 100)])
def test_encode_hashed_rank_table_every_row(kind, L, monkeypatch):
    """Vocabularies above DENSE_RANK_VOCAB keep the merge ranks in a hash of the merges; forced on these models."""
    from beast_tokenizer_b200 import B200ByteLevelBPE, bpe_model
    o, dm, R = model(kind)
    monkeypatch.setattr(bpe_model, "DENSE_RANK_VOCAB", 0)
    hashed = B200ByteLevelBPE(dm.tokens, dm.merges)
    w, ctas = apply_shape(0, L, R)
    n = rows_for([(w, ctas)])
    bins, status = encode_rows(kind, L, n, np.random.default_rng(L), R)
    assert len(bins) >= 3 * w * ctas
    check_encode(hashed, o, bins, status, R)
    assert hashed._tables(torch.device("cuda", torch.cuda.current_device()))["hash_bits"] > 0


@pytest.mark.parametrize("kind,L", [(1, 141), (3, 97), (2, 1600)])
def test_encode_thread_kernel_every_row(kind, L, monkeypatch):
    """BEAST_B200_BPE_THREAD_ENCODE=1: one thread per sequence, rows staged per CTA — over many CTAs."""
    o, dm, R = model(kind)
    monkeypatch.setenv("BEAST_B200_BPE_THREAD_ENCODE", "1")
    rows_per_cta = min(256, (180 * 1024) // ((L + 1) * 2 + 4))
    n = 3000
    assert n > 8 * rows_per_cta
    bins, status = encode_rows(kind, L, n, np.random.default_rng(L + 1), R)
    check_encode(dm, o, bins, status, R)


# ------------------------------------------------------------------ decode
def byte_ids(dm):
    """id of the single-byte token of every byte value (None where the vocabulary has none)."""
    out = [None] * 256
    for i, t in enumerate(dm.tokens):
        b = token_bytes(t)
        if len(b) == 1 and out[b[0]] is None:
            out[b[0]] = i
    return out


def decode_rows(o, dm, R, L, kind, rng, n):
    """Valid rows (the oracle's ids of random text) and every class of garbage."""
    V = len(dm.tokens)
    tb = [token_bytes(t) for t in dm.tokens]
    by = byte_ids(dm)
    n_valid = max(64, n // 3)
    text = text_rows(kind, n_valid, L, rng)
    ids, off = o.encode_batch(text)
    valid = [ids[off[i]:off[i + 1]] for i in range(n_valid)]
    long_tok = [i for i in range(V) if sum(1 for b in tb[i] if (b & 0xC0) != 0x80) > 6]
    two = [i for i in range(V) if len(tb[i]) == 2 and (tb[i][0] & 0xE0) == 0xC0 and (tb[i][1] & 0xC0) == 0x80]

    def from_bytes(bs):
        return np.array([by[b] for b in bs], dtype=np.int64) if all(by[b] is not None for b in bs) else None

    rows, k = list(valid), 0
    while len(rows) < n:
        k += 1
        r = valid[k % n_valid]
        c = k % 17
        if c == 0:                                          # random ids, random length
            rows.append(rng.integers(0, V, int(rng.integers(0, 2 * L))))
        elif c == 1 and len(r):                             # one id replaced
            r = r.copy(); r[rng.integers(0, len(r))] = rng.integers(0, V); rows.append(r)
        elif c == 2 and len(r):                             # ids -1 / n_vocab / beyond at the start, inside, at the end
            r = r.copy(); r[[0, len(r) // 2, -1][k % 3]] = [-1, V, V + 7][(k // 3) % 3]; rows.append(r)
        elif c == 3:                                        # a negative id after garbage
            g = rng.integers(0, V, 20); g[rng.integers(0, 20)] = -1; rows.append(g)
        elif c == 4:                                        # truncated / extended valid rows
            rows.append(np.concatenate([r[:len(r) // 2], r[:int(rng.integers(0, 4))]]))
        elif c == 5:                                        # more bytes than any valid row: the overflow path
            rows.append(rng.integers(0, V, 4 * L + 65))
        elif c == 6:                                        # empty
            rows.append(np.zeros(0, dtype=np.int64))
        elif c == 7:                                        # 32 / 33 / 64 ids (one group of lanes, the look-ahead)
            rows.append(rng.integers(0, V, (32, 33, 64)[k % 3]))
        elif c == 8 and long_tok:                           # tokens of more than 6 characters
            rows.append(np.array(rng.choice(long_tok, max(1, L // 8)), dtype=np.int64))
        elif c == 9:                                        # valid rows at L's length from single bytes: every 2- / 3-byte
            bs = "".join(map(chr, text[k % n_valid])).encode("utf-8")   # character split across tokens
            x = from_bytes(bs)
            if x is not None:
                rows.append(x)
        elif c == 10:                                       # a stray continuation byte starts the row
            x = from_bytes(b"\x80" + "".join(map(chr, text[k % n_valid][1:])).encode("utf-8"))
            if x is not None:
                rows.append(x)
        elif c == 11:                                       # overlong / surrogate / above-U+FFFF forms in valid text
            bad = [b"\xe0\x80\x80", b"\xed\xa0\x80", b"\xc0\x80", b"\xc1\xbf", b"\xf0\x90\x80\x80", b"\xf4\x90\x80\x80",
                   b"\xe0\x9f\xbf", b"\xed\xbf\xbf", b"\xe0", b"\xed", b"\xf5"][(k // 17) % 11]
            s = "".join(map(chr, text[k % n_valid])).encode("utf-8")
            q = int(rng.integers(0, len(s) + 1))
            while q < len(s) and (s[q] & 0xC0) == 0x80:
                q += 1
            x = from_bytes(s[:q] + bad + s[q:])
            if x is not None:
                rows.append(x[:len(x) - (k % 2)])           # also with the last byte cut
        elif c == 12 and two:                               # 2-byte characters cut at ids 31 | 32 and 63 | 64
            cut = [by[t] for t in (tb[two[k % len(two)]][0], tb[two[k % len(two)]][1])]
            if None not in cut:
                fill = rng.choice([i for i in range(V) if len(tb[i]) == 1 and tb[i][0] < 0x80], 64)
                x = np.concatenate([fill[:31], cut, fill[31:61], cut, fill[61:63]])
                rows.append(x)
        elif c == 13:                                       # many ids out of range
            rows.append(rng.integers(-3, V + 3, int(rng.integers(1, 80))))
        else:
            rows.append(r)
    rows = [np.asarray(r, dtype=np.int64) for r in rows[:n]]
    return [rows[i] for i in rng.permutation(n)], tb          # garbage in every pass of every warp


def run_decode(dm, rows, L):
    flat = torch.from_numpy(np.concatenate(rows).astype(np.int32) if rows else np.zeros(0, np.int32)).cuda()
    offs = torch.from_numpy(np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.int64)).cuda()
    bins, st, ln = dm.decode_ids(flat, offs, L, OFFSET)
    torch.cuda.synchronize()
    return bins.cpu().numpy(), st.cpu().numpy(), ln.cpu().numpy()


def check_decode(dm, rows, L, tb):
    bins, st, ln = run_decode(dm, rows, L)
    want = [ref_decode(r.tolist(), L, tb) for r in rows]
    ws = np.array([w[0] for w in want])
    bad = np.flatnonzero(st != ws)
    assert bad.size == 0, f"{bad.size} statuses differ, first rows {bad[:8]}: got {st[bad[:8]]}, want {ws[bad[:8]]}"
    for i, (s, n, cps) in enumerate(want):
        if s in (0, 3):
            assert ln[i] == n, (i, ln[i], n)
        if s == 0:
            assert np.array_equal(bins[i], np.asarray(cps) + OFFSET), i
    return ws


# (kind, slots of the per-token table, L)
DECODE_CASES = [(2, 6, 140), (2, 6, 141), (3, 6, 97), (1, 6, 141), (2, 2, 141), (3, 2, 100), ("drop", 6, 141)]


@pytest.mark.parametrize("kind,slots,L", DECODE_CASES)
def test_decode_every_row_equals_the_host_decoder(kind, slots, L):
    o, dm, R = model(kind, truncate_to_two_chars=slots == 2)
    dev = torch.device("cuda", torch.cuda.current_device())
    assert dm._tables(dev)["tab_slots"] == slots
    tw, tc = apply_shape(1, L, R)
    bw, bc = apply_shape(2, L, R)
    assert tw == 8 and bw >= 1
    n = rows_for([(tw, tc), (bw, bc)])
    rows, tb = decode_rows(o, dm, R, L, kind, np.random.default_rng(L + slots), n)
    assert len(rows) >= 3 * max(tw * tc, bw * bc)
    ws = check_decode(dm, rows, L, tb)
    assert ({0, 1, 3} if kind == 1 else {0, 1, 2, 3}) <= set(ws.tolist())     # ASCII tokens cannot form invalid UTF-8
    third = ws[2 * bw * bc:3 * bw * bc]                          # rows the byte-level kernel takes in its third pass
    assert ((third == 1) | (third == 2)).mean() > 0.05


def test_decode_thread_kernel_every_row(monkeypatch):
    """BEAST_B200_BPE_THREAD_DECODE=1: the sequential one-thread-per-sequence decoder, same rows, same answers."""
    o, dm, R = model(3)
    monkeypatch.setenv("BEAST_B200_BPE_THREAD_DECODE", "1")
    rows, tb = decode_rows(o, dm, R, 141, 3, np.random.default_rng(5), 20000)
    ws = check_decode(dm, rows, 141, tb)
    assert {0, 1, 2, 3} <= set(ws.tolist())


def test_decode_beyond_the_token_path_length():
    """L = 8193: the per-token kernel stops at 8192 bins, the byte-level kernel decodes every row alone (4 warps per
    CTA here).  Valid ids come from the oracle, which has no length limit."""
    o, dm, R = model(2)
    L = 8193
    assert apply_shape(1, L, R)[0] == 0
    bw, bc = apply_shape(2, L, R)
    assert bw < 8
    n = rows_for([(bw, bc)])
    rows, tb = decode_rows(o, dm, R, L, 2, np.random.default_rng(8193), n)
    assert len(rows) >= 3 * bw * bc
    ws = check_decode(dm, rows, L, tb)
    assert {0, 1, 2, 3} <= set(ws.tolist())


def test_overlong_and_surrogate_forms_are_invalid_in_every_decoder(monkeypatch):
    """E0 80 80 (overlong U+0000), ED A0 80 (a surrogate), C0 80, F4 90 80 80: strict UTF-8 rejects them, so the id
    stream does not decode to text (status 2) — in the per-token, the byte-level and the one-thread decoders, whether
    the form sits inside one token or is split after its lead."""
    o, dm, R = model(3)
    by = byte_ids(dm)
    tb = [token_bytes(t) for t in dm.tokens]
    L = 3
    ok = [by[b] for b in b"abc"]
    rows = [np.array(ok, dtype=np.int64)]
    for form in (b"\xe0\x80\x80", b"\xed\xa0\x80", b"\xc0\x80", b"\xf4\x90\x80\x80", b"\xe0\x9f\xbf", b"\xed\xbf\xbf"):
        x = [by[b] for b in form]
        rows += [np.array(ok[:2] + x, dtype=np.int64), np.array(x + ok[:2], dtype=np.int64)]
    for form in (b"\xe0\xa0\x80", b"\xed\x9f\xbf"):                        # the nearest valid forms
        rows.append(np.array(ok[:2] + [by[b] for b in form], dtype=np.int64))
    for mode in ("0", "1"):
        monkeypatch.setenv("BEAST_B200_BPE_THREAD_DECODE", mode)
        ws = check_decode(dm, rows, L, tb)
        assert ws.tolist() == [0] + [2] * 12 + [0, 0]


@pytest.mark.parametrize("slots", [2, 6])
def test_three_byte_lead_completed_by_the_next_token(slots, monkeypatch):
    """A token that ends in a bare 3-byte lead (E0, ED), the next token's two continuation bytes finishing the
    character: the per-token path hands such rows to the byte-level kernel, which must reject what strict UTF-8 rejects
    (E0 80 80 -> U+0000 is overlong, ED A0 80 is a surrogate) and keep what it accepts (E0 A0 80 = U+0800,
    ED 9F BF = U+D7FF).  A hand-made vocabulary: the 256 single bytes plus such pairs of tokens (and a 3-character
    token for the 6-slot table)."""
    from beast_tokenizer_b200 import B200ByteLevelBPE
    b2u = {b: c for c, b in U2B.items()}
    chars = lambda bs: "".join(b2u[b] for b in bs)
    extra = [b"A\xe0", b"A\xed", b"\x80\x80", b"\xa0\x80", b"\x9f\xbf", b"\xbf\xbf", b"\xa0\x80B"]
    if slots == 6:
        extra.append(b"abc")
    vocab = [chars(bytes([b])) for b in range(256)] + [chars(bs) for bs in extra]
    dm = B200ByteLevelBPE(vocab, [])
    assert dm._tables(torch.device("cuda", torch.cuda.current_device()))["tab_slots"] == slots
    tb = [token_bytes(t) for t in dm.tokens]
    tid = {bs: 256 + i for i, bs in enumerate(extra)}
    pairs = [(b"A\xe0", b"\x80\x80", 2), (b"A\xe0", b"\xa0\x80", 0), (b"A\xed", b"\xa0\x80", 2), (b"A\xed", b"\x9f\xbf", 0),
             (b"A\xed", b"\xbf\xbf", 2), (b"A\xe0", b"\x9f\xbf", 2), (b"A\xe0", b"\xa0\x80B", 3)]
    rows, want = [], []
    for a, b, st in pairs:
        for pre in (0, 31, 63):                           # the pair inside a lane group and across lanes 31 | 32, 63 | 64
            rows.append(np.array([ord("z")] * pre + [tid[a], tid[b]], dtype=np.int64))
            want.append(st if st != 0 or pre == 0 else 3)
    for mode in ("0", "1"):
        monkeypatch.setenv("BEAST_B200_BPE_THREAD_DECODE", mode)
        ws = check_decode(dm, rows, 2, tb)
        assert ws.tolist() == want
