"""ctypes wrapper of oracle/bpe_oracle.c (see that file for scope and citations).
TEST INFRASTRUCTURE ONLY."""
import ctypes as C
import json

import numpy as np

from . import build_oracle

_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build_oracle.build())
        _lib.bpe_oracle_train.restype = C.c_int
        _lib.bpe_oracle_train.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int, C.c_int,
                                          C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.POINTER(C.c_int32),
                                          C.POINTER(C.c_int32)]
        _lib.bpe_oracle_train_ex.restype = C.c_int
        _lib.bpe_oracle_train_ex.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_int64, C.c_int64, C.c_int,
                                             C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                             C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
        _lib.bpe_oracle_model_new.restype = C.c_void_p
        _lib.bpe_oracle_model_new.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int]
        _lib.bpe_oracle_model_free.argtypes = [C.c_void_p]
        _lib.bpe_oracle_encode.restype = C.c_int
        _lib.bpe_oracle_encode.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
        _lib.bpe_oracle_encode_batch.restype = C.c_int64
        _lib.bpe_oracle_encode_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_int64,
                                                 C.c_void_p]
        _lib.bpe_oracle_decode.restype = C.c_int
        _lib.bpe_oracle_decode.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int]
        _lib.bpe_oracle_pretokenize.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        _lib.bpe_oracle_set_classes.argtypes = [C.c_void_p, C.c_int]
        tab = unicode_classes(0xD800)
        _lib.bpe_oracle_set_classes(tab.ctypes.data, len(tab))
    return _lib


# letters added after Python 3.12's Unicode 15.0 that the library's regex engine already knows
_NEWER_LETTERS = (7305, 7306, 42955, 42956, 42957, 42970, 42971, 42972)
_WHITE_SPACE = {9, 10, 11, 12, 13, 32, 133, 160, 5760, 8232, 8233, 8239, 8287, 12288} | set(range(8192, 8203))


def unicode_classes(n):
    """0 = other, 1 = \\p{L}, 2 = \\p{N}, 3 = \\s for codepoints < n (SURVEY.md Appendix A.2, extended past
    Latin-1; checked codepoint by codepoint against the library's pre-tokenizer in tests/test_bpe_oracle.py)."""
    import unicodedata
    tab = np.zeros(n, dtype=np.uint8)
    for c in range(n):
        if c in _WHITE_SPACE:
            tab[c] = 3
        else:
            k = unicodedata.category(chr(c))[0]
            tab[c] = 1 if k == "L" else 2 if k == "N" else 0
    for c in _NEWER_LETTERS:
        if c < n:
            tab[c] = 1
    return tab


class OracleBPE:
    """Vocabulary (byte-level character strings in id order) + merges [(a, b, new_id)]."""

    def __init__(self, vocab_off, vocab_chars, merges):
        self.vocab_off = np.ascontiguousarray(vocab_off, dtype=np.int32)
        self.vocab_chars = np.ascontiguousarray(vocab_chars, dtype=np.uint16)
        self.merges = np.ascontiguousarray(merges, dtype=np.int32).reshape(-1, 3)
        self._model = None

    # ---- construction
    @classmethod
    def train(cls, bins, vocab_size, min_frequency=2):
        bins = np.ascontiguousarray(bins, dtype=np.int64)
        assert bins.ndim == 2
        min_token, max_token = int(bins.min()), int(bins.max())
        cap_v = max(vocab_size, 512)
        off = np.zeros(cap_v + 1, dtype=np.int32)
        cap = 4 * 1024 * 1024
        chars = np.zeros(cap, dtype=np.uint16)
        merges = np.zeros(3 * cap_v, dtype=np.int32)
        nv, nm = C.c_int32(0), C.c_int32(0)
        rc = lib().bpe_oracle_train(bins.ctypes.data, bins.shape[0], bins.shape[1], min_token, max_token, vocab_size,
                                    min_frequency, off.ctypes.data, chars.ctypes.data, cap, merges.ctypes.data,
                                    C.byref(nv), C.byref(nm))
        if rc != 0:
            raise RuntimeError(f"bpe_oracle_train failed: {rc}")
        o = cls(off[:nv.value + 1].copy(), chars[:off[nv.value]].copy(), merges[:3 * nm.value].copy())
        o.min_token, o.max_token = min_token, max_token
        return o

    @classmethod
    def train_ragged(cls, sequences, vocab_size, min_frequency=2, special_tokens=()):
        """FIGBPE.fit_from_sequences in full: sequences of unequal length, BpeTrainer special tokens."""
        rows = [np.asarray(r, dtype=np.int64).reshape(-1) for r in sequences]
        rows = [r for r in rows if r.size]
        flat = np.ascontiguousarray(np.concatenate(rows))
        row_off = np.zeros(len(rows) + 1, dtype=np.int64)
        np.cumsum([r.size for r in rows], out=row_off[1:])
        min_token, max_token = int(flat.min()), int(flat.max())
        sp_off = np.zeros(len(special_tokens) + 1, dtype=np.int32)
        sp_chars = []
        for i, t in enumerate(special_tokens):
            sp_chars.extend(ord(c) for c in t)
            sp_off[i + 1] = len(sp_chars)
        sp_chars = np.asarray(sp_chars or [0], dtype=np.uint16)
        cap_v = max(vocab_size, 512) + len(special_tokens)
        off = np.zeros(cap_v + 1, dtype=np.int32)
        cap = 4 * 1024 * 1024
        chars = np.zeros(cap, dtype=np.uint16)
        merges = np.zeros(3 * cap_v, dtype=np.int32)
        nv, nm = C.c_int32(0), C.c_int32(0)
        rc = lib().bpe_oracle_train_ex(flat.ctypes.data, len(rows), 0, row_off.ctypes.data, min_token, max_token,
                                       vocab_size, min_frequency, len(special_tokens), sp_off.ctypes.data,
                                       sp_chars.ctypes.data, off.ctypes.data, chars.ctypes.data, cap,
                                       merges.ctypes.data, C.byref(nv), C.byref(nm))
        if rc != 0:
            raise RuntimeError(f"bpe_oracle_train_ex failed: {rc}")
        o = cls(off[:nv.value + 1].copy(), chars[:off[nv.value]].copy(), merges[:3 * nm.value].copy())
        o.min_token, o.max_token = min_token, max_token
        return o

    @classmethod
    def from_strings(cls, vocab, merges_txt_lines):
        """vocab: {token string: id}; merges: ["a b", ...] (byte-level character strings)."""
        by_id = sorted(vocab.items(), key=lambda kv: kv[1])
        assert [i for _, i in by_id] == list(range(len(by_id)))
        off, chars = [0], []
        for tok, _ in by_id:
            chars.extend(ord(c) for c in tok)
            off.append(len(chars))
        merges = []
        for line in merges_txt_lines:
            a, b = line.split(" ")
            merges.append((vocab[a], vocab[b], vocab[a + b]))
        return cls(off, chars, merges)

    # ---- views
    def token_strings(self):
        return ["".join(map(chr, self.vocab_chars[self.vocab_off[i]:self.vocab_off[i + 1]]))
                for i in range(len(self.vocab_off) - 1)]

    def vocab_dict(self):
        return {t: i for i, t in enumerate(self.token_strings())}

    def merges_lines(self):
        toks = self.token_strings()
        return [f"{toks[a]} {toks[b]}" for a, b, _ in self.merges]

    def vocab_json(self):
        """Exactly the bytes HF's save_model writes: compact JSON in id order, non-ASCII unescaped."""
        return json.dumps(self.vocab_dict(), ensure_ascii=False, separators=(",", ":"))

    def merges_txt(self):
        return "#version: 0.2\n" + "".join(l + "\n" for l in self.merges_lines())

    # ---- apply
    def _m(self):
        if self._model is None:
            self._model = lib().bpe_oracle_model_new(self.vocab_off.ctypes.data, self.vocab_chars.ctypes.data,
                                                     len(self.vocab_off) - 1, self.merges.ctypes.data, len(self.merges))
        return self._model

    def encode(self, shifted):
        shifted = np.ascontiguousarray(shifted, dtype=np.int64)
        out = np.zeros(3 * len(shifted) + 3, dtype=np.int32)
        n = lib().bpe_oracle_encode(self._m(), shifted.ctypes.data, len(shifted), out.ctypes.data)
        return out[:n].tolist()

    def encode_batch(self, shifted):
        """Rows [N, L] of shifted bins -> (ids int32, offsets int64 [N + 1]): encode() of every row in one call."""
        shifted = np.ascontiguousarray(shifted, dtype=np.int64)
        n, L = shifted.shape
        width = 1 if n == 0 or shifted.max() < 0x80 else 2 if shifted.max() < 0x800 else 3   # ids <= UTF-8 bytes
        ids = np.zeros(max(width * n * L, 1), dtype=np.int32)
        off = np.zeros(n + 1, dtype=np.int64)
        total = lib().bpe_oracle_encode_batch(self._m(), shifted.ctypes.data, n, L, ids.ctypes.data, ids.size,
                                              off.ctypes.data)
        if total < 0:
            raise RuntimeError("bpe_oracle_encode_batch: id buffer too small")
        return ids[:total], off

    def decode(self, ids, cap=4096):
        ids = np.ascontiguousarray(ids, dtype=np.int32)
        out = np.zeros(cap, dtype=np.int64)
        n = lib().bpe_oracle_decode(self._m(), ids.ctypes.data, len(ids), out.ctypes.data, cap)
        if n < 0:
            raise ValueError(f"bpe_oracle_decode failed: {n}")
        return out[:n]

    def __del__(self):
        try:
            if self._model is not None:
                lib().bpe_oracle_model_free(self._model)
        except Exception:
            pass


def pretokenize(codepoints):
    cp = np.ascontiguousarray(codepoints, dtype=np.uint16)
    ws = np.zeros(len(cp), dtype=np.uint8)
    lib().bpe_oracle_pretokenize(cp.ctypes.data, len(cp), ws.ctypes.data)
    return ws
