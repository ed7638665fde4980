"""Byte-level BPE model (vocabulary + merge table) with device-side tables for the K5 kernels.

Stands in for HF `tokenizers.ByteLevelBPETokenizer` as used by the reference
(beast/beast_bpe_trainer.py:61-74, beast/beast_bspline_bpe_tokenizer.py:175-247, 336-388): same
vocab.json / merges.txt / tokenizer.json files, same ids.  Applying the model (ids <-> bins) runs
on the GPU through libbeast_b200.so (bpe_encode / bpe_decode); there is no host implementation.
"""
import json
import os
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib


def bytes_to_unicode() -> List[int]:
    """GPT-2 byte -> character map of the ByteLevel pre-tokenizer (SURVEY.md Appendix A.3): printable
    bytes map to themselves, the other 68 to U+0100.. in byte order."""
    out, n = [], 0
    for b in range(256):
        if 33 <= b <= 126 or 161 <= b <= 172 or 174 <= b <= 255:
            out.append(b)
        else:
            out.append(256 + n)
            n += 1
    return out


B2U = bytes_to_unicode()
U2B = {c: b for b, c in enumerate(B2U)}

MAX_SHIFT = 0xD7FF                      # shifted bins are codepoints below the surrogate range
MAX_APPLY_VOCAB = 65535                 # token ids are 16 bits wide in the encode kernel
DENSE_RANK_VOCAB = 4096                 # up to here the merge ranks live in a dense V x V table (64 MB), beyond in a hash of the merges
# letters added to Unicode after Python 3.12's tables (15.0) that the reference's regex engine already knows
_NEWER_LETTERS = (7305, 7306, 42955, 42956, 42957, 42970, 42971, 42972)
_WHITE_SPACE = {9, 10, 11, 12, 13, 32, 133, 160, 5760, 8232, 8233, 8239, 8287, 12288} | set(range(8192, 8203))
_CLASS_TABLE = None


def class_table() -> np.ndarray:
    """uint8 [0xD800]: GPT-2 pre-tokenizer class of every codepoint (0 other, 1 \\p{L}, 2 \\p{N}, 3 \\s) from the
    Unicode general categories — what Oniguruma's \\p{L} / \\p{N} / \\s match (SURVEY.md Appendix A.2 extended
    beyond Latin-1 for tokenizers with more than 256 bins).  Entries below 256 are not read by the kernels."""
    global _CLASS_TABLE
    if _CLASS_TABLE is None:
        import unicodedata
        tab = np.zeros(MAX_SHIFT + 1, dtype=np.uint8)
        for c in range(MAX_SHIFT + 1):
            if c in _WHITE_SPACE:
                tab[c] = 3
            else:
                k = unicodedata.category(chr(c))[0]
                tab[c] = 1 if k == "L" else 2 if k == "N" else 0
        for c in _NEWER_LETTERS:
            tab[c] = 1
        _CLASS_TABLE = tab
    return _CLASS_TABLE


_CLASS_DEV = {}


def class_table_device(dev: torch.device) -> torch.Tensor:
    key = (dev.type, dev.index)
    if key not in _CLASS_DEV:
        _CLASS_DEV[key] = torch.from_numpy(class_table()).to(dev)
    return _CLASS_DEV[key]


def utf8_len(max_shift: int) -> int:
    return 1 if max_shift < 0x80 else 2 if max_shift < 0x800 else 3


def token_char_entry(tb: bytes):
    """One row of the decode kernel's per-token character table (csrc/bpe.cu: bpe_decode_warp_kernel fast path): what
    the sequential UTF-8 state machine of A.6 does with this token's bytes, precomputed.  Returns 4 x uint32:
    x, y, z = six 16-bit slots with the token's characters in order (the last one = the partial accumulator, already
    shifted by the missing continuation bytes, when the token ends inside a character); w = characters started | bytes still needed << 3 | leading continuation bytes << 5
    | slow << 7 | payload of the leading continuation bytes << 8 | ends in a bare E0 lead << 26 | ends in a bare ED
    lead << 27.  slow = the token cannot be described this way (more than 6 characters or 3 leading continuation bytes,
    an invalid or 4-byte lead, a stray continuation byte, an overlong or surrogate form): sequences holding it decode on
    the byte-level path, which also reports the reference's errors.  So do sequences holding a token that ends in a bare
    E0 / ED lead (bits 26 / 27): strict UTF-8 restricts the next byte (A0..BF / 80..9F), which lies in the next token.
    The entry still describes such a token; only the kernel's choice of path reads the two bits."""
    SLOW = (0, 0, 0, 0x80)
    i, lead_cont, lead_bits = 0, 0, 0
    while i < len(tb) and (tb[i] & 0xC0) == 0x80:
        lead_bits = (lead_bits << 6) | (tb[i] & 0x3F)
        lead_cont += 1
        i += 1
    if lead_cont > 3:
        return SLOW
    cps, pending, acc, lo, hi, last = [], 0, 0, 0x80, 0xBF, 0
    for b in tb[i:]:
        last = b
        if pending:
            if not lo <= b <= hi:
                return SLOW
            lo, hi = 0x80, 0xBF
            acc = (acc << 6) | (b & 0x3F)
            pending -= 1
            if pending == 0:
                cps.append(acc)
        elif b < 0x80:
            cps.append(b)
        elif 0xC2 <= b < 0xE0:     # C0 / C1 only start overlong forms
            acc, pending = b & 0x1F, 1
        elif 0xE0 <= b < 0xF0:
            acc, pending = b & 0x0F, 2
            lo, hi = (0xA0 if b == 0xE0 else 0x80), (0x9F if b == 0xED else 0xBF)
        else:                      # 4-byte leads decode above U+FFFF (never a shifted bin), 0xF8.. and stray
            return SLOW            # continuation bytes are invalid: the byte-level path reports them
    if pending:
        cps.append(acc << (6 * pending))            # pre-shifted: the kernel ORs the next token's leading payload in
    if len(cps) > 6 or any(c > 0xFFFF for c in cps):
        return SLOW
    slots = cps + [0] * (6 - len(cps))
    lead3 = (1 if last == 0xE0 else 2 if last == 0xED else 0) if pending == 2 else 0
    meta = len(cps) | (pending << 3) | (lead_cont << 5) | (lead_bits << 8) | (lead3 << 26)
    return (slots[0] | (slots[1] << 16), slots[2] | (slots[3] << 16), slots[4] | (slots[5] << 16), meta)


class Encoding:
    """Minimal stand-in for tokenizers.Encoding (only `.ids` is used by the reference)."""

    def __init__(self, ids):
        self.ids = ids


class B200ByteLevelBPE:
    """vocab: token strings (byte-level characters) in id order; merges: [(id_a, id_b, id_new)]."""

    def __init__(self, vocab: Sequence[str], merges: Sequence[Tuple[int, int, int]],
                 special_tokens: Sequence[str] = ()):
        # BpeTrainer special tokens of THIS training run (HF registers them as added tokens on the trained object;
        # a tokenizer reloaded from vocab.json / merges.txt — what the reference's from_pretrained does,
        # beast_bspline_bpe_tokenizer.py:379-382 — no longer knows them, and neither does from_file here).
        self.special_tokens: List[str] = list(dict.fromkeys(special_tokens))
        self.tokens: List[str] = list(vocab)
        self.merges: List[Tuple[int, int, int]] = [tuple(int(x) for x in m) for m in merges]
        self._vocab: Dict[str, int] = {t: i for i, t in enumerate(self.tokens)}
        self._dev_tables = {}

    # ------------------------------------------------------------------ construction / files
    @classmethod
    def from_vocab_merges(cls, vocab: Dict[str, int], merge_pairs: Sequence[Tuple[str, str]]):
        by_id = sorted(vocab.items(), key=lambda kv: kv[1])
        if [i for _, i in by_id] != list(range(len(by_id))):
            raise ValueError("vocabulary ids must be 0..n-1")
        merges = []
        for a, b in merge_pairs:
            if a not in vocab or b not in vocab or (a + b) not in vocab:
                raise ValueError(f"merge {a!r} {b!r} refers to tokens outside the vocabulary")
            merges.append((vocab[a], vocab[b], vocab[a + b]))
        return cls([t for t, _ in by_id], merges)

    @classmethod
    def from_file(cls, vocab_path: str, merges_path: str):
        """Same inputs as ByteLevelBPETokenizer.from_file (reference bpe_tokenizer.py:379-382)."""
        with open(vocab_path, encoding="utf-8") as f:
            vocab = json.load(f)
        pairs = []
        with open(merges_path, encoding="utf-8") as f:
            for i, line in enumerate(f.read().split("\n")):
                if (i == 0 and line.startswith("#version")) or not line:
                    continue
                a, b = line.split(" ")
                pairs.append((a, b))
        return cls.from_vocab_merges(vocab, pairs)

    @classmethod
    def from_hf(cls, tokenizer):
        """Import a trained HF ByteLevelBPETokenizer / Tokenizer (e.g. one the reference produced)."""
        inner = getattr(tokenizer, "_tokenizer", tokenizer)
        model = json.loads(inner.to_str())["model"]
        pairs = [tuple(m.split(" ")) if isinstance(m, str) else tuple(m) for m in model["merges"]]
        return cls.from_vocab_merges(model["vocab"], pairs)

    def to_hf(self):
        """A real tokenizers.ByteLevelBPETokenizer with this vocabulary (needs the `tokenizers` wheel)."""
        from tokenizers import ByteLevelBPETokenizer
        return ByteLevelBPETokenizer(vocab=dict(self._vocab), merges=[(a, b) for a, b in self.merge_strings()])

    def get_vocab(self) -> Dict[str, int]:
        return dict(self._vocab)

    def get_vocab_size(self) -> int:
        return len(self.tokens)

    def token_to_id(self, token: str) -> Optional[int]:
        return self._vocab.get(token)

    def id_to_token(self, i: int) -> Optional[str]:
        return self.tokens[i] if 0 <= i < len(self.tokens) else None

    def merge_strings(self) -> List[Tuple[str, str]]:
        return [(self.tokens[a], self.tokens[b]) for a, b, _ in self.merges]

    def vocab_json(self) -> str:
        """The bytes HF's save_model writes: compact JSON in id order, non-ASCII unescaped."""
        return json.dumps(self._vocab, ensure_ascii=False, separators=(",", ":"))

    def merges_txt(self) -> str:
        return "#version: 0.2\n" + "".join(f"{a} {b}\n" for a, b in self.merge_strings())

    def save_model(self, directory: str, prefix: Optional[str] = None) -> List[str]:
        name = (lambda n: f"{prefix}-{n}" if prefix else n)
        vp, mp = os.path.join(directory, name("vocab.json")), os.path.join(directory, name("merges.txt"))
        with open(vp, "w", encoding="utf-8") as f:
            f.write(self.vocab_json())
        with open(mp, "w", encoding="utf-8") as f:
            f.write(self.merges_txt())
        return [vp, mp]

    def tokenizer_json(self) -> str:
        """tokenizer.json exactly as ByteLevelBPETokenizer.save writes it (tokenizers 0.2x layout)."""
        bl = lambda prefix, trim: {"type": "ByteLevel", "add_prefix_space": prefix, "trim_offsets": trim,
                                   "use_regex": True}
        doc = {
            "version": "1.0", "truncation": None, "padding": None,
            "added_tokens": [{"id": self._vocab[t], "content": t, "single_word": False, "lstrip": False, "rstrip": False,
                              "normalized": False, "special": True} for t in self.special_tokens],
            "normalizer": None,
            "pre_tokenizer": bl(False, True), "post_processor": bl(True, False), "decoder": bl(True, True),
            "model": {"type": "BPE", "dropout": None, "unk_token": None, "continuing_subword_prefix": None,
                      "end_of_word_suffix": None, "fuse_unk": False, "byte_fallback": False, "ignore_merges": False,
                      "vocab": self._vocab, "merges": [list(p) for p in self.merge_strings()]},
        }
        return json.dumps(doc, indent=2, ensure_ascii=False)

    def save(self, path: str, pretty: bool = True):
        with open(path, "w", encoding="utf-8") as f:
            f.write(self.tokenizer_json())

    # ------------------------------------------------------------------ device tables
    def token_bytes(self, i: int) -> bytes:
        return bytes(U2B[ord(c)] for c in self.tokens[i] if ord(c) in U2B)

    def _tables(self, dev: torch.device):
        key = (dev.type, dev.index)
        if key in self._dev_tables:
            return self._dev_tables[key]
        V = len(self.tokens)
        if V > MAX_APPLY_VOCAB:
            raise _lib.BeastB200Error(f"BPE vocabulary of {V} entries: token ids are 16 bits wide in the encode / decode kernels "
                                      f"(up to {MAX_APPLY_VOCAB} entries)")
        b2i = np.full(256, -1, dtype=np.int16)
        for b in range(256):
            b2i[b] = self._vocab.get(chr(B2U[b]), -1)
        if V <= DENSE_RANK_VOCAB:
            hash_bits = 0
            rank = np.full(V * V, 0xFFFFFFFF, dtype=np.uint32)
            for r, (a, b, c) in enumerate(self.merges):
                k = a * V + b
                if rank[k] == 0xFFFFFFFF:
                    rank[k] = (r << 16) | c
        else:
            # large vocabularies: an open-addressing hash of the merges only (O(#merges) memory; the dense table would
            # take 4 V^2 bytes — 4.3 GB at V = 32 768); same slot function and probing as csrc/bpe.cu: rank_lookup
            if len(self.merges) > 0xFFFE:
                raise _lib.BeastB200Error("more than 65 534 merges do not fit the 16-bit rank field of the encode kernel")
            hash_bits = max(10, int(2 * max(len(self.merges), 1) - 1).bit_length())
            size, mask = 1 << hash_bits, (1 << hash_bits) - 1
            table = np.full((size, 2), 0xFFFFFFFF, dtype=np.uint32)
            for r, (a, b, c) in enumerate(self.merges):
                key = (a << 16) | b
                slot = ((key * 0x9E3779B1) & 0xFFFFFFFF) >> (32 - hash_bits)
                while table[slot, 0] != 0xFFFFFFFF and table[slot, 0] != key:
                    slot = (slot + 1) & mask
                if table[slot, 0] == 0xFFFFFFFF:              # the first rule of a pair wins, as in the dense table
                    table[slot] = (key, (r << 16) | c)
            rank = table.reshape(-1)
        off = np.zeros(V + 1, dtype=np.int32)
        chunks = []
        special_ids = {self._vocab[t] for t in self.special_tokens}
        for i in range(V):
            if i in special_ids:                  # decode(skip_special_tokens=True), the library's default: no bytes
                chunks.append(b"")
                off[i + 1] = off[i]
                continue
            # HF's ByteLevel decoder maps characters back to bytes; a token holding any other
            # character (the unused raw chr(i) alphabet entries) contributes its own UTF-8 bytes
            tok = self.tokens[i]
            tb = bytes(U2B[ord(c)] for c in tok) if all(ord(c) in U2B for c in tok) else tok.encode("utf-8")
            chunks.append(tb)
            off[i + 1] = off[i] + len(tb)
        blob = np.frombuffer(b"".join(chunks) or b"\x00", dtype=np.uint8).copy()
        tab = np.stack([token_char_entry(tb) for tb in chunks]).astype(np.uint32)
        slots = 6
        fits2 = ((tab[:, 3] & 0x80) != 0) | ((tab[:, 3] & 7) <= 2)
        if bool(fits2.all()):                     # at most two characters per token: 8-byte entries {c0 | c1 << 16, meta}
            tab, slots = np.ascontiguousarray(tab[:, [0, 3]]), 2
        t = dict(V=V, hash_bits=hash_bits, b2i=torch.from_numpy(b2i).to(dev), rank=torch.from_numpy(rank.view(np.int32)).to(dev),
                 off=torch.from_numpy(off).to(dev), blob=torch.from_numpy(blob).to(dev),
                 tab=torch.from_numpy(tab.view(np.int32)).to(dev), tab_slots=slots)
        self._dev_tables[key] = t
        return t

    # ------------------------------------------------------------------ apply (GPU)
    def encode_bins(self, bins: torch.Tensor, min_token: int, max_token: Optional[int]):
        """bins [N, L] int64 (CUDA) -> (flat ids int32, offsets int64 [N+1], status int32 [N]).
        status bit 0 / 1 = a bin below min_token / above max_token (reference :182-192)."""
        dev = bins.device
        if dev.type != "cuda":
            raise _lib.BeastB200Error("BPE encode runs on the GPU only (no CPU fallback)")
        lib = _lib.load()
        t = self._tables(dev)
        bins = bins.to(torch.int64).contiguous()
        N, L = bins.shape
        self._reject_special_text(bins, int(min_token))
        max_shift = MAX_SHIFT if max_token is None else int(max_token) - int(min_token)
        if max_shift > MAX_SHIFT:
            raise ValueError("BPE over more than 55 296 distinct bin values is not representable (surrogate range)")
        stride = utf8_len(max_shift) * L
        padded = torch.empty((N, stride), device=dev, dtype=torch.int16)
        lens = torch.empty(N, device=dev, dtype=torch.int32)
        status = torch.empty(N, device=dev, dtype=torch.int32)
        with torch.cuda.device(dev):
            st = _lib.stream_ptr(dev)
            _lib.check(lib.bpe_encode(_lib.ptr(bins), N, L, int(min_token), max_shift, _lib.ptr(t["b2i"]),
                                      _lib.ptr(class_table_device(dev)), _lib.ptr(t["rank"]), t["V"], t["hash_bits"],
                                      _lib.ptr(padded), stride, _lib.ptr(lens), _lib.ptr(status), st), "bpe_encode")
            offsets = torch.zeros(N + 1, device=dev, dtype=torch.int64)
            torch.cumsum(lens, 0, out=offsets[1:])
            total = int(offsets[-1].item()) if N else 0
            flat = torch.empty(max(total, 1), device=dev, dtype=torch.int32)
            _lib.check(lib.bpe_compact(_lib.ptr(padded), stride, _lib.ptr(lens), _lib.ptr(offsets), N, _lib.ptr(flat),
                                       st), "bpe_compact")
        return flat[:total], offsets, status

    def _reject_special_text(self, bins: torch.Tensor, min_token: int):
        """The library matches special tokens in the TEXT before pre-tokenisation; a row whose chr() string
        contains one would encode differently there.  Not implemented on the GPU: detected and refused."""
        for t in self.special_tokens:
            m = len(t)
            if m == 0 or m > bins.shape[1] or bins.shape[0] == 0:
                continue
            pat = torch.tensor([ord(c) + min_token for c in t], device=bins.device, dtype=torch.int64)
            if bool((bins.unfold(1, m, 1) == pat).all(-1).any()):
                raise NotImplementedError(f"a sequence spells the special token {t!r}; the B200 encoder does not split "
                                          "special tokens out of the text (train without special_tokens, or reload "
                                          "the tokenizer from its files, which drops them as the reference does)")

    def decode_ids(self, flat: torch.Tensor, offsets: torch.Tensor, L: int, min_token: int):
        """CSR ids (CUDA) -> (bins int64 [N, L], status int32 [N], decoded length int32 [N])."""
        dev = flat.device
        if dev.type != "cuda":
            raise _lib.BeastB200Error("BPE decode runs on the GPU only (no CPU fallback)")
        lib = _lib.load()
        t = self._tables(dev)
        flat = flat.to(torch.int32).contiguous()
        offsets = offsets.to(dev, torch.int64).contiguous()
        N = offsets.numel() - 1
        bins = torch.empty((N, L), device=dev, dtype=torch.int64)
        status = torch.empty(N, device=dev, dtype=torch.int32)
        declen = torch.empty(N, device=dev, dtype=torch.int32)
        with torch.cuda.device(dev):
            _lib.check(lib.bpe_decode(_lib.ptr(flat), _lib.ptr(offsets), N, L, int(min_token), _lib.ptr(t["off"]),
                                      _lib.ptr(t["blob"]), _lib.ptr(t["tab"]), t["tab_slots"], t["V"], _lib.ptr(bins),
                                      _lib.ptr(status), _lib.ptr(declen), _lib.stream_ptr(dev)), "bpe_decode")
        return bins, status, declen

    # ------------------------------------------------------------------ HF-shaped convenience (single strings, on the GPU)
    def encode(self, text: str, add_special_tokens: bool = False) -> Encoding:
        cps = [ord(c) for c in text]
        if any(c > MAX_SHIFT for c in cps):
            raise ValueError("only codepoints below U+D800 are supported")
        if not cps:
            return Encoding([])
        dev = torch.device("cuda", torch.cuda.current_device()) if torch.cuda.is_available() else None
        if dev is None:
            raise _lib.BeastB200Error("BPE encode runs on the GPU only (no CPU fallback)")
        flat, _, _ = self.encode_bins(torch.tensor([cps], dtype=torch.int64, device=dev), 0, None)
        return Encoding(flat.cpu().tolist())

    def decode(self, ids: Sequence[int], skip_special_tokens: bool = True) -> str:
        """Token strings -> bytes -> text for ONE id list (a table lookup, kept for API parity with the
        HF object; batches go through decode_ids on the GPU)."""
        return bytes(U2B[ord(c)] for i in ids for c in self.tokens[i] if ord(c) in U2B).decode("utf-8", "replace")
