"""FIGBPE — trainer for byte-pair encoding over discretised BEAST tokens, on the GPU.

Drop-in for the reference trainer (beast/beast_bpe_trainer.py:32-160): same class names, arguments,
return type and exceptions.  The reference builds `chr(bin - min)` strings in Python and hands them to
HF `tokenizers`' Rust BpeTrainer; here the MP tokens never leave the GPU and the merge loop runs on
libbeast_b200.so kernels (csrc/bpe.cu): GPT-2 pre-tokenisation + byte-level expansion, a dense
L2-resident pair histogram, arg-max with the trainer's tie-break, in-place merges with compaction.

Sharded training: when torch.distributed is initialised with more than one rank (one process per
GPU), every rank passes ITS shard of the sequences; min/max, the seen-byte set, the initial histogram
and the per-merge 4 x V count deltas are all-reduced (NCCL), so every rank replays the same merges and
ends with the same vocabulary.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Iterable, List, Optional, Sequence, Union

import numpy as np
import torch

from . import _lib
from .beast_bspline_tokenizer import BEASTBsplineTokenizer
from .bpe_model import B2U, MAX_SHIFT, B200ByteLevelBPE, class_table_device, utf8_len

try:
    from tqdm.auto import tqdm
except Exception:  # pragma: no cover
    tqdm = None  # type: ignore[assignment]

ArrayLike = Union[Sequence[int], np.ndarray, torch.Tensor]

# symbol ids are 15 bits wide in the corpus (bit 15 = word start); the pair histogram is dense V x V int32 (4.3 GB at the limit;
# above 12 800 entries the rewrite kernel has no room for block-private counters and reduces into the global delta block)
MAX_TRAIN_VOCAB = 32766


@dataclass
class FIGBPEState:
    tokenizer: B200ByteLevelBPE
    min_token: int
    max_token: int


class _Collective:
    """The three reductions the sharded trainer needs; a no-op for a single rank."""

    def __init__(self, group=None, enabled=None):
        import torch.distributed as dist
        self.dist = dist
        self.on = bool(enabled) if enabled is not None else (dist.is_available() and dist.is_initialized()
                                                             and dist.get_world_size(group) > 1)
        self.group = group

    def reduce_(self, t: torch.Tensor, op: str):
        if self.on:
            self.dist.all_reduce(t, op={"sum": self.dist.ReduceOp.SUM, "min": self.dist.ReduceOp.MIN,
                                        "max": self.dist.ReduceOp.MAX}[op], group=self.group)
        return t


def build_alphabet(min_token: int, max_token: int, seen_bytes: Sequence[int], special_tokens: Sequence[str] = ()):
    """A.3: vocabulary = [special tokens, in order, duplicates skipped] + chr(0..max-min) U byte-level characters
    seen, by sorted codepoint; a character that already is a (single-character) special token keeps that id."""
    chars = set(range(max_token - min_token + 1)) | {B2U[b] for b in range(256) if seen_bytes[b]}
    tokens: List[str] = []
    index: dict = {}
    for t in list(special_tokens) + [chr(c) for c in sorted(chars)]:
        if t not in index:
            index[t] = len(tokens)
            tokens.append(t)
    byte_to_id = np.array([index.get(chr(B2U[b]), -1) for b in range(256)], dtype=np.int16)
    return tokens, byte_to_id


class GpuBpeEngine:
    """Device state of one shard: chunk-major symbols, lengths, replicated V x V histogram."""

    DEDUP_SAMPLE = 65536          # "auto": distinct-word statistics are taken on this many sequences first
    DEDUP_KEEP = 0.7              # ... and the corpus is de-duplicated when distinct symbols / symbols is below this
    DEDUP_PACK = 64               # symbols per pseudo-sequence of packed distinct words (plus one straddling word)

    def __init__(self, bins: torch.Tensor, min_token: int, byte_to_id: np.ndarray, V: int, max_shift: int = 255,
                 row_len: Optional[torch.Tensor] = None, dedup="auto", seen_bytes: Optional[np.ndarray] = None):
        self.lib = _lib.load()
        self.dev = bins.device
        self.N, self.L = bins.shape
        self.V = V
        self.stride = max(self.N, 1)
        cap = utf8_len(max_shift) * self.L                  # byte-level symbols per sequence
        with torch.cuda.device(self.dev):
            # chunk-major corpus: [ceil(cap / 8) chunks, sequences, 8 symbols] uint16 (see csrc/bpe.cu)
            self.sym = torch.empty(((cap + 7) // 8, self.stride, 8), device=self.dev, dtype=torch.int16)
            self.len = torch.zeros(self.stride, device=self.dev, dtype=torch.int32)
            self.hist = torch.zeros((V, V), device=self.dev, dtype=torch.int32)
            self.delta = torch.zeros(4 * V, device=self.dev, dtype=torch.int32)
            self.result = torch.zeros(256, device=self.dev, dtype=torch.int64)   # arg-max scratch (per-block maxima)
            self.work = torch.zeros(4 + 2 * self.stride, device=self.dev, dtype=torch.int32)   # scan -> rewrite work list
            self.mode = "single GPU"
            err = torch.zeros(1, device=self.dev, dtype=torch.int32)
            b2i = torch.from_numpy(byte_to_id).to(self.dev)
            st = _lib.stream_ptr(self.dev)
            _lib.check(self.lib.bpe_symbolize(_lib.ptr(bins), self.N, self.L, int(min_token), _lib.ptr(b2i),
                                              _lib.ptr(class_table_device(self.dev)), _lib.ptr(self.sym),
                                              _lib.ptr(self.len), self.stride, _lib.ptr(err), _lib.ptr(row_len), st),
                       "bpe_symbolize")
            if int(err.item()):
                raise ValueError("discrete tokens outside the representable range after subtracting min_token")
            self.weight = None
            self.dedup_stats = None
            if dedup and self.N > 0:
                self._dedup_words(force=dedup is True)
            # ids before any merge: the byte-level symbols of the bytes the corpus holds (all mapped bytes when unknown)
            live = byte_to_id >= 0 if seen_bytes is None else (byte_to_id >= 0) & (np.asarray(seen_bytes) != 0)
            used = np.unique(byte_to_id[live]).astype(np.int16)
            used_d = torch.from_numpy(used).to(self.dev)
            n_ids = int(used[-1]) + 1 if used.size else 0
            _lib.check(self.lib.bpe_count_pairs(_lib.ptr(self.sym), _lib.ptr(self.len), self.N, self.stride, V,
                                                n_ids, _lib.ptr(used_d), int(used.size), _lib.ptr(self.hist),
                                                _lib.ptr(self.weight), st),
                       "bpe_count_pairs")

    # ------------------------------------------------------------------ word de-duplication (SURVEY.md §8(f)4)
    def _word_table(self, n_seq: int, expect_distinct: Optional[int] = None):
        """Hash table over the words of the first n_seq sequences -> (locations, counts) of the distinct words
        (unordered), or None on a hash collision (exactness is never traded: the caller keeps the plain corpus).
        expect_distinct sizes the table (an estimate from a sample); when it proves too small the pass is repeated
        with the safe bound, the number of words."""
        dev, lib = self.dev, self.lib
        st = _lib.stream_ptr(dev)
        totals = torch.zeros(2, device=dev, dtype=torch.int64)
        _lib.check(lib.bpe_word_totals(_lib.ptr(self.sym), _lib.ptr(self.len), n_seq, self.stride, _lib.ptr(totals), st),
                   "bpe_word_totals")
        words, symbols = (int(v) for v in totals.tolist())
        if words == 0:
            return None
        flags = torch.zeros(4, device=dev, dtype=torch.int32)
        wlist = torch.empty((words, 4), device=dev, dtype=torch.int64)       # hash, location, first six symbols per word
        cursor = torch.zeros(1, device=dev, dtype=torch.int64)
        _lib.check(lib.bpe_word_list(_lib.ptr(self.sym), _lib.ptr(self.len), n_seq, self.stride, _lib.ptr(wlist), words,
                                     _lib.ptr(cursor), _lib.ptr(flags), st), "bpe_word_list")
        for bound in ([min(int(expect_distinct), words)] if expect_distinct else []) + [words]:
            size = 1 << max(10, (bound + bound // 2 - 1).bit_length())   # load factor <= 2/3 (linear probing)
            table = torch.zeros((size, 4), device=dev, dtype=torch.int64)    # key, representative, count | symbols
            flags[1:].zero_()
            _lib.check(lib.bpe_word_insert(_lib.ptr(self.sym), self.stride, _lib.ptr(wlist), words, _lib.ptr(table), size,
                                           _lib.ptr(flags), st), "bpe_word_insert")
            status, distinct = flags[:2].tolist()
            if status in (1, 2):
                return None
            if status != 3 and distinct <= size - size // 4:
                break
            if bound == words:
                return None
            flags.zero_()
        del wlist
        loc = torch.empty(distinct, device=dev, dtype=torch.int64)
        cnt = torch.empty(distinct, device=dev, dtype=torch.int32)
        _lib.check(lib.bpe_word_emit(_lib.ptr(table), size, _lib.ptr(flags), _lib.ptr(loc), _lib.ptr(cnt), distinct, st),
                   "bpe_word_emit")
        status, _, emitted = flags[:3].tolist()
        if status or emitted != distinct:
            return None
        return loc, cnt, words, symbols

    def _dedup_words(self, force: bool):
        """Replace the symbolised corpus by its distinct words, packed into pseudo-sequences of equal-count words,
        with one weight per pseudo-sequence.  "auto": only when a sample says the corpus is repetitive enough."""
        dev, lib = self.dev, self.lib
        expect = None
        if self.N > 2 * self.DEDUP_SAMPLE:
            probe = self._word_table(self.DEDUP_SAMPLE)
            if probe is None:
                return
            rep, cnt, words, symbols = probe
            ratio = float((rep & 0xFFFF).sum().item()) / max(symbols, 1)
            self.dedup_stats = {"sampled_sequences": self.DEDUP_SAMPLE, "sample_distinct_symbol_ratio": ratio, "applied": False}
            if not force and ratio >= self.DEDUP_KEEP:
                return
            # distinct words grow sub-linearly with the corpus: the sample's rate bounds the table from above
            expect = int(rep.numel() * (self.N / self.DEDUP_SAMPLE)) + 1024
        full = self._word_table(self.N, expect)
        if full is None:
            self.dedup_stats = {"applied": False, "reason": "64-bit word hash collision: trained on the plain corpus"}
            return
        rep, cnt, words, symbols = full
        lens = rep & 0xFFFF
        distinct_symbols = int(lens.sum().item())
        ratio = distinct_symbols / max(symbols, 1)
        stats = {"words": words, "distinct_words": int(rep.numel()), "symbols": symbols,
                 "distinct_symbols": distinct_symbols, "distinct_symbol_ratio": ratio, "applied": False}
        self.dedup_stats = {**(self.dedup_stats or {}), **stats}
        if not force and ratio >= self.DEDUP_KEEP:
            return
        # order by count (descending), pack words of equal count into pseudo-sequences of ~DEDUP_PACK symbols
        # (a dozen O(U) torch scans / gathers; no scatter, no cummax)
        cnt, order = torch.sort(cnt, descending=True)
        rep, lens = rep[order], lens[order]
        U = int(rep.numel())
        incl = torch.cumsum(lens, 0)
        excl = incl - lens                                                    # symbols before word i
        new_group = torch.ones(U, device=dev, dtype=torch.bool)
        new_group[1:] = cnt[1:] != cnt[:-1]
        gid = torch.cumsum(new_group, 0) - 1
        group_start = excl[torch.nonzero(new_group, as_tuple=False).flatten()][gid]
        bin_in_group = (excl - group_start) // self.DEDUP_PACK
        new_bin = new_group
        new_bin[1:] |= bin_in_group[1:] != bin_in_group[:-1]
        first = torch.nonzero(new_bin, as_tuple=False).flatten()              # first word of every pseudo-sequence
        P = int(first.numel())
        pid = torch.cumsum(new_bin, 0) - 1                                    # pseudo-sequence of word i
        bin_start = excl[first]
        off = excl - bin_start[pid]
        plen = torch.empty(P, device=dev, dtype=torch.int64)
        plen[:-1] = bin_start[1:] - bin_start[:-1]
        plen[-1] = incl[-1] - bin_start[-1]
        cap = int(plen.max().item())
        if cap > 32767 or P > 0x7FFFFFFF:
            return
        sym2 = torch.empty(((cap + 7) // 8, P, 8), device=dev, dtype=torch.int16)
        len2 = plen.to(torch.int32)
        # named temporaries: a tensor created inside the call would be freed (and its block reused) before the launch
        rep_c, pid32, off32 = rep.contiguous(), pid.to(torch.int32), off.to(torch.int32)
        _lib.check(lib.bpe_word_pack(_lib.ptr(self.sym), self.stride, _lib.ptr(rep_c), _lib.ptr(pid32), _lib.ptr(off32),
                                     U, _lib.ptr(sym2), _lib.ptr(len2), P, P, _lib.stream_ptr(dev)), "bpe_word_pack")
        self.sym, self.len, self.N, self.stride = sym2, len2, P, P
        self.weight = cnt[first].to(torch.int32).contiguous()
        self.work = torch.zeros(4 + 2 * P, device=dev, dtype=torch.int32)
        self.dedup_stats.update(applied=True, pseudo_sequences=P, longest_pseudo_sequence=cap)

    def argmax(self, n_active: int):
        with torch.cuda.device(self.dev):
            _lib.check(self.lib.bpe_argmax(_lib.ptr(self.hist), self.V, n_active, _lib.ptr(self.result),
                                           _lib.stream_ptr(self.dev)), "bpe_argmax")
        key = int(self.result[0].item()) & 0xFFFFFFFFFFFFFFFF
        if key == 0:
            return 0, -1, -1
        flat = 0xFFFFFFFF - (key & 0xFFFFFFFF)
        return key >> 32, flat // self.V, flat % self.V

    def merge(self, a: int, b: int, c: int):
        with torch.cuda.device(self.dev):
            _lib.check(self.lib.bpe_apply_merge(_lib.ptr(self.sym), _lib.ptr(self.len), self.N, self.stride, a, b, c,
                                                self.V, _lib.ptr(self.delta), _lib.ptr(self.work),
                                                _lib.ptr(self.weight), _lib.stream_ptr(self.dev)), "bpe_apply_merge")

    def apply_delta(self, a: int, b: int, c: int):
        with torch.cuda.device(self.dev):
            _lib.check(self.lib.bpe_apply_delta(_lib.ptr(self.hist), _lib.ptr(self.delta), a, b, c, self.V,
                                                _lib.stream_ptr(self.dev)), "bpe_apply_delta")

    def start_run(self, n_tokens: int, vocab_size: int, min_frequency: int, peers: Optional["_lib.BpePeers"] = None,
                  delta: Optional[torch.Tensor] = None) -> "_FastRun":
        return _FastRun(self, n_tokens, vocab_size, min_frequency, peers, delta)

    def run_fast(self, coll: "_Collective", n_tokens: int, vocab_size: int, min_frequency: int, progress=None):
        """Sync-free merge loop: arg-max, stop rules, id assignment and the merge log all stay on the device
        (bpe_train_step); the host only enqueues iterations and reads the log once (or once per 256-merge block
        when a progress bar is shown).  Sharded: the per-merge all-reduce of the 4 x V deltas is part of the
        iteration-head kernel (peer loads over NVLink, see _PeerBlock), so nothing runs on the host between
        merges either; without peer access the deltas go through one NCCL all-reduce per merge instead.
        Returns [(a, b, new_id, count)] assuming every merge creates a NEW token string; the caller verifies
        that and falls back to the exact host-driven loop otherwise."""
        if int(vocab_size) - int(n_tokens) <= 0:
            return []
        peers = delta = None
        if coll.on:
            block = _PeerBlock.get(self.dev, self.V, coll)
            if block is not None:
                peers, delta = block.begin_run(coll), block.delta_view
            self.mode = "peer-fused (NVLink loads inside bpe_iterate_kernel)" if block is not None else \
                "nccl all-reduce per merge (no peer access)"
        run = self.start_run(n_tokens, vocab_size, min_frequency, peers, delta)
        while not run.finished:
            if coll.on and peers is None:
                run.enqueue(limit=1)
                coll.reduce_(run.delta_half(run.enqueued - 1), "sum")
            else:
                run.enqueue()
            if progress is not None:
                progress(run.merges_done())
        return run.finish()


class _FastRun:
    """One pass of the device-driven merge loop over an engine: owns ctl / log / signatures, enqueues
    iterations in blocks that end at the signature (re)build points."""
    SIG_START, SIG_REBUILD = 64, 256

    def __init__(self, eng: GpuBpeEngine, n_tokens, vocab_size, min_frequency, peers=None, delta=None):
        self.eng, self.peers = eng, peers
        self.vocab_size, self.min_frequency = int(vocab_size), int(min_frequency)
        self.max_merges = max(int(vocab_size) - int(n_tokens), 0)
        self.enqueued = 0
        dev = eng.dev
        with torch.cuda.device(dev):
            # control block, double-buffered by iteration parity (iteration i reads ctl[i & 1], writes the other)
            self.ctl = torch.zeros((2, 16), device=dev, dtype=torch.int32)
            self.ctl[0, 4] = n_tokens
            self.log = torch.zeros(4 * max(self.max_merges, 1), device=dev, dtype=torch.int32)
            eng.result.zero_()
            # count deltas, double-buffered by merge parity: the peers' copy when sharded over NVLink
            self.delta = delta if delta is not None else torch.zeros(8 * eng.V, device=dev, dtype=torch.int32)
            # Pair signatures (two 4-byte column reads per merge tell which sequences can hold the pair).  The
            # first merges touch most sequences anyway, so the signatures are built after SIG_START merges and
            # rebuilt from the current corpus every SIG_REBUILD merges (0.6 ms at 1.6 M sequences) to drop stale bits.
            self.sig = torch.empty((int(eng.lib.bpe_signature_words()), eng.stride), device=dev, dtype=torch.int32)

    @property
    def finished(self) -> bool:
        return self.enqueued >= self.max_merges

    def delta_half(self, merge: int) -> torch.Tensor:
        V = self.eng.V
        return self.delta[(merge & 1) * 4 * V:((merge & 1) + 1) * 4 * V]

    def enqueue(self, limit: Optional[int] = None) -> int:
        """Enqueue the next block of iterations on the current stream (never synchronises)."""
        eng, i = self.eng, self.enqueued
        if i >= self.max_merges:
            return 0
        dev = eng.dev
        with torch.cuda.device(dev):
            st = _lib.stream_ptr(dev)
            if i >= self.SIG_START and (i - self.SIG_START) % self.SIG_REBUILD == 0:
                _lib.check(eng.lib.bpe_build_signatures(_lib.ptr(eng.sym), _lib.ptr(eng.len), eng.N, eng.stride,
                                                        _lib.ptr(self.sig), st), "bpe_build_signatures")
            nxt = self.SIG_START if i < self.SIG_START else i + self.SIG_REBUILD - (i - self.SIG_START) % self.SIG_REBUILD
            n = min(nxt, self.max_merges) - i
            if limit is not None:
                n = min(n, int(limit))
            _lib.check(eng.lib.bpe_train_step(_lib.ptr(eng.sym), _lib.ptr(eng.len), eng.N, eng.stride, eng.V,
                                              _lib.ptr(eng.hist), _lib.ptr(self.delta), _lib.ptr(self.ctl),
                                              _lib.ptr(self.log), _lib.ptr(eng.result), _lib.ptr(eng.work),
                                              self.vocab_size, self.min_frequency, self.max_merges,
                                              _lib.ptr(self.sig) if i >= self.SIG_START else None, int(i), int(n),
                                              C.byref(self.peers) if self.peers is not None else None,
                                              _lib.ptr(eng.weight), st),
                       "bpe_train_step")
        self.enqueued += n
        return n

    def merges_done(self) -> int:
        return int(self.ctl[self.enqueued & 1, 5].item())   # synchronises: progress display only

    def finish(self):
        ctl_h = self.ctl[self.enqueued & 1].cpu().tolist()
        if ctl_h[8]:
            raise _lib.BeastB200Error("sharded BPE training: a peer GPU did not publish its merge epoch within 5 s "
                                      "(ranks out of step or peer memory not reachable)")
        n = ctl_h[5]
        return self.log[:4 * n].cpu().view(-1, 4).tolist()


class _PeerBlock:
    """Peer-visible memory of one rank for the sharded trainer: int32 [2][4*V] count deltas + BPE_MAX_PEERS flags,
    allocated with cudaMalloc, exported over CUDA IPC and mapped by every other rank of the group (one process
    per GPU on one NVLink / NVSwitch node).  Cached per (device, V, group) for the life of the process."""
    _cache: dict = {}

    @classmethod
    def get(cls, dev, V, coll: "_Collective"):
        import os
        if os.environ.get("BEAST_B200_BPE_NO_PEER") == "1":
            return None
        key = (str(dev), int(V), id(coll.group))
        if key not in cls._cache:
            cls._cache[key] = cls._create(dev, V, coll)
        return cls._cache[key]

    @classmethod
    def _create(cls, dev, V, coll):
        dist, lib = coll.dist, _lib.load()
        world, rank = dist.get_world_size(coll.group), dist.get_rank(coll.group)
        if world > _lib.BPE_MAX_PEERS:
            return None
        self = cls()
        self.V, self.dev, self.world, self.rank = int(V), dev, world, rank
        n_delta = 8 * self.V
        nbytes = 4 * (n_delta + _lib.BPE_MAX_PEERS)
        own, handle, ok = C.c_void_p(), C.create_string_buffer(64), 1
        with torch.cuda.device(dev):
            if lib.beast_peer_alloc(nbytes, C.byref(own), handle) != 0:
                ok, own = 0, C.c_void_p()
            gathered = [None] * world
            dist.all_gather_object(gathered, (ok, bytes(handle.raw)), group=coll.group)
            ptrs = [None] * world
            ok = int(all(g[0] for g in gathered))
            if ok:
                for r, (_, h) in enumerate(gathered):
                    if r == rank:
                        ptrs[r] = own.value
                        continue
                    mapped = C.c_void_p()
                    if lib.beast_peer_open(C.create_string_buffer(h, 64), C.byref(mapped)) != 0:
                        ok = 0
                        break
                    ptrs[r] = mapped.value
            flag = torch.tensor([ok], device=dev, dtype=torch.int32)
            coll.reduce_(flag, "min")                       # every rank must have mapped every peer
            if not int(flag.item()):
                return None
        self.ptrs = ptrs
        # torch view of this rank's delta halves (reduced by NCCL only on the fallback path; otherwise just a pointer)
        self.delta_view = _wrap_device_int32(own.value, n_delta, dev)
        self.flags_view = _wrap_device_int32(own.value + 4 * n_delta, _lib.BPE_MAX_PEERS, dev)
        return self

    def begin_run(self, coll) -> "_lib.BpePeers":
        """Run boundary: no rank may touch peer memory for the new run while another still reads it for the old
        one, and no rank may publish an epoch before every rank has cleared its flags.  Two tiny all-reduces
        are those barriers (stream-ordered on every rank, no host synchronisation)."""
        t = torch.zeros(1, device=self.dev, dtype=torch.int32)
        coll.reduce_(t, "sum")
        self.flags_view.zero_()
        coll.reduce_(t, "sum")
        peers = _lib.BpePeers()
        peers.world, peers.rank, peers.grid_blocks, peers.epoch_base = self.world, self.rank, 0, 0
        for r in range(self.world):
            peers.delta[r] = self.ptrs[r]
            peers.flags[r] = self.ptrs[r] + 4 * 8 * self.V
        return peers


def _wrap_device_int32(ptr: int, n: int, dev) -> torch.Tensor:
    """A torch tensor over memory this library allocated (CUDA array interface; never freed by torch)."""
    class _Mem:
        __cuda_array_interface__ = {"shape": (n,), "typestr": "<i4", "data": (int(ptr), False), "version": 3,
                                    "strides": None}
    return torch.as_tensor(_Mem(), device=dev)


def scan_bins_gpu(bins: torch.Tensor, coll: _Collective):
    """Global min / max token and the set of UTF-8 bytes seen (A.1, A.3)."""
    lib = _lib.load()
    dev = bins.device
    with torch.cuda.device(dev):
        st = _lib.stream_ptr(dev)
        mm = torch.tensor([torch.iinfo(torch.int64).max, torch.iinfo(torch.int64).min], device=dev, dtype=torch.int64)
        if bins.numel():
            _lib.check(lib.bpe_scan_bins(_lib.ptr(bins), bins.numel(), 0, _lib.ptr(mm), None, None, 0, st), "bpe_scan_bins")
        lo, hi = mm[:1].clone(), mm[1:].clone()
        coll.reduce_(lo, "min")
        coll.reduce_(hi, "max")
        min_token, max_token = int(lo.item()), int(hi.item())
        if max_token - min_token > MAX_SHIFT:
            raise ValueError("BPE over more than 55 296 distinct bin values is not representable: chr() of the shifted "
                             "bins would enter the surrogate range")
        seen = torch.zeros(256, device=dev, dtype=torch.int32)
        err = torch.zeros(1, device=dev, dtype=torch.int32)
        if bins.numel():
            _lib.check(lib.bpe_scan_bins(_lib.ptr(bins), bins.numel(), min_token, None, _lib.ptr(seen), _lib.ptr(err), 1,
                                         st), "bpe_scan_bins")
        coll.reduce_(seen, "max")
    return min_token, max_token, seen.cpu().numpy()


def train_bpe(bins: torch.Tensor, vocab_size: int, min_frequency: int = 2, *, engine_factory=None,
              scan=None, coll: Optional[_Collective] = None, show_progress: bool = False,
              row_len: Optional[torch.Tensor] = None, special_tokens: Sequence[str] = (), dedup="auto"):
    """The merge loop (A.4) over this rank's shard `bins` [N, L] int64.  Returns
    (B200ByteLevelBPE, min_token, max_token).  `engine_factory` / `scan` are injection points for the
    CPU-only multi-process tests of the orchestration; production uses the GPU engine.
    row_len [N] int32: sequences of unequal length, padded to L with an in-range value of the same row (so the
    min / max / seen-byte scans need no mask).  special_tokens: BpeTrainer's, ids first.  dedup: train on the
    distinct pre-tokens with counts, as BpeTrainer does ("auto" = when a sample says it pays, True / False)."""
    coll = coll or _Collective()
    scan = scan or scan_bins_gpu
    engine_factory = engine_factory or GpuBpeEngine
    min_token, max_token, seen = scan(bins, coll)
    tokens, byte_to_id = build_alphabet(min_token, max_token, seen, special_tokens)
    V = max(int(vocab_size), len(tokens))
    if V > MAX_TRAIN_VOCAB:
        raise NotImplementedError(
            f"bpe_vocab_size {V} is above the trainer's limit of {MAX_TRAIN_VOCAB}: symbol ids are 15 bits wide in the corpus and "
            f"the merge loop keeps a dense V x V int32 pair histogram ({4 * V * V / 2**30:.1f} GiB here; reference FIGBPE "
            "default is 1024, BASELINE config 2048)")
    make_engine = lambda: (engine_factory(bins, min_token, byte_to_id, V, max_token - min_token, row_len, dedup, seen)
                           if engine_factory is GpuBpeEngine else engine_factory(bins, min_token, byte_to_id, V))
    eng = make_engine()
    coll.reduce_(eng.hist, "sum")                       # replicated global histogram
    index = {t: i for i, t in enumerate(tokens)}
    merges: List[tuple] = []
    if hasattr(eng, "run_fast"):
        bar = tqdm(total=max(vocab_size - len(tokens), 0), desc="BPE merges", leave=False) if (show_progress and tqdm) else None
        log = eng.run_fast(coll, len(tokens), vocab_size, min_frequency,
                           progress=(lambda n: bar.update(n - bar.n)) if bar is not None else None)
        if bar is not None:
            bar.close()
        fast_tokens, fast_index, ok = list(tokens), dict(index), True
        for a, b, c, _count in log:
            new = fast_tokens[a] + fast_tokens[b]
            if new in fast_index or c != len(fast_tokens):
                ok = False                              # an existing string must keep its id: replay exactly
                break
            fast_index[new] = c
            fast_tokens.append(new)
        if ok:
            model = B200ByteLevelBPE(fast_tokens, [(a, b, c) for a, b, c, _ in log], special_tokens=special_tokens)
            model.trainer_mode = getattr(eng, "mode", "single GPU")
            model.dedup_stats = getattr(eng, "dedup_stats", None)
            return model, min_token, max_token
        eng = make_engine()
        coll.reduce_(eng.hist, "sum")
    bar = tqdm(total=max(vocab_size - len(tokens), 0), desc="BPE merges", leave=False) if (show_progress and tqdm) else None
    while len(tokens) < vocab_size:
        count, a, b = eng.argmax(len(tokens))
        if a < 0 or count < 1 or count < min_frequency:
            break
        new = tokens[a] + tokens[b]
        c = index.get(new)
        if c is None:                                   # an existing string keeps its id (merge still recorded)
            c = len(tokens)
            tokens.append(new)
            index[new] = c
            if bar is not None:
                bar.update(1)
        merges.append((a, b, c))
        eng.merge(a, b, c)
        coll.reduce_(eng.delta, "sum")                  # per-merge count deltas: 4 x V int32
        eng.apply_delta(a, b, c)
    if bar is not None:
        bar.close()
    return B200ByteLevelBPE(tokens, merges, special_tokens=special_tokens), min_token, max_token


def _flatten_to_numpy(sequence: ArrayLike) -> np.ndarray:
    if isinstance(sequence, torch.Tensor):
        array = sequence.detach().cpu().numpy()
    else:
        array = np.asarray(sequence)
    if array.ndim > 1:
        array = array.reshape(-1)
    return array.astype(np.int64)


class FIGBPE:
    """Trainer for Byte Pair Encoding over discretised BEAST tokens (reference :39-160)."""

    def __init__(self, vocab_size: int = 1024, *, min_frequency: int = 2, special_tokens: Optional[Sequence[str]] = None,
                 show_progress: bool = True, max_token_length: int = 10000, device=None, process_group=None,
                 dedup="auto") -> None:
        self.vocab_size = vocab_size
        self.min_frequency = min_frequency
        self.special_tokens = list(special_tokens or [])
        self.show_progress = show_progress
        self.max_token_length = max_token_length
        self.device = device
        self.process_group = process_group
        self.dedup = dedup
        self.tokenizer: Optional[B200ByteLevelBPE] = None
        self.min_token: Optional[int] = None
        self.max_token: Optional[int] = None

    def _device(self):
        if self.device is not None:
            return _lib.require_cuda(self.device)
        if not torch.cuda.is_available():
            raise _lib.BeastB200Error("no CUDA device available: the BPE trainer has no CPU fallback")
        return torch.device("cuda", torch.cuda.current_device())

    def fit_from_bins(self, bins: torch.Tensor, row_len: Optional[torch.Tensor] = None) -> FIGBPEState:
        """bins [N, L] int64 on the GPU (this rank's shard when sharded); row_len [N]: see train_bpe."""
        # process_group=False forces a local (unsharded) fit even under torch.distributed
        coll = _Collective(enabled=False) if self.process_group is False else _Collective(self.process_group)
        dev = self._device()
        if row_len is not None:
            row_len = row_len.to(dev, torch.int32).contiguous()
        tok, mn, mx = train_bpe(bins.to(dev, torch.int64).contiguous(), self.vocab_size, self.min_frequency,
                                coll=coll, show_progress=self.show_progress, row_len=row_len,
                                special_tokens=self.special_tokens, dedup=self.dedup)
        self.tokenizer, self.min_token, self.max_token = tok, mn, mx
        return FIGBPEState(tokenizer=tok, min_token=mn, max_token=mx)

    def fit_from_sequences(self, sequences: Iterable[ArrayLike]) -> FIGBPEState:
        processed: List[np.ndarray] = []
        for seq in sequences:
            arr = _flatten_to_numpy(seq)
            if arr.size == 0:
                continue
            processed.append(arr)
        if not processed:
            raise ValueError("No non-empty sequences provided for BPE training.")
        lengths = np.fromiter((a.size for a in processed), dtype=np.int64, count=len(processed))
        if int(lengths.min()) == int(lengths.max()):
            return self.fit_from_bins(torch.from_numpy(np.stack(processed)))
        # unequal lengths (reference :76-98 takes any): pad every row with its own first value — in range, so
        # min / max / the seen-byte set are those of the real data — and hand the true lengths to the symboliser
        padded = np.empty((len(processed), int(lengths.max())), dtype=np.int64)
        for i, a in enumerate(processed):
            padded[i, :a.size] = a
            padded[i, a.size:] = a[0]
        return self.fit_from_bins(torch.from_numpy(padded), row_len=torch.from_numpy(lengths.astype(np.int32)))

    GATHER_ROWS = 4096      # loader batches are gathered on the device and fitted this many trajectories at a time

    def fit_from_trajectories(self, tokenizer: BEASTBsplineTokenizer, trajectories: Iterable[Union[ArrayLike, dict]], *,
                              update_bounds: bool = False, batch_key: str = "actions",
                              max_sequences: Optional[int] = None) -> FIGBPEState:
        """Reference :100-151: encode every loader batch to MP tokens, train on them.  The tokens of a trajectory
        do not depend on its batch (fixed bounds), so small loader batches (32 in the reference's script) are
        copied into a device staging block and fitted GATHER_ROWS at a time — one K1 launch per ~4 096
        trajectories instead of one per batch; the token chunks never leave the GPU."""
        chunks: List[torch.Tensor] = []
        collected = 0
        encode_fn = getattr(tokenizer, "encode_to_mp_tokens", None)
        offset = 0
        if encode_fn is None:
            encode_fn = tokenizer.encode
            offset = None                                # encode() adds the LLM offset when one is configured
        progress_bar = None
        if self.show_progress and tqdm is not None:
            progress_bar = tqdm(total=max_sequences, desc="Collecting BEAST sequences for BPE", unit="seq", leave=False)
        # gathering needs per-batch independence: fixed bounds, no boundary-condition state of "the last batch"
        can_gather = (not update_bounds and isinstance(tokenizer, BEASTBsplineTokenizer)
                      and not tokenizer._has_conditions and torch.cuda.is_available())
        staging, filled = None, 0
        T, D = (tokenizer.times.numel(), tokenizer.num_dof) if can_gather else (0, 0)
        # HOST batches beyond the first block are gathered in one of two pinned blocks (a plain memcpy per batch) and
        # uploaded GATHER_ROWS at a time by ONE asynchronous copy: a pageable 90 KB batch costs a synchronous staged
        # cudaMemcpy each (~15 us), 50 000 of them were most of the wall time of the reference's loader shape
        pinned, pin_events, pin_cur, block_on_host = None, [None, None], 0, False

        def flush():
            nonlocal filled, pin_cur, block_on_host
            if filled:
                if block_on_host:
                    staging[:filled].copy_(pinned[pin_cur][:filled], non_blocking=True)
                    ev = torch.cuda.Event()
                    ev.record()
                    pin_events[pin_cur] = ev
                    pin_cur ^= 1
                    if pin_events[pin_cur] is not None:      # the upload that last read the block we fill next
                        pin_events[pin_cur].synchronize()
                    block_on_host = False
                off = offset if offset is not None else (
                    tokenizer._llm_vocab_offset() if tokenizer.llm_vocab_size is not None else 0)
                chunks.append(tokenizer._fit(staging[:filled], want_tokens=True, offset=off)[0])
                filled = 0

        for batch in trajectories:
            if isinstance(batch, dict):
                if batch_key not in batch:
                    raise KeyError(f"Batch dictionary is missing required key '{batch_key}'.")
                data = batch[batch_key]
            else:
                data = batch
            if not torch.is_tensor(data):
                data = torch.as_tensor(data)
            n_new = None
            if (can_gather and data.dim() == 3 and data.shape[1] == T and data.shape[2] >= D
                    and 0 < data.shape[0] <= self.GATHER_ROWS):
                if max_sequences is not None and collected + data.shape[0] > max_sequences:
                    data = data[: max_sequences - collected]
                if staging is None:
                    staging = torch.empty((self.GATHER_ROWS, T, D), device=tokenizer._cuda(), dtype=torch.float32)
                via_host = data.device.type == "cpu" and collected >= self.GATHER_ROWS
                if filled and (filled + data.shape[0] > self.GATHER_ROWS or via_host != block_on_host):
                    flush()
                if via_host:
                    if pinned is None:
                        pinned = [torch.empty((self.GATHER_ROWS, T, D), dtype=torch.float32).pin_memory() for _ in range(2)]
                    pinned[pin_cur][filled:filled + data.shape[0]].copy_(data[..., :D])
                    block_on_host = True
                else:
                    staging[filled:filled + data.shape[0]].copy_(data[..., :D], non_blocking=True)
                filled += data.shape[0]
                n_new = data.shape[0]
            else:
                flush()                                  # keep the loader's order
                tokens, _ = encode_fn(data, update_bounds=update_bounds)       # stays on the GPU
                if max_sequences is not None and collected + tokens.shape[0] > max_sequences:
                    tokens = tokens[: max_sequences - collected]
                chunks.append(tokens)
                n_new = tokens.shape[0]
            collected += n_new
            if progress_bar is not None:
                progress_bar.update(n_new)
            if max_sequences is not None and collected >= max_sequences:
                break
        flush()
        if progress_bar is not None:
            progress_bar.close()
        if not chunks or collected == 0:
            raise ValueError("No non-empty sequences provided for BPE training.")
        return self.fit_from_bins(chunks[0] if len(chunks) == 1 else torch.cat(chunks, 0))

    def get_state(self) -> FIGBPEState:
        if self.tokenizer is None or self.min_token is None or self.max_token is None:
            raise RuntimeError("BPE tokenizer has not been trained yet.")
        return FIGBPEState(tokenizer=self.tokenizer, min_token=self.min_token, max_token=self.max_token)
