"""BEASTBsplineBPETokenizer — drop-in for the reference class (beast/beast_bspline_bpe_tokenizer.py:22-424):
the B-spline tokenizer with a learned byte-pair encoder over its discrete tokens.

Training (fit_from_trajectories), bins -> ids (_discrete_to_bpe) and ids -> bins (_bpe_to_discrete)
run on the GPU (csrc/bpe.cu); the reference loops over rows in Python around HF `tokenizers`.  The
ragged List[List[int]] return of `encode` is kept for API fidelity; `encode_csr` returns the same ids
as device CSR tensors without the host round trip.
"""
from __future__ import annotations

import json
import itertools
import numbers
from pathlib import Path
from typing import Iterable, List, Optional, Sequence, Union

import numpy as np
import torch

from .basis import check_orders
from .beast_bspline_tokenizer import CONFIG_FILENAME, BEASTBsplineTokenizer
from .bpe_model import B200ByteLevelBPE

TokenLike = Union[Sequence[int], torch.Tensor, np.ndarray]


def _coerce_bpe(tokenizer) -> B200ByteLevelBPE:
    if isinstance(tokenizer, B200ByteLevelBPE):
        return tokenizer
    try:                                    # a tokenizer trained by the reference / HF tokenizers
        from tokenizers import ByteLevelBPETokenizer
        if isinstance(tokenizer, ByteLevelBPETokenizer):
            return B200ByteLevelBPE.from_hf(tokenizer)
    except ImportError:
        pass
    raise TypeError("Expected a ByteLevelBPETokenizer instance.")


_PYLISTS = None


def _pylists():
    """The CPython helper `_pylists` (csrc/pylists.c, built in-tree by `build.py`); False when it cannot be had
    (no compiler): the pure-Python conversions below then do the same job, slower."""
    global _PYLISTS
    if _PYLISTS is None:
        try:
            from . import _pylists as mod
        except ImportError:
            try:
                from .build import build_pylists
                build_pylists()
                import importlib
                importlib.invalidate_caches()
                from . import _pylists as mod
            except Exception:
                mod = False
        _PYLISTS = mod
    return _PYLISTS


def _split_rows(flat_h: np.ndarray, off_h: np.ndarray) -> List[List[int]]:
    """CSR -> the ragged List[List[int]] the reference returns.  C helper: one list per row, one shared int object per
    distinct id.  Without it: one tolist() of the whole id array and pointer-copy slices of it, the cyclic collector
    paused meanwhile (tens of thousands of fresh lists would trigger repeated full collections that find nothing)."""
    import gc
    was_enabled = gc.isenabled()
    gc.disable()
    try:
        mod = _pylists()
        if mod:
            return mod.split_rows(np.ascontiguousarray(flat_h, dtype=np.int32),
                                  np.ascontiguousarray(off_h, dtype=np.int64))
        off = off_h.tolist()
        big = flat_h.tolist()
        return [big[off[i]:off[i + 1]] for i in range(len(off) - 1)]
    finally:
        if was_enabled:
            gc.enable()


def _flatten_rows(rows):
    """List / tuple of lists / tuples of Python ints -> (flat int32, offsets int64 [n+1]) numpy arrays, or None when the
    rows are of another kind (tensors, arrays, numpy scalars: the general path converts those)."""
    mod = _pylists()
    if mod:
        got = mod.flatten_rows(rows)
        if got is None:
            return None
        return np.frombuffer(got[0], dtype=np.int32), np.frombuffer(got[1], dtype=np.int64)
    if not (isinstance(rows, (list, tuple)) and all(type(t) in (list, tuple) for t in rows)):
        return None
    lens = np.fromiter(map(len, rows), dtype=np.int64, count=len(rows))
    try:
        flat = np.fromiter(itertools.chain.from_iterable(rows), dtype=np.int64, count=int(lens.sum()))
    except OverflowError:
        raise ValueError("BPE token id out of range") from None
    except (TypeError, ValueError):
        return None
    if flat.size and (flat.min() < -2 ** 31 or flat.max() >= 2 ** 31):
        raise ValueError("BPE token id out of range")
    offsets = np.zeros(len(lens) + 1, dtype=np.int64)
    np.cumsum(lens, out=offsets[1:])
    return flat.astype(np.int32), offsets


class BEASTBsplineBPETokenizer(BEASTBsplineTokenizer):
    """B-Spline tokenizer augmented with a learned Byte-Pair encoder."""

    bpe_subdir = "bpe_tokenizer"

    def __init__(self, *args, bpe_vocab_size: int = 1024, bpe_min_token: int = 0,
                 base_tokenizer: Optional[BEASTBsplineTokenizer] = None, **kwargs) -> None:
        kwargs = kwargs.copy()
        kwargs.pop("use_bpe", None)
        kwargs.pop("tokenizer_type", None)

        self.bpe_vocab_size = bpe_vocab_size
        self.bpe_tokenizer: Optional[B200ByteLevelBPE] = None
        self.bpe_min_token: int = int(bpe_min_token)
        self.bpe_max_token: Optional[int] = None

        if base_tokenizer is not None:
            if args:
                raise TypeError("Positional arguments are not supported when base_tokenizer is provided.")
            if not isinstance(base_tokenizer, BEASTBsplineTokenizer):
                raise TypeError("base_tokenizer must be a BEASTBsplineTokenizer instance.")
            base_state = base_tokenizer.state_dict()
            base_config = base_state.get("config", {}).copy()
            base_config.pop("tokenizer_type", None)
            base_config["use_bpe"] = True
            device_override = kwargs.pop("device", None)
            if kwargs:
                unexpected = ", ".join(sorted(kwargs.keys()))
                raise TypeError(f"Unexpected keyword arguments when base_tokenizer is provided: {unexpected}.")
            if device_override is not None:
                base_config["device"] = device_override
            super().__init__(**base_config)
        else:
            super().__init__(*args, use_bpe=True, **kwargs)

        self._config["bpe_vocab_size"] = bpe_vocab_size
        self._config["tokenizer_type"] = "beast_bspline_bpe"
        self._config["bpe_min_token"] = self.bpe_min_token

        if base_tokenizer is not None:
            self.load_state_dict(base_state)

    def to(self, device):
        super().to(device)
        self.device = device
        self._plan_cache = None
        return self

    # ------------------------------------------------------------------ utilities
    def _require_bpe(self) -> B200ByteLevelBPE:
        if self.bpe_tokenizer is None:
            raise RuntimeError("BPE tokenizer has not been trained. Call fit_from_trajectories() "
                               "or set_bpe_tokenizer() with a trained tokenizer.")
        return self.bpe_tokenizer

    @property
    def sequence_length(self) -> int:
        return self.num_basis * self.num_dof

    def set_bpe_tokenizer(self, tokenizer, *, min_token: int = 0, max_token: Optional[int] = None) -> None:
        self.bpe_tokenizer = _coerce_bpe(tokenizer)
        self.bpe_min_token = int(min_token)
        self.bpe_max_token = None if max_token is None else int(max_token)
        self._config["bpe_min_token"] = self.bpe_min_token

    def fit_from_trajectories(self, trajectories: Iterable[Union[TokenLike, dict]], *, update_bounds: bool = False,
                              batch_key: str = "actions", max_sequences: Optional[int] = None, min_frequency: int = 2,
                              special_tokens: Optional[Sequence[str]] = None, show_progress: bool = True,
                              max_token_length: int = 10000, process_group=None):
        """Train the internal BPE model on the GPU using BEAST discretised tokens (reference :111-146).
        Under torch.distributed (one process per GPU) `trajectories` is this rank's shard."""
        from .beast_bpe_trainer import FIGBPE
        fig_bpe = FIGBPE(vocab_size=self.bpe_vocab_size, min_frequency=min_frequency, special_tokens=special_tokens,
                         show_progress=show_progress, max_token_length=max_token_length, device=self.device,
                         process_group=process_group)
        state = fig_bpe.fit_from_trajectories(self, trajectories, update_bounds=update_bounds, batch_key=batch_key,
                                              max_sequences=max_sequences)
        self.set_bpe_tokenizer(state.tokenizer, min_token=state.min_token, max_token=state.max_token)
        return state

    # ------------------------------------------------------------------ bins <-> ids
    def _as_sequence_list(self, values: TokenLike) -> List[np.ndarray]:
        if isinstance(values, torch.Tensor):
            if values.ndim == 1:
                return [values.detach().cpu().numpy()]
            if values.ndim == 2:
                return [row.detach().cpu().numpy() for row in values]
            raise ValueError("Expected tensor with 1 or 2 dimensions for token sequences.")
        if isinstance(values, np.ndarray):
            if values.ndim == 1:
                return [values]
            if values.ndim == 2:
                return [row for row in values]
            raise ValueError("Expected numpy array with 1 or 2 dimensions for token sequences.")
        if isinstance(values, Sequence) and values and isinstance(values[0], numbers.Integral):
            return [np.asarray(values)]
        return [np.asarray(row) for row in values]  # type: ignore[arg-type]

    def _bins_matrix_groups(self, discrete_tokens: TokenLike, dev):
        """[(row indices, [n, L] int64 CUDA tensor)] — one group per distinct row length."""
        if isinstance(discrete_tokens, torch.Tensor) and discrete_tokens.ndim in (1, 2):
            m = discrete_tokens.reshape(1, -1) if discrete_tokens.ndim == 1 else discrete_tokens
            return m.shape[0], [(None, m.to(dev, torch.int64))]
        seqs = [np.asarray(s).reshape(-1).astype(np.int64) for s in self._as_sequence_list(discrete_tokens)]
        by_len = {}
        for i, s in enumerate(seqs):
            by_len.setdefault(s.size, []).append(i)
        groups = []
        for _, idx in by_len.items():
            groups.append((idx, torch.from_numpy(np.stack([seqs[i] for i in idx])).to(dev)))
        return len(seqs), groups

    def _raise_range(self, status: torch.Tensor):
        bad = int(status.max().item()) if status.numel() else 0
        if bad & 1:
            raise ValueError("Discrete tokens contain values smaller than the configured BPE minimum token.")
        if bad & 2:
            raise ValueError("Discrete tokens contain values greater than the configured BPE maximum token. "
                             "Either retrain the BPE tokenizer with a wider range or disable BPE for this run.")

    def _discrete_to_bpe_csr(self, bins: torch.Tensor):
        """bins [N, L] int64 (CUDA) -> (flat ids int32, offsets int64 [N+1]) on the device."""
        tokenizer = self._require_bpe()
        if bins.shape[1] == 0:
            return (torch.empty(0, device=bins.device, dtype=torch.int32),
                    torch.zeros(bins.shape[0] + 1, device=bins.device, dtype=torch.int64))
        flat, offsets, status = tokenizer.encode_bins(bins, self.bpe_min_token, self.bpe_max_token)
        self._raise_range(status)
        return flat, offsets

    def _discrete_to_bpe(self, discrete_tokens: TokenLike) -> List[List[int]]:
        """Reference :175-198 (shift by bpe_min_token, range checks, HF encode) — one GPU pass per row length."""
        self._require_bpe()
        dev = self._cuda()
        n, groups = self._bins_matrix_groups(discrete_tokens, dev)
        result: List[Optional[List[int]]] = [None] * n
        for idx, bins in groups:
            flat, offsets = self._discrete_to_bpe_csr(bins)
            rows = _split_rows(flat.cpu().numpy(), offsets.cpu().numpy())
            if idx is None:
                return rows
            for j, r in enumerate(rows):
                result[idx[j]] = r
        return result  # type: ignore[return-value]

    def _ids_to_csr(self, tokens: Iterable[TokenLike], dev):
        if isinstance(tokens, torch.Tensor):
            if tokens.ndim == 1:
                token_sequences = [tokens]
            elif tokens.ndim == 2:
                token_sequences = [row for row in tokens]
            else:
                raise ValueError("Expected tensor with 1 or 2 dimensions for BPE tokens.")
        elif isinstance(tokens, np.ndarray):
            if tokens.ndim == 1:
                token_sequences = [tokens]
            elif tokens.ndim == 2:
                token_sequences = [row for row in tokens]
            else:
                raise ValueError("Expected numpy array with 1 or 2 dimensions for BPE tokens.")
        elif isinstance(tokens, Sequence) and tokens and isinstance(tokens[0], numbers.Integral):
            token_sequences = [tokens]
        else:
            token_sequences = tokens
        fast = _flatten_rows(token_sequences) if isinstance(token_sequences, (list, tuple)) and token_sequences else None
        if fast is not None:
            # the ragged List[List[int]] that encode() returns: one C-level pass instead of an int() call per id
            flat32, offsets = fast
            return torch.from_numpy(flat32).to(dev), torch.from_numpy(offsets).to(dev)
        arrays = []
        for token in token_sequences:
            if isinstance(token, torch.Tensor):
                arrays.append(token.detach().cpu().numpy().astype(np.int64).reshape(-1))
            else:
                arrays.append(np.asarray([int(t) for t in token], dtype=np.int64).reshape(-1))
        lens = np.asarray([a.size for a in arrays], dtype=np.int64)
        flat = np.concatenate(arrays) if arrays else np.zeros(0, dtype=np.int64)
        offsets = np.zeros(len(lens) + 1, dtype=np.int64)
        np.cumsum(lens, out=offsets[1:])
        if flat.size and (flat.min() < -2 ** 31 or flat.max() >= 2 ** 31):
            raise ValueError("BPE token id out of range")
        return torch.from_numpy(flat.astype(np.int32)).to(dev), torch.from_numpy(offsets).to(dev)

    def _bpe_csr_to_discrete(self, flat: torch.Tensor, offsets: torch.Tensor) -> torch.Tensor:
        tokenizer = self._require_bpe()
        bins, status, declen = tokenizer.decode_ids(flat, offsets, self.sequence_length, self.bpe_min_token)
        if status.numel() and int(status.max().item()) != 0:
            i = int(torch.nonzero(status)[0].item())
            code = int(status[i].item())
            if code == 1:
                raise ValueError("BPE sequence contains ids outside the vocabulary.")
            if code == 2:
                raise ValueError("BPE sequence does not decode to valid text.")
            raise ValueError(f"Decoded sequence has length {int(declen[i].item())}, expected {self.sequence_length}.")
        return bins

    def _bpe_to_discrete(self, tokens: Iterable[TokenLike]) -> torch.Tensor:
        """Reference :200-247: ids -> token strings -> bytes -> codepoints + bpe_min_token, length checked."""
        self._require_bpe()
        dev = self._cuda()
        flat, offsets = self._ids_to_csr(tokens, dev)
        if offsets.numel() == 1:
            return torch.empty((0, self.sequence_length), dtype=torch.long, device=dev)
        return self._bpe_csr_to_discrete(flat, offsets)

    # ------------------------------------------------------------------ BEAST overridden
    def encode(self, trajs: torch.Tensor, update_bounds: bool = False, *, return_mp_tokens: bool = False,
               times: Optional[torch.Tensor] = None, mask: Optional[torch.Tensor] = None) -> tuple:
        mp_tokens, params = super().encode(trajs, update_bounds=update_bounds, respect_llm_vocab_size=False, times=times,
                                           mask=mask)
        bpe_tokens = self._discrete_to_bpe(mp_tokens)
        if return_mp_tokens:
            return bpe_tokens, params, mp_tokens
        return bpe_tokens, params

    def encode_csr(self, trajs: torch.Tensor, update_bounds: bool = False, *, times: Optional[torch.Tensor] = None,
                   mask: Optional[torch.Tensor] = None):
        """Device-resident variant of `encode`: (flat ids int32, offsets int64 [B+1], params_dict)."""
        mp_tokens, params = super().encode(trajs, update_bounds=update_bounds, respect_llm_vocab_size=False, times=times,
                                           mask=mask)
        flat, offsets = self._discrete_to_bpe_csr(mp_tokens)
        return flat, offsets, params

    def decode(self, tokens: Iterable[TokenLike], *, respect_llm_vocab_size: bool = False) -> torch.Tensor:
        discrete = self._bpe_to_discrete(tokens)
        return super().decode(discrete, respect_llm_vocab_size=respect_llm_vocab_size)

    def encode_to_mp_tokens(self, trajs: torch.Tensor, update_bounds: bool = False, *,
                            times: Optional[torch.Tensor] = None, mask: Optional[torch.Tensor] = None) -> tuple:
        """Expose the underlying MP-token encoding without BPE.  `times` [B, T]: per-row timestamps, `mask` [B, T]:
        the samples to fit (True = fitted, i.e. LeRobot's ~action_is_pad), as in BEASTBsplineTokenizer.encode."""
        return super().encode(trajs, update_bounds=update_bounds, respect_llm_vocab_size=False, times=times, mask=mask)

    def bpe_to_mp_tokens(self, tokens: Iterable[TokenLike]) -> torch.Tensor:
        return self._bpe_to_discrete(tokens)

    def reconstruct_traj(self, tokens: Iterable[TokenLike], times: Optional[torch.Tensor] = None, **kwargs) -> torch.Tensor:
        # the reference reaches its overridden decode() (respect_llm_vocab_size=False) through the base method
        discrete = self._bpe_to_discrete(tokens)
        return self._reconstruct_from_mp_tokens(discrete, 0, times, **kwargs)

    def reconstruct_traj_derivatives(self, tokens: Iterable[TokenLike], times: Optional[torch.Tensor] = None,
                                     orders=(0, 1, 2), **kwargs) -> tuple:
        # ids -> bins exactly as reconstruct_traj above (offset 0)
        orders = check_orders(orders)
        discrete = self._bpe_to_discrete(tokens)
        return self._derivatives_from_mp_tokens(discrete, 0, times, orders, **kwargs)

    def reconstruct_traj_csr(self, flat: torch.Tensor, offsets: torch.Tensor, times=None, **kwargs) -> torch.Tensor:
        return self._reconstruct_from_mp_tokens(self._bpe_csr_to_discrete(flat, offsets), 0, times, **kwargs)

    # ------------------------------------------------------------------ serialization
    def get_config(self):  # type: ignore[override]
        config = super().get_config()
        config["bpe_vocab_size"] = self.bpe_vocab_size
        config["use_bpe"] = True
        return config

    def state_dict(self):  # type: ignore[override]
        state = super().state_dict()
        state["bpe"] = {
            "min_token": self.bpe_min_token,
            "max_token": self.bpe_max_token,
            "vocab_size": self.bpe_vocab_size,
            "tokenizer_dir": self.bpe_subdir if self.bpe_tokenizer is not None else None,
        }
        return state

    def load_state_dict(self, state_dict):  # type: ignore[override]
        super().load_state_dict(state_dict)
        bpe_info = state_dict.get("bpe", {})
        self.bpe_min_token = int(bpe_info.get("min_token", self.bpe_min_token))
        max_token = bpe_info.get("max_token", self.bpe_max_token)
        self.bpe_max_token = None if max_token is None else int(max_token)
        self.bpe_vocab_size = int(bpe_info.get("vocab_size", self.bpe_vocab_size))
        self._config["bpe_min_token"] = self.bpe_min_token

    def save_pretrained(self, save_directory):  # type: ignore[override]
        save_directory = Path(save_directory)
        super().save_pretrained(save_directory)
        if self.bpe_tokenizer is not None:
            bpe_dir = save_directory / self.bpe_subdir
            bpe_dir.mkdir(parents=True, exist_ok=True)
            files = self.bpe_tokenizer.save_model(str(bpe_dir))
            self.bpe_tokenizer.save(str(bpe_dir / "tokenizer.json"))
            saved_files = ", ".join(Path(f).name for f in files)
            print(f"  - BPE tokenizer files: {saved_files} and tokenizer.json in {bpe_dir}")

    @classmethod
    def from_pretrained(cls, pretrained_path, device=None):  # type: ignore[override]
        pretrained_path = Path(pretrained_path)
        config_path = pretrained_path / CONFIG_FILENAME
        if not config_path.exists():
            raise FileNotFoundError(f"Config file not found: {config_path}")
        with open(config_path, "r", encoding="utf-8") as f:
            state = json.load(f)
        config = state["config"].copy()
        tokenizer_type = config.get("tokenizer_type")
        if tokenizer_type not in {"beast_bspline_bpe", None}:
            raise ValueError("Loaded configuration does not describe a BEAST B-Spline BPE tokenizer.")
        config["tokenizer_type"] = "beast_bspline_bpe"
        config["use_bpe"] = True
        if device is not None:
            config["device"] = device
        tokenizer = cls(**config)
        tokenizer.load_state_dict(state)
        bpe_info = state.get("bpe", {})
        bpe_dir_name = bpe_info.get("tokenizer_dir", cls.bpe_subdir)
        bpe_dir = pretrained_path / (bpe_dir_name or cls.bpe_subdir)
        if bpe_dir.exists():
            vocab_path = bpe_dir / "vocab.json"
            merges_path = bpe_dir / "merges.txt"
            if vocab_path.exists() and merges_path.exists():
                tokenizer.bpe_tokenizer = B200ByteLevelBPE.from_file(str(vocab_path), str(merges_path))
        tokenizer.bpe_min_token = int(bpe_info.get("min_token", tokenizer.bpe_min_token))
        max_token = bpe_info.get("max_token", tokenizer.bpe_max_token)
        tokenizer.bpe_max_token = None if max_token is None else int(max_token)
        tokenizer.bpe_vocab_size = int(bpe_info.get("vocab_size", tokenizer.bpe_vocab_size))
        tokenizer._config["bpe_min_token"] = tokenizer.bpe_min_token
        return tokenizer

    @classmethod
    def from_beast(cls, tokenizer: BEASTBsplineTokenizer, *, bpe_vocab_size: Optional[int] = None,
                   device: Optional[Union[str, torch.device]] = None) -> "BEASTBsplineBPETokenizer":
        """Instantiate a BPE-enabled tokenizer from a fitted BEAST tokenizer."""
        if not isinstance(tokenizer, BEASTBsplineTokenizer):
            raise TypeError("tokenizer must be a BEASTBsplineTokenizer instance.")
        init_kwargs = {"base_tokenizer": tokenizer}
        if bpe_vocab_size is not None:
            init_kwargs["bpe_vocab_size"] = bpe_vocab_size
        if device is not None:
            init_kwargs["device"] = device
        return cls(**init_kwargs)

    @classmethod
    def from_bspline_tokenizer(cls, tokenizer: BEASTBsplineTokenizer, *, bpe_vocab_size: Optional[int] = None,
                               device: Optional[Union[str, torch.device]] = None) -> "BEASTBsplineBPETokenizer":
        return cls.from_beast(tokenizer, bpe_vocab_size=bpe_vocab_size, device=device)
