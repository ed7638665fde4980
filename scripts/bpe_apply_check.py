"""Every row of bench.py's BPE apply workload against an independent encoder:  python scripts/bpe_apply_check.py

The bench's bpe_legs table (vocabulary 2048, trained on the GPU from its 1.6 M-sequence corpus) applied to 1 048 576
trajectories: the ids of every row are compared with HF tokenizers' encode_batch on the chr(bin - min) strings
(the C oracle when the wheel is absent), and the decode of the ids with the bins.  Prints the mismatch counts;
exits 1 if any row differs.  The bench itself only compares 64 rows."""
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from beast_tokenizer_b200 import BEASTBsplineBPETokenizer, BEASTBsplineTokenizer, FIGBPE  # noqa: E402
from beast_tokenizer_b200.synth import SyntheticLoader, synth_device  # noqa: E402

dev = torch.device("cuda:0")
tok = BEASTBsplineTokenizer(num_dof=bench.D, num_basis=bench.NB, seq_len=bench.T, vocab_size=bench.V,
                            gripper_zero_order=True, gripper_indices=bench.GRIP, device="cuda:0",
                            llm_vocab_size=bench.LLM_VOCAB)
tok.fit_parameters(SyntheticLoader(100, 32, bench.T, bench.D, seed0=1), verbose=False)
per_chunk = bench.BPE_BATCHES * bench.BPE_BATCH // bench.BPE_CHUNKS
corpus = torch.cat([tok.encode(synth_device(per_chunk, bench.T, bench.D, 1000 + c, dev), respect_llm_vocab_size=False)[0]
                    for c in range(bench.BPE_CHUNKS)])
state = FIGBPE(vocab_size=bench.BPE_VOCAB, show_progress=False, device="cuda:0").fit_from_bins(corpus)
del corpus
btok = BEASTBsplineBPETokenizer.from_beast(tok, bpe_vocab_size=bench.BPE_VOCAB, device="cuda:0")
btok.set_llm_vocab_size(None)
btok.set_bpe_tokenizer(state.tokenizer, min_token=state.min_token, max_token=state.max_token)
n = 1 << 20
mp, _ = btok.encode_to_mp_tokens(synth_device(n, bench.T, bench.D, 5, dev))
flat, offsets = btok._discrete_to_bpe_csr(mp)
back = btok._bpe_csr_to_discrete(flat, offsets)
decode_bad = int((back != mp).any(1).sum())
fl, of = flat.cpu().numpy(), offsets.cpu().numpy()
rows = mp.cpu().numpy() - state.min_token
t0 = time.perf_counter()
try:
    hf = state.tokenizer.to_hf()
    engine = "HF tokenizers encode_batch"
    text = rows.astype("<u4").tobytes().decode("utf-32-le")
    L = rows.shape[1]
    want = hf.encode_batch([text[i * L:(i + 1) * L] for i in range(n)], add_special_tokens=False)
    lens = np.array([len(e.ids) for e in want])
    ids = np.fromiter((t for e in want for t in e.ids), dtype=np.int64, count=int(lens.sum()))
except ImportError:
    from oracle.bpe_oracle import OracleBPE
    engine = "C oracle"
    o = OracleBPE.from_strings(state.tokenizer.get_vocab(), [f"{a} {b}" for a, b in state.tokenizer.merge_strings()])
    ids, off = o.encode_batch(rows)
    lens = np.diff(off)
want_off = np.concatenate([[0], np.cumsum(lens)])
bad = np.diff(of) != lens
same_len = np.flatnonzero(~bad)
if same_len.size and not np.array_equal(fl, ids) and not bad.any():
    pos = np.flatnonzero(fl != ids)
    bad[np.unique(np.searchsorted(of, pos, side="right") - 1)] = True
elif bad.any():                          # lengths differ somewhere: compare the rows of equal length one by one
    for i in same_len:
        if not np.array_equal(fl[of[i]:of[i + 1]], ids[want_off[i]:want_off[i + 1]]):
            bad[i] = True
print(f"reference: {engine} ({time.perf_counter() - t0:.1f} s); table: {len(state.tokenizer.merges)} merges")
print(f"encode: {int(bad.sum())} of {n} rows differ" + (f", first {np.flatnonzero(bad)[:10].tolist()}" if bad.any() else ""))
print(f"decode: {decode_bad} of {n} rows differ from the bins")
sys.exit(1 if bad.any() or decode_bad else 0)
