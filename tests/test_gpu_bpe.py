"""GPU BPE path (trainer, encode, decode) against the reference's golden files and the C oracle.
Run on the B200 box:  pytest -m gpu."""
import json
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN, GOLDEN_CASES, load_golden, rel_err
from oracle.bpe_oracle import OracleBPE

pytestmark = pytest.mark.gpu


def ref_files(name):
    d = os.path.join(GOLDEN, f"{name}_pretrained", "bpe_tokenizer")
    return (open(os.path.join(d, "vocab.json"), encoding="utf-8").read(),
            open(os.path.join(d, "merges.txt"), encoding="utf-8").read(),
            open(os.path.join(d, "tokenizer.json"), encoding="utf-8").read())


def ragged(g):
    return [r.tolist() for r in np.split(g["ids_flat"], np.cumsum(g["ids_len"])[:-1])]


@pytest.mark.parametrize("name", ["bpe_d14", "bpe_d14_small", "bpe_v1000"])
def test_trainer_reproduces_reference_files(name):
    from beast_tokenizer_b200 import FIGBPE
    g = load_golden(name)
    vocab_json, merges_txt, tok_json = ref_files(name)
    fig = FIGBPE(vocab_size=int(g["bpe_vocab_size"]), show_progress=False)
    state = fig.fit_from_bins(torch.from_numpy(g["corpus_bins"].astype(np.int64)).cuda())
    assert (state.min_token, state.max_token) == (int(g["min_token"]), int(g["max_token"]))
    assert state.tokenizer.merges_txt() == merges_txt            # byte-identical merges.txt
    assert state.tokenizer.vocab_json() == vocab_json            # byte-identical vocab.json
    assert state.tokenizer.tokenizer_json() == tok_json          # and tokenizer.json
    # the list-of-rows entry point of the reference API
    st2 = FIGBPE(vocab_size=int(g["bpe_vocab_size"]), show_progress=False).fit_from_sequences(
        [row for row in g["corpus_bins"][:64].astype(np.int64)])
    o = OracleBPE.train(g["corpus_bins"][:64].astype(np.int64), int(g["bpe_vocab_size"]))
    assert st2.tokenizer.merges_txt() == o.merges_txt() and st2.tokenizer.vocab_json() == o.vocab_json()


@pytest.mark.parametrize("name", ["bpe_d14", "bpe_d14_small", "bpe_v1000"])
def test_encode_decode_vs_reference(name):
    from beast_tokenizer_b200 import BEASTBsplineBPETokenizer
    g = load_golden(name)
    g2 = load_golden("cfg2_d14")
    tok = BEASTBsplineBPETokenizer.from_pretrained(os.path.join(GOLDEN, f"{name}_pretrained"), device="cuda")
    want = ragged(g)
    mp = torch.from_numpy(g["mp_tokens"])
    assert tok._discrete_to_bpe(mp) == want                       # ids bit-exact
    assert tok._discrete_to_bpe(g["mp_tokens"]) == want            # numpy input
    assert tok._discrete_to_bpe([r.tolist() for r in g["mp_tokens"][:5]]) == want[:5]
    assert tok._discrete_to_bpe(g["mp_tokens"][3].tolist()) == [want[3]]
    back = tok.bpe_to_mp_tokens(want)
    assert back.dtype == torch.long and back.is_cuda and np.array_equal(back.cpu().numpy(), g["mp_tokens"])
    assert np.array_equal(tok.decode(want).cpu().numpy(), g["decode"])
    assert rel_err(tok.reconstruct_traj(want).cpu().numpy(), g["recon"]) <= 1e-5
    # full pipeline from trajectories: ids equal wherever the MP tokens equal the reference's
    ids, pd, mp_ours = tok.encode(torch.from_numpy(g2["trajs"]), return_mp_tokens=True)
    same = (mp_ours.cpu().numpy() == g["mp_tokens"]).all(1)
    assert same.mean() > 0.9
    for i in np.nonzero(same)[0]:
        assert ids[i] == want[i]
    flat, offsets, _ = tok.encode_csr(torch.from_numpy(g2["trajs"]))
    assert flat.dtype == torch.int32 and offsets[-1].item() == sum(len(r) for r in ids)
    assert torch.equal(tok.reconstruct_traj_csr(flat, offsets), tok.reconstruct_traj(ids))
    # ragged API shapes
    out2 = tok.encode(torch.from_numpy(g2["trajs"][:4]))
    assert len(out2) == 2 and isinstance(out2[0], list) and isinstance(out2[0][0], list)


@pytest.mark.parametrize("kind,n,vocab", [("uniform", 20000, 1024), ("normal", 30000, 2048), ("letters", 3000, 700),
                                          ("narrow", 4000, 400), ("bins1000", 6000, 1800), ("bins5000", 2000, 5600),
                                          ("quotes", 6000, 420), ("quotes_thread_kernel", 1500, 380)])
def test_trainer_vs_oracle_large(kind, n, vocab, monkeypatch):
    """Synthetic corpora at sizes the C oracle trains in seconds: merges, vocabulary and ids identical."""
    from beast_tokenizer_b200 import FIGBPE
    rng = np.random.default_rng(3)
    if kind == "uniform":
        bins = rng.integers(0, 256, (n, 140))
    elif kind == "normal":
        bins = np.clip(rng.normal(128, 28, (n, 140)).round(), 0, 255).astype(np.int64)
    elif kind == "letters":                                        # long pre-tokens, repeated symbols (aaa -> Xa)
        bins = rng.choice([97, 97, 97, 98, 99, 32], (n, 60)) + 7
    elif kind == "bins1000":                                       # 1000-bin tokenizer: 2-byte UTF-8, classes past Latin-1
        bins = np.clip(rng.normal(500, 120, (n, 140)).round(), 0, 999).astype(np.int64)
    elif kind == "bins5000":                                       # 3-byte UTF-8
        bins = rng.integers(0, 5000, (n, 100))
    elif kind.startswith("quotes"):                                # contractions, blank / tab / NBSP runs, digits
        alphabet = [39, 39, 39, 32, 32, 32, 9, 10, 160] + [ord(ch) for ch in "stmdrevla12!?"] + [200, 178]
        bins = rng.choice(alphabet, (n, 57)) + 3
        if kind == "quotes_thread_kernel":                         # the one-thread-per-sequence encode kernel
            monkeypatch.setenv("BEAST_B200_BPE_THREAD_ENCODE", "1")
    else:
        bins = rng.integers(40, 91, (n, 140))
    o = OracleBPE.train(bins, vocab)
    state = FIGBPE(vocab_size=vocab, show_progress=False).fit_from_bins(torch.from_numpy(bins).cuda())
    assert state.tokenizer.merges_txt() == o.merges_txt()
    assert state.tokenizer.vocab_json() == o.vocab_json()
    assert (state.min_token, state.max_token) == (o.min_token, o.max_token)
    # encode / decode a held-out batch (includes values never seen in training for "narrow")
    test = np.concatenate([rng.permuted(bins[:256], axis=1),        # seen values in new orders
                           rng.integers(int(bins.min()), int(bins.max()) + 1, (256, bins.shape[1]))])
    flat, offsets, status = state.tokenizer.encode_bins(torch.from_numpy(test).cuda(), state.min_token, state.max_token)
    assert int(status.max()) == 0
    fl, of = flat.cpu().numpy(), offsets.cpu().numpy()
    for i in range(0, 512, 1 if kind.startswith("quotes") else 7):
        assert fl[of[i]:of[i + 1]].tolist() == o.encode(test[i] - o.min_token)
    dec, st, ln = state.tokenizer.decode_ids(flat, offsets, bins.shape[1], state.min_token)
    dec, st, ln = dec.cpu().numpy(), st.cpu().numpy(), ln.cpu().numpy()
    dropped = 0
    for i in range(512):
        try:
            want = o.decode(fl[of[i]:of[i + 1]]) + o.min_token
        except ValueError:        # a dropped continuation byte leaves invalid UTF-8 (HF would emit U+FFFD)
            dropped += 1
            assert st[i] == 2
            continue
        if want.size == bins.shape[1]:
            assert st[i] == 0 and np.array_equal(dec[i], test[i])
        else:                     # a bin never seen in training lost its symbol (SURVEY.md A.5): the reference's
            dropped += 1          # length ValueError, reported here as status 3 with the decoded length
            assert st[i] == 3 and ln[i] == want.size
    assert (st[:256] == 0).all()


def test_fit_from_trajectories_and_files(tmp_path):
    from beast_tokenizer_b200 import BEASTBsplineBPETokenizer, BEASTBsplineTokenizer, FIGBPEState
    from beast_tokenizer_b200.synth import SyntheticLoader, synth
    g2 = load_golden("cfg2_d14")
    cfg = {k: v for k, v in GOLDEN_CASES["cfg2_d14"].items() if k != "llm_vocab_size"}
    base = BEASTBsplineTokenizer(device="cuda", **cfg)
    base.w_min.copy_(torch.from_numpy(g2["w_min_fit"])); base.w_max.copy_(torch.from_numpy(g2["w_max_fit"]))
    tok = BEASTBsplineBPETokenizer.from_beast(base, bpe_vocab_size=512)
    with pytest.raises(RuntimeError):
        tok.encode(synth(2, 50, 14, 0))
    loader = SyntheticLoader(30, 32, 50, 14, seed0=1000)
    state = tok.fit_from_trajectories(loader, show_progress=False, max_sequences=900)
    assert isinstance(state, FIGBPEState) and tok.bpe_tokenizer is state.tokenizer
    corpus = torch.cat([tok.encode_to_mp_tokens(b["actions"])[0] for b in loader])[:900].cpu().numpy()
    o = OracleBPE.train(corpus, 512)
    assert state.tokenizer.merges_txt() == o.merges_txt() and state.tokenizer.vocab_json() == o.vocab_json()
    assert (tok.bpe_min_token, tok.bpe_max_token) == (o.min_token, o.max_token)
    x = synth(40, 50, 14, seed=9)
    ids, pd, mp = tok.encode(x, return_mp_tokens=True)
    for i in range(40):
        assert ids[i] == o.encode(mp[i].cpu().numpy() - o.min_token)
    assert torch.equal(tok.bpe_to_mp_tokens(ids), mp)
    assert torch.equal(tok.reconstruct_traj(ids), base.reconstruct_traj(mp))
    tok.save_pretrained(tmp_path)
    tok2 = BEASTBsplineBPETokenizer.from_pretrained(tmp_path, device="cuda")
    assert tok2.encode(x)[0] == ids and tok2.bpe_max_token == tok.bpe_max_token
    hf = pytest.importorskip("tokenizers")
    ref_tok = hf.ByteLevelBPETokenizer.from_file(str(tmp_path / "bpe_tokenizer" / "vocab.json"),
                                                 str(tmp_path / "bpe_tokenizer" / "merges.txt"))
    row = mp[0].cpu().numpy() - tok.bpe_min_token
    assert ref_tok.encode("".join(map(chr, row)), add_special_tokens=False).ids == ids[0]   # the library reads our files
    tok3 = BEASTBsplineBPETokenizer.from_beast(base, bpe_vocab_size=512)
    tok3.set_bpe_tokenizer(ref_tok, min_token=tok.bpe_min_token, max_token=tok.bpe_max_token)   # and we read its objects
    assert tok3.encode(x)[0] == ids
    with pytest.raises(TypeError):
        tok3.set_bpe_tokenizer(object())


def test_fit_from_trajectories_gathers_host_and_device_batches_in_order():
    """Reference beast/beast_bpe_trainer.py:100-151 encodes the loader batch by batch; here small batches are gathered
    (device batches in a device block, host batches beyond the first block in pinned blocks uploaded 4 096 rows at a
    time).  The bins handed to the trainer must be the loader's trajectories in the loader's order, whatever mix of
    host / device / float64 / oversized batches arrives."""
    from beast_tokenizer_b200 import BEASTBsplineTokenizer, FIGBPE
    from beast_tokenizer_b200.synth import synth
    tok = BEASTBsplineTokenizer(num_dof=14, num_basis=10, seq_len=50, vocab_size=256, gripper_zero_order=True,
                                gripper_indices=[6, 13], device="cuda")
    x = synth(15000, 50, 14, seed=21)
    tok.update_weights_bounds(x)
    want, _ = tok.encode(x)
    cuts = list(range(0, 9600, 32)) + [9600, 9607, 9700, 9700 + 4096 + 5, 14000, 14033, 15000]
    assert cuts == sorted(cuts)
    loader = []
    for j, (a, b) in enumerate(zip(cuts[:-1], cuts[1:])):
        part = x[a:b]
        if j % 7 == 3:
            part = part.cuda()                         # a device batch in the middle of host batches
        elif j % 11 == 5:
            part = part.double()                       # converted on the way into the pinned block
        loader.append({"actions": part} if j % 2 else part)
    got = {}
    fig = FIGBPE(vocab_size=300, show_progress=False, device="cuda", process_group=False)
    fig.fit_from_bins = lambda bins: got.setdefault("bins", bins)
    fig.fit_from_trajectories(tok, loader)
    assert torch.equal(got["bins"], want)
    got.clear()
    fig.fit_from_trajectories(tok, loader, max_sequences=9000)
    assert torch.equal(got["bins"], want[:9000])


def test_bpe_errors():
    from beast_tokenizer_b200 import BEASTBsplineBPETokenizer
    g = load_golden("bpe_d14")
    tok = BEASTBsplineBPETokenizer.from_pretrained(os.path.join(GOLDEN, "bpe_d14_pretrained"), device="cuda")
    mp = g["mp_tokens"][:4].copy()
    tok.bpe_min_token, tok.bpe_max_token = 5, 200
    bad = mp.copy(); bad[1, 3] = 2
    with pytest.raises(ValueError, match="smaller than the configured BPE minimum"):
        tok._discrete_to_bpe(np.clip(bad, 2, 200))
    bad = np.clip(mp, 5, 200); bad[2, 7] = 231
    with pytest.raises(ValueError, match="greater than the configured BPE maximum"):
        tok._discrete_to_bpe(bad)
    tok.bpe_min_token, tok.bpe_max_token = 0, 255
    ids = tok._discrete_to_bpe(mp)
    with pytest.raises(ValueError, match="Decoded sequence has length"):
        tok.bpe_to_mp_tokens([ids[0][:-1], ids[1]])
    with pytest.raises(ValueError):
        tok.bpe_to_mp_tokens([[10 ** 6]])
    with pytest.raises(ValueError):
        tok._discrete_to_bpe(torch.zeros(2, 2, 2, dtype=torch.long))
    assert tok._discrete_to_bpe(torch.zeros(0, 140, dtype=torch.long)) == []


def test_train_cli_flow(tmp_path):
    """The reference's train_beast.py flow (fit -> save -> BPE -> save -> eval) on synthetic loaders,
    at a 256-bin configuration the BPE path supports."""
    from beast_tokenizer_b200 import BEASTBsplineBPETokenizer
    from beast_tokenizer_b200.train_beast import main
    main(["--device", "cuda", "--num-basis", "10", "--degree", "4", "--vocab-size", "256", "--actions-len", "50",
          "--actions-dof", "14", "--train-batches", "40", "--eval-batches", "5", "--bpe-vocab-size", "500",
          "--beast-checkpoint-dir", str(tmp_path / "beast"), "--bpe-checkpoint-dir", str(tmp_path / "bpe"),
          "--eval-results-dir", str(tmp_path / "eval")])
    stats = json.load(open(tmp_path / "eval" / "total_stats.json"))["synthetic"]
    assert set(stats) == {f"{a}_{b}" for a in ("mean", "std", "max", "min") for b in ("l2", "l1")}
    assert 0 <= stats["mean_l2"] < 1e-4
    tok = BEASTBsplineBPETokenizer.from_pretrained(tmp_path / "bpe", device="cuda")
    assert tok.bpe_tokenizer.get_vocab_size() == 500
    errs = json.load(open(tmp_path / "eval" / "synthetic" / "errors.json"))
    assert len(errs["errors_l2"]) == 5 and len(errs["mean_tokens_length"]) == 5 * 32


def test_train_cli_flow_reference_defaults(tmp_path):
    """The reference's train.sh configuration: 50 basis functions, degree 0, 1000 bins, actions [10, 32]
    (sequences of 1600 bins, 2-byte UTF-8) — fit, BPE with vocab 2048, save, evaluate."""
    from beast_tokenizer_b200 import BEASTBsplineBPETokenizer
    from beast_tokenizer_b200.train_beast import main
    from beast_tokenizer_b200.synth import synth
    main(["--device", "cuda", "--train-batches", "12", "--eval-batches", "3", "--bpe-vocab-size", "2048",
          "--beast-checkpoint-dir", str(tmp_path / "beast"), "--bpe-checkpoint-dir", str(tmp_path / "bpe"),
          "--eval-results-dir", str(tmp_path / "eval")])
    tok = BEASTBsplineBPETokenizer.from_pretrained(tmp_path / "bpe", device="cuda")
    assert tok.sequence_length == 1600 and tok.vocab_size == 1000
    x = synth(6, 10, 32, seed=5)
    ids, pd, mp = tok.encode(x, return_mp_tokens=True)
    o = OracleBPE.from_strings(tok.bpe_tokenizer.get_vocab(), [f"{a} {b}" for a, b in tok.bpe_tokenizer.merge_strings()])
    for i in range(6):
        assert ids[i] == o.encode(mp[i].cpu().numpy() - tok.bpe_min_token)
    assert torch.equal(tok.bpe_to_mp_tokens(ids), mp)
    corpus = torch.cat([tok.encode_to_mp_tokens(b["actions"])[0] for b in
                        __import__("beast_tokenizer_b200.synth", fromlist=["SyntheticLoader"]).SyntheticLoader(12, 32, 10, 32, seed0=0)])
    o2 = OracleBPE.train(corpus.cpu().numpy(), 2048)
    assert tok.bpe_tokenizer.merges_txt() == o2.merges_txt()


def test_decode_kernels_agree_on_garbage(monkeypatch):
    """The warp-per-sequence decode and the one-thread-per-sequence decode (the sequential UTF-8 state
    machine) must report the same status for arbitrary id streams: random ids give stray continuation
    bytes, truncated characters, ids out of range, wrong lengths — and a few valid rows."""
    from beast_tokenizer_b200 import FIGBPE
    rng = np.random.default_rng(11)
    bins = np.clip(rng.normal(500, 150, (3000, 60)).round(), 0, 999).astype(np.int64)     # 2-byte UTF-8 symbols
    state = FIGBPE(vocab_size=1500, show_progress=False).fit_from_bins(torch.from_numpy(bins).cuda())
    tk = state.tokenizer
    n_vocab = len(tk.tokens)
    good, goff, st = tk.encode_bins(torch.from_numpy(bins[:200]).cuda(), state.min_token, state.max_token)
    good, goff = good.cpu().numpy(), goff.cpu().numpy()
    rows = [good[goff[i]:goff[i + 1]] for i in range(200)]                                # valid rows
    for i in range(600):
        kind = i % 6
        if kind == 0:                                                                       # random ids, random length
            rows.append(rng.integers(0, n_vocab, int(rng.integers(0, 140))))
        elif kind == 1:                                                                     # a valid row with one id replaced
            r = rows[i % 200].copy(); r[rng.integers(0, len(r))] = rng.integers(0, n_vocab); rows.append(r)
        elif kind == 2:                                                                     # id out of range somewhere
            r = rows[i % 200].copy(); r[rng.integers(0, len(r))] = n_vocab + int(rng.integers(0, 5)); rows.append(r)
        elif kind == 3:                                                                     # negative id after garbage
            r = rng.integers(0, n_vocab, 20); r[rng.integers(0, 20)] = -1; rows.append(r)
        elif kind == 4:                                                                     # truncated / extended valid rows
            r = rows[i % 200]; rows.append(np.concatenate([r[:len(r) // 2], r[:int(rng.integers(0, 4))]]))
        else:                                                                               # far too long: overflow path
            rows.append(rng.integers(0, n_vocab, 400))
    flat = torch.from_numpy(np.concatenate(rows).astype(np.int32)).cuda()
    offs = torch.from_numpy(np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.int64)).cuda()
    out = {}
    for mode in ("0", "1"):
        monkeypatch.setenv("BEAST_B200_BPE_THREAD_DECODE", mode)
        dec, stt, ln = tk.decode_ids(flat, offs, 60, state.min_token)
        out[mode] = (dec.cpu().numpy(), stt.cpu().numpy(), ln.cpu().numpy())
    (d0, s0, l0), (d1, s1, l1) = out["0"], out["1"]
    assert np.array_equal(s0, s1), np.flatnonzero(s0 != s1)[:10]
    assert set(np.unique(s0)) >= {0, 1, 2, 3}
    ok = s0 == 0
    assert ok[:200].all() and np.array_equal(d0[ok], d1[ok]) and np.array_equal(d0[:200], bins[:200])
    len_known = (s0 == 0) | (s0 == 3)
    assert np.array_equal(l0[len_known], l1[len_known])


def test_peer_fused_delta_reduction_two_ranks_on_one_gpu():
    """The sharded trainer's per-merge all-reduce lives inside bpe_iterate_kernel (peer loads of the other ranks'
    delta blocks, epoch flags, no host round).  Here two 'ranks' share ONE GPU: two engines, two streams, each
    rank's delta / flags are the other's peers; their iteration heads spin on each other's flags, so both grids
    must be co-resident (grid_blocks = half the SMs).  Every rank must log exactly the merges of the unsharded run."""
    import ctypes as C
    from beast_tokenizer_b200 import _lib
    from beast_tokenizer_b200.beast_bpe_trainer import GpuBpeEngine, _Collective, build_alphabet, scan_bins_gpu, train_bpe
    rng = np.random.default_rng(21)
    bins = np.clip(rng.normal(128, 30, (6000, 140)).round(), 0, 255).astype(np.int64)
    bins[::3] = np.clip(bins[::3] + 40, 0, 255)
    vocab = 700
    dev = torch.device("cuda", torch.cuda.current_device())
    full = torch.from_numpy(bins).to(dev)
    ref, mn0, mx0 = train_bpe(full, vocab, 2, coll=_Collective(enabled=False))
    mn, mx, seen = scan_bins_gpu(full, _Collective(enabled=False))
    tokens, b2i = build_alphabet(mn, mx, seen)
    world = 2
    engs = [GpuBpeEngine(full[r::world].contiguous(), mn, b2i, vocab, mx - mn) for r in range(world)]
    hist = sum(e.hist for e in engs)
    for e in engs:
        e.hist.copy_(hist)
    deltas = [torch.zeros(8 * vocab, device=dev, dtype=torch.int32) for _ in range(world)]
    flags = [torch.zeros(_lib.BPE_MAX_PEERS, device=dev, dtype=torch.int32) for _ in range(world)]
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    runs = []
    for r in range(world):
        p = _lib.BpePeers()
        p.world, p.rank, p.grid_blocks, p.epoch_base = world, r, max(1, sms // 2 - 4), 0
        for q in range(world):
            p.delta[q] = deltas[q].data_ptr()
            p.flags[q] = flags[q].data_ptr()
        runs.append(engs[r].start_run(len(tokens), vocab, 2, peers=p, delta=deltas[r]))
    torch.cuda.synchronize()
    streams = [torch.cuda.Stream(device=dev) for _ in range(world)]
    while not all(run.finished for run in runs):
        for r in range(world):                            # one iteration per rank and turn: neither queue runs ahead
            with torch.cuda.stream(streams[r]):
                runs[r].enqueue(limit=1)
    torch.cuda.synchronize()
    logs = [run.finish() for run in runs]
    assert logs[0] == logs[1]
    assert [(a, b, c) for a, b, c, _ in logs[0]] == list(ref.merges)
    assert len(logs[0]) == vocab - len(tokens)
    for e in engs:                                        # replicas stayed identical
        assert torch.equal(e.hist, engs[0].hist)


def test_ragged_sequences_and_special_tokens_vs_oracle():
    """FIGBPE.fit_from_sequences with sequences of unequal length and BpeTrainer special tokens (reference
    beast/beast_bpe_trainer.py:46, 53, 76-98): vocabulary / merges identical to the oracle (itself pinned to the
    library on such inputs); tokenizer.json lists the special tokens as added tokens; decode skips their ids."""
    from beast_tokenizer_b200 import FIGBPE
    rng = np.random.default_rng(23)
    cases = [
        ([rng.integers(40, 100, int(rng.integers(1, 60))) for _ in range(3000)], 300, []),
        ([rng.integers(0, 256, int(rng.integers(5, 140))) for _ in range(4000)], 900, ["<pad>", "<eos>", "<pad>"]),
        ([rng.integers(30, 90, 50) for _ in range(2000)], 330, ["<s>", chr(5), "ab"]),
        ([rng.integers(0, 900, int(rng.integers(2, 80))) for _ in range(3000)], 1300, ["<unk>"]),
    ]
    for rows, vs, special in cases:
        o = OracleBPE.train_ragged(rows, vs, special_tokens=special)
        fig = FIGBPE(vocab_size=vs, show_progress=False, special_tokens=special)
        st = fig.fit_from_sequences([torch.from_numpy(r) if i % 2 else r.tolist() for i, r in enumerate(rows)])
        assert (st.min_token, st.max_token) == (o.min_token, o.max_token)
        assert st.tokenizer.vocab_json() == o.vocab_json()
        assert st.tokenizer.merges_txt() == o.merges_txt()
        doc = json.loads(st.tokenizer.tokenizer_json())
        uniq = list(dict.fromkeys(special))
        assert [(t["id"], t["content"], t["special"]) for t in doc["added_tokens"]] == [(i, t, True) for i, t in enumerate(uniq)]
    # encode / decode with a model that carries special tokens: ids follow the shifted vocabulary, special ids decode
    # to nothing (skip_special_tokens), a row that spells a special token is refused
    rows, vs, special = cases[1]
    st = FIGBPE(vocab_size=vs, show_progress=False, special_tokens=special).fit_from_sequences(rows)
    o = OracleBPE.train_ragged(rows, vs, special_tokens=special)
    test = np.stack([r[:5] for r in rows[:64]])
    flat, offs, status = st.tokenizer.encode_bins(torch.from_numpy(test).cuda(), st.min_token, st.max_token)
    fl, of = flat.cpu().numpy(), offs.cpu().numpy()
    for i in range(64):
        assert fl[of[i]:of[i + 1]].tolist() == o.encode(test[i] - o.min_token)
    with_special = torch.cat([torch.tensor([0, 1], dtype=torch.int32, device="cuda"), flat[of[0]:of[1]]])
    dec, stt, ln = st.tokenizer.decode_ids(with_special, torch.tensor([0, with_special.numel()], device="cuda"), 5, st.min_token)
    assert int(stt[0]) == 0 and np.array_equal(dec[0].cpu().numpy(), test[0])
    spelled = test.copy()
    spelled[3, :5] = np.array([ord(c) for c in "<pad>"]) + st.min_token
    with pytest.raises(NotImplementedError):
        st.tokenizer.encode_bins(torch.from_numpy(spelled).cuda(), st.min_token, st.max_token)
    # the reloaded model (vocab.json + merges.txt, as the reference's from_pretrained) no longer knows them
    from beast_tokenizer_b200 import B200ByteLevelBPE
    re = B200ByteLevelBPE.from_vocab_merges(st.tokenizer.get_vocab(), st.tokenizer.merge_strings())
    assert re.special_tokens == [] and re.encode_bins(torch.from_numpy(spelled).cuda(), st.min_token, st.max_token)[2].max() == 0


def test_vocab_limits_are_reported_up_front():
    from beast_tokenizer_b200 import FIGBPE
    bins = torch.randint(0, 256, (64, 20), device="cuda")
    with pytest.raises(NotImplementedError, match="trainer's limit"):
        FIGBPE(vocab_size=40000, show_progress=False).fit_from_bins(bins)


def test_large_vocabulary_trains_and_applies():
    """bpe_vocab_size above 12 800 (no block-private delta counters in the rewrite kernel) and above 4 096 (hashed merge
    ranks in the encode kernel): the table must equal the library's, ids must round-trip."""
    tk = pytest.importorskip("tokenizers")
    from tokenizers import ByteLevelBPETokenizer
    from tokenizers.trainers import BpeTrainer
    from beast_tokenizer_b200 import FIGBPE
    rng = np.random.default_rng(61)
    base = rng.integers(0, 3000, (600, 80))
    bins = np.concatenate([base[rng.integers(0, 600, 9000)], rng.integers(0, 3000, (3000, 80))])    # repeats => many merges
    vocab = 14500
    st = FIGBPE(vocab_size=vocab, show_progress=False).fit_from_bins(torch.from_numpy(bins).cuda())
    mn, mx = int(bins.min()), int(bins.max())
    hf = ByteLevelBPETokenizer()
    trainer = BpeTrainer(vocab_size=vocab, min_frequency=2, show_progress=False, special_tokens=[],
                         initial_alphabet=[chr(i) for i in range(mx - mn + 1)], max_token_length=10000)
    hf._tokenizer.train_from_iterator(["".join(map(chr, r - mn)) for r in bins], trainer=trainer)
    model = json.loads(hf._tokenizer.to_str())["model"]
    hf_merges = [m if isinstance(m, str) else " ".join(m) for m in model["merges"]]
    assert len(st.tokenizer.merges) > 9000
    assert [f"{a} {b}" for a, b in st.tokenizer.merge_strings()] == hf_merges
    assert st.tokenizer.get_vocab() == hf.get_vocab()
    test = torch.from_numpy(bins[:400]).cuda()
    flat, offs, status = st.tokenizer.encode_bins(test, st.min_token, st.max_token)
    assert st.tokenizer._tables(test.device)["hash_bits"] > 0 and int(status.max()) == 0
    fl, of = flat.cpu().numpy(), offs.cpu().numpy()
    for i in range(0, 400, 17):
        assert fl[of[i]:of[i + 1]].tolist() == hf.encode("".join(map(chr, bins[i] - mn)), add_special_tokens=False).ids
    back, stt, _ = st.tokenizer.decode_ids(flat, offs, 80, st.min_token)
    assert int(stt.max()) == 0 and torch.equal(back, test)


@pytest.mark.parametrize("kind", ["repetitive", "iid", "letters", "bins1000"])
def test_word_dedup_gives_the_same_table(kind):
    """Training on the distinct pre-tokens with counts (SURVEY.md §8(f)4, what BpeTrainer does) must give exactly
    the table of the plain run and of the oracle — on a repetitive corpus (few distinct trajectories drawn many
    times), on an i.i.d. one, on long repeated-symbol words and on 2-byte symbols."""
    from beast_tokenizer_b200 import FIGBPE
    rng = np.random.default_rng(31)
    if kind == "repetitive":
        base = np.clip(rng.normal(128, 30, (300, 140)).round(), 0, 255).astype(np.int64)
        bins, vocab = base[rng.integers(0, 300, 20000)], 1200
    elif kind == "iid":
        bins, vocab = np.clip(rng.normal(128, 28, (8000, 140)).round(), 0, 255).astype(np.int64), 900
    elif kind == "letters":
        bins, vocab = rng.choice([97, 97, 97, 98, 99, 32], (3000, 60)) + 7, 500
    else:
        base = np.clip(rng.normal(500, 120, (500, 140)).round(), 0, 999).astype(np.int64)
        bins, vocab = np.concatenate([base[rng.integers(0, 500, 5000)], rng.integers(0, 1000, (500, 140))]), 1800
    o = OracleBPE.train(bins, vocab)
    dev_bins = torch.from_numpy(bins).cuda()
    tables = {}
    for mode in (True, False, "auto"):
        st = FIGBPE(vocab_size=vocab, show_progress=False, dedup=mode).fit_from_bins(dev_bins)
        tables[mode] = (st.tokenizer.merges_txt(), st.tokenizer.vocab_json())
        stats = st.tokenizer.dedup_stats
        if mode is True:
            assert stats["applied"] and stats["distinct_symbols"] <= stats["symbols"], stats
            if kind == "repetitive":
                assert stats["distinct_symbol_ratio"] < 0.1, stats
        if mode is False:
            assert stats is None
    assert tables[True] == tables[False] == tables["auto"] == (o.merges_txt(), o.vocab_json())
    # the exact host-driven loop (progress display off the fast path is no longer a separate loop; force it through
    # a vocabulary that re-creates an existing token string is covered elsewhere) also takes the weights:
    from beast_tokenizer_b200.beast_bpe_trainer import GpuBpeEngine, _Collective, build_alphabet, scan_bins_gpu
    mn, mx, seen = scan_bins_gpu(dev_bins, _Collective(enabled=False))
    tokens, b2i = build_alphabet(mn, mx, seen)
    engs = [GpuBpeEngine(dev_bins, mn, b2i, vocab, mx - mn, None, d) for d in (True, False)]
    assert engs[0].weight is not None and engs[1].weight is None
    assert torch.equal(engs[0].hist, engs[1].hist)                 # weighted initial counts == plain counts
    n_tok = len(tokens)
    for step in range(40):
        picks = [e.argmax(n_tok) for e in engs]
        assert picks[0] == picks[1]
        cnt, a, b = picks[0]
        for e in engs:
            e.merge(a, b, n_tok)
            e.apply_delta(a, b, n_tok)
        n_tok += 1
    assert torch.equal(engs[0].hist, engs[1].hist)


@pytest.mark.parametrize("kind", ["normal", "repetitive", "bins1000"])
def test_launch_chain_logs_the_oracle_merges(kind):
    """The merge loop runs three launches per merge chained with programmatic dependent launch, and never syncs with
    the host.  It must log exactly the oracle's merges, with and without word de-duplication."""
    from beast_tokenizer_b200 import FIGBPE
    rng = np.random.default_rng(41)
    if kind == "normal":
        bins, vocab = np.clip(rng.normal(128, 28, (12000, 140)).round(), 0, 255).astype(np.int64), 1500
    elif kind == "repetitive":
        base = np.clip(rng.normal(128, 30, (200, 140)).round(), 0, 255).astype(np.int64)
        bins, vocab = base[rng.integers(0, 200, 30000)], 2048            # merges run out before the vocabulary is full
    else:
        bins, vocab = np.clip(rng.normal(500, 120, (5000, 100)).round(), 0, 999).astype(np.int64), 2200
    dev_bins = torch.from_numpy(bins).cuda()
    out = {}
    for dedup in (True, False):
        st = FIGBPE(vocab_size=vocab, show_progress=False, dedup=dedup).fit_from_bins(dev_bins)
        out[dedup] = (st.tokenizer.merges_txt(), st.tokenizer.vocab_json())
    o = OracleBPE.train(bins, vocab)
    for key, val in out.items():
        assert val == (o.merges_txt(), o.vocab_json()), key


@pytest.mark.parametrize("kind", ["normal", "bins1000", "letters"])
def test_hashed_rank_table_gives_the_same_ids(kind, monkeypatch):
    """Vocabularies above 4 096 entries keep their merge ranks in an open-addressing hash of the merges (O(#merges)
    memory) instead of the dense V x V table.  Forced here on ordinary models: ids must equal the dense-table ids and
    the oracle's, in the warp-per-sequence kernel (lane-per-word and cooperative long-word paths) and in the
    one-thread-per-sequence kernel."""
    from beast_tokenizer_b200 import FIGBPE, B200ByteLevelBPE, bpe_model
    rng = np.random.default_rng(51)
    if kind == "normal":
        bins, vocab = np.clip(rng.normal(128, 28, (6000, 140)).round(), 0, 255).astype(np.int64), 1200
    elif kind == "bins1000":
        bins, vocab = np.clip(rng.normal(500, 120, (3000, 100)).round(), 0, 999).astype(np.int64), 1800
    else:
        bins, vocab = rng.choice([97, 97, 97, 98, 99, 32], (2000, 90)) + 7, 400      # long words, runs of one symbol
    dev_bins = torch.from_numpy(bins).cuda()
    st = FIGBPE(vocab_size=vocab, show_progress=False).fit_from_bins(dev_bins)
    o = OracleBPE.train(bins, vocab)
    test = torch.from_numpy(np.concatenate([bins[:300], rng.permuted(bins[:300], axis=1)])).cuda()
    dense = st.tokenizer.encode_bins(test, st.min_token, st.max_token)
    assert st.tokenizer._tables(test.device)["hash_bits"] == 0
    monkeypatch.setattr(bpe_model, "DENSE_RANK_VOCAB", 0)
    hashed_model = B200ByteLevelBPE(st.tokenizer.tokens, st.tokenizer.merges)
    for thread_kernel in ("0", "1"):
        monkeypatch.setenv("BEAST_B200_BPE_THREAD_ENCODE", thread_kernel)
        hashed = hashed_model.encode_bins(test, st.min_token, st.max_token)
        assert hashed_model._tables(test.device)["hash_bits"] > 0
        assert torch.equal(hashed[0], dense[0]) and torch.equal(hashed[1], dense[1])
    fl, of = dense[0].cpu().numpy(), dense[1].cpu().numpy()
    for i in range(0, 600, 13):
        assert fl[of[i]:of[i + 1]].tolist() == o.encode(test[i].cpu().numpy() - o.min_token)
