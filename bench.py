#!/usr/bin/env python
"""bench.py — BEAST tokenizer hot path on B200: trajectories/s, encode + decode.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Workload = BASELINE.json configs[1]: bimanual tokenizer (num_dof=14, num_basis=10, seq_len=50,
vocab 256, grippers [6, 13] zero-order, llm_vocab_size=32000), batch 65 536 per GPU, synthetic
trajectories.  One step = encode (K1) of one batch + reconstruct_traj (K3) of one batch of tokens.

  value   device-resident throughput: inputs already in HBM, C-ABI calls on preallocated buffers,
          timed with CUDA events on the launching stream, max over ranks.
  e2e     the same step through the public Python API from pinned HOST memory: H2D of the
          trajectories, both kernels, D2H of tokens and reconstructed trajectories inside the
          timed region.
  roofline  per-launch CUDA-event duration of the dominant kernel (encode) against the measured
          HBM copy bandwidth in MEASURED_PEAKS.json.
  cpu_baseline  the oracle's literal port of the reference algorithm on the host cores (rank 0, N=1).

`--impl reference` times that CPU port alone (rank 0 only under torchrun).
`--dump-outputs DIR` writes what the last timed step computed to DIR/<name>.npy (rank 0), so that two builds can be
compared output for output: the inputs depend only on the arguments.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BATCH = 65536
T, D, NB, V = 50, 14, 10, 256
GRIP = [6, 13]
LLM_VOCAB = 32000
WORKLOAD = ("bimanual num_dof=14 num_basis=10 seq_len=50 vocab=256 gripper_indices=[6,13] "
            "gripper_zero_order llm_vocab_size=32000, encode+reconstruct_traj batch 65536/GPU")
ENC_BYTES = 4 * T * D + 8 * NB * D + 4 * NB * D       # 4480 B / trajectory (SURVEY.md §8d)
DEC_BYTES = 8 * NB * D + 4 * T * D                    # 3920 B / trajectory
FALLBACK_HBM_GBS = 6650.0


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed regions run."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake", 0x2: "applications_clocks", 0x100: "display_clock"}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            pass

    def run(self):
        while self.ok and not self.stop_flag:
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                mask = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for bit, name in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.005)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": 0}
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


CPU_CHUNK = 8192          # BASELINE.md §5: the reference needs ~300 KB of scratch per trajectory, 8 192 fit comfortably


def make_port():
    """oracle/reference_port_torch.py: the reference's own sequence of torch CPU ops (basis rebuilt
    per call, dense block-diagonal basis, one 120x120 LU per trajectory — mp/uni_bspline.py:539-586);
    pinned to the live reference's golden vectors (coefficients within 1e-6 normwise, tokens equal up to
    the listed edge flips: tests/test_oracle_golden.py)."""
    from oracle.reference_port_torch import ReferencePort
    return ReferencePort(num_dof=D, num_basis=NB, seq_len=T, vocab_size=V, degree_p=4, gripper_zero_order=True,
                         gripper_indices=GRIP, llm_vocab_size=LLM_VOCAB)


def port_step(port, x):
    tokens, _ = port.encode(x)
    return port.reconstruct_traj(tokens)


def cpu_threads():
    import torch
    return int(torch.get_num_threads())


def use_all_host_threads():
    """torchrun exports OMP_NUM_THREADS=1 to every rank; the CPU arms must use the box's cores.  Call before the
    first `import torch` of the process when possible (the env var is read at import), and set the count anyway."""
    for k in ("OMP_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ.pop(k, None)
    import torch
    n = os.cpu_count() or 1
    if torch.get_num_threads() != n:
        torch.set_num_threads(n)
    os.environ.setdefault("RAYON_NUM_THREADS", str(n))
    os.environ.setdefault("TOKENIZERS_PARALLELISM", "true")
    return n


def cpu_baseline(budget_s=12.0):
    """Bounded sample of the same workload on the host cores (rank 0, N=1)."""
    use_all_host_threads()
    from beast_tokenizer_b200.synth import synth
    port = make_port()
    x = synth(CPU_CHUNK, T, D, seed=2)
    port_step(port, x[:256])                     # warm-up
    n, t0 = 0, time.perf_counter()
    while True:
        port_step(port, x)
        n += CPU_CHUNK
        el = time.perf_counter() - t0
        if el >= budget_s:
            break
    return {"value": n / el, "unit": "trajectories/s", "cores": cpu_threads(), "kind": "port",
            "sample": f"{n} trajectories in chunks of {CPU_CHUNK} (torch-CPU port of the reference's op sequence, "
                      f"encode + reconstruct_traj), {el:.1f} s; host has {os.cpu_count()} logical cores"}


def run_reference(args, rank):
    """--impl reference: the reference's CPU algorithm (torch-CPU port) on this box's host cores."""
    if rank != 0:
        return
    use_all_host_threads()
    from beast_tokenizer_b200.synth import synth
    port = make_port()
    x = synth(CPU_CHUNK, T, D, seed=2)
    for _ in range(max(1, min(args.warmup, 2))):
        port_step(port, x[:512])
    t0 = time.perf_counter()
    for _ in range(args.steps):
        port_step(port, x)
    el = time.perf_counter() - t0
    n = args.steps * CPU_CHUNK
    val = n / el
    line = {
        "impl": "reference", "metric": "trajectories/sec encode+decode", "value": val, "unit": "trajectories/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * el / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "sample_per_step": CPU_CHUNK},
        "cpu_baseline": {"value": val, "unit": "trajectories/s", "cores": cpu_threads(), "kind": "port",
                         "sample": f"{CPU_CHUNK} trajectories per step x {args.steps} steps (bounded sample of the "
                                   f"65536-trajectory batch), torch-CPU port of the reference's op sequence; host has "
                                   f"{os.cpu_count()} logical cores"},
        "e2e": {"value": val, "unit": "trajectories/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    try:                                                   # BPE-train merges/s of the reference trainer, bounded sample
        import numpy as np
        import torch
        n = 16384
        tokens, _ = port.encode(synth(n, T, D, seed=1000)[:n])
        bins = (tokens - (LLM_VOCAB - V)).numpy()
        cpu = hf_train_cpu(bins, BPE_VOCAB)
        line["bpe_train"] = {"metric": "BPE-train merges/sec", "value": cpu["merges"] / cpu["seconds"], "unit": "merges/s",
                             "engine": cpu["engine"], "merges": cpu["merges"], "seconds": cpu["seconds"],
                             "sample": f"{n} sequences x 140 bins (bounded sample; the trainer is ~linear in the corpus)"}
    except Exception as exc:                               # pragma: no cover
        line["bpe_train"] = {"unavailable": str(exc)}
    print(json.dumps(line), flush=True)


BPE_VOCAB = 2048
BPE_BATCHES, BPE_BATCH = 50_000, 32          # BASELINE configs[3]: 50k batches x 32 = 1.6 M sequences
BPE_CHUNKS = 200                             # corpus generated as 200 chunks of 250 batches, dealt round-robin to ranks
BPE_CPU_SAMPLE = 65_536


def hf_train_cpu(bins_np, vocab):
    """The reference's trainer: HF tokenizers' BpeTrainer behind FIGBPE._fit_from_strings
    (beast/beast_bpe_trainer.py:61-98) on the host cores; the C oracle if the wheel is absent."""
    mn, mx = int(bins_np.min()), int(bins_np.max())
    try:
        from tokenizers import ByteLevelBPETokenizer
        from tokenizers.trainers import BpeTrainer
    except ImportError:
        from oracle.bpe_oracle import OracleBPE
        t0 = time.perf_counter()
        o = OracleBPE.train(bins_np, vocab)
        return {"engine": "oracle/bpe_oracle.c (1 thread)", "seconds": time.perf_counter() - t0, "merges": len(o.merges),
                "merges_txt": o.merges_txt()}
    t0 = time.perf_counter()
    # chr(bin - min) per symbol (beast/beast_bpe_trainer.py:86-92), built with one UTF-32 decode
    flat = (bins_np - mn).astype("<u4")
    text = flat.tobytes().decode("utf-32-le")
    L = bins_np.shape[1]
    strings = [text[i * L:(i + 1) * L] for i in range(bins_np.shape[0])]
    t1 = time.perf_counter()
    hf = ByteLevelBPETokenizer()
    trainer = BpeTrainer(vocab_size=vocab, min_frequency=2, show_progress=False, special_tokens=[],
                         initial_alphabet=[chr(i) for i in range(mx - mn + 1)], max_token_length=10000)
    hf._tokenizer.train_from_iterator(strings, trainer=trainer)
    t2 = time.perf_counter()
    model = json.loads(hf._tokenizer.to_str())["model"]
    merges = [m if isinstance(m, str) else " ".join(m) for m in model["merges"]]
    import tokenizers
    return {"engine": f"tokenizers {tokenizers.__version__} BpeTrainer (rayon, {os.cpu_count()} logical cores)",
            "seconds": t2 - t1, "string_build_seconds": t1 - t0, "merges": len(merges),
            "merges_txt": "#version: 0.2\n" + "".join(m + "\n" for m in merges)}


def bpe_legs(tok, dev, rank, world, dist, with_cpu, cpu_full=False):
    """BPE-train merges/s on the 1.6 M-sequence corpus sharded over the ranks (strong scaling), and
    BPE encode / decode sequences/s on 1 M trajectories (rank 0's GPU)."""
    import torch
    from beast_tokenizer_b200 import BEASTBsplineBPETokenizer, FIGBPE
    from beast_tokenizer_b200.synth import synth_device
    per_chunk = BPE_BATCHES * BPE_BATCH // BPE_CHUNKS
    mine = [c for c in range(BPE_CHUNKS) if c % world == rank]
    bins = torch.cat([tok.encode(synth_device(per_chunk, T, D, 1000 + c, dev), respect_llm_vocab_size=False)[0]
                      for c in mine])
    torch.cuda.synchronize()
    fig = FIGBPE(vocab_size=BPE_VOCAB, show_progress=False, device=str(dev))
    fig.fit_from_bins(bins[:4096])                    # warm-up: kernels loaded, NCCL channels up
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    runs = []
    for _ in range(2):                                # the first full-size fit also pays the allocator's cudaMallocs (~1 GB of buffers)
        t0 = time.perf_counter()
        state = fig.fit_from_bins(bins)
        torch.cuda.synchronize()
        dt = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
            dist.barrier()
        runs.append(float(dt.item()))
    secs = min(runs)
    n_merges = len(state.tokenizer.merges)
    import hashlib
    table = state.tokenizer.merges_txt() + state.tokenizer.vocab_json()
    sha = hashlib.sha256(table.encode("utf-8")).hexdigest()
    out = {"metric": "BPE-train merges/sec", "value": n_merges / secs, "unit": "merges/s", "seconds": secs,
           "us_per_merge": 1e6 * secs / max(n_merges, 1),
           "runs_seconds": runs, "merges": n_merges, "vocab": BPE_VOCAB, "sequences": BPE_BATCHES * BPE_BATCH, "n_gpus": world,
           "scaling": "strong", "merge_table_sha256": sha,
           "delta_reduction": getattr(state.tokenizer, "trainer_mode", "single GPU"),
           "sharding": f"{BPE_CHUNKS} chunks of {per_chunk} sequences round-robin over ranks; min/max, seen bytes and the "
           "initial histogram all-reduced once (NCCL); per-merge 4xV deltas summed inside bpe_iterate_kernel over peer memory"}
    if world > 1:
        # every rank must hold the same table, and it must be the table of the unsharded corpus
        shas = [None] * world
        dist.all_gather_object(shas, sha)
        out["ranks_agree"] = all(h == sha for h in shas)
        if rank == 0:
            full = torch.cat([tok.encode(synth_device(per_chunk, T, D, 1000 + c, dev), respect_llm_vocab_size=False)[0]
                              for c in range(BPE_CHUNKS)])
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ref = FIGBPE(vocab_size=BPE_VOCAB, show_progress=False, device=str(dev), process_group=False).fit_from_bins(full)
            torch.cuda.synchronize()
            ref_secs = time.perf_counter() - t0
            ref_table = ref.tokenizer.merges_txt() + ref.tokenizer.vocab_json()
            out["identical_to_unsharded"] = ref_table == table
            out["unsharded_same_gpu"] = {"seconds": ref_secs, "merge_table_sha256": hashlib.sha256(ref_table.encode("utf-8")).hexdigest()}
            del full
        dist.barrier()
    if rank != 0:
        return out, None
    out["dedup"] = getattr(state.tokenizer, "dedup_stats", None)
    if world == 1:
        out["repetitive_corpus"] = bpe_repetitive_leg(tok, dev, bins, with_cpu)
        out["e2e_fit_from_trajectories"] = bpe_e2e_leg(tok, dev, with_cpu)
    if with_cpu:
        # the reference trainer on the same bins, bounded sample; the GPU trainer on that sample must agree
        sample = synth_bins_sample(tok, dev)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        st_s = FIGBPE(vocab_size=BPE_VOCAB, show_progress=False, device=str(dev), process_group=False).fit_from_bins(sample)
        torch.cuda.synchronize()
        g_secs = time.perf_counter() - t0
        cpu = hf_train_cpu(sample.cpu().numpy(), BPE_VOCAB)
        out["cpu_baseline"] = {"value": cpu["merges"] / cpu["seconds"], "unit": "merges/s", "kind": "reference",
                               "engine": cpu["engine"], "seconds": cpu["seconds"],
                               "sample": f"{BPE_CPU_SAMPLE} of the 1.6 M sequences (trainer cost is ~linear in the corpus)",
                               "gpu_same_sample": {"seconds": g_secs, "merges_per_s": len(st_s.tokenizer.merges) / g_secs},
                               "merge_table_identical": cpu["merges_txt"] == st_s.tokenizer.merges_txt()}
        if cpu_full and world == 1:
            # the reference trainer on the WHOLE 1.6 M-sequence corpus (about a minute of host time; --no-bpe-cpu-full skips it)
            full = hf_train_cpu(bins.cpu().numpy(), BPE_VOCAB)
            out["cpu_baseline"]["full_corpus"] = {
                "sequences": int(bins.shape[0]), "seconds": full["seconds"],
                "string_build_seconds": full.get("string_build_seconds"),
                "merges_per_s": full["merges"] / full["seconds"], "gpu_seconds": secs,
                "speedup_1gpu": full["seconds"] / secs,
                "merge_table_identical": full["merges_txt"] == state.tokenizer.merges_txt()}
    # BPE encode + reconstruct (configs[4]) on device-resident CSR
    btok = BEASTBsplineBPETokenizer.from_beast(tok, bpe_vocab_size=BPE_VOCAB, device=str(dev))
    btok.set_llm_vocab_size(None)
    btok.set_bpe_tokenizer(state.tokenizer, min_token=state.min_token, max_token=state.max_token)
    nb = 1 << 20
    x = synth_device(nb, T, D, 5, dev)
    mp, _ = btok.encode_to_mp_tokens(x)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    flat, offsets = btok._discrete_to_bpe_csr(mp)    # warm-up
    torch.cuda.synchronize()
    ev[0].record()
    flat, offsets = btok._discrete_to_bpe_csr(mp)
    ev[1].record()
    back = btok._bpe_csr_to_discrete(flat, offsets)
    ev[2].record()
    torch.cuda.synchronize()
    xs_api = x[:65536]
    btok.encode(xs_api[:1024])
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ids_list, _ = btok.encode(xs_api)                 # API-faithful: ragged List[List[int]] on the host
    t1 = time.perf_counter()
    rec_api = btok.reconstruct_traj(ids_list)
    torch.cuda.synchronize()
    t2 = time.perf_counter()
    apply = {"workload": "BPE encode / decode of 1 048 576 sequences x 140 bins, 2048-entry table, device CSR",
             "api_list_path": {"batch": 65536, "encode_traj_per_s": 65536 / (t1 - t0),
                               "reconstruct_traj_per_s": 65536 / (t2 - t1),
                               "note": "BEASTBsplineBPETokenizer.encode -> List[List[int]] -> reconstruct_traj; the lists are built / "
                                       "flattened by the CPython helper csrc/pylists.c (round 2 before it: 0.30 M / 0.22 M traj/s in Python)"},
             "encode_seq_per_s": nb / (ev[0].elapsed_time(ev[1]) * 1e-3),
             "decode_seq_per_s": nb / (ev[1].elapsed_time(ev[2]) * 1e-3),
             "ids_per_sequence": float(flat.numel()) / nb, "round_trip_exact": bool(torch.equal(back, mp))}
    # roofline of the two apply paths: 8 B x 140 bins + 4 B x ids per sequence (SURVEY.md §8d), against the measured HBM peak
    peak, _ = measured_peak()
    seq_bytes = 8 * mp.shape[1] + 4 * float(flat.numel()) / nb
    for name, secs in (("encode", ev[0].elapsed_time(ev[1]) * 1e-3), ("decode", ev[1].elapsed_time(ev[2]) * 1e-3)):
        gbs = seq_bytes * nb / secs / 1e9
        apply[f"roofline_bpe_{name}"] = {"bound": "hbm" if name == "decode" else "issue (ncu: 4 300 warp instructions per sequence)",
                                        "achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak,
                                        "bytes_per_sequence": seq_bytes, "ms": secs * 1e3,
                                        "path": "_discrete_to_bpe_csr (bpe_encode + cumsum + bpe_compact)" if name == "encode"
                                        else "_bpe_csr_to_discrete (bpe_decode: per-token table kernel + flagged fallback)"}
    if with_cpu:
        ref = bpe_apply_cpu_reference(btok, mp[:4096].cpu())
        if ref is not None:
            ids_gpu = btok._discrete_to_bpe(mp[:64])
            hf = btok.bpe_tokenizer.to_hf()
            ref["ids_identical_to_gpu"] = ids_gpu == [hf.encode("".join(map(chr, r))).ids
                                                      for r in (mp[:64].cpu() - btok.bpe_min_token).tolist()]
            apply["cpu_reference"] = ref
    return out, apply


def bpe_repetitive_leg(tok, dev, bins, with_cpu):
    """SURVEY.md §8(f)4: the trainer on a REPETITIVE corpus — 1.6 M sequences drawn from 20 000 distinct ones, the
    regime of real robot data — with and without word de-duplication (distinct pre-tokens with counts, as HF's
    BpeTrainer does); both must give the same table."""
    import hashlib
    import torch
    from beast_tokenizer_b200 import FIGBPE
    g = torch.Generator(device=dev).manual_seed(4)
    pick = torch.randint(0, 20_000, (bins.shape[0],), generator=g, device=dev)
    rep = bins[:20_000][pick].contiguous()
    out = {"workload": f"{rep.shape[0]} sequences drawn from 20 000 distinct ones, vocab {BPE_VOCAB}"}
    tables = {}
    for mode in ("auto", False):
        fig = FIGBPE(vocab_size=BPE_VOCAB, show_progress=False, device=str(dev), process_group=False, dedup=mode)
        runs = []
        for _ in range(2):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            st = fig.fit_from_bins(rep)
            torch.cuda.synchronize()
            runs.append(time.perf_counter() - t0)
        tables[mode] = st.tokenizer.merges_txt() + st.tokenizer.vocab_json()
        key = "dedup_auto" if mode == "auto" else "dedup_off"
        out[key] = {"seconds": min(runs), "runs_seconds": runs, "merges": len(st.tokenizer.merges),
                    "merges_per_s": len(st.tokenizer.merges) / min(runs), "stats": getattr(st.tokenizer, "dedup_stats", None)}
    out["same_table"] = tables["auto"] == tables[False]
    out["merge_table_sha256"] = hashlib.sha256(tables["auto"].encode("utf-8")).hexdigest()
    out["speedup_from_dedup"] = out["dedup_off"]["seconds"] / out["dedup_auto"]["seconds"]
    if with_cpu:
        cpu = hf_train_cpu(rep.cpu().numpy(), BPE_VOCAB)
        out["cpu_reference"] = {"engine": cpu["engine"], "seconds": cpu["seconds"], "string_build_seconds": cpu.get("string_build_seconds"),
                                "merges_per_s": cpu["merges"] / cpu["seconds"],
                                "merge_table_identical": cpu["merges_txt"] == st.tokenizer.merges_txt(),
                                "speedup_1gpu": cpu["seconds"] / out["dedup_auto"]["seconds"]}
    return out


def bpe_e2e_leg(tok, dev, with_cpu):
    """BASELINE configs[3] end to end through the public API: BEASTBsplineBPETokenizer.fit_from_trajectories over a
    loader of 50 000 HOST batches x 32 trajectories (wall clock: H2D of every batch, K1, symbolise, count, merge loop,
    vocabulary).  Beside it the reference flow (beast/beast_bpe_trainer.py:100-151: per-batch encode, D2H, chr strings,
    HF BpeTrainer) timed on a stated subset of the same loader."""
    import torch
    from beast_tokenizer_b200 import BEASTBsplineBPETokenizer
    from beast_tokenizer_b200.synth import synth_device
    n_batches, bs = BPE_BATCHES, BPE_BATCH
    # the loader's batches as views of host blocks (generated on the GPU, copied out once: 4.5 GB of host memory)
    blocks = []
    per = BPE_BATCHES * BPE_BATCH // BPE_CHUNKS
    for c in range(BPE_CHUNKS):
        blocks.append(synth_device(per, T, D, 1000 + c, dev).cpu())
    loader = [{"actions": blk[i:i + bs]} for blk in blocks for i in range(0, per, bs)]
    assert len(loader) == n_batches
    btok = BEASTBsplineBPETokenizer.from_beast(tok, bpe_vocab_size=BPE_VOCAB, device=str(dev))
    btok.set_llm_vocab_size(None)
    btok.fit_from_trajectories(loader[:64], show_progress=False)            # warm-up
    torch.cuda.synchronize()
    runs = []
    for _ in range(2):
        t0 = time.perf_counter()
        state = btok.fit_from_trajectories(loader, show_progress=False)
        torch.cuda.synchronize()
        runs.append(time.perf_counter() - t0)
    secs = min(runs)
    import hashlib
    out = {"workload": f"{n_batches} host batches x {bs} trajectories [32, 50, 14] fp32 (pageable host memory), "
                       f"bpe_vocab_size {BPE_VOCAB}", "seconds": secs, "runs_seconds": runs,
           "merges": len(state.tokenizer.merges), "sequences_per_s": n_batches * bs / secs,
           "merge_table_sha256": hashlib.sha256((state.tokenizer.merges_txt() + state.tokenizer.vocab_json()).encode("utf-8")).hexdigest(),
           "h2d_bytes": 4 * T * D * n_batches * bs, "timer": "host clock, device synchronised"}
    if with_cpu:
        # the reference's flow on the first `nb_cpu` batches: torch-CPU port encode per batch + HF trainer
        nb_cpu = 128
        port = make_port()
        port.offset = 0                                            # BPE works on MP tokens (encode_to_mp_tokens)
        lo, hi = tok._bounds(dev)
        port.w_min, port.w_max = lo.cpu(), hi.cpu()
        t0 = time.perf_counter()
        rows = []
        for b in loader[:nb_cpu]:
            tokens, _ = port.encode(b["actions"])
            rows.append(tokens.numpy())
        import numpy as np
        bins_cpu = np.concatenate(rows)
        t1 = time.perf_counter()
        cpu = hf_train_cpu(bins_cpu, BPE_VOCAB)
        t2 = time.perf_counter()
        enc_s = t1 - t0
        out["cpu_reference"] = {
            "kind": "port + tokenizers", "batches": nb_cpu, "encode_seconds": enc_s, "train_seconds": t2 - t1,
            "encode_seconds_extrapolated_full": enc_s * n_batches / nb_cpu,
            "note": f"reference flow on the first {nb_cpu} of {n_batches} batches: per-batch encode on the host ({cpu_threads()} "
                    "threads) scales linearly with the batch count; the trainer time on the full corpus is bpe_train.cpu_baseline.full_corpus"}
    return out


def bounds_cpu_reference(n=4096):
    """fit_parameters as the reference runs it (beast_bspline_tokenizer.py:181-220): per batch of 32 the fit on the
    host, weights concatenated, np.quantile(1 %, 99 %) — bounded sample, linear in the trajectory count."""
    import numpy as np
    import torch
    from beast_tokenizer_b200.synth import synth
    port = make_port()
    x = synth(n, T, D, seed=7)
    port.compute_weights(x[:32])
    t0 = time.perf_counter()
    w = torch.cat([port.compute_weights(x[i:i + 32]) for i in range(0, n, 32)]).numpy()
    np.quantile(w, 0.01, axis=0), np.quantile(w, 0.99, axis=0)
    dt = time.perf_counter() - t0
    return {"traj_per_s": n / dt, "seconds": dt, "sample": f"{n} trajectories in batches of 32, torch-CPU port + np.quantile, "
            f"{cpu_threads()} threads"}


def bpe_apply_cpu_reference(btok, mp_tokens_cpu, n=4096):
    """_discrete_to_bpe / _bpe_to_discrete as the reference runs them (beast_bspline_bpe_tokenizer.py:175-247): a Python
    loop over rows around HF tokenizer.encode / decode."""
    try:
        hf = btok.bpe_tokenizer.to_hf()
    except ImportError:
        return None
    rows = (mp_tokens_cpu[:n] - btok.bpe_min_token).tolist()
    t0 = time.perf_counter()
    ids = [hf.encode("".join(map(chr, r))).ids for r in rows]
    t1 = time.perf_counter()
    back = [[ord(ch) + btok.bpe_min_token for ch in hf.decode(i)] for i in ids]
    t2 = time.perf_counter()
    return {"batch": n, "encode_seq_per_s": n / (t1 - t0), "decode_seq_per_s": n / (t2 - t1),
            "round_trip_exact": back == mp_tokens_cpu[:n].tolist(), "engine": "tokenizers (per-row Python loop, as the reference)"}


def bounds_leg(tok, dev, with_cpu=False):
    """BASELINE configs[2]: weight bounds over 100 000 trajectories — the fused min/max reduction
    (update_weights_bounds) and the reference-faithful quantile fit (fit_parameters)."""
    import torch
    from beast_tokenizer_b200.synth import synth_device
    n = 100_000
    x = synth_device(n, T, D, 7, dev)
    saved = (tok.w_min.clone(), tok.w_max.clone())
    tok.update_weights_bounds(x)                      # warm-up
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 20
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        tok.update_weights_bounds(x)
    e1.record()
    torch.cuda.synchronize()
    mm_ms = e0.elapsed_time(e1) / reps
    out = {"workload": "100 000 trajectories [100000, 50, 14] resident in HBM",
           "update_weights_bounds": {"ms": mm_ms, "traj_per_s": n / (mm_ms * 1e-3),
                                     "GBps_read": 4 * T * D * n / (mm_ms * 1e-3) / 1e9}}
    for label, bs in (("3125 batches x 32 (the reference's loader shape)", 32), ("25 batches x 4000", 4000)):
        batches = [{"actions": x[i:i + bs]} for i in range(0, n, bs)]
        tok.fit_parameters(batches[:4], verbose=False)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        tok.fit_parameters(batches, verbose=False)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        out.setdefault("fit_parameters", {})[label] = {"seconds": dt, "traj_per_s": n / dt}
    tok.w_min.copy_(saved[0])
    tok.w_max.copy_(saved[1])
    if with_cpu:
        out["cpu_reference"] = bounds_cpu_reference()
    return out


def shipped_shape_leg(dev, with_cpu):
    """The reference's own shipped configuration (train.sh / train/train_beast.py:34-36): 50 basis functions, degree 0,
    1000 bins, actions [10, 32] — 1600 tokens per trajectory; write-bound: 1 280 B read, 12 800 B of int64 tokens +
    6 400 B of coefficients written per trajectory on encode, the reverse on decode."""
    import torch
    from beast_tokenizer_b200 import BEASTBsplineTokenizer
    from beast_tokenizer_b200.synth import synth, synth_device
    Ts, Ds, NBs, Vs = 10, 32, 50, 1000
    tok = BEASTBsplineTokenizer(num_dof=Ds, num_basis=NBs, seq_len=Ts, vocab_size=Vs, degree_p=0, device=str(dev))
    n = 32768
    x = synth_device(n, Ts, Ds, 11, dev)
    tok.update_weights_bounds(x)
    tokens, _ = tok.encode(x)
    rec = tok.reconstruct_traj(tokens)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
    reps = 10
    torch.cuda.synchronize()
    ev[0].record()
    for _ in range(reps):
        tokens, _ = tok.encode(x)
    ev[1].record()
    for _ in range(reps):
        rec = tok.reconstruct_traj(tokens)
    ev[2].record()
    torch.cuda.synchronize()
    api_enc_ms, api_dec_ms = ev[0].elapsed_time(ev[1]) / reps, ev[1].elapsed_time(ev[2]) / reps
    # the same kernels through the C ABI on preallocated buffers (what the roofline fraction is computed from; the API
    # path above also pays torch's allocation of 630 MB of outputs per call)
    from beast_tokenizer_b200 import _lib
    plan = tok._plan()
    lo, hi = tok._bounds(dev)
    toks_b = torch.empty((n, NBs * Ds), device=dev, dtype=torch.int64)
    pars_b = torch.empty((n, NBs * Ds), device=dev, dtype=torch.float32)
    out_b = torch.empty((n, Ts, Ds), device=dev, dtype=torch.float32)
    def enc_raw():
        _lib.check(plan._lib.beast_encode_f32(plan.handle, _lib.ptr(x), n, _lib.ptr(lo), _lib.ptr(hi), 0, _lib.ptr(pars_b),
                                              _lib.ptr(toks_b), _lib.stream_ptr(dev)), "encode")
    def dec_raw():
        _lib.check(plan._lib.beast_decode_f32(plan.handle, _lib.ptr(toks_b), n, _lib.ptr(lo), _lib.ptr(hi), 0, None,
                                              _lib.ptr(out_b), _lib.stream_ptr(dev)), "decode")
    enc_raw(); dec_raw()
    torch.cuda.synchronize()
    ev[2].record()
    for _ in range(reps):
        enc_raw()
    ev[3].record()
    for _ in range(reps):
        dec_raw()
    ev[4].record()
    torch.cuda.synchronize()
    enc_ms, dec_ms = ev[2].elapsed_time(ev[3]) / reps, ev[3].elapsed_time(ev[4]) / reps
    assert torch.equal(toks_b, tokens) and torch.equal(out_b, rec)
    enc_bytes = 4 * Ts * Ds + 8 * NBs * Ds + 4 * NBs * Ds
    dec_bytes = 8 * NBs * Ds + 4 * Ts * Ds
    peak, _ = measured_peak()
    used_rows = int((tok._plan().consts.phi_joint != 0).any(0).sum())
    dec_touched = 8 * used_rows * Ds + 4 * Ts * Ds
    out = {"workload": f"num_dof=32 num_basis=50 seq_len=10 vocab=1000 degree_p=0 (reference train.sh), batch {n}, device-resident; "
                       "C-ABI calls on preallocated buffers, CUDA events around 10 back-to-back launches",
           "api_path_ms": {"encode": api_enc_ms, "reconstruct_traj": api_dec_ms,
                           "note": "BEASTBsplineTokenizer.encode / reconstruct_traj incl. torch's allocation of the outputs (630 MB per encode); depends on "
                                   "the caching allocator's state inside this long process — 0.21 ms per encode in a fresh one (scripts/api_alloc_probe.py)"},
           "encode": {"ms": enc_ms, "traj_per_s": n / (enc_ms * 1e-3), "bytes_per_traj": enc_bytes,
                      "GBps": enc_bytes * n / (enc_ms * 1e-3) / 1e9, "frac_of_measured_hbm": enc_bytes * n / (enc_ms * 1e-3) / 1e9 / peak},
           "reconstruct_traj": {"ms": dec_ms, "traj_per_s": n / (dec_ms * 1e-3), "bytes_per_traj": dec_bytes,
                                "GBps": dec_bytes * n / (dec_ms * 1e-3) / 1e9,
                                "frac_of_measured_hbm": dec_bytes * n / (dec_ms * 1e-3) / 1e9 / peak,
                                "bytes_touched_per_traj": dec_touched,
                                "GBps_touched": dec_touched * n / (dec_ms * 1e-3) / 1e9,
                                "frac_of_measured_hbm_touched": dec_touched * n / (dec_ms * 1e-3) / 1e9 / peak,
                                "note": f"{used_rows} of {NBs} coefficient rows reach a trajectory sample (degree-0 basis functions over "
                                        f"{Ts} samples): the kernel loads only their tokens; bytes_per_traj counts every token as SURVEY 8(d) does"},
           "max_abs_reconstruction_error": float((rec - x).abs().max().item())}
    # the BPE stage of the same configuration (train.sh: --bpe-vocab-size 2048): 1 600-bin sequences, 2-byte UTF-8 symbols
    from beast_tokenizer_b200 import FIGBPE
    n_bpe = 16384
    bins = tokens[:n_bpe]
    fig = FIGBPE(vocab_size=2048, show_progress=False, device=str(dev), process_group=False)
    fig.fit_from_bins(bins[:1024])
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    st = fig.fit_from_bins(bins)
    torch.cuda.synchronize()
    bpe_s = time.perf_counter() - t0
    flat, offs, status = st.tokenizer.encode_bins(bins, st.min_token, st.max_token)
    back, st2, _ = st.tokenizer.decode_ids(flat, offs, bins.shape[1], st.min_token)
    torch.cuda.synchronize()
    enc_s = dec_s = float("inf")
    for _ in range(3):            # best of three calls: each allocates its outputs (210 MB of bins), and one call in a
        back = None               # long process can land on a cudaMalloc / cache flush of torch's allocator (~90 ms)
        t0 = time.perf_counter()
        flat, offs, status = st.tokenizer.encode_bins(bins, st.min_token, st.max_token)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        back, st2, _ = st.tokenizer.decode_ids(flat, offs, bins.shape[1], st.min_token)
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        enc_s, dec_s = min(enc_s, t1 - t0), min(dec_s, t2 - t1)
    out["bpe"] = {"sequences": n_bpe, "bins_per_sequence": int(bins.shape[1]), "vocab": 2048, "merges": len(st.tokenizer.merges),
                  "train_seconds": bpe_s, "merges_per_s": len(st.tokenizer.merges) / bpe_s,
                  "encode_seq_per_s": n_bpe / enc_s, "decode_seq_per_s": n_bpe / dec_s, "apply_timing": "host clock, best of 3 calls",
                  "ids_per_sequence": float(flat.numel()) / n_bpe, "round_trip_exact": bool(torch.equal(back, bins)),
                  "dedup": getattr(st.tokenizer, "dedup_stats", None)}
    if with_cpu:
        cpu = hf_train_cpu(bins.cpu().numpy(), 2048)
        out["bpe"]["cpu_reference"] = {"engine": cpu["engine"], "seconds": cpu["seconds"], "merges_per_s": cpu["merges"] / cpu["seconds"],
                                       "merge_table_identical": cpu["merges_txt"] == st.tokenizer.merges_txt(),
                                       "speedup_1gpu": cpu["seconds"] / bpe_s}
    if with_cpu:
        from oracle.reference_port_torch import ReferencePort
        use_all_host_threads()
        port = ReferencePort(num_dof=Ds, num_basis=NBs, seq_len=Ts, vocab_size=Vs, degree_p=0)
        port.w_min, port.w_max = tok.w_min.cpu(), tok.w_max.cpu()
        xs = synth(32, Ts, Ds, seed=12)
        t0 = time.perf_counter()
        tk, _ = port.encode(xs)
        t1 = time.perf_counter()
        port.reconstruct_traj(tk)
        t2 = time.perf_counter()
        mine, _ = tok.encode(xs)
        out["cpu_reference"] = {"kind": "port", "batch": 32, "encode_traj_per_s": 32 / (t1 - t0), "reconstruct_traj_per_s": 32 / (t2 - t1),
                                "cores": cpu_threads(), "tokens_equal_fraction": float((mine.cpu() == tk).float().mean().item()),
                                "note": "one loader batch of 32: the reference solves one 1600 x 1600 system per trajectory"}
    return out


def cfg1_latency_leg(dev, with_cpu):
    """BASELINE configs[0]: num_dof=7, 32 trajectories — per-call latency of encode + reconstruct_traj through the
    public API (host tensor in, host tensor out, synchronised), next to the reference's CPU path."""
    import torch
    from beast_tokenizer_b200 import BEASTBsplineTokenizer
    from beast_tokenizer_b200.synth import synth
    tok = BEASTBsplineTokenizer(num_dof=7, num_basis=10, seq_len=50, vocab_size=256, gripper_indices=[6], device=str(dev))
    x = synth(32, 50, 7, seed=0)

    def call():
        tokens, _ = tok.encode(x)
        return tok.reconstruct_traj(tokens).cpu()

    for _ in range(5):
        call()
    torch.cuda.synchronize()
    reps = 200
    t0 = time.perf_counter()
    for _ in range(reps):
        call()
    us = 1e6 * (time.perf_counter() - t0) / reps
    xd = x.to(dev)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    ev0.record()
    for _ in range(reps):
        tokens, _ = tok.encode(xd)
        tok.reconstruct_traj(tokens)
    ev1.record()
    torch.cuda.synchronize()
    out = {"workload": "num_dof=7 num_basis=10 seq_len=50 vocab=256 gripper_indices=[6], batch 32, encode + reconstruct_traj",
           "api_host_to_host_us_per_call": us, "traj_per_s": 32 / (us * 1e-6),
           "device_resident_us_per_call": 1e3 * ev0.elapsed_time(ev1) / reps}
    if with_cpu:
        from oracle.reference_port_torch import ReferencePort
        use_all_host_threads()
        port = ReferencePort(num_dof=7, num_basis=10, seq_len=50, vocab_size=256, degree_p=4, gripper_indices=[6])
        port_step(port, x)
        t0 = time.perf_counter()
        for _ in range(20):
            port_step(port, x)
        cpu_us = 1e6 * (time.perf_counter() - t0) / 20
        out["cpu_reference"] = {"kind": "port", "us_per_call": cpu_us, "traj_per_s": 32 / (cpu_us * 1e-6), "cores": cpu_threads()}
        out["speedup_per_call"] = cpu_us / us
    return out


def synth_bins_sample(tok, dev):
    from beast_tokenizer_b200.synth import synth_device
    return tok.encode(synth_device(BPE_CPU_SAMPLE, T, D, 1000, dev), respect_llm_vocab_size=False)[0]


DUMP_ROWS = 8192          # 8 192 x 4 480 B = 37 MB of .npy files whatever the batch


def dump_outputs(out_dir, tokens, params, trajectories):
    """What one timed step hands back — encode's tokens and coefficients, decode's trajectories — as
    out_dir/<name>.npy: the same seeded sample of rows (all rows of a batch up to DUMP_ROWS), tokens as
    float64 (exact), the rest float32."""
    import numpy as np
    import torch
    n = tokens.shape[0]
    rows = np.sort(np.random.default_rng(0).choice(n, size=min(n, DUMP_ROWS), replace=False))
    idx = torch.from_numpy(rows).to(tokens.device)
    os.makedirs(out_dir, exist_ok=True)
    for name, t, dtype in (("encode_tokens", tokens, np.float64), ("encode_params", params, np.float32),
                           ("decode_trajectories", trajectories, np.float32)):
        np.save(os.path.join(out_dir, f"{name}.npy"), t.index_select(0, idx).cpu().numpy().astype(dtype))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-bpe", action="store_true", help="skip the BPE-train / BPE-apply legs")
    ap.add_argument("--no-bpe-cpu-full", action="store_true",
                    help="skip the reference BPE trainer on the full 1.6 M-sequence corpus (about a minute of host time)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the tokens, coefficients and trajectories of the last one to "
                         f"DIR/<name>.npy (a fixed sample of {DUMP_ROWS} rows of the batch)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the B200 path; it does not apply to --impl reference")
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank)
        return

    import ctypes as C
    import numpy as np
    import torch
    import torch.distributed as dist
    from beast_tokenizer_b200 import BEASTBsplineTokenizer, _lib
    from beast_tokenizer_b200.synth import SyntheticLoader, synth

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    B = args.batch
    tok = BEASTBsplineTokenizer(num_dof=D, num_basis=NB, seq_len=T, vocab_size=V, gripper_zero_order=True,
                                gripper_indices=GRIP, device=f"cuda:{local_rank}", llm_vocab_size=LLM_VOCAB)
    tok.fit_parameters(SyntheticLoader(100, 32, T, D, seed0=1), verbose=False)
    plan = tok._plan()
    lib = plan._lib
    lo, hi = tok._bounds(dev)
    offset = LLM_VOCAB - V

    # ---- device-resident leg: R rotating buffer sets, each larger than L2 in aggregate; the decode of a
    # step reads tokens written two steps earlier, so no step input is L2-resident when it is read.
    R = 4
    xs = [synth(B, T, D, seed=2 + 1000 * rank + i, device=dev) for i in range(R)]
    toks = [torch.empty((B, NB * D), device=dev, dtype=torch.int64) for _ in range(R)]
    pars = [torch.empty((B, NB * D), device=dev, dtype=torch.float32) for _ in range(R)]
    outs = [torch.empty((B, T, D), device=dev, dtype=torch.float32) for _ in range(R)]
    def enc(i):
        _lib.check(lib.beast_encode_f32(plan.handle, _lib.ptr(xs[i]), B, _lib.ptr(lo), _lib.ptr(hi), offset,
                                        _lib.ptr(pars[i]), _lib.ptr(toks[i]), _lib.stream_ptr(dev)), "encode")

    def dec(i):
        _lib.check(lib.beast_decode_f32(plan.handle, _lib.ptr(toks[i]), B, _lib.ptr(lo), _lib.ptr(hi), offset,
                                        None, _lib.ptr(outs[i]), _lib.stream_ptr(dev)), "decode")

    def step(j):
        enc(j % R)
        dec((j + 2) % R)

    for i in range(R):
        enc(i)
    sampler = ClockSampler(local_rank)
    sampler.start()
    for j in range(args.warmup):
        step(j)
    torch.cuda.synchronize()
    K = args.steps

    # (a) per-kernel durations: CUDA events around every launch of the K timed steps
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(K)]
    for j in range(K):
        ev[j][0].record()
        enc(j % R)
        ev[j][1].record()
        dec((j + 2) % R)
        ev[j][2].record()
    torch.cuda.synchronize()
    enc_alt_ms = sum(e[0].elapsed_time(e[1]) for e in ev) / K
    dec_alt_ms = sum(e[1].elapsed_time(e[2]) for e in ev) / K
    # ... and K launches of ONE kernel back to back between two events (rotating buffer sets, no event record between
    # the launches): the kernel's average launch duration without the two event records that bracket every launch above
    e3 = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    e3[0].record()
    for j in range(K):
        enc(j % R)
    e3[1].record()
    for j in range(K):
        dec(j % R)
    e3[2].record()
    torch.cuda.synchronize()
    enc_ms, dec_ms = e3[0].elapsed_time(e3[1]) / K, e3[1].elapsed_time(e3[2]) / K
    enc_stream_ms, dec_stream_ms = enc_ms, dec_ms
    kernel_timing = f"CUDA events around {K} back-to-back launches of this kernel on the launching stream"
    # the same K launches replayed from a CUDA graph — the launch mode of the timed region below; plain stream launches
    # leave a ~2 us longer gap between two kernels (reported beside as ms_per_launch_stream)
    if os.environ.get("BEAST_BENCH_NO_GRAPH") != "1":
        try:
            per = []
            for fn in (enc, dec):
                g1 = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g1):
                    for j in range(K):
                        fn(j % R)
                g1.replay()
                torch.cuda.synchronize()
                ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                ea.record()
                g1.replay()
                eb.record()
                torch.cuda.synchronize()
                per.append(ea.elapsed_time(eb) / K)
                del g1
            enc_ms, dec_ms = per
            kernel_timing = (f"CUDA events around one replay of a CUDA graph holding {K} back-to-back launches of this kernel "
                             "(rotating buffer sets) on the launching stream — the launch mode of the timed region")
        except Exception as exc:                 # pragma: no cover
            print(f"[bench] per-kernel graph capture failed ({exc}); keeping the stream timing", file=sys.stderr)

    # (b) throughput: exactly K steps back to back, captured once into a CUDA graph (the launches are
    # the same C-ABI calls; the graph only removes the host launch gap between 60 us kernels)
    launch_mode = "cuda_graph"
    graph = None
    if os.environ.get("BEAST_BENCH_NO_GRAPH") != "1":
        try:
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                for j in range(K):
                    step(j)
            graph.replay()                       # one untimed replay (graph upload)
            torch.cuda.synchronize()
        except Exception as exc:                 # pragma: no cover
            print(f"[bench] graph capture failed ({exc}); timing plain stream launches", file=sys.stderr)
            graph = None
    if graph is None:
        launch_mode = "stream"
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    t_start = torch.cuda.Event(enable_timing=True)
    t_end = torch.cuda.Event(enable_timing=True)
    t_start.record()
    if graph is not None:
        graph.replay()
    else:
        for j in range(K):
            step(j)
    t_end.record()
    torch.cuda.synchronize()
    launches = (2 * K) if graph is not None else (_lib.launch_count() - n0)
    if world > 1:
        dist.barrier()
    ms_total = t_start.elapsed_time(t_end)
    if args.dump_outputs and rank == 0:
        last = K - 1                        # step(K - 1): encode of buffer set last % R, decode of set (last + 2) % R
        dump_outputs(args.dump_outputs, toks[last % R], pars[last % R], outs[(last + 2) % R])

    # ---- end-to-end leg: public API, pinned host input, results back on the host.  The step is the same
    # 65 536-trajectory batch, fed as 8 chunks over 3 streams so that the H2D copy of one chunk, the
    # kernels of another and the D2H copies of a third overlap (PCIe is full duplex).
    n_chunks = int(os.environ.get("BEAST_BENCH_E2E_CHUNKS", "8"))
    n_streams = int(os.environ.get("BEAST_BENCH_E2E_STREAMS", "3"))
    cb = B // n_chunks
    xh = [synth(B, T, D, seed=50 + 1000 * rank + i).pin_memory() for i in range(2)]
    tok_h = torch.empty((B, NB * D), dtype=torch.int64).pin_memory()
    rec_h = torch.empty((B, T, D), dtype=torch.float32).pin_memory()
    streams = [torch.cuda.Stream(device=dev) for _ in range(n_streams)]

    def e2e_step(i):
        src = xh[i % 2]
        for c in range(n_chunks):
            st = streams[c % n_streams]
            with torch.cuda.stream(st):
                sl = slice(c * cb, (c + 1) * cb if c < n_chunks - 1 else B)
                tokens, _ = tok.encode(src[sl])
                rec = tok.reconstruct_traj(tokens)
                tok_h[sl].copy_(tokens, non_blocking=True)
                rec_h[sl].copy_(rec, non_blocking=True)

    def e2e_sync():
        for st in streams:
            st.synchronize()

    Ke = max(3, min(K, 10))
    for i in range(3):
        e2e_step(i)
    e2e_sync()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    w0 = time.perf_counter()
    for i in range(Ke):
        e2e_step(i)
    e2e_sync()
    torch.cuda.synchronize()
    e2e_ms = 1e3 * (time.perf_counter() - w0)      # host clock around fully synchronised work on 3 streams
    # spot-check the pipelined results against a plain single-stream call
    chk_t, _ = tok.encode(xh[(Ke - 1) % 2][:cb])
    assert torch.equal(chk_t.cpu(), tok_h[:cb]), "pipelined e2e tokens differ"
    # copy-only ceiling of the same leg: the same pinned buffers, chunks and streams, no kernels — what the host
    # side (PCIe root, host DRAM) can move; e2e is to be read as a fraction of this
    dx = torch.empty((cb + n_chunks, T, D), device=dev, dtype=torch.float32)
    dtok = torch.empty((cb + n_chunks, NB * D), device=dev, dtype=torch.int64)
    drec = torch.empty((cb + n_chunks, T, D), device=dev, dtype=torch.float32)

    def copy_only_step(i):
        src = xh[i % 2]
        for c in range(n_chunks):
            st = streams[c % n_streams]
            with torch.cuda.stream(st):
                sl = slice(c * cb, (c + 1) * cb if c < n_chunks - 1 else B)
                n = sl.stop - sl.start
                dx[:n].copy_(src[sl], non_blocking=True)
                tok_h[sl].copy_(dtok[:n], non_blocking=True)
                rec_h[sl].copy_(drec[:n], non_blocking=True)

    copy_only_step(0)
    e2e_sync()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    c0 = time.perf_counter()
    for i in range(Ke):
        copy_only_step(i)
    e2e_sync()
    torch.cuda.synchronize()
    copy_ms = 1e3 * (time.perf_counter() - c0)
    del dx, dtok, drec
    sampler.stop_flag = True
    sampler.join(timeout=1.0)

    bounds = bounds_leg(tok, dev, with_cpu=world == 1 and not args.no_cpu_baseline) if rank == 0 else None
    shipped = cfg1 = None
    if rank == 0 and world == 1:
        shipped = shipped_shape_leg(dev, with_cpu=not args.no_cpu_baseline)
        cfg1 = cfg1_latency_leg(dev, with_cpu=not args.no_cpu_baseline)
    bpe_train = bpe_apply = None
    if not args.no_bpe:
        del xs, toks, pars, outs, xh
        torch.cuda.empty_cache()
        bpe_train, bpe_apply = bpe_legs(tok, dev, rank, world, dist, world == 1 and not args.no_cpu_baseline,
                                        cpu_full=not args.no_bpe_cpu_full)

    if world > 1:
        t = torch.tensor([ms_total, e2e_ms, enc_ms, dec_ms, copy_ms, enc_alt_ms, dec_alt_ms, enc_stream_ms, dec_stream_ms],
                         device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total, e2e_ms, enc_ms, dec_ms, copy_ms, enc_alt_ms, dec_alt_ms, enc_stream_ms, dec_stream_ms = [float(v) for v in t.tolist()]

    if rank == 0:
        peak, peak_src = measured_peak()
        enc_gbs = ENC_BYTES * B / (enc_ms * 1e-3) / 1e9
        dec_gbs = DEC_BYTES * B / (dec_ms * 1e-3) / 1e9
        line = {
            "metric": "trajectories/sec encode+decode", "value": world * B * K / (ms_total * 1e-3),
            "unit": "trajectories/s", "n_gpus": world, "steps": K, "warmup": args.warmup,
            "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "batch_per_gpu": B, "parallelism": f"dp{world} (batch sharded, no collective)",
                       "launch": launch_mode,
                       "l2": f"{R} rotating buffer sets ({R * (ENC_BYTES + DEC_BYTES) * B / 1e6:.0f} MB) > 126 MB L2; "
                             "decode reads tokens written two steps earlier"},
            "parity": {"tokens": "bit-exact given identical fp32 coefficients (beast_quantize_f32 on the reference's coefficients); fused K1 tokens == "
                                 "the exact quantiser applied to K1's own coefficients",
                       "flips_vs_reference": "profiles/flips_r02.json: 62 of 1 146 880 tokens (first 8 192 trajectories vs the reference's CPU path), all "
                                             "+-1 bin, reference coefficient within 3.7e-7 * max|w| of the rounding edge (criterion: coefficient tolerance "
                                             "1e-5 * max|w|, not 1 ulp — the reference's per-trajectory fp32 LU differs from the projector by ~2e-6)",
                       "coefficients_trajectories": "<= 1e-5 normwise vs the live reference's goldens (tests/test_gpu_spline.py)",
                       "bpe": "vocab.json / merges.txt / tokenizer.json byte-identical to the reference's files; ids bit-exact"},
            "e2e": {"value": world * B * Ke / (e2e_ms * 1e-3), "unit": "trajectories/s",
                    "h2d_bytes_per_step": 4 * T * D * B, "d2h_bytes_per_step": (8 * NB * D + 4 * T * D) * B,
                    "steps": Ke, "ms_per_step": e2e_ms / Ke, "copy_only_ms": copy_ms / Ke,
                    "frac_of_copy_only": copy_ms / e2e_ms,
                    "path": "BEASTBsplineTokenizer.encode(pinned host) -> reconstruct_traj -> tokens+trajectories to pinned host; "
                            f"{n_chunks} chunks over {n_streams} CUDA streams (H2D / kernels / D2H overlapped)", "timer": "host clock, all streams synchronised"},
            "gpu_launches": int(launches),
            "clocks": sampler.summary(),
            "roofline": {"bound": "hbm", "kernel": "encode_fast_kernel (K1)", "achieved": enc_gbs, "peak": peak,
                         "unit": "GB/s", "frac": enc_gbs / peak, "traffic": None, "peak_source": peak_src,
                         "bytes_per_launch": ENC_BYTES * B, "ms_per_launch": enc_ms,
                         "timing": kernel_timing, "ms_per_launch_stream": enc_stream_ms,
                         "ms_per_launch_alternating": enc_alt_ms, "frac_alternating": ENC_BYTES * B / (enc_alt_ms * 1e-3) / 1e9 / peak,
                         "alternating": "events around EVERY launch of the K1, K3, K1, ... step sequence (includes two event records per launch)",
                         "step_frac": (ENC_BYTES + DEC_BYTES) * B / (ms_total / K * 1e-3) / 1e9 / peak},
            "roofline_decode": {"bound": "hbm", "kernel": "decode_fast_kernel (K3)", "achieved": dec_gbs, "peak": peak,
                                "unit": "GB/s", "frac": dec_gbs / peak, "traffic": None,
                                "bytes_per_launch": DEC_BYTES * B, "ms_per_launch": dec_ms, "ms_per_launch_stream": dec_stream_ms,
                                "ms_per_launch_alternating": dec_alt_ms,
                                "frac_alternating": DEC_BYTES * B / (dec_alt_ms * 1e-3) / 1e9 / peak},
            "kernel_rates": {"encode_traj_per_s": B / (enc_ms * 1e-3), "decode_traj_per_s": B / (dec_ms * 1e-3)},
        }
        traffic_file = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(traffic_file):
            try:
                tr = json.load(open(traffic_file))
                line["roofline"]["traffic"] = tr.get("encode_fast_kernel")
                line["roofline_decode"]["traffic"] = tr.get("decode_fast_kernel")
            except Exception:
                pass
        if bounds is not None:
            line["bounds"] = bounds
        if shipped is not None:
            line["shipped_shape"] = shipped
        if cfg1 is not None:
            line["cfg1_latency"] = cfg1
        if bpe_train is not None:
            line["bpe_train"] = bpe_train
        if bpe_apply is not None:
            line["bpe_apply"] = bpe_apply
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline()
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
