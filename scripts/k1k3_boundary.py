"""Where the K1 / K3 step time goes: steady-state bandwidth against per-launch fixed cost.

    python scripts/k1k3_boundary.py [--out FILE.json]          # sweep
    python scripts/k1k3_boundary.py --ab [--out FILE.json]     # overlap on / forced off, same step graph

Sweep: the bench's workload (bimanual tokenizer, bounds from the bench's synthetic loader, the bench's seeds, 4 rotating
buffer sets larger than L2, the bench's C-ABI calls), timed as graph replays of K back-to-back K1 launches, K back-to-back
K3 launches and K alternating K1 / K3 steps (encode of set j, decode of set j+2) at B = 16 384 ... 262 144 trajectories.
A least-squares line t = a + b*B per series splits a launch into its per-launch intercept a (fill, drain and launch
boundary) and its steady-state rate: bytes / b.  The step's excess is what the alternating step costs beyond the sum of
its two kernels.

--ab: the bench's step graph (B = 65 536) captured twice, once as the library launches it (K1 / K3 overlap across the
launch boundary when their buffers are disjoint) and once with beast_debug_force_wait(1) (every launch waits for its
predecessor), replays alternated; median and min-max of us per step.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from bench import D, DEC_BYTES, ENC_BYTES, GRIP, LLM_VOCAB, NB, T, V, ClockSampler  # noqa: E402

R = 4
SIZES = (16384, 32768, 65536, 131072, 262144)


def device_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return dict(zip(q.split(","), (s.strip() for s in out.split(","))))
    except Exception as exc:  # pragma: no cover
        return {"name": torch.cuda.get_device_name(0), "nvidia_smi": f"unavailable ({exc})"}


class Workload:
    def __init__(self, dev):
        from beast_tokenizer_b200 import BEASTBsplineTokenizer, _lib
        from beast_tokenizer_b200.synth import SyntheticLoader
        self.dev, self._lib = dev, _lib
        self.tok = BEASTBsplineTokenizer(num_dof=D, num_basis=NB, seq_len=T, vocab_size=V, gripper_zero_order=True,
                                         gripper_indices=GRIP, device=str(dev), llm_vocab_size=LLM_VOCAB)
        self.tok.fit_parameters(SyntheticLoader(100, 32, T, D, seed0=1), verbose=False)
        self.plan = self.tok._plan()
        self.lib = self.plan._lib
        self.lo, self.hi = self.tok._bounds(dev)
        self.offset = LLM_VOCAB - V

    def buffers(self, B):
        from beast_tokenizer_b200.synth import synth
        self.B = B
        self.xs = [synth(B, T, D, seed=2 + i, device=self.dev) for i in range(R)]
        self.toks = [torch.empty((B, NB * D), device=self.dev, dtype=torch.int64) for _ in range(R)]
        self.pars = [torch.empty((B, NB * D), device=self.dev, dtype=torch.float32) for _ in range(R)]
        self.outs = [torch.empty((B, T, D), device=self.dev, dtype=torch.float32) for _ in range(R)]
        for i in range(R):
            self.enc(i)
        torch.cuda.synchronize()

    def enc(self, i):
        L, p = self._lib, self._lib.ptr
        L.check(self.lib.beast_encode_f32(self.plan.handle, p(self.xs[i]), self.B, p(self.lo), p(self.hi), self.offset,
                                          p(self.pars[i]), p(self.toks[i]), L.stream_ptr(self.dev)), "encode")

    def dec(self, i):
        L, p = self._lib, self._lib.ptr
        L.check(self.lib.beast_decode_f32(self.plan.handle, p(self.toks[i]), self.B, p(self.lo), p(self.hi), self.offset,
                                          None, p(self.outs[i]), L.stream_ptr(self.dev)), "decode")

    def step(self, j):
        self.enc(j % R)
        self.dec((j + 2) % R)


def capture(fn):
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fn()
    g.replay()                      # upload
    torch.cuda.synchronize()
    return g


def replay_us(g, n_units):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / n_units


def fit(xs, ys):
    b, a = np.polyfit(np.asarray(xs, float), np.asarray(ys, float), 1)
    resid = np.asarray(ys) - (a + b * np.asarray(xs, float))
    return float(a), float(b), float(np.abs(resid).max())


def sweep(w, K, reps):
    rows = []
    for B in SIZES:
        w.buffers(B)
        graphs = {
            "k1": capture(lambda: [w.enc(j % R) for j in range(K)]),
            "k3": capture(lambda: [w.dec(j % R) for j in range(K)]),
            "step": capture(lambda: [w.step(j) for j in range(K)]),
        }
        t = {k: [] for k in graphs}
        for _ in range(reps):           # interleaved, so that a slow phase of the machine hits every series alike
            for k, g in graphs.items():
                t[k].append(replay_us(g, K))
        row = {"B": B}
        for k in graphs:
            row[k + "_us"] = float(np.median(t[k]))
            row[k + "_us_min_max"] = [float(min(t[k])), float(max(t[k]))]
        row["step_excess_us"] = row["step_us"] - row["k1_us"] - row["k3_us"]
        rows.append(row)
        print(f"B={B:7d}  K1 {row['k1_us']:8.2f} us  K3 {row['k3_us']:8.2f} us  step {row['step_us']:8.2f} us  "
              f"excess {row['step_excess_us']:+6.2f} us", flush=True)
        del graphs
        torch.cuda.synchronize()
    Bs = [r["B"] for r in rows]
    res = {}
    for k, nbytes in (("k1", ENC_BYTES), ("k3", DEC_BYTES), ("step", ENC_BYTES + DEC_BYTES)):
        a, b, r = fit(Bs, [row[k + "_us"] for row in rows])
        res[k] = {"intercept_us": a, "us_per_1k_traj": b * 1e3, "steady_gbs": nbytes / b / 1e3, "max_resid_us": r}
        print(f"{k:5s} t = {a:6.2f} us + B * {b * 1e3:.4f} us/1k traj   steady state {nbytes / b / 1e3:7.0f} GB/s   "
              f"max residual {r:.2f} us", flush=True)
    return {"rows": rows, "fit": res}


def ab(w, K, pairs):
    lib = w.lib
    w.buffers(65536)
    graphs = {}
    for mode, flag in (("overlap", 0), ("forced_wait", 1)):
        prev = lib.beast_debug_force_wait(flag)
        n0 = lib.beast_overlap_count()
        graphs[mode] = capture(lambda: [w.step(j) for j in range(K)])
        graphs[mode + "_overlapped_launches"] = int(lib.beast_overlap_count() - n0)
        lib.beast_debug_force_wait(prev)
    t = {"overlap": [], "forced_wait": []}
    for _ in range(pairs):
        for mode in t:
            t[mode].append(replay_us(graphs[mode], K))
    out = {"K": K, "pairs": pairs, "launches_per_graph": 2 * K,
           "overlapped_launches": {m: graphs[m + "_overlapped_launches"] for m in t}}
    for mode, v in t.items():
        out[mode] = {"median_us": float(np.median(v)), "min_us": float(min(v)), "max_us": float(max(v)), "all_us": v}
        print(f"{mode:12s} median {np.median(v):7.2f} us/step   min {min(v):7.2f}   max {max(v):7.2f}   "
              f"({out['overlapped_launches'][mode]} of {2 * K} launches overlapped)", flush=True)
    out["gain_pct"] = 100.0 * (1.0 - out["overlap"]["median_us"] / out["forced_wait"]["median_us"])
    out["spreads_disjoint"] = out["overlap"]["max_us"] < out["forced_wait"]["min_us"]
    print(f"gain {out['gain_pct']:.1f} %   spreads disjoint: {out['spreads_disjoint']}", flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ab", action="store_true", help="A/B of the launch-boundary overlap instead of the sweep")
    ap.add_argument("--steps", type=int, default=40, help="launches (sweep) or steps (A/B) per graph")
    ap.add_argument("--reps", type=int, default=10, help="replays per series (sweep) or per mode (A/B)")
    ap.add_argument("--out", help="write the result as JSON here")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("k1k3_boundary.py measures on the GPU; no CUDA device is present")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    info = device_info()
    print(json.dumps(info), flush=True)
    sampler = ClockSampler(0)
    sampler.start()
    w = Workload(dev)
    result = {"device": info}
    if args.ab:
        result["ab"] = ab(w, args.steps, args.reps)
    else:
        result["sweep"] = sweep(w, args.steps, args.reps)
    sampler.stop_flag = True
    sampler.join()
    result["clocks"] = sampler.summary()
    print(json.dumps(result["clocks"]), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
