"""Time the masked spline fit and write profiles/r09_fit_mask_sweep.json.

Sweep: geometries cfg2 (D = 14, nb = 10, T = 50, degree 4, two gripper slots) and the shipped shape (D = 32, nb = 50,
T = 10, degree 0); B = 65 536; suffix padding (valid length uniform in [T/2, T-1]) on 0 %, 1 %, 10 % and 100 % of the
rows, the tokenizer's own times.  Per point (CUDA events over many calls after a warm-up; inputs rotate over copies
that together exceed twice the 126 MB L2):
  - encode_none_us / encode_mask_us: tok.encode(y) against tok.encode(y, mask=m) (K1, then beast_fit_masked_f32 over
    the rows with a masked sample, then one beast_quantize_f32);
  - kernel_partial_us: beast_fit_masked_f32 alone with partial_only = 1 on one grid (what encode launches);
    kernel_all_us: the same with partial_only = 0 (every row refitted);
  - fwd_bwd_none_us / fwd_bwd_mask_us: encode_continuous(y[, mask=m]) -> loss on the normalised coefficients ->
    backward;
  - workaround_us: what a user does without the mask: group the rows by valid count (one host sync) and call
    encode(y[rows, :k], times=[k]-grid) once per group, tokens scattered back.
The GPU name, power limit and SM clocks are read in the same call.

    python scripts/fit_mask_time.py [--out DIR]
"""
import argparse
import json
import math
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from beast_tokenizer_b200 import BEASTBsplineTokenizer, _lib  # noqa: E402

L2_BYTES = 126 * 2 ** 20
GEOMS = [
    ("cfg2", dict(num_dof=14, num_basis=10, seq_len=50, vocab_size=256, degree_p=4, gripper_zero_order=True,
                  gripper_indices=[6, 13])),
    ("shipped", dict(num_dof=32, num_basis=50, seq_len=10, vocab_size=1000, degree_p=0)),
]
B = 65536
FRACTIONS = (0.0, 0.01, 0.1, 1.0)


def device_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return dict(zip(q.split(","), (s.strip() for s in out.split(","))))
    except Exception as exc:  # pragma: no cover
        return {"name": torch.cuda.get_device_name(0), "nvidia_smi": f"unavailable ({exc})"}


def time_ms(fn, reps, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def suffix_mask(B, T, frac, dev, seed):
    g = torch.Generator(device=dev).manual_seed(seed)
    partial = torch.rand(B, 1, device=dev, generator=g) < frac
    n = torch.randint(T // 2, T, (B, 1), device=dev, generator=g)
    n = torch.where(partial, n, torch.full_like(n, T))
    return (torch.arange(T, device=dev).expand(B, T) < n).contiguous()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    res = {"device": device_info(), "B": B, "points": []}
    lib = _lib.load()
    st = _lib.stream_ptr(dev)
    for name, cfg in GEOMS:
        tok = BEASTBsplineTokenizer(device="cuda", **cfg)
        tok.w_min.fill_(-1.0)
        tok.w_max.fill_(1.0)
        plan = tok._plan()
        grid = plan.device_times()
        T, D, nb = cfg["seq_len"], cfg["num_dof"], cfg["num_basis"]
        per_call = B * (4 * T * D + T + 8 * D * nb)
        copies = max(1, min(16, math.ceil(2 * L2_BYTES / per_call)))
        g = torch.Generator(device=dev).manual_seed(T)
        ys = [0.02 * torch.randn(B, T, D, device=dev, generator=g) for _ in range(copies)]
        outs = [torch.empty(B, D * nb, device=dev) for _ in range(copies)]
        for frac in FRACTIONS:
            ms = [suffix_mask(B, T, frac, dev, 100 * i + int(frac * 100)) for i in range(copies)]
            i = [0]

            def nxt():
                k = i[0] % copies
                i[0] += 1
                return k

            def enc_none():
                tok.encode(ys[nxt()])

            def enc_mask():
                k = nxt()
                tok.encode(ys[k], mask=ms[k])

            def kern(partial):
                def f():
                    k = nxt()
                    rc = lib.beast_fit_masked_f32(plan.handle, _lib.ptr(ys[k]), B, T, _lib.ptr(grid), 0,
                                                  _lib.ptr(ms[k]), partial, None, None, _lib.ptr(outs[k]), st)
                    assert rc == 0, rc
                return f

            def fwd_bwd(masked):
                def f():
                    k = nxt()
                    x = ys[k].detach().requires_grad_(True)
                    n, _ = tok.encode_continuous(x, mask=ms[k] if masked else None)
                    n.sum().backward()
                return f

            def workaround():
                k = nxt()
                y, m = ys[k], ms[k]
                counts = m.sum(1)
                tokens = torch.empty(B, D * nb, device=dev, dtype=torch.int64)
                for c in torch.unique(counts).tolist():          # host sync: the groups' sizes
                    rows = (counts == c).nonzero().squeeze(1)
                    if c == T:
                        tokens[rows] = tok.encode(y[rows])[0]
                    else:
                        t = tok.times[:c].to(dev).expand(rows.numel(), -1)
                        tokens[rows] = tok.encode(y[rows, :c], times=t)[0]

            reps = 200 if T <= 10 else 100
            pt = {"geometry": name, "B": B, "T": T, "D": D, "nb": nb, "partial_fraction": frac,
                  "partial_rows": int((~ms[0].all(1)).sum()), "copies": copies, "reps": reps}
            pt["encode_none_us"] = time_ms(enc_none, reps) * 1e3
            pt["encode_mask_us"] = time_ms(enc_mask, reps) * 1e3
            pt["kernel_partial_us"] = time_ms(kern(1), reps) * 1e3
            pt["kernel_all_us"] = time_ms(kern(0), reps) * 1e3
            pt["fwd_bwd_none_us"] = time_ms(fwd_bwd(False), max(10, reps // 4)) * 1e3
            pt["fwd_bwd_mask_us"] = time_ms(fwd_bwd(True), max(10, reps // 4)) * 1e3
            pt["workaround_us"] = time_ms(workaround, 10, warm=1) * 1e3
            pt["encode_mask_over_none"] = pt["encode_mask_us"] / pt["encode_none_us"]
            # the timed masked encode agrees with the workaround's per-group fit
            k = 0
            tk, _ = tok.encode(ys[k], mask=ms[k])
            counts = ms[k].sum(1)
            agree = True
            for c in torch.unique(counts).tolist()[:4]:
                rows = (counts == c).nonzero().squeeze(1)[:64]
                t = tok.times[:c].to(dev).expand(rows.numel(), -1)
                agree &= bool(torch.equal(tk[rows], tok.encode(ys[k][rows, :c], times=t)[0])) if c < T else True
            pt["tokens_equal_per_group_fit"] = agree
            res["points"].append(pt)
            print(json.dumps(pt), flush=True)
        del ys, outs
        torch.cuda.empty_cache()
    res["device_after"] = device_info()
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "r09_fit_mask_sweep.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
