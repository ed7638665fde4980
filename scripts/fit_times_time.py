"""Time the spline fit on per-row times and write profiles/r07_fit_times_sweep.json.

Sweep: geometries cfg2 (D = 14, nb = 10, T = 50, degree 4, two gripper slots), odd_d5 (D = 5, nb = 8, T = 33,
degree 3), the shipped shape (D = 32, nb = 50, T = 10, degree 0) and T = 1987 (D = 7, nb = 10, degree 4, one gripper);
B = 32, 4 096 and 65 536; jittered per-row times.  Per point (CUDA events over many launches after a warm-up of every
shape):
  - kernel_us: beast_fit_times_f32 through the C ABI on preallocated buffers; inputs and outputs rotate over copies
    that together exceed twice the 126 MB L2 (B = 32 stays launch-bound).  Byte model 4 * T * (D + 1) read + 4 * D * nb
    written per row against the 6 543 GB/s copy peak of DESIGN §6;
  - backward_us: beast_fit_times_backward_f32 (gradient of params only) on the same rotation;
  - api_fwd_bwd_us: encode_continuous(y, times=t) -> loss on the normalised coefficients -> backward;
  - dense_fp32_us / dense_fp64_us: the route a user has without the kernel: per-row basis rows built as tensors
    (basis.bspline_basis on the device), bmm normal equations, torch.linalg.cholesky + cholesky_solve (TF32 off);
  - reference_cpu_rows_per_s: the reference's per-row fp32 fit (oracle/reference_port_torch.py ReferencePort._learn,
    which takes [B, T] times) on the host at B = 256.
The GPU name, power limit and SM clocks are read in the same call.

    python scripts/fit_times_time.py [--out DIR] [--quick]
"""
import argparse
import json
import math
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from beast_tokenizer_b200 import BEASTBsplineTokenizer, _lib, basis  # noqa: E402

PEAK_GBS = 6543.0
L2_BYTES = 126 * 2 ** 20
GEOMS = [
    ("cfg2", dict(num_dof=14, num_basis=10, seq_len=50, vocab_size=256, degree_p=4, gripper_zero_order=True,
                  gripper_indices=[6, 13])),
    ("odd_d5", dict(num_dof=5, num_basis=8, seq_len=33, vocab_size=1000, degree_p=3, gripper_zero_order=True,
                    gripper_indices=[0])),
    ("shipped", dict(num_dof=32, num_basis=50, seq_len=10, vocab_size=1000, degree_p=0)),
    ("t1987", dict(num_dof=7, num_basis=10, seq_len=1987, vocab_size=256, degree_p=4, gripper_zero_order=True,
                   gripper_indices=[3])),
]
BATCHES = (32, 4096, 65536)


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


def jitter_times(B, T, dur, dev, seed):
    g = torch.Generator(device=dev).manual_seed(seed)
    step = dur / (T - 1)
    t = torch.linspace(0, dur, T, device=dev).expand(B, -1) + 0.3 * step * (torch.rand(B, T, device=dev, generator=g) - 0.5)
    return t.clamp(0, dur).sort(dim=1).values.contiguous()


def dense_route(tok, y, t, dtype):
    """Per-row basis rows, normal equations by bmm, Cholesky solve (joint and gripper splines)."""
    nb, p = tok.num_basis, tok.degree_p
    outs = []
    for idx, deg in ((tok.joint_indices, p), (tok.gripper_indices, 0)):
        if not idx:
            continue
        phi = basis.bspline_basis(t, tok.duration, nb, deg).to(dtype)          # [B, T, nb]
        G = torch.bmm(phi.transpose(1, 2), phi) + 1e-9 * torch.eye(nb, device=y.device, dtype=dtype)
        rhs = torch.bmm(phi.transpose(1, 2), y[..., idx].to(dtype))          # [B, nb, d]
        outs.append(torch.cholesky_solve(rhs, torch.linalg.cholesky(G)).transpose(1, 2).reshape(y.shape[0], -1))
    return torch.cat(outs, dim=1).float()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    ap.add_argument("--quick", action="store_true", help="B = 32 and 4 096 only")
    args = ap.parse_args()
    torch.backends.cuda.matmul.allow_tf32 = False
    dev = torch.device("cuda", 0)
    info = device_info()
    res = {"device": info, "peak_copy_GBs": PEAK_GBS, "points": []}
    lib = _lib.load()
    for name, cfg in GEOMS:
        tok = BEASTBsplineTokenizer(device="cuda", **cfg)
        tok.w_min.fill_(-1.0)
        tok.w_max.fill_(1.0)
        plan = tok._plan()
        T, D, nb = cfg["seq_len"], cfg["num_dof"], cfg["num_basis"]
        for B in BATCHES if not args.quick else BATCHES[:2]:
            per_call = 4 * B * (T * (D + 1) + D * nb)
            copies = max(1, min(64, math.ceil(2 * L2_BYTES / per_call)))
            if copies * per_call > 40 * 2 ** 30:
                copies = 1
            g = torch.Generator(device=dev).manual_seed(B)
            ys = [0.02 * torch.randn(B, T, D, device=dev, generator=g) for _ in range(copies)]
            ts = [jitter_times(B, T, float(tok.duration), dev, B + i) for i in range(copies)]
            outs = [torch.empty(B, D * nb, device=dev) for _ in range(copies)]
            gys = [torch.empty(B, T, D, device=dev) for _ in range(copies)]
            i = [0]
            st = _lib.stream_ptr(dev)

            def fwd():
                k = i[0] % copies
                i[0] += 1
                rc = lib.beast_fit_times_f32(plan.handle, _lib.ptr(ys[k]), B, T, _lib.ptr(ts[k]), None, None,
                                             _lib.ptr(outs[k]), st)
                assert rc == 0, rc

            def bwd():
                k = i[0] % copies
                i[0] += 1
                rc = lib.beast_fit_times_backward_f32(plan.handle, B, T, _lib.ptr(ts[k]), None, _lib.ptr(outs[k]),
                                                      None, None, None, _lib.ptr(gys[k]), None, None, st)
                assert rc == 0, rc

            reps = max(20, min(2000, int(2e9 / per_call)))
            k_ms = time_ms(fwd, reps)
            b_ms = time_ms(bwd, reps)
            bytes_model = per_call
            pt = {"geometry": name, "B": B, "T": T, "D": D, "nb": nb, "copies": copies, "reps": reps,
                  "kernel_us": k_ms * 1e3, "bytes": bytes_model,
                  "GBs": bytes_model / (k_ms * 1e-3) / 1e9, "share_of_copy_peak": bytes_model / (k_ms * 1e-3) / 1e9 / PEAK_GBS,
                  "backward_us": b_ms * 1e3}
            # accuracy of the timed output against the dense fp64 route
            ref = dense_route(tok, ys[0][:256], ts[0][:256], torch.float64)
            pt["max_abs_err_vs_fp64_first256"] = float((outs[0][:256] - ref).abs().max())
            x = ys[0].clone().requires_grad_(True)

            def api():
                x.grad = None
                n, _ = tok.encode_continuous(x, times=ts[0])
                n.sum().backward()

            pt["api_fwd_bwd_us"] = time_ms(api, max(5, reps // 20)) * 1e3
            if B <= 4096 or T <= 50:
                for dt, key in ((torch.float32, "dense_fp32_us"), (torch.float64, "dense_fp64_us")):
                    pt[key] = time_ms(lambda: dense_route(tok, ys[0], ts[0], dt), 5, warm=1) * 1e3
            res["points"].append(pt)
            print(json.dumps(pt), flush=True)
            del ys, ts, outs, gys, x
            torch.cuda.empty_cache()
        # the reference's per-row fp32 fit on the host
        from oracle.reference_port_torch import ReferencePort
        ref = ReferencePort(**{k: v for k, v in cfg.items()})
        Bc = 256 if T <= 50 else 16
        tc = jitter_times(Bc, T, float(tok.duration), dev, 7).cpu()
        yc = 0.02 * torch.randn(Bc, T, D)
        t0 = time.perf_counter()
        ref._learn(tc, yc[..., ref.joint], cfg["degree_p"])
        if ref.grip:
            ref._learn(tc, yc[..., ref.grip], 0)
        dt = time.perf_counter() - t0
        res["points"].append({"geometry": name, "reference_cpu_B": Bc, "reference_cpu_rows_per_s": Bc / dt})
        print(json.dumps(res["points"][-1]), flush=True)
    res["device_after"] = device_info()
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "r07_fit_times_sweep.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
