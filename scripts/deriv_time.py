"""Time reconstruct_traj_derivatives' kernels through the C ABI on preallocated buffers (CUDA events over many launches
after warm-up) and write profiles/r04_deriv_sweep.json.

Sweep: geometries cfg2 (D = 14, T = 50, nb = 10, degree 4, two gripper slots), odd_d5 (D = 5, nb = 8, degree 3) and
the shipped shape (D = 32, nb = 50, degree 0); shared grids of Tq = 50 / 200 / 1000 samples over [0, duration];
orders (0,), (0, 1), (0, 1, 2); B = 1, 32, 65 536.  Per point: the tiled kernel (beast_decode_grid_f32) and, for
positions only, today's route to a custom grid, reconstruct_traj(times=grid.expand(B, -1)) = beast_decode_times_f32,
with a check that both return the same bits.  Byte model: the touched token bytes (the grid's token list) +
4 * D * Tq bytes per order written, per trajectory; achieved rate against the 6 543 GB/s copy peak of DESIGN §6.
Output buffers rotate so that consecutive launches write more than twice the 126 MB L2 (B = 1 / 32 stay launch-bound).

    python scripts/deriv_time.py [--out DIR]
"""
import argparse
import json
import math
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from beast_tokenizer_b200 import BEASTBsplineTokenizer, _lib  # noqa: E402
from beast_tokenizer_b200.synth import synth_device  # noqa: E402

PEAK_GBS = 6543.0
L2_BYTES = 126 * 2 ** 20
GEOMS = [
    ("cfg2", dict(num_dof=14, num_basis=10, seq_len=50, vocab_size=256, degree_p=4, gripper_zero_order=True,
                  gripper_indices=[6, 13])),
    ("odd_d5", dict(num_dof=5, num_basis=8, seq_len=33, vocab_size=1000, degree_p=3, gripper_zero_order=True,
                    gripper_indices=[0])),
    ("shipped", dict(num_dof=32, num_basis=50, seq_len=10, vocab_size=1000, degree_p=0)),
]
TQS = (50, 200, 1000)
ORDERS = ((0,), (0, 1), (0, 1, 2))
BATCHES = (1, 32, 65536)


def device_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return dict(zip(q.split(","), (s.strip() for s in out.split(","))))
    except Exception as exc:  # pragma: no cover
        return {"name": torch.cuda.get_device_name(0), "nvidia_smi": f"unavailable ({exc})"}


def touched_tokens(tok, grid_rows_j, grid_rows_g):
    """Tokens per trajectory the tiled kernel loads: (basis k, slot) pairs some row of the grid reads."""
    nj, ng = len(tok.joint_indices), len(tok.gripper_indices)
    used_j = int((grid_rows_j != 0).any(dim=1).any(dim=0).sum())
    used_g = int((grid_rows_g != 0).any(dim=1).any(dim=0).sum()) if grid_rows_g is not None else 0
    return used_j * nj + used_g * ng


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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles"))
    args = ap.parse_args()
    assert torch.cuda.is_available(), "deriv_time.py measures on a CUDA device"
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    info = device_info()
    print(json.dumps(info), flush=True)
    st = _lib.stream_ptr(dev)
    rows = []
    for gname, geom in GEOMS:
        tok = BEASTBsplineTokenizer(device="cuda", **geom)
        T, D, nb = geom["seq_len"], geom["num_dof"], geom["num_basis"]
        x = synth_device(max(BATCHES), T, D, 7, dev)
        tok.update_weights_bounds(x)
        tokens_all, _ = tok.encode(x)
        del x
        plan = tok._plan()
        lib = plan._lib
        lo, hi = tok._bounds(dev)
        for tq in TQS:
            grid_t = torch.linspace(0, float(tok.duration), tq)
            gr = tok._grid(plan, grid_t, 2)
            n_tok = touched_tokens(tok, gr._keep[1], gr._keep[2])
            for B in BATCHES:
                toks = tokens_all[:B].contiguous()
                out_bytes = B * tq * D * 4
                nbuf = max(1, min(16, math.ceil(2 * L2_BYTES / out_bytes))) if B >= 65536 else 1
                # today's route: per-row times, one thread per (row, sample)
                tt = grid_t.to(dev).expand(B, -1).contiguous()
                ref = [torch.empty((B, tq, D), device=dev) for _ in range(nbuf)]
                it = [0]

                def today():
                    o = ref[it[0] % nbuf]
                    it[0] += 1
                    _lib.check(lib.beast_decode_times_f32(plan.handle, _lib.ptr(toks), B, _lib.ptr(lo), _lib.ptr(hi),
                                                          0, None, _lib.ptr(tt), tq, _lib.ptr(o), st), "times")
                reps = 20 if B >= 65536 else 200
                t_today = time_ms(today, reps)
                for orders in ORDERS:
                    outs = [[torch.empty((B, tq, D), device=dev) if o in orders else None for o in range(3)]
                            for _ in range(nbuf)]
                    jt = [0]

                    def grid_call():
                        o = outs[jt[0] % nbuf]
                        jt[0] += 1
                        _lib.check(lib.beast_decode_grid_f32(plan.handle, gr.handle, _lib.ptr(toks), None, B, _lib.ptr(lo),
                                                             _lib.ptr(hi), 0, None, None, None,
                                                             *[_lib.ptr(t) for t in o], st), "grid")
                    t_grid = time_ms(grid_call, reps)
                    nbytes = B * (8 * n_tok + 4 * D * tq * len(orders))
                    row = dict(geometry=gname, Tq=tq, orders=list(orders), B=B, tiled_us=round(t_grid * 1e3, 2),
                               bytes=nbytes, tiled_GBs=round(nbytes / t_grid / 1e6, 1),
                               tiled_frac_of_copy_peak=round(nbytes / t_grid / 1e6 / PEAK_GBS, 3),
                               output_buffers=nbuf)
                    if orders == (0,):
                        torch.cuda.synchronize()
                        row["today_times_route_us"] = round(t_today * 1e3, 2)
                        row["speedup_vs_today"] = round(t_today / t_grid, 2)
                        # both wrote the positions of the same tokens on the same grid: the same bits
                        grid_call()
                        today()
                        torch.cuda.synchronize()
                        row["positions_bit_identical"] = bool(torch.equal(outs[(jt[0] - 1) % nbuf][0],
                                                                          ref[(it[0] - 1) % nbuf]))
                    rows.append(row)
                    print(json.dumps(row), flush=True)
                    del outs
                del ref, tt
                torch.cuda.empty_cache()
    result = dict(device=info, copy_peak_GBs=PEAK_GBS, byte_model="B * (8 * touched tokens + 4 * D * Tq * orders)",
                  rows=rows)
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "r04_deriv_sweep.json")
    with open(path, "w") as f:
        json.dump(result, f, indent=1)
    print(path)


if __name__ == "__main__":
    main()
