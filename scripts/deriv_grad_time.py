"""Time the backward of the continuous spline decode and write profiles/r05_deriv_grad_sweep.json.

Sweep: geometries cfg2 (D = 14, nb = 10, degree 4, two gripper slots), odd_d5 (D = 5, nb = 8, degree 3) and the
shipped shape (D = 32, nb = 50, degree 0); shared grids of Tq = 50 / 200 / 1000 samples over [0, duration]; orders
(0,), (0, 1, 2), (2,); B = 32 and 65 536.  Per point (CUDA events over many launches after warm-up):
  - kernel_us: beast_decode_grid_backward_f32 through the C ABI on preallocated buffers, against the byte model
    4 * D * Tq * NO bytes read + 4 * D * nb (+ 4 * D with init_p) written per trajectory and the 6 543 GB/s copy peak
    of DESIGN §6;
  - dense_us: the same gradient the way a user must compute it without this backward: the grid's basis rows as dense
    fp32 matrices, torch.einsum forward and autograd backward (TF32 off), forward + backward;
  - api_us: forward + backward through reconstruct_traj_continuous_derivatives (autograd, grads given).
The gradient buffers rotate so that consecutive launches read more than twice the 126 MB L2 (B = 32 stays
launch-bound).  The GPU name, power limit and SM clock are read in the same call.

    python scripts/deriv_grad_time.py [--out DIR]
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
ORDERS = ((0,), (0, 1, 2), (2,))
BATCHES = (32, 65536)
DENSE_MAX_BYTES = 4 << 30         # the dense einsum route is skipped above 4 GB of outputs


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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles"))
    args = ap.parse_args()
    assert torch.cuda.is_available(), "deriv_grad_time.py measures on a CUDA device"
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
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
        ct_all, _ = tok.encode_continuous(x)
        del x
        plan = tok._plan()
        lib = plan._lib
        nj = len(tok.joint_indices)
        perm = torch.tensor(tok.joint_indices + tok.gripper_indices, device=dev)
        inv = torch.empty_like(perm)
        inv[perm] = torch.arange(D, device=dev)
        for tq in TQS:
            grid_t = torch.linspace(0, float(tok.duration), tq)
            gr = tok._grid(plan, grid_t, 2)
            rj = gr._keep[1].to(dev)                                         # [3, Tq, nb] dense fp32
            rg = gr._keep[2].to(dev) if gr._keep[2] is not None else None
            for B in BATCHES:
                ct = ct_all[:B].contiguous()
                for orders in ORDERS:
                    no = len(orders)
                    g_bytes = B * tq * D * 4 * no
                    nbuf = max(1, min(8, math.ceil(2 * L2_BYTES / g_bytes))) if B >= 65536 else 1
                    grads = [[torch.randn((B, tq, D), device=dev) if o in orders else None for o in range(3)]
                             for _ in range(nbuf)]
                    gp = torch.empty((B, D * nb), device=dev)
                    it = [0]

                    def kernel():
                        g = grads[it[0] % nbuf]
                        it[0] += 1
                        _lib.check(lib.beast_decode_grid_backward_f32(plan.handle, gr.handle, B,
                                                                      *[_lib.ptr(t) for t in g], 0, _lib.ptr(gp),
                                                                      None, st), "backward")
                    reps = 20 if B >= 65536 else 200
                    t_k = time_ms(kernel, reps)
                    nbytes = B * (4 * D * tq * no + 4 * D * nb)
                    params = ct.clone().requires_grad_(True)
                    gsel = [grads[0][o] for o in orders]

                    def api():
                        params.grad = None
                        outs = tok.reconstruct_traj_continuous_derivatives(params, times=grid_t, orders=orders)
                        torch.autograd.backward(outs, gsel)
                    t_api = time_ms(api, reps)
                    api_grad = params.grad.clone()

                    def dense():
                        params.grad = None
                        c = tok._denormalize_continuous(params, dev).view(B, D, nb)
                        y = torch.einsum("otk,bsk->obts", rj[list(orders)], c[:, :nj])
                        if rg is not None:
                            yg = torch.einsum("otk,bsk->obts", rg[list(orders)], c[:, nj:])
                            y = torch.cat([y, yg], dim=-1)
                        y = y[..., inv]
                        torch.autograd.backward([y[i] for i in range(no)], gsel)
                    t_dense, dense_err = float("nan"), None
                    if g_bytes <= DENSE_MAX_BYTES:       # its intermediates hold several copies of the outputs
                        t_dense = time_ms(dense, max(5, reps // 4))
                        dense_err = float((params.grad - api_grad).abs().max() / api_grad.abs().max().clamp_min(1e-30))
                    row = dict(geometry=gname, Tq=tq, orders=list(orders), B=B, kernel_us=round(t_k * 1e3, 2),
                               bytes=nbytes, kernel_GBs=round(nbytes / t_k / 1e6, 1),
                               kernel_frac_of_copy_peak=round(nbytes / t_k / 1e6 / PEAK_GBS, 3),
                               api_fwd_bwd_us=round(t_api * 1e3, 2),
                               dense_einsum_fwd_bwd_us=None if dense_err is None else round(t_dense * 1e3, 2),
                               api_speedup_vs_dense=None if dense_err is None else round(t_dense / t_api, 2),
                               dense_vs_api_rel_diff=dense_err,
                               grad_buffers=nbuf)
                    rows.append(row)
                    print(json.dumps(row), flush=True)
                    del grads, gp, params, gsel
                    torch.cuda.empty_cache()
    result = dict(device=info, copy_peak_GBs=PEAK_GBS,
                  byte_model="B * (4 * D * Tq * orders read + 4 * D * nb written)", rows=rows)
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "r05_deriv_grad_sweep.json")
    with open(path, "w") as f:
        json.dump(result, f, indent=1)
    print(path)


if __name__ == "__main__":
    main()
