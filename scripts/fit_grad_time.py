"""Time the backward of the spline fit (encode_continuous) and write profiles/r06_fit_grad_sweep.json.

Sweep: geometries cfg2 (D = 14, nb = 10, T = 50, degree 4, two gripper slots), odd_d5 (D = 5, nb = 8, T = 33,
degree 3) and the shipped shape (D = 32, nb = 50, T = 10, degree 0); B = 32 and 65 536; the loss gradient on
`normalised` only, on `params` only, or on both.  Per point (CUDA events over many launches after a warm-up of every
shape):
  - kernel_us: beast_fit_backward_f32 through the C ABI on preallocated buffers, against the byte model
    4 * n_enc * (input arrays) bytes read + 4 * T * D written per trajectory (n_enc = coefficients whose projector
    row is not empty; grad_norm brings the coefficients along: two arrays, grad_params one) and the 6 543 GB/s copy
    peak of DESIGN §6, and against the sector model that counts the 32-byte sectors the listed entries fall in (on the
    shipped shape every fifth '(d t)' coefficient is listed, so whole rows of params / grad_params are fetched).  The
    output of the last timed launch is checked against the dense fp64 chain;
  - api_us: encode_continuous -> loss gradients -> backward (forward + backward through autograd);
  - dense_us: the route a user has without this backward: the plan's fp32 projectors as dense matrices, a
    torch.einsum fit, utils.normalize_tensor, autograd backward (TF32 off), forward + backward;
  - projection_us: the spline projection layer reconstruct_traj_continuous(encode_continuous(y)[0]), forward +
    backward, next to the same layer built from dense einsums (projector, then basis).
The gradient inputs and the coefficients rotate so that consecutive launches read more than twice the 126 MB L2 (B = 32 stays
launch-bound).  The GPU name, power limit and SM clocks are read in the same call.

    python scripts/fit_grad_time.py [--out DIR]
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
from beast_tokenizer_b200.utils import denormalize_tensor, normalize_tensor  # noqa: E402

PEAK_GBS = 6543.0
L2_BYTES = 126 * 2 ** 20
GEOMS = [
    ("cfg2", dict(num_dof=14, num_basis=10, seq_len=50, vocab_size=256, degree_p=4, gripper_zero_order=True,
                  gripper_indices=[6, 13])),
    ("odd_d5", dict(num_dof=5, num_basis=8, seq_len=33, vocab_size=1000, degree_p=3, gripper_zero_order=True,
                    gripper_indices=[0])),
    ("shipped", dict(num_dof=32, num_basis=50, seq_len=10, vocab_size=1000, degree_p=0)),
]
KINDS = ("norm", "params", "both")
BATCHES = (32, 65536)


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


def dense_tables(tok, dev):
    """[D, nb, T] fp32 projector and [D, T, nb] basis per slot, and the slot -> DoF permutation."""
    c = tok._plan().consts
    nj = len(c.joint_indices)
    P = torch.stack([c.proj_joint if s < nj else c.proj_grip for s in range(c.num_dof)]).to(dev)
    Phi = torch.stack([c.phi_joint if s < nj else c.phi_grip for s in range(c.num_dof)]).to(dev)
    slots = torch.tensor(c.slot_to_dof, device=dev)
    return P, Phi, slots


def ref64(tok, P, slots, params, lo, hi, gn, gp):
    """The dense fp64 chain of the backward (mask and scale on the fp32 coefficients and bounds)."""
    B = params.shape[0]
    D, nb = tok.num_dof, tok.num_basis
    gw = torch.zeros((B, D, nb), device=params.device, dtype=torch.float64)
    if gn is not None:
        mask = (params >= lo) & (params <= hi)
        scale = (hi.double() - lo.double()).clamp_min(1e-8)
        gw += (mask * gn.view(B, nb, D).transpose(1, 2).reshape(B, -1).double() * 2.0 / scale).view(B, D, nb)
    if gp is not None:
        gw += gp.double().view(B, D, nb)
    gy = torch.einsum("bsk,skt->bts", gw, P.double())
    out = torch.empty_like(gy)
    out[..., slots] = gy
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles"))
    args = ap.parse_args()
    assert torch.cuda.is_available(), "fit_grad_time.py measures on a CUDA device"
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
        x_all = synth_device(max(BATCHES), T, D, 7, dev)
        tok.update_weights_bounds(x_all[: max(BATCHES) // 2])       # the other half partly outside the bounds
        plan = tok._plan()
        lib = plan._lib
        P, Phi, slots = dense_tables(tok, dev)
        n_enc = sum(int((tab != 0).any(1).sum()) * n for tab, n in (
            (plan.consts.proj_joint, len(tok.joint_indices)),
            (plan.consts.proj_grip, len(tok.gripper_indices))) if tab is not None)
        lo, hi = tok.w_min.clone(), tok.w_max.clone()
        # bytes of the 32-byte sectors the listed entries fall in (over 64 consecutive rows), per input array: the
        # '(t d)' gradient of normalised, and the '(d t)' params / grad_params
        nj = len(tok.joint_indices)
        listed = [(k, s) for k in range(nb) for s in range(D)
                  if bool(((plan.consts.proj_joint if s < nj else plan.consts.proj_grip)[k] != 0).any())]
        row_b = D * nb * 4
        sec = {lay: len({(b * row_b + 4 * i) // 32 for b in range(64) for i in idx}) * 32 / 64 for lay, idx in (
            ("td", [k * D + s for k, s in listed]), ("dt", [s * nb + k for k, s in listed]))}
        for B in BATCHES:
            x = x_all[:B].contiguous()
            params = tok.compute_weights(x)
            for kind in KINDS:
                n_arr = {"norm": 2, "params": 1, "both": 3}[kind]
                in_bytes = B * D * nb * 4 * n_arr
                nbuf = max(1, min(8, math.ceil(2 * L2_BYTES / max(in_bytes, 1)))) if B >= 65536 else 1
                bufs = [[torch.randn((B, D * nb), device=dev) if kind in ("norm", "both") else None,
                         torch.randn((B, D * nb), device=dev) if kind in ("params", "both") else None,
                         params.clone() if kind in ("norm", "both") else params]
                        for _ in range(nbuf)]
                gy = torch.empty((B, T, D), device=dev)
                it = [0]

                def kernel():
                    gn, gp, par = bufs[it[0] % nbuf]
                    it[0] += 1
                    _lib.check(lib.beast_fit_backward_f32(plan.handle, B, _lib.ptr(gn), _lib.ptr(gp), _lib.ptr(par),
                                                          _lib.ptr(lo), _lib.ptr(hi), _lib.ptr(gy), st), "backward")
                reps = 50 if B >= 65536 else 200
                time_ms(kernel, 1, warm=3)
                it[0] = 0
                t_k = time_ms(kernel, reps, warm=0)
                last = bufs[(reps - 1) % nbuf]
                want = ref64(tok, P, slots, last[2], lo, hi, last[0], last[1])
                err = float((gy.double() - want).abs().max() / want.abs().max().clamp_min(1e-30))
                assert err <= 1e-5, (gname, B, kind, err)
                nbytes = B * (4 * n_enc * n_arr + 4 * T * D)
                lays = {"norm": ("td", "dt"), "params": ("dt",), "both": ("td", "dt", "dt")}[kind]
                sbytes = int(B * (sum(sec[lay] for lay in lays) + 4 * T * D))
                gn0, gp0 = bufs[0][:2]
                y = x.clone().requires_grad_(True)

                def api():
                    y.grad = None
                    norm, pd = tok.encode_continuous(y)
                    outs = [o for o, g in ((norm, gn0), (pd["params"], gp0)) if g is not None]
                    torch.autograd.backward(outs, [g for g in (gn0, gp0) if g is not None])
                t_api = time_ms(api, reps)
                api_grad = y.grad.clone()

                def dense():
                    y.grad = None
                    w = torch.einsum("skt,bts->bsk", P, y[..., slots]).reshape(B, D * nb)
                    outs, gs = [], []
                    if gn0 is not None:
                        nrm = normalize_tensor(w, lo, hi).view(B, D, nb).transpose(1, 2).reshape(B, nb * D)
                        outs.append(nrm)
                        gs.append(gn0)
                    if gp0 is not None:
                        outs.append(w)
                        gs.append(gp0)
                    torch.autograd.backward(outs, gs)
                t_dense = time_ms(dense, max(5, reps // 4))
                dense_diff = float((y.grad - api_grad).abs().max() / api_grad.abs().max().clamp_min(1e-30))
                row = dict(geometry=gname, B=B, grads=kind, n_enc=n_enc, kernel_us=round(t_k * 1e3, 2), bytes=nbytes,
                           kernel_GBs=round(nbytes / t_k / 1e6, 1),
                           kernel_frac_of_copy_peak=round(nbytes / t_k / 1e6 / PEAK_GBS, 3),
                           sector_bytes=sbytes, kernel_sector_frac_of_copy_peak=round(sbytes / t_k / 1e6 / PEAK_GBS, 3),
                           kernel_vs_fp64_rel_err=err, grad_buffers=nbuf,
                           api_fwd_bwd_us=round(t_api * 1e3, 2), dense_einsum_fwd_bwd_us=round(t_dense * 1e3, 2),
                           api_speedup_vs_dense=round(t_dense / t_api, 2), dense_vs_api_rel_diff=dense_diff)
                if kind == "norm":
                    wt = torch.randn((B, T, D), device=dev)

                    def proj():
                        y.grad = None
                        out = tok.reconstruct_traj_continuous(tok.encode_continuous(y)[0])
                        out.backward(wt)

                    def proj_dense():
                        y.grad = None
                        w = torch.einsum("skt,bts->bsk", P, y[..., slots]).reshape(B, D * nb)
                        nrm = normalize_tensor(w, lo, hi)
                        c = denormalize_tensor(nrm, lo, hi).view(B, D, nb)
                        out = torch.empty((B, T, D), device=dev)
                        out[..., slots] = torch.einsum("stk,bsk->bts", Phi, c)
                        out.backward(wt)
                    row["projection_api_us"] = round(time_ms(proj, reps) * 1e3, 2)
                    row["projection_dense_us"] = round(time_ms(proj_dense, max(5, reps // 4)) * 1e3, 2)
                rows.append(row)
                print(json.dumps(row), flush=True)
                del bufs, gy, y
                torch.cuda.empty_cache()
        del x_all
    result = dict(device=info, copy_peak_GBs=PEAK_GBS,
                  byte_model="B * (4 * n_enc * input arrays read + 4 * T * D written); input arrays: norm = grad_norm "
                             "+ params, params = grad_params, both = all three",
                  sector_byte_model="the same with every input array counted in the 32-byte sectors its listed entries "
                                    "fall in",
                  rows=rows)
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "r06_fit_grad_sweep.json")
    with open(path, "w") as f:
        json.dump(result, f, indent=1)
    print(path)


if __name__ == "__main__":
    main()
