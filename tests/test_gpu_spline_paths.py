"""The spline encode / decode fast paths at the batch sizes where their pipelines actually turn over, for every kernel
instantiation and branch, against an independent fp64 least-squares fit.

Every encode / reconstruct ends in one of three kernel families: the bulk-copy kernels (`encode_fast_kernel<50, 10, D>`,
`decode_fast_kernel<50, 10, D>`, csrc/spline_encode.cu / spline_decode.cu), the tiled kernels (`encode_tiled_kernel<R>`,
`decode_tiled_kernel<FROM_TOKENS>`, csrc/spline_tiled.cu) and the one-thread-per-column reference kernels
(`beast_debug_disable_fast`).  The small-batch tests give every CTA one tile; here each geometry runs at a batch large
enough that every persistent CTA walks at least three tiles (the double buffer's mbarrier parity flips twice, the
staging and template rows are reused, a ragged hand-loaded last tile follows bulk-loaded ones) or, for the bulk-copy
kernels, that every CTA's five-stage ring wraps at least twice with a ragged tail left to the tiled kernel.

Three independent anchors:
  * fast == reference kernels, bit for bit, on every row (on the GPU);
  * fused tokens == the exact quantiser applied to the kernel's own coefficients, on every row;
  * coefficients and trajectories against a float64 ridge fit / evaluation built here from `basis.bspline_basis`
    (pinned bit for bit to the live reference by test_oracle_golden.py) — not from the plan's fp32 projector, the
    oracle's fp32 operation sequence or any summation order the kernels share — on a sample of rows that always holds
    the first, second-tile, last-full-wave and ragged-tail rows of every launch.

`launch_plan` restates the launch arithmetic of launch_encode_tiled / launch_decode_tiled / launch_fast /
launch_dec_fast on the CPU; the table's expectations are checked against it without a GPU (at the B200's 148 SMs and
227 KB opt-in shared memory) and again with the device's own numbers before each GPU case runs.
"""
import math
import time

import numpy as np
import pytest
import torch

from conftest import rel_err
from oracle import beast_oracle as O
from beast_tokenizer_b200 import basis

TAU = 2 * math.pi
COEF_TOL = 1e-5      # coefficients vs fp64, relative to the row's largest |coefficient|
# decoded trajectories vs the fp64 evaluation of the same coefficients, same scale: a sum of at most degree_p + 1
# products whose basis weights add up to 1 is off by at most (degree_p + 2) * 2^-24 of the largest |coefficient| in fp32
# (3.6e-7 at degree 4, counting the rounding of the basis values); 1.7e-7 is the largest seen on a B200
TRAJ_TOL = 5e-7
N_RANDOM_ROWS = 500

B200_SMS = 148
B200_SMEM_OPTIN = 232448        # cudaDevAttrMaxSharedMemoryPerBlockOptin on sm_100
TILED_THREADS = 512
TILED_MAX_S = 64
BULK_COLUMNS = 7 * 32           # kEncColumns / kDecColumns
BULK_STAGES = 5
MAX_BATCH_BYTES = 6 << 30       # what one case holds on the device at once, fast and reference outputs together


# ---------------------------------------------------------------- geometries
def _cfg(num_dof, num_basis=10, seq_len=50, degree_p=4, vocab_size=256, grippers=None, llm_vocab_size=None):
    return dict(num_dof=num_dof, num_basis=num_basis, seq_len=seq_len, degree_p=degree_p, vocab_size=vocab_size,
                gripper_zero_order=bool(grippers), gripper_indices=list(grippers or []), llm_vocab_size=llm_vocab_size)


# name -> (config, expected branch summary (a subset of `branches`), kernels that must see several tiles per CTA)
GEOMETRIES = {
    # bulk-copy kernels, runtime-D instantiation <50, 10, 0>
    "bulk_d1": (_cfg(1), dict(bulk_S=224), ("bulk",)),
    "bulk_d6_v1000": (_cfg(6, vocab_size=1000), dict(bulk_S=36), ("bulk",)),
    "bulk_d16_grip_llm": (_cfg(16, grippers=[7, 15], llm_vocab_size=32000), dict(bulk_S=12), ("bulk",)),
    "bulk_d3_all_grip": (_cfg(3, grippers=[0, 1, 2]), dict(bulk_S=72, n_joint=0), ("bulk",)),
    "bulk_d32_grip_s4": (_cfg(32, grippers=[0]), dict(bulk_S=4), ("bulk",)),
    "bulk_d56_s4": (_cfg(56), dict(bulk_S=4), ("bulk",)),
    "bulk_d5_v2": (_cfg(5, vocab_size=2), dict(bulk_S=44), ("bulk",)),
    # T = 50 / nb = 10 past the bulk kernels' 224 columns: the whole batch takes the tiled kernels
    "tiled_d57_t50": (_cfg(57), dict(bulk_S=0, enc_R=4), ("enc", "dec")),
    # the reference's shipped shape: one-term sums, template rows (nb > T)
    "tiled_shipped_d32": (_cfg(32, num_basis=50, seq_len=10, degree_p=0, vocab_size=1000),
                          dict(bulk_S=None, enc_R=1, enc_p_smem=False, dec_phi_smem=False), ("enc", "dec")),
    "tiled_d9_deg1_grip": (_cfg(9, num_basis=6, seq_len=17, degree_p=1, vocab_size=64, grippers=[2, 8]),
                           dict(bulk_S=None, enc_R=4, enc_p_smem=True), ("enc", "dec")),
    # long sums, projector / basis rows staged in shared memory
    "tiled_odd_d5": (_cfg(5, num_basis=8, seq_len=33, degree_p=3, vocab_size=1000, grippers=[0]),
                     dict(bulk_S=None, enc_R=4, enc_p_smem=True, dec_phi_smem=True), ("enc", "dec")),
    "tiled_d3_nb20": (_cfg(3, num_basis=20, seq_len=64, degree_p=2, vocab_size=512),
                      dict(bulk_S=None, enc_R=4, enc_p_smem=True, dec_phi_smem=True), ("enc", "dec")),
    # tables above 32 KB: read through L1 from the plan's global copy
    "tiled_global_tables": (_cfg(4, num_basis=40, seq_len=128, degree_p=3),
                            dict(bulk_S=None, enc_R=4, enc_p_smem=False, dec_phi_smem=False), ("enc", "dec")),
    # V = 50 000 behind an LLM offset
    "tiled_v50000_llm": (_cfg(4, num_basis=12, seq_len=40, degree_p=2, vocab_size=50000, llm_vocab_size=60000),
                         dict(bulk_S=None, enc_R=4), ("enc", "dec")),
    # a trajectory just above the 108 KB two-CTA budget: S = 2 under the opt-in limit, tiles not 16-byte multiples
    "tiled_s2_t1987": (_cfg(7, seq_len=1987), dict(bulk_S=None, enc_S=2, in_bulk=0), ("enc",)),
    # 256 KB of samples per trajectory: over the opt-in limit, the one-thread-per-column encode kernel
    "generic_enc_t1000_d32": (_cfg(32, seq_len=1000), dict(bulk_S=None, enc_S=None), ()),
}


def layout(cfg):
    return O.slot_layout(cfg["num_dof"], cfg["gripper_zero_order"], cfg["gripper_indices"])


def offset(cfg):
    return 0 if cfg["llm_vocab_size"] is None else cfg["llm_vocab_size"] - cfg["vocab_size"]


# ---------------------------------------------------------------- the launch arithmetic, restated
def _up16(v):
    return (v + 15) & ~15


def _band(row):
    nz = np.flatnonzero(row != 0)
    return (int(nz[0]), int(nz[-1]) + 1) if nz.size else (0, 0)


def plan_tables(cfg):
    """What beast_plan_create derives from the fp32 host tables (csrc/plan.cu): the non-zero band of every projector
    row [k][t] and basis row [t][k], the tiled kernels' work lists and the longest bands."""
    T, D, nb = cfg["seq_len"], cfg["num_dof"], cfg["num_basis"]
    joint, grip = layout(cfg)
    c = basis.build_constants(basis.make_times(TAU, T), TAU, nb, cfg["degree_p"], joint, grip)
    pj, fj = c.proj_joint.numpy(), c.phi_joint.numpy()
    pg = c.proj_grip.numpy() if grip else np.zeros_like(pj)
    fg = c.phi_grip.numpy() if grip else np.zeros_like(fj)
    enc_bands = [[_band(p[k]) for k in range(nb)] for p in (pj, pg)]
    dec_bands = [[_band(f[t]) for t in range(T)] for f in (fj, fg)]
    used = [set(), set()]
    for s in (0, 1):
        for lo, hi in dec_bands[s]:
            used[s].update(range(lo, hi))
    nj = len(joint)
    n_enc = sum(1 for k in range(nb) for slot in range(D)
                if enc_bands[slot >= nj][k][0] < enc_bands[slot >= nj][k][1])
    n_dec = sum(1 for k in range(nb) for slot in range(D) if k in used[slot >= nj])
    return dict(T=T, D=D, nb=nb, n_joint=nj, n_enc=n_enc, n_dec=n_dec,
                enc_band_max=max(hi - lo for b in enc_bands for lo, hi in b),
                dec_band_max=max(hi - lo for b in dec_bands for lo, hi in b))


def enc_tiled(p, B, sms, optin, tokens=True, params=True, minmax=False, aligned=True):
    """launch_encode_tiled: None when it returns BEAST_E_UNSUPPORTED (the generic kernel runs instead)."""
    T, D, nb, n_enc = p["T"], p["D"], p["nb"], p["n_enc"]
    row_in, row_out = T * D, D * nb
    use_par = params or minmax
    per = 2 * row_in * 4 + (row_out * 8 if tokens else 0) + (row_out * 4 if use_par else 0)
    q_bytes = _up16(2 * row_out * 4 if minmax else (n_enc * 16 if tokens else 0))
    p_bytes = _up16(2 * T * nb * 4)
    p_smem = p_bytes <= 32 * 1024 and p["enc_band_max"] > 2
    extra = (q_bytes + _up16(n_enc * 4) + _up16(4 * nb * 4) + _up16(D * 4) + 16 + 4 * 16 +
             (p_bytes if p_smem else 0))
    budget = 108 * 1024
    if per + extra > budget:
        budget = optin
    if per + extra > budget:
        return None
    S = min(TILED_MAX_S, (budget - extra) // per)
    if S >= 4:
        S &= ~3
    y_bytes = _up16(S * row_in * 4)
    p_off = (2 * y_bytes + (_up16(S * row_out * 8) if tokens else 0) + (_up16(S * row_out * 4) if use_par else 0) +
             q_bytes + _up16(n_enc * 4) + _up16(4 * nb * 4) + _up16(D * 4) + 16)
    smem = p_off + (p_bytes if p_smem else 0)
    if smem > optin:
        return None
    per_sm = max(1, min(2048 // TILED_THREADS, (220 * 1024) // (smem + 1024)))
    n_tiles = -(-B // S)
    grid = min(n_tiles, sms * per_sm)
    return dict(kernel=f"encode_tiled_kernel<{4 if p['enc_band_max'] > 2 else 1}>", S=S, grid=grid,
                tiles_per_cta=-(-n_tiles // grid), smem=smem, p_smem=p_smem,
                in_bulk=int(aligned and (S * row_in) % 4 == 0),
                tok_bulk=int(tokens and aligned and (S * row_out) % 2 == 0),
                par_bulk=int(params and aligned and (S * row_out) % 4 == 0))


def dec_tiled(p, B, sms, optin, from_tokens=True):
    """launch_decode_tiled."""
    T, D, nb = p["T"], p["D"], p["nb"]
    row_in, row_out = D * nb, T * D
    per = row_in * 4
    phi_bytes = 2 * T * (nb | 1) * 4
    phi_smem = phi_bytes <= 32 * 1024 and p["dec_band_max"] > 2
    extra = (3 * p["n_dec"] + row_out + 4 * T + D) * 4 + 64 + (phi_bytes if phi_smem else 0)
    budget = 108 * 1024
    if per + extra > budget:
        budget = optin
    if per + extra > budget:
        return None
    S = min(TILED_MAX_S, (budget - extra) // per)
    smem = S * per + extra
    per_sm = max(1, min(2048 // TILED_THREADS, (220 * 1024) // (smem + 1024)))
    n_tiles = -(-B // S)
    grid = min(n_tiles, sms * per_sm)
    return dict(kernel=f"decode_tiled_kernel<{'true' if from_tokens else 'false'}>", S=S, grid=grid,
                tiles_per_cta=-(-n_tiles // grid), smem=smem, phi_smem=phi_smem)


def bulk_S(p):
    """S of encode_fast_kernel / decode_fast_kernel, None when the geometry is not T = 50 / nb = 10."""
    if p["T"] != 50 or p["nb"] != 10:
        return None
    S = (BULK_COLUMNS // p["D"]) & ~3
    return S if S >= 4 else 0


def launch_plan(p, B, sms, optin, call, aligned=True):
    """The launches of one C-ABI call as (kernel summary, first row, rows).  call: 'encode' (tokens + params),
    'fit' (params only), 'minmax', 'decode' (tokens -> trajectories), 'eval' (coefficients -> trajectories)."""
    out, done = [], 0
    S = bulk_S(p)
    if call in ("encode", "fit", "minmax", "decode") and aligned and S and B >= S:
        n_tiles = B // S
        grid = min(n_tiles, sms)
        name = ("encode" if call != "decode" else "decode") + f"_fast_kernel<50, 10, {p['D'] if p['D'] in (7, 14) else 0}>"
        out.append((dict(kernel=name, S=S, grid=grid, tiles_per_cta=-(-n_tiles // grid)), 0, n_tiles * S))
        done = n_tiles * S
    if done < B:
        rest = B - done
        if call in ("decode", "eval"):
            t = dec_tiled(p, rest, sms, optin, from_tokens=call == "decode")
        else:
            # a tail after the bulk kernel starts at a multiple of S rows: as aligned as the batch
            t = enc_tiled(p, rest, sms, optin, tokens=call == "encode", params=call in ("encode", "fit"),
                          minmax=call == "minmax", aligned=aligned)
        if t is None:
            t = dict(kernel="encode_generic_kernel" if call in ("encode", "fit", "minmax") else "decode_generic_kernel")
        out.append((t, done, rest))
    return out


def branches(cfg, sms=B200_SMS, optin=B200_SMEM_OPTIN):
    """The branch summary the geometry table asserts (batch-size independent)."""
    p = plan_tables(cfg)
    big = 10 ** 7
    e = enc_tiled(p, big, sms, optin)
    d = dec_tiled(p, big, sms, optin)
    return dict(bulk_S=bulk_S(p), n_joint=p["n_joint"],
                enc_R=None if e is None else int(e["kernel"][-2]), enc_S=None if e is None else e["S"],
                enc_p_smem=None if e is None else e["p_smem"], in_bulk=None if e is None else e["in_bulk"],
                dec_S=None if d is None else d["S"], dec_phi_smem=None if d is None else d["phi_smem"])


def batch_size(cfg, multi, sms, optin, universal=True):
    """A batch whose launches give every CTA of the listed kernels several tiles, with a ragged odd remainder.
    Bulk-copy: B >= 2 * 5 * sms * S + r (each CTA's five-stage ring wraps twice), r = S - 1 rows left to the tiled
    kernel.  Tiled: B >= 3 * (grid * S) of the launch that needs most rows, for every call type, and at least
    3 * 4 * sms * 64 when that fits MAX_BATCH_BYTES, plus an odd r that leaves every launch a ragged last tile."""
    p = plan_tables(cfg)
    S = bulk_S(p)
    if "bulk" in multi:
        return 2 * BULK_STAGES * sms * S + S - 1
    need = 0
    for call, kind in (("encode", "enc"), ("fit", "enc"), ("minmax", "enc"), ("decode", "dec"), ("eval", "dec")):
        if kind not in multi:
            continue
        t = launch_plan(p, 10 ** 7, sms, optin, call)[-1][0]
        need = max(need, 3 * t["grid"] * t["S"])
    # the launch-independent bound (S <= 64, grid <= 4 * sms) where the batch stays within a few GB on the device
    bound = 3 * 4 * sms * TILED_MAX_S
    row_bytes = 4 * p["T"] * p["D"] * 4 + p["D"] * p["nb"] * (2 * 8 + 3 * 4)    # 4 trajectories, 2 token + 3 coef rows
    base = max(need, 4096, bound if universal and bound * row_bytes <= MAX_BATCH_BYTES else 0)
    for r in range(1, 1000, 2):
        B = base + r
        ok = True
        for call in ("encode", "fit", "minmax", "decode", "eval"):
            t = launch_plan(p, B, sms, optin, call)[-1][0]
            if "S" in t and B % t["S"] == 0:
                ok = False
        if ok:
            return B
    raise AssertionError("no ragged batch size found")


def special_rows(p, B, sms, optin):
    """Rows 0, S-1, S, the first and last row of CTA 0's second tile, the first row of the last full wave and the
    last B mod S rows, of every launch of every call on this batch."""
    rows = set()
    for call in ("encode", "fit", "minmax", "decode", "eval"):
        for t, r0, n in launch_plan(p, B, sms, optin, call):
            if "S" not in t:
                rows.update((r0, r0 + n - 1))
                continue
            S, grid = t["S"], t["grid"]
            wave = S * grid
            cand = [0, S - 1, S, grid * S, grid * S + S - 1]
            if n // wave >= 1:
                cand.append((n // wave - 1) * wave)
            cand += list(range(n - n % S, n))
            rows.update(r0 + c for c in cand if 0 <= c < n)
    return sorted(rows)


# ---------------------------------------------------------------- the fp64 reference
def _phi64(T, nb, degree):
    return basis.bspline_basis(basis.make_times(TAU, T), TAU, nb, degree).to(torch.float64).numpy()


def _ridge64(phi):
    return np.linalg.solve(phi.T @ phi + 1e-9 * np.eye(phi.shape[1]), phi.T)


def fit64(x, cfg):
    """Coefficients [n, D*nb] '(d t)' of trajectories x [n, T, D]: the ridge solve of each spline (joints degree_p,
    grippers degree 0), in float64."""
    x = np.asarray(x, dtype=np.float64)
    T, nb = cfg["seq_len"], cfg["num_basis"]
    joint, grip = layout(cfg)
    parts = []
    for idx, deg in ((joint, cfg["degree_p"]), (grip, 0)):
        if idx:
            P = _ridge64(_phi64(T, nb, deg))                          # [nb, T]
            parts.append(np.einsum("kt,btd->bdk", P, x[..., idx]))
    return np.concatenate(parts, axis=1).reshape(x.shape[0], -1)


def eval64(coef, cfg, init_p=None):
    """Trajectories [n, T, D] of coefficients [n, D*nb] '(d t)' in float64; init_p replaces every joint's first
    coefficient.  Also returns each row's largest |coefficient| as evaluated."""
    T, nb, D = cfg["seq_len"], cfg["num_basis"], cfg["num_dof"]
    joint, grip = layout(cfg)
    c = np.asarray(coef, dtype=np.float64).reshape(-1, D, nb).copy()
    if init_p is not None:
        for s, dof in enumerate(joint):
            c[:, s, 0] = np.asarray(init_p, dtype=np.float64)[:, dof]
    out = np.zeros((c.shape[0], T, D))
    for slots, dofs, deg in ((range(len(joint)), joint, cfg["degree_p"]),
                             (range(len(joint), D), grip, 0)):
        if dofs:
            out[..., dofs] = np.einsum("tk,bsk->bts", _phi64(T, nb, deg), c[:, list(slots)])
    return out, np.abs(c).reshape(c.shape[0], -1).max(1)


def check_flips_rows(tokens, coef64, w_min, w_max, cfg):
    """Every token that differs from the exact quantiser of the fp64 coefficients must be a +-1 bin flip whose fp64
    coefficient lies within COEF_TOL of its row's largest |coefficient| from the rounding edge.  Returns the count."""
    D, nb, V = cfg["num_dof"], cfg["num_basis"], cfg["vocab_size"]
    ref = O.tokens_from_params(coef64.astype(np.float32), w_min, w_max, V, D, nb, offset(cfg))
    row_scale = np.abs(coef64).max(1)
    diff = np.argwhere(tokens != ref)
    for b, pos in diff:
        k, slot = divmod(int(pos), D)
        c = slot * nb + k
        w, lo, hi = float(coef64[b, c]), float(w_min[c]), float(w_max[c])
        assert abs(int(tokens[b, pos]) - int(ref[b, pos])) == 1, ("flip larger than one bin", int(b), int(pos))
        x = (min(max(w, lo), hi) - lo) / max(hi - lo, 1e-8) * (V - 1)
        dist = abs((x - math.floor(x)) - 0.5) * (hi - lo) / (V - 1)
        assert dist <= COEF_TOL * row_scale[b], (int(b), int(pos), dist, row_scale[b])
    return len(diff)


def test_fp64_reference_reproduces_the_golden_fits(golden_case):
    """The fp64 fit and evaluation against the live reference's outputs, before they judge a kernel."""
    name, cfg, g = golden_case
    assert np.array_equal(basis.make_times(TAU, cfg["seq_len"]).numpy(), g["times"])
    assert rel_err(fit64(g["trajs"], cfg), g["params"]) <= 1e-5
    assert rel_err(eval64(g["decode_fit"], cfg)[0], g["recon_fit"]) <= 1e-5
    assert rel_err(eval64(g["decode_fit"], cfg, g["init_p"])[0], g["recon_fit_initp"]) <= 1e-5


def test_geometry_table_reaches_the_stated_branches():
    """The restated launch arithmetic at 148 SMs / 227 KB: each row reaches the kernel and branch it is there for,
    and its batch size gives the listed kernels several tiles per CTA."""
    for name, (cfg, expect, multi) in GEOMETRIES.items():
        got = branches(cfg)
        assert {k: got[k] for k in expect} == expect, (name, got)
        B = batch_size(cfg, multi, B200_SMS, B200_SMEM_OPTIN)
        _assert_multi_tile(name, cfg, B, multi, B200_SMS, B200_SMEM_OPTIN)
    # the universal bound: S <= 64 and grid <= 4 * sms, so 3 * 4 * sms * 64 rows give any tiled launch three tiles
    p = plan_tables(GEOMETRIES["tiled_shipped_d32"][0])
    B = 3 * 4 * B200_SMS * TILED_MAX_S + 7
    for call in ("encode", "fit", "minmax", "decode", "eval"):
        assert launch_plan(p, B, B200_SMS, B200_SMEM_OPTIN, call)[-1][0]["tiles_per_cta"] >= 3


def _assert_multi_tile(name, cfg, B, multi, sms, optin):
    p = plan_tables(cfg)
    for call in ("encode", "fit", "minmax", "decode", "eval"):
        launches = launch_plan(p, B, sms, optin, call)
        kind = "enc" if call in ("encode", "fit", "minmax") else "dec"
        if "bulk" in multi and call != "eval":
            t = launches[0][0]
            assert "fast" in t["kernel"] and t["tiles_per_cta"] >= 2 * BULK_STAGES, (name, call, t)
            assert launches[-1][2] % 2 == 1 and launches[-1][0]["kernel"].startswith(kind), (name, call, launches)
        elif kind in multi:
            t = launches[-1][0]
            assert "tiled" in t["kernel"] and t["tiles_per_cta"] >= 3, (name, call, t)
            assert B % t["S"] != 0, (name, call, t)


# ---------------------------------------------------------------- GPU plumbing
def _lib():
    from beast_tokenizer_b200 import _lib as L
    return L


class _Slow:
    """The one-thread-per-column reference kernels for the duration of the block."""

    def __enter__(self):
        self.prev = _lib().load().beast_debug_disable_fast(1)

    def __exit__(self, *exc):
        _lib().load().beast_debug_disable_fast(self.prev)


def _device_limits():
    props = torch.cuda.get_device_properties(0)
    return props.multi_processor_count, int(props.shared_memory_per_block_optin)


def make_tok(cfg):
    from beast_tokenizer_b200 import BEASTBsplineTokenizer
    return BEASTBsplineTokenizer(device="cuda", **cfg)


def synth(B, cfg, seed):
    from beast_tokenizer_b200.synth import synth_device
    return synth_device(B, cfg["seq_len"], cfg["num_dof"], seed, "cuda")


def _equal(name, have, want):
    """Bit-identical on the GPU; otherwise name the rows that differ."""
    assert have.shape == want.shape and have.dtype == want.dtype, name
    if not torch.equal(have, want):
        bad = (have != want).reshape(have.shape[0], -1).any(1).nonzero().flatten()
        raise AssertionError(f"{name}: {bad.numel()} rows differ, first {bad[:8].tolist()}")


def _row_err(have, want, scale):
    """Largest |have - want| of each row over that row's scale."""
    d = np.abs(np.asarray(have, np.float64) - want).reshape(want.shape[0], -1).max(1)
    return d / np.maximum(scale, 1e-30)


def _bounds(tok):
    return tok.w_min.clone(), tok.w_max.clone()


# ---------------------------------------------------------------- the matrix
@pytest.mark.gpu
@pytest.mark.parametrize("name", list(GEOMETRIES))
def test_fast_paths_at_multi_tile_batches(name):
    """One geometry at a multi-tile batch: fast == reference kernels on every row for every entry point, fused tokens ==
    exact quantiser, bounds == column min / max, and the fp64 fit / evaluation on the boundary rows of every launch."""
    cfg, expect, multi = GEOMETRIES[name]
    sms, optin = _device_limits()
    got = branches(cfg, sms, optin)
    assert {k: got[k] for k in expect} == expect, (name, got)
    B = batch_size(cfg, multi, sms, optin)
    _assert_multi_tile(name, cfg, B, multi, sms, optin)
    p = plan_tables(cfg)
    t0 = time.perf_counter()
    torch.cuda.reset_peak_memory_stats()
    L = _lib()
    lib = L.load()
    off = offset(cfg)
    tok = make_tok(cfg)
    x = synth(B, cfg, seed=1000 + B)
    ip = x[:, 0, :].contiguous()

    # bounds: fused min / max == min / max of the coefficients, fast == reference, twice on different data
    params_f = tok.compute_weights(x)
    with _Slow():
        _equal("compute_weights", params_f, tok.compute_weights(x))
    x2 = synth(B - 2, cfg, seed=2000 + B)
    params2 = tok.compute_weights(x2)
    for data, par in ((x2, params2), (x, params_f)):
        tok.update_weights_bounds(data)
        lo, hi = _bounds(tok)
        assert torch.equal(lo, par.amin(0)) and torch.equal(hi, par.amax(0)), "update_weights_bounds"
        with _Slow():
            tok.update_weights_bounds(data)
        _equal("w_min", lo[None], tok.w_min[None])
        _equal("w_max", hi[None], tok.w_max[None])
    del x2
    # accumulate = 1 onto existing bounds, ragged batch
    Br = B - 3
    acc_lo, acc_hi = params2.amin(0).contiguous(), params2.amax(0).contiguous()
    plan = tok._plan()
    ws = plan.minmax_workspace()
    L.check(lib.beast_fit_minmax_ws_f32(plan.handle, L.ptr(x), Br, L.ptr(acc_lo), L.ptr(acc_hi), 1, L.ptr(ws),
                                        ws.numel() * 4, L.stream_ptr(x.device)), "beast_fit_minmax_ws_f32")
    assert torch.equal(acc_lo, torch.minimum(params2.amin(0), params_f[:Br].amin(0)))
    assert torch.equal(acc_hi, torch.maximum(params2.amax(0), params_f[:Br].amax(0)))
    del params2
    lo, hi = tok.w_min.clone(), tok.w_max.clone()         # bounds of x, as update_weights_bounds left them

    # encode: fast == reference, tokens == exact quantiser of the kernel's own coefficients
    tokens, pd = tok.encode(x)
    assert torch.equal(pd["params"], params_f)
    with _Slow():
        t_s, pd_s = tok.encode(x)
    _equal("tokens", tokens, t_s)
    _equal("params", pd["params"], pd_s["params"])
    del t_s, pd_s
    params_f = pd["params"]                              # the same bits: one copy
    assert torch.equal(tokens, tok._quantize(params_f, off)), "fused tokens != exact quantiser"

    # decode, with and without init_p
    rec = tok.reconstruct_traj(tokens)
    with _Slow():
        _equal("reconstruct_traj", rec, tok.reconstruct_traj(tokens))
    rec_i = tok.reconstruct_traj(tokens, init_p=ip)
    with _Slow():
        _equal("reconstruct_traj(init_p)", rec_i, tok.reconstruct_traj(tokens, init_p=ip))

    # fp64 on a row sample that holds every launch's boundary rows
    rng = np.random.default_rng(B)
    rows = sorted(set(special_rows(p, B, sms, optin)) | set(rng.choice(B, size=min(B, N_RANDOM_ROWS), replace=False).tolist()))
    ridx = torch.as_tensor(rows, device=x.device)
    xs = x[ridx].cpu().numpy()
    w64 = fit64(xs, cfg)
    par_s = params_f[ridx].cpu().numpy()
    coef_err = _row_err(par_s, w64, np.abs(w64).max(1))
    assert coef_err.max() <= COEF_TOL, ("coefficients", rows[int(coef_err.argmax())], float(coef_err.max()))
    lo_n, hi_n = lo.cpu().numpy(), hi.cpu().numpy()
    tk_s = tokens[ridx].cpu().numpy()
    n_flips = check_flips_rows(tk_s, w64, lo_n, hi_n, cfg)
    dec = O.decode(tk_s, lo_n, hi_n, cfg["vocab_size"], cfg["num_dof"], cfg["num_basis"], off)
    r64, scale = eval64(dec, cfg)
    traj_err = _row_err(rec[ridx].cpu().numpy(), r64, scale)
    assert traj_err.max() <= TRAJ_TOL, ("trajectories", rows[int(traj_err.argmax())], float(traj_err.max()))
    r64i, scale_i = eval64(dec, cfg, xs[:, 0, :])
    traj_err_i = _row_err(rec_i[ridx].cpu().numpy(), r64i, scale_i)
    assert traj_err_i.max() <= TRAJ_TOL, ("trajectories(init_p)", rows[int(traj_err_i.argmax())],
                                         float(traj_err_i.max()))
    del tokens, pd, params_f, rec, rec_i

    # continuous variants
    cont, _ = tok.encode_continuous(x)
    with _Slow():
        _equal("encode_continuous", cont, tok.encode_continuous(x)[0])
    rec_c = tok.reconstruct_traj_continuous(cont)
    with _Slow():
        _equal("reconstruct_traj_continuous", rec_c, tok.reconstruct_traj_continuous(cont))
    rec_ci = tok.reconstruct_traj_continuous(cont, init_p=ip)
    with _Slow():
        _equal("reconstruct_traj_continuous(init_p)", rec_ci, tok.reconstruct_traj_continuous(cont, init_p=ip))
    torch.cuda.synchronize()
    launches = {c: [t for t, _, _ in launch_plan(p, B, sms, optin, c)] for c in ("encode", "decode", "eval")}
    print(f"\n{name}: B={B} rows_checked={len(rows)} coef_err={coef_err.max():.2e} traj_err={traj_err.max():.2e} "
          f"traj_err_init_p={traj_err_i.max():.2e} flips={n_flips}/{tk_s.size} "
          f"peak_mem={torch.cuda.max_memory_allocated() / 2 ** 30:.2f}GiB wall={time.perf_counter() - t0:.1f}s "
          f"launches={launches}")


# ---------------------------------------------------------------- views and output windows
@pytest.mark.gpu
def test_public_api_unaligned_views_equal_aligned_calls():
    """Offset views reach the kernels without a copy and take the hand-loaded paths; results equal the aligned call
    bit for bit."""
    sms, _ = _device_limits()
    # rows of 660 B (odd_d5): buf[1:] starts 4 mod 16, every tile of the tiled encode is loaded by hand
    cfg = GEOMETRIES["tiled_odd_d5"][0]
    tok = make_tok(cfg)
    B = 3 * 2 * sms * 64 + 5
    buf = synth(B + 1, cfg, seed=11)
    assert buf[1:].data_ptr() % 16 == 4
    tok.update_weights_bounds(buf[1:].clone())
    t_al, p_al = tok.encode(buf[1:].clone())
    t_un, p_un = tok.encode(buf[1:])
    _equal("odd_d5 encode(buf[1:]) tokens", t_un, t_al)
    _equal("odd_d5 encode(buf[1:]) params", p_un["params"], p_al["params"])

    # T = 50 / nb = 10 samples one float into a flat buffer: the bulk-copy encode is refused, the tiled one loads by hand
    cfg = GEOMETRIES["bulk_d6_v1000"][0]
    D, n = cfg["num_dof"], cfg["num_dof"] * cfg["num_basis"]
    tok = make_tok(cfg)
    B = 2 * BULK_STAGES * sms * 36 + 35
    x = synth(B, cfg, seed=12)
    flat = torch.empty(B * 50 * D + 1, device="cuda")
    xv = flat[1:].view(B, 50, D)
    xv.copy_(x)
    assert xv.data_ptr() % 16 == 4
    tok.update_weights_bounds(x)
    lo, hi = _bounds(tok)
    tok.update_weights_bounds(xv)
    _equal("w_min (offset samples)", tok.w_min[None], lo[None])
    _equal("w_max (offset samples)", tok.w_max[None], hi[None])
    tokens, pd = tok.encode(x)
    t_v, pd_v = tok.encode(xv)
    _equal("encode(offset samples) tokens", t_v, tokens)
    _equal("encode(offset samples) params", pd_v["params"], pd["params"])
    cont = tok.encode_continuous(x)[0]
    _equal("encode_continuous(offset samples)", tok.encode_continuous(xv)[0], cont)
    # tokens one int64 into a flat buffer: the bulk-copy decode is refused (rows of 80 * D bytes keep tokbuf[1:] aligned)
    tflat = torch.empty(B * n + 1, dtype=torch.int64, device="cuda")
    tv = tflat[1:].view(B, n)
    tv.copy_(tokens)
    assert tv.data_ptr() % 16 == 8
    rec = tok.reconstruct_traj(tokens)
    _equal("reconstruct_traj(offset tokens)", tok.reconstruct_traj(tv), rec)
    # init_p one float into a flat buffer
    ip = x[:, 0, :].contiguous()
    ipf = torch.empty(B * D + 1, device="cuda")
    ipv = ipf[1:].view(B, D)
    ipv.copy_(ip)
    rec_i = tok.reconstruct_traj(tokens, init_p=ip)
    _equal("reconstruct_traj(offset init_p)", tok.reconstruct_traj(tokens, init_p=ipv), rec_i)
    _equal("reconstruct_traj(offset tokens, offset init_p)", tok.reconstruct_traj(tv, init_p=ipv), rec_i)
    # normalised coefficients one float into a flat buffer
    cf = torch.empty(B * n + 1, device="cuda")
    cv = cf[1:].view(B, n)
    cv.copy_(cont)
    _equal("reconstruct_traj_continuous(offset)", tok.reconstruct_traj_continuous(cv, init_p=ipv),
           tok.reconstruct_traj_continuous(cont, init_p=ip))

    # D * nb odd: token rows of 504 B, tokbuf[1:] starts 8 mod 16
    cfg = _cfg(3, num_basis=21, seq_len=30, degree_p=3)
    tok = make_tok(cfg)
    B = 3 * 2 * sms * 64 + 3
    x = synth(B + 1, cfg, seed=13)
    tok.update_weights_bounds(x)
    tokbuf = tok.encode(x)[0]
    assert tokbuf[1:].data_ptr() % 16 == 8
    _equal("reconstruct_traj(tokbuf[1:])", tok.reconstruct_traj(tokbuf[1:]), tok.reconstruct_traj(tokbuf[1:].clone()))
    ip = x[1:, 0, :].contiguous()
    _equal("reconstruct_traj(tokbuf[1:], init_p)", tok.reconstruct_traj(tokbuf[1:], init_p=x[1:, 0, :]),
           tok.reconstruct_traj(tokbuf[1:].clone(), init_p=ip))


SENT_F32 = 0x7FA5A5A5          # a NaN payload no kernel produces from finite data
SENT_I64 = 0x5A5A5A5A5A5A5A5A
GUARD = 512


def _guarded(n, dtype, shift):
    """(buffer, n-element window at GUARD + shift elements) with every element of the buffer set to a sentinel."""
    buf = torch.empty(n + 2 * GUARD + 1, dtype=dtype, device="cuda")
    if dtype == torch.float32:
        buf.view(torch.int32).fill_(SENT_F32)
    else:
        buf.fill_(SENT_I64)
    return buf, buf[GUARD + shift:GUARD + shift + n]


def _guards_intact(name, buf, n, shift):
    bits = buf.view(torch.int32) if buf.dtype == torch.float32 else buf
    sent = SENT_F32 if buf.dtype == torch.float32 else SENT_I64
    lo, hi = bits[:GUARD + shift], bits[GUARD + shift + n:]
    assert bool((lo == sent).all()) and bool((hi == sent).all()), f"{name}: a store left the output window"


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["bulk_d6_v1000", "bulk_d3_all_grip", "tiled_shipped_d32", "tiled_odd_d5"])
def test_c_abi_unaligned_outputs_and_guard_bands(name):
    """tokens_out at +8 B, params_out / traj_out at +4 B inside sentinel-filled buffers: the outputs equal the aligned
    call's, and no launch — bulk-copy, tiled with bulk stores, tiled with hand stores — writes outside its window."""
    cfg, _, multi = GEOMETRIES[name]
    sms, optin = _device_limits()
    L = _lib()
    tok = make_tok(cfg)
    plan = tok._plan()
    lib, h = plan._lib, plan.handle
    D, nb, T = cfg["num_dof"], cfg["num_basis"], cfg["seq_len"]
    B = batch_size(cfg, multi, sms, optin, universal=False)
    x = synth(B, cfg, seed=21)
    tok.update_weights_bounds(x)
    lo, hi = _bounds(tok)
    off = offset(cfg)
    st = L.stream_ptr(x.device)
    ip = x[:, 0, :].contiguous()
    res = {}
    for shift_t, shift_p in ((0, 0), (1, 1)):
        tb, tw = _guarded(B * D * nb, torch.int64, shift_t)
        pb, pw = _guarded(B * D * nb, torch.float32, shift_p)
        L.check(lib.beast_encode_f32(h, L.ptr(x), B, L.ptr(lo), L.ptr(hi), off, L.ptr(pw), L.ptr(tw), st), "encode")
        _guards_intact(f"encode tokens_out +{8 * shift_t} B", tb, B * D * nb, shift_t)
        _guards_intact(f"encode params_out +{4 * shift_p} B", pb, B * D * nb, shift_p)
        rb, rw = _guarded(B * T * D, torch.float32, shift_p)
        L.check(lib.beast_decode_f32(h, L.ptr(tw), B, L.ptr(lo), L.ptr(hi), off, None, L.ptr(rw), st), "decode")
        _guards_intact(f"decode traj_out +{4 * shift_p} B", rb, B * T * D, shift_p)
        ib, iw = _guarded(B * T * D, torch.float32, shift_p)
        L.check(lib.beast_decode_f32(h, L.ptr(tw), B, L.ptr(lo), L.ptr(hi), off, L.ptr(ip), L.ptr(iw), st),
                "decode init_p")
        _guards_intact(f"decode(init_p) traj_out +{4 * shift_p} B", ib, B * T * D, shift_p)
        eb, ew = _guarded(B * T * D, torch.float32, shift_p)
        L.check(lib.beast_eval_f32(h, L.ptr(pw), B, L.ptr(ip), None, 0, L.ptr(ew), st), "eval")
        _guards_intact(f"eval traj_out +{4 * shift_p} B", eb, B * T * D, shift_p)
        res[shift_t] = [w.clone() for w in (tw, pw, rw, iw, ew)]
        del tb, pb, rb, ib, eb
    for what, a, u in zip(("tokens", "params", "traj", "traj(init_p)", "eval"), res[0], res[1]):
        _equal(f"{name} {what} unaligned vs aligned", u.view(B, -1), a.view(B, -1))
    assert torch.equal(res[0][0].view(B, -1), tok.encode(x)[0])
