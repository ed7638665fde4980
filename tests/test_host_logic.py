"""CPU-only checks: host-side constants, the Python API surface that needs no GPU, the on-disk
format, and that the C-ABI library loads and exports every declared symbol."""
import ctypes
import json
import math
import os
import re

import numpy as np
import pytest
import torch

from conftest import GOLDEN, GOLDEN_CASES, ROOT, load_golden, rel_err


def test_host_constants_match_reference_basis(golden_case):
    from beast_tokenizer_b200.basis import build_constants, make_times
    from oracle import beast_oracle as O
    name, cfg, g = golden_case
    joint, grip = O.slot_layout(cfg["num_dof"], cfg["gripper_zero_order"], cfg["gripper_indices"])
    times = make_times(2 * math.pi, cfg["seq_len"])
    c = build_constants(times, 2 * math.pi, cfg["num_basis"], cfg["degree_p"], joint, grip)
    assert np.array_equal(c.times.numpy(), g["times"])
    assert np.array_equal(c.phi_joint.numpy(), g["phi_joint"])          # bit-identical to mp.basis_gn.basis
    assert np.array_equal(c.knots_joint.numpy(), g["knots_joint"])
    if grip:
        assert np.array_equal(c.phi_grip.numpy(), g["phi_grip"])
    assert c.slot_to_dof == joint + grip
    # the projector reproduces the reference's coefficients within the 1e-5 tolerance
    x = torch.from_numpy(g["trajs"])
    w = torch.einsum("kt,btd->bdk", c.proj_joint, x[..., joint]).reshape(x.shape[0], -1)
    if grip:
        wg = torch.einsum("kt,btd->bdk", c.proj_grip, x[..., grip]).reshape(x.shape[0], -1)
        w = torch.cat([w, wg], 1)
    err = np.abs(w.numpy() - g["params"]).max() / np.abs(g["params"]).max()
    assert err <= 1e-5


def test_library_exports_every_declared_symbol():
    from beast_tokenizer_b200 import _lib
    header = open(os.path.join(ROOT, "include", "beast_b200.h")).read()
    declared = set(re.findall(r"\b(beast_[a-z0-9_]+)\s*\(", header))
    declared |= set(re.findall(r"\b(bpe_[a-z0-9_]+)\s*\(", header))
    lib = _lib.load()
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} declared in include/beast_b200.h but not exported"
    assert declared == set(_lib.exported_symbols())
    assert b"sm_100a" in lib.beast_version()
    assert lib.beast_launch_count() == 0 or lib.beast_launch_count() > 0
    # argument validation needs no GPU
    assert lib.beast_plan_create(None, None) == -1
    assert lib.beast_minmax_f32(None, 0, 0, None, None, 0, None) == -1


def test_no_cpu_fallback():
    from beast_tokenizer_b200 import BEASTBsplineTokenizer, BeastB200Error
    tok = BEASTBsplineTokenizer(num_dof=7, device="cpu")
    with pytest.raises(BeastB200Error):
        tok.encode(torch.zeros(2, 50, 7))
    with pytest.raises(BeastB200Error):
        tok.reconstruct_traj(torch.zeros(2, 70, dtype=torch.long))
    if not torch.cuda.is_available():
        tok = BEASTBsplineTokenizer(num_dof=7, device="cuda")
        with pytest.raises(BeastB200Error):
            tok.compute_weights(torch.zeros(2, 50, 7))


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "beast_tokenizer_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in src.replace("oracle's", ""), f"{f} mentions the oracle"


def test_llm_vocab_size_api():
    from beast_tokenizer_b200 import BEASTBsplineTokenizer
    tok = BEASTBsplineTokenizer(num_dof=14, gripper_zero_order=True, gripper_indices=[13, 6], device="cpu")
    assert tok.joint_indices == [0, 1, 2, 3, 4, 5, 7, 8, 9, 10, 11, 12] and tok.gripper_indices == [6, 13]
    assert tok.joint_dof == 12 and tok.gripper_dof == 2 and tok.num_dof == 14
    with pytest.raises(ValueError, match="LLM vocab size is not set"):
        tok.tokens_to_llm_tokens(torch.zeros(1, 140, dtype=torch.long))
    with pytest.raises(ValueError):
        tok.llm_tokens_to_mp_tokens(torch.zeros(1, 140, dtype=torch.long))
    with pytest.raises(TypeError):
        tok.set_llm_vocab_size(3.5)
    with pytest.raises(ValueError):
        tok.set_llm_vocab_size(100)
    tok.set_llm_vocab_size(32000)
    assert tok._llm_vocab_offset() == 31744 and tok.get_config()["llm_vocab_size"] == 32000
    t = torch.arange(280).reshape(2, 140)
    assert torch.equal(tok.tokens_to_llm_tokens(t.reshape(2, 10, 14)), t + 31744)
    assert tok.llm_tokens_to_mp_tokens(t + 31744).shape == (2, 10, 14)
    tok.update_vlm_vocab_size(None)
    assert tok.llm_vocab_size is None and "llm_vocab_size" not in tok._config
    # gripper_indices are ignored unless gripper_zero_order (SURVEY.md trap 3)
    tok = BEASTBsplineTokenizer(num_dof=7, gripper_indices=[6], device="cpu")
    assert tok.gripper_indices == [] and tok.joint_dof == 7 and tok._config["gripper_indices"] == []


@pytest.mark.parametrize("name", sorted(GOLDEN_CASES))
def test_checkpoint_format_round_trip(name, tmp_path):
    """Reads the reference's save_pretrained output and writes byte-identical JSON back."""
    from beast_tokenizer_b200 import BEASTBsplineTokenizer
    ref_dir = os.path.join(GOLDEN, f"{name}_pretrained")
    tok = BEASTBsplineTokenizer.from_pretrained(ref_dir, device="cpu")
    g = load_golden(name)
    assert np.array_equal(tok.w_min.numpy(), g["w_min_fit"]) and np.array_equal(tok.w_max.numpy(), g["w_max_fit"])
    tok.save_pretrained(tmp_path)
    ours = json.load(open(tmp_path / "beast_tokenizer_config.json"))
    theirs = json.load(open(os.path.join(ref_dir, "beast_tokenizer_config.json")))
    assert ours == theirs
    assert open(tmp_path / "beast_tokenizer_config.json").read() == \
        open(os.path.join(ref_dir, "beast_tokenizer_config.json")).read()
    sd = tok.state_dict()
    assert set(sd) == {"config", "w_min", "w_max", "llm_vocab_size"}
    tok2 = BEASTBsplineTokenizer(**{k: v for k, v in sd["config"].items() if k not in ("tokenizer_type",)})
    tok2.load_state_dict(sd)
    assert torch.equal(tok2.w_min, tok.w_min) and tok2.llm_vocab_size == tok.llm_vocab_size


def test_from_pretrained_errors(tmp_path):
    from beast_tokenizer_b200 import BEASTBsplineTokenizer
    with pytest.raises(FileNotFoundError):
        BEASTBsplineTokenizer.from_pretrained(tmp_path / "nope")
    d = tmp_path / "bad"
    d.mkdir()
    json.dump({"config": {"tokenizer_type": "something_else"}}, open(d / "beast_tokenizer_config.json", "w"))
    with pytest.raises(ValueError):
        BEASTBsplineTokenizer.from_pretrained(d)


def test_utils_match_oracle():
    from beast_tokenizer_b200 import utils as U
    from oracle import beast_oracle as O
    rng = np.random.default_rng(0)
    x = rng.normal(0, 0.03, (64, 40)).astype(np.float32)
    lo = (-0.02 - rng.random(40) * 0.01).astype(np.float32)
    hi = (0.02 + rng.random(40) * 0.01).astype(np.float32)
    tx, tlo, thi = torch.from_numpy(x), torch.from_numpy(lo), torch.from_numpy(hi)
    q = U.continuous_to_discrete(torch.clamp(tx, tlo, thi), tlo, thi, 256).numpy()
    assert np.array_equal(q, O.continuous_to_discrete(np.clip(x, lo, hi), lo, hi, 256))
    assert np.array_equal(U.discrete_to_continuous(torch.from_numpy(q), tlo, thi, 256).numpy(),
                          O.discrete_to_continuous(q, lo, hi, 256))
    n = U.normalize_tensor(tx, tlo, thi).numpy()
    assert np.array_equal(n, O.normalize_tensor(x, lo, hi))
    assert np.array_equal(U.denormalize_tensor(torch.from_numpy(n), tlo, thi).numpy(), O.denormalize_tensor(n, lo, hi))


def test_synth_is_deterministic():
    from beast_tokenizer_b200.synth import synth, SyntheticLoader
    a, b = synth(4, 50, 14, 3), synth(4, 50, 14, 3)
    assert torch.equal(a, b) and a.dtype == torch.float32 and a.shape == (4, 50, 14)
    g = load_golden("cfg2_d14")
    assert np.array_equal(synth(96, 50, 14, 2).numpy(), g["trajs"])
    batches = list(SyntheticLoader(2, 32, 50, 14, seed0=1))
    assert len(batches) == 2 and batches[0]["actions"].shape == (32, 50, 14)


COND_CASES = {
    "cond_orders": dict(num_dof=14, num_basis=10, seq_len=50, degree_p=4, gripper_indices=[6, 13]),
    "cond_odd": dict(num_dof=5, num_basis=8, seq_len=33, degree_p=3, gripper_indices=[0]),
}


@pytest.mark.parametrize("case,orders", [("cond_orders", o) for o in [(1, 0), (2, 0), (0, 1), (0, 2), (1, 1), (2, 2)]] +
                         [("cond_odd", o) for o in [(2, 1), (1, 2)]])
def test_conditioned_projector_matches_reference(case, orders):
    """Non-zero init/end condition orders stay one linear map per joint: w = P_eff . y with the
    boundary terms folded in (basis.conditioned_projector) reproduces the reference's coefficients."""
    import torch
    from beast_tokenizer_b200.basis import build_constants, make_times
    io, eo = orders
    cfg = COND_CASES[case]
    g = load_golden(case)
    k = f"o{io}{eo}_"
    D, nb, T, p = cfg["num_dof"], cfg["num_basis"], cfg["seq_len"], cfg["degree_p"]
    grip = cfg["gripper_indices"]
    joint = [i for i in range(D) if i not in grip]
    c = build_constants(make_times(2 * math.pi, T), 2 * math.pi, nb, p, joint, grip, io, eo)
    assert np.array_equal(c.phi_joint.numpy(), g[k + "phi_joint"])
    assert np.array_equal(c.knots_joint.numpy(), g[k + "knots_joint"])
    assert tuple(c.proj_joint.shape) == (nb, T)
    x = torch.from_numpy(g["trajs"]).double()
    w = torch.einsum("kt,btd->bdk", c.proj_joint.double(), x[..., joint]).reshape(x.shape[0], -1).numpy()
    assert rel_err(w, g[k + "params"][:, :len(joint) * nb]) <= 1e-5


def test_condition_order_ctor_errors():
    from beast_tokenizer_b200 import BEASTBsplineTokenizer
    with pytest.raises(NotImplementedError):
        BEASTBsplineTokenizer(num_dof=2, end_cond_order=-1, device="cpu")
    with pytest.raises(NotImplementedError):
        BEASTBsplineTokenizer(num_dof=2, init_cond_order=3, device="cpu")
    tok = BEASTBsplineTokenizer(num_dof=2, init_cond_order=2, end_cond_order=1, device="cpu")
    assert tok._config["init_cond_order"] == 2 and tok._config["end_cond_order"] == 1


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (the CPU arm the driver runs beside ours) prints one JSON line with the
    contract's keys; it needs no GPU."""
    import subprocess
    import sys
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "1", "--no-bpe"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
                "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["impl"] == "reference" and line["value"] > 0 and line["unit"] == "trajectories/s"
    assert line["cpu_baseline"]["kind"] in ("port", "reference") and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in line["config"]


def test_bench_dump_outputs_writes_a_fixed_sample(tmp_path):
    """`bench.py --dump-outputs DIR`: float32 / float64 .npy files of at most 64 MB in all, the same seeded rows of
    every output on every run, every row of a small batch; out-of-range --steps and the reference arm are refused."""
    import importlib.util
    import subprocess
    import sys
    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    names = {"encode_tokens.npy", "encode_params.npy", "decode_trajectories.npy"}

    def dump(n, d):
        row = torch.arange(n, dtype=torch.int64)                   # every value of a row holds the row index
        bench.dump_outputs(str(d), row[:, None].repeat(1, 140) + 31744, row[:, None].repeat(1, 140).float(),
                           row[:, None, None].repeat(1, 50, 14).float())
        assert set(os.listdir(d)) == names
        out = {f[:-4]: np.load(d / f) for f in names}
        assert all(a.dtype in (np.float32, np.float64) for a in out.values())
        assert sum(os.path.getsize(d / f) for f in names) <= 64 << 20
        rows = out["encode_tokens"][:, 0] - 31744
        assert np.array_equal(out["encode_params"][:, 0], rows) and np.array_equal(out["decode_trajectories"][:, 0, 0], rows)
        return rows

    n = bench.DUMP_ROWS + 4099
    a, b = dump(n, tmp_path / "a"), dump(n, tmp_path / "b")
    assert a.shape == (bench.DUMP_ROWS,) and np.array_equal(a, b) and np.all(np.diff(a) > 0) and a[-1] < n
    assert np.array_equal(dump(300, tmp_path / "small"), np.arange(300))
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path / "ref")]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True,
                             timeout=120, cwd=ROOT)
        assert out.returncode == 2 and "error" in out.stderr, out.stderr[-2000:]
    assert not os.path.exists(tmp_path / "ref")


def test_fit_parameters_gathers_small_batches():
    """fit_parameters fits the loader's small batches ~4 096 trajectories at a time (host logic only: the fit and
    the quantile select are stubbed)."""
    from beast_tokenizer_b200 import BEASTBsplineTokenizer
    tok = BEASTBsplineTokenizer(num_dof=3, num_basis=4, seq_len=10, vocab_size=16, device="cpu")
    calls = []
    tok._cuda = lambda: torch.device("cpu")

    def fake_fit(x):
        calls.append(tuple(x.shape))
        return x.reshape(x.shape[0], -1)[:, :12].float()

    tok.compute_weights = fake_fit
    tok._column_quantiles = lambda p, qs: (p.min(0).values, p.max(0).values)
    batches = [{"actions": torch.randn(32, 10, 5)} for _ in range(300)]
    tok.fit_parameters(batches, verbose=False)
    assert calls == [(4096, 10, 3), (4096, 10, 3), (1408, 10, 3)]
    want_lo = torch.cat([b["actions"][..., :3] for b in batches]).reshape(9600, -1)[:, :12].min(0).values
    assert torch.equal(tok.w_min, want_lo)
    calls.clear()
    tok.fit_parameters(batches, max_samples=5, verbose=False)
    assert calls == [(160, 10, 3)]
    calls.clear()
    odd = [{"actions": torch.randn(32, 10, 5)}, {"actions": torch.randn(4, 7, 5)}, {"actions": torch.randn(8, 10, 5)}]
    tok.fit_parameters(odd, verbose=False)                       # an odd-shaped batch is passed through on its own
    assert calls == [(32, 10, 3), (4, 7, 3), (8, 10, 3)]
    calls.clear()
    tok.fit_parameters(batches, max_samples=0, verbose=False)    # the reference's loop fits one batch before it checks
    assert calls == [(32, 10, 3)]
    calls.clear()
    grow = [{"actions": torch.randn(8, 10, 3)}] + [{"actions": torch.randn(3000, 10, 3)} for _ in range(9)]
    tok.fit_parameters(grow, verbose=False)                      # later batches far larger than the first: bounded blocks
    assert calls == [(6008, 10, 3), (6000, 10, 3), (6000, 10, 3), (6000, 10, 3), (3000, 10, 3)]
    want_hi = torch.cat([b["actions"] for b in grow]).reshape(27008, -1)[:, :12].max(0).values
    assert torch.equal(tok.w_max, want_hi)
    calls.clear()
    mixed = [{"actions": torch.randn(16, 10, 3)}, {"actions": torch.randn(16, 10, 3).double()},
             {"actions": torch.randn(16, 10, 3).numpy()}]
    tok.compute_weights = lambda x: fake_fit(torch.as_tensor(x))
    tok.fit_parameters(mixed, verbose=False)                     # a numpy batch in the block: batch by batch, in order
    assert calls == [(16, 10, 3)] * 3
    calls.clear()
    tok.fit_parameters(mixed[:2], verbose=False)                 # a change of dtype starts a new block
    assert calls == [(16, 10, 3), (16, 10, 3)]
    with pytest.raises(KeyError):
        tok.fit_parameters([{"x": 1}], verbose=False)
    with pytest.raises(KeyError):
        tok.fit_parameters(batches[:3] + [{"x": 1}], verbose=False)
    with pytest.raises(RuntimeError):
        tok.fit_parameters([], verbose=False)


def test_tiled_kernel_work_lists_are_exact_shortcuts():
    """The tiled kernels (csrc/spline_tiled.cu, lists built by csrc/plan.cu) recompute only the token positions whose
    projector row is not empty and load only the tokens whose coefficient some basis row reads.  Restated on the host
    tables: (a) band sums equal full sums bit for bit (the skipped terms are exact zeros, t / k ascending FMA order),
    (b) an empty projector row gives coefficient +0.0 for any trajectory, (c) a coefficient outside every basis band
    cannot change a trajectory sample.  Geometries: the reference's shipped shape (train.sh) and a cubic one."""
    from beast_tokenizer_b200.basis import build_constants, make_times
    rng = np.random.default_rng(3)
    for T, nb, deg in ((10, 50, 0), (33, 8, 3), (64, 20, 2)):
        c = build_constants(make_times(2 * math.pi, T), 2 * math.pi, nb, deg, list(range(3)), [])
        P, Phi = c.proj_joint.numpy(), c.phi_joint.numpy()          # [nb, T], [T, nb]
        assert P.dtype == np.float32 and Phi.dtype == np.float32

        def band(row):
            nz = np.nonzero(row)[0]
            return (0, 0) if nz.size == 0 else (int(nz[0]), int(nz[-1]) + 1)

        def fma_sum(coef, vals, lo, hi):                            # fp32 FMA chain, ascending index
            acc = np.float32(0.0)
            for i in range(lo, hi):
                acc = np.float32(np.float64(coef[i]) * np.float64(vals[i]) + np.float64(acc))   # one rounding: an FMA
            return acc

        y = rng.standard_normal(T).astype(np.float32)
        w = rng.standard_normal(nb).astype(np.float32)
        used = np.zeros(nb, bool)
        for t in range(T):
            lo, hi = band(Phi[t])
            used[lo:hi] = True
            assert fma_sum(Phi[t], w, lo, hi).tobytes() == fma_sum(Phi[t], w, 0, nb).tobytes()
        n_empty = 0
        for k in range(nb):
            lo, hi = band(P[k])
            full = fma_sum(P[k], y, 0, T)
            assert fma_sum(P[k], y, lo, hi).tobytes() == full.tobytes()
            if lo == hi:
                n_empty += 1
                assert full.tobytes() == np.float32(0.0).tobytes()   # +0.0: the token is a per-column constant
        # (c): garbage in the coefficients no basis row reads leaves every sample unchanged
        w2 = w.copy()
        w2[~used] = 1e30
        for t in range(T):
            lo, hi = band(Phi[t])
            assert fma_sum(Phi[t], w2, lo, hi).tobytes() == fma_sum(Phi[t], w, lo, hi).tobytes()
        if (T, nb, deg) == (10, 50, 0):
            assert n_empty == 40 and int(used.sum()) == 10           # one token in five is recomputed / loaded
        else:
            assert n_empty == 0 and used.all()
