"""ctypes binding of libbeast_b200.so (the C ABI declared in include/beast_b200.h).

There is no CPU fallback: if the library cannot be loaded, or no CUDA device is present,
every compute entry point raises.  torch is used only for device memory and streams.
"""
import ctypes as C
import os
import threading

import torch

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "libbeast_b200.so")

_lib = None
_lock = threading.Lock()

c_f32p = C.c_void_p     # device pointers travel as integers
c_i64p = C.c_void_p


class BeastB200Error(RuntimeError):
    pass


class PlanDesc(C.Structure):
    _fields_ = [
        ("seq_len", C.c_int32), ("num_dof", C.c_int32), ("num_basis", C.c_int32), ("n_joint", C.c_int32),
        ("degree_p", C.c_int32), ("vocab_size", C.c_int32), ("tau", C.c_float),
        ("slot_to_dof_h", C.POINTER(C.c_int32)),
        ("proj_joint_h", C.POINTER(C.c_float)), ("proj_grip_h", C.POINTER(C.c_float)),
        ("phi_joint_h", C.POINTER(C.c_float)), ("phi_grip_h", C.POINTER(C.c_float)),
        ("knots_joint_h", C.POINTER(C.c_float)), ("knots_grip_h", C.POINTER(C.c_float)),
        ("init_cond_order", C.c_int32), ("end_cond_order", C.c_int32),
    ]


class GridDesc(C.Structure):
    """beast_grid_desc_t: one shared time grid and its basis rows of orders 0..max_order (host pointers)."""
    _fields_ = [
        ("n_times", C.c_int32), ("max_order", C.c_int32), ("times_h", C.POINTER(C.c_float)),
        ("rows_joint_h", C.POINTER(C.c_float)), ("rows_grip_h", C.POINTER(C.c_float)),
    ]


BPE_MAX_PEERS = 16


class BpePeers(C.Structure):
    """bpe_peers_t (include/beast_b200.h): the ranks' delta blocks / flag arrays as device pointers."""
    _fields_ = [("world", C.c_int32), ("rank", C.c_int32), ("grid_blocks", C.c_int32), ("epoch_base", C.c_int32),
                ("delta", C.c_void_p * BPE_MAX_PEERS), ("flags", C.c_void_p * BPE_MAX_PEERS)]


_SIGNATURES = {
    "beast_plan_create": (C.c_int, [C.POINTER(PlanDesc), C.POINTER(C.c_void_p)]),
    "beast_plan_destroy": (C.c_int, [C.c_void_p]),
    "beast_version": (C.c_char_p, []),
    "beast_launch_count": (C.c_int64, []),
    "beast_debug_disable_fast": (C.c_int, [C.c_int32]),
    "beast_overlap_count": (C.c_int64, []),
    "beast_debug_force_wait": (C.c_int, [C.c_int32]),
    "beast_debug_ranges_conflict": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32]),
    "beast_encode_f32": (C.c_int, [C.c_void_p, c_f32p, C.c_int64, c_f32p, c_f32p, C.c_int64, c_f32p, c_i64p, C.c_void_p]),
    "beast_quantize_f32": (C.c_int, [C.c_void_p, c_f32p, C.c_int64, c_f32p, c_f32p, C.c_int64, c_i64p, C.c_void_p]),
    "beast_normalize_f32": (C.c_int, [C.c_void_p, c_f32p, C.c_int64, c_f32p, c_f32p, c_f32p, C.c_void_p]),
    "beast_decode_f32": (C.c_int, [C.c_void_p, c_i64p, C.c_int64, c_f32p, c_f32p, C.c_int64, c_f32p, c_f32p, C.c_void_p]),
    "beast_decode_times_f32": (C.c_int, [C.c_void_p, c_i64p, C.c_int64, c_f32p, c_f32p, C.c_int64, c_f32p, c_f32p,
                                         C.c_int32, c_f32p, C.c_void_p]),
    "beast_dequantize_f32": (C.c_int, [C.c_void_p, c_i64p, C.c_int64, c_f32p, c_f32p, C.c_int64, c_f32p, C.c_void_p]),
    "beast_eval_f32": (C.c_int, [C.c_void_p, c_f32p, C.c_int64, c_f32p, c_f32p, C.c_int32, c_f32p, C.c_void_p]),
    "beast_reconstruct_bc_f32": (C.c_int, [C.c_void_p, c_i64p, c_f32p, C.c_int64, c_f32p, c_f32p, C.c_int64, c_f32p, c_f32p,
                                           C.c_int32, c_f32p, c_f32p, c_f32p, C.c_void_p]),
    "beast_grid_create": (C.c_int, [C.c_void_p, C.POINTER(GridDesc), C.POINTER(C.c_void_p)]),
    "beast_grid_destroy": (C.c_int, [C.c_void_p]),
    "beast_decode_grid_f32": (C.c_int, [C.c_void_p, C.c_void_p, c_i64p, c_f32p, C.c_int64, c_f32p, c_f32p, C.c_int64,
                                        c_f32p, c_f32p, c_f32p, c_f32p, c_f32p, c_f32p, C.c_void_p]),
    "beast_decode_deriv_times_f32": (C.c_int, [C.c_void_p, c_i64p, c_f32p, C.c_int64, c_f32p, c_f32p, C.c_int64, c_f32p,
                                               c_f32p, C.c_int32, c_f32p, c_f32p, c_f32p, c_f32p, c_f32p, C.c_void_p]),
    "beast_decode_grid_backward_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, c_f32p, c_f32p, c_f32p, C.c_int32,
                                                 c_f32p, c_f32p, C.c_void_p]),
    "beast_decode_deriv_times_backward_f32": (C.c_int, [C.c_void_p, C.c_int64, c_f32p, C.c_int32, c_f32p, c_f32p, c_f32p,
                                                        C.c_int32, c_f32p, c_f32p, C.c_void_p]),
    "beast_fit_backward_f32": (C.c_int, [C.c_void_p, C.c_int64, c_f32p, c_f32p, c_f32p, c_f32p, c_f32p, c_f32p,
                                         C.c_void_p]),
    "beast_fit_times_f32": (C.c_int, [C.c_void_p, c_f32p, C.c_int64, C.c_int32, c_f32p, c_f32p, c_f32p, c_f32p,
                                      C.c_void_p]),
    "beast_fit_times_backward_f32": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, c_f32p, c_f32p, c_f32p, c_f32p,
                                               c_f32p, c_f32p, c_f32p, c_f32p, c_f32p, C.c_void_p]),
    "beast_fit_minmax_f32":(C.c_int, [C.c_void_p, c_f32p, C.c_int64, c_f32p, c_f32p, C.c_int32, C.c_void_p]),
    "beast_fit_minmax_workspace_bytes": (C.c_int64, [C.c_void_p]),
    "beast_fit_minmax_ws_f32": (C.c_int, [C.c_void_p, c_f32p, C.c_int64, c_f32p, c_f32p, C.c_int32, C.c_void_p, C.c_int64,
                                          C.c_void_p]),
    "beast_minmax_f32": (C.c_int, [c_f32p, C.c_int64, C.c_int32, c_f32p, c_f32p, C.c_int32, C.c_void_p]),
    "beast_bounds_expand_f32": (C.c_int, [c_f32p, c_f32p, c_f32p, c_f32p, C.c_int32, C.c_float, C.c_void_p]),
    "beast_colselect_scratch_bytes": (C.c_int64, [C.c_int64, C.c_int32, C.c_int32]),
    "bpe_scan_bins": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "bpe_symbolize": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "bpe_count_pairs": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_int32,
                                  C.c_void_p, C.c_void_p, C.c_void_p]),
    "bpe_word_totals": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p]),
    "bpe_word_list": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p,
                                C.c_void_p, C.c_void_p]),
    "bpe_word_insert": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p,
                                  C.c_void_p]),
    "bpe_word_emit": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "bpe_word_pack": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p,
                                C.c_void_p, C.c_int64, C.c_int64, C.c_void_p]),
    "bpe_argmax": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
    "bpe_apply_merge": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                  C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "bpe_apply_delta": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "bpe_train_step": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p,
                                 C.c_int32, C.c_int32, C.POINTER(BpePeers), C.c_void_p, C.c_void_p]),
    "beast_peer_alloc": (C.c_int, [C.c_int64, C.POINTER(C.c_void_p), C.c_void_p]),
    "beast_peer_open": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "beast_peer_close": (C.c_int, [C.c_void_p]),
    "beast_peer_free": (C.c_int, [C.c_void_p]),
    "bpe_signature_words": (C.c_int32, []),
    "bpe_build_signatures": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p]),
    "bpe_encode": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                             C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "bpe_apply_shape": (C.c_int, [C.c_int32, C.c_int32, C.c_int64, C.c_void_p, C.c_void_p]),
    "bpe_compact": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "bpe_decode": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                             C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "beast_selftest_div": (C.c_int, [C.c_int32, C.c_int32, C.c_uint64, C.c_void_p, C.c_void_p]),
    "beast_colselect_f32": (C.c_int, [c_f32p, C.c_int64, C.c_int32, C.POINTER(C.c_int64), C.c_int32, c_f32p,
                                      C.c_void_p, C.c_void_p]),
}

_ERRORS = {-1: "null pointer", -2: "bad shape", -3: "misaligned pointer", -4: "unsupported configuration",
           -5: "out of memory"}


def exported_symbols():
    """Names include/beast_b200.h declares (checked by the CPU test-suite)."""
    return sorted(_SIGNATURES)


def load(build_if_missing=True):
    """Load the shared library (building it in-tree with nvcc when absent)."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH) and build_if_missing:
            from . import build as _build
            _build.build()
        if not os.path.exists(LIB_PATH):
            raise BeastB200Error(
                f"{LIB_PATH} is missing: build it with `python -m beast_tokenizer_b200.build` "
                "(there is no CPU fallback for the BEAST hot path)")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(rc, what):
    if rc == 0:
        return
    if rc < 0:
        raise BeastB200Error(f"{what}: {_ERRORS.get(rc, 'error')} ({rc})")
    raise BeastB200Error(f"{what}: CUDA error {rc}")


def require_cuda(device):
    dev = torch.device(device)
    if dev.type != "cuda":
        raise BeastB200Error(
            f"device={device!r}: beast_tokenizer_b200 runs the BEAST hot path on B200 GPUs only "
            "(no CPU fallback); construct the tokenizer with device='cuda'")
    if not torch.cuda.is_available():
        raise BeastB200Error("no CUDA device available: beast_tokenizer_b200 has no CPU fallback")
    return dev


def ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def stream_ptr(device):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def launch_count():
    return int(load().beast_launch_count())


def overlap_count():
    return int(load().beast_overlap_count())
