"""BEASTBsplineTokenizer — drop-in for the reference class of the same name
(beast/beast_bspline_tokenizer.py:45-597) with the hot path on B200 CUDA kernels.

Same constructor, methods, return types, exceptions and on-disk format; underneath, the
movement-primitive library, the per-trajectory LU solve and the elementwise quantiser are
replaced by the C-ABI kernels of libbeast_b200.so (include/beast_b200.h).

Limits next to the reference (also in README "Out of scope"): the three visualize_* methods raise
NotImplementedError (plotting); num_dof <= 64 (BEAST_MAX_DOF); init / end condition orders 0, 1, 2 only;
non-finite trajectories are not rejected — the fused min / max and the clamp use IEEE fmin / fmax, which
drop a NaN where torch.min / torch.clamp would propagate it.  Entry points:

    encode / compute_weights / encode_continuous  -> beast_encode_f32 (+ quantize / normalize)
    decode / reconstruct_traj(_continuous)        -> beast_decode_f32 / _times / dequantize / eval
    reconstruct_traj(_continuous)_derivatives     -> beast_decode_grid_f32 / beast_decode_deriv_times_f32
    reconstruct_traj_continuous(_derivatives)
        backward (autograd)                       -> beast_decode_grid_backward_f32 / beast_decode_deriv_times_backward_f32
    encode_continuous backward (autograd)         -> beast_fit_backward_f32
    update_weights_bounds(_per_batch)             -> beast_minmax_f32 + beast_bounds_expand_f32
    fit_parameters                                -> beast_encode_f32 + beast_colselect_f32

There is no CPU fallback: compute methods raise BeastB200Error without a CUDA device.
"""
import ctypes as C
import json
import numbers
from pathlib import Path
from typing import Optional

import numpy as np
import torch
from torch.autograd.function import once_differentiable

from . import _dist, _lib
from .base_tokenizer import TokenizerBase
from .basis import SplineConstants, bspline_basis_derivatives, build_constants, check_orders, make_times

CONFIG_FILENAME = "beast_tokenizer_config.json"


class _Plan:
    """Owns one beast_plan_t (immutable device tables for one geometry)."""

    def __init__(self, consts: SplineConstants, vocab_size: int, device: torch.device):
        self.consts = consts
        self.device = device
        lib = _lib.load()

        def fptr(t):
            return None if t is None else t.contiguous().numpy().ctypes.data_as(C.POINTER(C.c_float))

        self._keep = [consts.proj_joint, consts.proj_grip, consts.phi_joint, consts.phi_grip,
                      consts.knots_joint, consts.knots_grip]
        slots = (C.c_int32 * consts.num_dof)(*consts.slot_to_dof)
        desc = _lib.PlanDesc(
            seq_len=consts.seq_len, num_dof=consts.num_dof, num_basis=consts.num_basis,
            n_joint=len(consts.joint_indices), degree_p=consts.degree_p, vocab_size=int(vocab_size),
            tau=consts.tau, slot_to_dof_h=slots,
            proj_joint_h=fptr(consts.proj_joint), proj_grip_h=fptr(consts.proj_grip),
            phi_joint_h=fptr(consts.phi_joint), phi_grip_h=fptr(consts.phi_grip),
            knots_joint_h=fptr(consts.knots_joint), knots_grip_h=fptr(consts.knots_grip),
            init_cond_order=consts.init_order, end_cond_order=consts.end_order)
        handle = C.c_void_p()
        with torch.cuda.device(device):
            _lib.check(lib.beast_plan_create(C.byref(desc), C.byref(handle)), "beast_plan_create")
        self.handle = handle
        self._lib = lib
        self._workspaces = {}

    def minmax_workspace(self) -> torch.Tensor:
        """Zero-initialised scratch of beast_fit_minmax_ws_f32, one per (plan, stream)."""
        key = torch.cuda.current_stream(self.device).cuda_stream
        ws = self._workspaces.get(key)
        if ws is None:
            n = int(self._lib.beast_fit_minmax_workspace_bytes(self.handle)) // 4
            ws = self._workspaces[key] = torch.zeros(max(n, 1), device=self.device, dtype=torch.float32)
        return ws

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                self._lib.beast_plan_destroy(self.handle)
                self.handle = None
        except Exception:
            pass


class _Grid:
    """Owns one beast_grid_t: the basis rows of orders 0..max_order on one time grid shared by every trajectory
    (basis.bspline_basis_derivatives), for the plan it was built for (kept alive with it)."""

    def __init__(self, plan: _Plan, times: torch.Tensor, max_order: int):
        c = plan.consts
        nc = c.num_basis + c.init_order + c.end_order
        times = times.to("cpu", torch.float32).contiguous()
        rows_j = bspline_basis_derivatives(times, c.tau, nc, c.degree_p, max_order)
        rows_g = bspline_basis_derivatives(times, c.tau, c.num_basis, 0, max_order) if c.gripper_indices else None

        def fptr(t):
            return None if t is None else t.numpy().ctypes.data_as(C.POINTER(C.c_float))

        self._keep = [times, rows_j, rows_g]
        desc = _lib.GridDesc(n_times=int(times.numel()), max_order=int(max_order), times_h=fptr(times),
                             rows_joint_h=fptr(rows_j), rows_grip_h=fptr(rows_g))
        handle = C.c_void_p()
        with torch.cuda.device(plan.device):
            _lib.check(plan._lib.beast_grid_create(plan.handle, C.byref(desc), C.byref(handle)), "beast_grid_create")
        self.handle = handle
        self.plan = plan
        self.n_times = int(times.numel())

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                self.plan._lib.beast_grid_destroy(self.handle)
                self.handle = None
        except Exception:
            pass


class _Adjoint:
    """The backward launch of one continuous decode: the gradients of its outputs (orders `orders`) -> the gradients
    of the de-normalised '(d t)' coefficients [B, D*nb] and of init_p [B, num_dof].  A grid (shared times) takes
    beast_decode_grid_backward_f32, per-row times [B, Tq] beast_decode_deriv_times_backward_f32."""

    def __init__(self, plan: _Plan, batch: int, orders, grid: Optional[_Grid], times, tq: int, init_p_used: bool):
        self.plan, self.batch, self.orders, self.grid = plan, batch, orders, grid
        self.times, self.tq, self.init_p_used = times, tq, init_p_used

    def __call__(self, grads, want_init_p):
        plan, B, dev = self.plan, self.batch, self.plan.device
        by_order = dict(zip(self.orders, grads))
        g = [by_order.get(o) for o in range(3)]
        if all(x is None for x in g):
            return None, None
        g = [None if x is None else x.to(dev, torch.float32).contiguous() for x in g]
        c = plan.consts
        grad_params = torch.empty((B, c.num_dof * c.num_basis), device=dev, dtype=torch.float32)
        grad_init_p = (torch.empty((B, c.num_dof), device=dev, dtype=torch.float32)
                       if self.init_p_used and want_init_p else None)
        if B == 0 or self.tq == 0:      # no sample reads a coefficient
            grad_params.zero_()
            if grad_init_p is not None:
                grad_init_p.zero_()
            return grad_params, grad_init_p
        args = (*[_lib.ptr(x) for x in g], int(self.init_p_used), _lib.ptr(grad_params), _lib.ptr(grad_init_p),
                _lib.stream_ptr(dev))
        with torch.cuda.device(dev):
            if self.grid is not None:
                _lib.check(plan._lib.beast_decode_grid_backward_f32(plan.handle, self.grid.handle, B, *args),
                           "beast_decode_grid_backward_f32")
            else:                       # per-row times, or an empty grid (every gradient is then 0)
                _lib.check(plan._lib.beast_decode_deriv_times_backward_f32(plan.handle, B, _lib.ptr(self.times),
                                                                           self.tq, *args),
                           "beast_decode_deriv_times_backward_f32")
        return grad_params, grad_init_p


class _SplineDecodeFn(torch.autograd.Function):
    """The coefficient contraction of reconstruct_traj_continuous(_derivatives) as an autograd node: forward = the
    decode launch (`decode(params, init_p)` -> tuple of outputs), backward = its adjoint launch.  Denormalising and the
    layout transposition stay torch ops in front of it.  Outputs the loss does not use arrive as None and are passed
    to the kernel as NULL.  The map is linear, so the backward needs no saved tensors; it is not itself differentiable."""

    @staticmethod
    def forward(ctx, decode, adjoint, params, init_p):
        ctx.set_materialize_grads(False)
        ctx.adjoint = adjoint
        return decode(params, init_p)

    @staticmethod
    @once_differentiable
    def backward(ctx, *grads):
        grad_params, grad_init_p = ctx.adjoint(grads, ctx.needs_input_grad[3])
        return None, None, grad_params if ctx.needs_input_grad[2] else None, grad_init_p


class _FitFn(torch.autograd.Function):
    """encode_continuous's fit and normalisation as an autograd node: forward = `fit(x)` (the K1 launch, the optional
    bounds expansion and beast_normalize_f32, unchanged) -> (normalised, params, (w_min, w_max) snapshot), backward =
    one beast_fit_backward_f32 launch.  The unclamped params and the bounds the forward normalised with are saved; an
    output the loss does not use arrives as None and is passed to the kernel as NULL.  Not itself differentiable."""

    @staticmethod
    def forward(ctx, fit, plan, x):
        ctx.set_materialize_grads(False)
        normalised, params, bounds = fit(x)
        ctx.plan, ctx.bounds = plan, bounds
        ctx.save_for_backward(params)
        return normalised, params

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_norm, grad_params):
        if grad_norm is None and grad_params is None:
            return None, None, None
        plan = ctx.plan
        (params,), (lo, hi) = ctx.saved_tensors, ctx.bounds
        dev = plan.device
        c = plan.consts
        grad_norm, grad_params = (None if g is None else g.to(dev, torch.float32).contiguous()
                                  for g in (grad_norm, grad_params))
        B = params.shape[0]
        grad_traj = torch.empty((B, c.seq_len, c.num_dof), device=dev, dtype=torch.float32)
        if B == 0:                      # empty tensors carry no data pointer
            return None, None, grad_traj
        with torch.cuda.device(dev):
            _lib.check(plan._lib.beast_fit_backward_f32(
                plan.handle, B, _lib.ptr(grad_norm), _lib.ptr(grad_params), _lib.ptr(params), _lib.ptr(lo),
                _lib.ptr(hi), _lib.ptr(grad_traj), _lib.stream_ptr(dev)), "beast_fit_backward_f32")
        return None, None, grad_traj


class BEASTBsplineTokenizer(TokenizerBase):

    def __init__(self, num_dof=1, num_basis=10, duration=2 * torch.pi, seq_len=50, vocab_size=256,
                 degree_p=4, gripper_zero_order=False, gripper_indices=None,
                 init_cond_order=0, end_cond_order=0, init_pos=True,
                 use_bpe=False, device="cuda", llm_vocab_size: Optional[int] = None):
        super().__init__()
        if init_cond_order not in (0, 1, 2) or end_cond_order not in (0, 1, 2):
            # the reference's end order -1 / goal basis variants are not reachable from its own tokenizer config
            raise NotImplementedError("init_cond_order / end_cond_order must be 0, 1 or 2")
        if (init_cond_order == 2 or end_cond_order == 2) and degree_p < 1:
            raise NotImplementedError("velocity conditions need degree_p >= 1")
        self.init_cond_order = int(init_cond_order)
        self.end_cond_order = int(end_cond_order)
        # The reference's joint MP keeps the pinned boundary control points of its LAST fit as object
        # state and reconstruct_traj silently uses them (mp/uni_bspline.py:68-104, 126-136); same here.
        self._boundary = None

        self.dt = 0.01
        # gripper handling exactly as the reference (:55-70): indices are dropped unless zero-order
        if gripper_indices is None or not gripper_zero_order:
            gripper_indices = []
        self.gripper_indices = sorted(gripper_indices)
        self.gripper_dof = len(self.gripper_indices) if gripper_zero_order else 0
        self.joint_dof = num_dof - self.gripper_dof
        self.joint_indices = sorted(set(range(num_dof)) - set(self.gripper_indices))
        self.init_pos = init_pos

        self.device = device
        self.num_dof = self.joint_dof + self.gripper_dof
        self.num_basis = num_basis
        self.degree_p = degree_p
        self.vocab_size = vocab_size
        self.duration = duration
        self.seq_length = seq_len
        self.use_bpe = use_bpe

        self.times = make_times(duration, seq_len)
        self._times_version = 0
        self._plan_cache = None
        # sharded fitting is opt-in (set_process_group): an implicit collective inside update_weights_bounds /
        # fit_parameters would hang every caller that fits on one rank of an initialised job
        self.process_group = False
        if self.gripper_dof > 0:
            print(f"Gripper MP initialized with {num_basis} basis functions for "
                  f"{self.gripper_dof} DOFs at indices {self.gripper_indices}")

        buf_dev = self._buffer_device()
        self.register_buffer("w_min", -0.02 * torch.ones(num_dof * num_basis, device=buf_dev))
        self.register_buffer("w_max", 0.02 * torch.ones(num_dof * num_basis, device=buf_dev))
        self.llm_vocab_size = None

        self._config = {
            'tokenizer_type': 'beast_bspline',
            'num_dof': num_dof,
            'num_basis': num_basis,
            'duration': float(duration),
            'seq_len': seq_len,
            'vocab_size': vocab_size,
            'degree_p': degree_p,
            'gripper_zero_order': gripper_zero_order,
            'gripper_indices': list(self.gripper_indices),
            'init_cond_order': init_cond_order,
            'end_cond_order': end_cond_order,
            'init_pos': init_pos,
            'use_bpe': use_bpe,
            'device': device,
        }
        if llm_vocab_size is not None:
            self.set_llm_vocab_size(llm_vocab_size)

    # ------------------------------------------------------------------ plumbing
    def _buffer_device(self):
        try:
            dev = torch.device(self.device)
        except (TypeError, RuntimeError):
            return "cpu"
        return dev if (dev.type == "cuda" and torch.cuda.is_available()) else "cpu"

    def _cuda(self) -> torch.device:
        dev = _lib.require_cuda(self.device)
        if dev.index is None:
            dev = torch.device("cuda", torch.cuda.current_device())
        return dev

    def _plan(self) -> _Plan:
        dev = self._cuda()
        # `times` is part of the geometry: update_times() bumps the version; in-place edits of tok.times are picked up
        # through the content hash of the (short) vector
        key = (dev, self._times_version, hash(self.times.numpy().tobytes()), int(self.vocab_size))
        if self._plan_cache is None or self._plan_cache[0] != key:
            consts = build_constants(self.times, self.duration, self.num_basis, self.degree_p,
                                     self.joint_indices, self.gripper_indices,
                                     self.init_cond_order, self.end_cond_order)
            self._plan_cache = (key, _Plan(consts, self.vocab_size, dev), self.times)
        return self._plan_cache[1]

    _GRID_CACHE_SIZE = 8

    def _grid(self, plan: _Plan, times: torch.Tensor, max_order: int) -> _Grid:
        """The grid of `times` [Tq] (CPU fp32) for `plan`, cached per (device, plan key, grid bytes, max order)."""
        plan_key = self._plan_cache[0]
        cache = self.__dict__.setdefault("_grid_cache", {})
        key = (plan_key, times.numpy().tobytes(), int(max_order))
        grid = cache.get(key)
        if grid is None:
            for k in [k for k in cache if k[0] != plan_key]:       # grids of a replaced plan
                del cache[k]
            while len(cache) >= self._GRID_CACHE_SIZE:
                cache.pop(next(iter(cache)))
            grid = cache[key] = _Grid(plan, times, max_order)
        return grid

    def _bounds(self, dev):
        return (self.w_min.to(dev, torch.float32).contiguous(), self.w_max.to(dev, torch.float32).contiguous())

    def _prep_trajs(self, trajs, dev):
        # pinned host batches are uploaded asynchronously on the current stream (stream-ordered before
        # the kernel), so callers can overlap the copy of one chunk with the compute of another
        trajs = trajs.to(dev, dtype=torch.float32, non_blocking=bool(trajs.device.type == "cpu" and trajs.is_pinned()))
        if trajs.dim() != 3:
            raise AssertionError(f"expected trajectories [batch, time, dof], got {tuple(trajs.shape)}")
        if trajs.shape[1] != self.times.numel():
            raise AssertionError(f"trajectory has {trajs.shape[1]} samples, tokenizer times has {self.times.numel()}")
        if trajs.shape[2] < self.num_dof:
            raise IndexError(f"trajectory has {trajs.shape[2]} DoF, tokenizer expects {self.num_dof}")
        if trajs.shape[2] > self.num_dof:          # extra trailing DoF are never indexed by the reference
            trajs = trajs[..., :self.num_dof]
        return trajs.contiguous()

    def _fit(self, trajs, want_tokens, offset=0, bounds=None):
        """One K1 launch: (tokens | None, unclamped params)."""
        plan = self._plan()
        dev = plan.device
        x = self._prep_trajs(trajs, dev)
        B = x.shape[0]
        n = self.num_dof * self.num_basis
        params = torch.empty((B, n), device=dev, dtype=torch.float32)
        tokens = torch.empty((B, n), device=dev, dtype=torch.int64) if want_tokens else None
        lo, hi = bounds if bounds is not None else (self._bounds(dev) if want_tokens else (None, None))
        with torch.cuda.device(dev):
            _lib.check(plan._lib.beast_encode_f32(plan.handle, _lib.ptr(x), B, _lib.ptr(lo), _lib.ptr(hi),
                                                  int(offset), _lib.ptr(params), _lib.ptr(tokens),
                                                  _lib.stream_ptr(dev)), "beast_encode_f32")
        self._remember_boundary(x, plan)
        return tokens, params

    @property
    def _has_conditions(self) -> bool:
        return (self.init_cond_order != 0 or self.end_cond_order != 0) and self.joint_dof > 0

    def _remember_boundary(self, x, plan):
        """Boundary state of a fit with non-zero condition orders (mp/uni_bspline.py:500-531,
        basis_gn/uni_bspline_basis.py:192-274): the pinned control points are functions of the four
        boundary samples y[0], y[1], y[-2], y[-1] only — O(B*D) elementwise work next to the fit."""
        if not self._has_conditions:
            return
        self._boundary = self._boundary_state(x, plan)

    def _boundary_state(self, x, plan):
        """The boundary state of `x` (torch ops: attached to the graph of `x` under grad mode)."""
        io, eo, p = self.init_cond_order, self.end_cond_order, self.degree_p
        c = plan.consts
        nc = self.num_basis + io + eo
        t = c.times
        inv_dt = float(torch.tensor(1.0) / (t[1] - t[0]))
        tau = c.tau
        ji = torch.as_tensor(self.joint_indices, device=x.device)
        y0, y1, ym2, ym1 = (x[:, i, :].index_select(1, ji) for i in (0, 1, -2, -1))
        st = {"init_pos": None, "init_vel": None, "end_pos": None, "end_vel": None}
        parts = []
        if io != 0:
            st["init_pos"] = y0
            st["init_vel"] = (y1 - y0) * inv_dt
            parts.append(torch.zeros_like(y0))
            if io == 2:
                dk = float(c.knots_joint[1 + p] - c.knots_joint[1])
                parts.append(st["init_vel"] * tau * dk / p + 0.0)
        if eo != 0:
            end_pos = ym1 - y0 if io != 0 else ym1
            st["end_vel"] = (ym1 - ym2) * inv_dt
            if eo == 2:
                dk = float(c.knots_joint[nc - 1 + p] - c.knots_joint[nc - 1])
                parts.append(end_pos - st["end_vel"] * tau * dk / p)
            parts.append(end_pos)
            st["end_pos"] = end_pos + y0 if io != 0 else end_pos       # returned absolute (:600)
        st["bc"] = torch.stack(parts, dim=-1).contiguous()             # [B, n_joint, io + eo]
        st["bias"] = y0.contiguous() if io != 0 else None
        return st

    def _params_dict(self, params, st=None):
        # keys of UniformBSpline.learn_mp_params_from_trajs (mp/uni_bspline.py:597-602); `st` overrides the kept state
        if st is None:
            st = self._boundary if self._has_conditions else None
        if st is None:
            return {"params": params, "init_pos": None, "init_vel": None, "end_pos": None, "end_vel": None}
        return {"params": params, "init_pos": st["init_pos"], "init_vel": st["init_vel"],
                "end_pos": st["end_pos"], "end_vel": st["end_vel"]}

    def _pinned(self, batch):
        """(bc, bias) of the last fit for a reconstruct of `batch` trajectories."""
        if not self._has_conditions:
            return None, None
        st = self._boundary
        if st is None:
            raise RuntimeError("init_cond_order / end_cond_order != 0: reconstruct needs the boundary conditions "
                               "of a previous encode (the reference keeps them as state of its MP object)")
        if st["bc"].shape[0] != batch:
            raise RuntimeError(f"boundary conditions were fitted for a batch of {st['bc'].shape[0]}, "
                               f"cannot reconstruct a batch of {batch}")
        return st["bc"], st["bias"]

    # ------------------------------------------------------------------ preparation
    def set_llm_vocab_size(self, llm_vocab_size: Optional[int]):
        if llm_vocab_size is None:
            self.llm_vocab_size = None
            self._config.pop('llm_vocab_size', None)
            return
        if not isinstance(llm_vocab_size, numbers.Integral):
            raise TypeError("llm_vocab_size must be an integer or None")
        llm_vocab_size = int(llm_vocab_size)
        if llm_vocab_size < self.vocab_size:
            raise ValueError("llm_vocab_size must be greater or equal to tokenizer vocab size")
        self.llm_vocab_size = llm_vocab_size
        self._config['llm_vocab_size'] = llm_vocab_size

    def set_process_group(self, process_group="world"):
        """Shard the FITTING calls over torch.distributed ranks (one process per GPU, every rank passes its shard of
        the data): update_weights_bounds all-reduces MIN / MAX of the two D*nb vectors, fit_parameters all-gathers
        the coefficient rows before the exact quantile selection, update_weights_bounds_per_batch all-reduces the
        batch min / max.  "world" = the default group, a ProcessGroup = that group, False = local (the default).
        encode / decode shard by rows and never communicate."""
        self.process_group = process_group
        return self

    def _group(self, process_group):
        return self.process_group if process_group is None else process_group

    def update_vlm_vocab_size(self, vlm_vocab_size):
        self.set_llm_vocab_size(vlm_vocab_size)

    def _llm_vocab_offset(self) -> int:
        if self.llm_vocab_size is None:
            raise ValueError("LLM vocab size is not set.")
        return self.llm_vocab_size - self.vocab_size

    @torch.no_grad()
    def fit_parameters(self, dataloader, max_samples=None, verbose=True, process_group=None):
        """1 % / 99 % per-column quantiles of the fitted coefficients (reference :181-220).
        Coefficients stay on the GPU; the order statistics np.quantile needs are selected
        exactly by beast_colselect_f32 and interpolated with numpy's own lerp.
        Sharded (set_process_group, or process_group= here; every rank iterates ITS shard of the loader): the
        ranks' coefficient rows are all-gathered (56 MB per 100 k trajectories) before the exact selection, so
        every rank ends with the quantiles of the whole data set."""
        params = []
        sample_limit = max_samples if max_samples is not None else float("inf")
        iterator = dataloader
        if verbose:
            try:
                from tqdm import tqdm
                iterator = tqdm(dataloader, total=max_samples, desc="precomputing weight normalizer of MP", unit="batch")
            except Exception:
                iterator = dataloader
        sample_count = 0
        # The reference fits batch by batch; the coefficients of a trajectory do not depend on its position in a
        # batch, so small loader batches (32 in the reference's training script) are gathered on the device and
        # fitted ~4 096 at a time: one K1 launch per chunk instead of one per batch.  The gathered batches are READ at
        # the flush (up to ~128 batches later): a loader must yield fresh tensors, as torch's DataLoader does, not one
        # buffer it overwrites in place (FIGBPE.fit_from_trajectories copies every batch at once and has no such rule).
        dev = self._cuda()
        pending, pending_rows, pending_key = [], 0, None
        T, D, gatherable = self.times.numel(), self.num_dof, not self._has_conditions

        def flush():
            nonlocal pending_rows
            if pending:
                x = pending[0] if len(pending) == 1 else torch.cat(pending, dim=0)     # one copy kernel / memcpy pass
                params.append(self.compute_weights(x[..., :D] if x.shape[2] != D else x))
                pending.clear()
                pending_rows = 0

        # the per-batch work is a handful of Python operations (the loader's 3 125 batches of 32 are otherwise bound
        # by ~3 us of tensor-op dispatch each); conversion, slicing and the upload happen once per ~4 096 rows
        for batch in iterator:
            try:
                x = batch["actions"]
            except KeyError:
                raise KeyError("Expected batch to contain an 'actions' entry.") from None
            if gatherable and type(x) is torch.Tensor and x.dim() == 3 and x.shape[1] == T and x.shape[2] >= D:
                key = (x.device, x.dtype, x.shape[2])
                if key != pending_key:
                    flush()
                    pending_key = key
                pending.append(x)
                pending_rows += x.shape[0]
                if pending_rows >= 4096:
                    flush()
            else:                                   # odd shapes raise here, as they would per batch; boundary-condition
                flush()                             # tokenizers keep the reference's "state of the last batch" semantics
                params.append(self.compute_weights(x[..., : self.num_dof]))
            sample_count += 1
            if sample_count >= sample_limit:
                if verbose:
                    print("Precomputed enough samples for weight normalizer of MP")
                break
        flush()
        dist, group = _dist.resolve(self._group(process_group), implicit=False)
        if not params and dist is None:
            raise RuntimeError("No parameters were gathered from the dataloader.")
        params = (torch.cat(params, dim=0) if params else
                  torch.empty((0, self.num_dof * self.num_basis), device=dev, dtype=torch.float32))
        if dist is not None:
            params = _dist.gather_rows(params, _dist.WORLD if group is None else group)
            if params.shape[0] == 0:
                raise RuntimeError("No parameters were gathered from the dataloader.")
        lo, hi = self._column_quantiles(params, (0.01, 0.99))
        self.w_min.copy_(lo.to(self.w_min.device))
        self.w_max.copy_(hi.to(self.w_max.device))

    def _column_quantiles(self, params, qs):
        """np.quantile(params, q, axis=0) for each q (numpy 'linear' method, fp32 input)."""
        plan = self._plan()
        dev = plan.device
        params = params.to(dev, torch.float32).contiguous()
        n, cols = params.shape
        ks, gammas = [], []
        for q in qs:
            q32 = np.asanyarray(q, dtype=np.float32)           # numpy >= 2 matches q to the array dtype
            virt = (n - 1) * q32
            prev = int(np.floor(virt))
            nxt = prev + 1
            if virt >= n - 1:
                prev = nxt = n - 1
            if virt < 0:
                prev = nxt = 0
            gammas.append(np.asanyarray(virt - np.float32(np.floor(virt)), dtype=np.float32))
            ks += [prev, nxt]
        ks_arr = (C.c_int64 * len(ks))(*ks)
        out = torch.empty((len(ks), cols), device=dev, dtype=torch.float32)
        nbytes = int(plan._lib.beast_colselect_scratch_bytes(n, cols, len(ks)))
        scratch = torch.empty(nbytes, device=dev, dtype=torch.uint8)
        with torch.cuda.device(dev):
            _lib.check(plan._lib.beast_colselect_f32(_lib.ptr(params), n, cols, ks_arr, len(ks), _lib.ptr(out),
                                                     _lib.ptr(scratch), _lib.stream_ptr(dev)), "beast_colselect_f32")
        sel = out.cpu().numpy()
        res = []
        for i, g in enumerate(gammas):
            # numpy's own _lerp on the two neighbouring order statistics (virtual index = gamma on 2 rows)
            pair = np.stack([sel[2 * i], sel[2 * i + 1]])
            res.append(torch.from_numpy(np.asarray(np.quantile(pair, np.float32(g), 0), dtype=np.float32)))
        return res

    # ------------------------------------------------------------------ serialization
    def get_config(self):
        config = self._config.copy()
        if self.llm_vocab_size is not None:
            config['llm_vocab_size'] = self.llm_vocab_size
        return config

    def state_dict(self):
        return {
            'config': self.get_config(),
            'w_min': self.w_min.cpu().numpy().tolist(),
            'w_max': self.w_max.cpu().numpy().tolist(),
            'llm_vocab_size': self.llm_vocab_size,
        }

    def load_state_dict(self, state_dict):
        if 'w_min' in state_dict:
            self.w_min.copy_(torch.tensor(state_dict['w_min'], dtype=torch.float32).to(self.w_min.device))
        if 'w_max' in state_dict:
            self.w_max.copy_(torch.tensor(state_dict['w_max'], dtype=torch.float32).to(self.w_max.device))
        llm_size = state_dict.get('llm_vocab_size')
        if llm_size is None:
            llm_size = state_dict.get('vlm_vocab_size')
        if llm_size is not None:
            self.set_llm_vocab_size(llm_size)
        print(f"✓ Loaded fitted parameters (w_min, w_max) with shape {self.w_min.shape}")

    def save_pretrained(self, save_directory):
        save_directory = Path(save_directory)
        save_directory.mkdir(parents=True, exist_ok=True)
        config_path = save_directory / CONFIG_FILENAME
        with open(config_path, 'w') as f:
            json.dump(self.state_dict(), f, indent=2)
        print(f"✓ Saved tokenizer to {save_directory}")
        print(f"  - Config: {config_path}")

    @classmethod
    def from_pretrained(cls, pretrained_path, device=None):
        pretrained_path = Path(pretrained_path)
        config_path = pretrained_path / CONFIG_FILENAME
        if not config_path.exists():
            raise FileNotFoundError(f"Config file not found: {config_path}")
        with open(config_path, 'r') as f:
            state = json.load(f)
        config = state['config'].copy()
        tokenizer_type = config.get('tokenizer_type')
        if tokenizer_type not in {'beast_bspline', None}:
            raise ValueError("Loaded configuration does not describe a BEAST B-Spline tokenizer.")
        config.pop('tokenizer_type', None)
        if device is not None:
            config['device'] = device
        print(f"✓ Loading tokenizer from {pretrained_path}")
        print(f"  - Config: num_dof={config['num_dof']}, num_basis={config['num_basis']}, "
              f"gripper_indices={config['gripper_indices']}")
        tokenizer = cls(**config)
        tokenizer.load_state_dict(state)
        return tokenizer

    # ------------------------------------------------------------------ utils
    @torch.no_grad()
    def compute_weights(self, demos):
        """Unclamped spline coefficients [B, D*nb] '(d t)', joints first (reference :344-360)."""
        return self._fit(demos, want_tokens=False)[1]

    @torch.no_grad()
    def update_weights_bounds(self, demos, process_group=None):
        """Global per-column min / max of the coefficients (reference :362-378): one fused launch,
        the coefficients are reduced in registers and never written.  Sharded (set_process_group, or
        process_group= here; every rank passes its shard): one MIN and one MAX all-reduce of the D*nb vectors."""
        plan = self._plan()
        dev = plan.device
        x = self._prep_trajs(demos, dev)
        n = self.num_dof * self.num_basis
        # one launch, results written straight into the w_min / w_max buffers when they live on this device
        direct = (self.w_min.device == dev and self.w_max.device == dev and self.w_min.dtype == torch.float32
                  and self.w_max.dtype == torch.float32 and self.w_min.is_contiguous() and self.w_max.is_contiguous())
        lo = self.w_min if direct else torch.empty(n, device=dev, dtype=torch.float32)
        hi = self.w_max if direct else torch.empty(n, device=dev, dtype=torch.float32)
        ws = plan.minmax_workspace()
        with torch.cuda.device(dev):
            _lib.check(plan._lib.beast_fit_minmax_ws_f32(plan.handle, _lib.ptr(x), x.shape[0], _lib.ptr(lo), _lib.ptr(hi), 0,
                                                         _lib.ptr(ws), ws.numel() * 4, _lib.stream_ptr(dev)),
                       "beast_fit_minmax_ws_f32")
        self._remember_boundary(x, plan)
        _dist.allreduce_minmax(lo, hi, self._group(process_group), implicit=False)
        if not direct:
            self.w_min.copy_(lo.to(self.w_min.device))
            self.w_max.copy_(hi.to(self.w_max.device))

    def _minmax(self, weights):
        dev = weights.device
        lib = _lib.load()
        n = weights.shape[1]
        lo = torch.empty(n, device=dev, dtype=torch.float32)
        hi = torch.empty(n, device=dev, dtype=torch.float32)
        with torch.cuda.device(dev):
            _lib.check(lib.beast_minmax_f32(_lib.ptr(weights), weights.shape[0], n, _lib.ptr(lo), _lib.ptr(hi), 0,
                                            _lib.stream_ptr(dev)), "beast_minmax_f32")
        return lo, hi

    @torch.no_grad()
    def update_weights_bounds_per_batch(self, weights, process_group=None):
        """Monotone expansion with 1e-4 hysteresis (reference :379-389).  Sharded (set_process_group, or
        process_group= here): the batch min / max are all-reduced first, so every rank expands identically."""
        dev = self._cuda()
        weights = weights.to(dev, torch.float32).reshape(-1, self.num_dof * self.num_basis).contiguous()
        lo, hi = self._minmax(weights)
        _dist.allreduce_minmax(lo, hi, self._group(process_group), implicit=False)
        on_dev = self.w_min.device == dev and self.w_max.device == dev
        w_min = self.w_min if on_dev else self.w_min.to(dev)
        w_max = self.w_max if on_dev else self.w_max.to(dev)
        lib = _lib.load()
        with torch.cuda.device(dev):
            _lib.check(lib.beast_bounds_expand_f32(_lib.ptr(lo), _lib.ptr(hi), _lib.ptr(w_min), _lib.ptr(w_max),
                                                   w_min.numel(), 1e-4, _lib.stream_ptr(dev)),
                       "beast_bounds_expand_f32")
        if not on_dev:
            self.w_min.copy_(w_min.to(self.w_min.device))
            self.w_max.copy_(w_max.to(self.w_max.device))

    def update_times(self, times):
        self.times = times.detach().to("cpu", torch.float32).reshape(-1).contiguous()
        self._times_version += 1
        self._plan_cache = None

    # ------------------------------------------------------------------ encoding
    @torch.no_grad()
    def encode(self, trajs, update_bounds=False, *, respect_llm_vocab_size=True):
        """trajs [B, T, D] -> (tokens int64 [B, nb*D] '(t d)', params_dict) — reference :399-428."""
        offset = 0
        if respect_llm_vocab_size and self.llm_vocab_size is not None:
            offset = self._llm_vocab_offset()
        if not update_bounds:
            tokens, params = self._fit(trajs, want_tokens=True, offset=offset)
            return tokens, self._params_dict(params)
        # bounds move before quantisation: fit, expand, then the exact quantiser on the coefficients
        _, params = self._fit(trajs, want_tokens=False)
        self.update_weights_bounds_per_batch(params)
        tokens = self._quantize(params, offset)
        return tokens, self._params_dict(params)

    def _quantize(self, params, offset=0):
        plan = self._plan()
        dev = plan.device
        params = params.to(dev, torch.float32).contiguous()
        lo, hi = self._bounds(dev)
        tokens = torch.empty(params.shape, device=dev, dtype=torch.int64)
        with torch.cuda.device(dev):
            _lib.check(plan._lib.beast_quantize_f32(plan.handle, _lib.ptr(params), params.shape[0], _lib.ptr(lo),
                                                    _lib.ptr(hi), int(offset), _lib.ptr(tokens),
                                                    _lib.stream_ptr(dev)), "beast_quantize_f32")
        return tokens

    def encode_continuous(self, trajs, update_bounds=False):
        """Normalised [-1, 1] coefficients in '(t d)' order (reference :430-450).

        Differentiable with respect to `trajs` when `trajs` requires grad under grad mode: the backward of `normalised`
        and `params_dict['params']` is beast_fit_backward_f32 (the adjoint of the fit; the normaliser's clamp passes
        the gradient where w_min <= params <= w_max, inclusive), and the condition-order entries of `params_dict` are
        torch ops on the boundary samples.  w_min / w_max as the call normalised with (after the expansion of
        update_bounds=True), the times and the tokenizer state are constants; the boundary state the tokenizer keeps
        for later reconstructs is detached.  Otherwise the call runs under no_grad, as before."""
        if not (torch.is_grad_enabled() and isinstance(trajs, torch.Tensor) and trajs.requires_grad):
            with torch.no_grad():
                _, params = self._fit(trajs, want_tokens=False)
                if update_bounds:
                    self.update_weights_bounds_per_batch(params)
                return self._normalize(params), self._params_dict(params)
        plan = self._plan()
        x = self._prep_trajs(trajs, plan.device)          # differentiable: .to() / slicing / .contiguous()

        def fit(x):
            _, params = self._fit(x, want_tokens=False)
            if update_bounds:
                self.update_weights_bounds_per_batch(params)
            normalised = self._normalize(params)
            # the bounds this call normalised with: a later update_weights_bounds* changes the buffers in place
            lo, hi = self._bounds(plan.device)
            return normalised, params, (lo.clone(), hi.clone())

        normalised, params = _FitFn.apply(fit, plan, x)
        st = self._boundary_state(x, plan) if self._has_conditions else None
        return normalised, self._params_dict(params, st)

    def _normalize(self, params):
        plan = self._plan()
        dev = plan.device
        params = params.to(dev, torch.float32).contiguous()
        lo, hi = self._bounds(dev)
        out = torch.empty_like(params)
        with torch.cuda.device(dev):
            _lib.check(plan._lib.beast_normalize_f32(plan.handle, _lib.ptr(params), params.shape[0], _lib.ptr(lo),
                                                     _lib.ptr(hi), _lib.ptr(out), _lib.stream_ptr(dev)),
                       "beast_normalize_f32")
        return out

    # ------------------------------------------------------------------ LLM token helpers
    def tokens_to_llm_tokens(self, tokens):
        tokens = tokens.to(self._buffer_device())
        if len(tokens.shape) == 3:
            tokens = tokens.reshape(tokens.shape[0], -1)
        if self.llm_vocab_size is None:
            raise ValueError("LLM vocab size is not set.")
        return tokens + self._llm_vocab_offset()

    def llm_tokens_to_mp_tokens(self, llm_tokens):
        if self.llm_vocab_size is None:
            raise ValueError("LLM vocab size is not set.")
        tokens = llm_tokens - self._llm_vocab_offset()
        if len(tokens.shape) == 2:
            tokens = tokens.reshape(tokens.shape[0], self.num_basis, self.num_dof)
        return tokens

    # ------------------------------------------------------------------ decoding
    def reconstruct_from_llm_tokens(self, llm_tokens, times=None, **kwargs):
        tokens = self.llm_tokens_to_mp_tokens(llm_tokens)
        return self.reconstruct_traj(tokens, times=times, **kwargs)

    def _flatten_tokens(self, tokens, dev):
        tokens = tokens.to(dev)
        if tokens.dim() == 3:
            tokens = tokens.reshape(tokens.shape[0], -1)
        elif tokens.dim() != 2:
            raise ValueError(f"Unexpected token shape {tokens.shape}")
        return tokens.to(torch.int64).contiguous()

    @torch.no_grad()
    def decode(self, tokens, *, respect_llm_vocab_size=True):
        """tokens -> coefficients [B, D*nb] '(d t)' (reference :483-496)."""
        plan = self._plan()
        dev = plan.device
        tokens = self._flatten_tokens(tokens, dev)
        offset = self._llm_vocab_offset() if (respect_llm_vocab_size and self.llm_vocab_size is not None) else 0
        lo, hi = self._bounds(dev)
        out = torch.empty(tokens.shape, device=dev, dtype=torch.float32)
        with torch.cuda.device(dev):
            _lib.check(plan._lib.beast_dequantize_f32(plan.handle, _lib.ptr(tokens), tokens.shape[0], _lib.ptr(lo),
                                                      _lib.ptr(hi), int(offset), _lib.ptr(out),
                                                      _lib.stream_ptr(dev)), "beast_dequantize_f32")
        return out

    def _init_p(self, kwargs, dev, batch):
        init_p = kwargs.get("init_p") if self.init_pos else None
        if init_p is None:
            return None
        init_p = torch.as_tensor(init_p).to(dev, torch.float32)
        if init_p.dim() != 2 or init_p.shape[0] != batch or init_p.shape[1] < self.num_dof:
            raise IndexError(f"init_p must be [batch, >= num_dof], got {tuple(init_p.shape)}")
        return init_p[:, :self.num_dof].contiguous()

    def _check_times(self, times, dev, batch):
        times = torch.as_tensor(times).to(dev, torch.float32)
        if times.dim() != 2 or times.shape[0] != batch:
            raise AssertionError(f"times must be [batch, T'], got {tuple(times.shape)}")
        return times.contiguous()

    @torch.no_grad()
    def reconstruct_traj(self, tokens, times=None, **kwargs):
        """tokens -> trajectories [B, T, D] (reference :498-536): one fused K3 launch."""
        offset = self._llm_vocab_offset() if self.llm_vocab_size is not None else 0   # decode() default
        return self._reconstruct_from_mp_tokens(tokens, offset, times, **kwargs)

    def _reconstruct_from_mp_tokens(self, tokens, offset, times=None, **kwargs):
        plan = self._plan()
        dev = plan.device
        tokens = self._flatten_tokens(tokens, dev)
        B = tokens.shape[0]
        lo, hi = self._bounds(dev)
        init_p = self._init_p(kwargs, dev, B)
        bc, bias = self._pinned(B)
        with torch.cuda.device(dev):
            if bc is not None:
                tq = 0
                if times is not None:
                    times = self._check_times(times, dev, B)
                    tq = times.shape[1]
                out = torch.empty((B, tq if times is not None else plan.consts.seq_len, self.num_dof), device=dev,
                                  dtype=torch.float32)
                _lib.check(plan._lib.beast_reconstruct_bc_f32(
                    plan.handle, _lib.ptr(tokens), None, B, _lib.ptr(lo), _lib.ptr(hi), int(offset), _lib.ptr(init_p),
                    _lib.ptr(times), tq, _lib.ptr(bc), _lib.ptr(bias), _lib.ptr(out), _lib.stream_ptr(dev)),
                    "beast_reconstruct_bc_f32")
            elif times is None:
                out = torch.empty((B, plan.consts.seq_len, self.num_dof), device=dev, dtype=torch.float32)
                _lib.check(plan._lib.beast_decode_f32(plan.handle, _lib.ptr(tokens), B, _lib.ptr(lo), _lib.ptr(hi),
                                                      int(offset), _lib.ptr(init_p), _lib.ptr(out),
                                                      _lib.stream_ptr(dev)), "beast_decode_f32")
            else:
                times = self._check_times(times, dev, B)
                out = torch.empty((B, times.shape[1], self.num_dof), device=dev, dtype=torch.float32)
                _lib.check(plan._lib.beast_decode_times_f32(plan.handle, _lib.ptr(tokens), B, _lib.ptr(lo),
                                                            _lib.ptr(hi), int(offset), _lib.ptr(init_p),
                                                            _lib.ptr(times), times.shape[1], _lib.ptr(out),
                                                            _lib.stream_ptr(dev)), "beast_decode_times_f32")
        return out

    def _continuous_needs_grad(self, params, kwargs) -> bool:
        """Grad mode is on and `params` or a used init_p requires grad: the continuous decode is then recorded."""
        if not torch.is_grad_enabled():
            return False
        init_p = kwargs.get("init_p") if self.init_pos else None
        return any(isinstance(t, torch.Tensor) and t.requires_grad for t in (params, init_p))

    def reconstruct_traj_continuous(self, params, times=None, **kwargs):
        """Normalised '(t d)' coefficients -> trajectories (reference :538-582).  Upstream this
        method raises TypeError (beast/utils.py:42 clamps a Python float); here it works.

        Differentiable with respect to `params` and `init_p` (when `params` or `init_p` requires grad under grad
        mode): the backward is beast_decode_grid_backward_f32 (times None) / beast_decode_deriv_times_backward_f32
        (times [B, T']).  `times`, the condition-order boundary state and w_min / w_max as the kernels see them are
        constants; the clamp of the normalised coefficients passes no gradient where |params| > 1."""
        if not self._continuous_needs_grad(params, kwargs):
            with torch.no_grad():
                return self._reconstruct_continuous(params, times, kwargs, False)
        return self._reconstruct_continuous(params, times, kwargs, True)

    def _reconstruct_continuous(self, params, times, kwargs, grad):
        plan = self._plan()
        dev = plan.device
        params = self._denormalize_continuous(params, dev)
        B = params.shape[0]
        init_p = self._init_p(kwargs, dev, B)
        tq = 0
        if times is not None:
            times = self._check_times(times, dev, B)
            tq = times.shape[1]
        bc, bias = self._pinned(B)

        def decode(params, init_p):
            out = torch.empty((B, tq if times is not None else plan.consts.seq_len, self.num_dof), device=dev,
                              dtype=torch.float32)
            with torch.cuda.device(dev):
                if bc is not None:
                    _lib.check(plan._lib.beast_reconstruct_bc_f32(
                        plan.handle, None, _lib.ptr(params), B, None, None, 0, _lib.ptr(init_p), _lib.ptr(times), tq,
                        _lib.ptr(bc), _lib.ptr(bias), _lib.ptr(out), _lib.stream_ptr(dev)), "beast_reconstruct_bc_f32")
                else:
                    _lib.check(plan._lib.beast_eval_f32(plan.handle, _lib.ptr(params), B, _lib.ptr(init_p),
                                                        _lib.ptr(times), tq, _lib.ptr(out), _lib.stream_ptr(dev)),
                               "beast_eval_f32")
            return (out,)

        if not grad:
            return decode(params, init_p)[0]
        # the positions on the tokenizer's own times are the order-0 rows of its grid bit for bit
        grid = self._grid(plan, self.times.contiguous(), 0) if times is None else None
        adjoint = _Adjoint(plan, B, (0,), grid, times, tq if times is not None else plan.consts.seq_len,
                           init_p is not None)
        return _SplineDecodeFn.apply(decode, adjoint, params, init_p)[0]

    def _denormalize_continuous(self, params, dev):
        """Normalised '(t d)' coefficients -> de-normalised '(d t)' coefficients [B, D*nb] on `dev`."""
        from .utils import denormalize_tensor
        params = params.to(dev)
        if len(params.shape) == 3:
            params = params.reshape(params.shape[0], -1)
        if params.shape[-1] != self.num_basis * self.num_dof:
            raise ValueError(
                f"Token dimension {params.shape[-1]} does not match expected {self.num_basis * self.num_dof}.")
        B = params.shape[0]
        n = self.num_basis * self.num_dof
        params = params.reshape(B, self.num_basis, self.num_dof).transpose(1, 2).reshape(B, n)
        lo, hi = self._bounds(dev)
        return denormalize_tensor(params.to(torch.float32), w_min=lo, w_max=hi).contiguous()

    # ------------------------------------------------------------------ derivatives
    @torch.no_grad()
    def reconstruct_traj_derivatives(self, tokens, times=None, orders=(0, 1, 2), **kwargs):
        """tokens -> (d^o/dt^o of the decoded trajectory for o in `orders`), each fp32 [B, Tq, num_dof].

        Order 0 is reconstruct_traj's position bit for bit, orders 1 / 2 velocity and acceleration in the units of
        `times` (exact spline derivatives; one-sided at t = 0 and t = duration, right-hand at an interior knot,
        exactly 0 outside [0, duration] and for gripper slots).  `times`: None (the tokenizer's own times), one grid
        [Tq] shared by every trajectory, or [B, Tq] per trajectory.  Tokens, the LLM offset, init_p and the
        condition-order state behave as in reconstruct_traj."""
        orders = check_orders(orders)
        offset = self._llm_vocab_offset() if self.llm_vocab_size is not None else 0   # as reconstruct_traj
        return self._derivatives_from_mp_tokens(tokens, offset, times, orders, **kwargs)

    def reconstruct_traj_continuous_derivatives(self, params, times=None, orders=(0, 1, 2), **kwargs):
        """reconstruct_traj_derivatives from the normalised coefficients of encode_continuous.

        Differentiable with respect to `params` and `init_p` (when either requires grad under grad mode), for every
        form of `times` and any subset of `orders`: the backward is beast_decode_grid_backward_f32 on the grid the
        forward used (times None or [Tq]) / beast_decode_deriv_times_backward_f32 (times [B, Tq]).  `times`, the
        condition-order boundary state and w_min / w_max as the kernels see them are constants; the clamp of the
        normalised coefficients passes no gradient where |params| > 1."""
        orders = check_orders(orders)
        if not self._continuous_needs_grad(params, kwargs):
            with torch.no_grad():
                plan = self._plan()
                params = self._denormalize_continuous(params, plan.device)
                return self._derivatives(plan, None, params, None, None, 0, times, orders, kwargs)
        plan = self._plan()
        params = self._denormalize_continuous(params, plan.device)
        return self._derivatives(plan, None, params, None, None, 0, times, orders, kwargs, grad=True)

    def _derivatives_from_mp_tokens(self, tokens, offset, times, orders, **kwargs):
        plan = self._plan()
        dev = plan.device
        tokens = self._flatten_tokens(tokens, dev)
        lo, hi = self._bounds(dev)
        return self._derivatives(plan, tokens, None, lo, hi, offset, times, orders, kwargs)

    def _derivatives(self, plan, tokens, params, lo, hi, offset, times, orders, kwargs, grad=False):
        dev = plan.device
        B = (tokens if tokens is not None else params).shape[0]
        init_p = self._init_p(kwargs, dev, B)
        bc, bias = self._pinned(B)
        shared = times is None or torch.as_tensor(times).dim() == 1
        if shared:                                  # one grid for every trajectory: the tiled kernel
            grid_t = self.times if times is None else torch.as_tensor(times).detach().to("cpu", torch.float32)
            grid_t = grid_t.contiguous()
            tq = grid_t.numel()
        else:
            times = self._check_times(times, dev, B)
            tq = times.shape[1]
        grid = self._grid(plan, grid_t, max(orders)) if shared and B > 0 and tq > 0 else None

        def decode(params, init_p):
            outs = {o: torch.empty((B, tq, self.num_dof), device=dev, dtype=torch.float32) for o in orders}
            o0, o1, o2 = (_lib.ptr(outs.get(o)) for o in range(3))
            if B == 0 or tq == 0:
                return tuple(outs[o] for o in orders)
            with torch.cuda.device(dev):
                if shared:
                    _lib.check(plan._lib.beast_decode_grid_f32(
                        plan.handle, grid.handle, _lib.ptr(tokens), _lib.ptr(params), B, _lib.ptr(lo), _lib.ptr(hi),
                        int(offset), _lib.ptr(init_p), _lib.ptr(bc), _lib.ptr(bias), o0, o1, o2,
                        _lib.stream_ptr(dev)), "beast_decode_grid_f32")
                else:
                    _lib.check(plan._lib.beast_decode_deriv_times_f32(
                        plan.handle, _lib.ptr(tokens), _lib.ptr(params), B, _lib.ptr(lo), _lib.ptr(hi), int(offset),
                        _lib.ptr(init_p), _lib.ptr(times), tq, _lib.ptr(bc), _lib.ptr(bias), o0, o1, o2,
                        _lib.stream_ptr(dev)), "beast_decode_deriv_times_f32")
            return tuple(outs[o] for o in orders)

        if not grad:
            return decode(params, init_p)
        adjoint = _Adjoint(plan, B, orders, grid, None if shared else times, tq, init_p is not None)
        return _SplineDecodeFn.apply(decode, adjoint, params, init_p)

    # ------------------------------------------------------------------ evaluation
    def _no_plotting(self, name):
        raise NotImplementedError(
            f"{name} is matplotlib plotting around encode -> reconstruct_traj (reference beast_bspline_tokenizer.py:600-720), "
            "outside the B200 hot path; use compute_reconstruction_error(raw_traj, return_tokens=True) and plot the result")

    def visualize_reconstruction_error(self, raw_traj, max_vis_samples=5, update_bounds=True, save_path=None):
        self._no_plotting("visualize_reconstruction_error")

    def visualize_reconstruction_error_with_llm_tokenizer(self, raw_traj, save_path=None):
        self._no_plotting("visualize_reconstruction_error_with_llm_tokenizer")

    def visualize_reconstruction_error_with_cont_tokenizer(self, raw_traj, save_path=None):
        self._no_plotting("visualize_reconstruction_error_with_cont_tokenizer")

    def compute_reconstruction_error(self, raw_traj, return_tokens: bool = False):
        """(mean squared error, mean signed error) of encode -> reconstruct (reference :589-597).
        `return_tokens=True` also returns the tokens — the call train/eval.py:34 makes upstream, where
        the one-argument signature makes it fail."""
        raw_traj = raw_traj.to(self._cuda(), dtype=torch.float32)
        if len(raw_traj.shape) == 2:
            raw_traj = raw_traj.unsqueeze(0)
        tokens = self.encode(raw_traj)[0]
        reconstruct_trajs = self.reconstruct_traj(tokens)
        error_l2 = torch.mean((raw_traj - reconstruct_trajs) ** 2)
        error_l1 = torch.mean(raw_traj - reconstruct_trajs)
        if return_tokens:
            return error_l2, error_l1, tokens
        return error_l2, error_l1
