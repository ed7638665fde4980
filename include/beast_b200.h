/*
 * beast_b200.h — C ABI of libbeast_b200.so: the B200 (sm_100a) implementation of the
 * BEAST tokenizer hot path.
 *
 * The reference (Dont4rootMe/beast_tokenizer) has no FFI layer: the path sits behind plain
 * Python classes.  Each entry point below replaces the torch/numpy/`tokenizers` call
 * sequence of one reference method; the Python classes in beast_tokenizer_b200/ (same names
 * and signatures as the reference's) are the only callers.  Citations are relative to the
 * reference tree.
 *
 * Conventions
 *   - every function returns int: 0 = ok, <0 = BEAST_E_* argument error, >0 = cudaError_t;
 *   - nothing throws, nothing synchronises the device, nothing allocates device memory
 *     except beast_plan_create (small constant tables, freed by beast_plan_destroy);
 *   - the caller owns every buffer and passes its stream (cudaStream_t as void*);
 *   - pointers are DEVICE pointers unless the name ends in _h;
 *   - a plan is immutable after creation: calls on it are thread-safe per stream.
 */
#ifndef BEAST_B200_H
#define BEAST_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BEAST_MAX_DOF 64

enum {
    BEAST_OK = 0,
    BEAST_E_NULL = -1,       /* required pointer is NULL */
    BEAST_E_SHAPE = -2,      /* bad size / dimension */
    BEAST_E_ALIGN = -3,      /* pointer not aligned for its element type */
    BEAST_E_UNSUPPORTED = -4,
    BEAST_E_NOMEM = -5
};

/* Geometry of one tokenizer (constructor arguments of BEASTBsplineTokenizer,
 * beast/beast_bspline_tokenizer.py:47-116) plus the precomputed constant tables.
 * All table pointers are HOST pointers, copied at plan creation.
 *   slot_to_dof_h[num_dof] : joint_indices followed by gripper_indices (:56-70, :351-358)
 *   proj_joint_h [num_basis*seq_len] row-major [k][t] : P = (Phi^T Phi + 1e-9 I)^-1 Phi^T, the
 *        closed form of the ridge solve at MP_lite_PyTorch/mp_pytorch/mp/uni_bspline.py:559-586
 *   proj_grip_h  same for the degree-0 gripper spline (NULL when n_joint == num_dof)
 *   phi_joint_h  [seq_len*num_ctrlp] row-major [t][c] : basis at the tokenizer's own times
 *        (basis_gn/uni_bspline_basis.py:59-113), num_ctrlp = num_basis + init_cond_order +
 *        end_cond_order (:40); phi_grip_h [seq_len*num_basis] likewise (NULL if no grippers)
 *   knots_joint_h [num_ctrlp+degree_p+1], knots_grip_h [num_basis+1] : knot vectors (:48-55),
 *        used when the caller supplies its own evaluation times.
 *   init_cond_order / end_cond_order (0, 1 or 2): how many leading / trailing control points of
 *        every JOINT spline are pinned by boundary conditions instead of being tokens
 *        (mp/uni_bspline.py:500-537).  proj_joint_h then already folds the conditions in
 *        (they are linear in the trajectory); decode takes the pinned points per trajectory
 *        through beast_reconstruct_bc_f32. */
typedef struct beast_plan_desc {
    int32_t seq_len;
    int32_t num_dof;
    int32_t num_basis;
    int32_t n_joint;
    int32_t degree_p;
    int32_t vocab_size;
    float   tau;            /* fp32(duration): phase = clip(t / tau, 0, 1), linear_phase.py:22-23 */
    const int32_t* slot_to_dof_h;
    const float* proj_joint_h;
    const float* proj_grip_h;
    const float* phi_joint_h;
    const float* phi_grip_h;
    const float* knots_joint_h;
    const float* knots_grip_h;
    int32_t init_cond_order;
    int32_t end_cond_order;
} beast_plan_desc_t;

typedef struct beast_plan beast_plan_t;

int beast_plan_create(const beast_plan_desc_t* desc, beast_plan_t** plan_out);
int beast_plan_destroy(beast_plan_t* plan);

/* Library / build information: "beast_b200 <version> sm_100a". */
const char* beast_version(void);
/* Number of kernels this library has launched in this process (bench.py's gpu_launches). */
int64_t beast_launch_count(void);
/* Test hook: flag != 0 makes the spline entry points take the one-thread-per-column reference kernels only (as
 * BEAST_B200_DISABLE_FAST=1 does from the environment); returns the previous setting.  The parity tests compare the
 * tiled / bulk-copy kernels with them bit for bit. */
int beast_debug_disable_fast(int32_t flag);
/* Number of bulk-copy K1 / K3 launches made so far that may overlap the launch before them (they stream while it
 * drains).  Only launches captured into a CUDA graph overlap, and only directly after the previous bulk-copy K1 / K3
 * launch of this library on the same stream when the two touch disjoint memory. */
int64_t beast_overlap_count(void);
/* Test hook: flag != 0 makes every bulk-copy K1 / K3 launch wait for the launch before it (no overlap); returns the
 * previous setting. */
int beast_debug_force_wait(int32_t flag);
/* Test hook: the hazard predicate of the overlap.  prev / next hold n_prev / n_next triples (first byte, end byte,
 * written != 0) of two launches; returns 1 on a read-after-write, write-after-read or write-after-write conflict,
 * 0 otherwise (touching and empty ranges never conflict). */
int beast_debug_ranges_conflict(const int64_t* prev, int32_t n_prev, const int64_t* next, int32_t n_next);

/* ---- K1: fused fit + quantise.  Replaces BEASTBsplineTokenizer.encode
 * (beast/beast_bspline_tokenizer.py:399-428) and compute_weights (:344-360):
 *   traj   [B, seq_len, num_dof] fp32
 *   params_out [B, num_dof*num_basis] fp32, UNclamped, '(d t)' slot layout     (nullable)
 *   tokens_out [B, num_basis*num_dof] int64, '(t d)' layout, + offset           (nullable)
 *   w_min / w_max [num_dof*num_basis] fp32 ('(d t)'); required when tokens_out != NULL
 *   offset = llm_vocab_size - vocab_size or 0 (:424-426). */
int beast_encode_f32(const beast_plan_t* plan, const float* traj, int64_t B,
                     const float* w_min, const float* w_max, int64_t offset,
                     float* params_out, int64_t* tokens_out, void* stream);

/* Quantise given coefficients (the bit-exact contract of beast/utils.py:4-17 applied as in
 * beast_bspline_tokenizer.py:419-426): params [B, D*nb] '(d t)' -> tokens [B, nb*D] '(t d)'. */
int beast_quantize_f32(const beast_plan_t* plan, const float* params, int64_t B,
                       const float* w_min, const float* w_max, int64_t offset,
                       int64_t* tokens_out, void* stream);

/* encode_continuous (:430-450, utils.py:29-35): params -> normalised [-1,1] '(t d)' fp32. */
int beast_normalize_f32(const beast_plan_t* plan, const float* params, int64_t B,
                        const float* w_min, const float* w_max, float* out, void* stream);

/* ---- K3: fused dequantise + spline evaluation.  Replaces decode (:483-496) +
 * reconstruct_traj (:498-536) + UniformBSpline.get_traj_pos (mp/uni_bspline.py:114-177):
 *   tokens [B, nb*D] int64 '(t d)';  init_p [B, num_dof] fp32 or NULL (first control point
 *   of every JOINT slot := init_p[:, dof], :505-510);  traj_out [B, seq_len, num_dof] fp32. */
int beast_decode_f32(const beast_plan_t* plan, const int64_t* tokens, int64_t B,
                     const float* w_min, const float* w_max, int64_t offset,
                     const float* init_p, float* traj_out, void* stream);

/* Same with caller-supplied evaluation times [B, Tq] (reconstruct_traj(times=...)):
 * the basis is evaluated in-kernel (Cox-de Boor, same fp32 op order).  traj_out [B, Tq, num_dof]. */
int beast_decode_times_f32(const beast_plan_t* plan, const int64_t* tokens, int64_t B,
                           const float* w_min, const float* w_max, int64_t offset,
                           const float* init_p, const float* times, int32_t Tq,
                           float* traj_out, void* stream);

/* ---- K3 with pinned control points (init/end condition orders 1, 2).  Replaces
 * UniformBSpline.get_traj_pos when `params_init` / `params_end` are set
 * (MP_lite_PyTorch/mp_pytorch/mp/uni_bspline.py:126-166, as reached from reconstruct_traj /
 * reconstruct_traj_continuous, beast/beast_bspline_tokenizer.py:498-582):
 *   exactly one of tokens [B, nb*D] int64 / params [B, D*nb] fp32 ('(d t)') is non-NULL
 *   bc   [B, n_joint, init_cond_order + end_cond_order] fp32: the pinned control points of every
 *        joint slot (leading ones first), as the reference's MP object holds them after a fit
 *   bias [B, n_joint] fp32 (nullable): added to every sample (the fit's init_pos)
 *   times [B, Tq] (nullable: the plan's own times, Tq ignored)
 * A plan with both orders 0 accepts bc = bias = NULL and then equals beast_decode_times_f32 /
 * beast_eval_f32. */
int beast_reconstruct_bc_f32(const beast_plan_t* plan, const int64_t* tokens, const float* params, int64_t B,
                             const float* w_min, const float* w_max, int64_t offset, const float* init_p,
                             const float* times, int32_t Tq, const float* bc, const float* bias,
                             float* traj_out, void* stream);

/* decode() alone (:483-496, utils.py:20-26): tokens -> coefficients [B, D*nb] '(d t)'. */
int beast_dequantize_f32(const beast_plan_t* plan, const int64_t* tokens, int64_t B,
                         const float* w_min, const float* w_max, int64_t offset,
                         float* params_out, void* stream);

/* Evaluate given coefficients (reconstruct_traj_continuous after denormalise, :549-582):
 * params [B, D*nb] '(d t)' (already de-normalised) -> traj_out. times/Tq as above or NULL/0. */
int beast_eval_f32(const beast_plan_t* plan, const float* params, int64_t B,
                   const float* init_p, const float* times, int32_t Tq,
                   float* traj_out, void* stream);

/* ---- Derivatives of the decoded spline: position, velocity and acceleration (orders 0, 1, 2) on any time grid.
 *   x^(o)(t) = (1/tau)^o * sum_k N_k^(o)(u(t)) * c_k (+ bias for order 0),  u = clip(t / tau, 0, 1),
 * with the coefficients of beast_decode_f32 / beast_reconstruct_bc_f32 (tokens or params, init_p, pinned points).
 * Order 0 equals beast_decode_times_f32 / beast_reconstruct_bc_f32 on the same times bit for bit.  Orders 1 / 2 are
 * d/dt and d2/dt2 in the units of the times: bias does not contribute, intervals are half-open with the last one
 * closed (right-hand derivative at an interior knot, one-sided at t = 0 and t = tau), and outside [0, tau] (phase
 * clamped, position held) they are exactly 0, as are the orders 1 / 2 of degree-0 (gripper) slots.
 *
 * A grid: immutable device tables for one time grid [n_times] shared by every trajectory.
 *   times_h      [n_times] fp32 (host)
 *   rows_joint_h [max_order+1][n_times][num_ctrlp] fp32 (host): d^o/dt^o of the joint basis at the times, from
 *                basis.py: bspline_basis_derivatives (num_ctrlp = num_basis + init_cond_order + end_cond_order)
 *   rows_grip_h  [max_order+1][n_times][num_basis] likewise for the degree-0 gripper basis (NULL without grippers)
 * beast_grid_create allocates and copies (it synchronises); the grid belongs to `plan` and must be destroyed before
 * it.  Decoding with a grid reads only the tokens some row of the grid reads. */
typedef struct beast_grid_desc {
    int32_t n_times;
    int32_t max_order;       /* 0, 1 or 2: the highest order the grid can decode */
    const float* times_h;
    const float* rows_joint_h;
    const float* rows_grip_h;
} beast_grid_desc_t;

typedef struct beast_grid beast_grid_t;

int beast_grid_create(const beast_plan_t* plan, const beast_grid_desc_t* desc, beast_grid_t** grid_out);
int beast_grid_destroy(beast_grid_t* grid);

/* Orders 0..2 on a grid: exactly one of tokens [B, nb*D] int64 '(t d)' / params [B, D*nb] fp32 '(d t)' (already
 * de-normalised) is non-NULL; w_min / w_max / offset as beast_decode_f32 (tokens only); init_p [B, num_dof] or NULL;
 * bc / bias as beast_reconstruct_bc_f32 (required / nullable when the plan pins control points, else ignored).
 * outO [B, n_times, num_dof] fp32 receives order O; any of them may be NULL, at least one is set, and none above
 * the grid's max_order.  Without pinned points one tiled kernel writes every requested order in one pass over the
 * tokens; with pinned points (or beast_debug_disable_fast) the generic kernel evaluates the basis in-kernel. */
int beast_decode_grid_f32(const beast_plan_t* plan, const beast_grid_t* grid, const int64_t* tokens,
                          const float* params, int64_t B, const float* w_min, const float* w_max, int64_t offset,
                          const float* init_p, const float* bc, const float* bias,
                          float* out0, float* out1, float* out2, void* stream);

/* Same with per-trajectory times [B, Tq]: one thread per (trajectory, sample) runs the de Boor recursion in-kernel
 * and takes orders 1 / 2 from the levels below the top one.  BEAST_E_UNSUPPORTED when num_ctrlp + degree_p + 1 > 320.
 * outO [B, Tq, num_dof]. */
int beast_decode_deriv_times_f32(const beast_plan_t* plan, const int64_t* tokens, const float* params, int64_t B,
                                 const float* w_min, const float* w_max, int64_t offset, const float* init_p,
                                 const float* times, int32_t Tq, const float* bc, const float* bias,
                                 float* out0, float* out1, float* out2, void* stream);

/* ---- Adjoint of the two calls above for given coefficients (reconstruct_traj_continuous(_derivatives) backward):
 *   grad_params[b, slot, k] = sum_t sum_o R_o[t, k] * gradO[b, t, dof(slot)]
 * with R_o the rows the forward multiplies coefficient k of that slot with (joint basis for joint slots; the degree-0
 * basis and order 0 only for gripper slots, whose orders 1 / 2 are 0).  gradO [B, n_times (Tq), num_dof] fp32 is the
 * gradient of outO, NULL = zero (at least one is set, none above the grid's max_order).  grad_params [B, D*nb]
 * '(d t)' receives the gradient of params.  Pinned control points, bias and the times are constants: with pinned
 * points only the nb free columns exist in params.  init_p_used != 0: the forward took init_p (coefficient 0 of every
 * joint slot := init_p[b, dof]); that entry of grad_params is then 0 and grad_init_p [B, num_dof] (nullable; NULL
 * unless init_p_used) receives it, 0 for gripper DoFs.  Every element of grad_params / grad_init_p is written (no
 * accumulation, no memset needed).  Deterministic, no atomics: each element is one fp32 sum over t ascending and, for
 * each t, the orders ascending (fmaf); terms with an exactly-zero basis value may be skipped, which does not change
 * the value for finite gradients, so the tiled and generic kernels agree.  On a grid without pinned points a tiled
 * kernel streams the gradients through shared memory once; otherwise (and under beast_debug_disable_fast) the generic
 * kernel evaluates the basis in-kernel.  Per-row times: BEAST_E_UNSUPPORTED when num_ctrlp + degree_p + 1 > 320. */
int beast_decode_grid_backward_f32(const beast_plan_t* plan, const beast_grid_t* grid, int64_t B,
                                   const float* grad0, const float* grad1, const float* grad2, int32_t init_p_used,
                                   float* grad_params, float* grad_init_p, void* stream);
int beast_decode_deriv_times_backward_f32(const beast_plan_t* plan, int64_t B, const float* times, int32_t Tq,
                                          const float* grad0, const float* grad1, const float* grad2,
                                          int32_t init_p_used, float* grad_params, float* grad_init_p, void* stream);

/* ---- Adjoint of beast_encode_f32's coefficients (+ beast_normalize_f32) for encode_continuous backward:
 *   g_w[b, slot, k] = grad_params[b, slot*nb + k]
 *                   + (w_min[c] <= w <= w_max[c] ? (grad_norm[b, k*D + slot] * 2) / max(w_max[c] - w_min[c], 1e-8) : 0)
 *   grad_traj[b, t, dof(slot)] = sum_k P_s[k, t] * g_w[b, slot, k]
 * with c = slot*nb + k, w = params[b, c] the UNclamped forward coefficient, w_min / w_max [D*nb] the bounds the
 * forward normalised with (inclusive: torch's clamp rule; each operation one fp32 rounding, in the order written) and
 * P_s the fp32 projector K1 multiplies with (joint: proj_joint_h, which folds in the condition orders; gripper slots:
 * the degree-0 proj_grip_h).  grad_norm [B, nb*D] '(t d)' and grad_params [B, D*nb] '(d t)' are nullable (NULL =
 * zero, at least one is set); params, w_min and w_max are required with grad_norm.  grad_traj [B, seq_len, num_dof]
 * fp32: every element is written (no accumulation, no memset needed).  Deterministic, no atomics: each element is
 * one fp32 sum over k ascending (fmaf); terms with an exactly-zero projector entry may be skipped, which does not
 * change the value for finite gradients, so the two kernels agree.  NaN inputs are not treated specially.
 * Dispatch: a tiled kernel (persistent CTAs over tiles of trajectories, only the coefficients of non-empty projector
 * rows loaded; the projector in shared memory when its column sums have more than two terms and it fits in 32 KB, else
 * read through L1) whenever one trajectory's coefficients and the tables fit in shared memory; otherwise, and under
 * beast_debug_disable_fast, a generic one-thread-per-element kernel. */
int beast_fit_backward_f32(const beast_plan_t* plan, int64_t B, const float* grad_norm, const float* grad_params,
                           const float* params, const float* w_min, const float* w_max, float* grad_traj,
                           void* stream);

/* ---- Fit on per-row times (encode / encode_continuous / compute_weights with times [B, T]).
 * Row b solves its own ridge system on Phi_b = the basis at times[b] (phase clip(t / tau, 0, 1), the rows the per-row
 * decode evaluates): joint slots w = (Phi_f^T Phi_f + 1e-9 I)^-1 Phi_f^T (y - bias - Phi_pin bc) on the nb free
 * columns, gripper slots the same on the degree-0 basis.  traj [B, T, num_dof] and times [B, T] fp32, T >= 1 (>= 2
 * when the plan pins control points) and independent of seq_len; times need not be sorted and are clamped to
 * [0, tau] like the decode's; NaN and repeated first times (dt = 0 upstream) are not treated specially.  bc
 * [B, n_joint, init_cond_order + end_cond_order] (required when the plan pins points, else ignored) and bias
 * [B, n_joint] (nullable) as beast_reconstruct_bc_f32 takes them.  params_out [B, D*nb] '(d t)' unclamped.  Gram
 * matrix, right-hand sides, band Cholesky and solves in fp64, one fp32 rounding per output; a coefficient whose basis
 * function holds no sample is exactly 0.  Each element depends only on its row (no atomics, fixed summation order).
 * BEAST_E_UNSUPPORTED when num_ctrlp + degree_p + 1 > 320 (as the per-row decode).  Tokens: beast_quantize_f32. */
int beast_fit_times_f32(const beast_plan_t* plan, const float* traj, int64_t B, int32_t T, const float* times,
                        const float* bc, const float* bias, float* params_out, void* stream);
/* Its adjoint: g_w exactly as beast_fit_backward_f32 forms it (same arguments and nullability), v = G_b^-1 g_w and
 * u = Phi_f v per row; grad_traj [B, T, num_dof] = u, grad_bc = -Phi_pin^T u (required when the plan pins points) and
 * grad_bias [B, n_joint] = -sum_t u (nullable).  Every element of the given outputs is written; no atomics. */
int beast_fit_times_backward_f32(const beast_plan_t* plan, int64_t B, int32_t T, const float* times,
                                 const float* grad_norm, const float* grad_params, const float* params,
                                 const float* w_min, const float* w_max, float* grad_traj, float* grad_bc,
                                 float* grad_bias, void* stream);

/* ---- Masked fit (encode / encode_continuous / compute_weights / update_weights_bounds with mask [B, T]).
 * mask [B, T] bytes, non-zero = the sample is fitted (LeRobot's action_is_pad is its negation).  Row b is fitted as
 * beast_fit_times_f32 fits the compacted row y[b, mask[b]] on times[b, mask[b]], bit for bit: same fp64 Gram matrix,
 * right-hand sides, band Cholesky, single fp32 rounding and t-ascending order.  A masked sample's time and trajectory
 * value are never read and add no term anywhere.  times_row_stride is T (times [B, T]) or 0 (one grid [T] for every
 * row); any other value is BEAST_E_SHAPE.  bc / bias are the row's boundary state computed from its valid samples.
 * A row without valid samples gets exactly 0 (without pinned points); with pinned points a row with fewer than two
 * valid samples is not treated specially.  partial_only != 0: a row whose mask is all non-zero is skipped and its
 * outputs are left untouched (the shared-grid path lets K1 write those rows first).  NULL mask is BEAST_E_NULL;
 * the other NULL, shape, alignment and support rules are beast_fit_times_f32's.  An ordinary launch. */
int beast_fit_masked_f32(const beast_plan_t* plan, const float* traj, int64_t B, int32_t T, const float* times,
                         int64_t times_row_stride, const uint8_t* mask, int32_t partial_only, const float* bc,
                         const float* bias, float* params_out, void* stream);
/* Its adjoint, as beast_fit_times_backward_f32 on the compacted row: masked samples get grad_traj exactly 0 and add
 * nothing to grad_bc / grad_bias.  With partial_only, rows whose mask is all non-zero are left untouched in every
 * output (grad_traj, grad_bc, grad_bias). */
int beast_fit_masked_backward_f32(const beast_plan_t* plan, int64_t B, int32_t T, const float* times,
                                  int64_t times_row_stride, const uint8_t* mask, int32_t partial_only,
                                  const float* grad_norm, const float* grad_params, const float* params,
                                  const float* w_min, const float* w_max, float* grad_traj, float* grad_bc,
                                  float* grad_bias, void* stream);

/* ---- K2: bounds.
 * Column min/max of x [rows, cols] (update_weights_bounds :377-378; the reduction inside
 * update_weights_bounds_per_batch :382-383).  accumulate != 0 folds into the existing
 * contents of min_out / max_out (used when the rows arrive in several batches or shards);
 * accumulate == 0 with rows == 0 leaves min_out = +inf, max_out = -inf.  Any column count
 * cols >= 1 and any 4-byte-aligned x are accepted.  The sign of a zero result is not kept
 * (-0 comes back as +0). */
int beast_minmax_f32(const float* x, int64_t rows, int32_t cols,
                     float* min_out, float* max_out, int32_t accumulate, void* stream);

/* update_weights_bounds fused (:362-378): column min / max of the fitted coefficients straight from the
 * trajectories — K1 without any output but 2 x D*nb floats (2 800 B read per trajectory). */
int beast_fit_minmax_f32(const beast_plan_t* plan, const float* traj, int64_t B, float* min_out,
                         float* max_out, int32_t accumulate, void* stream);
/* Same in ONE launch: with a zero-initialised workspace of beast_fit_minmax_workspace_bytes(plan) bytes (per-CTA
 * partials + a ticket that the kernel resets itself; one workspace per concurrent stream, shared by calls of any batch
 * size) the last CTA to finish
 * combines the partials and writes min_out / max_out with plain stores — no initialisation pass, no float atomics; the
 * destination may be the tokenizer's own w_min / w_max buffers.  workspace == NULL behaves as beast_fit_minmax_f32. */
int64_t beast_fit_minmax_workspace_bytes(const beast_plan_t* plan);
int beast_fit_minmax_ws_f32(const beast_plan_t* plan, const float* traj, int64_t B, float* min_out, float* max_out,
                            int32_t accumulate, void* workspace, int64_t workspace_bytes, void* stream);

/* update_weights_bounds_per_batch (:384-389): w_min[i] = bmin[i] where bmin[i] < w_min[i]-hyst,
 * w_max[i] = bmax[i] where bmax[i] > w_max[i]+hyst. */
int beast_bounds_expand_f32(const float* batch_min, const float* batch_max,
                            float* w_min, float* w_max, int32_t n, float hyst, void* stream);

/* Exact per-column order statistics for fit_parameters' np.quantile (:211-214):
 * x [rows, cols]; for every column c and every j < nk writes the ks_h[j]-th smallest value
 * (0-based) to out[j*cols + c].  scratch: at least beast_colselect_scratch_bytes() bytes. */
int64_t beast_colselect_scratch_bytes(int64_t rows, int32_t cols, int32_t nk);
int beast_colselect_f32(const float* x, int64_t rows, int32_t cols,
                        const int64_t* ks_h, int32_t nk, float* out,
                        void* scratch, void* stream);

/* ---- K4 / K5: byte-level BPE over discretised bins.  Replaces the HF `tokenizers` calls under
 * FIGBPE (beast/beast_bpe_trainer.py:61-98: ByteLevelBPETokenizer + BpeTrainer.train_from_iterator) and
 * BEASTBsplineBPETokenizer._discrete_to_bpe / _bpe_to_discrete (beast/beast_bspline_bpe_tokenizer.py:
 * 175-247: tokenizer.encode(...).ids / tokenizer.decode).  Algorithm: SURVEY.md Appendix A.
 * Corpus layout: chunk-major symbols sym[((p >> 3) * n_stride + seq) * 8 + (p & 7)] (uint16, bit 15 = first
 * symbol of a pre-token, 0xffff padding in the last 8-symbol chunk; ceil(2L / 8) chunks), len[seq] live symbols; sequences may be sharded over GPUs, the V x V pair histogram is
 * replicated.  All functions below take DEVICE pointers.
 *
 * bpe_scan_bins  phase 0: minmax[0] = min(minmax[0], bins), minmax[1] = max(minmax[1], bins)
 *                         (caller initialises to INT64_MAX / INT64_MIN; global min_token / max_token, A.1);
 *                phase 1: seen[b] = 1 for every UTF-8 byte of chr(bin - min_token) (alphabet, A.3);
 *                         *err = 1 if a shifted bin is outside 0..0xD7FF (1 / 2 / 3 UTF-8 bytes per bin).
 * bpe_symbolize  bins [N, L] int64 -> sym / len through the GPT-2 pre-tokeniser (A.2) and the byte-level
 *                expansion (A.3); byte_to_id[256] int16 (-1 = not in the vocabulary: dropped); cls_tab[max
 *                shifted bin + 1] uint8: character class of every codepoint >= 256 (0 other, 1 \p{L}, 2 \p{N}, 3 \s).
 *                row_len [N] int32 (nullable): sequences of unequal length (FIGBPE.fit_from_sequences,
 *                beast/beast_bpe_trainer.py:76-98) arrive padded to L with any in-range value; the text of
 *                sequence s ends at row_len[s].
 * bpe_count_pairs  hist[a*V + b] += #adjacent (a, b) inside pre-tokens (int32, V x V).  Optional hint:
 *                used_ids[n_used] = the distinct ids that can occur in sym (ascending, all < n_ids: the
 *                byte-level symbols before any merge; an id of sym that is missing from the list is NOT counted) —
 *                the count then runs on block-private shared-memory histograms, the rows dealt to up to 8 blocks
 *                per group of sequences when n_used^2 counters do not fit in one; NULL / 0 = global atomics.
 * bpe_argmax     result = count << 32 | (0xffffffff - (a*V + b)) of the best pair (0 if none): maximum
 *                count, ties -> smallest (a, b) (BpeTrainer's heap order).
 * bpe_apply_merge  replace (a, b) by c left to right, non-overlapping, compacting in place; the count
 *                changes are ADDED to delta[4*V] = {column a lost, row b lost, column c gained, row c gained}.
 *                Two kernels: a scan that lists the sequences containing the pair, a rewrite over that list;
 *                work: int32 [4 + 2*N] scratch (list length, sequence ids, first-hit positions).
 * bpe_apply_delta  hist += delta (after the cross-GPU sum when sharded); hist[a][b] = 0; delta = 0.
 * bpe_encode     bins -> ids: per pre-token repeatedly merge the lowest-rank pair, leftmost first (A.5).
 *                rank_tab: hash_bits == 0: dense [a*V + b] = rank << 16 | new_id or 0xffffffff; hash_bits > 0: an
 *                open-addressing hash of the merges only, 2^hash_bits uint2 slots {a << 16 | b, rank << 16 | new_id}, empty
 *                key 0xffffffff, slot = (key * 0x9E3779B1) >> (32 - hash_bits), linear probing (large vocabularies:
 *                O(#merges) memory instead of 4 V^2 bytes).  ids_padded [N, out_stride >= 2L]
 *                uint16, len_out [N], status_out [N]: bit 0 = bin below min_token, bit 1 = bin above
 *                min_token + max_shift (the two range ValueErrors of bpe_tokenizer.py:182-192).
 * bpe_compact    padded rows -> CSR flat int32 (offsets = exclusive scan of len, by the caller).
 * bpe_decode     CSR ids -> bins [N, L] int64 (A.6); status 1 = unknown id, 2 = invalid UTF-8,
 *                3 = decoded length != L (bpe_tokenizer.py:241-244); declen_out = decoded length.
 *                tok_tab (nullable): the per-token character table of the fast path (one lane per token; sequences it
 *                cannot describe are decoded by the byte-level kernel in a second launch).  tok_tab_slots = 6:
 *                16 bytes per token {c0|c1<<16, c2|c3<<16, c4|c5<<16, meta}; tok_tab_slots = 2: 8 bytes {c0|c1<<16, meta}.
 *                c = the token's characters (16-bit codepoints; the last one pre-shifted when it is cut off),
 *                meta = characters started | continuation bytes the last character still needs << 3 | continuation
 *                bytes the token begins with << 5 | not representable << 7 | payload of those leading bytes << 8. */
int bpe_scan_bins(const int64_t* bins, int64_t n, int64_t min_token, int64_t* minmax, int32_t* seen,
                  int32_t* err, int32_t phase, void* stream);
int bpe_symbolize(const int64_t* bins, int64_t N, int32_t L, int64_t min_token, const int16_t* byte_to_id,
                  const uint8_t* cls_tab, uint16_t* sym, int32_t* len, int64_t n_stride, int32_t* err,
                  const int32_t* row_len, void* stream);
int bpe_count_pairs(const uint16_t* sym, const int32_t* len, int64_t N, int64_t n_stride, int32_t V,
                    int32_t n_ids, const int16_t* used_ids, int32_t n_used, int32_t* hist, const int32_t* weight,
                    void* stream);
int bpe_argmax(const int32_t* hist, int32_t V, int32_t n_active, uint64_t* result, void* stream);
int bpe_apply_merge(uint16_t* sym, int32_t* len, int64_t N, int64_t n_stride, int32_t a, int32_t b,
                    int32_t c, int32_t V, int32_t* delta, int32_t* work, const int32_t* weight, void* stream);
int bpe_apply_delta(int32_t* hist, int32_t* delta, int32_t a, int32_t b, int32_t c, int32_t V, void* stream);
/* Peers of a sharded training run (one process per GPU, sequences sharded, V x V histogram replicated).
 * delta[r] / flags[r] are rank r's count-delta block (int32 [2][4*V], double-buffered by merge parity) and
 * flag array (int32 [BPE_MAX_PEERS]) as DEVICE pointers valid on the calling rank's GPU: its own allocation for
 * r == rank, a peer mapping (beast_peer_open) otherwise.  The per-merge SUM all-reduce of the 4 x V deltas is
 * folded into the iteration head: every rank publishes "rewrite of merge m done" by storing the epoch into
 * flags[p][rank] of every peer p (release, system scope), waits for its own flags, then sums the ranks' delta
 * blocks with peer loads over NVLink while it folds them into its histogram replica.  No host round, no NCCL call
 * between merges.  grid_blocks: blocks of the iteration-head kernel (0 = one per SM); tests that run several
 * ranks on ONE GPU pass a smaller grid so that all ranks' (spinning) kernels are co-resident. */
#define BPE_MAX_PEERS 16
typedef struct bpe_peers {
    int32_t world, rank;
    int32_t grid_blocks;
    int32_t epoch_base;      /* added to the merge index in the flags (lets a caller reuse flags without clearing) */
    int32_t* delta[BPE_MAX_PEERS];
    int32_t* flags[BPE_MAX_PEERS];
} bpe_peers_t;

/* Peer-visible device memory for bpe_peers_t: cudaMalloc + CUDA IPC.  beast_peer_alloc returns a zeroed
 * allocation on the current device and its 64-byte IPC handle (handle_out_h, host); another PROCESS on the same
 * node maps it with beast_peer_open (peer access is enabled lazily); beast_peer_close unmaps, beast_peer_free
 * releases the owner's allocation.  These four calls synchronise / allocate (set-up, not the hot path). */
int beast_peer_alloc(int64_t bytes, void** ptr_out, void* handle_out_h);
int beast_peer_open(const void* handle_h, void** ptr_out);
int beast_peer_close(void* ptr);
int beast_peer_free(void* ptr);

/* Sync-free training loop: one iteration = three launches: (1) iterate: arg-max of the histogram, folding the
 * previous merge's delta (summed over the peers when sharded) on the way, clearing the delta half of the coming
 * merge and the work list; (2) pick + scan: every block picks the merge from the per-block maxima (BpeTrainer's stop
 * rules: vocabulary full / count < min_frequency; next id; block 0 logs it), then scans its tiles of sequences for the
 * pair (signature filter) into the work list; (3) rewrite: the listed sequences, count changes into delta[merge & 1].
 * ctl: int32 [2][16] device block, double-buffered by iteration parity — iteration i reads ctl[i & 1] = {a, b, c, count,
 * n_tokens, n_merges, done, has_delta, err, ...} and writes ctl[(i + 1) & 1]; the caller sets ctl[0].n_tokens =
 * alphabet size and zeroes the rest; first_iter = index of the first iteration enqueued by this call.
 * delta: int32 [2][4*V] (== peers->delta[peers->rank] when sharded); work: int32 [4 + 2*N] scratch; log: int32
 * [4 * max_merges] receives (a, b, new_id, count) per merge; result: arg-max scratch, 256 x uint64 (per-block maxima).
 * Nothing is read back until the end (ctl[(first_iter + iters) & 1]).  iters: iterations enqueued by this call.
 * peers_h: NULL (or world == 1) = unsharded.  weight: int32 [N] multiplicity of every (pseudo-)sequence, NULL = 1
 * (see word de-duplication below). */
int bpe_train_step(uint16_t* sym, int32_t* len, int64_t N, int64_t n_stride, int32_t V, int32_t* hist,
                   int32_t* delta, void* ctl, int32_t* log, uint64_t* result, int32_t* work, int32_t vocab_size,
                   int32_t min_frequency, int32_t max_merges, uint32_t* sig, int32_t first_iter, int32_t iters,
                   const bpe_peers_t* peers_h, const int32_t* weight, void* stream);

/* Word de-duplication in front of the merge loop (what BpeTrainer does with the strings FIGBPE hands it,
 * beast/beast_bpe_trainer.py:61-74: distinct pre-tokens with counts).  csrc/bpe_dedup.cu.
 * bpe_word_totals  totals[0] = pre-tokens, totals[1] = symbols of the symbolised corpus (device, 2 x uint64).
 * bpe_word_list    the flat list of the corpus' words: words [W][4] uint64 = (64-bit hash over symbol ids and length,
 *                  location = sequence << 32 | first symbol << 16 | symbols, the first six symbol ids + 1 in the
 *                  upper 32 + 64 bits of the rest), W = totals[0], in no particular order;
 *                  cursor: one device uint64 of scratch (zeroed by the call); flags[0] = 2 reports W too small.
 * bpe_word_insert  one thread per word over an open-addressing table of 32-byte slots (table: uint64
 *                  [table_size][4] = key, representative location, count | two symbols, four symbols; 32-byte aligned; table_size a
 *                  power of two above the distinct words (the trainer keeps the load below 3/4); the caller zeroes table and flags [3]): an empty
 *                  slot is claimed with one 128-bit compare-and-swap of (hash, location), occurrences are counted,
 *                  and every word that is not the slot's representative is compared with it symbol by symbol (against the
 *                  slot's copy of the first six symbols, else in the corpus):
 *                  flags[0] = 1 reports a 64-bit hash collision — the table is then unusable and the caller trains
 *                  on the plain corpus; flags[0] = 3 = table too small (retry with a larger one); flags[1] = slots
 *                  claimed.
 * bpe_word_emit    reads the distinct words off the table: (location, count) of every claimed slot to out_loc /
 *                  out_cnt [capacity >= flags[1]]; flags[2] = entries written.
 * bpe_word_pack    copies U distinct words (loc[i] as above) to position dst_off[i] of pseudo-sequence dst_seq[i]
 *                  of a second corpus in the same chunk-major layout (first symbol flagged as a word start) and
 *                  pads the last chunk of each of the P pseudo-sequences (dst_len[P] symbols each).
 * The merge loop then runs on the packed corpus with weight[P] = occurrences of the words of each pseudo-sequence
 * (words of equal count are packed together): bpe_count_pairs / bpe_apply_merge / bpe_train_step multiply their
 * count updates by weight[seq] (NULL = 1). */
int bpe_word_totals(const uint16_t* sym, const int32_t* len, int64_t N, int64_t n_stride, uint64_t* totals,
                    void* stream);
int bpe_word_list(const uint16_t* sym, const int32_t* len, int64_t N, int64_t n_stride, uint64_t* words, int64_t W,
                  uint64_t* cursor, int32_t* flags, void* stream);
int bpe_word_insert(const uint16_t* sym, int64_t n_stride, const uint64_t* words, int64_t W, uint64_t* table,
                    int64_t table_size, int32_t* flags, void* stream);
int bpe_word_emit(const uint64_t* table, int64_t table_size, int32_t* flags, uint64_t* out_loc, int32_t* out_cnt,
                  int64_t capacity, void* stream);
int bpe_word_pack(const uint16_t* src, int64_t src_stride, const uint64_t* loc, const int32_t* dst_seq,
                  const int32_t* dst_off, int64_t U, uint16_t* dst, const int32_t* dst_len, int64_t P,
                  int64_t dst_stride, void* stream);

/* Pair signatures for bpe_train_step (optional, sig = NULL scans every sequence): uint32
 * [bpe_signature_words()][n_stride], bit hash(a, b) of sequence s set when s holds (or ever held) the
 * in-word pair (a, b).  The scan for a merge reads one 4-byte column and skips the sequences whose bit
 * is clear; the rewrite adds the bits of the pairs it creates.  Build once after bpe_symbolize. */
int32_t bpe_signature_words(void);
int bpe_build_signatures(const uint16_t* sym, const int32_t* len, int64_t N, int64_t n_stride, uint32_t* sig,
                         void* stream);
int bpe_encode(const int64_t* bins, int64_t N, int32_t L, int64_t min_token, int64_t max_shift,
               const int16_t* byte_to_id, const uint8_t* cls_tab, const uint32_t* rank_tab, int32_t V,
               int32_t hash_bits, uint16_t* ids_padded, int32_t out_stride, int32_t* len_out, int32_t* status_out,
               void* stream);
/* Launch shape of a warp-per-sequence apply kernel on the current device (kernel 0 = bpe_encode's, 1 = bpe_decode's
 * per-token fast path, 2 = bpe_decode's byte-level kernel) for rows of L bins: warps per CTA (0 = the kernel is not
 * used at this L) and the CTA cap of its grid.  Each warp strides over the rows, warps * max_ctas of them per pass. */
int bpe_apply_shape(int32_t kernel, int32_t L, int64_t max_shift, int32_t* warps, int64_t* max_ctas);
int bpe_compact(const uint16_t* ids_padded, int32_t stride, const int32_t* len, const int64_t* offsets,
                int64_t N, int32_t* flat, void* stream);
int bpe_decode(const int32_t* flat, const int64_t* offsets, int64_t N, int32_t L, int64_t min_token,
               const int32_t* tok_off, const uint8_t* tok_bytes, const void* tok_tab, int32_t tok_tab_slots,
               int32_t n_vocab, int64_t* bins_out, int32_t* status_out, int32_t* declen_out, void* stream);

/* Device self-test of the exact invariant-divisor division inside K1 / K3 (csrc/common.cuh) against
 * IEEE division: n_divisors random divisors x 2^24 + 2^22 numerators each, and float(tok)/(V-1)
 * for every V <= vmax.  mismatches (device, 20 x uint64): [0], [1] = number of differing results of the
 * two forms, [2] = examples recorded, [4..19] = up to 8 x (a|b, want|got) bit patterns. */
int beast_selftest_div(int32_t n_divisors, int32_t vmax, uint64_t seed, unsigned long long* mismatches,
                       void* stream);

#ifdef __cplusplus
}
#endif
#endif /* BEAST_B200_H */
