// Spline fit on per-row times (encode / encode_continuous / compute_weights with times [B, T]) and its adjoint.
//
// Row b has its own basis Phi_b = bspline_basis(times[b]) (phase clip(t / tau, 0, 1), the Cox-de Boor rows the
// per-row decode evaluates), so every row solves its own ridge system:
//   joint slot s:   w = (Phi_f^T Phi_f + 1e-9 I)^-1 Phi_f^T (y_s - bias_s - Phi_pin bc_s)
//   gripper slot s: w = (Phi_g^T Phi_g + 1e-9 I)^-1 Phi_g^T y_s          (degree 0: the Gram matrix is diagonal)
// Phi_f = the nb free columns ico .. ico+nb-1 of the nc-column joint basis, Phi_pin the pinned ones (bc [B, n_joint,
// ico+eco] in the layout of beast_reconstruct_bc_f32: cat[bc[:ico], w, bc[ico:]]).  The Gram matrix of a row is shared
// by all its joint slots: it is factored once (band Cholesky) and solved for n_joint right-hand sides.
// Adjoint: v = G^-1 g_w (G is symmetric), u = Phi_f v -> grad_traj = u, grad_bc = -Phi_pin^T u, grad_bias = -sum_t u.
//
// One warp per row, persistent over rows.  Samples stream through shared memory in chunks of 32: lane t evaluates
// only the p + 1 non-zero basis values of its sample (the local triangle of deboor_basis, same operations, so the same
// values) and stages (first column, values); the chunk's targets are staged as fp64.  Every Gram entry and right-hand
// side has one owner lane that adds the chunk's terms in t ascending order, so a row's result depends on nothing but
// the row.  Gram, rhs, factorisation and solves are fp64 (products of fp32 values are exact); each output is rounded
// once to fp32.  No atomics.
//
// Masked fit (beast_fit_masked_f32 / _backward_f32, the kMasked instantiations): a byte mask [B, T] marks the samples
// that are fitted.  Each chunk of 32 raw samples stages only its valid samples, compacted in t order (a ballot and a
// prefix popcount), so the owners see exactly the samples, values and order the unmasked kernel sees on the compacted
// row y[b, mask[b]] on times[b, mask[b]]: the results are bit-identical to it.  A masked sample's time and trajectory
// value are never loaded, it adds no term anywhere, and its grad_traj is written as 0.  The times may be one grid [T]
// for every row (row stride 0).  partial_only: a warp first reads its row's mask and leaves a row whose samples are all
// valid untouched (its outputs stay what another launch wrote there).
#include <climits>
#include <initializer_list>
#include "common.cuh"

namespace beast {

constexpr int kFitTimesChunk = 32;       // samples per staging chunk (one per lane)
constexpr int kFitTimesMaxWarps = 8;     // warps (rows in flight) per CTA
// 64 registers: four 8-warp CTAs fit the register file; without the bound ptxas picked 40-48 and spilled around the
// slow-path calls of the fp32 divisions
constexpr int kFitTimesMinCtas = 4;

struct FitTimesArgs {
    long long B;
    int T, D, nb, n_joint, p, ico, eco, nc;
    float tau;
    const float* knots_j;        // [nc + p + 1]
    const float* knots_g;        // [nb + 1] or nullptr
    const int* slot_to_dof;
    const float* times;          // [B, T] (row stride times_stride: T, or 0 for one grid [T])
    // forward
    const float* traj;           // [B, T, D]
    const float* bc;             // [B, n_joint, ico + eco] (pinned points only)
    const float* bias;           // [B, n_joint] or nullptr
    float* params_out;           // [B, D*nb] '(d t)'
    // backward
    const float* grad_norm;      // [B, nb*D] '(t d)' or nullptr
    const float* grad_params;    // [B, D*nb] or nullptr
    const float* params;         // [B, D*nb] unclamped forward coefficients (with grad_norm)
    const float* w_min;
    const float* w_max;
    float* grad_traj;            // [B, T, D]
    float* grad_bc;              // [B, n_joint, ico + eco] (pinned points only)
    float* grad_bias;            // [B, n_joint] or nullptr
    size_t warp_bytes;           // shared memory per warp
    // masked kernels only
    const uint8_t* mask;         // [B, T] non-zero = fitted
    long long times_stride;
    int partial_only;            // skip rows whose mask is all non-zero
};

// Per-warp shared memory: fp64 arrays first (8-byte aligned), then fp32 / int.
struct FitTimesWarp {
    double* G;       // [nb][p+1]: G[k][d] = Gram(k, k-d) of the free joint columns, then L of its Cholesky factor
    double* cnt;     // [nb] gripper Gram diagonal (sample count per interval)
    double* inv;     // [nb] 1 / L(k, k)
    double* rhs;     // [D][nb] right-hand sides, then the solutions ('(d t)' order)
    double* yc;      // [chunk][D] staged targets (forward) / u (backward), slot order
    double* acc;     // [n_joint][ico + eco + 1] grad_bc / grad_bias sums (backward)
    float* v;        // [chunk][p+2] non-zero joint basis values of each sample (+ a zero sentinel)
    int* f;          // [chunk] first joint column (of nc) of each sample's values
    int* g;          // [chunk] gripper interval of each sample
    int* r;          // [chunk] raw index of each staged sample (masked kernels only)
};

static size_t fit_times_doubles(int D, int nb, int p, int n_joint, int nbc) {
    return (size_t)nb * (p + 1) + 2 * (size_t)nb + (size_t)D * nb + (size_t)kFitTimesChunk * D +
           (size_t)n_joint * (nbc + 1);
}
static size_t fit_times_warp_bytes(int D, int nb, int p, int n_joint, int nbc, bool masked) {
    const size_t b = fit_times_doubles(D, nb, p, n_joint, nbc) * 8 + (size_t)kFitTimesChunk * (p + 2) * 4 +
                     (masked ? 3 : 2) * (size_t)kFitTimesChunk * 4;
    return (b + 15) & ~(size_t)15;
}

__device__ __forceinline__ FitTimesWarp fit_times_warp(const FitTimesArgs& a, char* base) {
    FitTimesWarp w;
    const int nbc = a.ico + a.eco;
    double* d = (double*)base;
    w.G = d;   d += (size_t)a.nb * (a.p + 1);
    w.cnt = d; d += a.nb;
    w.inv = d; d += a.nb;
    w.rhs = d; d += (size_t)a.D * a.nb;
    w.yc = d;  d += (size_t)kFitTimesChunk * a.D;
    w.acc = d; d += (size_t)a.n_joint * (nbc + 1);
    w.v = (float*)d;
    w.f = (int*)(w.v + kFitTimesChunk * (a.p + 2));
    w.g = w.f + kFitTimesChunk;
    w.r = w.g + kFitTimesChunk;
    return w;
}

// Largest i in [lo, hi] with kn[i] <= u (kn non-decreasing, kn[lo] <= u): the interval deboor_basis's level 0 sets to
// 1 — [kn[i], kn[i+1]) with the last basis interval closed on the right; the intervals below lo / above hi are empty.
__device__ __forceinline__ int knot_span(const float* kn, int lo, int hi, float u) {
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (kn[mid] <= u) lo = mid; else hi = mid - 1;
    }
    return lo;
}

// Stages one sample at time tv into slot `lane`: joint span values v[0..p] of columns f .. f+p (deboor_basis's
// recursion restricted to the triangle of non-zero entries, same operations in the same order) and the gripper interval.
__device__ __forceinline__ void fit_times_stage_one(const FitTimesArgs& a, const FitTimesWarp& w, const float* kj,
                                                    const float* kg, float tv, int lane) {
    const int p = a.p;
    const float u = clampf(__fdiv_rn(__fsub_rn(tv, 0.0f), a.tau), 0.0f, 1.0f);   // as decode_generic_kernel
    float* N = w.v + lane * (p + 2);                       // N[m] = basis j - p + m, N[p + 1] = 0 (basis j + 1)
    if (a.n_joint > 0) {
        const int j = knot_span(kj, p, a.nc - 1, u);
        for (int m = 0; m <= p + 1; ++m) N[m] = m == p ? 1.0f : 0.0f;
        for (int k = 1; k <= p; ++k) {
            for (int i = j - k; i <= j; ++i) {             // ascending i, in place, as deboor_basis
                const int m = i - (j - p);
                const float d1 = __fsub_rn(kj[i + k], kj[i]);
                const float d2 = __fsub_rn(kj[i + k + 1], kj[i + 1]);
                const bool h1 = d1 != 0.0f, h2 = d2 != 0.0f;
                const float t1 = h1 ? __fmul_rn(__fdiv_rn(__fsub_rn(u, kj[i]), d1), N[m]) : 0.0f;
                const float t2 = h2 ? __fmul_rn(__fdiv_rn(__fsub_rn(kj[i + k + 1], u), d2), N[m + 1]) : 0.0f;
                N[m] = (h1 && h2) ? __fadd_rn(t1, t2) : (h1 ? t1 : t2);
            }
        }
        w.f[lane] = j - p;
    } else {
        w.f[lane] = 0;
    }
    w.g[lane] = kg ? knot_span(kg, 0, a.nb - 1, u) : 0;
}

// Stages the n raw samples t0 .. t0+n-1 of row b and returns how many were staged (slots 0 .. nt-1, t ascending).
// Unmasked: lane < n stages sample t0 + lane.  Masked: only the valid samples, each at slot = the number of valid samples
// before it in the chunk, its raw index in w.r; *valid = the chunk's ballot (bit i: sample t0 + i is fitted).
template <bool kMasked>
__device__ __forceinline__ int fit_times_stage(const FitTimesArgs& a, const FitTimesWarp& w, const float* kj,
                                               const float* kg, long long b, int t0, int n, int lane,
                                               unsigned* valid = nullptr) {
    if constexpr (!kMasked) {
        if (lane < n) fit_times_stage_one(a, w, kj, kg, a.times[b * a.T + t0 + lane], lane);
        return n;
    } else {
        const bool on = lane < n && a.mask[b * a.T + t0 + lane] != 0;
        const unsigned bal = __ballot_sync(0xffffffffu, on);
        if (on) {
            const int slot = __popc(bal & ((1u << lane) - 1u));
            fit_times_stage_one(a, w, kj, kg, a.times[b * a.times_stride + t0 + lane], slot);
            w.r[slot] = t0 + lane;
        }
        if (valid) *valid = bal;
        return __popc(bal);
    }
}

// partial_only: true when every sample of row b is valid (the warp then leaves the row to the launch that wrote it)
template <bool kMasked>
__device__ __forceinline__ bool fit_times_skip_row(const FitTimesArgs& a, long long b, int lane) {
    if constexpr (!kMasked) {
        return false;
    } else {
        if (!a.partial_only) return false;
        bool full = true;
        for (int t = lane; t < a.T; t += 32) full &= a.mask[b * a.T + t] != 0;
        return __all_sync(0xffffffffu, full);
    }
}

// Owners of the Gram entries add the chunk's terms, t ascending.  Joint: entry (k, k-d) of the free columns; gripper:
// the sample count of interval k.  A per-sample weight would multiply each term here.
__device__ __forceinline__ void fit_times_gram(const FitTimesArgs& a, const FitTimesWarp& w, int nt, int lane, int fmin,
                                               int fmax, int gmin, int gmax) {
    const int p = a.p, nb = a.nb, pp = p + 2;
    const int n_g = a.n_joint > 0 ? nb * (p + 1) : 0, n_c = a.knots_g ? nb : 0;
    for (int e = lane; e < n_g + n_c; e += 32) {
        if (e < n_g) {
            const int k = e / (p + 1), d = e - k * (p + 1);
            const int c = k + a.ico;
            if (k < d || c - d < fmin || c - p > fmax) continue;     // no sample of the chunk has both columns
            double s = w.G[e];
#pragma unroll 4
            for (int t = 0; t < nt; ++t) {            // a sample outside the entry's support adds 0 * 0
                const int q = c - w.f[t];
                const bool hit = q >= d && q <= p;
                const float* r = w.v + t * pp;
                s = fma((double)r[hit ? q : p + 1], (double)r[hit ? q - d : p + 1], s);
            }
            w.G[e] = s;
        } else {
            const int k = e - n_g;
            if (k < gmin || k > gmax) continue;
            double s = w.cnt[k];
            for (int t = 0; t < nt; ++t)
                if (w.g[t] == k) s += 1.0;
            w.cnt[k] = s;
        }
    }
}

// Band Cholesky of Gram + 1e-9 I in place (one lane): G[k][d] <- L(k, k-d), inv[k] = 1 / L(k, k).
__device__ __forceinline__ void fit_times_factor(const FitTimesArgs& a, const FitTimesWarp& w) {
    const int p = a.p, nb = a.nb, w1 = p + 1;
    double* G = w.G;
    for (int k = 0; k < nb; ++k) {
        const int m0 = k - p > 0 ? k - p : 0;
        for (int i = m0; i < k; ++i) {
            double s = G[k * w1 + (k - i)];
            for (int m = m0; m < i; ++m) s -= G[k * w1 + (k - m)] * G[i * w1 + (i - m)];
            G[k * w1 + (k - i)] = s * w.inv[i];
        }
        double s = G[k * w1] + 1e-9;
        for (int m = m0; m < k; ++m) s -= G[k * w1 + (k - m)] * G[k * w1 + (k - m)];
        const double l = sqrt(s);
        G[k * w1] = l;
        w.inv[k] = 1.0 / l;
    }
}

// Solve every slot's system in place in rhs (lanes over slots): joint slots L L^T x = r, gripper slots r / (count + 1e-9).
__device__ __forceinline__ void fit_times_solve(const FitTimesArgs& a, const FitTimesWarp& w, int lane) {
    const int p = a.p, nb = a.nb, w1 = p + 1;
    for (int s = lane; s < a.D; s += 32) {
        double* r = w.rhs + (size_t)s * nb;
        if (s < a.n_joint) {
            for (int k = 0; k < nb; ++k) {
                double z = r[k];
                for (int m = (k - p > 0 ? k - p : 0); m < k; ++m) z -= w.G[k * w1 + (k - m)] * r[m];
                r[k] = z * w.inv[k];
            }
            for (int k = nb - 1; k >= 0; --k) {
                double x = r[k];
                const int i1 = k + p < nb - 1 ? k + p : nb - 1;
                for (int i = k + 1; i <= i1; ++i) x -= w.G[i * w1 + (i - k)] * r[i];
                r[k] = x * w.inv[k];
            }
        } else {
            for (int k = 0; k < nb; ++k) r[k] = r[k] / (w.cnt[k] + 1e-9);
        }
    }
}

__device__ __forceinline__ void warp_range(int nt, int lane, const FitTimesWarp& w, int& fmin, int& fmax, int& gmin,
                                           int& gmax) {
    const bool on = lane < nt;
    fmin = __reduce_min_sync(0xffffffffu, on ? w.f[lane] : INT_MAX);
    fmax = __reduce_max_sync(0xffffffffu, on ? w.f[lane] : INT_MIN);
    gmin = __reduce_min_sync(0xffffffffu, on ? w.g[lane] : INT_MAX);
    gmax = __reduce_max_sync(0xffffffffu, on ? w.g[lane] : INT_MIN);
}

// Common prologue: knots and the dof -> slot map in shared memory, then this warp's region.
__device__ __forceinline__ FitTimesWarp fit_times_setup(const FitTimesArgs& a, char* smem, const float*& kj,
                                                        const float*& kg, int*& dof_slot) {
    const int nkj = a.nc + a.p + 1, nkg = a.knots_g ? a.nb + 1 : 0;
    float* k_s = (float*)smem;
    dof_slot = (int*)(k_s + nkj + nkg);
    for (int i = threadIdx.x; i < nkj; i += blockDim.x) k_s[i] = a.knots_j[i];
    for (int i = threadIdx.x; i < nkg; i += blockDim.x) k_s[nkj + i] = a.knots_g[i];
    for (int i = threadIdx.x; i < a.D; i += blockDim.x) dof_slot[a.slot_to_dof[i]] = i;
    __syncthreads();
    kj = k_s;
    kg = a.knots_g ? k_s + nkj : nullptr;
    const size_t head = (((size_t)(nkj + nkg + a.D) * 4) + 15) & ~(size_t)15;
    return fit_times_warp(a, smem + head + (threadIdx.x >> 5) * a.warp_bytes);
}

template <bool kMasked>
__global__ void __launch_bounds__(kFitTimesMaxWarps * 32, kFitTimesMinCtas)
fit_times_kernel(const __grid_constant__ FitTimesArgs a) {
    extern __shared__ __align__(16) char smem_c[];
    const float* kj;
    const float* kg;
    int* dof_slot;
    const FitTimesWarp w = fit_times_setup(a, smem_c, kj, kg, dof_slot);
    const int lane = threadIdx.x & 31, warps = blockDim.x >> 5;
    const int T = a.T, D = a.D, nb = a.nb, p = a.p, pp = p + 2, nj = a.n_joint, nbc = a.ico + a.eco;
    const int n_g = nj > 0 ? nb * (p + 1) : 0;
    for (long long b = (long long)blockIdx.x * warps + (threadIdx.x >> 5); b < a.B; b += (long long)gridDim.x * warps) {
        if (fit_times_skip_row<kMasked>(a, b, lane)) continue;
        for (int i = lane; i < n_g; i += 32) w.G[i] = 0.0;
        for (int i = lane; i < nb; i += 32) w.cnt[i] = 0.0;
        for (int i = lane; i < D * nb; i += 32) w.rhs[i] = 0.0;
        for (int t0 = 0; t0 < T; t0 += kFitTimesChunk) {
            const int n = T - t0 < kFitTimesChunk ? T - t0 : kFitTimesChunk;
            __syncwarp();                                  // previous chunk consumed, accumulators zeroed
            const int nt = fit_times_stage<kMasked>(a, w, kj, kg, b, t0, n, lane);
            __syncwarp();
            // targets in slot order; joint slots minus bias and the pinned points' contribution
            const float* y = a.traj + (b * T + t0) * D;
            for (int i = lane; i < nt * D; i += 32) {
                const int t = i / D, dof = i - t * D, s = dof_slot[dof];
                double v;
                if constexpr (kMasked) v = (double)__ldcs(a.traj + (b * T + w.r[t]) * D + dof);
                else v = (double)__ldcs(y + i);
                if (s < nj && (nbc > 0 || a.bias)) {
                    if (a.bias) v -= (double)a.bias[b * nj + s];
                    const float* pin = a.bc + (b * nj + s) * nbc;
                    const int f = w.f[t];
                    for (int c = 0; c < nbc; ++c) {
                        const int col = c < a.ico ? c : nb + c, q = col - f;
                        if (q >= 0 && q <= p) v -= (double)w.v[t * pp + q] * (double)pin[c];
                    }
                }
                w.yc[t * D + s] = v;
            }
            __syncwarp();
            int fmin, fmax, gmin, gmax;
            warp_range(nt, lane, w, fmin, fmax, gmin, gmax);
            fit_times_gram(a, w, nt, lane, fmin, fmax, gmin, gmax);
            for (int e = lane; e < D * nb; e += 32) {      // rhs owners: (slot, k), t ascending
                const int s = e / nb, k = e - s * nb;
                double acc = w.rhs[e];
                if (s < nj) {
                    const int c = k + a.ico;
                    if (c < fmin || c > fmax + p) continue;
#pragma unroll 4
                    for (int t = 0; t < nt; ++t) {    // branch-free: a sample outside the support adds 0 * y
                        const int q = c - w.f[t];
                        const bool hit = (unsigned)q <= (unsigned)p;
                        acc = fma((double)w.v[t * pp + (hit ? q : p + 1)], w.yc[t * D + s], acc);
                    }
                } else {
                    if (k < gmin || k > gmax) continue;
                    for (int t = 0; t < nt; ++t)
                        if (w.g[t] == k) acc += w.yc[t * D + s];
                }
                w.rhs[e] = acc;
            }
        }
        __syncwarp();
        if (nj > 0 && lane == 0) fit_times_factor(a, w);
        __syncwarp();
        fit_times_solve(a, w, lane);
        __syncwarp();
        float* out = a.params_out + b * D * nb;
        for (int i = lane; i < D * nb; i += 32) __stcs(out + i, __double2float_rn(w.rhs[i]));
        __syncwarp();
    }
}

template <bool kMasked>
__global__ void __launch_bounds__(kFitTimesMaxWarps * 32, kFitTimesMinCtas)
fit_times_backward_kernel(const __grid_constant__ FitTimesArgs a) {
    extern __shared__ __align__(16) char smem_c[];
    const float* kj;
    const float* kg;
    int* dof_slot;
    const FitTimesWarp w = fit_times_setup(a, smem_c, kj, kg, dof_slot);
    const int lane = threadIdx.x & 31, warps = blockDim.x >> 5;
    const int T = a.T, D = a.D, nb = a.nb, p = a.p, pp = p + 2, nj = a.n_joint, nbc = a.ico + a.eco;
    const int n_g = nj > 0 ? nb * (p + 1) : 0;
    const int n_acc = a.grad_bc ? nj * (nbc + 1) : 0;
    for (long long b = (long long)blockIdx.x * warps + (threadIdx.x >> 5); b < a.B; b += (long long)gridDim.x * warps) {
        if (fit_times_skip_row<kMasked>(a, b, lane)) continue;
        for (int i = lane; i < n_g; i += 32) w.G[i] = 0.0;
        for (int i = lane; i < nb; i += 32) w.cnt[i] = 0.0;
        for (int i = lane; i < n_acc; i += 32) w.acc[i] = 0.0;
        // pass 1: the row's Gram matrices, exactly as the forward builds them
        for (int t0 = 0; t0 < T; t0 += kFitTimesChunk) {
            const int n = T - t0 < kFitTimesChunk ? T - t0 : kFitTimesChunk;
            __syncwarp();
            const int nt = fit_times_stage<kMasked>(a, w, kj, kg, b, t0, n, lane);
            __syncwarp();
            int fmin, fmax, gmin, gmax;
            warp_range(nt, lane, w, fmin, fmax, gmin, gmax);
            fit_times_gram(a, w, nt, lane, fmin, fmax, gmin, gmax);
        }
        // g_w as beast_fit_backward_f32 forms it, then v = G^-1 g_w
        for (int i = lane; i < D * nb; i += 32) {
            const int s = i / nb, k = i - s * nb;
            w.rhs[i] = (double)fit_grad_coeff(a.grad_norm, a.grad_params, a.params, a.w_min, a.w_max, b * D * nb, D,
                                              nb, s, k);
        }
        __syncwarp();
        if (nj > 0 && lane == 0) fit_times_factor(a, w);
        __syncwarp();
        fit_times_solve(a, w, lane);
        // pass 2: u = Phi v per sample (output order), then the pinned points' and the bias's sums, t ascending
        for (int t0 = 0; t0 < T; t0 += kFitTimesChunk) {
            const int n = T - t0 < kFitTimesChunk ? T - t0 : kFitTimesChunk;
            __syncwarp();
            unsigned valid = 0;
            const int nt = fit_times_stage<kMasked>(a, w, kj, kg, b, t0, n, lane, &valid);
            __syncwarp();
            float* gy = a.grad_traj + (b * T + t0) * D;
            if constexpr (kMasked) {                       // masked samples: exactly 0
                for (int i = lane; i < n * D; i += 32)
                    if (!((valid >> (i / D)) & 1u)) __stcs(gy + i, 0.0f);
            }
            for (int i = lane; i < nt * D; i += 32) {
                const int t = i / D, dof = i - t * D, s = dof_slot[dof];
                const double* v = w.rhs + (size_t)s * nb;
                double u = 0.0;
                if (s < nj) {
                    const int f = w.f[t] - a.ico;
                    for (int q = 0; q <= p; ++q) {
                        const int k = f + q;
                        if (k >= 0 && k < nb) u = fma((double)w.v[t * pp + q], v[k], u);
                    }
                } else {
                    u = v[w.g[t]];
                }
                if constexpr (kMasked) __stcs(a.grad_traj + (b * T + w.r[t]) * D + dof, __double2float_rn(u));
                else __stcs(gy + i, __double2float_rn(u));
                w.yc[t * D + s] = u;
            }
            __syncwarp();
            for (int e = lane; e < n_acc; e += 32) {
                const int s = e / (nbc + 1), c = e - s * (nbc + 1);
                double acc = w.acc[e];
                if (c < nbc) {
                    const int col = c < a.ico ? c : nb + c;
                    for (int t = 0; t < nt; ++t) {
                        const int q = col - w.f[t];
                        if (q >= 0 && q <= p) acc = fma((double)w.v[t * pp + q], w.yc[t * D + s], acc);
                    }
                } else {
                    for (int t = 0; t < nt; ++t) acc += w.yc[t * D + s];
                }
                w.acc[e] = acc;
            }
        }
        __syncwarp();
        for (int e = lane; e < n_acc; e += 32) {
            const int s = e / (nbc + 1), c = e - s * (nbc + 1);
            const float r = __double2float_rn(-w.acc[e]);
            if (c < nbc) a.grad_bc[(b * nj + s) * nbc + c] = r;
            else if (a.grad_bias) a.grad_bias[b * nj + s] = r;
        }
        __syncwarp();
    }
}

template <typename K>
static int launch_fit_times(const Plan* p, FitTimesArgs& a, K kernel, cudaStream_t st, size_t (&granted)[kMaxDevices]) {
    const int nbc = p->ico + p->eco;
    const size_t head = (((size_t)(p->nc + p->degree_p + 1 + (p->n_joint < p->D ? p->nb + 1 : 0) + p->D) * 4) + 15) &
                        ~(size_t)15;
    a.warp_bytes = fit_times_warp_bytes(p->D, p->nb, p->degree_p, p->n_joint, nbc, a.mask != nullptr);
    long long warps = ((long long)p->max_smem_optin - (long long)head) / (long long)a.warp_bytes;
    if (warps < 1) return BEAST_E_UNSUPPORTED;
    if (warps > kFitTimesMaxWarps) warps = kFitTimesMaxWarps;
    const size_t smem = head + (size_t)warps * a.warp_bytes;
    if (int rc = opt_in_smem(kernel, smem, granted)) return rc;
    int per_sm = 0;
    cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, (int)warps * 32, smem);
    if (e != cudaSuccess) return (int)e;
    if (per_sm < 1) per_sm = 1;
    const long long ctas = (a.B + warps - 1) / warps;
    const long long cap = (long long)p->num_sms * per_sm;
    kernel<<<(unsigned)(ctas < cap ? ctas : cap), (unsigned)warps * 32, smem, st>>>(a);
    count_launch();
    BEAST_CHECK_LAUNCH();
    return BEAST_OK;
}

static void fit_times_common(const Plan* p, FitTimesArgs& a, long long B, int T, const float* times) {
    a.B = B; a.T = T; a.D = p->D; a.nb = p->nb; a.n_joint = p->n_joint; a.p = p->degree_p;
    a.ico = p->ico; a.eco = p->eco; a.nc = p->nc; a.tau = p->tau;
    a.knots_j = p->knots_joint_d;
    a.knots_g = p->n_joint < p->D ? p->knots_grip_d : nullptr;
    a.slot_to_dof = p->slot_to_dof_d;
    a.times = times;
    a.times_stride = T;
}

static bool misaligned4(std::initializer_list<const void*> ps) {
    for (const void* q : ps)
        if ((uintptr_t)q & 3u) return true;
    return false;
}

}  // namespace beast

using namespace beast;

extern "C" int beast_fit_times_f32(const beast_plan_t* plan, const float* traj, int64_t B, int32_t T,
                                   const float* times, const float* bc, const float* bias, float* params_out,
                                   void* stream) {
    const Plan* p = (const Plan*)plan;
    if (!p) return BEAST_E_NULL;
    const bool pinned = p->ico + p->eco > 0 && p->n_joint > 0;
    if (B < 0 || T < 1 || (pinned && T < 2)) return BEAST_E_SHAPE;
    if (p->nc + p->degree_p + 1 > kMaxEvalKnots) return BEAST_E_UNSUPPORTED;
    if (B > 0 && (!traj || !times || !params_out || (pinned && !bc))) return BEAST_E_NULL;
    if (misaligned4({traj, times, bc, bias, params_out})) return BEAST_E_ALIGN;
    if (B == 0) return BEAST_OK;
    FitTimesArgs a = {};
    fit_times_common(p, a, B, T, times);
    a.traj = traj;
    a.bc = pinned ? bc : nullptr;
    a.bias = pinned ? bias : nullptr;
    a.params_out = params_out;
    static size_t granted[kMaxDevices] = {};
    return launch_fit_times(p, a, fit_times_kernel<false>, (cudaStream_t)stream, granted);
}

extern "C" int beast_fit_times_backward_f32(const beast_plan_t* plan, int64_t B, int32_t T, const float* times,
                                            const float* grad_norm, const float* grad_params, const float* params,
                                            const float* w_min, const float* w_max, float* grad_traj, float* grad_bc,
                                            float* grad_bias, void* stream) {
    const Plan* p = (const Plan*)plan;
    if (!p) return BEAST_E_NULL;
    const bool pinned = p->ico + p->eco > 0 && p->n_joint > 0;
    if (B < 0 || T < 1 || (pinned && T < 2)) return BEAST_E_SHAPE;
    if (p->nc + p->degree_p + 1 > kMaxEvalKnots) return BEAST_E_UNSUPPORTED;
    if (!grad_norm && !grad_params) return BEAST_E_NULL;
    if (grad_norm && (!params || !w_min || !w_max)) return BEAST_E_NULL;
    if (B > 0 && (!times || !grad_traj || (pinned && !grad_bc))) return BEAST_E_NULL;
    if (misaligned4({times, grad_norm, grad_params, params, w_min, w_max, grad_traj, grad_bc, grad_bias}))
        return BEAST_E_ALIGN;
    if (B == 0) return BEAST_OK;
    FitTimesArgs a = {};
    fit_times_common(p, a, B, T, times);
    a.grad_norm = grad_norm; a.grad_params = grad_params;
    a.params = grad_norm ? params : nullptr;
    a.w_min = grad_norm ? w_min : nullptr; a.w_max = grad_norm ? w_max : nullptr;
    a.grad_traj = grad_traj;
    a.grad_bc = pinned ? grad_bc : nullptr;
    a.grad_bias = pinned ? grad_bias : nullptr;
    static size_t granted[kMaxDevices] = {};
    return launch_fit_times(p, a, fit_times_backward_kernel<false>, (cudaStream_t)stream, granted);
}

extern "C" int beast_fit_masked_f32(const beast_plan_t* plan, const float* traj, int64_t B, int32_t T,
                                    const float* times, int64_t times_row_stride, const uint8_t* mask,
                                    int32_t partial_only, const float* bc, const float* bias, float* params_out,
                                    void* stream) {
    const Plan* p = (const Plan*)plan;
    if (!p) return BEAST_E_NULL;
    const bool pinned = p->ico + p->eco > 0 && p->n_joint > 0;
    if (B < 0 || T < 1 || (pinned && T < 2)) return BEAST_E_SHAPE;
    if (times_row_stride != 0 && times_row_stride != T) return BEAST_E_SHAPE;
    if (p->nc + p->degree_p + 1 > kMaxEvalKnots) return BEAST_E_UNSUPPORTED;
    if (B > 0 && (!traj || !times || !mask || !params_out || (pinned && !bc))) return BEAST_E_NULL;
    if (misaligned4({traj, times, bc, bias, params_out})) return BEAST_E_ALIGN;
    if (B == 0) return BEAST_OK;
    FitTimesArgs a = {};
    fit_times_common(p, a, B, T, times);
    a.times_stride = times_row_stride;
    a.mask = mask;
    a.partial_only = partial_only ? 1 : 0;
    a.traj = traj;
    a.bc = pinned ? bc : nullptr;
    a.bias = pinned ? bias : nullptr;
    a.params_out = params_out;
    static size_t granted[kMaxDevices] = {};
    return launch_fit_times(p, a, fit_times_kernel<true>, (cudaStream_t)stream, granted);
}

extern "C" int beast_fit_masked_backward_f32(const beast_plan_t* plan, int64_t B, int32_t T, const float* times,
                                             int64_t times_row_stride, const uint8_t* mask, int32_t partial_only,
                                             const float* grad_norm, const float* grad_params, const float* params,
                                             const float* w_min, const float* w_max, float* grad_traj, float* grad_bc,
                                             float* grad_bias, void* stream) {
    const Plan* p = (const Plan*)plan;
    if (!p) return BEAST_E_NULL;
    const bool pinned = p->ico + p->eco > 0 && p->n_joint > 0;
    if (B < 0 || T < 1 || (pinned && T < 2)) return BEAST_E_SHAPE;
    if (times_row_stride != 0 && times_row_stride != T) return BEAST_E_SHAPE;
    if (p->nc + p->degree_p + 1 > kMaxEvalKnots) return BEAST_E_UNSUPPORTED;
    if (!grad_norm && !grad_params) return BEAST_E_NULL;
    if (grad_norm && (!params || !w_min || !w_max)) return BEAST_E_NULL;
    if (B > 0 && (!times || !mask || !grad_traj || (pinned && !grad_bc))) return BEAST_E_NULL;
    if (misaligned4({times, grad_norm, grad_params, params, w_min, w_max, grad_traj, grad_bc, grad_bias}))
        return BEAST_E_ALIGN;
    if (B == 0) return BEAST_OK;
    FitTimesArgs a = {};
    fit_times_common(p, a, B, T, times);
    a.times_stride = times_row_stride;
    a.mask = mask;
    a.partial_only = partial_only ? 1 : 0;
    a.grad_norm = grad_norm; a.grad_params = grad_params;
    a.params = grad_norm ? params : nullptr;
    a.w_min = grad_norm ? w_min : nullptr; a.w_max = grad_norm ? w_max : nullptr;
    a.grad_traj = grad_traj;
    a.grad_bc = pinned ? grad_bc : nullptr;
    a.grad_bias = pinned ? grad_bias : nullptr;
    static size_t granted[kMaxDevices] = {};
    return launch_fit_times(p, a, fit_times_backward_kernel<true>, (cudaStream_t)stream, granted);
}
