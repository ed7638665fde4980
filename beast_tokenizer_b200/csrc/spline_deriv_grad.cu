// Adjoint of the spline decode of orders 0..2 (spline_deriv.cu): gradients of positions, velocities and accelerations
// back to the de-normalised coefficients and to init_p.
//
//   g_c[b, slot, k] = sum_t sum_o R_o[t, ico + k] * g_o[b, t, dof(slot)]      (joint slots, o over the given orders)
//   g_c[b, slot, k] = sum_t N_g[t, k] * g_0[b, t, dof(slot)]                  (gripper slots: degree 0, position only)
//
// R_o are the rows the forward multiplies the coefficients with (d^o/dt^o of the basis, zero outside [0, tau] for
// o >= 1).  Pinned control points (ico leading / eco trailing) are constants: only the nb free columns receive a
// gradient.  With init_p, coefficient 0 of every joint slot is init_p[b, dof]: that sum goes to grad_init_p[b, dof]
// and grad_params[b, slot, 0] is 0; gripper columns of grad_init_p are 0.
//
// Every coefficient is one fp32 sum in a fixed order: t ascending over the rows that read it, for each t the orders
// ascending, one fmaf per term.  The terms a kernel skips are exact zeros (R_o[t, k] == 0), which leave a sum of
// finite values unchanged, so both kernels return the same values.  No atomics.
//
// Generic kernel: one CTA per trajectory; the basis rows of a chunk of samples are evaluated in-kernel (deboor_deriv,
// bit for bit the host rows) into shared memory, then every thread adds them into the coefficients it owns.  Times per
// row ([B, Tq]) or one shared grid (row stride 0).
// Tiled kernel (one shared grid, no pinned points): a CTA owns a tile of S = 4 Q trajectories.  The tile's gradient
// rows stream through shared memory in chunks of samples, transposed so that one float4 holds one (order, sample, dof)
// of four trajectories.  Each thread keeps register sums of fixed (slot, k, quad) items and adds, per chunk, the rows
// of the grid's column support of k (colsup_d).  At the end of a tile the sums go through shared memory and leave in
// grad_params order.
#include "spline_deriv.cuh"

namespace beast {

constexpr int kGradThreads = 512;     // tiled kernel
constexpr int kGradItems = 4;         // (slot, k, quad) items per thread of the tiled kernel
constexpr int kGradGenericThreads = 128;

struct GradGenericArgs {
    long long B;
    int Tq, times_stride;          // times of trajectory b start at times + b * times_stride (0: one shared grid)
    int D, nb, n_joint, degree_p, ico, nc;
    const int* slot_to_dof;
    const float* times;
    const float* knots_j;
    const float* knots_g;
    float tau;
    const float* grad[3];          // [B, Tq, D] by order (nullable)
    int max_order;                 // highest given order
    int TC, row_floats;            // samples per chunk; floats of one sample's rows in shared memory
    int init_p_used;
    float* grad_params;            // [B, D*nb] '(d t)'
    float* grad_init_p;            // [B, D] or nullptr
};

__global__ void __launch_bounds__(kGradGenericThreads, 2)
deriv_grad_generic_kernel(const __grid_constant__ GradGenericArgs a) {
    extern __shared__ __align__(16) float smem_f[];
    const int D = a.D, nb = a.nb, nc = a.nc, ico = a.ico, Tq = a.Tq, TC = a.TC, mo = a.max_order;
    const int rf = a.row_floats, row = D * nb;
    float* rows_s = smem_f;                              // [TC][rf]: orders 0..mo of the joint basis [nc], gripper [nb]
    float* g_s = rows_s + (size_t)TC * rf;               // [TC][3][D]
    const int tid = threadIdx.x;
    const int n_chunks = (Tq + TC - 1) / TC;
    const int grip_off = (mo + 1) * nc;
    float N[kMaxEvalKnots], D1[kMaxEvalKnots], D2[kMaxEvalKnots];
    for (long long b = blockIdx.x; b < a.B; b += gridDim.x) {
        float* gp = a.grad_params + b * row;
        for (int c = 0; c < (n_chunks > 0 ? n_chunks : 1); ++c) {
            const int t0 = c * TC;
            const int tc = n_chunks > 0 ? (Tq - t0 < TC ? Tq - t0 : TC) : 0;
            __syncthreads();                             // previous chunk consumed
            if (tid < tc) {
                const float raw = __fdiv_rn(__fsub_rn(a.times[b * a.times_stride + t0 + tid], 0.0f), a.tau);
                const float u = clampf(raw, 0.0f, 1.0f);
                const bool outside = raw < 0.0f || raw > 1.0f;
                float* r = rows_s + (size_t)tid * rf;
                deboor_deriv(a.knots_j, nc, a.degree_p, u, mo, N, D1, D2);
                for (int i = 0; i < nc; ++i) {
                    r[i] = N[i];
                    if (mo >= 1) r[nc + i] = outside ? 0.0f : __fdiv_rn(D1[i], a.tau);
                    if (mo >= 2) r[2 * nc + i] = outside ? 0.0f : __fdiv_rn(__fdiv_rn(D2[i], a.tau), a.tau);
                }
                if (a.n_joint < D) {
                    deboor_deriv(a.knots_g, nb, 0, u, 0, N, nullptr, nullptr);
                    for (int k = 0; k < nb; ++k) r[grip_off + k] = N[k];
                }
            }
            for (int o = 0; o <= mo; ++o) {
                if (!a.grad[o]) continue;
                const float* src = a.grad[o] + (b * Tq + t0) * D;
                for (int idx = tid; idx < tc * D; idx += kGradGenericThreads) {
                    const int i = idx / D, dof = idx - i * D;
                    g_s[(i * 3 + o) * D + dof] = src[idx];
                }
            }
            __syncthreads();
            const bool last = c + 1 >= n_chunks;
            for (int j = tid; j < row; j += kGradGenericThreads) {
                const int slot = j / nb, k = j - slot * nb;
                const int dof = a.slot_to_dof[slot];
                const bool joint = slot < a.n_joint;
                float acc = c == 0 ? 0.0f : gp[j];
                for (int i = 0; i < tc; ++i) {
                    const float* r = rows_s + (size_t)i * rf;
                    const float* g = g_s + i * 3 * D + dof;
                    if (joint) {
                        for (int o = 0; o <= mo; ++o)
                            if (a.grad[o]) acc = fmaf(r[o * nc + ico + k], g[o * D], acc);
                    } else if (a.grad[0]) {
                        acc = fmaf(r[grip_off + k], g[0], acc);
                    }
                }
                if (last && k == 0 && a.init_p_used) {
                    if (a.grad_init_p) a.grad_init_p[b * D + dof] = joint ? acc : 0.0f;
                    if (joint) acc = 0.0f;
                }
                gp[j] = acc;
            }
        }
    }
}

struct GradTiledArgs {
    long long B;
    int Tq, D, nb, n_joint;
    const int* slot_to_dof;
    const int* colsup;             // [joint | gripper][nb][lo, hi)
    const float* rows[3];          // joint rows [Tq][nb] of the NO given orders, ascending
    const float* rows_grip0;       // gripper order-0 rows [Tq][nb] (nullptr without grippers)
    const float* grad[3];          // [B, Tq, D] of the NO given orders, ascending
    int has0;                      // order 0 is given (then it is grad[0]): gripper slots receive a gradient
    int S, Q, TC, TS;              // trajectories per tile (4 Q), quads, samples per chunk, floats per sample row
    int buf_floats;                // floats of the chunk / output buffer
    int init_p_used;
    float* grad_params;
    float* grad_init_p;
};

template <int NO>
__global__ void __launch_bounds__(kGradThreads, 2)
deriv_grad_tiled_kernel(const __grid_constant__ GradTiledArgs a) {
    extern __shared__ __align__(16) float smem_f[];
    const int D = a.D, nb = a.nb, Tq = a.Tq, S = a.S, Q = a.Q, TC = a.TC, TS = a.TS;
    const int row = D * nb, n_items = row * Q;
    float* buf = smem_f;                   // chunk [NO][TC][TS] (TS >= D * S: [dof][S]); then the tile's sums [S][row]
    int* s_dof = (int*)(smem_f + a.buf_floats);          // [D] slot -> dof
    int* s_slot = s_dof + D;                             // [D] dof -> slot
    int* s_sup = s_slot + D;                             // [2][nb][lo, hi)
    const int tid = threadIdx.x;
    for (int i = tid; i < D; i += kGradThreads) {
        s_dof[i] = a.slot_to_dof[i];
        s_slot[a.slot_to_dof[i]] = i;
    }
    for (int i = tid; i < 4 * nb; i += kGradThreads) s_sup[i] = a.colsup[i];
    const long long n_tiles = (a.B + S - 1) / S;
    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const long long b0 = tile * S;
        const int ns = (int)((a.B - b0) < S ? (a.B - b0) : S);
        float acc[kGradItems][4];
#pragma unroll
        for (int m = 0; m < kGradItems; ++m) acc[m][0] = acc[m][1] = acc[m][2] = acc[m][3] = 0.0f;
        for (int t0 = 0; t0 < Tq; t0 += TC) {
            const int tc = Tq - t0 < TC ? Tq - t0 : TC;
            const int per_q = tc * D;
            __syncthreads();                             // tables ready / previous chunk or tile consumed
            // four trajectories per float4; four float4 per thread in flight before the first store (16 loads)
            const int total = NO * Q * per_q;
            const size_t stride = (size_t)Tq * D;
            for (int base = tid; base < total; base += 4 * kGradThreads) {
                float4 v[4];
                int dst[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int idx = base + u * kGradThreads;
                    dst[u] = -1;
                    v[u] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
                    if (idx >= total) continue;
                    const int e = idx % per_q, r = idx / per_q;
                    const int q = r % Q, o = r / Q;
                    const int t = e / D, dof = e - t * D;
                    const float* src = a.grad[o] + ((b0 + 4 * q) * Tq + t0) * D + e;
                    const int tr = 4 * q;
                    if (tr < ns) v[u].x = __ldcs(src);
                    if (tr + 1 < ns) v[u].y = __ldcs(src + stride);
                    if (tr + 2 < ns) v[u].z = __ldcs(src + 2 * stride);
                    if (tr + 3 < ns) v[u].w = __ldcs(src + 3 * stride);
                    dst[u] = (o * TC + t) * TS + dof * S + tr;
                }
#pragma unroll
                for (int u = 0; u < 4; ++u)
                    if (dst[u] >= 0) *(float4*)(buf + dst[u]) = v[u];
            }
            __syncthreads();
#pragma unroll
            for (int m = 0; m < kGradItems; ++m) {
                const int j = tid + m * kGradThreads;
                if (j >= n_items) continue;
                const int q = j % Q, sk = j / Q;
                const int slot = sk / nb, k = sk - slot * nb;
                const bool grip = slot >= a.n_joint;
                if (grip && !a.has0) continue;
                const int dof = s_dof[slot];
                const int2 sup = *(const int2*)(s_sup + 2 * ((grip ? nb : 0) + k));
                const int lo = sup.x > t0 ? sup.x : t0;
                const int hi = sup.y < t0 + tc ? sup.y : t0 + tc;
                const float* gq = buf + dof * S + 4 * q;
                if (grip) {
                    for (int t = lo; t < hi; ++t) {
                        const float r = __ldg(a.rows_grip0 + (size_t)t * nb + k);
                        const float4 g = *(const float4*)(gq + (size_t)(t - t0) * TS);
                        acc[m][0] = fmaf(r, g.x, acc[m][0]); acc[m][1] = fmaf(r, g.y, acc[m][1]);
                        acc[m][2] = fmaf(r, g.z, acc[m][2]); acc[m][3] = fmaf(r, g.w, acc[m][3]);
                    }
                } else {
                    for (int t = lo; t < hi; ++t) {
#pragma unroll
                        for (int o = 0; o < NO; ++o) {
                            const float r = __ldg(a.rows[o] + (size_t)t * nb + k);
                            const float4 g = *(const float4*)(gq + (size_t)(o * TC + t - t0) * TS);
                            acc[m][0] = fmaf(r, g.x, acc[m][0]); acc[m][1] = fmaf(r, g.y, acc[m][1]);
                            acc[m][2] = fmaf(r, g.z, acc[m][2]); acc[m][3] = fmaf(r, g.w, acc[m][3]);
                        }
                    }
                }
            }
        }
        __syncthreads();                                 // last chunk consumed: the buffer takes the sums
#pragma unroll
        for (int m = 0; m < kGradItems; ++m) {
            const int j = tid + m * kGradThreads;
            if (j >= n_items) continue;
            const int q = j % Q, sk = j / Q;
#pragma unroll
            for (int i = 0; i < 4; ++i) buf[(size_t)(4 * q + i) * row + sk] = acc[m][i];
        }
        __syncthreads();
        float* gp = a.grad_params + b0 * row;
        for (int idx = tid; idx < ns * row; idx += kGradThreads) {
            const int j = idx % row;
            const int slot = j / nb, k = j - slot * nb;
            const float v = (a.init_p_used && k == 0 && slot < a.n_joint) ? 0.0f : buf[idx];
            __stcs(gp + idx, v);
        }
        if (a.grad_init_p)
            for (int idx = tid; idx < ns * D; idx += kGradThreads) {
                const int tr = idx / D, dof = idx - tr * D;
                const int slot = s_slot[dof];
                a.grad_init_p[b0 * D + idx] = slot < a.n_joint ? buf[(size_t)tr * row + slot * nb] : 0.0f;
            }
    }
}

static int launch_grad_generic(const Plan* p, long long B, int Tq, const float* times, int times_stride,
                               const float* const grad[3], int init_p_used, float* grad_params, float* grad_init_p,
                               cudaStream_t st) {
    if (p->nc + p->degree_p + 1 > kMaxEvalKnots) return BEAST_E_UNSUPPORTED;
    GradGenericArgs a;
    a.B = B; a.Tq = Tq; a.times_stride = times_stride;
    a.D = p->D; a.nb = p->nb; a.n_joint = p->n_joint; a.degree_p = p->degree_p; a.ico = p->ico; a.nc = p->nc;
    a.slot_to_dof = p->slot_to_dof_d; a.times = times; a.knots_j = p->knots_joint_d; a.knots_g = p->knots_grip_d;
    a.tau = p->tau;
    a.max_order = 0;
    for (int o = 0; o < 3; ++o) {
        a.grad[o] = grad[o];
        if (grad[o]) a.max_order = o;
    }
    a.row_floats = (a.max_order + 1) * p->nc + (p->n_joint < p->D ? p->nb : 0);
    const size_t per_sample = ((size_t)a.row_floats + 3 * (size_t)p->D) * sizeof(float);
    int TC = (int)((size_t)(40 * 1024) / per_sample);
    if (TC > kGradGenericThreads) TC = kGradGenericThreads;
    if (TC < 1) TC = 1;
    a.TC = TC;
    a.init_p_used = init_p_used; a.grad_params = grad_params; a.grad_init_p = grad_init_p;
    const size_t smem = (size_t)TC * per_sample;
    static size_t granted[kMaxDevices] = {};
    if (int rc = opt_in_smem(deriv_grad_generic_kernel, smem, granted)) return rc;
    const long long cap = (long long)p->num_sms * 8;
    const int grid = (int)(B < cap ? B : cap);
    deriv_grad_generic_kernel<<<grid, kGradGenericThreads, smem, st>>>(a);
    count_launch();
    BEAST_CHECK_LAUNCH();
    return BEAST_OK;
}

template <int NO>
static int launch_grad_tiled_no(const GradTiledArgs& a, size_t smem, long long grid, cudaStream_t st) {
    static size_t granted[kMaxDevices] = {};
    if (int rc = opt_in_smem(deriv_grad_tiled_kernel<NO>, smem, granted)) return rc;
    deriv_grad_tiled_kernel<NO><<<(unsigned)grid, kGradThreads, smem, st>>>(a);
    return BEAST_OK;
}

static int launch_grad_tiled(const Plan* p, const Grid* gr, long long B, const float* const grad[3], int init_p_used,
                             float* grad_params, float* grad_init_p, cudaStream_t st) {
    const int Tq = gr->Tq, D = p->D, nb = p->nb, row = D * nb;
    if (p->nc != nb || !gr->colsup_d) return BEAST_E_UNSUPPORTED;
    if (row > kGradThreads * kGradItems) return BEAST_E_UNSUPPORTED;
    GradTiledArgs a;
    int no = 0;
    a.has0 = grad[0] != nullptr;
    for (int o = 0; o < 3; ++o) {
        if (!grad[o]) continue;
        a.rows[no] = gr->rows_j_d + (size_t)o * Tq * nb;
        a.grad[no] = grad[o];
        ++no;
    }
    for (int o = no; o < 3; ++o) { a.rows[o] = nullptr; a.grad[o] = nullptr; }
    a.rows_grip0 = gr->rows_g_d;
    // two CTAs per SM; a tile of at most 64 trajectories, and small batches spread over the CTA slots
    const long long slots = (long long)p->num_sms * 2;
    long long Q = (kGradThreads * kGradItems) / row;
    if (Q > 16) Q = 16;
    const long long q_spread = (B + 4 * slots - 1) / (4 * slots);
    if (Q > q_spread) Q = q_spread;
    if (Q < 1) Q = 1;
    const int S = 4 * (int)Q;
    const int TS = D * S + 4;                           // one float4 of padding per sample row: fewer bank conflicts
    const size_t budget_floats = (100 * 1024 - 16 * 1024) / sizeof(float);   // chunk / sums, below 100 KB in all
    int TC = (int)(budget_floats / ((size_t)no * TS));
    if (TC > Tq) TC = Tq;
    if (TC < 1) TC = 1;
    size_t buf = (size_t)no * TC * TS;
    if ((size_t)S * row > buf) buf = (size_t)S * row;
    buf = (buf + 3) & ~(size_t)3;
    const size_t smem = buf * sizeof(float) + ((size_t)2 * D + 4 * (size_t)nb) * sizeof(int);
    if (smem > (size_t)p->max_smem_optin) return BEAST_E_UNSUPPORTED;
    a.B = B; a.Tq = Tq; a.D = D; a.nb = nb; a.n_joint = p->n_joint; a.slot_to_dof = p->slot_to_dof_d;
    a.colsup = gr->colsup_d; a.S = S; a.Q = (int)Q; a.TC = TC; a.TS = TS; a.buf_floats = (int)buf;
    a.init_p_used = init_p_used; a.grad_params = grad_params; a.grad_init_p = grad_init_p;
    const long long n_tiles = (B + S - 1) / S;
    const long long grid = n_tiles < slots ? n_tiles : slots;
    const int rc = no == 1 ? launch_grad_tiled_no<1>(a, smem, grid, st)
                 : no == 2 ? launch_grad_tiled_no<2>(a, smem, grid, st) : launch_grad_tiled_no<3>(a, smem, grid, st);
    if (rc) return rc;
    count_launch();
    BEAST_CHECK_LAUNCH();
    return BEAST_OK;
}

// Shared argument checks of the two backward entry points.
static int check_grad_args(const Plan* p, int64_t B, const float* const grad[3], int32_t init_p_used,
                           const float* grad_params, const float* grad_init_p) {
    if (!p) return BEAST_E_NULL;
    if (!grad[0] && !grad[1] && !grad[2]) return BEAST_E_NULL;
    if (!grad_params) return BEAST_E_NULL;
    if (B < 0) return BEAST_E_SHAPE;
    if (grad_init_p && !init_p_used) return BEAST_E_SHAPE;           // no init_p in the forward: nothing to receive
    for (int o = 0; o < 3; ++o)
        if ((uintptr_t)grad[o] & 3u) return BEAST_E_ALIGN;
    if (((uintptr_t)grad_params & 3u) || ((uintptr_t)grad_init_p & 3u)) return BEAST_E_ALIGN;
    return BEAST_OK;
}

}  // namespace beast

using namespace beast;

extern "C" int beast_decode_grid_backward_f32(const beast_plan_t* plan, const beast_grid_t* grid, int64_t B,
                                              const float* grad0, const float* grad1, const float* grad2,
                                              int32_t init_p_used, float* grad_params, float* grad_init_p,
                                              void* stream) {
    const Plan* p = (const Plan*)plan;
    const Grid* g = (const Grid*)grid;
    const float* const grad[3] = {grad0, grad1, grad2};
    if (!g) return BEAST_E_NULL;
    if (int rc = check_grad_args(p, B, grad, init_p_used, grad_params, grad_init_p)) return rc;
    if (g->plan != p) return BEAST_E_SHAPE;
    for (int o = g->max_order + 1; o < 3; ++o)
        if (grad[o]) return BEAST_E_SHAPE;                          // the grid holds no rows of that order
    if (B == 0) return BEAST_OK;
    cudaStream_t st = (cudaStream_t)stream;
    const bool pinned = p->ico + p->eco > 0 && p->n_joint > 0;
    if (!pinned && !fast_paths_disabled()) {
        const int rc = launch_grad_tiled(p, g, B, grad, init_p_used, grad_params, grad_init_p, st);
        if (rc != BEAST_E_UNSUPPORTED) return rc;
    }
    return launch_grad_generic(p, B, g->Tq, g->times_d, 0, grad, init_p_used, grad_params, grad_init_p, st);
}

extern "C" int beast_decode_deriv_times_backward_f32(const beast_plan_t* plan, int64_t B, const float* times,
                                                     int32_t Tq, const float* grad0, const float* grad1,
                                                     const float* grad2, int32_t init_p_used, float* grad_params,
                                                     float* grad_init_p, void* stream) {
    const Plan* p = (const Plan*)plan;
    const float* const grad[3] = {grad0, grad1, grad2};
    if (int rc = check_grad_args(p, B, grad, init_p_used, grad_params, grad_init_p)) return rc;
    if (Tq < 0) return BEAST_E_SHAPE;
    if (B == 0) return BEAST_OK;
    if (Tq > 0 && !times) return BEAST_E_NULL;
    if ((uintptr_t)times & 3u) return BEAST_E_ALIGN;
    return launch_grad_generic(p, B, Tq, times, Tq, grad, init_p_used, grad_params, grad_init_p, (cudaStream_t)stream);
}
