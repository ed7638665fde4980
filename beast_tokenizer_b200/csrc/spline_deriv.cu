// Derivatives of the decoded action spline: position, velocity and acceleration (orders 0, 1, 2) on any time grid.
//
//   x^(o)(t) = (1/tau)^o * sum_k N_k^(o)(u(t)) * c_k (+ bias for o = 0),   u = clip(t / tau, 0, 1)
//
// with the coefficients of reconstruct_traj (dequantised tokens or given coefficients, init_p, pinned boundary
// control points).  The basis derivatives are the derivative form of the Cox-de Boor recursion,
// N'_{i,q} = q * (N_{i,q-1} / (k_{i+q} - k_i) - N_{i+1,q-1} / (k_{i+q+1} - k_{i+1})), zero-denominator terms dropped,
// taken from the levels below the top one that the recursion computes anyway; then divided by tau once per order.
// Outside [0, tau] (t / tau outside [0, 1]) orders 1 and 2 are exactly 0: the clamped phase holds the position.
// basis.py: bspline_basis_derivatives runs the same fp32 operation sequence on the host.
//
// Generic kernel: one thread per (trajectory, sample), basis and derivatives evaluated in-kernel; times per row
// ([B, Tq]) or one shared grid (row stride 0).  Order 0 is decode_generic_kernel's sum, bit for bit.
// Tiled kernel (one shared grid, no pinned points): the grid's host rows (a beast_grid_t), summed over the non-zero
// band of each row.  Only the tokens some row reads are loaded, dequantised once into shared memory; then one output
// sample per thread in output order, every requested order from the same coefficient loads.
#include <cstdlib>
#include <cstring>
#include <new>
#include "spline_deriv.cuh"

namespace beast {

constexpr int kDerivThreads = 512;

struct DerivGenericArgs {
    const long long* tokens;
    const float* params;
    long long n_rows;
    int Tq, times_stride;          // times of trajectory b start at times + b * times_stride (0: one shared grid)
    int D, nb, n_joint, degree_p, ico, eco;
    const int* slot_to_dof;
    const float* times;
    const float* knots_j;
    const float* knots_g;
    float tau;
    const float* w_min;
    const float* w_max;
    float vm1;
    long long offset;
    const float* init_p;
    const float* bc;
    const float* bias;
    float* out[3];                 // orders 0, 1, 2 (nullable)
};

template <bool FROM_TOKENS>
__global__ void __launch_bounds__(128, 2)     // 128 registers: the default 72 spilled
deriv_generic_kernel(const __grid_constant__ DerivGenericArgs a) {
    const int nb = a.nb, D = a.D, n_joint = a.n_joint, ico = a.ico, eco = a.eco;
    const int nc = nb + ico + eco, nbc = ico + eco;
    const int max_order = a.out[2] ? 2 : (a.out[1] ? 1 : 0);
    float N[kMaxEvalKnots], D1[kMaxEvalKnots], D2[kMaxEvalKnots], Ng[kMaxEvalKnots];
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < a.n_rows;
         idx += (long long)gridDim.x * blockDim.x) {
        const long long b = idx / a.Tq;
        const int t = (int)(idx - b * a.Tq);
        const float raw = __fdiv_rn(__fsub_rn(a.times[b * a.times_stride + t], 0.0f), a.tau);
        const float u = clampf(raw, 0.0f, 1.0f);
        const bool outside = raw < 0.0f || raw > 1.0f;
        deboor_deriv(a.knots_j, nc, a.degree_p, u, max_order, N, D1, D2);
        for (int i = 0; i < nc; ++i) {
            if (max_order >= 1) D1[i] = outside ? 0.0f : __fdiv_rn(D1[i], a.tau);
            if (max_order >= 2) D2[i] = outside ? 0.0f : __fdiv_rn(__fdiv_rn(D2[i], a.tau), a.tau);
        }
        if (n_joint < D) deboor_deriv(a.knots_g, nb, 0, u, 0, Ng, nullptr, nullptr);
        const long long row = (long long)D * nb;
        for (int slot = 0; slot < D; ++slot) {
            const int dof = a.slot_to_dof[slot];
            const bool joint = slot < n_joint;
            const bool pinned = nbc > 0 && joint;
            const float* pin = pinned ? a.bc + (b * n_joint + slot) * nbc : nullptr;
            float acc0 = 0.0f, acc1 = 0.0f, acc2 = 0.0f;
            if (pinned)
                for (int c = 0; c < ico; ++c) {
                    acc0 = fmaf(N[c], pin[c], acc0);
                    if (max_order >= 1) acc1 = fmaf(D1[c], pin[c], acc1);
                    if (max_order >= 2) acc2 = fmaf(D2[c], pin[c], acc2);
                }
            const float* r0 = joint ? N + ico : Ng;
            for (int k = 0; k < nb; ++k) {
                float c;
                if (FROM_TOKENS) {
                    const int j = slot * nb + k;
                    c = dequantize_one(a.tokens[b * row + (long long)k * D + slot] - a.offset, a.w_min[j], a.w_max[j], a.vm1);
                } else {
                    c = a.params[b * row + (long long)slot * nb + k];
                }
                if (k == 0 && a.init_p && joint) c = a.init_p[b * D + dof];
                acc0 = fmaf(r0[k], c, acc0);
                if (joint) {                                  // gripper slots are degree 0: orders 1 / 2 stay 0
                    if (max_order >= 1) acc1 = fmaf(D1[ico + k], c, acc1);
                    if (max_order >= 2) acc2 = fmaf(D2[ico + k], c, acc2);
                }
            }
            if (pinned) {
                for (int c = 0; c < eco; ++c) {
                    acc0 = fmaf(N[ico + nb + c], pin[ico + c], acc0);
                    if (max_order >= 1) acc1 = fmaf(D1[ico + nb + c], pin[ico + c], acc1);
                    if (max_order >= 2) acc2 = fmaf(D2[ico + nb + c], pin[ico + c], acc2);
                }
                if (a.bias) acc0 = __fadd_rn(acc0, a.bias[b * n_joint + slot]);
            }
            const long long o = idx * D + dof;
            if (a.out[0]) a.out[0][o] = acc0;
            if (a.out[1]) a.out[1][o] = acc1;
            if (a.out[2]) a.out[2][o] = acc2;
        }
    }
}

struct DerivTiledArgs {
    const long long* tokens;
    const float* params;
    long long B;
    int Tq, D, nb, n_joint;
    const int* slot_to_dof;
    const float* rows_j;           // [(max_order+1)][Tq][nb]
    const float* rows_g;
    const int* bands;
    const int* list;
    int n_dec;
    const float* w_min;
    const float* w_max;
    float vm1;
    long long offset;
    const float* init_p;
    const float* rows[3];          // rows of the NO requested orders (joint), in output order
    const float* rows_grip[3];
    float* out[3];
    int S, G1, G2;                 // trajectories per tile; trajectory groups per token entry / per output sample
    int qsplit, qchunk;            // a tile's output samples in qsplit slices of qchunk (small batches: more CTAs)
};

// NO = number of requested orders.  Phase 1 is decode_tiled_kernel's (spline_tiled.cu); phase 2 sums the band of one
// output sample for four trajectories per pass and every requested order: one coefficient load feeds NO sums, one
// basis load four.
template <bool FROM_TOKENS, int NO>
__global__ void __launch_bounds__(kDerivThreads, 2)
deriv_tiled_kernel(const __grid_constant__ DerivTiledArgs a) {
    extern __shared__ __align__(16) float smem_f[];
    const int Tq = a.Tq, D = a.D, nb = a.nb, S = a.S, n_dec = a.n_dec;
    const int row_in = D * nb, row_out = Tq * D;
    float* c_s = smem_f;                                            // [S][nb][D] coefficients, token order
    float* lohi = c_s + (((size_t)S * row_in + 3) & ~(size_t)3);    // [n_dec][2]
    int* lst = (int*)(lohi + (size_t)2 * n_dec);                    // [n_dec]
    int* s_dof = lst + n_dec;                                       // [D] slot -> dof
    int* s_slot = s_dof + D;                                        // [D] dof -> slot
    const int tid = threadIdx.x;
    const float rcp_vm1 = __frcp_rn(a.vm1);
    for (int i = tid; i < n_dec; i += kDerivThreads) {
        const int e = a.list[i];
        lst[i] = e;
        if (FROM_TOKENS) {
            const int k = e & 0xffff, slot = (e >> 16) & 0x7fff;
            lohi[2 * i] = a.w_min[slot * nb + k];
            lohi[2 * i + 1] = a.w_max[slot * nb + k];
        }
    }
    for (int i = tid; i < D; i += kDerivThreads) {
        s_dof[i] = a.slot_to_dof[i];
        s_slot[a.slot_to_dof[i]] = i;
    }
    const long long n_tiles = (a.B + S - 1) / S;
    const int items1 = n_dec * a.G1;
    const int nd = n_dec > 0 ? n_dec : 1;
    for (long long w = blockIdx.x; w < n_tiles * a.qsplit; w += gridDim.x) {
        const long long tile = w / a.qsplit;
        const int q0 = (int)(w - tile * a.qsplit) * a.qchunk;
        const int nq = row_out - q0 < a.qchunk ? row_out - q0 : a.qchunk;
        const int items2 = nq * a.G2;
        const long long b0 = tile * S;
        const int ns = (int)((a.B - b0) < S ? (a.B - b0) : S);
        __syncthreads();                                            // tables ready / previous tile's coefficients consumed
        const long long* tok_tile = FROM_TOKENS ? a.tokens + b0 * row_in : nullptr;
        const float* par_tile = FROM_TOKENS ? nullptr : a.params + b0 * row_in;
        const float* ip_tile = a.init_p ? a.init_p + b0 * D : nullptr;
        const int g1_step = kDerivThreads / nd, i1_step = kDerivThreads - g1_step * n_dec;
        int g = tid / nd, i = tid - g * n_dec;
        for (int j = tid; j < items1; j += kDerivThreads, g += g1_step, i += i1_step) {   // phase 1: tokens -> coefficients
            if (i >= n_dec) { i -= n_dec; ++g; }
            const int e = lst[i];
            const int k = e & 0xffff, slot = (e >> 16) & 0x7fff;
            const int r = k * D + slot;
            float lo = 0.0f, hi = 0.0f;
            if (FROM_TOKENS) { lo = lohi[2 * i]; hi = lohi[2 * i + 1]; }
            const int cpar = slot * nb + k;
            const int stride = a.G1 * row_in;
            for (int tr = g, off = g * row_in; tr < ns; tr += 4 * a.G1, off += 4 * stride) {
                const int o1 = off + stride, o2 = o1 + stride, o3 = o2 + stride;
                const bool h1 = tr + a.G1 < ns, h2 = tr + 2 * a.G1 < ns, h3 = tr + 3 * a.G1 < ns;
                float v0, v1 = 0.0f, v2 = 0.0f, v3 = 0.0f;
                if (FROM_TOKENS) {
                    const long long q0 = __ldcs(tok_tile + off + r);
                    const long long q1 = h1 ? __ldcs(tok_tile + o1 + r) : 0;
                    const long long q2 = h2 ? __ldcs(tok_tile + o2 + r) : 0;
                    const long long q3 = h3 ? __ldcs(tok_tile + o3 + r) : 0;
                    v0 = dequantize_fast(q0 - a.offset, lo, hi, a.vm1, rcp_vm1);
                    v1 = dequantize_fast(q1 - a.offset, lo, hi, a.vm1, rcp_vm1);
                    v2 = dequantize_fast(q2 - a.offset, lo, hi, a.vm1, rcp_vm1);
                    v3 = dequantize_fast(q3 - a.offset, lo, hi, a.vm1, rcp_vm1);
                } else {
                    v0 = par_tile[off + cpar];
                    if (h1) v1 = par_tile[o1 + cpar];
                    if (h2) v2 = par_tile[o2 + cpar];
                    if (h3) v3 = par_tile[o3 + cpar];
                }
                c_s[off + r] = v0;
                if (h1) c_s[o1 + r] = v1;
                if (h2) c_s[o2 + r] = v2;
                if (h3) c_s[o3 + r] = v3;
            }
            if (k == 0 && ip_tile != nullptr && slot < a.n_joint) {
                const int dof = s_dof[slot];
                for (int tr = g; tr < ns; tr += a.G1) c_s[tr * row_in + r] = ip_tile[tr * D + dof];
            }
        }
        __syncthreads();
        for (int j = tid; j < items2; j += kDerivThreads) {          // phase 2: one output sample per thread, output order
            const int g2 = j / nq, q = q0 + (j - g2 * nq);
            const int t = q / D, dof = q - t * D;
            const int slot = s_slot[dof];
            const bool grip = slot >= a.n_joint;
            const int2 band = __ldg((const int2*)a.bands + (grip ? Tq : 0) + t);
            const float* rw[NO];
#pragma unroll
            for (int o = 0; o < NO; ++o) rw[o] = (grip ? a.rows_grip[o] : a.rows[o]) + (size_t)t * nb;
            for (int tr = g2; tr < ns; tr += 4 * a.G2) {
                const int tr1 = tr + a.G2, tr2 = tr + 2 * a.G2, tr3 = tr + 3 * a.G2, last = ns - 1;
                const float* c0 = c_s + tr * row_in + slot;
                const float* c1 = c_s + (tr1 < last ? tr1 : last) * row_in + slot;
                const float* c2 = c_s + (tr2 < last ? tr2 : last) * row_in + slot;
                const float* c3 = c_s + (tr3 < last ? tr3 : last) * row_in + slot;
                float acc[NO][4];
#pragma unroll
                for (int o = 0; o < NO; ++o) acc[o][0] = acc[o][1] = acc[o][2] = acc[o][3] = 0.0f;
                for (int k = band.x; k < band.y; ++k) {
                    const int off = k * D;
                    const float v0 = c0[off], v1 = c1[off], v2 = c2[off], v3 = c3[off];
#pragma unroll
                    for (int o = 0; o < NO; ++o) {
                        const float pv = __ldg(rw[o] + k);
                        acc[o][0] = fmaf(pv, v0, acc[o][0]); acc[o][1] = fmaf(pv, v1, acc[o][1]);
                        acc[o][2] = fmaf(pv, v2, acc[o][2]); acc[o][3] = fmaf(pv, v3, acc[o][3]);
                    }
                }
#pragma unroll
                for (int o = 0; o < NO; ++o) {
                    float* dst = a.out[o] + (b0 + tr) * row_out + q;
                    __stcs(dst, acc[o][0]);
                    if (tr1 < ns) __stcs(dst + (size_t)a.G2 * row_out, acc[o][1]);
                    if (tr2 < ns) __stcs(dst + (size_t)2 * a.G2 * row_out, acc[o][2]);
                    if (tr3 < ns) __stcs(dst + (size_t)3 * a.G2 * row_out, acc[o][3]);
                }
            }
        }
    }
}

static int deriv_grid_for(long long n, int block, int num_sms) {
    long long g = (n + block - 1) / block;
    const long long cap = (long long)num_sms * 16;
    if (g > cap) g = cap;
    if (g < 1) g = 1;
    return (int)g;
}

static int launch_deriv_generic(const Plan* p, const long long* tokens, const float* params, long long B, int Tq,
                                const float* times, int times_stride, const float* w_min, const float* w_max,
                                long long offset, const float* init_p, const float* bc, const float* bias,
                                float* const out[3], cudaStream_t st) {
    if (p->nc + p->degree_p + 1 > kMaxEvalKnots) return BEAST_E_UNSUPPORTED;
    DerivGenericArgs a;
    a.tokens = tokens; a.params = params; a.n_rows = B * Tq; a.Tq = Tq; a.times_stride = times_stride;
    a.D = p->D; a.nb = p->nb; a.n_joint = p->n_joint; a.degree_p = p->degree_p; a.ico = p->ico; a.eco = p->eco;
    a.slot_to_dof = p->slot_to_dof_d; a.times = times; a.knots_j = p->knots_joint_d; a.knots_g = p->knots_grip_d;
    a.tau = p->tau; a.w_min = w_min; a.w_max = w_max; a.vm1 = tokens ? (float)(p->V - 1) : 0.0f;
    a.offset = tokens ? offset : 0; a.init_p = init_p; a.bc = bc; a.bias = bias;
    for (int o = 0; o < 3; ++o) a.out[o] = out[o];
    const int grid = deriv_grid_for(a.n_rows, 128, p->num_sms);
    if (tokens) deriv_generic_kernel<true><<<grid, 128, 0, st>>>(a);
    else deriv_generic_kernel<false><<<grid, 128, 0, st>>>(a);
    count_launch();
    BEAST_CHECK_LAUNCH();
    return BEAST_OK;
}

template <bool FROM_TOKENS, int NO>
static int launch_tiled_no(const DerivTiledArgs& a, size_t smem, long long grid, cudaStream_t st) {
    static size_t granted[kMaxDevices] = {};
    if (int rc = opt_in_smem(deriv_tiled_kernel<FROM_TOKENS, NO>, smem, granted)) return rc;
    deriv_tiled_kernel<FROM_TOKENS, NO><<<(unsigned)grid, kDerivThreads, smem, st>>>(a);
    return BEAST_OK;
}

static int launch_deriv_tiled(const Plan* p, const Grid* gr, const long long* tokens, const float* params, long long B,
                              const float* w_min, const float* w_max, long long offset, const float* init_p,
                              float* const out[3], cudaStream_t st) {
    const int Tq = gr->Tq, D = p->D, nb = p->nb;
    if (p->nc != nb || !gr->bands_d || !gr->list_d) return BEAST_E_UNSUPPORTED;
    if (nb > 0xffff || D > 0x7fff || (long long)Tq * D > 0x7fffffff / 4) return BEAST_E_UNSUPPORTED;
    const size_t row_in = (size_t)D * nb, row_out = (size_t)Tq * D;
    const size_t per_traj = row_in * sizeof(float);
    const size_t extra = ((size_t)3 * gr->n_dec + 2 * (size_t)D) * sizeof(float) + 64;
    size_t budget = 108 * 1024;                                     // two CTAs per SM, as the tiled decode
    if (per_traj + extra > budget) budget = (size_t)p->max_smem_optin;
    if (per_traj + extra > budget) return BEAST_E_UNSUPPORTED;
    int S = (int)((budget - extra) / per_traj);
    if (S > 64) S = 64;
    const size_t smem = (size_t)S * per_traj + extra;
    // a tile's output offsets are 32-bit: S * Tq * D < 2^31
    if ((long long)S * (long long)row_out >= 0x7fffffffLL) return BEAST_E_UNSUPPORTED;
    DerivTiledArgs a;
    a.tokens = tokens; a.params = params; a.B = B; a.Tq = Tq; a.D = D; a.nb = nb; a.n_joint = p->n_joint;
    a.slot_to_dof = p->slot_to_dof_d; a.rows_j = gr->rows_j_d; a.rows_g = gr->rows_g_d; a.bands = gr->bands_d;
    a.list = gr->list_d; a.n_dec = gr->n_dec;
    a.w_min = w_min; a.w_max = w_max; a.vm1 = tokens ? (float)(p->V - 1) : 0.0f; a.offset = tokens ? offset : 0;
    a.init_p = init_p;
    int no = 0;
    for (int o = 0; o < 3; ++o) {
        if (!out[o]) continue;
        a.rows[no] = gr->rows_j_d + (size_t)o * Tq * nb;
        a.rows_grip[no] = gr->rows_g_d ? gr->rows_g_d + (size_t)o * Tq * nb : a.rows[no];
        a.out[no] = out[o];
        ++no;
    }
    for (int o = no; o < 3; ++o) { a.rows[o] = nullptr; a.rows_grip[o] = nullptr; a.out[o] = nullptr; }
    a.S = S;
    auto groups = [&](long long entries) {
        long long g = entries > 0 ? (kDerivThreads + entries - 1) / entries : 1;
        if (g > S) g = S;
        return (int)(g < 1 ? 1 : g);
    };
    a.G1 = groups(gr->n_dec);
    const long long n_tiles = (B + S - 1) / S;
    long long per_sm = (long long)(220 * 1024) / (long long)(smem + 1024);
    if (per_sm > 2048 / kDerivThreads) per_sm = 2048 / kDerivThreads;
    if (per_sm < 1) per_sm = 1;
    const long long slots = (long long)p->num_sms * per_sm;
    // fewer tiles than CTA slots (small batches, long grids): every tile's output samples are dealt to several CTAs,
    // each of which dequantises the tile's tokens itself; slices of at least one thread's worth of samples per thread
    long long qsplit = n_tiles < slots ? slots / n_tiles : 1;
    const long long max_split = ((long long)row_out + kDerivThreads - 1) / kDerivThreads;
    if (qsplit > max_split) qsplit = max_split;
    if (qsplit < 1) qsplit = 1;
    a.qsplit = (int)qsplit;
    a.qchunk = (int)(((long long)row_out + qsplit - 1) / qsplit);
    a.G2 = groups(a.qchunk);
    const long long work = n_tiles * qsplit;
    const long long grid = work < slots ? work : slots;
    int rc;
    if (tokens) rc = no == 1 ? launch_tiled_no<true, 1>(a, smem, grid, st)
                   : no == 2 ? launch_tiled_no<true, 2>(a, smem, grid, st) : launch_tiled_no<true, 3>(a, smem, grid, st);
    else rc = no == 1 ? launch_tiled_no<false, 1>(a, smem, grid, st)
            : no == 2 ? launch_tiled_no<false, 2>(a, smem, grid, st) : launch_tiled_no<false, 3>(a, smem, grid, st);
    if (rc) return rc;
    count_launch();
    BEAST_CHECK_LAUNCH();
    return BEAST_OK;
}

// Shared argument checks of the two decode entry points.
static int check_deriv_args(const Plan* p, const int64_t* tokens, const float* params, int64_t B, const float* w_min,
                            const float* w_max, const float* init_p, const float* bc, float* const out[3]) {
    if (!p) return BEAST_E_NULL;
    if (!out[0] && !out[1] && !out[2]) return BEAST_E_NULL;
    if (tokens && params) return BEAST_E_SHAPE;
    if (B < 0) return BEAST_E_SHAPE;
    if (B > 0 && !tokens && !params) return BEAST_E_NULL;
    if (tokens && (!w_min || !w_max)) return BEAST_E_NULL;
    if (B > 0 && p->ico + p->eco > 0 && p->n_joint > 0 && !bc) return BEAST_E_NULL;   // pinned points are required
    if (((uintptr_t)tokens & 7u) || ((uintptr_t)params & 3u) || ((uintptr_t)init_p & 3u) || ((uintptr_t)bc & 3u))
        return BEAST_E_ALIGN;
    for (int o = 0; o < 3; ++o)
        if ((uintptr_t)out[o] & 3u) return BEAST_E_ALIGN;
    return BEAST_OK;
}

}  // namespace beast

using namespace beast;

extern "C" int beast_grid_create(const beast_plan_t* plan, const beast_grid_desc_t* d, beast_grid_t** out) {
    if (!plan || !d || !out) return BEAST_E_NULL;
    *out = nullptr;
    const Plan* p = (const Plan*)plan;
    if (d->n_times < 1 || d->max_order < 0 || d->max_order > 2) return BEAST_E_SHAPE;
    const bool has_grip = p->n_joint < p->D;
    if (!d->times_h || !d->rows_joint_h || (has_grip && !d->rows_grip_h)) return BEAST_E_NULL;
    const int Tq = d->n_times, nc = p->nc, nb = p->nb, no = d->max_order + 1;
    Grid* g = new (std::nothrow) Grid();
    if (!g) return BEAST_E_NOMEM;
    memset(g, 0, sizeof(Grid));
    g->plan = p; g->Tq = Tq; g->max_order = d->max_order;
    const size_t n_rj = (size_t)no * Tq * nc, n_rg = has_grip ? (size_t)no * Tq * nb : 0;
    const size_t total = (size_t)Tq + n_rj + n_rg;
    cudaError_t e = cudaMalloc((void**)&g->dev_block, total * sizeof(float));
    if (e != cudaSuccess) { beast_grid_destroy((beast_grid_t*)g); return (int)e; }
    g->times_d = g->dev_block;
    g->rows_j_d = g->times_d + Tq;
    g->rows_g_d = has_grip ? g->rows_j_d + n_rj : nullptr;
    e = cudaMemcpy(g->times_d, d->times_h, (size_t)Tq * sizeof(float), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(g->rows_j_d, d->rows_joint_h, n_rj * sizeof(float), cudaMemcpyHostToDevice);
    if (e == cudaSuccess && has_grip) e = cudaMemcpy(g->rows_g_d, d->rows_grip_h, n_rg * sizeof(float), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) { beast_grid_destroy((beast_grid_t*)g); return (int)e; }
    if (nc == nb && nb <= 0xffff && p->D <= 0x7fff) {
        // bands [joint | gripper][t] = union over the orders of the non-zero columns; the dec_list as in plan.cu
        int* bands = (int*)calloc((size_t)4 * Tq, sizeof(int));
        char* used = (char*)calloc((size_t)2 * nb, 1);
        int* list = (int*)malloc(((size_t)p->D * nb + 1) * sizeof(int));
        int* colsup = (int*)malloc((size_t)4 * nb * sizeof(int));    // column supports of the adjoint (no row: [0, 0))
        if (!bands || !used || !list || !colsup) {
            free(bands); free(used); free(list); free(colsup);
            beast_grid_destroy((beast_grid_t*)g);
            return BEAST_E_NOMEM;
        }
        for (int i = 0; i < 2 * nb; ++i) { colsup[2 * i] = Tq; colsup[2 * i + 1] = 0; }
        for (int side = 0; side < (has_grip ? 2 : 1); ++side) {
            const float* rows = side ? d->rows_grip_h : d->rows_joint_h;
            for (int t = 0; t < Tq; ++t) {
                int lo = nb, hi = 0;
                for (int o = 0; o < no; ++o)
                    for (int k = 0; k < nb; ++k)
                        if (rows[((size_t)o * Tq + t) * nb + k] != 0.0f) { if (k < lo) lo = k; if (k + 1 > hi) hi = k + 1; }
                if (lo >= hi) lo = hi = 0;
                bands[2 * (side * Tq + t)] = lo;
                bands[2 * (side * Tq + t) + 1] = hi;
                for (int k = lo; k < hi; ++k) {
                    used[side * nb + k] = 1;
                    int* cs = colsup + 2 * (side * nb + k);
                    if (t < cs[0]) cs[0] = t;
                    cs[1] = t + 1;
                }
                if (hi - lo > g->band_max) g->band_max = hi - lo;
            }
        }
        for (int i = 0; i < 2 * nb; ++i)
            if (colsup[2 * i] >= colsup[2 * i + 1]) colsup[2 * i] = colsup[2 * i + 1] = 0;
        int n_dec = 0;
        for (int k = 0; k < nb; ++k)
            for (int slot = 0; slot < p->D; ++slot) {
                const bool grip = slot >= p->n_joint;
                if (used[(grip ? nb : 0) + k]) list[n_dec++] = k | (slot << 16) | (grip ? (int)0x80000000u : 0);
            }
        g->n_dec = n_dec;
        e = cudaMalloc((void**)&g->bands_d, (size_t)4 * Tq * sizeof(int));
        if (e == cudaSuccess) e = cudaMemcpy(g->bands_d, bands, (size_t)4 * Tq * sizeof(int), cudaMemcpyHostToDevice);
        if (e == cudaSuccess) e = cudaMalloc((void**)&g->list_d, ((size_t)n_dec + 1) * sizeof(int));
        if (e == cudaSuccess && n_dec) e = cudaMemcpy(g->list_d, list, (size_t)n_dec * sizeof(int), cudaMemcpyHostToDevice);
        if (e == cudaSuccess) e = cudaMalloc((void**)&g->colsup_d, (size_t)4 * nb * sizeof(int));
        if (e == cudaSuccess) e = cudaMemcpy(g->colsup_d, colsup, (size_t)4 * nb * sizeof(int), cudaMemcpyHostToDevice);
        free(bands); free(used); free(list); free(colsup);
        if (e != cudaSuccess) { beast_grid_destroy((beast_grid_t*)g); return (int)e; }
    }
    *out = (beast_grid_t*)g;
    return BEAST_OK;
}

extern "C" int beast_grid_destroy(beast_grid_t* grid) {
    if (!grid) return BEAST_OK;
    Grid* g = (Grid*)grid;
    if (g->dev_block) cudaFree(g->dev_block);
    if (g->bands_d) cudaFree(g->bands_d);
    if (g->list_d) cudaFree(g->list_d);
    if (g->colsup_d) cudaFree(g->colsup_d);
    delete g;
    return BEAST_OK;
}

extern "C" int beast_decode_grid_f32(const beast_plan_t* plan, const beast_grid_t* grid, const int64_t* tokens,
                                     const float* params, int64_t B, const float* w_min, const float* w_max,
                                     int64_t offset, const float* init_p, const float* bc, const float* bias,
                                     float* out0, float* out1, float* out2, void* stream) {
    const Plan* p = (const Plan*)plan;
    const Grid* g = (const Grid*)grid;
    float* const out[3] = {out0, out1, out2};
    if (!g) return BEAST_E_NULL;
    if (int rc = check_deriv_args(p, tokens, params, B, w_min, w_max, init_p, bc, out)) return rc;
    if (g->plan != p) return BEAST_E_SHAPE;
    for (int o = g->max_order + 1; o < 3; ++o)
        if (out[o]) return BEAST_E_SHAPE;                           // the grid holds no rows of that order
    if (B == 0) return BEAST_OK;
    cudaStream_t st = (cudaStream_t)stream;
    const bool pinned = p->ico + p->eco > 0 && p->n_joint > 0;
    if (!pinned && !fast_paths_disabled()) {
        const int rc = launch_deriv_tiled(p, g, (const long long*)tokens, params, B, w_min, w_max, offset, init_p, out, st);
        if (rc != BEAST_E_UNSUPPORTED) return rc;
    }
    return launch_deriv_generic(p, (const long long*)tokens, params, B, g->Tq, g->times_d, 0, w_min, w_max, offset,
                                init_p, bc, bias, out, st);
}

extern "C" int beast_decode_deriv_times_f32(const beast_plan_t* plan, const int64_t* tokens, const float* params,
                                            int64_t B, const float* w_min, const float* w_max, int64_t offset,
                                            const float* init_p, const float* times, int32_t Tq, const float* bc,
                                            const float* bias, float* out0, float* out1, float* out2, void* stream) {
    const Plan* p = (const Plan*)plan;
    float* const out[3] = {out0, out1, out2};
    if (int rc = check_deriv_args(p, tokens, params, B, w_min, w_max, init_p, bc, out)) return rc;
    if (Tq < 0) return BEAST_E_SHAPE;
    if (B == 0 || Tq == 0) return BEAST_OK;
    if (!times) return BEAST_E_NULL;
    if ((uintptr_t)times & 3u) return BEAST_E_ALIGN;
    return launch_deriv_generic(p, (const long long*)tokens, params, B, Tq, times, Tq, w_min, w_max, offset, init_p,
                                bc, bias, out, (cudaStream_t)stream);
}
