// K3 — fused dequantise + B-spline evaluation  (replaces decode, beast/beast_bspline_tokenizer.py:483-496,
// reconstruct_traj :498-536 and UniformBSpline.get_traj_pos, mp/uni_bspline.py:114-177).
//
//   c[slot, k] = clamp(float(tok - offset)/(V-1) * (w_max - w_min) + w_min)       (beast/utils.py:20-26)
//   c[joint slot, 0] = init_p[dof]                       when init_p is given     (:505-510)
//   pos[t, dof(slot)] = sum_k Phi[t, k] * c[slot, k]                              (uni_bspline.py:165)
//
// Fast kernel (seq_len = 50, num_basis = 10, tokenizer's own times): the mirror image of K1 — one
// persistent CTA per SM cycling five shared-memory stages; bulk-TMA load of the int64 token tile
// (+ init_p), one thread per (trajectory, slot) column pulls its ten tokens into registers, the
// [t][dof] output rows are staged over the consumed tile and leave with one bulk store.
// Phi comes from the constant bank (uniform LDCU.128 loads); the degree-0 gripper basis has one
// non-zero per sample and is walked interval by interval.
// Generic kernel: any geometry, optional caller-supplied times [B, Tq] with the basis evaluated
// in-kernel by the Cox-de Boor recursion in the reference's fp32 operation order
// (basis_gn/uni_bspline_basis.py:82-113, phase_gn/linear_phase.py:22-23).
#include <cstdlib>
#include "common.cuh"

namespace beast {

constexpr int kDecGroupWarps = 7;
constexpr int kDecGroups = 2;
constexpr int kDecStages = 5;
constexpr int kDecCopyWarp = kDecGroups * kDecGroupWarps;
constexpr int kDecPdlWarp = kDecCopyWarp + 1;          // griddepcontrol only (as in K1)
constexpr int kDecThreads = (kDecPdlWarp + 1) * 32;
constexpr int kDecColumns = kDecGroupWarps * 32;

template <int T, int NB>
struct alignas(16) DecTables {
    static constexpr int NBP = (NB + 3) & ~3;
    float fj[T * NBP];   // Phi_joint [t][k], k padded
    float fgv[T];        // Phi_grip[t][k(t)] — the single non-zero of row t
    int gstart[NB + 1];  // rows gstart[k] <= t < gstart[k+1] belong to interval k
};

struct DecArgs {
    const long long* tokens;
    const float* init_p;
    float* out;
    const float* w_min;
    const float* w_max;
    long long offset;
    float vm1;
    int D, n_joint, S, n_tiles;
    int wait_first;        // 0 = may stream while the previous launch drains (disjoint buffers, common.cuh)
    int slot_to_dof[BEAST_MAX_SLOTS];
};

template <int T, int NB>
__device__ __forceinline__ void eval_joint(const DecTables<T, NB>& tab, const float (&c)[NB], float* __restrict__ o,
                                           int D) {
    constexpr int NBP = DecTables<T, NB>::NBP;
#pragma unroll
    for (int t = 0; t < T; ++t) {
        float acc = 0.0f;
#pragma unroll
        for (int k = 0; k < NB; ++k) acc = fmaf(tab.fj[t * NBP + k], c[k], acc);
        o[t * D] = acc;
    }
}

template <int T, int NB>
__device__ __forceinline__ void eval_grip(const DecTables<T, NB>& tab, const float (&c)[NB], float* __restrict__ o,
                                          int D) {
#pragma unroll
    for (int k = 0; k < NB; ++k) {
        const int t1 = tab.gstart[k + 1];
        for (int t = tab.gstart[k]; t < t1; ++t) o[t * D] = fmaf(tab.fgv[t], c[k], 0.0f);
    }
}

// Persistent CTA, one per SM; same stage life cycle as K1 (spline_encode.cu): bulk load of the token
// tile (+ init_p) -> one 7-warp group pulls its tokens into registers and evaluates -> [t][dof] rows
// staged over the tile -> bulk store -> reload.  Warp 15 and wait_first as in K1.
template <int T, int NB, int DT>
__global__ void __launch_bounds__(kDecThreads, 1)
decode_fast_kernel(const __grid_constant__ DecTables<T, NB> tab, const __grid_constant__ DecArgs a) {
    if (a.wait_first) pdl_wait();
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ __align__(8) uint64_t full_bar[kDecStages];
    __shared__ __align__(8) uint64_t out_full_bar[kDecStages];
    const int D = DT ? DT : a.D;
    const int S = a.S;
    const bool has_init = a.init_p != nullptr;
    const uint32_t tok_bytes = (uint32_t)S * NB * D * 8u;
    const uint32_t ini_bytes = (uint32_t)S * D * 4u;
    const uint32_t out_bytes = (uint32_t)S * T * D * 4u;
    const uint32_t load_bytes = tok_bytes + (has_init ? ini_bytes : 0u);
    const uint32_t stride = (out_bytes + 127u) & ~127u;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int first = blockIdx.x, step = gridDim.x;
    const int n_my = first < a.n_tiles ? (a.n_tiles - first + step - 1) / step : 0;
    const size_t tile_tok = (size_t)S * NB * D, tile_ini = (size_t)S * D, tile_out = (size_t)S * T * D;
    if (tid == 0) {
        for (int s = 0; s < kDecStages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&out_full_bar[s], kDecGroupWarps); }
        mbar_fence_init();
    }
    __syncthreads();

    if (warp == kDecPdlWarp) {
        pdl_wait();
        pdl_launch();
        return;
    }
    if (warp == kDecCopyWarp) {
        if (lane == 0) {
            auto load = [&](int j) {
                const int s = j % kDecStages;
                const size_t tile = (size_t)first + (size_t)j * step;
                mbar_arrive_expect_tx(&full_bar[s], load_bytes);
                bulk_g2s(smem + s * stride, a.tokens + tile * tile_tok, tok_bytes, &full_bar[s]);
                if (has_init) bulk_g2s(smem + s * stride + tok_bytes, a.init_p + tile * tile_ini, ini_bytes, &full_bar[s]);
            };
            for (int j = 0; j < kDecStages && j < n_my; ++j) load(j);
            for (int i = 0; i < n_my; ++i) {
                const int s = i % kDecStages;
                const size_t tile = (size_t)first + (size_t)i * step;
                mbar_wait(&out_full_bar[s], (i / kDecStages) & 1);
                bulk_s2g(a.out + tile * tile_out, smem + s * stride, out_bytes);
                bulk_commit();
                if (i + kDecStages < n_my) {
                    bulk_wait_read<0>();
                    load(i + kDecStages);
                }
            }
            bulk_wait_all<0>();
        }
        return;
    }

    const int group = warp / kDecGroupWarps;
    const int gtid = tid - group * (kDecGroupWarps * 32);
    const int nj = a.n_joint, ng = D - nj;
    const bool active = gtid < S * D;
    int tl = 0, slot = 0;
    if (active) {
        if (gtid < S * nj) { tl = gtid / nj; slot = gtid - tl * nj; }
        else { const int c = gtid - S * nj; tl = c / ng; slot = nj + (c - tl * ng); }
    }
    const int dof = a.slot_to_dof[slot];
    float wmin[NB], wmax[NB];
#pragma unroll
    for (int k = 0; k < NB; ++k) { wmin[k] = a.w_min[slot * NB + k]; wmax[k] = a.w_max[slot * NB + k]; }
    const float rcp_vm1 = __frcp_rn(a.vm1);

    for (int i = group; i < n_my; i += kDecGroups) {
        const int s = i % kDecStages;
        unsigned char* stage = smem + s * stride;
        mbar_wait(&full_bar[s], (i / kDecStages) & 1);
        float c[NB];
        if (active) {
            const long long* tk = (const long long*)stage + tl * (NB * D) + slot;
#pragma unroll
            for (int k = 0; k < NB; ++k) c[k] = dequantize_fast(tk[k * D] - a.offset, wmin[k], wmax[k], a.vm1, rcp_vm1);
            if (has_init && slot < nj) c[0] = ((const float*)(stage + tok_bytes))[tl * D + dof];
        }
        asm volatile("bar.sync %0, %1;" ::"r"(group + 1), "r"(kDecGroupWarps * 32) : "memory");   // tokens are in registers
        if (active) {
            float* o = (float*)stage + tl * (T * D) + dof;
            if (slot < nj) eval_joint<T, NB>(tab, c, o, D);
            else eval_grip<T, NB>(tab, c, o, D);
        }
        fence_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(&out_full_bar[s]);
    }
}

// Cox-de Boor on the knot vector `kn` (nb + p + 1 knots): N[0..nb) <- basis values at phase u.
// Level 0 exactly as uni_bspline_basis.py:94-104 (basis nb-1 closed on the right); higher levels
// as :106-113, terms with a zero denominator dropped.  In place, ascending i.
__device__ inline void deboor_basis(const float* __restrict__ kn, int nb, int p, float u, float* N) {
    const int n0 = nb + p;
    for (int i = 0; i < n0; ++i) {
        const bool in = (u >= kn[i]) && (i == nb - 1 ? (u <= kn[i + 1]) : (u < kn[i + 1]));
        N[i] = in ? 1.0f : 0.0f;
    }
    for (int k = 1; k <= p; ++k) {
        for (int i = 0; i < n0 - k; ++i) {
            const float d1 = __fsub_rn(kn[i + k], kn[i]);
            const float d2 = __fsub_rn(kn[i + k + 1], kn[i + 1]);
            const bool h1 = d1 != 0.0f, h2 = d2 != 0.0f;
            const float t1 = h1 ? __fmul_rn(__fdiv_rn(__fsub_rn(u, kn[i]), d1), N[i]) : 0.0f;
            const float t2 = h2 ? __fmul_rn(__fdiv_rn(__fsub_rn(kn[i + k + 1], u), d2), N[i + 1]) : 0.0f;
            N[i] = (h1 && h2) ? __fadd_rn(t1, t2) : (h1 ? t1 : t2);
        }
    }
}

// One thread per (trajectory, time sample): basis row from the plan's table or evaluated in-kernel,
// then every slot.  FROM_TOKENS: coefficients dequantised on the fly; else read from `params`.
template <bool FROM_TOKENS>
__global__ void __launch_bounds__(128)
decode_generic_kernel(const long long* __restrict__ tokens, const float* __restrict__ params, long long n_rows,
                      int Tq, int D, int nb, int n_joint, int degree_p, const int* __restrict__ slot_to_dof,
                      const float* __restrict__ phi_j, const float* __restrict__ phi_g,
                      const float* __restrict__ times, const float* __restrict__ knots_j,
                      const float* __restrict__ knots_g, float tau, const float* __restrict__ w_min,
                      const float* __restrict__ w_max, float vm1, long long offset,
                      const float* __restrict__ init_p, int ico, int eco, const float* __restrict__ bc,
                      const float* __restrict__ bias, float* __restrict__ out) {
    // Pinned control points (init/end condition orders, mp/uni_bspline.py:126-166): joint slot s of
    // trajectory b evaluates cat[bc[b,s,:ico], c[0..nb), bc[b,s,ico:]] against the nc-column basis and
    // adds bias[b,s] (the trajectory's init_pos).
    const int nc = nb + ico + eco, nbc = ico + eco;
    float Nj[kMaxEvalKnots];
    float Ng[kMaxEvalKnots];
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < n_rows;
         idx += (long long)gridDim.x * blockDim.x) {
        const long long b = idx / Tq;
        const int t = (int)(idx - b * Tq);
        const float* rj;
        const float* rg;
        if (times) {
            // linear_phase.py:22-23 with delay = 0: clip(t / tau, 0, 1)
            const float u = clampf(__fdiv_rn(__fsub_rn(times[idx], 0.0f), tau), 0.0f, 1.0f);
            deboor_basis(knots_j, nc, degree_p, u, Nj);
            rj = Nj;
            if (n_joint < D) deboor_basis(knots_g, nb, 0, u, Ng);
            rg = Ng;
        } else {
            rj = phi_j + (long long)t * nc;
            rg = phi_g + (long long)t * nb;
        }
        const long long row = (long long)D * nb;
        for (int slot = 0; slot < D; ++slot) {
            const int dof = slot_to_dof[slot];
            const bool pinned = nbc > 0 && slot < n_joint;
            const float* r = slot < n_joint ? rj + ico : rg;
            const float* pin = pinned ? bc + (b * n_joint + slot) * nbc : nullptr;
            float acc = 0.0f;
            if (pinned)
                for (int c = 0; c < ico; ++c) acc = fmaf(rj[c], pin[c], acc);
            for (int k = 0; k < nb; ++k) {
                float c;
                if (FROM_TOKENS) {
                    const int j = slot * nb + k;
                    c = dequantize_one(tokens[b * row + (long long)k * D + slot] - offset, w_min[j], w_max[j], vm1);
                } else {
                    c = params[b * row + (long long)slot * nb + k];
                }
                if (k == 0 && init_p && slot < n_joint) c = init_p[b * D + dof];
                acc = fmaf(r[k], c, acc);
            }
            if (pinned) {
                for (int c = 0; c < eco; ++c) acc = fmaf(rj[ico + nb + c], pin[ico + c], acc);
                if (bias) acc = __fadd_rn(acc, bias[b * n_joint + slot]);
            }
            out[idx * D + dof] = acc;
        }
    }
}

__global__ void __launch_bounds__(256)
dequantize_kernel(const long long* __restrict__ tokens, long long n, int D, int nb, const float* __restrict__ w_min,
                  const float* __restrict__ w_max, float vm1, long long offset, float* __restrict__ params_out) {
    const int row = D * nb;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < n;
         idx += (long long)gridDim.x * blockDim.x) {
        const long long b = idx / row;
        const int c = (int)(idx - b * row);          // output position slot*nb + k
        const int slot = c / nb, k = c - slot * nb;
        params_out[idx] = dequantize_one(tokens[b * row + (long long)k * D + slot] - offset, w_min[c], w_max[c], vm1);
    }
}

static inline bool dec_aligned16(const void* p) { return ((uintptr_t)p & 15u) == 0; }
static int dec_grid_for(long long n, int block, int num_sms) {
    long long g = (n + block - 1) / block;
    const long long cap = (long long)num_sms * 16;
    if (g > cap) g = cap;
    if (g < 1) g = 1;
    return (int)g;
}

// Degree-0 basis structure: one non-zero per row, rows of an interval contiguous.
template <int T, int NB>
static bool dec_grip_structure(const float* fg, float* fgv, int* gstart) {
    int k_prev = 0;
    for (int k = 0; k <= NB; ++k) gstart[k] = -1;
    gstart[0] = 0;
    for (int t = 0; t < T; ++t) {
        int kk = -1;
        for (int k = 0; k < NB; ++k) {
            if (fg[t * NB + k] != 0.0f) {
                if (kk >= 0) return false;
                kk = k;
            }
        }
        if (kk < 0) { fgv[t] = 0.0f; kk = k_prev; }
        else fgv[t] = fg[t * NB + kk];
        if (kk < k_prev) return false;
        for (int k = k_prev + 1; k <= kk; ++k) gstart[k] = t;
        k_prev = kk;
    }
    for (int k = k_prev + 1; k <= NB; ++k) gstart[k] = T;
    return true;
}

template <int T, int NB, int DT>
static int launch_dec_fast(const Plan* p, const long long* tokens, long long n_tiles, int S, const float* w_min,
                           const float* w_max, long long offset, const float* init_p, float* out,
                           cudaStream_t st) {
    DecTables<T, NB> tab;
    constexpr int NBP = DecTables<T, NB>::NBP;
    for (int t = 0; t < T; ++t)
        for (int k = 0; k < NBP; ++k) tab.fj[t * NBP + k] = k < NB ? p->phi_joint_h[t * NB + k] : 0.0f;
    if (p->phi_grip_h) {
        if (!dec_grip_structure<T, NB>(p->phi_grip_h, tab.fgv, tab.gstart)) return BEAST_E_UNSUPPORTED;
    } else {
        for (int t = 0; t < T; ++t) tab.fgv[t] = 0.0f;
        for (int k = 0; k <= NB; ++k) tab.gstart[k] = 0;
    }
    DecArgs a;
    a.tokens = tokens; a.init_p = init_p; a.out = out; a.w_min = w_min; a.w_max = w_max;
    a.offset = offset; a.vm1 = (float)(p->V - 1);
    a.D = p->D; a.n_joint = p->n_joint; a.S = S; a.n_tiles = (int)n_tiles;
    for (int i = 0; i < BEAST_MAX_SLOTS; ++i) a.slot_to_dof[i] = i < p->D ? p->slot_to_dof[i] : 0;
    static_assert(8 * NB + 4 <= 4 * T, "token tile (+ init_p) must fit under the output tile");
    const size_t smem = (size_t)kDecStages * ((((size_t)S * T * p->D * 4u) + 127u) & ~(size_t)127u);
    if ((int)smem > p->max_smem_optin) return BEAST_E_UNSUPPORTED;
    static size_t granted[kMaxDevices] = {};
    if (int rc = opt_in_smem(decode_fast_kernel<T, NB, DT>, smem, granted)) return rc;
    const int grid = (int)(n_tiles < p->num_sms ? n_tiles : p->num_sms);
    LaunchRanges rg;
    const size_t n_traj = (size_t)n_tiles * S, n_col = (size_t)p->D * NB;
    rg.add(tokens, n_traj * n_col * sizeof(long long), false);
    rg.add(init_p, n_traj * p->D * sizeof(float), false);
    rg.add(w_min, n_col * sizeof(float), false);
    rg.add(w_max, n_col * sizeof(float), false);
    rg.add(out, n_traj * T * p->D * sizeof(float), true);
    const bool overlap = overlap_begin(st, rg);
    a.wait_first = overlap ? 0 : 1;
    const cudaError_t e = launch_maybe_overlapped(decode_fast_kernel<T, NB, DT>, grid, kDecThreads, smem, st, overlap, tab, a);
    overlap_end(st, rg, overlap, e);
    count_launch();
    BEAST_CHECK_LAUNCH();
    return BEAST_OK;
}

static int launch_generic(const Plan* p, const long long* tokens, const float* params, long long B, int Tq,
                          const float* times, const float* w_min, const float* w_max, long long offset,
                          const float* init_p, const float* bc, const float* bias, float* out, cudaStream_t st) {
    if (times && p->nc + p->degree_p + 1 > kMaxEvalKnots) return BEAST_E_UNSUPPORTED;
    if ((p->ico + p->eco > 0) && p->n_joint > 0 && !bc) return BEAST_E_NULL;   // pinned points are required
    const long long n_rows = B * Tq;
    const int grid = dec_grid_for(n_rows, 128, p->num_sms);
    if (tokens)
        decode_generic_kernel<true><<<grid, 128, 0, st>>>(tokens, nullptr, n_rows, Tq, p->D, p->nb, p->n_joint,
                                                          p->degree_p, p->slot_to_dof_d, p->phi_joint_d, p->phi_grip_d,
                                                          times, p->knots_joint_d, p->knots_grip_d, p->tau, w_min,
                                                          w_max, (float)(p->V - 1), offset, init_p, p->ico, p->eco,
                                                          bc, bias, out);
    else
        decode_generic_kernel<false><<<grid, 128, 0, st>>>(nullptr, params, n_rows, Tq, p->D, p->nb, p->n_joint,
                                                           p->degree_p, p->slot_to_dof_d, p->phi_joint_d,
                                                           p->phi_grip_d, times, p->knots_joint_d, p->knots_grip_d,
                                                           p->tau, nullptr, nullptr, 0.0f, 0, init_p, p->ico, p->eco,
                                                           bc, bias, out);
    count_launch();
    BEAST_CHECK_LAUNCH();
    return BEAST_OK;
}

}  // namespace beast

using namespace beast;

extern "C" int beast_decode_f32(const beast_plan_t* plan, const int64_t* tokens, int64_t B, const float* w_min,
                                const float* w_max, int64_t offset, const float* init_p, float* traj_out,
                                void* stream) {
    const Plan* p = (const Plan*)plan;
    if (!p || !w_min || !w_max || (B > 0 && (!tokens || !traj_out))) return BEAST_E_NULL;
    if (B < 0) return BEAST_E_SHAPE;
    if (B == 0) return BEAST_OK;
    if (((uintptr_t)tokens & 7u) || ((uintptr_t)traj_out & 3u) || ((uintptr_t)init_p & 3u)) return BEAST_E_ALIGN;
    cudaStream_t st = (cudaStream_t)stream;
    const int T = p->T, D = p->D, nb = p->nb;
    long long done = 0;
    if (T == 50 && nb == 10 && p->nc == nb && !fast_paths_disabled() && dec_aligned16(tokens) && dec_aligned16(traj_out) &&
        (!init_p || dec_aligned16(init_p))) {
        const int S = (kDecColumns / D) & ~3;
        if (S >= 4 && B >= S) {
            const long long n_tiles = B / S;
            int rc;
            if (D == 14)
                rc = launch_dec_fast<50, 10, 14>(p, (const long long*)tokens, n_tiles, S, w_min, w_max, offset, init_p, traj_out, st);
            else if (D == 7)
                rc = launch_dec_fast<50, 10, 7>(p, (const long long*)tokens, n_tiles, S, w_min, w_max, offset, init_p, traj_out, st);
            else
                rc = launch_dec_fast<50, 10, 0>(p, (const long long*)tokens, n_tiles, S, w_min, w_max, offset, init_p, traj_out, st);
            if (rc == BEAST_OK) done = n_tiles * S;
            else if (rc != BEAST_E_UNSUPPORTED) return rc;
        }
    }
    if (done < B && !fast_paths_disabled()) {
        const int rc = launch_decode_tiled(p, (const long long*)tokens + done * (long long)D * nb, nullptr, B - done, w_min,
                                           w_max, offset, init_p ? init_p + done * D : nullptr,
                                           traj_out + done * (long long)T * D, st);
        if (rc == BEAST_OK) done = B;
        else if (rc != BEAST_E_UNSUPPORTED) return rc;
    }
    if (done < B)
        return launch_generic(p, (const long long*)tokens + done * (long long)D * nb, nullptr, B - done, T, nullptr,
                              w_min, w_max, offset, init_p ? init_p + done * D : nullptr, nullptr, nullptr,
                              traj_out + done * (long long)T * D, st);
    return BEAST_OK;
}

extern "C" int beast_decode_times_f32(const beast_plan_t* plan, const int64_t* tokens, int64_t B,
                                      const float* w_min, const float* w_max, int64_t offset, const float* init_p,
                                      const float* times, int32_t Tq, float* traj_out, void* stream) {
    const Plan* p = (const Plan*)plan;
    if (!p || !w_min || !w_max || (B > 0 && (!tokens || !traj_out || !times))) return BEAST_E_NULL;
    if (B < 0 || Tq < 0) return BEAST_E_SHAPE;
    if (B == 0 || Tq == 0) return BEAST_OK;
    return launch_generic(p, (const long long*)tokens, nullptr, B, Tq, times, w_min, w_max, offset, init_p, nullptr,
                          nullptr, traj_out, (cudaStream_t)stream);
}

extern "C" int beast_eval_f32(const beast_plan_t* plan, const float* params, int64_t B, const float* init_p,
                              const float* times, int32_t Tq, float* traj_out, void* stream) {
    const Plan* p = (const Plan*)plan;
    if (!p || (B > 0 && (!params || !traj_out))) return BEAST_E_NULL;
    if (B < 0 || Tq < 0) return BEAST_E_SHAPE;
    if (B == 0) return BEAST_OK;
    const int tq = times ? Tq : p->T;
    if (tq == 0) return BEAST_OK;
    if (!times && !fast_paths_disabled()) {
        const int rc = launch_decode_tiled(p, nullptr, params, B, nullptr, nullptr, 0, init_p, traj_out, (cudaStream_t)stream);
        if (rc != BEAST_E_UNSUPPORTED) return rc;
    }
    return launch_generic(p, nullptr, params, B, tq, times, nullptr, nullptr, 0, init_p, nullptr, nullptr, traj_out,
                          (cudaStream_t)stream);
}

extern "C" int beast_reconstruct_bc_f32(const beast_plan_t* plan, const int64_t* tokens, const float* params,
                                        int64_t B, const float* w_min, const float* w_max, int64_t offset,
                                        const float* init_p, const float* times, int32_t Tq, const float* bc,
                                        const float* bias, float* traj_out, void* stream) {
    const Plan* p = (const Plan*)plan;
    if (!p || (B > 0 && (!traj_out || (!tokens && !params)))) return BEAST_E_NULL;
    if (tokens && params) return BEAST_E_SHAPE;
    if (tokens && (!w_min || !w_max)) return BEAST_E_NULL;
    if (B < 0 || Tq < 0) return BEAST_E_SHAPE;
    if (B == 0) return BEAST_OK;
    const int tq = times ? Tq : p->T;
    if (tq == 0) return BEAST_OK;
    return launch_generic(p, (const long long*)tokens, params, B, tq, times, w_min, w_max, offset, init_p, bc, bias,
                          traj_out, (cudaStream_t)stream);
}

extern "C" int beast_dequantize_f32(const beast_plan_t* plan, const int64_t* tokens, int64_t B, const float* w_min,
                                    const float* w_max, int64_t offset, float* params_out, void* stream) {
    const Plan* p = (const Plan*)plan;
    if (!p || !w_min || !w_max || (B > 0 && (!tokens || !params_out))) return BEAST_E_NULL;
    if (B < 0) return BEAST_E_SHAPE;
    if (B == 0) return BEAST_OK;
    const long long n = (long long)B * p->D * p->nb;
    dequantize_kernel<<<dec_grid_for(n, 256, p->num_sms), 256, 0, (cudaStream_t)stream>>>(
        (const long long*)tokens, n, p->D, p->nb, w_min, w_max, (float)(p->V - 1), offset, params_out);
    count_launch();
    BEAST_CHECK_LAUNCH();
    return BEAST_OK;
}
