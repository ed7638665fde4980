// K1 — fused B-spline least-squares fit + quantisation  (replaces
// BEASTBsplineTokenizer.encode, beast/beast_bspline_tokenizer.py:399-428, and the
// UniformBSpline.learn_mp_params_from_trajs calls under it, mp/uni_bspline.py:471-602).
//
// Math: every trajectory shares self.times, so the reference's per-trajectory ridge solve
// collapses to  w[slot, k] = sum_t P[k, t] * y[t, dof(slot)]  with one P = (Phi^T Phi + 1e-9 I)^-1 Phi^T
// per spline (joint degree_p, gripper degree 0), computed once on the host.
//
// Fast kernel (seq_len = 50, num_basis = 10 — every BASELINE config): HBM-bound streaming.
//   * tile = S trajectories (S*D <= 224 columns, 44.8 KB); one persistent CTA per SM cycles five
//     shared-memory stages through load -> compute -> staged outputs -> store, two 7-warp groups
//     computing two tiles at once while the other stages have bulk copies in flight;
//   * every HBM byte moves by 1-D bulk TMA (cp.async.bulk, SASS UBLKCP): global->shared completes on
//     an mbarrier; the outputs are staged over the consumed input tile and leave with bulk
//     shared->global stores — 16-byte-aligned bursts, nothing through registers;
//   * one thread per (trajectory, slot) column: 50 LDS + 250 packed FFMA2 (fma.rn.f32x2: two fp32
//     FMAs per instruction) whose P operand pair comes from the constant bank (the table travels as
//     a __grid_constant__ kernel parameter and is read with uniform LDCU.128 loads straight into the
//     uniform-register operand of FFMA2), then the exact quantiser; joint columns fill warps 0-5, gripper
//     columns warp 6 (degree-0 projector = one non-zero per sample, walked interval by interval).
// Generic kernel: any geometry, one thread per column, same accumulation order (bit-identical
// coefficients), plain loads/stores.  Also handles the ragged tail of the fast path.
#include <cstdlib>
#include "common.cuh"

namespace beast {

constexpr int kEncGroupWarps = 7;                       // 224 columns per tile
constexpr int kEncGroups = 2;                           // tiles computed concurrently per SM
constexpr int kEncStages = 5;                           // 5 x 44.8 KB of the 227 KB shared memory
constexpr int kEncCopyWarp = kEncGroups * kEncGroupWarps;
constexpr int kEncPdlWarp = kEncCopyWarp + 1;          // griddepcontrol only: no copies, no compute
constexpr int kEncThreads = (kEncPdlWarp + 1) * 32;
constexpr int kEncColumns = kEncGroupWarps * 32;

__device__ __forceinline__ void group_barrier(int group) {
    asm volatile("bar.sync %0, %1;" ::"r"(group + 1), "r"(kEncGroupWarps * 32) : "memory");
}

// Projector tables as the kernel sees them.  Joint: [t][k] with k padded to a multiple of 4 so one
// 16-byte uniform constant load (LDCU.128) feeds four FFMAs.  Gripper (degree 0): sample t belongs
// to exactly one interval k, P_grip[k][t] = pgv[t] for gstart[k] <= t < gstart[k+1], zero elsewhere.
template <int T, int NB>
struct alignas(16) EncTables {
    static constexpr int NBP = (NB + 3) & ~3;
    float pj[T * NBP];
    float pgv[T];
    int gstart[NB + 1];
};

struct EncArgs {
    const float* traj;
    float* params_out;
    long long* tokens_out;
    const float* w_min;
    const float* w_max;
    float* bmin;           // optional [D*NB]: column min / max of the coefficients
    float* bmax;
    float* mm_ws;          // workspace of the single-launch reduction: [grid][2][D*NB] per-CTA partials + ticket; NULL = atomics
    int mm_accumulate;     // fold the existing contents of bmin / bmax into the result
    int wait_first;        // 0 = may stream while the previous launch drains (disjoint buffers, common.cuh)
    long long offset;
    float vm1;
    int D, n_joint, S, n_tiles;
    int slot_to_dof[BEAST_MAX_SLOTS];
};

template <int T, int NB>
__device__ __forceinline__ void fit_joint(const EncTables<T, NB>& tab, const float* __restrict__ y, int D,
                                          float (&acc)[NB]) {
    constexpr int NBP = EncTables<T, NB>::NBP;
    constexpr int NP = NB / 2;
    unsigned long long acc2[NP > 0 ? NP : 1];             // (k, k+1) accumulator pairs -> FFMA2
    float tail = 0.0f;
#pragma unroll
    for (int p = 0; p < NP; ++p) acc2[p] = 0ull;
#pragma unroll
    for (int t = 0; t < T; ++t) {
        const float v = y[t * D];
#pragma unroll
        for (int p = 0; p < NP; ++p) ffma2_bcast(acc2[p], tab.pj[t * NBP + 2 * p], tab.pj[t * NBP + 2 * p + 1], v);
        if (NB & 1) tail = fmaf(tab.pj[t * NBP + NB - 1], v, tail);
    }
#pragma unroll
    for (int p = 0; p < NP; ++p) { acc[2 * p] = lo_f32(acc2[p]); acc[2 * p + 1] = hi_f32(acc2[p]); }
    if (NB & 1) acc[NB - 1] = tail;
}

// Same sums as the dense form (the skipped terms are exact zeros), t ascending inside each interval.
template <int T, int NB>
__device__ __forceinline__ void fit_grip(const EncTables<T, NB>& tab, const float* __restrict__ y, int D,
                                         float (&acc)[NB]) {
#pragma unroll
    for (int k = 0; k < NB; ++k) {
        float s = 0.0f;
        const int t1 = tab.gstart[k + 1];
        for (int t = tab.gstart[k]; t < t1; ++t) s = fmaf(tab.pgv[t], y[t * D], s);
        acc[k] = s;
    }
}

// Persistent CTA, one per SM.  kEncStages tiles of shared memory cycle through
//   bulk load in flight -> computed by one 7-warp group -> outputs staged over the tile -> bulk store -> reload.
// Two groups compute two different tiles at once; the copy thread (warp 14, lane 0) issues every
// bulk copy.  full[s] (tx-count) hands a stage to its group, out_full[s] (7 warp arrivals) hands it back.
// Warp 15 waits for the previous grid and only then lets the next one launch (common.cuh: overlap_begin); with
// wait_first every thread waits before its first global access instead.
template <int T, int NB, int DT>
__global__ void __launch_bounds__(kEncThreads, 1)
encode_fast_kernel(const __grid_constant__ EncTables<T, NB> tab, const __grid_constant__ EncArgs a) {
    if (a.wait_first) pdl_wait();
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ __align__(8) uint64_t full_bar[kEncStages];
    __shared__ __align__(8) uint64_t out_full_bar[kEncStages];
    const int D = DT ? DT : a.D;          // compile-time DoF count for the common shapes (7, 14)
    const int S = a.S;
    const uint32_t in_bytes = (uint32_t)S * T * D * 4u;
    const uint32_t tok_bytes = (uint32_t)S * NB * D * 8u;
    const uint32_t par_bytes = (uint32_t)S * NB * D * 4u;
    const uint32_t stride = (in_bytes + 127u) & ~127u;
    const bool want_tok = a.tokens_out != nullptr, want_par = a.params_out != nullptr;
    const uint32_t par_off = want_tok ? tok_bytes : 0u;   // outputs staged over the consumed input tile

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int first = blockIdx.x, step = gridDim.x;
    const int n_my = first < a.n_tiles ? (a.n_tiles - first + step - 1) / step : 0;
    const size_t tile_in = (size_t)S * T * D, tile_out = (size_t)S * NB * D;
    // optional column min / max of the coefficients: CTA-level partials (shared-memory atomics),
    // then one global atomic per column and CTA
    __shared__ float s_mn[BEAST_MAX_SLOTS * NB];
    __shared__ float s_mx[BEAST_MAX_SLOTS * NB];
    const bool want_mm = a.bmin != nullptr;
    if (want_mm)
        for (int c = tid; c < D * NB; c += blockDim.x) { s_mn[c] = __int_as_float(0x7f800000); s_mx[c] = __int_as_float(0xff800000); }
    if (tid == 0) {
        for (int s = 0; s < kEncStages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&out_full_bar[s], kEncGroupWarps); }
        mbar_fence_init();
    }
    __syncthreads();

    if (warp == kEncPdlWarp) {
        pdl_wait();
        pdl_launch();
        return;
    }
    if (warp == kEncCopyWarp) {
        // ---------------- copy thread ----------------
        if (lane == 0) {
            auto load = [&](int j) {
                const int s = j % kEncStages;
                mbar_arrive_expect_tx(&full_bar[s], in_bytes);
                bulk_g2s(smem + s * stride, a.traj + ((size_t)first + (size_t)j * step) * tile_in, in_bytes, &full_bar[s]);
            };
            for (int j = 0; j < kEncStages && j < n_my; ++j) load(j);
            for (int i = 0; i < n_my; ++i) {
                const int s = i % kEncStages;
                const size_t tile = (size_t)first + (size_t)i * step;
                mbar_wait(&out_full_bar[s], (i / kEncStages) & 1);
                if (want_tok) bulk_s2g(a.tokens_out + tile * tile_out, smem + s * stride, tok_bytes);
                if (want_par) bulk_s2g(a.params_out + tile * tile_out, smem + s * stride + par_off, par_bytes);
                bulk_commit();
                if (i + kEncStages < n_my) {
                    bulk_wait_read<0>();                   // the stage has been drained -> refill it
                    load(i + kEncStages);
                }
            }
            bulk_wait_all<0>();
        }
        return;
    }

    // ---------------- compute groups: one (trajectory, slot) column per thread ----------------
    const int group = warp / kEncGroupWarps;
    const int gtid = tid - group * (kEncGroupWarps * 32);
    const int nj = a.n_joint, ng = D - nj;
    const bool active = gtid < S * D;
    int tl = 0, slot = 0;
    if (active) {
        if (gtid < S * nj) { tl = gtid / nj; slot = gtid - tl * nj; }     // joint columns first: uniform warps
        else { const int c = gtid - S * nj; tl = c / ng; slot = nj + (c - tl * ng); }
    }
    const int dof = a.slot_to_dof[slot];
    QuantCol qc[NB];
#pragma unroll
    for (int k = 0; k < NB; ++k)
        qc[k].init(want_tok ? a.w_min[slot * NB + k] : 0.0f, want_tok ? a.w_max[slot * NB + k] : 0.0f);

    float tmin[NB], tmax[NB];
#pragma unroll
    for (int k = 0; k < NB; ++k) { tmin[k] = __int_as_float(0x7f800000); tmax[k] = __int_as_float(0xff800000); }

    for (int i = group; i < n_my; i += kEncGroups) {
        const int s = i % kEncStages;
        unsigned char* stage = smem + s * stride;
        mbar_wait(&full_bar[s], (i / kEncStages) & 1);
        float acc[NB];
        if (active) {
            const float* y = (const float*)stage + tl * (T * D) + dof;
            if (slot < nj) fit_joint<T, NB>(tab, y, D, acc);
            else fit_grip<T, NB>(tab, y, D, acc);
        }
        if (want_mm && active) {
#pragma unroll
            for (int k = 0; k < NB; ++k) { tmin[k] = fminf(tmin[k], acc[k]); tmax[k] = fmaxf(tmax[k], acc[k]); }
        }
        // every column of the tile has been read before the outputs overwrite it (the reduction-only launch of
        // update_weights_bounds writes nothing: its warps release the stage one by one and run ahead)
        if (want_tok || want_par) group_barrier(group);
        if (active) {
            if (want_tok) {
                long long* to = (long long*)stage + tl * (NB * D) + slot;
#pragma unroll
                for (int k = 0; k < NB; ++k) to[k * D] = quantize_col(acc[k], qc[k], a.vm1) + a.offset;
            }
            if (want_par) {
                float* po = (float*)(stage + par_off) + tl * (NB * D) + slot * NB;
                if (NB % 2 == 0) {
#pragma unroll
                    for (int k = 0; k < NB; k += 2) *(float2*)(po + k) = make_float2(acc[k], acc[k + 1]);
                } else {
#pragma unroll
                    for (int k = 0; k < NB; ++k) po[k] = acc[k];
                }
            }
        }
        fence_async_smem();                                // generic-proxy writes -> visible to the bulk store
        __syncwarp();
        if (lane == 0) mbar_arrive(&out_full_bar[s]);
    }
    if (want_mm) {
        // a thread keeps its (slot) columns for the whole launch: registers -> shared -> global
        if (active && n_my > group) {
#pragma unroll
            for (int k = 0; k < NB; ++k) {
                atomic_min_f32(&s_mn[slot * NB + k], tmin[k]);
                atomic_max_f32(&s_mx[slot * NB + k], tmax[k]);
            }
        }
        constexpr int kComputeThreads = kEncGroups * kEncGroupWarps * 32;
        asm volatile("bar.sync %0, %1;" ::"r"(kEncGroups + 1), "r"(kComputeThreads) : "memory");
        const int n_col = D * NB;
        if (a.mm_ws == nullptr) {
            for (int c = tid; c < n_col; c += kComputeThreads) {
                if (s_mn[c] <= s_mx[c]) { atomic_min_f32(a.bmin + c, s_mn[c]); atomic_max_f32(a.bmax + c, s_mx[c]); }
            }
        } else {
            // single-launch reduction: every CTA stores its partials, the LAST one to arrive (ticket) combines
            // them and writes the result with plain stores — no initialisation pass, no float atomics, and the
            // caller can pass the tokenizer's own w_min / w_max as the destination
            float* part = a.mm_ws + (size_t)blockIdx.x * 2 * n_col;
            unsigned int* ticket = (unsigned int*)(a.mm_ws + (size_t)gridDim.x * 2 * n_col);
            for (int c = tid; c < n_col; c += kComputeThreads) { part[c] = s_mn[c]; part[n_col + c] = s_mx[c]; }
            __threadfence();
            asm volatile("bar.sync %0, %1;" ::"r"(kEncGroups + 1), "r"(kComputeThreads) : "memory");
            __shared__ int s_last;
            if (tid == 0) s_last = atomicAdd(ticket, 1u) == gridDim.x - 1 ? 1 : 0;
            asm volatile("bar.sync %0, %1;" ::"r"(kEncGroups + 1), "r"(kComputeThreads) : "memory");
            if (s_last) {
                __threadfence();
                for (int c = tid; c < n_col; c += kComputeThreads) {
                    float mn = a.mm_accumulate ? a.bmin[c] : __int_as_float(0x7f800000);
                    float mx = a.mm_accumulate ? a.bmax[c] : __int_as_float(0xff800000);
                    for (unsigned int bk = 0; bk < gridDim.x; ++bk) {
                        const float* q = a.mm_ws + (size_t)bk * 2 * n_col;
                        mn = fminf(mn, __ldcg(q + c));
                        mx = fmaxf(mx, __ldcg(q + n_col + c));
                    }
                    a.bmin[c] = mn;
                    a.bmax[c] = mx;
                }
                if (tid == 0) *ticket = 0u;                    // ready for the next launch
            }
        }
    }
}

// One thread per (trajectory, slot) column; any geometry.  Accumulates in the same order
// (t ascending, fused multiply-add) as the fast kernel.
__global__ void __launch_bounds__(256)
encode_generic_kernel(const float* __restrict__ traj, long long ncol, int T, int D, int nb, int n_joint,
                      const int* __restrict__ slot_to_dof, const float* __restrict__ Pj,
                      const float* __restrict__ Pg, const float* __restrict__ w_min,
                      const float* __restrict__ w_max, float vm1, long long offset,
                      float* __restrict__ params_out, long long* __restrict__ tokens_out,
                      float* __restrict__ bmin, float* __restrict__ bmax) {
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < ncol;
         idx += (long long)gridDim.x * blockDim.x) {
        const long long b = idx / D;
        const int slot = (int)(idx - b * D);
        const int dof = slot_to_dof[slot];
        const float* P = slot < n_joint ? Pj : Pg;
        const float* y = traj + b * (long long)T * D + dof;
        for (int k = 0; k < nb; ++k) {
            float acc = 0.0f;
            const float* pk = P + (long long)k * T;
            for (int t = 0; t < T; ++t) acc = fmaf(__ldg(pk + t), __ldg(y + (long long)t * D), acc);
            if (params_out) params_out[b * (long long)D * nb + (long long)slot * nb + k] = acc;
            if (bmin) { atomic_min_f32(bmin + slot * nb + k, acc); atomic_max_f32(bmax + slot * nb + k, acc); }
            if (tokens_out) {
                const float lo = w_min[slot * nb + k], hi = w_max[slot * nb + k];
                tokens_out[b * (long long)D * nb + (long long)k * D + slot] =
                    quantize_one(acc, lo, hi, quant_scale(lo, hi), vm1) + offset;
            }
        }
    }
}

// params '(d t)' -> tokens '(t d)' (bit-exact quantiser) or normalised fp32 '(t d)'.
template <bool NORMALIZE>
__global__ void __launch_bounds__(256)
quantize_kernel(const float* __restrict__ params, long long n, int D, int nb, const float* __restrict__ w_min,
                const float* __restrict__ w_max, float vm1, long long offset, long long* __restrict__ tokens_out,
                float* __restrict__ norm_out) {
    const int row = D * nb;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < n;
         idx += (long long)gridDim.x * blockDim.x) {
        const long long b = idx / row;
        const int r = (int)(idx - b * row);          // output position k*D + slot
        const int k = r / D, slot = r - k * D;
        const int c = slot * nb + k;
        const float w = params[b * row + c], lo = w_min[c], hi = w_max[c];
        if (NORMALIZE) {
            // beast/utils.py:32-34 with norm_min=-1, norm_max=1: (clip-lo)/scale * 2.0 + (-1.0)
            const float nrm = __fdiv_rn(__fsub_rn(clampf(w, lo, hi), lo), quant_scale(lo, hi));
            norm_out[idx] = __fadd_rn(__fmul_rn(nrm, 2.0f), -1.0f);
        } else {
            tokens_out[idx] = quantize_one(w, lo, hi, quant_scale(lo, hi), vm1) + offset;
        }
    }
}


static inline bool aligned16(const void* p) { return ((uintptr_t)p & 15u) == 0; }

static int grid_for(long long n, int block, int num_sms) {
    long long g = (n + block - 1) / block;
    const long long cap = (long long)num_sms * 16;
    if (g > cap) g = cap;
    if (g < 1) g = 1;
    return (int)g;
}

// Degree-0 projector structure: exactly one non-zero per sample, intervals contiguous in t.
template <int T, int NB>
static bool grip_structure(const float* pg, float* pgv, int* gstart) {
    int k_prev = 0;
    for (int k = 0; k <= NB; ++k) gstart[k] = -1;
    gstart[0] = 0;
    for (int t = 0; t < T; ++t) {
        int kk = -1;
        for (int k = 0; k < NB; ++k) {
            if (pg[k * T + t] != 0.0f) {
                if (kk >= 0) return false;
                kk = k;
            }
        }
        if (kk < 0) { pgv[t] = 0.0f; kk = k_prev; }        // sample outside every interval: contributes 0
        else pgv[t] = pg[kk * T + t];
        if (kk < k_prev) return false;
        for (int k = k_prev + 1; k <= kk; ++k) gstart[k] = t;
        k_prev = kk;
    }
    for (int k = k_prev + 1; k <= NB; ++k) gstart[k] = T;
    return true;
}

template <int T, int NB, int DT>
static int launch_fast(const Plan* p, const float* traj, long long n_tiles, int S, const float* w_min,
                       const float* w_max, long long offset, float* params_out, long long* tokens_out,
                       float* bmin, float* bmax, float* mm_ws, int mm_accumulate, cudaStream_t st) {
    const int D = p->D;
    EncTables<T, NB> tab;
    constexpr int NBP = EncTables<T, NB>::NBP;
    for (int t = 0; t < T; ++t)
        for (int k = 0; k < NBP; ++k) tab.pj[t * NBP + k] = k < NB ? p->proj_joint_h[k * T + t] : 0.0f;
    if (p->proj_grip_h) {
        if (!grip_structure<T, NB>(p->proj_grip_h, tab.pgv, tab.gstart)) return BEAST_E_UNSUPPORTED;
    } else {
        for (int t = 0; t < T; ++t) tab.pgv[t] = 0.0f;
        for (int k = 0; k <= NB; ++k) tab.gstart[k] = 0;
    }
    EncArgs a;
    a.traj = traj; a.params_out = params_out; a.tokens_out = tokens_out;
    a.w_min = w_min; a.w_max = w_max; a.bmin = bmin; a.bmax = bmax; a.offset = offset; a.vm1 = (float)(p->V - 1);
    a.mm_ws = mm_ws; a.mm_accumulate = mm_accumulate;
    a.D = p->D; a.n_joint = p->n_joint; a.S = S; a.n_tiles = (int)n_tiles;
    for (int i = 0; i < BEAST_MAX_SLOTS; ++i) a.slot_to_dof[i] = i < p->D ? p->slot_to_dof[i] : 0;
    // outputs (12 B * NB per column) alias the 4*T B per column input tile
    const size_t smem = (size_t)kEncStages * ((((size_t)S * T * p->D * 4u) + 127u) & ~(size_t)127u);
    static_assert(12 * NB <= 4 * T, "staged outputs must fit over the input tile");
    if ((int)smem > p->max_smem_optin) return BEAST_E_UNSUPPORTED;
    static size_t granted[kMaxDevices] = {};
    if (int rc = opt_in_smem(encode_fast_kernel<T, NB, DT>, smem, granted)) return rc;
    const int grid = (int)(n_tiles < p->num_sms ? n_tiles : p->num_sms);
    LaunchRanges rg;
    const size_t n_traj = (size_t)n_tiles * S, n_col = (size_t)D * NB;
    rg.add(traj, n_traj * T * D * sizeof(float), false);
    if (tokens_out) { rg.add(w_min, n_col * sizeof(float), false); rg.add(w_max, n_col * sizeof(float), false); }
    rg.add(params_out, n_traj * n_col * sizeof(float), true);
    rg.add(tokens_out, n_traj * n_col * sizeof(long long), true);
    rg.add(bmin, n_col * sizeof(float), true);
    rg.add(bmax, n_col * sizeof(float), true);
    rg.add(mm_ws, (size_t)beast_fit_minmax_workspace_bytes((const beast_plan_t*)p), true);   // partials + ticket
    const bool overlap = overlap_begin(st, rg);
    a.wait_first = overlap ? 0 : 1;
    const cudaError_t e = launch_maybe_overlapped(encode_fast_kernel<T, NB, DT>, grid, kEncThreads, smem, st, overlap, tab, a);
    overlap_end(st, rg, overlap, e);
    count_launch();
    BEAST_CHECK_LAUNCH();
    return BEAST_OK;
}


// Shared body of beast_encode_f32 / beast_fit_minmax_f32.
static int encode_impl(const Plan* p, const float* traj, long long B, const float* w_min, const float* w_max,
                       long long offset, float* params_out, long long* tokens_out, float* bmin, float* bmax,
                       cudaStream_t st, float* mm_ws = nullptr, int mm_accumulate = 1, bool* fast_ran = nullptr) {
    const int T = p->T, D = p->D, nb = p->nb;
    long long done = 0;
    if (T == 50 && nb == 10 && !fast_paths_disabled() && aligned16(traj) && (!params_out || aligned16(params_out)) &&
        (!tokens_out || aligned16(tokens_out))) {
        const int S = (kEncColumns / D) & ~3;
        if (S >= 4 && B >= S) {
            const long long n_tiles = B / S;
            int rc;
            if (D == 14)
                rc = launch_fast<50, 10, 14>(p, traj, n_tiles, S, w_min, w_max, offset, params_out, tokens_out, bmin, bmax, mm_ws, mm_accumulate, st);
            else if (D == 7)
                rc = launch_fast<50, 10, 7>(p, traj, n_tiles, S, w_min, w_max, offset, params_out, tokens_out, bmin, bmax, mm_ws, mm_accumulate, st);
            else
                rc = launch_fast<50, 10, 0>(p, traj, n_tiles, S, w_min, w_max, offset, params_out, tokens_out, bmin, bmax, mm_ws, mm_accumulate, st);
            if (rc == BEAST_OK) { done = n_tiles * S; if (fast_ran) *fast_ran = true; }
            else if (rc != BEAST_E_UNSUPPORTED) return rc;
        }
    }
    if (done < B && !fast_paths_disabled()) {
        // any other geometry (and long ragged tails): tiles of trajectories through shared memory
        const int rc = launch_encode_tiled(p, traj + done * (long long)T * D, B - done, w_min, w_max, offset,
                                           params_out ? params_out + done * (long long)D * nb : nullptr,
                                           tokens_out ? tokens_out + done * (long long)D * nb : nullptr, bmin, bmax, st);
        if (rc == BEAST_OK) done = B;
        else if (rc != BEAST_E_UNSUPPORTED) return rc;
    }
    if (done < B) {
        const long long ncol = (B - done) * D;
        encode_generic_kernel<<<grid_for(ncol, 256, p->num_sms), 256, 0, st>>>(
            traj + done * (long long)T * D, ncol, T, D, nb, p->n_joint, p->slot_to_dof_d, p->proj_joint_d,
            p->proj_grip_d, w_min, w_max, (float)(p->V - 1), offset,
            params_out ? params_out + done * (long long)D * nb : nullptr,
            tokens_out ? tokens_out + done * (long long)D * nb : nullptr, bmin, bmax);
        count_launch();
        BEAST_CHECK_LAUNCH();
    }
    return BEAST_OK;
}

__global__ void bounds_init_kernel(float* mn, float* mx, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) { mn[i] = __int_as_float(0x7f800000); mx[i] = __int_as_float(0xff800000); }
}

}  // namespace beast

using namespace beast;

extern "C" int beast_encode_f32(const beast_plan_t* plan, const float* traj, int64_t B, const float* w_min,
                                const float* w_max, int64_t offset, float* params_out, int64_t* tokens_out,
                                void* stream) {
    const Plan* p = (const Plan*)plan;
    if (!p) return BEAST_E_NULL;
    if (B < 0) return BEAST_E_SHAPE;
    if (B == 0) return BEAST_OK;
    if (!traj || (!params_out && !tokens_out)) return BEAST_E_NULL;
    if (tokens_out && (!w_min || !w_max)) return BEAST_E_NULL;
    if (((uintptr_t)traj & 3u) || ((uintptr_t)params_out & 3u) || ((uintptr_t)tokens_out & 7u)) return BEAST_E_ALIGN;
    return encode_impl(p, traj, B, w_min, w_max, offset, params_out, (long long*)tokens_out, nullptr, nullptr,
                       (cudaStream_t)stream);
}

extern "C" int beast_fit_minmax_f32(const beast_plan_t* plan, const float* traj, int64_t B, float* min_out,
                                    float* max_out, int32_t accumulate, void* stream) {
    return beast_fit_minmax_ws_f32(plan, traj, B, min_out, max_out, accumulate, nullptr, 0, stream);
}

extern "C" int64_t beast_fit_minmax_workspace_bytes(const beast_plan_t* plan) {
    const Plan* p = (const Plan*)plan;
    if (!p) return 0;
    return ((int64_t)p->num_sms * 2 * p->D * p->nb + 4) * (int64_t)sizeof(float);
}

extern "C" int beast_fit_minmax_ws_f32(const beast_plan_t* plan, const float* traj, int64_t B, float* min_out,
                                       float* max_out, int32_t accumulate, void* workspace, int64_t workspace_bytes,
                                       void* stream) {
    const Plan* p = (const Plan*)plan;
    if (!p || !min_out || !max_out) return BEAST_E_NULL;
    if (B < 0) return BEAST_E_SHAPE;
    if (B > 0 && !traj) return BEAST_E_NULL;
    if ((uintptr_t)traj & 3u) return BEAST_E_ALIGN;
    cudaStream_t st = (cudaStream_t)stream;
    const int n = p->D * p->nb;
    float* ws = (workspace && workspace_bytes >= beast_fit_minmax_workspace_bytes(plan) && !((uintptr_t)workspace & 3u))
                    ? (float*)workspace : nullptr;
    // With a workspace the tiled kernel reduces in ONE launch (its last CTA combines the per-CTA partials and writes
    // min_out / max_out with plain stores, folding the previous contents in when accumulate != 0); the ragged tail
    // then accumulates with atomics.  Without one (or when no full tile exists) the outputs are initialised first.
    const int S = (kEncColumns / p->D) & ~3;
    const bool tiled = ws && p->T == 50 && p->nb == 10 && !fast_paths_disabled() && S >= 4 && B >= S && aligned16(traj);
    if (!tiled) {
        if (!accumulate) {
            bounds_init_kernel<<<(n + 255) / 256, 256, 0, st>>>(min_out, max_out, n);
            count_launch();
            BEAST_CHECK_LAUNCH();
        }
        if (B == 0) return BEAST_OK;
        return encode_impl(p, traj, B, nullptr, nullptr, 0, nullptr, nullptr, min_out, max_out, st);
    }
    bool fast_ran = false;
    const long long n_full = (B / S) * S;
    int rc = encode_impl(p, traj, n_full, nullptr, nullptr, 0, nullptr, nullptr, min_out, max_out, st, ws, accumulate ? 1 : 0,
                         &fast_ran);
    if (rc != BEAST_OK) return rc;
    if (!fast_ran) return BEAST_E_UNSUPPORTED;
    if (n_full < B)
        rc = encode_impl(p, traj + n_full * (long long)p->T * p->D, B - n_full, nullptr, nullptr, 0, nullptr, nullptr, min_out,
                         max_out, st);
    return rc;
}

extern "C" int beast_quantize_f32(const beast_plan_t* plan, const float* params, int64_t B, const float* w_min,
                                  const float* w_max, int64_t offset, int64_t* tokens_out, void* stream) {
    const Plan* p = (const Plan*)plan;
    if (!p || !w_min || !w_max || (B > 0 && (!params || !tokens_out))) return BEAST_E_NULL;
    if (B < 0) return BEAST_E_SHAPE;
    if (B == 0) return BEAST_OK;
    const long long n = (long long)B * p->D * p->nb;
    quantize_kernel<false><<<grid_for(n, 256, p->num_sms), 256, 0, (cudaStream_t)stream>>>(
        params, n, p->D, p->nb, w_min, w_max, (float)(p->V - 1), offset, (long long*)tokens_out, nullptr);
    count_launch();
    BEAST_CHECK_LAUNCH();
    return BEAST_OK;
}

extern "C" int beast_normalize_f32(const beast_plan_t* plan, const float* params, int64_t B, const float* w_min,
                                   const float* w_max, float* out, void* stream) {
    const Plan* p = (const Plan*)plan;
    if (!p || !w_min || !w_max || (B > 0 && (!params || !out))) return BEAST_E_NULL;
    if (B < 0) return BEAST_E_SHAPE;
    if (B == 0) return BEAST_OK;
    const long long n = (long long)B * p->D * p->nb;
    quantize_kernel<true><<<grid_for(n, 256, p->num_sms), 256, 0, (cudaStream_t)stream>>>(
        params, n, p->D, p->nb, w_min, w_max, 0.0f, 0, nullptr, out);
    count_launch();
    BEAST_CHECK_LAUNCH();
    return BEAST_OK;
}
