// Adjoint of the spline fit (beast_encode_f32's coefficients, then beast_normalize_f32): gradients of encode_continuous's
// outputs back to the trajectories.
//
//   g_w[b, slot, k] = grad_params[b, slot*nb + k]
//                   + (w_min <= w <= w_max ? (grad_norm[b, k*D + slot] * 2) / max(w_max - w_min, 1e-8) : 0)
//   g_y[b, t, dof(slot)] = sum_k P_s[k, t] * g_w[b, slot, k]
//
// w is the unclamped forward coefficient params[b, slot*nb + k] and the bounds are those of its column (torch's rules
// for utils.normalize_tensor: the clamp passes the gradient where the bounds hold inclusively, then * 2 and / scale,
// each one fp32 rounding).  P_s is the fp32 table K1 multiplies with: the plan's joint projector (which already folds
// the boundary conditions in, basis.py: conditioned_projector) or the degree-0 gripper projector.  Each output is one
// fp32 sum over k ascending (fmaf); the terms a kernel skips are exact zeros of the table, which leave a sum of finite
// values unchanged, so both kernels return the same values.  No atomics; every output element is written.
//
// Tiled kernel: a persistent CTA walks tiles of S trajectories.  Phase 1 loads only the coefficients of the plan's
// enc_list (a coefficient whose projector row is empty reaches no sample) from grad_norm / params / grad_params and
// combines them into g_w in shared memory, in token order [k][slot] (the other entries stay 0 for the whole launch).
// Phase 2 writes one output sample per thread in output order: the sum over the column band of P (plan.cu) for four
// trajectories per pass, one table load feeding four sums.  The table is staged in shared memory as [t][k] with an odd
// pitch when its sums are long and it fits in 32 KB; otherwise it is read through L1 from the plan's [k][t] copy.
// Generic kernel: one thread per output element, the whole column with the zero entries skipped.  It is the reference
// the tiled kernel is compared with and the path under beast_debug_disable_fast.
#include "common.cuh"

namespace beast {

constexpr int kFitGradThreads = 512;
// Resident CTAs per SM: __launch_bounds__ lets ptxas use 64 registers, so two 512-thread CTAs fill the register file.  The
// grid still asks for up to four per SM (as the other tiled launchers do): the second half runs as a second wave, restages
// the tables and takes over the remaining tiles.  With grad_norm only at B = 65 536 on a B200 that measured faster than a
// grid of two per SM: cfg2 154 vs 188 us, odd_d5 45 vs 53 us (scripts/fit_grad_time.py).  Why was not checked.
constexpr int kFitGradCtasPerSm = 2;
constexpr int kFitGradGridPerSm = 4;

struct FitGradArgs {
    const float* grad_norm;        // [B, nb*D] '(t d)' (nullable)
    const float* grad_params;      // [B, D*nb] '(d t)' (nullable)
    const float* params;           // [B, D*nb] '(d t)' unclamped (with grad_norm)
    const float* w_min;
    const float* w_max;
    long long B;
    int T, D, nb, n_joint;
    const int* slot_to_dof;
    const float* Pj;               // [nb][T]
    const float* Pg;               // [nb][T] or nullptr
    const int* col_bands;          // [joint | gripper][T][lo, hi) over k
    const int* list;               // enc_list: k | slot << 16 | gripper << 31, token order
    int n_enc;
    float* grad_traj;              // [B, T, D]
    int S, G1, G2;                 // trajectories per tile; trajectory groups per list entry / per output sample
    int p_smem;                    // projector staged in shared memory as [joint | gripper][t][nb | 1]
};

__global__ void __launch_bounds__(kFitGradThreads, kFitGradCtasPerSm)
fit_grad_tiled_kernel(const __grid_constant__ FitGradArgs a) {
    extern __shared__ __align__(16) float smem_f[];
    const int T = a.T, D = a.D, nb = a.nb, S = a.S, n_enc = a.n_enc;
    const int row_in = D * nb, row_out = T * D;
    const bool has_n = a.grad_norm != nullptr, has_p = a.grad_params != nullptr;
    float* g_s = smem_f;                                        // [S][nb][D] g_w, token order (slot minor)
    float* lohi = g_s + (((size_t)S * row_in + 3) & ~(size_t)3);   // [n_enc][2] bounds of the listed coefficients
    int* lst = (int*)(lohi + (size_t)2 * n_enc);                // [n_enc]
    int* s_band = lst + n_enc;                                  // [2][2*T] column bands
    int* s_slot = s_band + 4 * T;                               // [D] dof -> slot
    float* P_s = (float*)(s_slot + D);                          // [2][T][pitch]
    const int pitch = nb | 1;
    const int tid = threadIdx.x;
    for (int i = tid; i < n_enc; i += kFitGradThreads) {
        const int e = a.list[i];
        lst[i] = e;
        if (has_n) {
            const int c = ((e >> 16) & 0x7fff) * nb + (e & 0xffff);
            lohi[2 * i] = a.w_min[c];
            lohi[2 * i + 1] = a.w_max[c];
        }
    }
    for (int i = tid; i < D; i += kFitGradThreads) s_slot[a.slot_to_dof[i]] = i;
    for (int i = tid; i < 4 * T; i += kFitGradThreads) s_band[i] = a.col_bands[i];
    if (a.p_smem)
        for (int i = tid; i < T * nb; i += kFitGradThreads) {
            const int k = i / T, t = i - k * T;
            P_s[t * pitch + k] = a.Pj[i];
            if (a.Pg) P_s[(T + t) * pitch + k] = a.Pg[i];
        }
    for (int i = tid; i < S * row_in; i += kFitGradThreads) g_s[i] = 0.0f;   // entries outside the list: exactly 0
    const long long n_tiles = (a.B + S - 1) / S;
    const int items1 = n_enc * a.G1, items2 = row_out * a.G2;
    const int nd = n_enc > 0 ? n_enc : 1;
    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const long long b0 = tile * S;
        const int ns = (int)((a.B - b0) < S ? (a.B - b0) : S);
        __syncthreads();                                        // tables ready / previous tile's g_w consumed
        const float* gn_tile = has_n ? a.grad_norm + b0 * row_in : nullptr;
        const float* par_tile = has_n ? a.params + b0 * row_in : nullptr;
        const float* gp_tile = has_p ? a.grad_params + b0 * row_in : nullptr;
        float* out_tile = a.grad_traj + b0 * row_out;
        // phase 1: the listed coefficients -> g_w; work item j -> (trajectory group, entry) tracked by increments
        const int g1_step = kFitGradThreads / nd, i1_step = kFitGradThreads - g1_step * n_enc;
        int g = tid / nd, i = tid - g * n_enc;
        for (int j = tid; j < items1; j += kFitGradThreads, g += g1_step, i += i1_step) {
            if (i >= n_enc) { i -= n_enc; ++g; }
            const int e = lst[i];
            const int k = e & 0xffff, slot = (e >> 16) & 0x7fff;
            const int r = k * D + slot, c = slot * nb + k;
            float lo = 0.0f, hi = 0.0f;
            if (has_n) { lo = lohi[2 * i]; hi = lohi[2 * i + 1]; }
            const int stride = a.G1 * row_in;
            // four trajectories per pass, every load of the pass issued before the first shared-memory store
            for (int tr = g, off = g * row_in; tr < ns; tr += 4 * a.G1, off += 4 * stride) {
                const int o[4] = {off, off + stride, off + 2 * stride, off + 3 * stride};
                const bool h[4] = {true, tr + a.G1 < ns, tr + 2 * a.G1 < ns, tr + 3 * a.G1 < ns};
                float gn[4], w[4], gp[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    gn[u] = 0.0f; w[u] = 0.0f; gp[u] = 0.0f;
                    if (!h[u]) continue;
                    if (has_n) { gn[u] = __ldcs(gn_tile + o[u] + r); w[u] = __ldcs(par_tile + o[u] + c); }
                    if (has_p) gp[u] = __ldcs(gp_tile + o[u] + c);
                }
#pragma unroll
                for (int u = 0; u < 4; ++u)
                    if (h[u]) g_s[o[u] + r] = fit_grad_weight(has_n, gn[u], w[u], lo, hi, has_p, gp[u]);
            }
        }
        __syncthreads();
        // phase 2: one output sample per thread, output order
        const int g2_step = kFitGradThreads / row_out, q_step = kFitGradThreads - g2_step * row_out;
        int g2 = tid / row_out, q = tid - g2 * row_out;
        for (int j = tid; j < items2; j += kFitGradThreads, g2 += g2_step, q += q_step) {
            if (q >= row_out) { q -= row_out; ++g2; }
            const int t = q / D, dof = q - t * D;
            const int slot = s_slot[dof];
            const bool grip = slot >= a.n_joint;
            // generic pointer + stride over k: the shared-memory copy [t][k] or the plan's global table [k][t]
            const float* col = a.p_smem ? P_s + (size_t)((grip ? T : 0) + t) * pitch : (grip ? a.Pg : a.Pj) + t;
            const int pst = a.p_smem ? 1 : T;
            const int k0 = s_band[(grip ? 2 * T : 0) + 2 * t], k1 = s_band[(grip ? 2 * T : 0) + 2 * t + 1];
            for (int tr = g2; tr < ns; tr += 4 * a.G2) {
                const int tr1 = tr + a.G2, tr2 = tr + 2 * a.G2, tr3 = tr + 3 * a.G2, last = ns - 1;
                const float* c0 = g_s + tr * row_in + slot;
                const float* c1 = g_s + (tr1 < last ? tr1 : last) * row_in + slot;
                const float* c2 = g_s + (tr2 < last ? tr2 : last) * row_in + slot;
                const float* c3 = g_s + (tr3 < last ? tr3 : last) * row_in + slot;
                float a0 = 0.0f, a1 = 0.0f, a2 = 0.0f, a3 = 0.0f;
                for (int k = k0; k < k1; ++k) {
                    const float pv = col[k * pst];
                    const int o = k * D;
                    a0 = fmaf(pv, c0[o], a0); a1 = fmaf(pv, c1[o], a1); a2 = fmaf(pv, c2[o], a2); a3 = fmaf(pv, c3[o], a3);
                }
                __stcs(out_tile + tr * row_out + q, a0);
                if (tr1 < ns) __stcs(out_tile + tr1 * row_out + q, a1);
                if (tr2 < ns) __stcs(out_tile + tr2 * row_out + q, a2);
                if (tr3 < ns) __stcs(out_tile + tr3 * row_out + q, a3);
            }
        }
    }
}

__global__ void fit_grad_generic_kernel(const __grid_constant__ FitGradArgs a) {
    const int T = a.T, D = a.D, nb = a.nb;
    const long long row_in = (long long)D * nb, row_out = (long long)T * D, n = a.B * row_out;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < n;
         idx += (long long)gridDim.x * blockDim.x) {
        const long long b = idx / row_out;
        const int q = (int)(idx - b * row_out);
        const int t = q / D, dof = q - t * D;
        int slot = 0;
        for (int s = 0; s < D; ++s) if (a.slot_to_dof[s] == dof) slot = s;
        const float* P = slot < a.n_joint ? a.Pj : a.Pg;
        float acc = 0.0f;
        for (int k = 0; k < nb; ++k) {
            const float pv = P[(size_t)k * T + t];
            if (pv == 0.0f) continue;
            acc = fmaf(pv, fit_grad_coeff(a.grad_norm, a.grad_params, a.params, a.w_min, a.w_max, b * row_in, D, nb,
                                          slot, k), acc);
        }
        a.grad_traj[idx] = acc;
    }
}

static inline int fit_groups_for(int entries, int S) {
    int g = entries > 0 ? (kFitGradThreads + entries - 1) / entries : 1;
    if (g > S) g = S;
    return g < 1 ? 1 : g;
}

// BEAST_E_UNSUPPORTED when one trajectory's g_w and the tables do not fit in shared memory (the caller then takes the
// generic kernel).
static int launch_fit_grad_tiled(const Plan* p, FitGradArgs a, cudaStream_t st) {
    const int T = p->T, D = p->D, nb = p->nb;
    if (!p->bands_d || !p->enc_list_d || nb > 0xffff || D > 0x7fff) return BEAST_E_UNSUPPORTED;
    const size_t per_traj = (size_t)D * nb * sizeof(float);
    const size_t p_bytes = (size_t)2 * T * (nb | 1) * sizeof(float);
    // sums of one or two terms read every table entry once per pass: nothing to stage for (as in launch_decode_tiled)
    const bool p_smem = p_bytes <= 32 * 1024 && p->fit_band_max > 2;
    const size_t extra = ((size_t)3 * p->n_enc + (size_t)4 * T + D) * sizeof(float) + 16 + (p_smem ? p_bytes : 0);
    size_t budget = 108 * 1024;                                 // two CTAs per SM
    if (per_traj + extra > budget) budget = (size_t)p->max_smem_optin;
    if (per_traj + extra > budget) return BEAST_E_UNSUPPORTED;
    int S = (int)((budget - extra) / per_traj);
    if (S > 64) S = 64;
    const size_t smem = (size_t)S * per_traj + extra;
    static size_t granted[kMaxDevices] = {};
    if (int rc = opt_in_smem(fit_grad_tiled_kernel, smem, granted)) return rc;
    a.col_bands = p->bands_d + 4 * nb + 4 * T;
    a.list = p->enc_list_d; a.n_enc = p->n_enc;
    a.S = S; a.G1 = fit_groups_for(p->n_enc, S); a.G2 = fit_groups_for(T * D, S);
    a.p_smem = p_smem ? 1 : 0;
    const long long n_tiles = (a.B + S - 1) / S;
    long long per_sm = (long long)(220 * 1024) / (long long)(smem + 1024);
    if (per_sm > kFitGradGridPerSm) per_sm = kFitGradGridPerSm;
    if (per_sm < 1) per_sm = 1;
    const long long grid = n_tiles < (long long)p->num_sms * per_sm ? n_tiles : (long long)p->num_sms * per_sm;
    fit_grad_tiled_kernel<<<(unsigned)grid, kFitGradThreads, smem, st>>>(a);
    count_launch();
    BEAST_CHECK_LAUNCH();
    return BEAST_OK;
}

static int launch_fit_grad_generic(const Plan* p, const FitGradArgs& a, cudaStream_t st) {
    const long long n = a.B * (long long)p->T * p->D;
    long long grid = (n + 255) / 256;
    const long long cap = (long long)p->num_sms * 16;
    if (grid > cap) grid = cap;
    fit_grad_generic_kernel<<<(unsigned)grid, 256, 0, st>>>(a);
    count_launch();
    BEAST_CHECK_LAUNCH();
    return BEAST_OK;
}

}  // namespace beast

using namespace beast;

extern "C" int beast_fit_backward_f32(const beast_plan_t* plan, int64_t B, const float* grad_norm,
                                      const float* grad_params, const float* params, const float* w_min,
                                      const float* w_max, float* grad_traj, void* stream) {
    const Plan* p = (const Plan*)plan;
    if (!p) return BEAST_E_NULL;
    if (!grad_norm && !grad_params) return BEAST_E_NULL;
    if (!grad_traj) return BEAST_E_NULL;
    if (grad_norm && (!params || !w_min || !w_max)) return BEAST_E_NULL;
    if (B < 0) return BEAST_E_SHAPE;
    for (const void* q : {(const void*)grad_norm, (const void*)grad_params, (const void*)params, (const void*)w_min,
                          (const void*)w_max, (const void*)grad_traj})
        if ((uintptr_t)q & 3u) return BEAST_E_ALIGN;
    if (B == 0) return BEAST_OK;
    FitGradArgs a = {};
    a.grad_norm = grad_norm; a.grad_params = grad_params;
    a.params = grad_norm ? params : nullptr;
    a.w_min = grad_norm ? w_min : nullptr; a.w_max = grad_norm ? w_max : nullptr;
    a.B = B; a.T = p->T; a.D = p->D; a.nb = p->nb; a.n_joint = p->n_joint;
    a.slot_to_dof = p->slot_to_dof_d; a.Pj = p->proj_joint_d; a.Pg = p->proj_grip_d;
    a.grad_traj = grad_traj;
    cudaStream_t st = (cudaStream_t)stream;
    if (!fast_paths_disabled()) {
        const int rc = launch_fit_grad_tiled(p, a, st);
        if (rc != BEAST_E_UNSUPPORTED) return rc;
    }
    return launch_fit_grad_generic(p, a, st);
}
