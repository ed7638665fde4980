// Shared device helpers for libbeast_b200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <cstdlib>
#include <utility>
#include "beast_b200.h"

#ifndef __CUDA_ARCH__
#define BEAST_HOST 1
#endif

#define BEAST_MAX_SLOTS BEAST_MAX_DOF

namespace beast {

// ---------------------------------------------------------------- plan
struct Plan {
    int T, D, nb, n_joint, degree_p, V;
    int ico, eco, nc;      // pinned leading / trailing joint control points; nc = nb + ico + eco
    float tau;
    int slot_to_dof[BEAST_MAX_SLOTS];
    // host copies
    float* proj_joint_h;   // [nb*T]  [k][t]
    float* proj_grip_h;    // [nb*T] or nullptr
    float* phi_joint_h;    // [T*nc]  [t][c]
    float* phi_grip_h;
    // device copies (one allocation)
    float* dev_block;
    float* proj_joint_d;
    float* proj_grip_d;
    float* phi_joint_d;
    float* phi_grip_d;
    float* knots_joint_d;  // [nc+degree_p+1]
    float* knots_grip_d;   // [nb+1]
    int* slot_to_dof_d;
    // Band tables of the tiled kernels (csrc/spline_tiled.cu), pairs [lo, hi): the non-zero range of every projector
    // row (encode: samples t of basis k) and of every basis row (decode: basis k of sample t); the terms outside are
    // exact zeros, skipping them leaves the fp32 sums unchanged.  Layout: enc_joint[2*nb], enc_grip[2*nb],
    // dec_joint[2*T], dec_grip[2*T], then the non-zero range over k of every projector column (the fit's adjoint,
    // csrc/spline_fit_grad.cu): fit_joint[2*T], fit_grip[2*T].
    int* bands_d;
    // Work lists of the tiled kernels, token order (r = k*D + slot ascending), entries k | slot << 16 | gripper << 31:
    // enc_list = token positions whose projector row is not empty (every other coefficient is exactly 0 for every
    // trajectory and its token a per-column constant); dec_list = token positions whose coefficient some basis row
    // actually reads (with more basis functions than samples most coefficients never reach a trajectory sample, so
    // their tokens need not even be loaded).  One allocation: enc_list_d[n_enc] followed by dec_list_d[n_dec].
    int* enc_list_d;
    int* dec_list_d;
    int n_enc, n_dec;
    int enc_band_max, dec_band_max;   // longest projector-row / basis-row band (terms per sum)
    int fit_band_max;                 // longest projector-column band
    int num_sms;
    int max_smem_optin;
};

// Tiled kernels for any geometry on the tokenizer's own times (csrc/spline_tiled.cu); BEAST_E_UNSUPPORTED when a
// trajectory's working set does not fit shared memory (the caller then takes the one-thread-per-column kernels).
int launch_encode_tiled(const Plan* p, const float* traj, long long B, const float* w_min, const float* w_max,
                        long long offset, float* params_out, long long* tokens_out, float* bmin, float* bmax,
                        cudaStream_t st);
int launch_decode_tiled(const Plan* p, const long long* tokens, const float* params, long long B, const float* w_min,
                        const float* w_max, long long offset, const float* init_p, float* out, cudaStream_t st);

// Generic kernels that evaluate the basis in-kernel (spline_decode.cu, spline_deriv.cu) keep one level of the
// recursion per thread: num_ctrlp + degree_p <= 319.
constexpr int kMaxEvalKnots = 320;

extern long long g_launch_count;
inline void count_launch(int n = 1) { g_launch_count += n; }

// ---------------------------------------------------------------- launch-boundary overlap of K1 / K3 (csrc/plan.cu)
// A bulk-copy K1 / K3 launch may start streaming while the launch before it drains (it skips griddepcontrol.wait)
// only when that launch provably is the previous bulk-copy K1 / K3 launch of this library and the two touch disjoint
// memory.  Adjacency can only be proven inside a stream capture: the dependency set the next captured node gets must
// be exactly the node recorded right after that launch.  Eager launches never overlap (the library cannot see
// foreign work enqueued between two of its calls).  Every CTA issues griddepcontrol.launch_dependents only after its
// own griddepcontrol.wait has returned, so a successor starts only once its predecessor's predecessor has completed:
// checking against the immediate predecessor is enough.
struct MemRange {
    uintptr_t lo, hi;      // bytes [lo, hi)
    int write;             // 0 = read, 1 = written (or read and written)
};
struct LaunchRanges {
    static constexpr int kMax = 8;
    MemRange r[kMax];
    int n = 0;
    void add(const void* p, size_t bytes, bool write) {
        if (p && bytes && n < kMax) r[n++] = MemRange{(uintptr_t)p, (uintptr_t)p + bytes, write ? 1 : 0};
    }
};
// read-after-write, write-after-read or write-after-write between two launches; touching and empty ranges never conflict
bool ranges_conflict(const LaunchRanges& prev, const LaunchRanges& next);
// Before a bulk-copy K1 / K3 launch on `st`: true when it may overlap its predecessor (launch it with the programmatic
// stream serialization attribute and wait_first = 0).
bool overlap_begin(cudaStream_t st, const LaunchRanges& mine);
// Right after it: records the launch's capture node and ranges for the next launch on `st` (or forgets the stream's
// record when the launch was eager or failed) and counts overlapped launches.
void overlap_end(cudaStream_t st, const LaunchRanges& mine, bool overlapped, cudaError_t launch_error);
// 1 = every bulk-copy K1 / K3 launch waits for its predecessor (beast_debug_force_wait): the A/B measurement and the
// overlap tests compare against it
extern int g_force_wait;

template <typename... P, typename... A>
static inline cudaError_t launch_maybe_overlapped(void (*kernel)(P...), int grid, int block, size_t smem,
                                                  cudaStream_t st, bool overlap, A&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(block);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = overlap ? 1 : 0;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, std::forward<A>(args)...);
}

// Programmatic dependent launch: pdl_wait() blocks until the previous grid has completed and its writes are visible
// (a no-op when the launch did not allow programmatic serialization); pdl_launch() lets the next grid start being
// scheduled once every CTA of this one has issued it or exited.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
// 1 = take the one-thread-per-column reference kernels only (beast_debug_disable_fast, or BEAST_B200_DISABLE_FAST=1
// read once at the first call): the parity tests compare them with the tiled / bulk-copy kernels bit for bit.
extern int g_disable_fast;
inline bool fast_paths_disabled() {
    if (g_disable_fast < 0) { const char* e = getenv("BEAST_B200_DISABLE_FAST"); g_disable_fast = (e && e[0] == '1') ? 1 : 0; }
    return g_disable_fast == 1;
}

// ---------------------------------------------------------------- quantiser (bit-exact contract)
// beast/beast_bspline_tokenizer.py:419 (clamp) + beast/utils.py:12-16: every step is one
// separately rounded IEEE fp32 operation; the _rn intrinsics are never contracted into FMAs.
__device__ __forceinline__ float clampf(float x, float lo, float hi) {
    // torch.clamp(x, lo, hi) == min(max(x, lo), hi)
    return fminf(fmaxf(x, lo), hi);
}

__device__ __forceinline__ float quant_scale(float w_min, float w_max) {
    return fmaxf(__fsub_rn(w_max, w_min), 1e-8f);               // utils.py:12
}

// Correctly rounded a / b for a divisor that is reused many times: y = RN(1/b) is computed once
// (IEEE reciprocal), then two FMA residual corrections.  After the first correction q is a faithful
// quotient, so the second residual is exact and Markstein's theorem gives q2 == RN(a / b) — the
// same bits as the reference's true division, without div.rn's data-dependent slow path (taken
// for a == 0, i.e. for every clamped coefficient).  Bit-exact for 2^-27 <= b <= 2^100 (callers check
// div_fast_ok(b) once per divisor and fall back to __fdiv_rn) whenever a / b >= 2^-60: then every
// residual is a normal number.  For a smaller (possibly subnormal) quotient the last bit may
// differ, but the token is bin 0 either way ((V-1) * 2^-60 rounds to 0).  Verified against __fdiv_rn on ~10^10 operand
// pairs by beast_selftest_div (tests/test_gpu_spline.py).
__device__ __forceinline__ bool div_fast_ok(float b) {
    return b >= 7.4505805969238281e-09f && b <= 1.2676506002282294e+30f;   // 2^-27 .. 2^100
}
__device__ __forceinline__ float div_invariant(float a, float b, float y) {
    float q = __fmul_rn(a, y);
    float r = __fmaf_rn(-b, q, a);
    q = __fmaf_rn(r, y, q);
    r = __fmaf_rn(-b, q, a);
    return __fmaf_rn(r, y, q);
}

// Per-column constants of the quantiser, loaded once per thread.
struct QuantCol {
    float lo, hi, scale, rcp;      // rcp == 0 -> use __fdiv_rn (divisor outside the safe range)
    __device__ __forceinline__ void init(float w_min, float w_max) {
        lo = w_min; hi = w_max;
        scale = quant_scale(w_min, w_max);
        rcp = div_fast_ok(scale) ? __frcp_rn(scale) : 0.0f;
    }
};

__device__ __forceinline__ long long quantize_col(float w, const QuantCol& c, float vm1) {
    const float p = clampf(w, c.lo, c.hi);                      // tokenizer.py:419
    const float num = __fsub_rn(p, c.lo);
    // utils.py:13 (true division); |num| <= 2^101 here unless the inputs are non-finite
    float n = (c.rcp != 0.0f && fabsf(num) <= 2.5353012004564588e+30f) ? div_invariant(num, c.scale, c.rcp)
                                                                         : __fdiv_rn(num, c.scale);
    n = clampf(n, 0.0f, 1.0f);                                  // utils.py:14
    return __float2ll_rn(__fmul_rn(n, vm1));                    // utils.py:16: round half to even, to int64
}

__device__ __forceinline__ long long quantize_one(float w, float w_min, float w_max, float scale, float vm1) {
    float p = clampf(w, w_min, w_max);                          // tokenizer.py:419
    float n = __fdiv_rn(__fsub_rn(p, w_min), scale);            // utils.py:13 (true division)
    n = clampf(n, 0.0f, 1.0f);                                  // utils.py:14
    return (long long)rintf(__fmul_rn(n, vm1));                 // utils.py:16 (half-to-even)
}

// beast/utils.py:23-25: float(tok)/(V-1), mul, add (two roundings), clamp.
__device__ __forceinline__ float dequantize_one(long long tok, float w_min, float w_max, float vm1) {
    float n = __fdiv_rn(__ll2float_rn(tok), vm1);
    float c = __fadd_rn(__fmul_rn(n, __fsub_rn(w_max, w_min)), w_min);
    return clampf(c, w_min, w_max);
}
// Same with the invariant divisor V-1 (rcp_vm1 = RN(1 / (V-1)); V-1 <= 2^31 is always in range).
__device__ __forceinline__ float dequantize_fast(long long tok, float w_min, float w_max, float vm1, float rcp_vm1) {
    const float n = div_invariant(__ll2float_rn(tok), vm1, rcp_vm1);
    const float c = __fadd_rn(__fmul_rn(n, __fsub_rn(w_max, w_min)), w_min);
    return clampf(c, w_min, w_max);
}

// ---------------------------------------------------------------- packed fp32 FMA (Blackwell FFMA2)
// fma.rn.f32x2: two IEEE fp32 FMAs per instruction (SASS FFMA2, which takes a uniform-register pair
// and a broadcast scalar directly).  Bit-identical to two fmaf calls; halves the issue slots of the
// K = 50 / N = 10 contractions in K1 / K3.
__device__ __forceinline__ unsigned long long pack_f32x2(float lo, float hi) {
    return ((unsigned long long)__float_as_uint(hi) << 32) | (unsigned long long)__float_as_uint(lo);
}
__device__ __forceinline__ float lo_f32(unsigned long long v) { return __uint_as_float((unsigned int)v); }
__device__ __forceinline__ float hi_f32(unsigned long long v) { return __uint_as_float((unsigned int)(v >> 32)); }
// acc.{lo,hi} = fma(a.{lo,hi}, b, acc.{lo,hi})
__device__ __forceinline__ void ffma2_bcast(unsigned long long& acc, float a_lo, float a_hi, float b) {
    const unsigned long long a = pack_f32x2(a_lo, a_hi);
    const unsigned long long bb = pack_f32x2(b, b);
    asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(acc) : "l"(a), "l"(bb));
}

// ---------------------------------------------------------------- mbarrier / bulk-copy PTX
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// Bounded wait: a protocol bug traps (kernel fails with an error) instead of hanging the GPU.  The bound is wall
// time on the global timer (60 s): a healthy launch that is merely descheduled (time-slicing with another process,
// MPS oversubscription, a debugger) never comes near it, whereas SM-clock ticks keep running while descheduled.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    if (mbar_try_wait(bar, parity)) return;
    unsigned long long t0 = 0;
    unsigned int spins = 0;
    while (!mbar_try_wait(bar, parity)) {
        if ((++spins & 0xfffu) == 0) {
            unsigned long long now;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
            if (t0 == 0) t0 = now;
            else if (now - t0 > 60000000000ull) __trap();
        }
    }
}
// global -> shared, completion counted in bytes on an mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
// shared -> global, tracked by the issuing thread's bulk async-group
__device__ __forceinline__ void bulk_s2g(void* dst_gmem, const void* src_smem, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem),
                 "r"(smem_u32(src_smem)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() {
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void bulk_wait_all() {
    asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}
// make generic-proxy shared-memory writes visible to the async proxy (before a bulk store)
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// float atomics through the order-preserving integer views (outputs hold +inf / -inf initially).
__device__ __forceinline__ void atomic_min_f32(float* addr, float v) {
    v = __fadd_rn(v, 0.0f);                                  // -0.0 -> +0.0 (its int view is INT_MIN)
    if (v >= 0.0f) atomicMin((int*)addr, __float_as_int(v));
    else atomicMax((unsigned int*)addr, __float_as_uint(v));
}
__device__ __forceinline__ void atomic_max_f32(float* addr, float v) {
    v = __fadd_rn(v, 0.0f);
    if (v >= 0.0f) atomicMax((int*)addr, __float_as_int(v));
    else atomicMin((unsigned int*)addr, __float_as_uint(v));
}

__device__ __forceinline__ float warp_min(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// Opt-in to more than 48 KB of dynamic shared memory. The attribute is per (kernel, device), so the
// granted size is remembered per device: a process that drives several GPUs sets it on each.
constexpr int kMaxDevices = 64;
template <typename F>
static inline int opt_in_smem(F kernel, size_t smem, size_t (&granted)[kMaxDevices]) {
    if (smem <= 48 * 1024) return BEAST_OK;
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return (int)e;
    if (dev < 0 || dev >= kMaxDevices) return BEAST_E_UNSUPPORTED;
    if (smem > granted[dev]) {
        e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return (int)e;
        granted[dev] = smem;
    }
    return BEAST_OK;
}


}  // namespace beast

#define BEAST_CHECK_LAUNCH()                     \
    do {                                         \
        cudaError_t e__ = cudaGetLastError();    \
        if (e__ != cudaSuccess) return (int)e__; \
    } while (0)
