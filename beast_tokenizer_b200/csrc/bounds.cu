// K2 — weight-bound reductions.
//   beast_minmax_f32        column min/max             (update_weights_bounds, beast_bspline_tokenizer.py:377-378;
//                                                       the batch reduction of update_weights_bounds_per_batch :382-383)
//   beast_bounds_expand_f32 1e-4 hysteresis expansion  (:384-389)
//   beast_colselect_f32     exact per-column order statistics for fit_parameters' np.quantile (:211-214)
// min/max are order independent, so the results are bit-exact however the rows are split over
// threads, CTAs or GPUs (NCCL MIN/MAX all-reduce of the two vectors when the rows are sharded).
#include <cfloat>
#include "common.cuh"

namespace beast {

__global__ void minmax_init_kernel(float* mn, float* mx, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) { mn[i] = __int_as_float(0x7f800000); mx[i] = __int_as_float(0xff800000); }
}

// The columns are cut into chunks of `chunk_groups` column groups (VEC adjacent columns each; at most
// 1024 groups, so a chunk fits one block); the last chunk may be shorter.  Block b works on chunk
// b / row_blocks and on rows (b % row_blocks) * rows_per_block + ..., stepping by row_blocks *
// rows_per_block.  Every thread owns one column group of its chunk for its whole life, and
// consecutive threads read consecutive 16-byte words.  Partials meet in shared memory; one warp per
// column finishes with shuffles.
template <int VEC>
__global__ void __launch_bounds__(1024)
minmax_kernel(const float* __restrict__ x, long long rows, int cols, int chunk_groups, int rows_per_block,
              int row_blocks, float* __restrict__ mn_out, float* __restrict__ mx_out) {
    extern __shared__ float sm[];                 // [2][rows_per_block][chunk_groups * VEC]
    const int chunk = blockIdx.x / row_blocks, rb = blockIdx.x - chunk * row_blocks;
    const int ccols = chunk_groups * VEC;         // columns of a full chunk
    const int c0 = chunk * ccols;
    const int ncols = min(ccols, cols - c0);      // columns of this chunk (VEC divides it)
    const int tid = threadIdx.x;
    const int g = tid % chunk_groups, rl = tid / chunk_groups;
    float mn[VEC], mx[VEC];
#pragma unroll
    for (int v = 0; v < VEC; ++v) { mn[v] = __int_as_float(0x7f800000); mx[v] = __int_as_float(0xff800000); }
    const long long row_stride = (long long)row_blocks * rows_per_block;
    const long long row_end = g * VEC < ncols ? rows : 0;      // a group past the end of a short last chunk reads nothing
    for (long long r = (long long)rb * rows_per_block + rl; r < row_end; r += row_stride) {
        const float* p = x + r * cols + c0 + g * VEC;
        if (VEC == 4) {
            const float4 q = __ldg((const float4*)p);
            mn[0] = fminf(mn[0], q.x); mx[0] = fmaxf(mx[0], q.x);
            mn[1] = fminf(mn[1], q.y); mx[1] = fmaxf(mx[1], q.y);
            mn[2] = fminf(mn[2], q.z); mx[2] = fmaxf(mx[2], q.z);
            mn[3] = fminf(mn[3], q.w); mx[3] = fmaxf(mx[3], q.w);
        } else {
            const float q = __ldg(p);
            mn[0] = fminf(mn[0], q); mx[0] = fmaxf(mx[0], q);
        }
    }
    float* smn = sm;
    float* smx = sm + (size_t)rows_per_block * ccols;
#pragma unroll
    for (int v = 0; v < VEC; ++v) {
        smn[rl * ccols + g * VEC + v] = mn[v];
        smx[rl * ccols + g * VEC + v] = mx[v];
    }
    __syncthreads();
    // full warps only (the block need not be a multiple of 32, and the shuffles name all 32 lanes); a block has
    // at least 257 threads, so 8 full warps or more
    const int warp = tid >> 5, lane = tid & 31, nwarps = blockDim.x >> 5;
    if (warp >= nwarps) return;
    for (int c = warp; c < ncols; c += nwarps) {
        float a = __int_as_float(0x7f800000), b = __int_as_float(0xff800000);
        for (int r = lane; r < rows_per_block; r += 32) {
            a = fminf(a, smn[r * ccols + c]);
            b = fmaxf(b, smx[r * ccols + c]);
        }
        a = warp_min(a);
        b = warp_max(b);
        if (lane == 0) { atomic_min_f32(mn_out + c0 + c, a); atomic_max_f32(mx_out + c0 + c, b); }
    }
}

__global__ void bounds_expand_kernel(const float* __restrict__ bmin, const float* __restrict__ bmax,
                                     float* __restrict__ w_min, float* __restrict__ w_max, int n, float hyst) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    // masks are taken against the bounds as they were on entry (:384-385)
    const float lo = w_min[i], hi = w_max[i];
    if (bmin[i] < __fsub_rn(lo, hyst)) w_min[i] = bmin[i];
    if (bmax[i] > __fadd_rn(hi, hyst)) w_max[i] = bmax[i];
}

// ---------------------------------------------------------------- exact order statistics
__global__ void transpose_kernel(const float* __restrict__ x, long long rows, int cols, float* __restrict__ xt) {
    __shared__ float tile[32][33];
    const long long r0 = (long long)blockIdx.x * 32;
    const int c0 = blockIdx.y * 32;
    for (int j = threadIdx.y; j < 32; j += blockDim.y) {
        const long long r = r0 + j;
        const int c = c0 + threadIdx.x;
        if (r < rows && c < cols) tile[j][threadIdx.x] = x[r * cols + c];
    }
    __syncthreads();
    for (int j = threadIdx.y; j < 32; j += blockDim.y) {
        const int c = c0 + j;
        const long long r = r0 + threadIdx.x;
        if (r < rows && c < cols) xt[(long long)c * rows + r] = tile[threadIdx.x][j];
    }
}

__device__ __forceinline__ unsigned int f32_key(float f) {
    const unsigned int u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float key_f32(unsigned int k) {
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

struct SelectKs { long long k[8]; };

// One CTA per (column, rank): MSD radix select, 4 passes of 8 bits over the transposed column.
// Warp-aggregated shared-memory atomics (lanes that hit the same bin elect one adder).
__global__ void __launch_bounds__(512)
colselect_kernel(const float* __restrict__ xt, long long rows, int cols, SelectKs ks, float* __restrict__ out) {
    __shared__ unsigned int hist[256];
    __shared__ unsigned int s_prefix;
    __shared__ unsigned long long s_k;
    const int col = blockIdx.x;
    const float* colp = xt + (long long)col * rows;
    unsigned int prefix = 0, mask = 0;
    unsigned long long k = (unsigned long long)ks.k[blockIdx.y];
    for (int shift = 24; shift >= 0; shift -= 8) {
        for (int i = threadIdx.x; i < 256; i += blockDim.x) hist[i] = 0;
        __syncthreads();
        const long long rows_pad = (rows + 31) & ~31LL;
        for (long long i = threadIdx.x; i < rows_pad; i += blockDim.x) {
            const bool valid = i < rows;
            const unsigned int key = valid ? f32_key(colp[i]) : 0u;
            const bool hit = valid && ((key & mask) == prefix);
            const unsigned int bin = (key >> shift) & 255u;
            const unsigned int act = __ballot_sync(0xffffffffu, hit);
            if (hit) {
                const unsigned int peers = __match_any_sync(act, bin);
                if ((threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&hist[bin], __popc(peers));
            }
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            unsigned long long cum = 0;
            int d = 0;
            for (; d < 255; ++d) {
                if (cum + hist[d] > k) break;
                cum += hist[d];
            }
            s_k = k - cum;
            s_prefix = prefix | ((unsigned int)d << shift);
        }
        __syncthreads();
        k = s_k;
        prefix = s_prefix;
        mask |= 255u << shift;
        __syncthreads();
    }
    if (threadIdx.x == 0) out[(long long)blockIdx.y * cols + col] = key_f32(prefix);
}

}  // namespace beast

using namespace beast;

extern "C" int beast_minmax_f32(const float* x, int64_t rows, int32_t cols, float* min_out, float* max_out,
                                int32_t accumulate, void* stream) {
    if (!min_out || !max_out || (rows > 0 && !x)) return BEAST_E_NULL;
    if (rows < 0 || cols < 1) return BEAST_E_SHAPE;
    cudaStream_t st = (cudaStream_t)stream;
    if (!accumulate) {
        minmax_init_kernel<<<(cols + 255) / 256, 256, 0, st>>>(min_out, max_out, cols);
        count_launch();
        BEAST_CHECK_LAUNCH();
    }
    if (rows == 0) return BEAST_OK;
    const bool vec4 = (cols % 4 == 0) && (((uintptr_t)x & 15u) == 0);
    const int vec = vec4 ? 4 : 1;
    const int groups = cols / vec;
    // up to 1024 groups: one chunk, the whole row in one block; wider: the fewest chunks of <= 1024 groups, as even
    // as possible, sharing the same 4 * SMs block budget
    const int chunks = (groups + 1023) / 1024;
    const int chunk_groups = (groups + chunks - 1) / chunks;
    int rpb = 512 / chunk_groups;
    if (rpb < 1) rpb = 1;
    const int block = chunk_groups * rpb;
    const size_t smem = 2 * (size_t)rpb * chunk_groups * vec * sizeof(float);     // <= 32 KB
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    long long row_blocks = (rows + rpb - 1) / rpb;
    long long cap = (long long)sms * 4 / chunks;
    if (cap < 1) cap = 1;
    if (row_blocks > cap) row_blocks = cap;
    const long long grid = row_blocks * chunks;
    if (vec4) minmax_kernel<4><<<(unsigned)grid, block, smem, st>>>(x, rows, cols, chunk_groups, rpb, (int)row_blocks,
                                                                   min_out, max_out);
    else minmax_kernel<1><<<(unsigned)grid, block, smem, st>>>(x, rows, cols, chunk_groups, rpb, (int)row_blocks,
                                                              min_out, max_out);
    count_launch();
    BEAST_CHECK_LAUNCH();
    return BEAST_OK;
}

extern "C" int beast_bounds_expand_f32(const float* batch_min, const float* batch_max, float* w_min, float* w_max,
                                       int32_t n, float hyst, void* stream) {
    if (!batch_min || !batch_max || !w_min || !w_max) return BEAST_E_NULL;
    if (n < 0) return BEAST_E_SHAPE;
    if (n == 0) return BEAST_OK;
    bounds_expand_kernel<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(batch_min, batch_max, w_min, w_max, n, hyst);
    count_launch();
    BEAST_CHECK_LAUNCH();
    return BEAST_OK;
}

extern "C" int64_t beast_colselect_scratch_bytes(int64_t rows, int32_t cols, int32_t nk) {
    (void)nk;
    if (rows < 0 || cols < 0) return 0;
    return ((rows * (int64_t)cols * 4 + 255) / 256) * 256;
}

extern "C" int beast_colselect_f32(const float* x, int64_t rows, int32_t cols, const int64_t* ks_h, int32_t nk,
                                   float* out, void* scratch, void* stream) {
    if (!x || !ks_h || !out || !scratch) return BEAST_E_NULL;
    if (rows < 1 || cols < 1 || nk < 1 || nk > 8 || cols > 65535) return BEAST_E_SHAPE;
    SelectKs ks;
    for (int i = 0; i < 8; ++i) {
        ks.k[i] = i < nk ? ks_h[i] : 0;
        if (ks.k[i] < 0 || ks.k[i] >= rows) return BEAST_E_SHAPE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    float* xt = (float*)scratch;
    dim3 tb(32, 8), tg((unsigned)((rows + 31) / 32), (unsigned)((cols + 31) / 32));
    transpose_kernel<<<tg, tb, 0, st>>>(x, rows, cols, xt);
    count_launch();
    BEAST_CHECK_LAUNCH();
    colselect_kernel<<<dim3(cols, nk), 512, 0, st>>>(xt, rows, cols, ks, out);
    count_launch();
    BEAST_CHECK_LAUNCH();
    return BEAST_OK;
}
