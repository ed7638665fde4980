// K4 / K5 — byte-level BPE over discretised BEAST bins on the GPU.
//
// The reference trains and applies HF `tokenizers`' ByteLevelBPETokenizer on chr(bin - min_token)
// strings (beast/beast_bpe_trainer.py:61-98, beast/beast_bspline_bpe_tokenizer.py:175-247).  These
// kernels implement the same algorithm (SURVEY.md Appendix A) on integer symbols:
//
//   symbolise   bins -> GPT-2 pre-tokenisation -> UTF-8 bytes -> symbol ids, word-start flag in bit 15
//   count       adjacent-pair histogram, dense V x V int32 (L2-resident: 16 MB at V = 2048), counted in
//               block-private shared-memory histograms over the distinct byte-level symbols
//   iterate     fold the previous merge's 4 x V delta block, arg-max: max count, ties -> smallest (a, b)
//   pick        BpeTrainer's stop rules, next id, merge log (all on the device: the loop never syncs)
//   scan        which sequences hold (a, b): per-sequence 2048-bit pair signatures (Bloom filter, word-major)
//               filter the corpus down to the survivors, which are walked in lock step; hits -> work list
//   rewrite     left to right, non-overlapping, in-place compaction — one warp per sequence (short lists)
//               or one thread per sequence (long lists); the count changes are confined to column a, row b,
//               column c, row c of the histogram and are collected in the 4 x V delta block (summed over
//               GPUs with one small all-reduce when sharded)
//   encode      one warp per sequence: token starts by a local rule, per word repeatedly merge the
//               lowest-rank pair, leftmost first
//   decode      one warp per sequence: ids -> token bytes -> UTF-8 -> codepoints + min_token
//
// Corpus layout: CHUNK-MAJOR — 8 consecutive symbols (16 bytes) of one sequence form a chunk and chunk c
// of all sequences is contiguous: sym[((p >> 3) * n_stride + seq) * 8 + (p & 7)] (uint16).  A warp that
// walks 32 sequences reads / writes chunk c of all of them as 512 contiguous bytes, one 128-bit access
// per lane.
#include <cstring>
#include <cooperative_groups.h>
#include "bpe_common.cuh"

namespace beast {

// Pair signatures: kSigBits bits per sequence, bit hash(a, b) set for every in-word adjacent pair the
// sequence holds or ever held (bits are only added, so the set is a superset).  Stored word-major
// (sig[word * n_stride + seq]) so that the scan for one pair reads a single 4-byte column.
constexpr int kScanTile = 2048;          // sequences filtered per block and step by the signature scan
constexpr int kDirectDeltaWork = 1 << 17; // rewrite: work lists up to this size are rewritten one warp per sequence
constexpr int kGlobalDeltaWork = 1 << 14; // ... and up to this size their count changes go straight to the global delta block // rewrite: work lists up to this size update the global delta directly
constexpr int kSigWords = 64;
constexpr int kSigBits = kSigWords * 32;
// Two independent hash positions per pair (a Bloom filter with k = 2): a sequence passes the scan's
// filter only if both bits are set, which squares the false-positive rate for one more 4-byte column.
__device__ __forceinline__ unsigned int sig_hash(unsigned int a, unsigned int b) {
    return ((a * 0x9E3779B1u + b * 0x85EBCA77u) >> 15) & (unsigned int)(kSigBits - 1);
}
__device__ __forceinline__ unsigned int sig_hash2(unsigned int a, unsigned int b) {
    return ((a * 0xC2B2AE3Du + b * 0x27D4EB2Fu + 0x165667B1u) >> 13) & (unsigned int)(kSigBits - 1);
}

// Device-side control block of the sync-free training loop (bpe_train_step).
struct BpeCtl {
    int a, b, c, count;     // the merge selected for this iteration
    int n_tokens;           // vocabulary size so far (= next new id)
    int n_merges;           // merges logged
    int done;               // sticky: no pair reached min_frequency, or the vocabulary is full
    int has_delta;          // the delta block of merge (a, b, c) still has to be folded into the histogram
    int err;                // sticky: 1 = a peer did not publish its epoch in time (sharded runs)
    int pad[7];
};

// Sharded training: the ranks' delta blocks and flag arrays as seen from this GPU (bpe_peers_t of the C ABI).
struct BpePeersDev {
    int world, rank, epoch_base;
    int* delta[BPE_MAX_PEERS];
    int* flags[BPE_MAX_PEERS];
};
__device__ __forceinline__ void st_release_sys(int* p, int v) {
    asm volatile("st.release.sys.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ int ld_acquire_sys(const int* p) {
    int v;
    asm volatile("ld.acquire.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ int ld_relaxed_sys(const int* p) {
    int v;
    asm volatile("ld.relaxed.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned long long global_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
constexpr unsigned long long kPeerWaitNs = 5000000000ull;     // a peer that stays silent for 5 s is reported, not waited for
// Programmatic dependent launch (pdl_wait / pdl_launch, common.cuh): the three kernels of a merge iteration are
// launched with cudaLaunchAttributeProgrammaticStreamSerialization, so the blocks of the next kernel are scheduled
// while the previous one drains.


// GPT-2 pre-tokeniser character classes for codepoints 0..255 (SURVEY.md Appendix A.2)
enum { CLS_O = 0, CLS_L = 1, CLS_N = 2, CLS_S = 3 };
__device__ __forceinline__ int cp_class_latin1(int c) {
    if (c == 32 || (c >= 9 && c <= 13) || c == 133 || c == 160) return CLS_S;
    if ((c >= 48 && c <= 57) || c == 178 || c == 179 || c == 185 || (c >= 188 && c <= 190)) return CLS_N;
    if ((c >= 65 && c <= 90) || (c >= 97 && c <= 122) || c == 170 || c == 181 || c == 186 ||
        (c >= 192 && c <= 214) || (c >= 216 && c <= 246) || c >= 248)
        return CLS_L;
    return CLS_O;
}

// Codepoints >= 256 (tokenizers with more than 256 bins) look their class up in a table built on the
// host from the Unicode general categories (L*, N*, White_Space — Oniguruma's \p{L}, \p{N}, \s).
__device__ __forceinline__ int cp_class(int c, const uint8_t* __restrict__ cls_tab) {
    return c < 256 ? cp_class_latin1(c) : (int)__ldg(cls_tab + c);
}

// UTF-8 bytes of codepoint c (< 0x10000, never a surrogate here).
__device__ __forceinline__ int utf8_encode(int c, int (&b)[3]) {
    if (c < 0x80) { b[0] = c; return 1; }
    if (c < 0x800) { b[0] = 0xC0 | (c >> 6); b[1] = 0x80 | (c & 0x3F); return 2; }
    b[0] = 0xE0 | (c >> 12); b[1] = 0x80 | ((c >> 6) & 0x3F); b[2] = 0x80 | (c & 0x3F);
    return 3;
}

// Length of the pre-token starting at codepoint i of cp[0..n) (shared memory).
template <typename CP>
__device__ __forceinline__ int pretoken_len(const CP* cp, int i, int n, const uint8_t* __restrict__ cls_tab) {
    const int c = cp[i];
    if (c == 39 && i + 1 < n) {                              // 's|'t|'re|'ve|'m|'ll|'d
        const int d = cp[i + 1];
        if (d == 's' || d == 't' || d == 'm' || d == 'd') return 2;
        if (i + 2 < n) {
            const int e = cp[i + 2];
            if ((d == 'r' && e == 'e') || (d == 'v' && e == 'e') || (d == 'l' && e == 'l')) return 3;
        }
    }
    int start = i;
    if (c == 32 && i + 1 < n && cp_class(cp[i + 1], cls_tab) != CLS_S) start = i + 1;     // " ?" prefix
    const int k = cp_class(cp[start], cls_tab);
    if (k != CLS_S) {                                        // one run of L, N or O
        int j = start + 1;
        while (j < n && cp_class(cp[j], cls_tab) == k) ++j;
        return j - i;
    }
    int j = i + 1;                                           // whitespace run [i, j)
    while (j < n && cp_class(cp[j], cls_tab) == CLS_S) ++j;
    if (j == n) return j - i;                                // \s+(?!\S) at end of text
    if (j - i >= 2) return j - 1 - i;                        // \s+(?!\S): leave the last blank
    return 1;                                                // \s+
}

// Cooperative load of rows of bins into shared memory as shifted codepoints (CP = uint8_t when every
// valid shifted bin is below 256 — half the footprint, twice the resident sequences — else uint16_t).
// status: bit 0 = a value below min_token, bit 1 = a value above max_token (per sequence).
template <typename CP>
__device__ __forceinline__ void stage_rows(const long long* __restrict__ bins, long long base, long long N, int L,
                                           long long min_token, long long max_shift, CP* s_cp, int LP,
                                           int* s_status, int rows_per_block) {
    constexpr long long kCpMax = sizeof(CP) == 1 ? 0xFF : 0xD7FF;
    const long long rows = (N - base) < rows_per_block ? (N - base) : rows_per_block;
    for (long long idx = threadIdx.x; idx < rows * L; idx += blockDim.x) {
        const int r = (int)(idx / L), p = (int)(idx - (long long)r * L);
        const long long v = bins[(base + r) * L + p] - min_token;
        if (v < 0) atomicOr(&s_status[r], 1);
        else if (v > max_shift) atomicOr(&s_status[r], 2);
        s_cp[r * LP + p] = (CP)(v < 0 ? 0 : (v > kCpMax ? kCpMax : v));
    }
}

// ---------------------------------------------------------------- alphabet discovery
__global__ void __launch_bounds__(256)
bpe_minmax_kernel(const long long* __restrict__ bins, long long n, long long* mn, long long* mx) {
    long long a = 0x7fffffffffffffffLL, b = -0x7fffffffffffffffLL - 1;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const long long v = bins[i];
        a = v < a ? v : a;
        b = v > b ? v : b;
    }
    for (int o = 16; o > 0; o >>= 1) {
        const long long a2 = __shfl_xor_sync(0xffffffffu, a, o), b2 = __shfl_xor_sync(0xffffffffu, b, o);
        a = a2 < a ? a2 : a;
        b = b2 > b ? b2 : b;
    }
    if ((threadIdx.x & 31) == 0) { atomicMin(mn, a); atomicMax(mx, b); }
}

// seen[b] = 1 for every UTF-8 byte that occurs (the byte-level characters "seen in words", A.3)
__global__ void __launch_bounds__(256)
bpe_seen_kernel(const long long* __restrict__ bins, long long n, long long min_token, int* seen, int* err) {
    __shared__ int s_seen[256];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) s_seen[i] = 0;
    __syncthreads();
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const long long v = bins[i] - min_token;
        if (v < 0 || v > 0xD7FF) { *err = 1; continue; }
        int bt[3];
        const int nbt = utf8_encode((int)v, bt);
        for (int q = 0; q < nbt; ++q) s_seen[bt[q]] = 1;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 256; i += blockDim.x) if (s_seen[i]) seen[i] = 1;
}

// ---------------------------------------------------------------- symbolise
__global__ void __launch_bounds__(kBpeBlock)
bpe_symbolize_kernel(const long long* __restrict__ bins, long long N, int L, long long min_token,
                     const short* __restrict__ byte_to_id, const uint8_t* __restrict__ cls_tab,
                     uint16_t* __restrict__ sym, int* __restrict__ len, long long n_stride, int* err, int rows,
                     const int* __restrict__ row_len) {
    extern __shared__ uint8_t s_raw[];
    const int LP = L + 1;
    uint16_t* s_cp = (uint16_t*)s_raw;
    int* s_status = (int*)(s_raw + (((size_t)rows * LP * 2 + 3) & ~(size_t)3));
    __shared__ short s_b2i[256];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) s_b2i[i] = byte_to_id[i];
    for (int i = threadIdx.x; i < rows; i += blockDim.x) s_status[i] = 0;
    __syncthreads();
    const long long base = (long long)blockIdx.x * rows;
    stage_rows<uint16_t>(bins, base, N, L, min_token, 0xD7FF, s_cp, LP, s_status, rows);
    __syncthreads();
    const long long seq = base + threadIdx.x;
    if (threadIdx.x >= rows || seq >= N) return;
    if (s_status[threadIdx.x]) *err = 1;
    const uint16_t* cp = s_cp + threadIdx.x * LP;
    // sequences of unequal length arrive padded to L; the text of this one ends at row_len[seq]
    const int Lr = row_len ? min(max(row_len[seq], 0), L) : L;
    // pretoken_len's rules as ONE pass with constant work per codepoint (the lanes of a warp hold different
    // sequences: nested run loops made the warp execute every lane's path, ~630 instructions per codepoint):
    // run_cls = class of the run being extended (-1: the next codepoint opens a pre-token), ws_run = inside a
    // whitespace run of two or more, skip = codepoints left of a contraction ('s 't 're 've 'm 'll 'd).
    int m = 0, run_cls = -1, skip = 0;
    bool ws_run = false;
    unsigned long long lo = 0ull, hi = 0ull;                 // the open chunk of eight symbols
    unsigned int pending = 0u;
    int c = Lr > 0 ? cp[0] : 0, k = Lr > 0 ? cp_class(c, cls_tab) : 0;
    for (int p = 0; p < Lr; ++p) {
        const bool has1 = p + 1 < Lr;
        const int c1 = has1 ? cp[p + 1] : 0;
        const int k1 = has1 ? cp_class(c1, cls_tab) : -1;
        bool start;
        if (skip > 0) {
            start = false;
            --skip;
        } else if (k == CLS_S) {
            const bool next_s = k1 == CLS_S;
            if (!ws_run) {                                   // a whitespace run opens a pre-token
                start = true;
                if (next_s) ws_run = true;
                else run_cls = (has1 && c == 32) ? k1 : -1;  // " ?X+": one blank joins the run behind it
            } else if (next_s || !has1) {
                start = false;                               // \s+(?!\S): inside the run, or the run ends the text
            } else {                                         // ... which leaves the run's last blank to the next match
                start = true;
                ws_run = false;
                run_cls = c == 32 ? k1 : -1;
            }
        } else if (k == run_cls) {
            start = false;
        } else {
            start = true;
            run_cls = k;
            if (c == 39 && has1) {
                const int c2 = p + 2 < Lr ? cp[p + 2] : 0;
                int cl = 0;
                if (c1 == 's' || c1 == 't' || c1 == 'm' || c1 == 'd') cl = 2;
                else if ((c1 == 'r' && c2 == 'e') || (c1 == 'v' && c2 == 'e') || (c1 == 'l' && c2 == 'l')) cl = 3;
                if (cl) { skip = cl - 1; run_cls = -1; }
            }
        }
        if (start) pending = kWordStart;
        int bt[3];
        const int nbt = utf8_encode(c, bt);
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            if (r >= nbt) break;
            const int id = s_b2i[bt[r]];
            if (id < 0) continue;
            const unsigned long long v = (unsigned long long)((unsigned int)id | pending);
            pending = 0u;
            const int pos = m & 7;
            if (pos < 4) lo |= v << (16 * pos);
            else hi |= v << (16 * (pos - 4));
            if (pos == 7) {
                *(uint4*)(sym + ((long long)(m >> 3) * n_stride + seq) * kChunk) =
                    make_uint4((unsigned int)lo, (unsigned int)(lo >> 32), (unsigned int)hi, (unsigned int)(hi >> 32));
                lo = hi = 0ull;
            }
            ++m;
        }
        c = c1;
        k = k1;
    }
    len[seq] = m;
    if (m & 7) {                                             // pad the last chunk
        for (int pos = m & 7; pos < 8; ++pos) {
            if (pos < 4) lo |= 0xffffull << (16 * pos);
            else hi |= 0xffffull << (16 * (pos - 4));
        }
        *(uint4*)(sym + ((long long)(m >> 3) * n_stride + seq) * kChunk) =
            make_uint4((unsigned int)lo, (unsigned int)(lo >> 32), (unsigned int)hi, (unsigned int)(hi >> 32));
    }
}

// ---------------------------------------------------------------- pair histogram
__global__ void __launch_bounds__(256)
bpe_count_kernel(const uint16_t* __restrict__ sym, const int* __restrict__ len, long long N, long long n_stride,
                 int V, int* __restrict__ hist, const int* __restrict__ weight) {
    for (long long seq = (long long)blockIdx.x * blockDim.x + threadIdx.x; seq < N;
         seq += (long long)gridDim.x * blockDim.x) {
        const int n = len[seq];
        if (n < 2) continue;
        const int wgt = weight ? weight[seq] : 1;
        int prev = sym[sym_index(0, seq, n_stride)] & kIdMask;
        for (int q = 1; q < n; ++q) {
            const uint16_t cur = sym[sym_index(q, seq, n_stride)];
            if (!(cur & kWordStart)) atomicAdd(&hist[(long long)prev * V + (cur & kIdMask)], wgt);
            prev = cur & kIdMask;
        }
    }
}

// Same count with a block-private histogram in shared memory over the A DISTINCT ids of the corpus (the
// byte-level symbols before any merge: 194 for a 256-bin tokenizer, 150 KB; their ids are sparse in [0, n_ids),
// so they are renumbered through `used_ids`): the ~200 pair increments per sequence become shared-memory
// atomics, one global atomic per non-zero cell and block at the end.  When A x A counters do not fit, the rows
// (first symbol of the pair) are dealt round-robin to `parts` blocks that read the same sequences — the corpus is
// read `parts` times, which is cheap next to global atomics on a few hundred hot cells.
// 128-bit chunk loads, one thread per sequence.
__global__ void __launch_bounds__(1024)
bpe_count_smem_kernel(const uint16_t* __restrict__ sym, const int* __restrict__ len, long long N, long long n_stride,
                      int V, int n_ids, const short* __restrict__ used_ids, int A, int parts, int* __restrict__ hist,
                      const int* __restrict__ weight) {
    extern __shared__ int s_hist[];                          // [rows*A] counters, then u16 inverse map [n_ids]
    const int rows = (A + parts - 1) / parts, part = (int)(blockIdx.x % (unsigned int)parts);
    const int cells = rows * A;
    unsigned short* s_inv = (unsigned short*)(s_hist + cells);
    for (int i = threadIdx.x; i < cells; i += blockDim.x) s_hist[i] = 0;
    for (int i = threadIdx.x; i < n_ids; i += blockDim.x) s_inv[i] = 0xffffu;
    __syncthreads();
    for (int i = threadIdx.x; i < A; i += blockDim.x) s_inv[used_ids[i]] = (unsigned short)i;
    __syncthreads();
    const long long group = blockIdx.x / (unsigned int)parts, groups = gridDim.x / (unsigned int)parts;
    for (long long seq = group * blockDim.x + threadIdx.x; seq < N; seq += groups * blockDim.x) {
        const int n = len[seq];
        const int wgt = weight ? weight[seq] : 1;
        unsigned int prev = 0xffffu;
        for (int c = 0; c * kChunk < n; ++c) {
            const int4 q = __ldcs((const int4*)(sym + ((long long)c * n_stride + seq) * kChunk));
            const unsigned int w[4] = {(unsigned int)q.x, (unsigned int)q.y, (unsigned int)q.z, (unsigned int)q.w};
#pragma unroll
            for (int j = 0; j < kChunk; ++j) {
                if (c * kChunk + j >= n) break;
                const unsigned int cur = (w[j >> 1] >> ((j & 1) * 16)) & 0xffffu;
                const unsigned int id = cur & kIdMask;
                const unsigned int ci = id < (unsigned int)n_ids ? s_inv[id] : 0xffffu;
                if (prev != 0xffffu && ci != 0xffffu && !(cur & kWordStart)) {
                    if (parts == 1) atomicAdd(&s_hist[prev * A + ci], wgt);
                    else if ((int)(prev % (unsigned int)parts) == part) atomicAdd(&s_hist[(prev / (unsigned int)parts) * A + ci], wgt);
                }
                prev = ci;
            }
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < cells; i += blockDim.x) {
        const int v = s_hist[i];
        const int first = (i / A) * parts + part;
        if (v && first < A) atomicAdd(&hist[(long long)used_ids[first] * V + used_ids[i % A]], v);
    }
}

// Build the pair signatures of every sequence: thread-private bit sets in shared memory (word-major, so
// neither the updates nor the final coalesced column writes conflict), 128-bit chunk loads.
constexpr int kSigBlock = 128;
__global__ void __launch_bounds__(kSigBlock)
bpe_signature_kernel(const uint16_t* __restrict__ sym, const int* __restrict__ len, long long N, long long n_stride,
                     unsigned int* __restrict__ sig) {
    __shared__ unsigned int s_sig[kSigWords * kSigBlock];
    for (long long base = (long long)blockIdx.x * kSigBlock; base < N; base += (long long)gridDim.x * kSigBlock) {
        for (int wd = 0; wd < kSigWords; ++wd) s_sig[wd * kSigBlock + threadIdx.x] = 0;
        const long long seq = base + threadIdx.x;
        if (seq < N) {
            const int n = len[seq];
            unsigned int prev = 0;
            for (int c = 0; c * kChunk < n; ++c) {
                const int4 q = __ldcs((const int4*)(sym + ((long long)c * n_stride + seq) * kChunk));
                const unsigned int w[4] = {(unsigned int)q.x, (unsigned int)q.y, (unsigned int)q.z, (unsigned int)q.w};
#pragma unroll
                for (int j = 0; j < kChunk; ++j) {
                    if (c * kChunk + j >= n) break;
                    const unsigned int cur = (w[j >> 1] >> ((j & 1) * 16)) & 0xffffu;
                    const unsigned int id = cur & kIdMask;
                    if ((c | j) && !(cur & kWordStart)) {
                        const unsigned int h = sig_hash(prev, id), h2 = sig_hash2(prev, id);
                        s_sig[(h >> 5) * kSigBlock + threadIdx.x] |= 1u << (h & 31u);
                        s_sig[(h2 >> 5) * kSigBlock + threadIdx.x] |= 1u << (h2 & 31u);
                    }
                    prev = id;
                }
            }
            for (int wd = 0; wd < kSigWords; ++wd) sig[(long long)wd * n_stride + seq] = s_sig[wd * kSigBlock + threadIdx.x];
        }
    }
}

// ---------------------------------------------------------------- arg-max with the trainer's tie-break
// key = count << 32 | ~flat: the largest key is the largest count and, among equals, the smallest
// flat index a*V + b, i.e. the lexicographically smallest (a, b).
__global__ void __launch_bounds__(256)
bpe_argmax_kernel(const int* __restrict__ hist, int V, int n_active, const BpeCtl* __restrict__ ctl,
                  unsigned long long* __restrict__ result) {
    if (ctl) {
        if (ctl->done) return;
        n_active = ctl->n_tokens;
    }
    unsigned long long best = 0;
    const long long total = (long long)n_active * n_active;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
         i += (long long)gridDim.x * blockDim.x) {
        const int a = (int)(i / n_active), b = (int)(i - (long long)a * n_active);
        const unsigned int flat = (unsigned int)a * (unsigned int)V + (unsigned int)b;
        const int c = hist[flat];
        if (c > 0) {
            const unsigned long long key = ((unsigned long long)(unsigned int)c << 32) | (0xffffffffu - flat);
            best = key > best ? key : best;
        }
    }
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long other = __shfl_xor_sync(0xffffffffu, best, o);
        best = other > best ? other : best;
    }
    __shared__ unsigned long long s_best[8];
    if ((threadIdx.x & 31) == 0) s_best[threadIdx.x >> 5] = best;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < (int)(blockDim.x >> 5); ++w) best = s_best[w] > best ? s_best[w] : best;
        if (best) atomicMax(result, best);
    }
}

// ---------------------------------------------------------------- merge (a, b) -> c
// delta block: [0] column a (pairs (x, a) lost), [1] row b (pairs (b, y) lost),
//              [2] column c (pairs (x, c) gained), [3] row c (pairs (c, y) gained).
// Block-private copies live in shared memory (4*V ints) and are flushed once per block.
// One thread per sequence, one warp per 32 consecutive sequences; the warp walks the chunks in LOCK
// STEP, so every load / store is one 128-bit access per lane over 512 contiguous bytes.
//   pass 1 (read-only): first position q0 whose id is a and whose successor is b inside the same
//           pre-token (b with the word-start bit clear is the 16-bit value b itself; padding never matches);
//   pass 2 (only if some lane found one): streaming rewrite from the warp's first hit chunk — an `a` is
//           held back one step, so no look-ahead is needed: next symbol == b -> emit c (merge),
//           otherwise emit the held symbol unchanged.  Emitted symbols are packed into a 128-bit
//           register window and stored chunk-wise; nothing is stored before a lane's first merge.
__device__ __forceinline__ int warp_max_i(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = max(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ int warp_min_i(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = min(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ uint16_t chunk_get(const uint4& w, int j) {        // j is a compile-time index
    const unsigned int word = j < 2 ? w.x : (j < 4 ? w.y : (j < 6 ? w.z : w.w));
    return (uint16_t)((j & 1) ? (word >> 16) : (word & 0xffffu));
}

// First position q0 whose id is a and whose successor is b inside the same pre-token (b with the word-start
// bit clear is the 16-bit value b itself; padding never matches), or -1.  One lane per sequence, the warp walks
// the chunks in LOCK STEP (512 contiguous bytes per step; all 32 lanes must call).  SWAR search, two symbols per
// 32-bit word: most chunks contain no `a` at all and cost four XOR-AND-ADD-ANDN groups.  `deep`: four independent
// 128-bit loads in flight per lane (few rows: the walk is a chain of dependent round trips) instead of two.
__device__ __forceinline__ int find_first_pair(const uint4* __restrict__ sym4, long long n_stride, long long seq,
                                               bool valid, int n, int a, int b, bool deep) {
    const unsigned int A2 = (unsigned int)a | ((unsigned int)a << 16);
    const unsigned int B2 = (unsigned int)b | ((unsigned int)b << 16);
    const int nch = valid ? (n + kChunk - 1) >> 3 : 0;
    const long long row0 = valid ? seq : 0;
    const int nch_max = warp_max_i(nch);
    int q0 = -1;
    unsigned int carry = 0;                               // bit 15: previous chunk ended with `a`
    auto test_chunk = [&](const uint4& w, int ci) {
        const unsigned int wd[4] = {w.x, w.y, w.z, w.w};
        unsigned int fa[4];                               // bit 15 / 31: half-word has id == a
#pragma unroll
        for (int k = 0; k < 4; ++k) fa[k] = ~(((wd[k] ^ A2) & 0x7fff7fffu) + 0x7fff7fffu) & 0x80008000u;
        if (carry | fa[0] | fa[1] | fa[2] | fa[3]) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const unsigned int y = wd[k] ^ B2;            // fb: half-word == b exactly
                const unsigned int fb = ~((((y & 0x7fff7fffu) + 0x7fff7fffu)) | y) & 0x80008000u;
                const unsigned int h = ((fa[k] << 16) | (k ? fa[k - 1] >> 16 : carry)) & fb;
                if (h && q0 < 0) q0 = ci * kChunk + 2 * k + ((h & 0x8000u) ? 0 : 1) - 1;
            }
        }
        carry = fa[3] >> 16;
    };
    const uint4 pad = make_uint4(0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu);
    if (deep) {
        for (int ci = 0; ci < nch_max; ci += 4) {
            if (ci < nch && q0 < 0) {
                const uint4 w0 = __ldcs(&sym4[(long long)ci * n_stride + row0]);
                const uint4 w1 = ci + 1 < nch ? __ldcs(&sym4[(long long)(ci + 1) * n_stride + row0]) : pad;
                const uint4 w2 = ci + 2 < nch ? __ldcs(&sym4[(long long)(ci + 2) * n_stride + row0]) : pad;
                const uint4 w3 = ci + 3 < nch ? __ldcs(&sym4[(long long)(ci + 3) * n_stride + row0]) : pad;
                test_chunk(w0, ci);
                if (q0 < 0) test_chunk(w1, ci + 1);
                if (q0 < 0) test_chunk(w2, ci + 2);
                if (q0 < 0) test_chunk(w3, ci + 3);
            }
            if (__all_sync(0xffffffffu, q0 >= 0 || ci + 4 >= nch)) break;
        }
    } else {
        for (int ci = 0; ci < nch_max; ci += 2) {         // whole corpus: two loads in flight per lane
            if (ci < nch && q0 < 0) {
                // streaming (evict-first) loads: the corpus pass must not push the V x V histogram out of L2
                const uint4 w0 = __ldcs(&sym4[(long long)ci * n_stride + row0]);
                const uint4 w1 = ci + 1 < nch ? __ldcs(&sym4[(long long)(ci + 1) * n_stride + row0]) : pad;
                test_chunk(w0, ci);
                if (q0 < 0) test_chunk(w1, ci + 1);
            }
            if (__all_sync(0xffffffffu, q0 >= 0 || ci + 2 >= nch)) break;
        }
    }
    return q0;
}

// Scan kernel of the host-driven loop (bpe_apply_merge): sequences with a hit are appended to the work list
// (warp-aggregated atomic), the rewrite kernel below consumes it.
__global__ void __launch_bounds__(256)
bpe_scan_kernel(const uint16_t* __restrict__ sym, const int* __restrict__ len, long long N, long long n_stride,
                int a, int b, int* __restrict__ work_count, int* __restrict__ work_seq, int* __restrict__ work_q0) {
    const uint4* sym4 = (const uint4*)sym;
    const int lane = threadIdx.x & 31;
    for (long long base = (long long)blockIdx.x * blockDim.x + (threadIdx.x & ~31); base < N;
         base += (long long)gridDim.x * blockDim.x) {
        const long long seq = base + lane;
        const bool valid = seq < N;
        const int q0 = find_first_pair(sym4, n_stride, seq, valid, valid ? len[seq] : 0, a, b, false);
        const unsigned int hits = __ballot_sync(0xffffffffu, q0 >= 0);
        if (hits) {
            int slot0 = 0;
            if (lane == 0) slot0 = atomicAdd(work_count, __popc(hits));
            slot0 = __shfl_sync(0xffffffffu, slot0, 0);
            if (q0 >= 0) {
                const int slot = slot0 + __popc(hits & ((1u << lane) - 1u));
                work_seq[slot] = (int)seq;
                work_q0[slot] = q0;
            }
        }
    }
}

// Rewrite kernel (pass 2): one thread per work-list entry.  Streaming state machine from the chunk of
// q0: an `a` is held back one step, so no look-ahead is needed — next symbol == b -> emit c (merge),
// otherwise emit the held symbol unchanged.  Emitted symbols are packed into a 128-bit register window
// and stored chunk-wise (in place: the write position never overtakes the read position); nothing is
// stored before the first merge.  Count changes go to the block-private delta block.
__device__ __forceinline__ void rewrite_sequence(uint16_t* __restrict__ sym, int* __restrict__ len, long long seq,
                                                 int q0, long long n_stride, int a, int b, int c, int V,
                                                 int* s_delta, unsigned int* __restrict__ sig, int wgt) {
    auto sig_add = [&](int x, int y) {                        // the rewritten sequence now holds the pair (x, y)
        if (sig) {
            const unsigned int h = sig_hash((unsigned int)x, (unsigned int)y), h2 = sig_hash2((unsigned int)x, (unsigned int)y);
            atomicOr(&sig[(long long)(h >> 5) * n_stride + seq], 1u << (h & 31u));   // no return value: fire and forget
            atomicOr(&sig[(long long)(h2 >> 5) * n_stride + seq], 1u << (h2 & 31u));
        }
    };
    // s_delta: block-private counters in shared memory (long work lists) or the global delta block itself
    // (short lists: the few changes go out as fire-and-forget reductions); inlined per call site
    int* col_a = s_delta;
    int* row_b = s_delta + V;
    int* col_c = s_delta + 2 * V;
    int* row_c = s_delta + 3 * V;
    const uint16_t bsym = (uint16_t)b;
    uint4* sym4 = (uint4*)sym;
    const int n = len[seq];
    const int nch = (n + kChunk - 1) >> 3;
    const int cs = q0 >> 3;
    int o = cs * kChunk;                                      // output position
    unsigned long long olo = 0ull, ohi = 0ull;                // 8 x 16-bit output window
    bool prev_merged = false, pend = false, dirty = false;
    uint16_t pend_sym = 0;
    int prev_old = 0, prev_new = 0;                           // left neighbour ids (old / emitted)
    if (cs > 0) {
        const uint4 w = sym4[(long long)(cs - 1) * n_stride + seq];
        prev_old = prev_new = (w.w >> 16) & kIdMask;
    }
    auto push = [&](uint16_t x) {                             // append to the window, store when a chunk fills
        const int k = o & 7;
        if (k < 4) olo |= (unsigned long long)x << (16 * k);
        else ohi |= (unsigned long long)x << (16 * (k - 4));
        ++o;
        if ((o & 7) == 0) {
            if (dirty)
                sym4[(long long)((o >> 3) - 1) * n_stride + seq] =
                    make_uint4((unsigned int)olo, (unsigned int)(olo >> 32), (unsigned int)ohi, (unsigned int)(ohi >> 32));
            olo = 0ull;
            ohi = 0ull;
        }
    };
    auto emit_plain = [&](uint16_t x) {
        const int id = x & kIdMask;
        if (prev_merged && !(x & kWordStart)) {              // right neighbour of a merge
            atomicAdd(&row_b[id], -wgt);                     // (b, y) disappears
            atomicAdd(&row_c[id], wgt);                      // (c, y) appears
            sig_add(c, id);
        }
        prev_merged = false;
        prev_old = id;
        prev_new = id;
        push(x);
    };
    // the chunks of one sequence are n_stride * 16 bytes apart: pull the next few towards L1 ahead of the
    // one-deep register pipeline (reads run ahead of the in-place writes, which never pass chunk ci)
    auto prefetch_chunk = [&](int ci) {
        if (ci < nch) asm volatile("prefetch.global.L1 [%0];" ::"l"(&sym4[(long long)ci * n_stride + seq]));
    };
    uint4 w_next = sym4[(long long)cs * n_stride + seq];
    prefetch_chunk(cs + 1); prefetch_chunk(cs + 2); prefetch_chunk(cs + 3); prefetch_chunk(cs + 4);
    for (int ci = cs; ci < nch; ++ci) {
        const uint4 w = w_next;
        if (ci + 1 < nch) w_next = sym4[(long long)(ci + 1) * n_stride + seq];   // next chunk in flight while this one is processed
        prefetch_chunk(ci + 5);
#pragma unroll
        for (int j = 0; j < kChunk; ++j) {
            if (ci * kChunk + j >= n) break;
            const uint16_t cur = chunk_get(w, j);
            if (pend) {
                pend = false;
                if (cur == bsym) {                           // merge (held a, b) -> c
                    if (!(pend_sym & kWordStart)) {          // the pair with the left neighbour changes
                        atomicAdd(&col_a[prev_old], -wgt);   // (old left, a) disappears
                        atomicAdd(&col_c[prev_new], wgt);    // (new left, c) appears
                        sig_add(prev_new, c);
                    }
                    dirty = true;
                    prev_merged = true;
                    prev_old = b;
                    prev_new = c;
                    push((uint16_t)c | (pend_sym & kWordStart));
                    continue;
                }
                emit_plain(pend_sym);
            }
            if ((cur & kIdMask) == a) { pend = true; pend_sym = cur; }
            else emit_plain(cur);
        }
    }
    if (pend) emit_plain(pend_sym);
    const int n_new = o;
    while (o & 7) push(kPad);                                 // pad and flush the last chunk
    len[seq] = n_new;
}

// Warp-cooperative rewrite of ONE sequence (short work lists: the steady state of training, where the
// latency of a single divergent thread per sequence is the cost).  Lane l owns chunk cs + l (eight
// symbols in registers); the caller guarantees at most 32 chunks from cs on.
//   cand[p]  = id[p] == a and the next symbol is exactly b (same pre-token)
//   match[p] = cand[p] and not match[p-1]          (left-to-right, non-overlapping; matters only for a == b)
// The recurrence is a composition of one-bit functions, so each lane evaluates its chunk for both possible
// inputs and a warp scan of the compositions yields every lane's true input.  Symbol p+1 of a match is
// dropped, symbol p becomes c; output positions are a prefix sum of the kept counts; count changes of
// the neighbours go to the global delta block (and the signature) as fire-and-forget reductions.
__device__ __forceinline__ void rewrite_sequence_warp(uint16_t* __restrict__ sym, int* __restrict__ len, long long seq,
                                                      int q0, int n, long long n_stride, int a, int b, int c, int V,
                                                      int* __restrict__ delta, unsigned int* __restrict__ sig,
                                                      uint16_t* s_out, int wgt) {
    const unsigned int FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    uint4* sym4 = (uint4*)sym;
    const int nch = (n + kChunk - 1) >> 3;
    const int cs = q0 >> 3;
    const int ci = cs + lane;
    const uint16_t bsym = (uint16_t)b;
    uint4 w = make_uint4(0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu);
    if (ci < nch) w = sym4[(long long)ci * n_stride + seq];
    unsigned int s[kChunk];
#pragma unroll
    for (int j = 0; j < kChunk; ++j) s[j] = chunk_get(w, j);
    // neighbours across lanes: two symbols ahead, one behind
    unsigned int nx0 = __shfl_down_sync(FULL, s[0], 1), nx1 = __shfl_down_sync(FULL, s[1], 1);
    unsigned int pv7 = __shfl_up_sync(FULL, s[7], 1);
    if (lane == 31) { nx0 = kPad; nx1 = kPad; }
    if (lane == 0) {
        pv7 = kPad;
        if (cs > 0) pv7 = (sym4[(long long)(cs - 1) * n_stride + seq].w >> 16) & 0xffffu;
    }
    const int p0 = ci * kChunk;                               // position of s[0]
    auto at = [&](int j) -> unsigned int { return j < 0 ? pv7 : (j < kChunk ? s[j < 0 ? 0 : (j > 7 ? 7 : j)] : (j == 8 ? nx0 : nx1)); };
    unsigned int cand = 0;
#pragma unroll
    for (int j = 0; j < kChunk; ++j) {
        const unsigned int nxt = j + 1 < kChunk ? s[j + 1 < kChunk ? j + 1 : 7] : nx0;
        if (p0 + j + 1 < n && (s[j] & kIdMask) == (unsigned int)a && nxt == bsym) cand |= 1u << j;
    }
    // match bits for incoming 0 / 1, then the lane's true input by a scan over function compositions
    auto run = [&](unsigned int m_in) {
        unsigned int m = 0, prev = m_in;
#pragma unroll
        for (int j = 0; j < kChunk; ++j) {
            const unsigned int mj = ((cand >> j) & 1u) & (prev ^ 1u);
            m |= mj << j;
            prev = mj;
        }
        return m;
    };
    const unsigned int m_if0 = run(0u), m_if1 = run(1u);
    unsigned int f = ((m_if0 >> 7) & 1u) | (((m_if1 >> 7) & 1u) << 1);     // bit x = output for input x
    for (int o = 1; o < 32; o <<= 1) {                        // inclusive scan: F_l = f_l o F_{l-o}
        const unsigned int g = __shfl_up_sync(FULL, f, o);
        if (lane >= o) f = ((f >> (g & 1u)) & 1u) | (((f >> ((g >> 1) & 1u)) & 1u) << 1);
    }
    unsigned int m_in = __shfl_up_sync(FULL, f & 1u, 1);      // the sequence enters chunk cs with input 0
    if (lane == 0) m_in = 0;
    const unsigned int match = m_in ? m_if1 : m_if0;
    const unsigned int match_prev = __shfl_up_sync(FULL, match, 1), match_next = __shfl_down_sync(FULL, match, 1);
    auto is_match = [&](int j) -> bool {                      // j in [-2, 9]
        if (j < 0) return lane > 0 && ((match_prev >> (j + kChunk)) & 1u);
        if (j < kChunk) return (match >> j) & 1u;
        return lane < 31 && ((match_next >> (j - kChunk)) & 1u);
    };
    auto sig_add = [&](int x, int y) {
        if (sig) {
            const unsigned int h = sig_hash((unsigned int)x, (unsigned int)y), h2 = sig_hash2((unsigned int)x, (unsigned int)y);
            atomicOr(&sig[(long long)(h >> 5) * n_stride + seq], 1u << (h & 31u));
            atomicOr(&sig[(long long)(h2 >> 5) * n_stride + seq], 1u << (h2 & 31u));
        }
    };
    // kept symbols of this lane and their values
    int kept = 0;
    unsigned int outv[kChunk];
#pragma unroll
    for (int j = 0; j < kChunk; ++j) {
        const bool valid = p0 + j < n;
        const bool dropped = j == 0 ? (m_in != 0) : ((match >> (j - 1)) & 1u);
        outv[j] = 0xffffffffu;                                // not kept
        if (valid && !dropped) {
            outv[j] = ((match >> j) & 1u) ? ((unsigned int)c | (s[j] & kWordStart)) : s[j];
            ++kept;
        }
        if ((match >> j) & 1u) {                              // neighbour counts of the merge at p0 + j
            if (!(s[j] & kWordStart)) {                       // a left neighbour inside the pre-token
                const bool left_merged = is_match(j - 2);
                const int prev_old = left_merged ? b : (int)(at(j - 1) & kIdMask);
                const int prev_new = left_merged ? c : prev_old;
                atomicAdd(&delta[prev_old], -wgt);            // (old left, a) disappears
                atomicAdd(&delta[2 * V + prev_new], wgt);     // (new left, c) appears
                sig_add(prev_new, c);
            }
            const unsigned int r = at(j + 2);
            if (p0 + j + 2 < n && !(r & kWordStart) && !is_match(j + 2)) {
                const int id = (int)(r & kIdMask);
                atomicAdd(&delta[V + id], -wgt);              // (b, y) disappears
                atomicAdd(&delta[3 * V + id], wgt);           // (c, y) appears
                sig_add(c, id);
            }
        }
    }
    int inc = kept;
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(FULL, inc, o);
        if (lane >= o) inc += t;
    }
    const int total = __shfl_sync(FULL, inc, 31);
    int o = inc - kept;
#pragma unroll
    for (int j = 0; j < kChunk; ++j)
        if (outv[j] != 0xffffffffu) s_out[o++] = (uint16_t)outv[j];
    const int padded = (total + kChunk - 1) & ~(kChunk - 1);
    for (int i = total + lane; i < padded; i += 32) s_out[i] = kPad;
    __syncwarp();
    if (lane * kChunk < padded) {
        const uint16_t* src = s_out + lane * kChunk;
        sym4[(long long)(cs + lane) * n_stride + seq] =
            make_uint4((unsigned int)src[0] | ((unsigned int)src[1] << 16), (unsigned int)src[2] | ((unsigned int)src[3] << 16),
                       (unsigned int)src[4] | ((unsigned int)src[5] << 16), (unsigned int)src[6] | ((unsigned int)src[7] << 16));
    }
    if (lane == 0) len[seq] = cs * kChunk + total;
    __syncwarp();
}

// A "virtual block": the scan and rewrite phases are written for blocks of 256 threads.  As stand-alone kernels a
// virtual block is a CUDA block (barrier 0); inside the persistent loop kernel a 1024-thread block hosts four of them
// (named barriers 1..4, private shared-memory regions), so that the same code runs in both.
struct VBlock {
    int tid, bid, nblocks, nthreads, bar;
};
__device__ __forceinline__ void vb_sync(const VBlock& vb) {
    asm volatile("bar.sync %0, %1;" ::"r"(vb.bar), "r"(vb.nthreads) : "memory");
}
__device__ __forceinline__ VBlock real_block() {
    VBlock vb;
    vb.tid = (int)threadIdx.x; vb.bid = (int)blockIdx.x; vb.nblocks = (int)gridDim.x; vb.nthreads = (int)blockDim.x; vb.bar = 0;
    return vb;
}

// Block-private 4 x V delta counters in (dynamic, 16-byte aligned) shared memory: zero / flush with
// 128-bit accesses; only non-zero counters reach the global delta block.
__device__ __forceinline__ void zero_delta_block(const VBlock& vb, int* s_delta, int V) {
    int4* p = (int4*)s_delta;
    for (int i = vb.tid; i < V; i += vb.nthreads) p[i] = make_int4(0, 0, 0, 0);      // 4 V ints = V int4
}
__device__ __forceinline__ void flush_delta_block(const VBlock& vb, const int* s_delta, int* __restrict__ delta, int V) {
    const int4* p = (const int4*)s_delta;
    for (int i = vb.tid; i < V; i += vb.nthreads) {
        const int4 d = p[i];
        if (d.x | d.y | d.z | d.w) {
            if (d.x) atomicAdd(&delta[4 * i], d.x);
            if (d.y) atomicAdd(&delta[4 * i + 1], d.y);
            if (d.z) atomicAdd(&delta[4 * i + 2], d.z);
            if (d.w) atomicAdd(&delta[4 * i + 3], d.w);
        }
    }
}

constexpr int kRewriteOut = 32 * kChunk + kChunk;            // staging of one warp-rewritten sequence (symbols)
__device__ __forceinline__ void
rewrite_body(const VBlock& vb, int* s_delta, uint16_t (*s_out)[kRewriteOut],
             uint16_t* __restrict__ sym, int* __restrict__ len, long long n_stride, int a, int b, int c, int V,
             const BpeCtl* __restrict__ ctl, const int* __restrict__ work_count,
             const int* __restrict__ work_seq, const int* __restrict__ work_q0, int* __restrict__ delta,
             unsigned int* __restrict__ sig, const int* __restrict__ weight) {
    if (ctl) {                                                // the state the scan kernel's pick wrote
        if (ctl->done) return;
        a = ctl->a; b = ctl->b; c = ctl->c;
        delta += ((ctl->n_merges - 1) & 1) * 4 * V;           // double-buffered by merge parity (peers may still read the other half)
    }
    const int n_work = *work_count;
    if (n_work > kDirectDeltaWork && (long long)vb.bid * vb.nthreads >= n_work) return;       // nothing for this block
    if (n_work <= kDirectDeltaWork) {
        // short work list (the steady state after the first ~100 merges): the few count changes go straight
        // to the global delta block as fire-and-forget reductions, no 4 x V block-private counters to zero and
        // flush; one WARP per sequence (entries with more than 32 chunks left take the one-thread state machine)
        const int lane = vb.tid & 31, warp = vb.tid >> 5, nw = vb.nthreads >> 5;
        // a warp's entries are e0 + k * stride: the lanes fetch the (sequence, position, length) triples of up to
        // 32 of them at once, so that dependent-load chain is paid once per batch; the chunks of entry k + 1 are
        // pulled towards L1 while entry k is rewritten
        const long long stride = (long long)vb.nblocks * nw;
        const uint4* sym4 = (const uint4*)sym;
        const bool use_smem = n_work > kGlobalDeltaWork && s_delta != nullptr;   // nullptr: 4 x V counters do not fit shared memory
        if (use_smem) {
            if ((long long)vb.bid * nw >= n_work) return;        // no entry for this block
            zero_delta_block(vb, s_delta, V);
            vb_sync(vb);
        }
        for (long long e0 = (long long)vb.bid * nw + warp; e0 < n_work; e0 += 32 * stride) {
            const long long my_e = e0 + lane * stride;
            const bool have = my_e < n_work;
            const int my_seq = have ? work_seq[my_e] : 0, my_q0 = have ? work_q0[my_e] : 0;
            const int my_n = have ? len[my_seq] : 0;
            const int my_w = (have && weight) ? weight[my_seq] : 1;
            const int cnt = __popc(__ballot_sync(0xffffffffu, have));
            for (int k = 0; k < cnt; ++k) {
                const long long seq = __shfl_sync(0xffffffffu, my_seq, k);
                const int q0 = __shfl_sync(0xffffffffu, my_q0, k), n = __shfl_sync(0xffffffffu, my_n, k);
                const int wgt = __shfl_sync(0xffffffffu, my_w, k);
                if (k + 1 < cnt) {
                    const long long seq2 = __shfl_sync(0xffffffffu, my_seq, k + 1);
                    const int ci2 = (__shfl_sync(0xffffffffu, my_q0, k + 1) >> 3) + lane;
                    const int nch2 = (__shfl_sync(0xffffffffu, my_n, k + 1) + kChunk - 1) >> 3;
                    if (ci2 < nch2) asm volatile("prefetch.global.L1 [%0];" ::"l"(&sym4[(long long)ci2 * n_stride + seq2]));
                }
                const int chunks_left = ((n + kChunk - 1) >> 3) - (q0 >> 3);
                if (use_smem) {                               // block-private counters: hot neighbours would serialise in L2
                    if (chunks_left <= 32) rewrite_sequence_warp(sym, len, seq, q0, n, n_stride, a, b, c, V, s_delta, sig, s_out[warp], wgt);
                    else if (lane == 0) rewrite_sequence(sym, len, seq, q0, n_stride, a, b, c, V, s_delta, sig, wgt);
                } else {
                    if (chunks_left <= 32) rewrite_sequence_warp(sym, len, seq, q0, n, n_stride, a, b, c, V, delta, sig, s_out[warp], wgt);
                    else if (lane == 0) rewrite_sequence(sym, len, seq, q0, n_stride, a, b, c, V, delta, sig, wgt);
                }
                __syncwarp();
            }
        }
        if (use_smem) {
            vb_sync(vb);
            flush_delta_block(vb, s_delta, delta, V);
        }
        return;
    }
    if (s_delta != nullptr) {
        zero_delta_block(vb, s_delta, V);
        vb_sync(vb);
    }
    int* target = s_delta != nullptr ? s_delta : delta;         // very large vocabularies: straight to the global block
    for (long long i = (long long)vb.bid * vb.nthreads + vb.tid; i < n_work;
         i += (long long)vb.nblocks * vb.nthreads)
        rewrite_sequence(sym, len, work_seq[i], work_q0[i], n_stride, a, b, c, V, target, sig,
                         weight ? weight[work_seq[i]] : 1);
    if (s_delta != nullptr) {
        vb_sync(vb);
        flush_delta_block(vb, s_delta, delta, V);
    }
}

__global__ void __launch_bounds__(256)
bpe_rewrite_kernel(uint16_t* __restrict__ sym, int* __restrict__ len, long long n_stride, int a, int b, int c, int V,
                   const BpeCtl* __restrict__ ctl, const int* __restrict__ work_count,
                   const int* __restrict__ work_seq, const int* __restrict__ work_q0, int* __restrict__ delta,
                   unsigned int* __restrict__ sig, const int* __restrict__ weight) {
    extern __shared__ int s_delta[];
    __shared__ uint16_t s_out[8][kRewriteOut];
    if (ctl) {
        pdl_wait();
        pdl_launch();
    }
    // V < 0: launched without the 16 |V|-byte dynamic shared memory (vocabularies above 12 800 entries)
    const bool has_smem = V > 0;
    V = V > 0 ? V : -V;
    rewrite_body(real_block(), has_smem ? s_delta : nullptr, s_out, sym, len, n_stride, a, b, c, V, ctl, work_count, work_seq, work_q0,
                 delta, sig, weight);
}

// Iteration head of the sync-free loop: arg-max of the histogram, folding the delta block of the previous merge
// on the way.  The delta touches only column a, row b, column c and row c of the previous merge (a, b) -> c: the
// bulk pass skips those entries (four compares), a short second pass folds and weighs them.
// Sharded runs: the per-merge all-reduce of the 4 x V deltas lives HERE.  Block 0 publishes "my rewrite of merge
// m - 1 is complete" into every peer's flag array (release, system scope) as soon as the kernel starts; the bulk
// pass — which needs nothing from the peers — hides the NVLink round trip; then every block waits for its own
// flags and the fold pass sums the ranks' delta blocks with peer loads.  The histogram replicas stay identical, so
// every rank picks the same merge without a broadcast.
// (One block of 1024 threads per SM writes its maximum to partial[block]; every block of the scan kernel reduces them.)
__device__ __forceinline__ void
iterate_body(int* __restrict__ hist, int V, BpeCtl* __restrict__ ctl, int* __restrict__ delta,
             unsigned long long* __restrict__ partial, int* __restrict__ work_count, const BpePeersDev& peers,
             unsigned long long* s_best) {
    if (ctl->done) return;
    const int n_active = ctl->n_tokens;
    const bool fold = ctl->has_delta != 0;
    const int pa = ctl->a, pb = ctl->b, pc = ctl->c;
    const int epoch = peers.epoch_base + ctl->n_merges;
    const int world = peers.world;
    if (world > 1 && blockIdx.x == 0 && threadIdx.x < world) {
        __threadfence_system();
        st_release_sys(peers.flags[threadIdx.x] + peers.rank, epoch);
    }
    unsigned long long best = 0;
    const int warps_per_block = blockDim.x >> 5, lane = threadIdx.x & 31;
    const bool vec = (V & 3) == 0;
    auto consider = [&](int x, int y, int v) {
        if (v > 0) {
            const unsigned int flat = (unsigned int)x * (unsigned int)V + (unsigned int)y;
            const unsigned long long key = ((unsigned long long)(unsigned int)v << 32) | (0xffffffffu - flat);
            best = key > best ? key : best;
        }
    };
    auto visit = [&](int* row, int x, int y, int v) {
        if (fold) {
            if (y == pa || x == pb || y == pc || x == pc) return;
            if (x == pa && y == pb) { row[y] = 0; return; }
        }
        consider(x, y, v);
    };
    if (vec) {
        // the live n_active x n_active corner as a flat list of 128-bit units, dealt round-robin to ALL
        // threads (a warp reads 512 contiguous bytes), four independent loads in flight per thread
        const unsigned int n4 = (unsigned int)(n_active + 3) >> 2;
        const unsigned int total = (unsigned int)n_active * n4;
        const unsigned int nthreads = gridDim.x * blockDim.x;
        for (unsigned int u0 = blockIdx.x * blockDim.x + threadIdx.x; u0 < total; u0 += 4u * nthreads) {
            int4 q[4];
            unsigned int xs[4], ys[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const unsigned int u = u0 + (unsigned int)k * nthreads;
                xs[k] = u / n4;
                ys[k] = (u - xs[k] * n4) * 4u;
                if (u < total) q[k] = *(const int4*)(hist + (long long)xs[k] * V + ys[k]);
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                if (u0 + (unsigned int)k * nthreads >= total) break;
                int* row = hist + (long long)xs[k] * V;
                const int x = (int)xs[k], y0 = (int)ys[k];
                visit(row, x, y0, q[k].x);
                if (y0 + 1 < n_active) visit(row, x, y0 + 1, q[k].y);
                if (y0 + 2 < n_active) visit(row, x, y0 + 2, q[k].z);
                if (y0 + 3 < n_active) visit(row, x, y0 + 3, q[k].w);
            }
        }
    } else {
        for (int x = blockIdx.x * warps_per_block + (threadIdx.x >> 5); x < n_active; x += gridDim.x * warps_per_block) {
            int* row = hist + (long long)x * V;
            for (int y = lane; y < n_active; y += 32) visit(row, x, y, row[y]);
        }
    }
    if (fold) {
        const int* dloc = delta + ((ctl->n_merges - 1) & 1) * 4 * V;      // this rank's half for merge m - 1
        if (world > 1) {
            // every peer has finished the rewrite of merge m - 1 once its epoch shows up in OUR flag array
            if (threadIdx.x < world && !ctl->err) {
                const int* f = peers.flags[peers.rank] + threadIdx.x;
                if (ld_acquire_sys(f) < epoch) {
                    const unsigned long long t0 = global_ns();
                    while (ld_acquire_sys(f) < epoch) {
                        __nanosleep(64);
                        if (global_ns() - t0 > kPeerWaitNs) { atomicExch(&ctl->err, 1); break; }
                    }
                }
            }
            __syncthreads();
        }
        const int boff = ((ctl->n_merges - 1) & 1) * 4 * V;
        auto dsum = [&](int idx) {
            int acc = dloc[idx];
            if (world > 1) {
                int v[BPE_MAX_PEERS];
#pragma unroll
                for (int r = 0; r < BPE_MAX_PEERS; ++r)
                    v[r] = (r < world && r != peers.rank) ? ld_relaxed_sys(peers.delta[r] + boff + idx) : 0;
#pragma unroll
                for (int r = 0; r < BPE_MAX_PEERS; ++r) acc += v[r];
            }
            return acc;
        };
        // 4 x n_active special entries, one per thread: which = 0 column a (j, a), 1 row b (b, j), 2 column c
        // (j, c), 3 row c (c, j).  An entry on two of the lines belongs to the first one in that order and takes
        // both deltas; the delta half itself is cleared by the iteration head two merges later.
        const unsigned int nthreads = gridDim.x * blockDim.x;
        for (unsigned int i = blockIdx.x * blockDim.x + threadIdx.x; i < 4u * (unsigned int)n_active; i += nthreads) {
            const int which = (int)(i / (unsigned int)n_active), j = (int)(i - (unsigned int)which * n_active);
            const int x = which == 0 ? j : (which == 1 ? pb : (which == 2 ? j : pc));
            const int y = which == 0 ? pa : (which == 1 ? j : (which == 2 ? pc : j));
            const bool on0 = y == pa, on1 = x == pb, on2 = y == pc;
            if ((which == 1 && on0) || (which == 2 && (on0 || on1)) || (which == 3 && (on0 || on1 || on2))) continue;
            int d = 0;
            if (on0) d += dsum(x);
            if (on1) d += dsum(V + y);
            if (on2) d += dsum(2 * V + x);
            if (x == pc) d += dsum(3 * V + y);
            int* cell = hist + (long long)x * V + y;
            int v = *cell + d;
            if (x == pa && y == pb) v = 0;
            if (d != 0 || v == 0) *cell = v;
            consider(x, y, v);
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) *work_count = 0;      // the scan of this iteration refills the work list
    {   // the half that the rewrite of THIS merge fills: it held merge m - 2, which every rank has consumed (the
        // peers published epoch m — awaited above — after their fold of m - 2)
        int4* d4 = (int4*)(delta + (ctl->n_merges & 1) * 4 * V);
        for (unsigned int i = blockIdx.x * blockDim.x + threadIdx.x; i < (unsigned int)V; i += gridDim.x * blockDim.x)
            d4[i] = make_int4(0, 0, 0, 0);
    }
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long other = __shfl_xor_sync(0xffffffffu, best, o);
        best = other > best ? other : best;
    }
    if (lane == 0) s_best[threadIdx.x >> 5] = best;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < warps_per_block; ++w) best = s_best[w] > best ? s_best[w] : best;
        partial[blockIdx.x] = best;                          // plain store: the scan kernel's pick runs after this grid
    }
}

__global__ void __launch_bounds__(1024)
bpe_iterate_kernel(int* __restrict__ hist, int V, BpeCtl* __restrict__ ctl, int* __restrict__ delta,
                   unsigned long long* __restrict__ partial, int* __restrict__ work_count,
                   const __grid_constant__ BpePeersDev peers) {
    __shared__ unsigned long long s_best[32];
    pdl_wait();
    pdl_launch();
    iterate_body(hist, V, ctl, delta, partial, work_count, peers, s_best);
}

// Second kernel of an iteration: pick + scan.
//   pick   EVERY block reduces the per-block maxima of the iteration head and applies BpeTrainer's stop rules
//          (vocabulary full, count < min_frequency) itself — the state is read from ctl_in and the new state written
//          (by block 0) to the OTHER control block, so no block waits for another and no separate launch is
//          needed; block 0 logs the merge.  (A one-block pick kernel cost ~4 us per merge in launch + drain.)
//   scan   a block filters a tile of <= kScanTile sequences by the pair's two signature columns (12.8 MB per merge
//          at 1.6 M sequences instead of the 440 MB corpus), compacts the survivors in shared memory and walks only
//          those (lane per sequence, lock step) for the first hit; hits go to the global work list by
//          warp-aggregated atomics — the rewrite kernel deals them evenly over all warps of the GPU (a fused
//          scan + rewrite was measured 25 % slower: the hits of one warp's 32 survivors then serialise in that warp).
struct ScanSmem {
    int list[kScanTile];
    unsigned long long best[8];
    int pick[4];
    int n;
};
template <bool DEEP>
__device__ __forceinline__ void
pick_scan_body(const VBlock& vb, ScanSmem& sm,
               const uint16_t* __restrict__ sym, const int* __restrict__ len, long long N, long long n_stride, int V,
               const BpeCtl* __restrict__ ctl_in, BpeCtl* __restrict__ ctl_out,
               const unsigned long long* __restrict__ partial, int n_partial, int* __restrict__ log,
               int vocab_size, int min_frequency, int max_merges, int* __restrict__ work_count,
               int* __restrict__ work_seq, int* __restrict__ work_q0, const unsigned int* __restrict__ sig,
               int tile_size) {
    int* s_list = sm.list;
    int& s_n = sm.n;
    unsigned long long* s_best = sm.best;
    int* s_pick = sm.pick;
    const int lane = vb.tid & 31, warp = vb.tid >> 5;
    // ---------------- pick
    const BpeCtl cur = *ctl_in;
    if (cur.done) {
        if (vb.bid == 0 && vb.tid == 0) *ctl_out = cur;
        return;
    }
    unsigned long long best = 0;
    for (int i = vb.tid; i < n_partial; i += vb.nthreads) best = partial[i] > best ? partial[i] : best;
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long other = __shfl_xor_sync(0xffffffffu, best, o);
        best = other > best ? other : best;
    }
    if (lane == 0) s_best[warp] = best;
    vb_sync(vb);
    if (vb.tid == 0) {
        for (int w = 1; w < (int)(vb.nthreads >> 5); ++w) best = s_best[w] > best ? s_best[w] : best;
        const int count = (int)(best >> 32);
        const bool stop = best == 0 || count < 1 || count < min_frequency || cur.n_tokens >= vocab_size ||
                          cur.n_merges >= max_merges || cur.err;
        BpeCtl next = cur;
        next.has_delta = 0;
        if (stop) next.done = 1;
        else {
            const unsigned int flat = 0xffffffffu - (unsigned int)(best & 0xffffffffu);
            next.a = (int)(flat / (unsigned int)V);
            next.b = (int)(flat % (unsigned int)V);
            next.c = cur.n_tokens;
            next.count = count;
            next.n_tokens = cur.n_tokens + 1;
            next.n_merges = cur.n_merges + 1;
            next.has_delta = 1;
        }
        s_pick[0] = next.a; s_pick[1] = next.b; s_pick[3] = stop ? 1 : 0;
        if (vb.bid == 0) {
            *ctl_out = next;
            if (!stop) {
                int* e = log + 4 * cur.n_merges;
                e[0] = next.a; e[1] = next.b; e[2] = next.c; e[3] = count;
            }
        }
    }
    vb_sync(vb);
    if (s_pick[3]) return;
    const int a = s_pick[0], b = s_pick[1];
    // ---------------- scan
    const uint4* sym4 = (const uint4*)sym;
    auto scan_warp = [&](long long seq, bool valid, bool deep) {
        const int q0 = find_first_pair(sym4, n_stride, seq, valid, valid ? len[seq] : 0, a, b, deep);
        const unsigned int hits = __ballot_sync(0xffffffffu, q0 >= 0);
        if (hits) {
            int slot0 = 0;
            if (lane == 0) slot0 = atomicAdd(work_count, __popc(hits));
            slot0 = __shfl_sync(0xffffffffu, slot0, 0);
            if (q0 >= 0) {
                const int slot = slot0 + __popc(hits & ((1u << lane) - 1u));
                work_seq[slot] = (int)seq;
                work_q0[slot] = q0;
            }
        }
    };
    if (!sig) {
        for (long long base = (long long)vb.bid * vb.nthreads + (vb.tid & ~31); base < N;
             base += (long long)vb.nblocks * vb.nthreads)
            scan_warp(base + lane, base + lane < N, false);
        return;
    }
    // signature columns of this pair: sequences whose bits are clear cannot contain (a, b) and are never read
    const unsigned int sh = sig_hash((unsigned int)a, (unsigned int)b), sh2 = sig_hash2((unsigned int)a, (unsigned int)b);
    const unsigned int* sig_col = sig + (long long)(sh >> 5) * n_stride;
    const unsigned int* sig_col2 = sig + (long long)(sh2 >> 5) * n_stride;
    const unsigned int sig_bit = 1u << (sh & 31u), sig_bit2 = 1u << (sh2 & 31u);
    for (long long tile = (long long)vb.bid * tile_size; tile < N; tile += (long long)vb.nblocks * tile_size) {
        if (vb.tid == 0) s_n = 0;
        vb_sync(vb);
        // all signature words of the tile first (up to 16 loads in flight per thread), then the ballots
        unsigned int pass_bits = 0;
#pragma unroll
        for (int r = 0; r < kScanTile / 256; ++r) {
            const int k = vb.tid + r * 256;
            const long long seq = tile + k;
            if (k < tile_size && seq < N && (__ldg(sig_col + seq) & sig_bit) && (__ldg(sig_col2 + seq) & sig_bit2))
                pass_bits |= 1u << r;
        }
        for (int r = 0; r * 256 < tile_size; ++r) {
            const int k = vb.tid + r * 256;
            const bool pass = (pass_bits >> r) & 1u;
            const unsigned int m = __ballot_sync(0xffffffffu, pass);
            if (m) {
                int base = 0;
                if (lane == 0) base = atomicAdd(&s_n, __popc(m));
                base = __shfl_sync(0xffffffffu, base, 0);
                if (pass) s_list[base + __popc(m & ((1u << lane) - 1u))] = k;
            }
        }
        vb_sync(vb);
        const int n_pass = s_n;
        for (int i0 = vb.tid & ~31; i0 < n_pass; i0 += vb.nthreads) {
            const int i = i0 + lane;
            const bool valid = i < n_pass;
            scan_warp(valid ? tile + s_list[i] : 0, valid, DEEP);
        }
        vb_sync(vb);
    }
}

template <bool DEEP>
__global__ void __launch_bounds__(256)
bpe_pick_scan_kernel(const uint16_t* __restrict__ sym, const int* __restrict__ len, long long N, long long n_stride, int V,
                     const BpeCtl* __restrict__ ctl_in, BpeCtl* __restrict__ ctl_out,
                     const unsigned long long* __restrict__ partial, int n_partial, int* __restrict__ log,
                     int vocab_size, int min_frequency, int max_merges, int* __restrict__ work_count,
                     int* __restrict__ work_seq, int* __restrict__ work_q0, const unsigned int* __restrict__ sig,
                     int tile_size) {
    __shared__ ScanSmem sm;
    pdl_wait();
    pdl_launch();
    pick_scan_body<DEEP>(real_block(), sm, sym, len, N, n_stride, V, ctl_in, ctl_out, partial, n_partial, log, vocab_size,
                         min_frequency, max_merges, work_count, work_seq, work_q0, sig, tile_size);
}

// The whole merge loop in ONE cooperative kernel (opt-in, BEAST_B200_BPE_LOOP=persistent): the three phases of an
// iteration are separated by grid barriers instead of kernel boundaries, and the host enqueues one launch per block of
// up to 256 merges.  Slower than the PDL-chained launches on every size measured (see bpe_train_step).  One 1024-thread block per SM; the scan and rewrite phases
// run as four 256-thread virtual blocks per block (VBlock), the code is the stand-alone kernels' code.
struct LoopArgs {
    uint16_t* sym; int* len; long long N, n_stride; int V;
    int* hist; int* delta; BpeCtl* ctl; int* log; unsigned long long* partial;
    int* work_count; int* work_seq; int* work_q0;
    int vocab_size, min_frequency, max_merges;
    unsigned int* sig; const int* weight; int tile_size, first_iter, iters;
};
template <bool DEEP>
__global__ void __launch_bounds__(1024, 1)
bpe_loop_kernel(const __grid_constant__ LoopArgs a, const __grid_constant__ BpePeersDev peers) {
    extern __shared__ __align__(16) int s_dyn[];              // four private 4 x V delta blocks, then the rewrite staging
    __shared__ unsigned long long s_best[32];
    __shared__ ScanSmem s_scan[4];
    uint16_t (*s_out)[8][kRewriteOut] = (uint16_t (*)[8][kRewriteOut])(s_dyn + (size_t)16 * a.V);
    cooperative_groups::grid_group grid = cooperative_groups::this_grid();
    const int sub = (int)(threadIdx.x >> 8);
    VBlock vb;
    vb.tid = (int)(threadIdx.x & 255); vb.bid = (int)blockIdx.x * 4 + sub; vb.nblocks = (int)gridDim.x * 4; vb.nthreads = 256;
    vb.bar = 1 + sub;
    int* s_delta = s_dyn + (size_t)sub * 4 * a.V;
    for (int it = 0; it < a.iters; ++it) {
        const int i = a.first_iter + it;
        BpeCtl* cin = a.ctl + (i & 1);
        BpeCtl* cout = a.ctl + ((i + 1) & 1);
        iterate_body(a.hist, a.V, cin, a.delta, a.partial, a.work_count, peers, s_best);
        grid.sync();
        pick_scan_body<DEEP>(vb, s_scan[sub], a.sym, a.len, a.N, a.n_stride, a.V, cin, cout, a.partial, (int)gridDim.x, a.log,
                             a.vocab_size, a.min_frequency, a.max_merges, a.work_count, a.work_seq, a.work_q0, a.sig, a.tile_size);
        grid.sync();
        if (cout->done) {                                     // uniform: every block reads the state block 0 wrote before the barrier
            if (blockIdx.x == 0 && threadIdx.x == 0) *cin = *cout;       // both control blocks hold the final state
            break;
        }
        if (a.N > 0)
            rewrite_body(vb, s_delta, s_out[sub], a.sym, a.len, a.n_stride, 0, 0, 0, a.V, cout, a.work_count, a.work_seq, a.work_q0,
                         a.delta, a.sig, a.weight);
        grid.sync();
    }
}

// hist += delta (after the optional cross-GPU sum), then the merged pair is gone for good.
__global__ void __launch_bounds__(1024)
bpe_apply_delta_kernel(int* __restrict__ hist, int* __restrict__ delta, int a, int b, int c, int V,
                       const BpeCtl* __restrict__ ctl) {
    if (ctl) {
        if (ctl->done) return;
        a = ctl->a; b = ctl->b; c = ctl->c;
    }
    for (int i = threadIdx.x; i < V; i += blockDim.x) hist[(long long)i * V + a] += delta[i];
    __syncthreads();
    for (int i = threadIdx.x; i < V; i += blockDim.x) hist[(long long)b * V + i] += delta[V + i];
    __syncthreads();
    for (int i = threadIdx.x; i < V; i += blockDim.x) hist[(long long)i * V + c] += delta[2 * V + i];
    __syncthreads();
    for (int i = threadIdx.x; i < V; i += blockDim.x) hist[(long long)c * V + i] += delta[3 * V + i];
    __syncthreads();
    if (threadIdx.x == 0) hist[(long long)a * V + b] = 0;
    for (int i = threadIdx.x; i < 4 * V; i += blockDim.x) delta[i] = 0;
}

// ---------------------------------------------------------------- encode (K5a)
// Merge-rank look-up: rank << 16 | new_id of the pair (a, b), 0xffffffff when it is no merge.  Two table forms:
// dense V x V uint32 (hash_bits == 0: 16 MB at V = 2048, L2-resident) or, for large vocabularies, an open-addressing hash
// of the merges only (2^hash_bits uint2 slots {a << 16 | b, rank << 16 | new_id}, empty key 0xffffffff): O(#merges) memory.
__device__ __forceinline__ unsigned int rank_lookup(const unsigned int* __restrict__ tab, int V, int hash_bits,
                                                    unsigned int a, unsigned int b) {
    if (hash_bits == 0) return __ldg(&tab[(size_t)a * V + b]);
    const unsigned int key = (a << 16) | b, mask = (1u << hash_bits) - 1u;
    const uint2* ht = (const uint2*)tab;
    unsigned int slot = (key * 0x9E3779B1u) >> (32 - hash_bits);
    for (;;) {
        const uint2 e = __ldg(&ht[slot]);
        if (e.x == key) return e.y;
        if (e.x == 0xffffffffu) return 0xffffffffu;
        slot = (slot + 1) & mask;
    }
}

// rank_tab[a*V + b] = rank << 16 | new_id, or 0xffffffff.  One thread per sequence; the word being
// merged lives in local memory with its pair keys cached, so a merge costs one scan + two lookups.
template <int MAXW, typename CP>
__global__ void __launch_bounds__(kBpeBlock)
bpe_encode_kernel(const long long* __restrict__ bins, long long N, int L, long long min_token, long long max_shift,
                  const short* __restrict__ byte_to_id, const uint8_t* __restrict__ cls_tab,
                  const unsigned int* __restrict__ rank_tab, int V, uint16_t* __restrict__ ids_out, int out_stride,
                  int* __restrict__ len_out, int* __restrict__ status_out, int rows, int hash_bits) {
    extern __shared__ uint8_t s_raw[];
    const int LP = L + 1;
    CP* s_cp = (CP*)s_raw;
    int* s_status = (int*)(s_raw + (((size_t)rows * LP * sizeof(CP) + 3) & ~(size_t)3));
    __shared__ short s_b2i[256];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) s_b2i[i] = byte_to_id[i];
    for (int i = threadIdx.x; i < rows; i += blockDim.x) s_status[i] = 0;
    __syncthreads();
    const long long base = (long long)blockIdx.x * rows;
    stage_rows<CP>(bins, base, N, L, min_token, max_shift, s_cp, LP, s_status, rows);
    __syncthreads();
    const long long seq = base + threadIdx.x;
    if (threadIdx.x >= rows || seq >= N) return;
    status_out[seq] = s_status[threadIdx.x];
    if (s_status[threadIdx.x]) { len_out[seq] = 0; return; }
    const CP* cp = s_cp + threadIdx.x * LP;
    uint16_t* out = ids_out + seq * (long long)out_stride;
    uint16_t w[MAXW];
    unsigned int key[MAXW];
    int m = 0, i = 0;
    while (i < L) {
        const int pl = pretoken_len(cp, i, L, cls_tab);
        int wl = 0;
        for (int q = i; q < i + pl; ++q) {
            int bt[3];
            const int nbt = utf8_encode(cp[q], bt);
            for (int r = 0; r < nbt; ++r) {
                const int id = s_b2i[bt[r]];
                if (id >= 0) w[wl++] = (uint16_t)id;
            }
        }
        i += pl;
        for (int q = 0; q + 1 < wl; ++q) key[q] = rank_lookup(rank_tab, V, hash_bits, w[q], w[q + 1]);
        while (wl >= 2) {
            unsigned int best = 0xffffffffu, best_rank = 0xffffffffu;
            int bp = -1;
            for (int q = 0; q + 1 < wl; ++q) {               // lowest rank, leftmost first
                const unsigned int kq = key[q];
                if (kq != 0xffffffffu && (kq >> 16) < best_rank) { best = kq; best_rank = kq >> 16; bp = q; }
            }
            if (bp < 0) break;
            w[bp] = (uint16_t)(best & 0xffffu);
            for (int q = bp + 1; q + 1 < wl; ++q) { w[q] = w[q + 1]; key[q] = key[q + 1]; }
            --wl;
            if (bp > 0) key[bp - 1] = rank_lookup(rank_tab, V, hash_bits, w[bp - 1], w[bp]);
            if (bp + 1 < wl) key[bp] = rank_lookup(rank_tab, V, hash_bits, w[bp], w[bp + 1]);
        }
        for (int q = 0; q < wl; ++q) out[m++] = w[q];
    }
    len_out[seq] = m;
}

// ---------------------------------------------------------------- encode (K5a), one warp per sequence
// The GPT-2 pre-tokeniser is a left-to-right regex, but its token starts are a LOCAL function of the
// codepoints: a class run starts where the class changes (a single U+0020 before a non-space run joins
// it), the last blank of a longer whitespace run splits off when text follows, and an apostrophe that
// starts a token and is followed by s/t/m/d/re/ve/ll swallows those letters and forces a restart after
// them.  (Checked against the sequential matcher on adversarial strings by the CPU test suite.)
// class of a codepoint: Latin-1 from a 256-entry shared-memory copy, the rest from the host-built table
__device__ __forceinline__ int cls_of(int c, const uint8_t* s_cls, const uint8_t* __restrict__ cls_tab) {
    return c < 256 ? (int)s_cls[c] : (int)__ldg(cls_tab + c);
}
__device__ __forceinline__ bool base_start(const uint16_t* cp, int i, int n, const uint8_t* s_cls, const uint8_t* __restrict__ cls_tab) {
    if (i == 0) return true;
    const int k = cls_of(cp[i], s_cls, cls_tab), kp = cls_of(cp[i - 1], s_cls, cls_tab);
    if (k != CLS_S) {
        if (kp == k) return false;
        if (kp == CLS_S) return cp[i - 1] != 32;             // " ?" prefix: the blank belongs to this token
        return true;
    }
    if (kp != CLS_S) return true;
    return i + 1 < n && cls_of(cp[i + 1], s_cls, cls_tab) != CLS_S;  // \s+(?!\S) leaves the last blank
}
__device__ __forceinline__ int contraction_len(const uint16_t* cp, int i, int n) {
    if (i + 1 < n) {
        const int d = cp[i + 1];
        if (d == 's' || d == 't' || d == 'm' || d == 'd') return 2;
        if (i + 2 < n) {
            const int e = cp[i + 2];
            if ((d == 'r' && e == 'e') || (d == 'v' && e == 'e') || (d == 'l' && e == 'l')) return 3;
        }
    }
    return 0;
}
__device__ __forceinline__ bool token_start(const uint16_t* cp, int i, int n, const uint8_t* s_cls, const uint8_t* __restrict__ cls_tab) {
    for (int back = 1; back <= 3 && back <= i; ++back) {
        const int j = i - back;
        if (cp[j] == 39) {
            const int len = contraction_len(cp, j, n);
            if (len > 0 && base_start(cp, j, n, s_cls, cls_tab)) {
                if (back < len) return false;                // inside 's / 're ...
                if (back == len) return true;                // the matcher restarts right after it
            }
        }
    }
    return base_start(cp, i, n, s_cls, cls_tab);
}

// Per warp in shared memory: key u32[M], sym u16[M], wid u16[M], cp u16[L], wbeg u16[L+2]  (M = symbols max).
// A: stage the row (coalesced), B: every lane expands its slice of codepoints into byte-level symbols
// tagged with their word number (one packed warp scan gives symbol and word offsets), C: pair ranks for
// all adjacent symbols in parallel (slot = rank << 16 | symbol) + ordered word list, D: one lane per word
// applies the merges lowest rank first inside its own segment, E: scan of the final word lengths, ids
// written in order.
__global__ void __launch_bounds__(256)
bpe_encode_warp_kernel(const long long* __restrict__ bins, long long N, int L, long long min_token,
                       long long max_shift, const short* __restrict__ byte_to_id,
                       const uint8_t* __restrict__ cls_tab, const unsigned int* __restrict__ rank_tab, int V,
                       uint16_t* __restrict__ ids_out, int out_stride, int* __restrict__ len_out,
                       int* __restrict__ status_out, int M, int warp_bytes, int key2_off, int hash_bits) {
    extern __shared__ __align__(16) uint8_t s_raw[];
    __shared__ short s_b2i[256];
    __shared__ uint8_t s_cls[256];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) { s_b2i[i] = byte_to_id[i]; s_cls[i] = (uint8_t)cp_class_latin1(i); }
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    uint8_t* mine = s_raw + (size_t)warp * warp_bytes;
    unsigned int* key = (unsigned int*)mine;
    uint16_t* sym = (uint16_t*)(key + M);
    uint16_t* wid = sym + M;
    uint16_t* cp = wid + M;
    uint16_t* wbeg = cp + ((L + 1) & ~1);
    unsigned int* key2 = (unsigned int*)(mine + key2_off);      // ping-pong buffer of the cooperative long-word path
    const int P = (L + 31) >> 5;
    const unsigned int FULL = 0xffffffffu, NONE = 0xffffffffu, lt_mask = (1u << lane) - 1u;
    for (long long seq = (long long)blockIdx.x * nw + warp; seq < N; seq += (long long)gridDim.x * nw) {
        // ---- A
        int st = 0;
        const long long* row = bins + seq * L;
        for (int i = lane; i < L; i += 32) {
            const long long v = row[i] - min_token;
            if (v < 0) st |= 1;
            else if (v > max_shift) st |= 2;
            if (v == 39) st |= 4;                              // an apostrophe: the contraction rule may apply
            cp[i] = (uint16_t)(v < 0 ? 0 : (v > 0xD7FF ? 0xD7FF : v));
        }
        st = __reduce_or_sync(FULL, st);
        const bool apos = (st & 4) != 0;                       // warp-uniform: most sequences hold none and skip the look-back
        st &= 3;
        __syncwarp();
        if (st) {
            if (lane == 0) { status_out[seq] = st; len_out[seq] = 0; }
            continue;
        }
        // ---- B
        const int p0 = lane * P, p1 = min(L, p0 + P);
        int ns = 0, nst = 0;
        unsigned int smask = 0;
        for (int i = p0; i < p1; ++i) {
            int bt[3];
            const int nbt = utf8_encode(cp[i], bt);
            for (int r = 0; r < nbt; ++r) ns += s_b2i[bt[r]] >= 0;
            const bool t = apos ? token_start(cp, i, L, s_cls, cls_tab) : base_start(cp, i, L, s_cls, cls_tab);
            nst += t;
            if (t && i - p0 < 32) smask |= 1u << (i - p0);
        }
        const unsigned int packed = ((unsigned int)ns << 16) | (unsigned int)nst;
        unsigned int inc = packed;
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned int t = __shfl_up_sync(FULL, inc, o);
            if (lane >= o) inc += t;
        }
        const int total = (int)(__shfl_sync(FULL, inc, 31) >> 16);
        int off = (int)((inc - packed) >> 16), w = (int)((inc - packed) & 0xffffu);
        for (int i = p0; i < p1; ++i) {
            const bool t = i - p0 < 32 ? ((smask >> (i - p0)) & 1u) != 0
                                       : (apos ? token_start(cp, i, L, s_cls, cls_tab) : base_start(cp, i, L, s_cls, cls_tab));
            w += t;
            int bt[3];
            const int nbt = utf8_encode(cp[i], bt);
            for (int r = 0; r < nbt; ++r) {
                const int id = s_b2i[bt[r]];
                if (id >= 0) { sym[off] = (uint16_t)id; wid[off] = (uint16_t)w; ++off; }
            }
        }
        __syncwarp();
        // ---- C
        int nwords = 0;
        for (int s0 = 0; s0 < total; s0 += 32) {
            const int s = s0 + lane;
            bool isb = false;
            if (s < total) {
                isb = s == 0 || wid[s] != wid[s - 1];
                // slot = rank of the pair (s, s+1) in the high half (0xffff: none), symbol s in the low half
                const unsigned int me = sym[s];
                const unsigned int r = (s + 1 < total && wid[s + 1] == wid[s])
                                           ? rank_lookup(rank_tab, V, hash_bits, me, sym[s + 1]) : NONE;
                key[s] = (r & 0xffff0000u) | me;
            }
            const unsigned int m = __ballot_sync(FULL, isb);
            if (isb) wbeg[nwords + __popc(m & ((1u << lane) - 1u))] = (uint16_t)s;
            nwords += __popc(m);
        }
        if (lane == 0) wbeg[nwords] = (uint16_t)total;
        __syncwarp();
        // ---- D: one lane per word; a word's slots are only touched by its lane.  Lanes that sit in different
        // loops of the merge code serialise, so words are handed out longest class first (>= 7 symbols, 3-6, 2; finer classes cost more in ballots than they save):
        // the lanes of one round then run words of similar length.  Single symbols need no work at all.
        // (`sym` is free after phase C and holds the order list.)
        // Long words (>= kCoopWord symbols: the reference's shipped 1000-bin / 50-basis configuration produces words of
        // ~60 symbols, runs of one character class) are merged by the WHOLE WARP, one word at a time and one RANK per
        // step: the ranks a word's merges are applied in never decrease (a pair created by a merge involves the new
        // token, whose rules were all learned later), so "lowest rank, leftmost first, one merge at a time" equals
        // "for the lowest rank present, merge ALL its occurrences left to right".  A step is a strided min-scan, the
        // left-to-right resolution of overlapping candidates by run parity, a compaction by ballot prefix sums and
        // the re-evaluation of the pair ranks — all lanes busy, all rank look-ups of a step in flight together — instead
        // of one lane's O(length) scan + shift per single merge.
        int n_long = 0;
        for (int w0 = 0; w0 < nwords; w0 += 32) {
            const int wq = w0 + lane;
            const int wl = wq < nwords ? wbeg[wq + 1] - wbeg[wq] : 0;
            const bool in = wl >= kCoopWord;
            const unsigned int m = __ballot_sync(FULL, in);
            if (in) cp[n_long + __popc(m & lt_mask)] = (uint16_t)wq;     // `cp` is free after phase B
            n_long += __popc(m);
        }
        __syncwarp();
        for (int li = 0; li < n_long; ++li) {
            const int wq = cp[li];
            const int b = wbeg[wq];
            int n = wbeg[wq + 1] - b;
            unsigned int* cur = key + b;
            unsigned int* nxt = key2 + b;
            for (;;) {
                unsigned int best = 0xffffu;                  // lowest rank present
                for (int q = lane; q + 1 < n; q += 32) best = min(best, cur[q] >> 16);
                best = __reduce_min_sync(FULL, best);
                if (best == 0xffffu) break;
                int out_n = 0;
                unsigned int m_prev = 0;                      // was the last position of the previous chunk a match
                for (int q0 = 0; q0 < n; q0 += 32) {
                    const int q = q0 + lane;
                    const unsigned int slot = q < n ? cur[q] : NONE;
                    const bool cand = q + 1 < n && (slot >> 16) == best;
                    const unsigned int C = __ballot_sync(FULL, cand);
                    // match[q] = cand[q] and not match[q-1]: inside a run of candidates the matches alternate from the
                    // run's first position (from its second when the run continues a matched position of the last chunk)
                    const unsigned int zeros_below = ~C & lt_mask;
                    const int run_start = zeros_below ? 32 - __clz(zeros_below) : 0;
                    const bool match = cand && ((((lane - run_start) + ((run_start == 0) ? (int)m_prev : 0)) & 1) == 0);
                    const unsigned int Mb = __ballot_sync(FULL, match);
                    const bool dropped = q < n && (lane == 0 ? m_prev != 0 : ((Mb >> (lane - 1)) & 1u) != 0);
                    const bool kept = q < n && !dropped;
                    const unsigned int K = __ballot_sync(FULL, kept);
                    if (kept) {
                        unsigned int v = slot & 0xffffu;
                        if (match) v = rank_lookup(rank_tab, V, hash_bits, v, cur[q + 1] & 0xffffu) & 0xffffu;   // the merged token
                        nxt[out_n + __popc(K & lt_mask)] = v;
                    }
                    out_n += __popc(K);
                    m_prev = (Mb >> 31) & 1u;
                }
                __syncwarp();
                n = out_n;
                for (int q = lane; q < n; q += 32) {          // pair ranks of the shorter word
                    const unsigned int me = nxt[q];
                    const unsigned int r = q + 1 < n ? rank_lookup(rank_tab, V, hash_bits, me, nxt[q + 1]) : NONE;
                    cur[q] = (r & 0xffff0000u) | me;
                }
                __syncwarp();
            }
            if (lane == 0) wid[b] = (uint16_t)n;              // final length, kept in the word's own segment
            __syncwarp();
        }
        int n_order = 0;
        for (int cls = 0; cls < 3; ++cls) {
            for (int w0 = 0; w0 < nwords; w0 += 32) {
                const int wq = w0 + lane;
                int wl = wq < nwords ? wbeg[wq + 1] - wbeg[wq] : 0;
                if (wl >= kCoopWord) wl = 0;                  // done above
                const bool in = cls == 0 ? wl >= 7 : (cls == 1 ? (wl >= 3 && wl <= 6) : wl == 2);
                const unsigned int m = __ballot_sync(FULL, in);
                if (in) sym[n_order + __popc(m & lt_mask)] = (uint16_t)wq;
                n_order += __popc(m);
                if (cls == 0 && wl == 1) wid[wbeg[wq]] = 1;
            }
        }
        __syncwarp();
        for (int oi = lane; oi < n_order; oi += 32) {
            const int wq = sym[oi];
            const int b = wbeg[wq];
            int wl = wbeg[wq + 1] - b;
            unsigned int* wk = key + b;
            while (wl >= 2) {
                // lowest rank, leftmost first: equal ranks mean the same pair, hence equal slots, and the
                // strict compare keeps the first
                unsigned int best = 0xffff0000u;
                int bp = -1;
                for (int q = 0; q + 1 < wl; ++q) {
                    const unsigned int v = wk[q];
                    if (v < best) { best = v; bp = q; }
                }
                if (bp < 0) break;
                const unsigned int left = best & 0xffffu, right = wk[bp + 1] & 0xffffu;
                const unsigned int nid = rank_lookup(rank_tab, V, hash_bits, left, right) & 0xffffu;
                for (int q = bp + 1; q + 1 < wl; ++q) wk[q] = wk[q + 1];
                --wl;
                unsigned int r = 0xffff0000u;
                if (bp + 1 < wl) r = rank_lookup(rank_tab, V, hash_bits, nid, wk[bp + 1] & 0xffffu) & 0xffff0000u;
                wk[bp] = r | nid;
                if (bp > 0) {
                    const unsigned int ls = wk[bp - 1] & 0xffffu;
                    wk[bp - 1] = (rank_lookup(rank_tab, V, hash_bits, ls, nid) & 0xffff0000u) | ls;
                }
            }
            wid[b] = (uint16_t)wl;                           // final length, kept in the word's own segment
        }
        __syncwarp();
        // ---- E
        uint16_t* out = ids_out + seq * (long long)out_stride;
        int done = 0;
        for (int w0 = 0; w0 < nwords; w0 += 32) {
            const int wq = w0 + lane;
            int b = 0, wl = 0;
            if (wq < nwords) { b = wbeg[wq]; wl = wid[b]; }
            int run = wl;
            for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_up_sync(FULL, run, o);
                if (lane >= o) run += t;
            }
            const int o0 = done + run - wl;
            for (int q = 0; q < wl; ++q) out[o0 + q] = (uint16_t)(key[b + q] & 0xffffu);
            done += __shfl_sync(FULL, run, 31);
        }
        if (lane == 0) { len_out[seq] = done; status_out[seq] = 0; }
        __syncwarp();
    }
}

// padded rows -> CSR (offsets are an exclusive scan of len, computed by the caller)
__global__ void __launch_bounds__(256)
bpe_compact_kernel(const uint16_t* __restrict__ padded, int stride, const int* __restrict__ len,
                   const long long* __restrict__ offsets, long long N, int* __restrict__ flat) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (long long seq = (long long)blockIdx.x * (blockDim.x >> 5) + warp; seq < N;
         seq += (long long)gridDim.x * (blockDim.x >> 5)) {
        const int n = len[seq];
        const long long off = offsets[seq];
        for (int q = lane; q < n; q += 32) flat[off + q] = padded[seq * (long long)stride + q];
    }
}

// ---------------------------------------------------------------- decode (K5b)
// ids (CSR) -> token bytes -> UTF-8 -> codepoints + min_token.  status: 1 = id out of range,
// 2 = invalid UTF-8, 3 = decoded length != L (the reference's ValueError, bpe_tokenizer.py:241-244).
__global__ void __launch_bounds__(kBpeBlock)
bpe_decode_kernel(const int* __restrict__ flat, const long long* __restrict__ offsets, long long N, int L,
                  long long min_token, const int* __restrict__ tok_off, const uint8_t* __restrict__ tok_bytes,
                  int n_vocab, long long* __restrict__ bins_out, int* __restrict__ status_out,
                  int* __restrict__ declen_out, int rows_per_block) {
    extern __shared__ uint8_t s_raw[];
    const int LP = L + 1;
    uint16_t* s_cp = (uint16_t*)s_raw;                       // decoded codepoints, [kBpeBlock][LP]
    const long long base = (long long)blockIdx.x * rows_per_block;
    const long long seq = base + threadIdx.x;
    int status = 0, cnt = 0;
    if (threadIdx.x < rows_per_block && seq < N) {
        uint16_t* cp = s_cp + threadIdx.x * LP;
        int pending = 0, acc = 0;
        for (long long p = offsets[seq]; p < offsets[seq + 1] && !status; ++p) {
            const int id = flat[p];
            if (id < 0 || id >= n_vocab) { status = 1; break; }
            for (int q = tok_off[id]; q < tok_off[id + 1]; ++q) {
                const int bt = tok_bytes[q];
                int out_c = -1;
                if (pending) {
                    if ((bt & 0xC0) != 0x80) { status = 2; break; }
                    acc = (acc << 6) | (bt & 0x3F);
                    if (--pending == 0) out_c = acc;
                } else if (bt < 0x80) out_c = bt;
                else if ((bt & 0xE0) == 0xC0) { acc = bt & 0x1F; pending = 1; }
                else if ((bt & 0xF0) == 0xE0) { acc = bt & 0x0F; pending = 2; }
                else if ((bt & 0xF8) == 0xF0) { acc = bt & 0x07; pending = 3; }
                else { status = 2; break; }
                if (out_c >= 0) {
                    if (out_c > 0xFFFF) { status = 2; break; }   // not a shifted bin
                    if (cnt < L) cp[cnt] = (uint16_t)out_c;
                    ++cnt;
                }
            }
        }
        if (!status && pending) status = 2;
        if (!status && cnt != L) status = 3;
        status_out[seq] = status;
        declen_out[seq] = cnt;
    }
    __syncthreads();
    const long long rows = (N - base) < rows_per_block ? (N - base) : rows_per_block;
    for (long long idx = threadIdx.x; idx < rows * L; idx += blockDim.x) {
        const int r = (int)(idx / L), p = (int)(idx - (long long)r * L);
        bins_out[(base + r) * L + p] = (long long)s_cp[r * LP + p] + min_token;
    }
}

// ---------------------------------------------------------------- decode (K5b), fast path: one lane per TOKEN
// The table holds, per token, what the sequential UTF-8 state machine (A.6) does with its bytes: its characters
// (the last one pre-shifted by the continuation bytes it still needs), the continuation bytes the token starts
// with (they finish the previous token's last character) and their payload.  A sequence decodes here when every id
// is in range, no token is flagged slow and every boundary matches (needed == supplied); a token's character index
// is a prefix sum of the tokens' character counts.  Anything else — stray / missing continuation bytes, ids out of
// range, tokens of more than SLOTS characters — is flagged (status kDecodeNeedsBytes) and decoded by the byte-level
// kernel below, which also decides WHICH of the reference's errors the sequence has.
//   SLOTS = 2: 8-byte entries {c0 | c1 << 16, meta}; SLOTS = 6: 16-byte entries {c0|c1, c2|c3, c4|c5, meta};
//   meta = characters started | bytes still needed << 3 | leading continuation bytes << 5 | slow << 7 | payload << 8.
constexpr int kDecodeNeedsBytes = 0x100;
template <int SLOTS>
__global__ void __launch_bounds__(256, 8)
bpe_decode_token_kernel(const int* __restrict__ flat, const long long* __restrict__ offsets, long long N, int L,
                        long long min_token, const void* __restrict__ tok_tab, int n_vocab,
                        long long* __restrict__ bins_out, int* __restrict__ status_out, int* __restrict__ declen_out) {
    extern __shared__ __align__(16) uint8_t s_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const int LP = (L + 7) & ~7;
    uint16_t* s_cp = (uint16_t*)s_raw + (size_t)warp * LP;
    const unsigned int FULL = 0xffffffffu, lt = (1u << lane) - 1u;
    struct Entry { unsigned int c01, c23, c45, meta; };
    auto load_entry = [&](int id, bool in_range) -> Entry {
        Entry e{0u, 0u, 0u, 0u};                               // beyond the end: supplies nothing, needs nothing
        if (!in_range) return e;
        if (id < 0 || id >= n_vocab) { e.meta = 0x80u; return e; }
        if (SLOTS == 2) { const uint2 t = __ldg((const uint2*)tok_tab + id); e.c01 = t.x; e.meta = t.y; }
        else { const uint4 t = __ldg((const uint4*)tok_tab + id); e.c01 = t.x; e.c23 = t.y; e.c45 = t.z; e.meta = t.w; }
        return e;
    };
    for (long long seq = (long long)blockIdx.x * nw + warp; seq < N; seq += (long long)gridDim.x * nw) {
        const long long p0 = offsets[seq];
        const int n = (int)(offsets[seq + 1] - p0);
        const int* ids = flat + p0;
        bool bad = false;
        int cnt = 0;
        Entry cur = load_entry(lane < n ? ids[lane] : 0, lane < n);
        if (n > 0 && (__shfl_sync(FULL, cur.meta, 0) & 0x60u)) bad = true;          // the text starts inside a character
        for (int g0 = 0; g0 < n; g0 += 32) {
            const int qn = g0 + 32 + lane;
            const Entry nxt = load_entry(qn < n ? ids[qn] : 0, qn < n);              // in flight while this group is decoded
            const unsigned int meta = cur.meta;
            unsigned int nmeta = __shfl_down_sync(FULL, meta, 1);
            const unsigned int nmeta0 = __shfl_sync(FULL, nxt.meta, 0);
            if (lane == 31) nmeta = nmeta0;
            const int nst = (int)(meta & 7u);
            const unsigned int need = (meta >> 3) & 3u;
            if ((meta & 0x80u) || need != ((nmeta >> 5) & 3u)) bad = true;
            const unsigned int tail = need ? ((nmeta >> 8) & 0x3ffffu) : 0u;
            int at, total;
            if (SLOTS == 2) {                                   // counts of 0 / 1 / 2: two ballots
                const unsigned int b1 = __ballot_sync(FULL, nst >= 1), b2 = __ballot_sync(FULL, nst >= 2);
                at = cnt + __popc(b1 & lt) + __popc(b2 & lt);
                total = __popc(b1) + __popc(b2);
                unsigned int v0 = cur.c01 & 0xffffu, v1 = cur.c01 >> 16;
                if (nst == 1) v0 |= tail;
                if (nst == 2) v1 |= tail;
                if (nst >= 1 && at < L) s_cp[at] = (uint16_t)v0;
                if (nst >= 2 && at + 1 < L) s_cp[at + 1] = (uint16_t)v1;
            } else {
                int inc = nst;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const int t = __shfl_up_sync(FULL, inc, o);
                    if (lane >= o) inc += t;
                }
                at = cnt + inc - nst;
                total = __shfl_sync(FULL, inc, 31);
                const unsigned int c[6] = {cur.c01 & 0xffffu, cur.c01 >> 16, cur.c23 & 0xffffu, cur.c23 >> 16,
                                           cur.c45 & 0xffffu, cur.c45 >> 16};
#pragma unroll
                for (int k = 0; k < 6; ++k)
                    if (k < nst && at + k < L) s_cp[at + k] = (uint16_t)(k == nst - 1 ? c[k] | tail : c[k]);
            }
            cnt += total;
            cur = nxt;
        }
        if (__any_sync(FULL, bad)) {
            if (lane == 0) status_out[seq] = kDecodeNeedsBytes;
            continue;
        }
        __syncwarp();
        if (lane == 0) { status_out[seq] = cnt != L ? 3 : 0; declen_out[seq] = cnt; }
        long long* out = bins_out + seq * L;
        if ((L & 1) == 0 && (((uintptr_t)bins_out) & 15u) == 0) {
            for (int i = 2 * lane; i < L; i += 64) {
                const unsigned int two = *(const unsigned int*)(s_cp + i);
                *(longlong2*)(out + i) = make_longlong2((long long)(two & 0xffffu) + min_token, (long long)(two >> 16) + min_token);
            }
        } else {
            for (int i = lane; i < L; i += 32) out[i] = (long long)s_cp[i] + min_token;
        }
        __syncwarp();
    }
}

// ---------------------------------------------------------------- decode (K5b), one warp per sequence
// Lanes read the ids (coalesced), a warp scan of the token byte lengths places every token's bytes in
// shared memory, then UTF-8 is decoded in parallel: a byte that is not a continuation byte starts a
// character whose index is the number of such bytes before it (ballot + popcount).  Errors follow the
// sequential decoder's order: the byte stream ends at the first id out of range; an invalid byte before
// that point gives status 2, else the bad id gives 1, else an unfinished character at the end gives 2,
// else a character count != L gives 3 (the reference's length ValueError, bpe_tokenizer.py:241-244).
__device__ __forceinline__ int utf8_lead_len(int b) {
    return b < 0x80 ? 1 : ((b & 0xE0) == 0xC0 ? 2 : ((b & 0xF0) == 0xE0 ? 3 : ((b & 0xF8) == 0xF0 ? 4 : 0)));
}

__global__ void __launch_bounds__(256)
bpe_decode_warp_kernel(const int* __restrict__ flat, const long long* __restrict__ offsets, long long N, int L,
                       long long min_token, const int* __restrict__ tok_off, const uint8_t* __restrict__ tok_bytes,
                       int n_vocab, long long* __restrict__ bins_out, int* __restrict__ status_out,
                       int* __restrict__ declen_out, int cap, int warp_bytes, int only_flagged) {
    extern __shared__ __align__(16) uint8_t s_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    uint8_t* s_b = s_raw + (size_t)warp * warp_bytes;
    uint16_t* s_cp = (uint16_t*)(s_b + ((cap + 15) & ~15));
    const unsigned int FULL = 0xffffffffu, lt = (1u << lane) - 1u;
    for (long long seq = (long long)blockIdx.x * nw + warp; seq < N; seq += (long long)gridDim.x * nw) {
        const long long p0 = offsets[seq], p1 = offsets[seq + 1];
        if (only_flagged && status_out[seq] != kDecodeNeedsBytes) continue;   // decoded by the per-token fast kernel
        int B = 0, status = 0, cnt = 0;
        bool bad_tok = false, overflow = false;
        for (long long q0 = p0; q0 < p1; q0 += 32) {
            const long long q = q0 + lane;
            const int id = q < p1 ? flat[q] : 0;
            const bool isbad = q < p1 && (id < 0 || id >= n_vocab);
            const unsigned int badm = __ballot_sync(FULL, isbad);
            const int nvalid = badm ? __ffs(badm) - 1 : 32;
            int b0 = 0, len = 0;
            if (q < p1 && lane < nvalid) { b0 = tok_off[id]; len = tok_off[id + 1] - b0; }
            int inc = len;
            for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_up_sync(FULL, inc, o);
                if (lane >= o) inc += t;
            }
            const int total = __shfl_sync(FULL, inc, 31);
            if (B + total > cap) { overflow = true; break; }
            const int at = B + inc - len;
            for (int k = 0; k < len; ++k) s_b[at + k] = tok_bytes[b0 + k];
            B += total;
            if (badm) { bad_tok = true; break; }
        }
        __syncwarp();
        if (overflow) {
            // more bytes than any valid sequence can have: the sequential state machine decides which error
            // comes first (rare; one lane, straight from global memory)
            if (lane == 0) {
                int pending = 0, acc = 0;
                for (long long p = p0; p < p1 && !status; ++p) {
                    const int id = flat[p];
                    if (id < 0 || id >= n_vocab) { status = 1; break; }
                    for (int q = tok_off[id]; q < tok_off[id + 1]; ++q) {
                        const int bt = tok_bytes[q];
                        int out_c = -1;
                        if (pending) {
                            if ((bt & 0xC0) != 0x80) { status = 2; break; }
                            acc = (acc << 6) | (bt & 0x3F);
                            if (--pending == 0) out_c = acc;
                        } else if (bt < 0x80) out_c = bt;
                        else if (utf8_lead_len(bt) >= 2) { pending = utf8_lead_len(bt) - 1; acc = bt & (0x3F >> pending); }
                        else { status = 2; break; }
                        if (out_c >= 0) {
                            if (out_c > 0xFFFF) { status = 2; break; }
                            if (cnt < L) s_cp[cnt] = (uint16_t)out_c;
                            ++cnt;
                        }
                    }
                }
                if (!status && pending) status = 2;
                if (!status && cnt != L) status = 3;
            }
            status = __shfl_sync(FULL, status, 0);
            cnt = __shfl_sync(FULL, cnt, 0);
        } else {
            int first_err = 0x7fffffff, n_start = 0;
            bool pend_end = false;
            for (int i0 = 0; i0 < B; i0 += 32) {
                const int i = i0 + lane;
                const bool valid = i < B;
                const int b = valid ? s_b[i] : 0;
                const bool cont = valid && (b & 0xC0) == 0x80;
                const bool start = valid && !cont;
                int err = 0x7fffffff, cpv = -1;
                if (start) {
                    const int n = utf8_lead_len(b);
                    if (n == 0) err = i;                      // 0xF8..0xFF
                    else {
                        int acc = n == 1 ? b : (b & (0x7F >> n));
                        bool complete = true;
                        for (int k = 1; k < n; ++k) {
                            if (i + k >= B) { pend_end = true; complete = false; break; }
                            const int c = s_b[i + k];
                            if ((c & 0xC0) != 0x80) { err = i + k; complete = false; break; }
                            acc = (acc << 6) | (c & 0x3F);
                        }
                        if (complete) {
                            if (acc > 0xFFFF) err = i + n - 1;
                            else cpv = acc;
                        }
                    }
                } else if (cont) {                            // must lie inside the span of the lead before it
                    bool covered = false;
                    for (int k = 1; k <= 3 && k <= i; ++k) {
                        const int c = s_b[i - k];
                        if ((c & 0xC0) != 0x80) { covered = utf8_lead_len(c) > k; break; }
                    }
                    if (!covered) err = i;
                }
                const unsigned int sm = __ballot_sync(FULL, start);
                const int idx = n_start + __popc(sm & lt);
                if (cpv >= 0 && idx < L) s_cp[idx] = (uint16_t)cpv;
                n_start += __popc(sm);
                first_err = min(first_err, __reduce_min_sync(FULL, err));
            }
            pend_end = __any_sync(FULL, pend_end);
            cnt = n_start - (pend_end ? 1 : 0);
            if (first_err != 0x7fffffff) status = 2;
            else if (bad_tok) status = 1;
            else if (pend_end) status = 2;
            else if (cnt != L) status = 3;
        }
        __syncwarp();
        if (lane == 0) { status_out[seq] = status; declen_out[seq] = cnt; }
        long long* out = bins_out + seq * L;
        for (int i = lane; i < L; i += 32) out[i] = (long long)s_cp[i] + min_token;
        __syncwarp();
    }
}

static int bpe_grid(long long n, int block) {
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    long long g = (n + block - 1) / block;
    const long long cap = (long long)sms * 16;
    if (g > cap) g = cap;
    if (g < 1) g = 1;
    return (int)g;
}

// rows of bins staged per block: as many as fit in ~180 KB of shared memory, at most one per thread
static int stage_rows_per_block(int L, int cp_bytes = 2) {
    long long r = (180 * 1024) / ((long long)(L + 1) * cp_bytes + 4);
    if (r > kBpeBlock) r = kBpeBlock;
    return (int)r;
}
static size_t stage_smem(int L, int rows, int cp_bytes = 2) {
    return (((size_t)rows * (L + 1) * cp_bytes + 3) & ~(size_t)3) + (size_t)rows * sizeof(int);
}

}  // namespace beast

using namespace beast;

extern "C" int bpe_scan_bins(const int64_t* bins, int64_t n, int64_t min_token, int64_t* minmax, int32_t* seen,
                             int32_t* err, int32_t phase, void* stream) {
    if (!bins || n < 1) return n == 0 ? BEAST_OK : BEAST_E_NULL;
    cudaStream_t st = (cudaStream_t)stream;
    if (phase == 0) {
        if (!minmax) return BEAST_E_NULL;
        bpe_minmax_kernel<<<bpe_grid(n, 256), 256, 0, st>>>((const long long*)bins, n, (long long*)minmax,
                                                           (long long*)minmax + 1);
    } else {
        if (!seen || !err) return BEAST_E_NULL;
        bpe_seen_kernel<<<bpe_grid(n, 256), 256, 0, st>>>((const long long*)bins, n, min_token, seen, err);
    }
    count_launch();
    BEAST_CHECK_LAUNCH();
    return BEAST_OK;
}

extern "C" int bpe_symbolize(const int64_t* bins, int64_t N, int32_t L, int64_t min_token, const int16_t* byte_to_id,
                             const uint8_t* cls_tab, uint16_t* sym, int32_t* len, int64_t n_stride, int32_t* err,
                             const int32_t* row_len, void* stream) {
    if (N == 0) return BEAST_OK;
    if (!bins || !byte_to_id || !cls_tab || !sym || !len || !err) return BEAST_E_NULL;
    if (N < 0 || L < 1 || n_stride < N || 3 * L > 32767) return BEAST_E_SHAPE;
    const int rows = stage_rows_per_block(L);
    if (rows < 1) return BEAST_E_UNSUPPORTED;
    const size_t smem = stage_smem(L, rows);
    static size_t granted[kMaxDevices] = {};
    if (int rc = opt_in_smem(bpe_symbolize_kernel, smem, granted)) return rc;
    const long long grid = (N + rows - 1) / rows;
    bpe_symbolize_kernel<<<(unsigned)grid, kBpeBlock, smem, (cudaStream_t)stream>>>(
        (const long long*)bins, N, L, min_token, byte_to_id, cls_tab, sym, len, n_stride, err, rows, row_len);
    count_launch();
    BEAST_CHECK_LAUNCH();
    return BEAST_OK;
}

extern "C" int bpe_count_pairs(const uint16_t* sym, const int32_t* len, int64_t N, int64_t n_stride, int32_t V,
                               int32_t n_ids, const int16_t* used_ids, int32_t n_used, int32_t* hist,
                               const int32_t* weight, void* stream) {
    if (N == 0) return BEAST_OK;
    if (!sym || !len || !hist) return BEAST_E_NULL;
    if (N < 0 || V < 1 || V > 32767 || n_ids < 0 || n_ids > V || n_used < 0 || n_used > n_ids) return BEAST_E_SHAPE;
    if (used_ids && n_used > 0 && ((uintptr_t)sym & 15u) == 0) {
        const size_t map = ((size_t)n_ids * 2 + 15) & ~(size_t)15;
        int parts = 1;
        auto bytes = [&](int p) { return (size_t)((n_used + p - 1) / p) * n_used * sizeof(int) + map; };
        while (parts < 8 && bytes(parts) > 200 * 1024) ++parts;
        if (bytes(parts) <= 200 * 1024) {
            const size_t smem = bytes(parts);
            static size_t granted[kMaxDevices] = {};
            if (int rc = opt_in_smem(bpe_count_smem_kernel, smem, granted)) return rc;
            int dev = 0, sms = 148;
            cudaGetDevice(&dev);
            cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
            long long groups = (N + 1023) / 1024;
            if (groups > sms / parts) groups = sms / parts;
            if (groups < 1) groups = 1;
            bpe_count_smem_kernel<<<(unsigned)(groups * parts), 1024, smem, (cudaStream_t)stream>>>(
                sym, len, N, n_stride, V, n_ids, used_ids, n_used, parts, hist, weight);
            count_launch();
            BEAST_CHECK_LAUNCH();
            return BEAST_OK;
        }
    }
    bpe_count_kernel<<<bpe_grid(N, 256), 256, 0, (cudaStream_t)stream>>>(sym, len, N, n_stride, V, hist, weight);
    count_launch();
    BEAST_CHECK_LAUNCH();
    return BEAST_OK;
}

extern "C" int bpe_argmax(const int32_t* hist, int32_t V, int32_t n_active, uint64_t* result, void* stream) {
    if (!hist || !result) return BEAST_E_NULL;
    if (V < 1 || n_active < 1 || n_active > V || (long long)V * V > 0xffffffffLL) return BEAST_E_SHAPE;
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaMemsetAsync(result, 0, sizeof(uint64_t), st);
    if (e != cudaSuccess) return (int)e;
    bpe_argmax_kernel<<<bpe_grid((long long)n_active * n_active, 256 * 4), 256, 0, st>>>(
        hist, V, n_active, nullptr, (unsigned long long*)result);
    count_launch();
    BEAST_CHECK_LAUNCH();
    return BEAST_OK;
}

static int merge_grid(long long n) {
    static int sms = 0;
    if (!sms) { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev); }
    long long grid = (n + 255) / 256;
    const long long cap = (long long)sms * 8;
    if (grid > cap) grid = cap;
    return grid < 1 ? 1 : (int)grid;
}

static int rewrite_smem_attr(size_t smem) {
    if (smem > 200 * 1024) return BEAST_OK;               // launched without block-private counters (V passed negated)
    static size_t granted[kMaxDevices] = {};
    return opt_in_smem(bpe_rewrite_kernel, smem, granted);
}

extern "C" int bpe_apply_merge(uint16_t* sym, int32_t* len, int64_t N, int64_t n_stride, int32_t a, int32_t b,
                               int32_t c, int32_t V, int32_t* delta, int32_t* work, const int32_t* weight,
                               void* stream) {
    if (!delta || !work) return BEAST_E_NULL;
    if (V < 1 || a < 0 || b < 0 || c < 0 || a >= V || b >= V || c >= V || c > 32766) return BEAST_E_SHAPE;
    if (N == 0) return BEAST_OK;
    if (!sym || !len) return BEAST_E_NULL;
    const size_t smem = (size_t)4 * V * sizeof(int);
    int rc = rewrite_smem_attr(smem);
    if (rc != BEAST_OK) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    int* work_count = work;                  // work = {count, pad[3], seq[N], q0[N]}
    int* work_seq = work + 4;
    int* work_q0 = work + 4 + N;
    cudaError_t e = cudaMemsetAsync(work_count, 0, sizeof(int), st);
    if (e != cudaSuccess) return (int)e;
    const int grid = merge_grid(N);
    bpe_scan_kernel<<<grid, 256, 0, st>>>(sym, len, N, n_stride, a, b, work_count, work_seq, work_q0);
    const bool big_v = smem > 200 * 1024;                  // no room for block-private counters: global reductions only
    bpe_rewrite_kernel<<<grid, 256, big_v ? 0 : smem, st>>>(sym, len, n_stride, a, b, c, big_v ? -V : V, nullptr, work_count, work_seq,
                                                            work_q0, delta, nullptr, weight);
    count_launch(2);
    BEAST_CHECK_LAUNCH();
    return BEAST_OK;
}

extern "C" int bpe_apply_delta(int32_t* hist, int32_t* delta, int32_t a, int32_t b, int32_t c, int32_t V, void* stream) {
    if (!hist || !delta) return BEAST_E_NULL;
    if (V < 1 || a < 0 || b < 0 || c < 0 || a >= V || b >= V || c >= V) return BEAST_E_SHAPE;
    bpe_apply_delta_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(hist, delta, a, b, c, V, nullptr);
    count_launch();
    BEAST_CHECK_LAUNCH();
    return BEAST_OK;
}

extern "C" int32_t bpe_signature_words(void) { return kSigWords; }

extern "C" int bpe_build_signatures(const uint16_t* sym, const int32_t* len, int64_t N, int64_t n_stride, uint32_t* sig,
                                    void* stream) {
    if (N == 0) return BEAST_OK;
    if (!sym || !len || !sig) return BEAST_E_NULL;
    if (N < 0 || n_stride < N) return BEAST_E_SHAPE;
    if ((uintptr_t)sym & 15u) return BEAST_E_ALIGN;
    bpe_signature_kernel<<<bpe_grid(N, kSigBlock), kSigBlock, 0, (cudaStream_t)stream>>>(sym, len, N, n_stride, sig);
    count_launch();
    BEAST_CHECK_LAUNCH();
    return BEAST_OK;
}

// `iters` iterations of the sync-free training loop, each THREE launches: the iteration head (arg-max + fold of the
// previous merge's delta, summed over the peers' blocks when sharded), pick + scan (work list), rewrite (fills
// delta[merge & 1]).  The control block is double-buffered by iteration parity (first_iter = index of the first
// iteration of this call): iteration i reads ctl[i & 1] and writes ctl[(i + 1) & 1].  The caller enqueues up to
// (vocab_size - alphabet) iterations without reading anything back; ctl / log are read once at the end.
extern "C" int bpe_train_step(uint16_t* sym, int32_t* len, int64_t N, int64_t n_stride, int32_t V, int32_t* hist,
                              int32_t* delta, void* ctl, int32_t* log, uint64_t* result, int32_t* work,
                              int32_t vocab_size, int32_t min_frequency, int32_t max_merges, uint32_t* sig,
                              int32_t first_iter, int32_t iters, const bpe_peers_t* peers_h, const int32_t* weight,
                              void* stream) {
    if (!hist || !delta || !ctl || !log || !result || !work) return BEAST_E_NULL;
    if (N > 0 && (!sym || !len)) return BEAST_E_NULL;
    if (V < 1 || V > 32767 || (long long)V * V > 0xffffffffLL || first_iter < 0) return BEAST_E_SHAPE;
    if (((uintptr_t)delta & 15u) || ((uintptr_t)ctl & 15u)) return BEAST_E_ALIGN;
    cudaStream_t st = (cudaStream_t)stream;
    const size_t smem = (size_t)4 * V * sizeof(int);
    int rc = rewrite_smem_attr(smem);
    if (rc != BEAST_OK) return rc;
    static int sms = 0;
    if (!sms) { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev); }
    BpePeersDev peers;
    memset(&peers, 0, sizeof(peers));
    peers.world = 1;
    int n_part = sms < 256 ? sms : 256;                       // `result` holds 256 words
    if (peers_h && peers_h->world > 1) {
        if (peers_h->world > BPE_MAX_PEERS || peers_h->rank < 0 || peers_h->rank >= peers_h->world) return BEAST_E_SHAPE;
        peers.world = peers_h->world; peers.rank = peers_h->rank; peers.epoch_base = peers_h->epoch_base;
        for (int r = 0; r < peers.world; ++r) {
            if (!peers_h->delta[r] || !peers_h->flags[r]) return BEAST_E_NULL;
            peers.delta[r] = peers_h->delta[r];
            peers.flags[r] = peers_h->flags[r];
        }
        if (peers.delta[peers.rank] != delta) return BEAST_E_SHAPE;
    }
    if (peers_h && peers_h->grid_blocks > 0 && peers_h->grid_blocks < n_part) n_part = peers_h->grid_blocks;
    int* work_count = work;                  // work = {count, pad[3], seq[N], q0[N]}
    int* work_seq = work + 4;
    int* work_q0 = work + 4 + N;
    // tile of the signature scan: large enough to fill warps with survivors, small enough to use every SM
    // (a multiple of the block size, so every thread takes part in the ballots)
    long long tile = ((N / ((long long)sms * 2) + 255) / 256) * 256;
    if (tile < 256) tile = 256;
    if (tile > kScanTile) tile = kScanTile;
    const int grid = merge_grid(N > 0 ? N : 1);
    // small shards are latency-bound (few tiles per SM): walk the survivors with four loads in flight; large
    // ones are better off with two (measured: 65 k sequences 0.056 -> 0.053 s, 1.6 M sequences 0.214 -> 0.228 s)
    const bool deep_walk = N <= (1 << 19);
    BpeCtl* ctl2 = (BpeCtl*)ctl;
    static int use_pdl = -1;
    if (use_pdl < 0) { const char* e = getenv("BEAST_B200_BPE_NO_PDL"); use_pdl = (e && e[0] == '1') ? 0 : 1; }
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    auto config = [&](unsigned g, unsigned b, size_t sm) {
        cudaLaunchConfig_t c;
        memset(&c, 0, sizeof(c));
        c.gridDim = dim3(g); c.blockDim = dim3(b); c.dynamicSmemBytes = sm; c.stream = st;
        c.attrs = attr; c.numAttrs = use_pdl ? 1 : 0;
        return c;
    };
    // BEAST_B200_BPE_LOOP=persistent: the whole block of iterations in ONE cooperative kernel, grid barriers instead of
    // kernel boundaries.  Measured SLOWER than the PDL-chained launches (200 k-sequence shard 62.6 vs 40.2 ms, 12 000
    // pseudo-sequences 54.3 vs 31.3 ms: three grid barriers of a 148 x 1024-thread grid cost more than three
    // programmatic launch boundaries), so it is opt-in; kept because it is the same device code and is tested.
    const char* loop_env = getenv("BEAST_B200_BPE_LOOP");      // re-read per call: the tests run both forms in one process
    const int loop_mode = (loop_env && loop_env[0] == 'p') ? 1 : 0;
    const size_t loop_smem = (size_t)64 * V + (size_t)4 * 8 * kRewriteOut * sizeof(uint16_t);
    if (loop_mode == 1 && loop_smem <= 176 * 1024) {
        static size_t granted_ld[kMaxDevices] = {}, granted_lf[kMaxDevices] = {};
        int rc2 = deep_walk ? opt_in_smem(bpe_loop_kernel<true>, loop_smem, granted_ld) : opt_in_smem(bpe_loop_kernel<false>, loop_smem, granted_lf);
        int per_sm = 0, coop = 0, dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev);
        if (rc2 == BEAST_OK) {
            if (deep_walk) cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, bpe_loop_kernel<true>, 1024, loop_smem);
            else cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, bpe_loop_kernel<false>, 1024, loop_smem);
        }
        if (rc2 == BEAST_OK && coop && per_sm >= 1) {
            LoopArgs la;
            la.sym = sym; la.len = len; la.N = N; la.n_stride = n_stride; la.V = V;
            la.hist = hist; la.delta = delta; la.ctl = ctl2; la.log = log; la.partial = (unsigned long long*)result;
            la.work_count = work_count; la.work_seq = work_seq; la.work_q0 = work_q0;
            la.vocab_size = vocab_size; la.min_frequency = min_frequency; la.max_merges = max_merges;
            la.sig = sig; la.weight = weight; la.tile_size = (int)tile; la.first_iter = first_iter; la.iters = iters < 1 ? 1 : iters;
            void* args[2] = {&la, &peers};
            const void* fn = deep_walk ? (const void*)bpe_loop_kernel<true> : (const void*)bpe_loop_kernel<false>;
            cudaError_t e = cudaLaunchCooperativeKernel(fn, dim3((unsigned)n_part), dim3(1024), args, loop_smem, st);
            if (e != cudaSuccess) return (int)e;
            count_launch();
            return BEAST_OK;
        }
    }
    const unsigned long long* partial = (const unsigned long long*)result;
    const uint16_t* csym = sym;
    const int32_t* clen = len;
    const unsigned int* csig = sig;
    const int tile_i = (int)tile;
    for (int it = 0; it < (iters < 1 ? 1 : iters); ++it) {
        const int i = first_iter + it;
        BpeCtl* cin = ctl2 + (i & 1);
        BpeCtl* cout = ctl2 + ((i + 1) & 1);
        const BpeCtl* ccin = cin;
        const BpeCtl* ccout = cout;
        cudaLaunchConfig_t c1 = config((unsigned)n_part, 1024, 0);
        cudaError_t e = cudaLaunchKernelEx(&c1, bpe_iterate_kernel, hist, V, cin, delta, (unsigned long long*)result, work_count, peers);
        if (e != cudaSuccess) return (int)e;
        cudaLaunchConfig_t c2 = config((unsigned)grid, 256, 0);
        if (deep_walk)
            e = cudaLaunchKernelEx(&c2, bpe_pick_scan_kernel<true>, csym, clen, (long long)N, (long long)n_stride, V, ccin, cout, partial,
                                   n_part, log, vocab_size, min_frequency, max_merges, work_count, work_seq, work_q0, csig, tile_i);
        else
            e = cudaLaunchKernelEx(&c2, bpe_pick_scan_kernel<false>, csym, clen, (long long)N, (long long)n_stride, V, ccin, cout, partial,
                                   n_part, log, vocab_size, min_frequency, max_merges, work_count, work_seq, work_q0, csig, tile_i);
        if (e != cudaSuccess) return (int)e;
        count_launch(2);
        if (N > 0) {
            const bool big_v = smem > 200 * 1024;          // no room for block-private counters: global reductions only
            cudaLaunchConfig_t c3 = config((unsigned)grid, 256, big_v ? 0 : smem);
            const int v_arg = big_v ? -V : V;
            const int* cwc = work_count;
            const int* cws = work_seq;
            const int* cwq = work_q0;
            e = cudaLaunchKernelEx(&c3, bpe_rewrite_kernel, sym, len, (long long)n_stride, 0, 0, 0, v_arg, ccout, cwc, cws, cwq, delta, sig, weight);
            if (e != cudaSuccess) return (int)e;
            count_launch();
        }
    }
    BEAST_CHECK_LAUNCH();
    return BEAST_OK;
}

// Peer-visible device memory (CUDA IPC) for the sharded trainer's delta blocks and flags.
extern "C" int beast_peer_alloc(int64_t bytes, void** ptr_out, void* handle_out_h) {
    if (!ptr_out || !handle_out_h) return BEAST_E_NULL;
    if (bytes < 1) return BEAST_E_SHAPE;
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size is part of the C ABI");
    void* p = nullptr;
    cudaError_t e = cudaMalloc(&p, (size_t)bytes);
    if (e != cudaSuccess) return (int)e;
    e = cudaMemset(p, 0, (size_t)bytes);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    cudaIpcMemHandle_t h;
    if (e == cudaSuccess) e = cudaIpcGetMemHandle(&h, p);
    if (e != cudaSuccess) { cudaFree(p); cudaGetLastError(); return (int)e; }
    memcpy(handle_out_h, &h, sizeof(h));
    *ptr_out = p;
    return BEAST_OK;
}
extern "C" int beast_peer_open(const void* handle_h, void** ptr_out) {
    if (!handle_h || !ptr_out) return BEAST_E_NULL;
    cudaIpcMemHandle_t h;
    memcpy(&h, handle_h, sizeof(h));
    void* p = nullptr;
    cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) { cudaGetLastError(); return (int)e; }
    *ptr_out = p;
    return BEAST_OK;
}
extern "C" int beast_peer_close(void* ptr) {
    if (!ptr) return BEAST_E_NULL;
    cudaError_t e = cudaIpcCloseMemHandle(ptr);
    if (e != cudaSuccess) { cudaGetLastError(); return (int)e; }
    return BEAST_OK;
}
extern "C" int beast_peer_free(void* ptr) {
    if (!ptr) return BEAST_E_NULL;
    cudaError_t e = cudaFree(ptr);
    if (e != cudaSuccess) { cudaGetLastError(); return (int)e; }
    return BEAST_OK;
}

extern "C" int bpe_encode(const int64_t* bins, int64_t N, int32_t L, int64_t min_token, int64_t max_shift,
                          const int16_t* byte_to_id, const uint8_t* cls_tab, const uint32_t* rank_tab, int32_t V,
                          int32_t hash_bits, uint16_t* ids_padded, int32_t out_stride, int32_t* len_out,
                          int32_t* status_out, void* stream) {
    if (N == 0) return BEAST_OK;
    if (!bins || !byte_to_id || !cls_tab || !rank_tab || !ids_padded || !len_out || !status_out) return BEAST_E_NULL;
    const int mult = max_shift < 0x80 ? 1 : (max_shift < 0x800 ? 2 : 3);       // UTF-8 bytes per bin
    if (N < 0 || L < 1 || mult * L > kMaxWordLong || out_stride < mult * L || V < 1 || V > 65535 || max_shift > 0xD7FF ||
        hash_bits < 0 || hash_bits > 30 || ((uintptr_t)rank_tab & 7u))
        return BEAST_E_SHAPE;
    const int M = mult * L;
    if (M > 65535) return BEAST_E_SHAPE;
    // one warp per sequence, working arrays in shared memory; sequences too long for that (or
    // BEAST_B200_BPE_THREAD_ENCODE=1) take the one-thread-per-sequence kernel
    const size_t key2_off = ((size_t)8 * M + 2 * (size_t)((L + 1) & ~1) + 2 * (size_t)(L + 2) + 3) & ~(size_t)3;
    const size_t warp_bytes = (key2_off + (size_t)4 * M + 15) & ~(size_t)15;
    int warps = (int)((200 * 1024) / warp_bytes);
    if (warps > 8) warps = 8;
    // test hook, re-read per call (the tests toggle it): one getenv is noise next to a launch
    const char* env = getenv("BEAST_B200_BPE_THREAD_ENCODE");
    if (warps >= 1 && !(env && env[0] == '1')) {
        const size_t smem = warp_bytes * warps;
        static size_t granted[kMaxDevices] = {};
        if (int rc = opt_in_smem(bpe_encode_warp_kernel, smem, granted)) return rc;
        int dev = 0, sms = 148;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        long long per_sm = (long long)(220 * 1024) / (long long)(smem + 1024);
        if (per_sm > 2048 / (warps * 32)) per_sm = 2048 / (warps * 32);
        if (per_sm < 1) per_sm = 1;
        long long grid = (N + warps - 1) / warps;
        if (grid > sms * per_sm) grid = sms * per_sm;
        bpe_encode_warp_kernel<<<(unsigned)grid, warps * 32, smem, (cudaStream_t)stream>>>(
            (const long long*)bins, N, L, min_token, max_shift, byte_to_id, cls_tab, rank_tab, V, ids_padded, out_stride,
            len_out, status_out, M, (int)warp_bytes, (int)key2_off, hash_bits);
        count_launch();
        BEAST_CHECK_LAUNCH();
        return BEAST_OK;
    }
    const int rows = stage_rows_per_block(L);
    if (rows < 1) return BEAST_E_UNSUPPORTED;
    const size_t smem = stage_smem(L, rows);
    static size_t granted[kMaxDevices] = {};
    if (int rc = opt_in_smem(bpe_encode_kernel<kMaxWordLong, uint16_t>, smem, granted)) return rc;
    const long long grid = (N + rows - 1) / rows;
    bpe_encode_kernel<kMaxWordLong, uint16_t><<<(unsigned)grid, kBpeBlock, smem, (cudaStream_t)stream>>>(
        (const long long*)bins, N, L, min_token, max_shift, byte_to_id, cls_tab, rank_tab, V, ids_padded, out_stride,
        len_out, status_out, rows, hash_bits);
    count_launch();
    BEAST_CHECK_LAUNCH();
    return BEAST_OK;
}

extern "C" int bpe_compact(const uint16_t* ids_padded, int32_t stride, const int32_t* len, const int64_t* offsets,
                           int64_t N, int32_t* flat, void* stream) {
    if (N == 0) return BEAST_OK;
    if (!ids_padded || !len || !offsets || !flat) return BEAST_E_NULL;
    bpe_compact_kernel<<<bpe_grid(N, 8), 256, 0, (cudaStream_t)stream>>>(ids_padded, stride, len,
                                                                        (const long long*)offsets, N, flat);
    count_launch();
    BEAST_CHECK_LAUNCH();
    return BEAST_OK;
}

extern "C" int bpe_decode(const int32_t* flat, const int64_t* offsets, int64_t N, int32_t L, int64_t min_token,
                          const int32_t* tok_off, const uint8_t* tok_bytes, const void* tok_tab, int32_t tok_tab_slots,
                          int32_t n_vocab, int64_t* bins_out, int32_t* status_out, int32_t* declen_out, void* stream) {
    if (N == 0) return BEAST_OK;
    if (!offsets || !tok_off || !tok_bytes || !bins_out || !status_out || !declen_out) return BEAST_E_NULL;
    if (N < 0 || L < 1 || n_vocab < 1) return BEAST_E_SHAPE;
    if (tok_tab && tok_tab_slots != 2 && tok_tab_slots != 6) return BEAST_E_SHAPE;
    if ((uintptr_t)tok_tab & 15u) return BEAST_E_ALIGN;
    cudaStream_t st = (cudaStream_t)stream;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    // test hook, re-read per call (the tests toggle it between calls): one getenv is noise next to a launch
    const char* env_thread = getenv("BEAST_B200_BPE_THREAD_DECODE");
    const int force_thread = (env_thread && env_thread[0] == '1') ? 1 : 0;
    int only_flagged = 0;
    if (tok_tab && !force_thread && L <= 8192) {
        // fast path: one lane per token from the per-token character table; sequences it cannot describe are flagged
        const size_t smem = (size_t)8 * (((size_t)L + 7) & ~(size_t)7) * 2;
        static size_t granted2[kMaxDevices] = {}, granted6[kMaxDevices] = {};
        int rc = tok_tab_slots == 2 ? opt_in_smem(bpe_decode_token_kernel<2>, smem, granted2)
                                    : opt_in_smem(bpe_decode_token_kernel<6>, smem, granted6);
        if (rc) return rc;
        long long grid = (N + 7) / 8;
        if (grid > (long long)sms * 8) grid = (long long)sms * 8;
        if (tok_tab_slots == 2)
            bpe_decode_token_kernel<2><<<(unsigned)grid, 256, smem, st>>>(flat, (const long long*)offsets, N, L, min_token, tok_tab,
                                                                         n_vocab, (long long*)bins_out, status_out, declen_out);
        else
            bpe_decode_token_kernel<6><<<(unsigned)grid, 256, smem, st>>>(flat, (const long long*)offsets, N, L, min_token, tok_tab,
                                                                         n_vocab, (long long*)bins_out, status_out, declen_out);
        count_launch();
        BEAST_CHECK_LAUNCH();
        only_flagged = 1;
    }
    {   // byte-level path, one warp per sequence (all sequences, or only the ones the fast kernel flagged);
        // BEAST_B200_BPE_THREAD_DECODE=1 (or rows too long for shared memory) takes the one-thread-per-sequence kernel
        const int cap = 4 * L + 64;                          // a valid sequence has at most 3 L bytes
        const size_t warp_bytes = (((size_t)cap + 15) & ~(size_t)15) + (((size_t)L * 2 + 15) & ~(size_t)15);
        int warps = (int)((200 * 1024) / warp_bytes);
        if (warps > 8) warps = 8;
        if (warps >= 1 && !force_thread) {
            const size_t smem = warp_bytes * warps;
            static size_t granted_w[kMaxDevices] = {};
            if (int rc = opt_in_smem(bpe_decode_warp_kernel, smem, granted_w)) return rc;
            long long per_sm = (long long)(220 * 1024) / (long long)(smem + 1024);
            if (per_sm > 2048 / (warps * 32)) per_sm = 2048 / (warps * 32);
            if (per_sm < 1) per_sm = 1;
            long long grid = (N + warps - 1) / warps;
            if (grid > sms * per_sm) grid = sms * per_sm;
            bpe_decode_warp_kernel<<<(unsigned)grid, warps * 32, smem, st>>>(
                flat, (const long long*)offsets, N, L, min_token, tok_off, tok_bytes, n_vocab, (long long*)bins_out,
                status_out, declen_out, cap, (int)warp_bytes, only_flagged);
            count_launch();
            BEAST_CHECK_LAUNCH();
            return BEAST_OK;
        }
    }
    const int rows = stage_rows_per_block(L);
    if (rows < 1) return BEAST_E_UNSUPPORTED;
    const size_t smem = (size_t)rows * (L + 1) * 2;
    static size_t granted[kMaxDevices] = {};
    if (int rc = opt_in_smem(bpe_decode_kernel, smem, granted)) return rc;
    const long long grid = (N + rows - 1) / rows;
    bpe_decode_kernel<<<(unsigned)grid, kBpeBlock, smem, st>>>(
        flat, (const long long*)offsets, N, L, min_token, tok_off, tok_bytes, n_vocab, (long long*)bins_out, status_out,
        declen_out, rows);
    count_launch();
    BEAST_CHECK_LAUNCH();
    return BEAST_OK;
}
