// Plan: immutable per-tokenizer constants (geometry, projector / basis tables) on host and device.
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <new>
#include "common.cuh"

namespace beast {
long long g_launch_count = 0;
int g_disable_fast = -1;
int g_force_wait = 0;

bool ranges_conflict(const LaunchRanges& prev, const LaunchRanges& next) {
    for (int i = 0; i < prev.n; ++i)
        for (int j = 0; j < next.n; ++j) {
            const MemRange &p = prev.r[i], &q = next.r[j];
            if ((p.write || q.write) && p.lo < q.hi && q.lo < p.hi && p.lo < p.hi && q.lo < q.hi) return true;
        }
    return false;
}

namespace {
// The last bulk-copy K1 / K3 launch captured on a (device, stream): its capture sequence, its node and its ranges.
struct LaunchRecord {
    unsigned long long capture_id;
    cudaGraphNode_t node;
    LaunchRanges ranges;
};
std::mutex g_record_mutex;
std::map<std::pair<int, cudaStream_t>, LaunchRecord> g_records;
long long g_overlap_count = 0;

// The dependency set the next node captured on `st` gets, when it is exactly one node over a plain edge.
bool single_capture_dependency(cudaStream_t st, unsigned long long* id, cudaGraphNode_t* node) {
    cudaStreamCaptureStatus status = cudaStreamCaptureStatusNone;
    const cudaGraphNode_t* deps = nullptr;
    const cudaGraphEdgeData* edges = nullptr;
    size_t n = 0;
    if (cudaStreamGetCaptureInfo_v3(st, &status, id, nullptr, &deps, &edges, &n) != cudaSuccess) {
        cudaGetLastError();                      // the launch that follows reports any real stream error itself
        return false;
    }
    if (status != cudaStreamCaptureStatusActive || n != 1) return false;
    if (edges && (edges[0].type != cudaGraphDependencyTypeDefault || edges[0].from_port != 0 || edges[0].to_port != 0))
        return false;
    *node = deps[0];
    return true;
}
}  // namespace

bool overlap_begin(cudaStream_t st, const LaunchRanges& mine) {
    if (g_force_wait) return false;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return false;
    unsigned long long id = 0;
    cudaGraphNode_t dep = nullptr;
    if (!single_capture_dependency(st, &id, &dep)) return false;
    std::lock_guard<std::mutex> lock(g_record_mutex);
    auto it = g_records.find({dev, st});
    return it != g_records.end() && it->second.capture_id == id && it->second.node == dep &&
           !ranges_conflict(it->second.ranges, mine);
}

void overlap_end(cudaStream_t st, const LaunchRanges& mine, bool overlapped, cudaError_t launch_error) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return;
    unsigned long long id = 0;
    cudaGraphNode_t node = nullptr;
    const bool captured = launch_error == cudaSuccess && single_capture_dependency(st, &id, &node);
    std::lock_guard<std::mutex> lock(g_record_mutex);
    if (captured) g_records[{dev, st}] = LaunchRecord{id, node, mine};
    else g_records.erase({dev, st});
    if (overlapped && launch_error == cudaSuccess) ++g_overlap_count;
}
}  // namespace beast
using beast::Plan;

static float* dup_h(const float* src, size_t n) {
    if (!src) return nullptr;
    float* p = (float*)malloc(n * sizeof(float));
    if (p) memcpy(p, src, n * sizeof(float));
    return p;
}

extern "C" const char* beast_version(void) { return "beast_b200 0.1 sm_100a"; }
extern "C" int64_t beast_launch_count(void) { return beast::g_launch_count; }
extern "C" int beast_debug_disable_fast(int32_t flag) {
    const int prev = beast::g_disable_fast == 1 ? 1 : 0;
    beast::g_disable_fast = flag ? 1 : 0;
    return prev;
}
extern "C" int64_t beast_overlap_count(void) {
    std::lock_guard<std::mutex> lock(beast::g_record_mutex);
    return beast::g_overlap_count;
}
extern "C" int beast_debug_force_wait(int32_t flag) {
    const int prev = beast::g_force_wait;
    beast::g_force_wait = flag ? 1 : 0;
    return prev;
}
extern "C" int beast_debug_ranges_conflict(const int64_t* prev, int32_t n_prev, const int64_t* next, int32_t n_next) {
    if (n_prev < 0 || n_next < 0 || n_prev > beast::LaunchRanges::kMax || n_next > beast::LaunchRanges::kMax) return BEAST_E_SHAPE;
    if ((n_prev && !prev) || (n_next && !next)) return BEAST_E_NULL;
    beast::LaunchRanges a, b;
    for (int i = 0; i < n_prev; ++i) a.r[a.n++] = beast::MemRange{(uintptr_t)prev[3 * i], (uintptr_t)prev[3 * i + 1], prev[3 * i + 2] ? 1 : 0};
    for (int i = 0; i < n_next; ++i) b.r[b.n++] = beast::MemRange{(uintptr_t)next[3 * i], (uintptr_t)next[3 * i + 1], next[3 * i + 2] ? 1 : 0};
    return beast::ranges_conflict(a, b) ? 1 : 0;
}

extern "C" int beast_plan_create(const beast_plan_desc_t* d, beast_plan_t** out) {
    if (!d || !out) return BEAST_E_NULL;
    *out = nullptr;
    if (d->seq_len < 1 || d->num_basis < 1 || d->num_dof < 1 || d->num_dof > BEAST_MAX_DOF) return BEAST_E_SHAPE;
    if (d->n_joint < 0 || d->n_joint > d->num_dof || d->vocab_size < 2 || d->degree_p < 0) return BEAST_E_SHAPE;
    if (d->init_cond_order < 0 || d->init_cond_order > 2 || d->end_cond_order < 0 || d->end_cond_order > 2)
        return BEAST_E_UNSUPPORTED;
    if (!d->slot_to_dof_h || !d->proj_joint_h || !d->phi_joint_h || !d->knots_joint_h) return BEAST_E_NULL;
    const bool has_grip = d->n_joint < d->num_dof;
    if (has_grip && (!d->proj_grip_h || !d->phi_grip_h || !d->knots_grip_h)) return BEAST_E_NULL;
    for (int i = 0; i < d->num_dof; ++i)
        if (d->slot_to_dof_h[i] < 0 || d->slot_to_dof_h[i] >= d->num_dof) return BEAST_E_SHAPE;

    Plan* p = new (std::nothrow) Plan();
    if (!p) return BEAST_E_NOMEM;
    memset(p, 0, sizeof(Plan));
    p->T = d->seq_len; p->D = d->num_dof; p->nb = d->num_basis; p->n_joint = d->n_joint;
    p->degree_p = d->degree_p; p->V = d->vocab_size; p->tau = d->tau;
    p->ico = d->init_cond_order; p->eco = d->end_cond_order; p->nc = p->nb + p->ico + p->eco;
    for (int i = 0; i < p->D; ++i) p->slot_to_dof[i] = d->slot_to_dof_h[i];
    const size_t nt = (size_t)p->nb * p->T, ntc = (size_t)p->nc * p->T;
    const size_t nkj = (size_t)p->nc + p->degree_p + 1, nkg = (size_t)p->nb + 1;
    p->proj_joint_h = dup_h(d->proj_joint_h, nt);
    p->phi_joint_h = dup_h(d->phi_joint_h, ntc);
    p->proj_grip_h = has_grip ? dup_h(d->proj_grip_h, nt) : nullptr;
    p->phi_grip_h = has_grip ? dup_h(d->phi_grip_h, nt) : nullptr;

    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&p->num_sms, cudaDevAttrMultiProcessorCount, dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&p->max_smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    // one device block: 4 tables + 2 knot vectors + slot map (all 4-byte elements)
    const size_t total = 3 * nt + ntc + nkj + nkg + BEAST_MAX_SLOTS;
    if (e == cudaSuccess) e = cudaMalloc((void**)&p->dev_block, total * sizeof(float));
    if (e != cudaSuccess) { beast_plan_destroy((beast_plan_t*)p); return (int)e; }
    float* host = (float*)calloc(total, sizeof(float));
    if (!host) { beast_plan_destroy((beast_plan_t*)p); return BEAST_E_NOMEM; }
    size_t off = 0;
    auto put = [&](const float* src, size_t n, float** dptr) {
        if (src) memcpy(host + off, src, n * sizeof(float));
        *dptr = p->dev_block + off;
        off += n;
    };
    put(d->proj_joint_h, nt, &p->proj_joint_d);
    put(has_grip ? d->proj_grip_h : nullptr, nt, &p->proj_grip_d);
    put(d->phi_joint_h, ntc, &p->phi_joint_d);
    put(has_grip ? d->phi_grip_h : nullptr, nt, &p->phi_grip_d);
    put(d->knots_joint_h, nkj, &p->knots_joint_d);
    put(has_grip ? d->knots_grip_h : nullptr, nkg, &p->knots_grip_d);
    memcpy(host + off, p->slot_to_dof, BEAST_MAX_SLOTS * sizeof(int));
    p->slot_to_dof_d = (int*)(p->dev_block + off);
    e = cudaMemcpy(p->dev_block, host, total * sizeof(float), cudaMemcpyHostToDevice);
    free(host);
    if (e != cudaSuccess) { beast_plan_destroy((beast_plan_t*)p); return (int)e; }
    {   // band tables: non-zero range of every projector row [k][t], of every basis row [t][k] and of every projector
        // column
        const int T = p->T, nb = p->nb;
        const size_t n_band = (size_t)4 * nb + (size_t)8 * T;
        int* bands = (int*)calloc(n_band, sizeof(int));
        if (!bands) { beast_plan_destroy((beast_plan_t*)p); return BEAST_E_NOMEM; }
        auto row_band = [](const float* row, int n, int stride, int* lo_hi) {
            int lo = n, hi = 0;
            for (int i = 0; i < n; ++i)
                if (row[(size_t)i * stride] != 0.0f) { if (i < lo) lo = i; hi = i + 1; }
            if (lo >= hi) lo = hi = 0;
            lo_hi[0] = lo; lo_hi[1] = hi;
        };
        for (int k = 0; k < nb; ++k) {
            row_band(p->proj_joint_h + (size_t)k * T, T, 1, bands + 2 * k);
            if (has_grip) row_band(p->proj_grip_h + (size_t)k * T, T, 1, bands + 2 * nb + 2 * k);
        }
        for (int t = 0; t < T; ++t) {
            if (p->nc == nb) row_band(p->phi_joint_h + (size_t)t * nb, nb, 1, bands + 4 * nb + 2 * t);
            if (has_grip) row_band(p->phi_grip_h + (size_t)t * nb, nb, 1, bands + 4 * nb + 2 * T + 2 * t);
            int* fit = bands + 4 * nb + 4 * T;
            row_band(p->proj_joint_h + t, nb, T, fit + 2 * t);
            if (has_grip) row_band(p->proj_grip_h + t, nb, T, fit + 2 * T + 2 * t);
            for (int s = 0; s < 2; ++s)
                if (fit[2 * (s * T + t) + 1] - fit[2 * (s * T + t)] > p->fit_band_max)
                    p->fit_band_max = fit[2 * (s * T + t) + 1] - fit[2 * (s * T + t)];
        }
        e = cudaMalloc((void**)&p->bands_d, n_band * sizeof(int));
        if (e == cudaSuccess) e = cudaMemcpy(p->bands_d, bands, n_band * sizeof(int), cudaMemcpyHostToDevice);
        // work lists of the tiled kernels (see Plan): non-empty projector rows / coefficients a basis row reads
        const int D = p->D, n_joint = p->n_joint;
        int* lists = nullptr;
        if (e == cudaSuccess && nb <= 0xffff && D <= 0x7fff) {
            lists = (int*)malloc((size_t)2 * D * nb * sizeof(int) + sizeof(int));
            char* used = (char*)calloc((size_t)2 * nb, 1);          // [joint | gripper][k]
            if (!lists || !used) { free(lists); free(used); free(bands); beast_plan_destroy((beast_plan_t*)p); return BEAST_E_NOMEM; }
            for (int t = 0; t < T; ++t) {
                for (int k = bands[4 * nb + 2 * t]; k < bands[4 * nb + 2 * t + 1]; ++k) used[k] = 1;
                for (int k = bands[4 * nb + 2 * T + 2 * t]; k < bands[4 * nb + 2 * T + 2 * t + 1]; ++k) used[nb + k] = 1;
            }
            for (int k = 0; k < 2 * nb; ++k)
                if (bands[2 * k + 1] - bands[2 * k] > p->enc_band_max) p->enc_band_max = bands[2 * k + 1] - bands[2 * k];
            for (int t = 0; t < 2 * T; ++t)
                if (bands[4 * nb + 2 * t + 1] - bands[4 * nb + 2 * t] > p->dec_band_max)
                    p->dec_band_max = bands[4 * nb + 2 * t + 1] - bands[4 * nb + 2 * t];
            int n_enc = 0, n_dec = 0;
            int* dec = lists + (size_t)D * nb;
            for (int k = 0; k < nb; ++k)
                for (int slot = 0; slot < D; ++slot) {
                    const bool grip = slot >= n_joint;
                    const int entry = k | (slot << 16) | (grip ? (int)0x80000000u : 0);
                    const int* b = bands + (grip ? 2 * nb : 0) + 2 * k;
                    if (b[0] < b[1]) lists[n_enc++] = entry;
                    if (used[(grip ? nb : 0) + k]) dec[n_dec++] = entry;
                }
            free(used);
            p->n_enc = n_enc; p->n_dec = n_dec;
            e = cudaMalloc((void**)&p->enc_list_d, ((size_t)n_enc + n_dec + 1) * sizeof(int));
            if (e == cudaSuccess && n_enc) e = cudaMemcpy(p->enc_list_d, lists, (size_t)n_enc * sizeof(int), cudaMemcpyHostToDevice);
            if (e == cudaSuccess) p->dec_list_d = p->enc_list_d + n_enc;
            if (e == cudaSuccess && n_dec) e = cudaMemcpy(p->dec_list_d, dec, (size_t)n_dec * sizeof(int), cudaMemcpyHostToDevice);
            free(lists);
        }
        free(bands);
        if (e != cudaSuccess) { beast_plan_destroy((beast_plan_t*)p); return (int)e; }
    }
    *out = (beast_plan_t*)p;
    return BEAST_OK;
}

extern "C" int beast_plan_destroy(beast_plan_t* plan) {
    if (!plan) return BEAST_OK;
    Plan* p = (Plan*)plan;
    free(p->proj_joint_h); free(p->proj_grip_h); free(p->phi_joint_h); free(p->phi_grip_h);
    if (p->dev_block) cudaFree(p->dev_block);
    if (p->bands_d) cudaFree(p->bands_d);
    if (p->enc_list_d) cudaFree(p->enc_list_d);
    delete p;
    return BEAST_OK;
}
