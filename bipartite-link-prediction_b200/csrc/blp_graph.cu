// Graph handle: de-duplicated bipartite adjacency as two padded CSR arrays resident in HBM.
// Replaces snap.LoadEdgeList / snap.Nodes / GetNI().GetDeg() of the reference
// (similarity.py:16, 22, 65, 121).
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstdio>
#include <map>
#include <mutex>
#include <tuple>
#include <vector>

#include "blp_internal.h"

namespace blp {
static thread_local std::string g_last_error;

void set_error(const std::string& msg) { g_last_error = msg; }

int cuda_fail(cudaError_t e, const char* what, const char* file, int line) {
    char buf[512];
    snprintf(buf, sizeof(buf), "CUDA error %d (%s) at %s:%d: %s", (int)e, cudaGetErrorString(e),
             file, line, what);
    g_last_error = buf;
    // clear the sticky-less error so that the next call starts clean
    (void)cudaGetLastError();
    return e == cudaErrorMemoryAllocation ? BLP_ERR_OOM : BLP_ERR_CUDA;
}

// Stream-ordered scratch (graph construction on the device, the per-call scratch of the scoring
// kernels) comes from ONE pool per device that the library owns and shares between its handles:
// its release threshold is the maximum, so repeated calls and repeated graph builds reuse the same
// memory instead of going back to the driver at every synchronisation.  The device's default pool
// keeps its settings.  When the last handle on a device is destroyed the pool is trimmed to zero,
// so nothing stays cached once the application is done with the library.
namespace {
constexpr int kPoolDevices = 64;
std::mutex g_pool_mutex;
cudaMemPool_t g_pool[kPoolDevices] = {};
int g_pool_refs[kPoolDevices] = {};
}  // namespace

cudaMemPool_t acquire_scratch_pool(int device) {
    if (device < 0 || device >= kPoolDevices) return nullptr;
    std::lock_guard<std::mutex> lock(g_pool_mutex);
    if (!g_pool[device]) {
        cudaMemPoolProps props = {};
        props.allocType = cudaMemAllocationTypePinned;
        props.handleTypes = cudaMemHandleTypeNone;
        props.location.type = cudaMemLocationTypeDevice;
        props.location.id = device;
        if (cudaMemPoolCreate(&g_pool[device], &props) != cudaSuccess) {
            (void)cudaGetLastError();
            g_pool[device] = nullptr;
            return nullptr;
        }
        uint64_t keep = UINT64_MAX;
        cudaMemPoolSetAttribute(g_pool[device], cudaMemPoolAttrReleaseThreshold, &keep);
    }
    ++g_pool_refs[device];
    return g_pool[device];
}

// stream-ordered allocation for code that has no handle at hand (sort, scan, evaluation): the
// library pool of the current device while some handle keeps it alive, else the default pool
cudaError_t scratch_alloc(void** p, size_t bytes, cudaStream_t st) {
    int device = -1;
    if (cudaGetDevice(&device) == cudaSuccess && device >= 0 && device < kPoolDevices) {
        cudaMemPool_t pool = nullptr;
        {
            std::lock_guard<std::mutex> lock(g_pool_mutex);
            if (g_pool_refs[device] > 0) pool = g_pool[device];
        }
        if (pool) return cudaMallocFromPoolAsync(p, bytes, pool, st);
    }
    return cudaMallocAsync(p, bytes, st);
}

void release_scratch_pool(int device) {
    if (device < 0 || device >= kPoolDevices) return;
    std::lock_guard<std::mutex> lock(g_pool_mutex);
    if (g_pool[device] && --g_pool_refs[device] <= 0) {
        g_pool_refs[device] = 0;
        cudaMemPoolTrimTo(g_pool[device], 0);   // last handle gone: give the cached scratch back
        (void)cudaGetLastError();
    }
}

// The dynamic shared-memory opt-in is a property of (kernel, device) for the whole PROCESS, not of
// a graph handle: handles of different size, possibly on different host threads, share it.  So it
// is kept here, under one lock, and only ever raised: a small graph scored between two calls on a
// large one cannot lower it under the large one's launch.  The occupancy of a (kernel, device,
// block size, shared-memory size) does not change either, so it is queried once.
namespace {
std::mutex g_kernel_mutex;
std::map<std::pair<const void*, int>, size_t> g_smem_optin;
std::map<std::tuple<const void*, int, int, size_t>, int> g_ctas_per_sm;
}  // namespace

int kernel_ctas_per_sm(const void* kernel, int device, int threads, size_t smem, int* ctas_per_sm) {
    std::lock_guard<std::mutex> lock(g_kernel_mutex);
    size_t& granted = g_smem_optin[{kernel, device}];
    if (smem > granted) {
        BLP_CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        granted = smem;
    }
    if (!ctas_per_sm) return BLP_OK;
    const auto key = std::make_tuple(kernel, device, threads, smem);
    auto it = g_ctas_per_sm.find(key);
    if (it == g_ctas_per_sm.end()) {
        int n = 0;
        BLP_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kernel, threads, smem));
        it = g_ctas_per_sm.emplace(key, n).first;
    }
    *ctas_per_sm = it->second;
    return BLP_OK;
}

// Device properties, tuning (read_tuning, called once by the builder), the scratch pool and the
// timing events of a new handle.
int init_device_state(blp_graph* g, int device, const blp_tuning& tune) {
    cudaDeviceProp prop;
    BLP_CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    g->device = device;
    g->sm_count = prop.multiProcessorCount;
    g->max_smem_optin = (int)prop.sharedMemPerBlockOptin;
    g->tune = tune;
    g->pool = acquire_scratch_pool(device);   // nullptr: fall back to the default pool, untouched
    for (int sd = 0; sd < 2; ++sd)
        for (int k = 0; k < 4; ++k) BLP_CUDA_TRY(cudaEventCreate(&g->ev[sd][k]));
    for (int sd = 0; sd < 2; ++sd)
        BLP_CUDA_TRY(cudaEventCreateWithFlags(&g->ev_fork[sd], cudaEventDisableTiming));
    BLP_CUDA_TRY(cudaStreamCreateWithFlags(&g->side_stream, cudaStreamNonBlocking));
    // id-range plan of both sides (n_users / n_biz are set by the builder before this call)
    range_plan(g->n_users, g->max_smem_optin, g->tune.ranges, &g->n_ranges[0], &g->range_words[0]);
    range_plan(g->n_biz, g->max_smem_optin, g->tune.ranges, &g->n_ranges[1], &g->range_words[1]);
    for (int sd = 0; sd < 2; ++sd) {
        BLP_CUDA_TRY(cudaMalloc((void**)&g->d_counts[sd], sizeof(int) * 2));
        BLP_CUDA_TRY(cudaMemset(g->d_counts[sd], 0, sizeof(int) * 2));
    }
    return BLP_OK;
}

blp_tuning read_tuning() {
    blp_tuning t;
    if (const char* e = getenv("BLP_RANGES")) t.ranges = atoi(e);
    if (const char* e = getenv("BLP_HUB_MIN_DEG")) t.hub_min_deg = std::max(0, atoi(e));
    if (const char* e = getenv("BLP_PROBE_MIN_DEG")) t.probe_min_deg = std::max(0, atoi(e));
    if (const char* e = getenv("BLP_PROBE_RATIO")) t.probe_ratio = std::max(1, atoi(e));
    if (const char* e = getenv("BLP_LIGHT")) t.light = atoi(e) != 0;
    if (const char* e = getenv("BLP_LIGHT_HUBS")) t.light_hubs = atoi(e) != 0;
    if (const char* e = getenv("BLP_HOP3_GLOBAL")) t.hop3_global = atoi(e) != 0;
    if (const char* e = getenv("BLP_BIZ_INDEX")) t.biz_index = atoi(e) != 0 ? 1 : 0;
    if (const char* e = getenv("BLP_BIZ_INDEX_MAX_MB")) t.biz_index_cap = atoll(e) << 20;
    return t;
}

// 1/ln(d) in Q1.31 for d = 0..max_deg (0 for d <= 1), evaluated with the host libm.
void weight_lut(int32_t max_deg, std::vector<unsigned>& lut) {
    lut.assign((size_t)max_deg + 1, 0u);
    for (int32_t d = 2; d <= max_deg; ++d)
        lut[d] = (unsigned)llrint(ldexp(1.0 / log((double)d), BLP_AA_FRAC_BITS));
}
}  // namespace blp

extern "C" int blp_version(void) { return BLP_VERSION; }

extern "C" const char* blp_last_error(void) { return blp::g_last_error.c_str(); }

extern "C" int blp_device_count(int* count) {
    if (!count) {
        blp::set_error("blp_device_count: null argument");
        return BLP_ERR_INVALID;
    }
    *count = 0;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0) {
        (void)cudaGetLastError();
        blp::set_error(std::string("no usable CUDA device: ") + cudaGetErrorString(e));
        return BLP_ERR_CUDA;
    }
    *count = n;
    return BLP_OK;
}

extern "C" int blp_graph_destroy(blp_graph* g) {
    if (!g) return BLP_OK;
    blp::DeviceGuard device_guard__(g->device);
    cudaDeviceSynchronize();   // scratch of calls still in flight goes back to the pool first
    blp::host_state_destroy(g);
    cudaFree(g->u_row);
    cudaFree(g->b_row);
    cudaFree(g->u_adj);
    cudaFree(g->b_adj);
    cudaFree(g->u_deg);
    cudaFree(g->b_deg);
    cudaFree(g->u_adjw);
    cudaFree(g->b_adjw);
    for (int sd = 0; sd < 2; ++sd) {
        cudaFree(g->seg_off[sd]);
        cudaFree(g->xrow[sd]);
        cudaFree(g->hub_bm[sd]);
        cudaFree(g->node_wt[sd]);
        cudaFree(g->light[sd]);
        cudaFree(g->hubtab_cn[sd]);
        cudaFree(g->hubtab_aa[sd]);
    }
    cudaFree(g->biz_index);
    cudaFree(g->biz_hop2);
    cudaFree(g->biz_radj);
    cudaFree(g->biz_rank);
    for (int sd = 0; sd < 2; ++sd)
        for (int k = 0; k < 4; ++k)
            if (g->ev[sd][k]) cudaEventDestroy(g->ev[sd][k]);
    for (int sd = 0; sd < 2; ++sd)
        if (g->ev_fork[sd]) cudaEventDestroy(g->ev_fork[sd]);
    if (g->side_stream) cudaStreamDestroy(g->side_stream);
    for (int sd = 0; sd < 2; ++sd) cudaFree(g->d_counts[sd]);
    if (g->pool) blp::release_scratch_pool(g->device);
    (void)cudaGetLastError();
    delete g;
    return BLP_OK;
}

extern "C" int blp_graph_info(const blp_graph* g, blp_graph_info_t* info) {
    if (!g || !info) {
        blp::set_error("blp_graph_info: null argument");
        return BLP_ERR_INVALID;
    }
    info->n_users = g->n_users;
    info->n_biz = g->n_biz;
    info->n_edges_in = g->n_edges_in;
    info->n_edges = g->n_edges;
    info->n_users_in_graph = g->n_users_in;
    info->n_biz_in_graph = g->n_biz_in;
    info->max_user_degree = g->max_udeg;
    info->max_biz_degree = g->max_bdeg;
    info->device_bytes = g->device_bytes;
    info->device = g->device;
    info->sm_count = g->sm_count;
    info->n_hub_biz = g->n_hubs[0];
    info->n_hub_users = g->n_hubs[1];
    info->hub_min_biz_degree = g->n_hubs[0] ? g->hub_min_deg[0] : 0;
    info->hub_min_user_degree = g->n_hubs[1] ? g->hub_min_deg[1] : 0;
    info->biz_index_bytes = g->biz_index ? g->biz_index_bytes : 0;
    info->biz_index_build_ms = g->biz_index ? g->biz_index_build_ms : 0.f;
    return BLP_OK;
}

extern "C" int blp_graph_degrees(const blp_graph* g, int side, int32_t* host_out) {
    if (!g || !host_out || (side != BLP_SIDE_USER && side != BLP_SIDE_BUSINESS)) {
        blp::set_error("blp_graph_degrees: bad argument");
        return BLP_ERR_INVALID;
    }
    BLP_ON_DEVICE(g->device);
    const int* src = side == BLP_SIDE_USER ? g->u_deg : g->b_deg;
    size_t n = (size_t)(side == BLP_SIDE_USER ? g->n_users : g->n_biz);
    BLP_CUDA_TRY(cudaMemcpy(host_out, src, n * sizeof(int32_t), cudaMemcpyDeviceToHost));
    return BLP_OK;
}

extern "C" int blp_graph_reserve_sms(blp_graph* g, int n_sms) {
    if (!g || n_sms < 0 || n_sms >= g->sm_count) {
        blp::set_error("blp_graph_reserve_sms: bad argument");
        return BLP_ERR_INVALID;
    }
    g->reserve_sms = n_sms;
    return BLP_OK;
}

extern "C" int blp_score_stats(const blp_graph* g, int side, blp_score_stats_t* stats) {
    if (!g || !stats || (side != BLP_SIDE_USER && side != BLP_SIDE_BUSINESS)) {
        blp::set_error("blp_score_stats: bad argument");
        return BLP_ERR_INVALID;
    }
    *stats = g->stats[side];
    if (g->ev_recorded[side] && stats->path == BLP_PATH_BIZ_INDEX) {
        // one kernel, no grouping: its time is the whole call's
        BLP_ON_DEVICE(g->device);
        BLP_CUDA_TRY(cudaEventSynchronize(g->ev[side][2]));
        BLP_CUDA_TRY(cudaEventElapsedTime(&stats->score_ms, g->ev[side][1], g->ev[side][2]));
    } else if (g->ev_recorded[side]) {
        BLP_ON_DEVICE(g->device);
        BLP_CUDA_TRY(cudaEventSynchronize(g->ev[side][2]));
        BLP_CUDA_TRY(cudaEventElapsedTime(&stats->group_ms, g->ev[side][0], g->ev[side][1]));
        BLP_CUDA_TRY(cudaEventElapsedTime(&stats->score_ms, g->ev[side][1], g->ev[side][2]));
        if (g->ev_light[side])
            BLP_CUDA_TRY(cudaEventElapsedTime(&stats->light_ms, g->ev[side][1], g->ev[side][3]));
        int counts[2] = {0, 0};
        BLP_CUDA_TRY(cudaMemcpy(counts, g->d_counts[side], sizeof(counts), cudaMemcpyDeviceToHost));
        stats->n_groups = counts[0];
        stats->light_groups = counts[1];
    }
    return BLP_OK;
}
