// Graph handle: de-duplicated bipartite adjacency as two padded CSR arrays resident in HBM.
// Replaces snap.LoadEdgeList / snap.Nodes / GetNI().GetDeg() of the reference
// (similarity.py:16, 22, 65, 121).
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <new>
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

template <typename T>
static int upload(T** dptr, const std::vector<T>& h, int64_t* bytes) {
    size_t n = h.size() * sizeof(T);
    BLP_CUDA_TRY(cudaMalloc((void**)dptr, n ? n : sizeof(T)));
    if (n) BLP_CUDA_TRY(cudaMemcpy(*dptr, h.data(), n, cudaMemcpyHostToDevice));
    *bytes += (int64_t)n;
    return BLP_OK;
}

// Least-significant-digit radix sort of 64-bit keys on the host, only over the bits in use.
static void radix_sort_u64(std::vector<uint64_t>& keys, int bits_used) {
    const int RB = 11;
    const size_t n = keys.size();
    std::vector<uint64_t> tmp(n);
    std::vector<size_t> cnt((size_t)1 << RB);
    uint64_t* src = keys.data();
    uint64_t* dst = tmp.data();
    for (int shift = 0; shift < bits_used; shift += RB) {
        std::fill(cnt.begin(), cnt.end(), 0);
        const uint64_t mask = ((uint64_t)1 << RB) - 1;
        for (size_t i = 0; i < n; ++i) cnt[(src[i] >> shift) & mask]++;
        size_t run = 0;
        for (size_t d = 0; d < cnt.size(); ++d) {
            size_t c = cnt[d];
            cnt[d] = run;
            run += c;
        }
        for (size_t i = 0; i < n; ++i) dst[cnt[(src[i] >> shift) & mask]++] = src[i];
        std::swap(src, dst);
    }
    if (src != keys.data()) memcpy(keys.data(), src, n * sizeof(uint64_t));
}

static int bits_for(uint64_t v) {
    int b = 0;
    while (v) {
        ++b;
        v >>= 1;
    }
    return b ? b : 1;
}

// Row offsets of one padded CSR direction (each row rounded up to a multiple of four ids).
static void padded_offsets(int32_t n_rows, const std::vector<int32_t>& deg,
                           std::vector<long long>& off) {
    off.assign((size_t)n_rows + 1, 0);
    for (int32_t r = 0; r < n_rows; ++r) off[r + 1] = off[r] + (((long long)deg[r] + 3) & ~3LL);
}

// Bank striping.  The kernels probe a shared-memory bitmap with one 32-bit load per id; word
// id>>5 lives in bank (id>>5)&31, so 32 random ids cost ~3 wavefronts instead of 1.  Nothing in
// the algorithm needs a row in ascending order, so every row longer than the sub-warp path is
// permuted once here: the 32 ids that ONE load instruction touches (lane l reads component q of
// the int4 at index 32*block + l, i.e. slots 128*block + 4*l + q) are drawn from 32 different
// banks for as long as every bank still has ids left (largest remaining bucket first).
static void bank_stripe_row(int32_t* row, int len, std::vector<int32_t>& tmp,
                            std::vector<int32_t> (&bucket)[32]) {
    for (auto& b : bucket) b.clear();
    for (int i = 0; i < len; ++i) bucket[(row[i] >> 5) & 31].push_back(row[i]);
    tmp.assign((size_t)len, 0);
    const int n4 = (len + 3) >> 2;
    int order[32];
    for (int blk = 0; blk * 32 < n4; ++blk) {
        const int lanes = std::min(32, n4 - blk * 32);
        for (int q = 0; q < 4; ++q) {
            // real slots of this wave: lane l is real iff its slot index is < len
            int cap = 0;
            for (int l = 0; l < lanes; ++l) cap += (128 * blk + 4 * l + q) < len;
            if (cap == 0) continue;
            for (int b = 0; b < 32; ++b) order[b] = b;
            std::sort(order, order + 32, [&](int a, int b) {
                return bucket[a].size() > bucket[b].size();
            });
            int filled = 0, l = 0;
            while (filled < cap) {
                // one id from each of the fullest buckets; wrap around only when fewer than
                // `cap` buckets are left (then a bank repeats inside the wave)
                for (int k = 0; k < 32 && filled < cap; ++k) {
                    std::vector<int32_t>& bk = bucket[order[k]];
                    if (bk.empty()) continue;
                    while (l < lanes && (128 * blk + 4 * l + q) >= len) ++l;
                    tmp[(size_t)(128 * blk + 4 * l + q)] = bk.back();
                    bk.pop_back();
                    ++l;
                    ++filled;
                }
            }
        }
    }
    memcpy(row, tmp.data(), sizeof(int32_t) * (size_t)len);
}

// Per-entry weights: adjw[k] = Q1.31(1 / ln(deg(adj[k]))), with the degree taken on the side the
// entry names.  1/ln(deg) is evaluated once per distinct degree with the host libm (the kernels
// do no transcendental math); deg <= 1 contributes 0 (similarity.py:122-125), padding too.
static void entry_weights(const std::vector<int32_t>& adj, int32_t sentinel,
                          const std::vector<int32_t>& deg_of_entry_side, int32_t max_deg,
                          std::vector<unsigned>& adjw) {
    std::vector<unsigned> lut((size_t)max_deg + 1, 0u);
    for (int32_t d = 2; d <= max_deg; ++d)
        lut[d] = (unsigned)llrint(ldexp(1.0 / log((double)d), BLP_AA_FRAC_BITS));
    adjw.resize(adj.size());
    for (size_t k = 0; k < adj.size(); ++k)
        adjw[k] = adj[k] == sentinel ? 0u : lut[deg_of_entry_side[adj[k]]];
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

// Device properties, the scratch pool and the timing events of a new handle.
int init_device_state(blp_graph* g, int device) {
    cudaDeviceProp prop;
    BLP_CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    g->device = device;
    g->sm_count = prop.multiProcessorCount;
    g->max_smem_optin = (int)prop.sharedMemPerBlockOptin;
    read_tuning(&g->tune);
    g->pool = acquire_scratch_pool(device);   // nullptr: fall back to the default pool, untouched
    for (int sd = 0; sd < 2; ++sd)
        for (int k = 0; k < 4; ++k) BLP_CUDA_TRY(cudaEventCreate(&g->ev[sd][k]));
    for (int sd = 0; sd < 2; ++sd)
        BLP_CUDA_TRY(cudaEventCreateWithFlags(&g->ev_fork[sd], cudaEventDisableTiming));
    BLP_CUDA_TRY(cudaStreamCreateWithFlags(&g->side_stream, cudaStreamNonBlocking));
    // id-range plan of both sides (n_users / n_biz are set by the builders before this call)
    range_plan(g->n_users, g->max_smem_optin, g->tune.ranges, &g->n_ranges[0], &g->range_words[0]);
    range_plan(g->n_biz, g->max_smem_optin, g->tune.ranges, &g->n_ranges[1], &g->range_words[1]);
    for (int sd = 0; sd < 2; ++sd) {
        BLP_CUDA_TRY(cudaMalloc((void**)&g->d_counts[sd], sizeof(int) * 2));
        BLP_CUDA_TRY(cudaMemset(g->d_counts[sd], 0, sizeof(int) * 2));
    }
    return BLP_OK;
}

void read_tuning(blp_tuning* t) {
    if (const char* e = getenv("BLP_RANGES")) t->ranges = atoi(e);
    if (const char* e = getenv("BLP_GROUPING"))
        t->grouping = !strcmp(e, "runs") ? 1 : (!strcmp(e, "sort") ? 0 : -1);   // MODE_RUNS / MODE_SORT
    if (const char* e = getenv("BLP_NT")) t->nt = atoi(e);
    if (const char* e = getenv("BLP_LIGHT_STREAM")) t->light_stream = atoi(e) != 0;
    if (const char* e = getenv("BLP_SLICE_GROWTH")) t->slice_growth = atof(e);
    if (getenv("BLP_NO_BANK_STRIPE")) t->bank_stripe = false;
    if (const char* e = getenv("BLP_HOP3_GLOBAL")) t->hop3_global = atoi(e) != 0;
    if (const char* e = getenv("BLP_BIZ_INDEX")) t->biz_index = atoi(e) != 0 ? 1 : 0;
    if (const char* e = getenv("BLP_BIZ_INDEX_MAX_MB")) t->biz_index_cap = atoll(e) << 20;
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

extern "C" int blp_graph_create(int32_t n_users, int32_t n_biz, int64_t n_edges,
                                const int32_t* edge_u, const int32_t* edge_b, int device,
                                blp_graph** out) {
    if (!out) {
        blp::set_error("blp_graph_create: out is null");
        return BLP_ERR_INVALID;
    }
    *out = nullptr;
    if (n_users <= 0 || n_biz <= 0 || n_edges < 0 || (n_edges > 0 && (!edge_u || !edge_b))) {
        blp::set_error("blp_graph_create: need n_users>0, n_biz>0, n_edges>=0 and edge arrays");
        return BLP_ERR_INVALID;
    }
    int ndev = 0;
    int rc = blp_device_count(&ndev);
    if (rc != BLP_OK) return rc;
    if (device < 0 || device >= ndev) {
        blp::set_error("blp_graph_create: device index out of range");
        return BLP_ERR_INVALID;
    }
    BLP_ON_DEVICE(device);

    blp_graph* g = nullptr;
    try {
        // ---- de-duplicate: sort (u,b) keys, keep one of each (SNAP TUNGraph ignores repeats)
        const int bb = blp::bits_for((uint64_t)n_biz);      // key = u << bb | b, bits in use only
        const uint64_t bmask = ((uint64_t)1 << bb) - 1;
        std::vector<uint64_t> keys((size_t)n_edges);
        for (int64_t i = 0; i < n_edges; ++i) {
            int32_t u = edge_u[i], b = edge_b[i];
            if (u < 0 || u >= n_users || b < 0 || b >= n_biz) {
                char buf[160];
                snprintf(buf, sizeof(buf),
                         "blp_graph_create: edge %lld = (%d,%d) outside [0,%d) x [0,%d)",
                         (long long)i, u, b, n_users, n_biz);
                blp::set_error(buf);
                return BLP_ERR_RANGE;
            }
            keys[i] = ((uint64_t)(uint32_t)u << bb) | (uint32_t)b;
        }
        if (n_edges > (1 << 16))
            blp::radix_sort_u64(keys, bb + blp::bits_for((uint64_t)n_users));
        else
            std::sort(keys.begin(), keys.end());
        keys.erase(std::unique(keys.begin(), keys.end()), keys.end());
        const size_t m = keys.size();

        std::vector<int32_t> u_deg((size_t)n_users, 0), b_deg((size_t)n_biz, 0);
        for (size_t i = 0; i < m; ++i) {
            u_deg[keys[i] >> bb]++;
            b_deg[keys[i] & bmask]++;
        }
        std::vector<long long> u_off, b_off;
        blp::padded_offsets(n_users, u_deg, u_off);
        blp::padded_offsets(n_biz, b_deg, b_off);
        std::vector<int32_t> u_adj((size_t)u_off[n_users], n_biz);   // pre-filled with sentinels
        std::vector<int32_t> b_adj((size_t)b_off[n_biz], n_users);
        {
            // keys ascend by (u,b): user rows fill in order; business rows receive users in
            // ascending order too, so both directions come out sorted.
            std::vector<long long> bcur(b_off.begin(), b_off.end() - 1);
            size_t i = 0;
            for (int32_t u = 0; u < n_users; ++u) {
                long long w = u_off[u];
                for (int32_t k = 0; k < u_deg[u]; ++k, ++i) {
                    int32_t b = (int32_t)(keys[i] & bmask);
                    u_adj[w++] = b;
                    b_adj[bcur[b]++] = u;
                }
            }
        }
        std::vector<uint64_t>().swap(keys);
        blp_tuning tune;
        blp::read_tuning(&tune);
        // a side that needs id-range passes keeps its middle rows ascending (= partitioned by
        // range): business rows serve the user side, user rows the business side
        int optin = 0, nr_user = 1, nr_biz = 1, rw = 0;
        BLP_CUDA_TRY(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));
        blp::range_plan(n_users, optin, tune.ranges, &nr_user, &rw);
        blp::range_plan(n_biz, optin, tune.ranges, &nr_biz, &rw);
        if (tune.bank_stripe) {   // (BLP_NO_BANK_STRIPE: tuning switch)
            std::vector<int32_t> tmp;
            std::vector<int32_t> bucket[32];
            if (nr_biz == 1)
                for (int32_t u = 0; u < n_users; ++u)
                    if (u_deg[u] > 16) blp::bank_stripe_row(&u_adj[u_off[u]], u_deg[u], tmp, bucket);
            if (nr_user == 1)
                for (int32_t b = 0; b < n_biz; ++b)
                    if (b_deg[b] > 16) blp::bank_stripe_row(&b_adj[b_off[b]], b_deg[b], tmp, bucket);
        }

        g = new blp_graph();
        g->device = device;
        g->n_users = n_users;
        g->n_biz = n_biz;
        g->n_edges_in = n_edges;
        g->n_edges = (int64_t)m;
        for (int32_t d : u_deg) {
            g->n_users_in += d > 0;
            g->max_udeg = std::max(g->max_udeg, d);
        }
        for (int32_t d : b_deg) {
            g->n_biz_in += d > 0;
            g->max_bdeg = std::max(g->max_bdeg, d);
        }
        // packed row descriptors
        // (first entry / 4) has BLP_ROW_FIRST4_BITS bits in the descriptor: 2^30 padded entries
        if (u_off[n_users] / 4 >= (1LL << BLP_ROW_FIRST4_BITS) ||
            b_off[n_biz] / 4 >= (1LL << BLP_ROW_FIRST4_BITS) ||
            g->max_udeg >= (1 << 24) || g->max_bdeg >= (1 << 24)) {
            delete g;
            blp::set_error("blp_graph_create: graph too large for the packed row descriptors");
            return BLP_ERR_UNSUPPORTED;
        }
        g->u_adj_len = u_off[n_users];
        g->b_adj_len = b_off[n_biz];
        std::vector<unsigned long long> u_row((size_t)n_users), b_row((size_t)n_biz);
        for (int32_t u = 0; u < n_users; ++u)
            u_row[u] = ((unsigned long long)(u_off[u] >> 2) << 24) | (unsigned)u_deg[u];
        for (int32_t b = 0; b < n_biz; ++b)
            b_row[b] = ((unsigned long long)(b_off[b] >> 2) << 24) | (unsigned)b_deg[b];
        std::vector<unsigned> u_adjw, b_adjw;
        blp::entry_weights(u_adj, n_biz, b_deg, g->max_bdeg, u_adjw);   // user rows name businesses
        blp::entry_weights(b_adj, n_users, u_deg, g->max_udeg, b_adjw); // business rows name users

        rc = blp::init_device_state(g, device);
        if (rc == BLP_OK) rc = blp::upload(&g->u_row, u_row, &g->device_bytes);
        if (rc == BLP_OK) rc = blp::upload(&g->b_row, b_row, &g->device_bytes);
        if (rc == BLP_OK) rc = blp::upload(&g->u_adj, u_adj, &g->device_bytes);
        if (rc == BLP_OK) rc = blp::upload(&g->b_adj, b_adj, &g->device_bytes);
        if (rc == BLP_OK) rc = blp::upload(&g->u_deg, u_deg, &g->device_bytes);
        if (rc == BLP_OK) rc = blp::upload(&g->b_deg, b_deg, &g->device_bytes);
        if (rc == BLP_OK) rc = blp::upload(&g->u_adjw, u_adjw, &g->device_bytes);
        if (rc == BLP_OK) rc = blp::upload(&g->b_adjw, b_adjw, &g->device_bytes);
        if (rc == BLP_OK) rc = blp::build_range_segments(g, /*reorder=*/false, nullptr, nullptr);
        if (rc == BLP_OK) rc = blp::build_hub_bitmaps(g, u_deg.data(), b_deg.data());
        if (rc != BLP_OK) {
            std::string keep = blp_last_error();
            blp_graph_destroy(g);
            blp::set_error(keep);
            return rc;
        }
    } catch (const std::bad_alloc&) {
        if (g) blp_graph_destroy(g);
        blp::set_error("blp_graph_create: host allocation failed");
        return BLP_ERR_OOM;
    }
    *out = g;
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
