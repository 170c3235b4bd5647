// Internal declarations shared by the graph builder and the scoring kernels (not part of the ABI).
#ifndef BLP_INTERNAL_H_
#define BLP_INTERNAL_H_

#include <cuda_runtime.h>
#include <stdint.h>
#include <string>
#include <vector>

#include "blp.h"

// Packed row descriptor fields (see blp_graph below).
#define BLP_ROW_FIRST4_BITS 28
#define BLP_ROW_SLOT_SHIFT 52
#define BLP_ROW_MAX_SLOTS 2047
// expansion-side entry of a hub (xrow): 1 << 63 | table row << 35 | bitmap slot << 24 | degree
#define BLP_XROW_ORIDX_SHIFT 35

// Fixed point for the Adamic-Adar weights: integer sums are order independent.  A weight is at
// most 1/ln 2 = 1.4427 < 2, so Q1.31 fits 32 bits; sums are kept in 64 bits.
#define BLP_AA_FRAC_BITS 31

struct blp_host_state;   // staging buffers and streams of blp_score_pairs_host (blp_host.cu)

// BLP_* tuning variables (developer overrides).  Read ONCE, when a handle is created -- never on
// the scoring path.
struct blp_tuning {
    int ranges = 0;            // BLP_RANGES: at least this many id-range passes
    int hub_min_deg = -1;      // BLP_HUB_MIN_DEG: hub bitmaps from this degree on (0 = none, -1 = by bitmap size)
    int probe_min_deg = -1;    // BLP_PROBE_MIN_DEG: probe bitmaps from this degree on (0 = none, -1 = by hub degree)
    int probe_ratio = 0;       // BLP_PROBE_RATIO: probe when deg(y) >= ratio * |hop2(x)| (0 = kProbeRatio)
    bool light = true;         // BLP_LIGHT=0: no warp-per-group kernel
    bool light_hubs = true;    // BLP_LIGHT_HUBS=0: the warp-per-group kernel takes hub-free groups only
    bool hop3_global = false;  // BLP_HOP3_GLOBAL=1: hop-3 user bitmap in global scratch even when it fits shared memory
    int biz_index = -1;        // BLP_BIZ_INDEX=0|1: never / always (cap ignored) build the business index (-1 = by size)
    long long biz_index_cap = 0;  // BLP_BIZ_INDEX_MAX_MB: byte cap of the automatic choice (0 = default)
};

struct blp_graph {
    blp_host_state* host = nullptr;
    int device = 0;
    int sm_count = 0;
    int max_smem_optin = 0;  // bytes of dynamic shared memory one CTA may opt in to
    int reserve_sms = 0;     // SMs left out of the persistent scoring grids
    blp_tuning tune;         // developer overrides, read when the handle was created
    // stream-ordered scratch comes from the library's own per-device pool (shared by its handles,
    // kept warm, trimmed when the last handle goes; see acquire_scratch_pool) -- the device's
    // default pool and other libraries' allocators are left alone
    cudaMemPool_t pool = nullptr;
    int32_t n_users = 0, n_biz = 0;
    int64_t n_edges_in = 0, n_edges = 0;
    int32_t n_users_in = 0, n_biz_in = 0, max_udeg = 0, max_bdeg = 0;
    int64_t device_bytes = 0;
    int64_t u_adj_len = 0, b_adj_len = 0;   // padded entries of u_adj / b_adj
    // Both CSR directions.  Every row is padded AT ITS TAIL to a multiple of four ids with the
    // sentinel n_biz (user rows) / n_users (business rows), so every row starts 16-byte aligned and
    // is read with 128-bit loads without a tail; the first deg(row) entries are the real ids
    // (blp_hop3 and the light-kernel prefetch rely on that).  Nothing else about the order inside
    // a row may be assumed (business rows are filled through atomic cursors, longer rows are
    // bank-striped, see k_bank_stripe), so no binary search over rows.
    // Row descriptors: (first padded entry / 4) << 24 | true degree -- one 8-byte load per list.
    // Bits 52..62 hold (hub-bitmap slot + 1) of a node whose neighbour list is also kept as a
    // bitmap (0 = none); they are set only when every first-entry index fits 28 bits.
    unsigned long long* u_row = nullptr;  // [n_users]
    unsigned long long* b_row = nullptr;  // [n_biz]
    int* u_adj = nullptr;        // user -> businesses
    int* b_adj = nullptr;        // business -> users
    int* u_deg = nullptr;        // true (unpadded, de-duplicated) degrees
    int* b_deg = nullptr;
    // Adamic-Adar weight 1/ln(deg(id)) (0 where deg <= 1 and in padding) of every adjacency
    // entry, Q1.31, parallel to u_adj / b_adj: the weight streams in beside the id it belongs to.
    unsigned* u_adjw = nullptr;
    unsigned* b_adjw = nullptr;
    // Hub bitmaps.  For side s (0 = user side, 1 = business side) the middle nodes of degree >=
    // hub_min_deg[s] have their whole neighbour list precomputed as a bitmap over the grouping
    // side, so the two-hop expansion ORs 128-bit words instead of walking the list id by id.
    // Middle nodes of degree >= probe_min_deg[s] (<= hub_min_deg[s]) get a bitmap as well, used only
    // by the intersection phase: when hop2(x) is small it is kept as an id list and a pair whose
    // partner has a bitmap is scored by probing that bitmap with the list instead of streaming N(y).
    unsigned long long* xrow[2] = {nullptr, nullptr};   // expansion-side row descriptors (hubs tagged)
    unsigned* hub_bm[2] = {nullptr, nullptr};     // [n_hubs][bm_words]
    unsigned char* light[2] = {nullptr, nullptr}; // per grouping node of side s: 1 = warp-per-group kernel
    // |N(h) & N(y)| and its weight sum, OR-hub h (row) x bitmap node y (column), per side
    int* hubtab_cn[2] = {nullptr, nullptr};
    unsigned long long* hubtab_aa[2] = {nullptr, nullptr};
    unsigned* node_wt[2] = {nullptr, nullptr};    // Q1.31 1/ln(deg) per grouping-side node of side s
    // Id ranges.  When the bitmap over side s's universe does not fit one CTA's shared memory (or
    // BLP_RANGES asks for it) k_score_side processes every group of side s once per id range.  The
    // rows of that side's MIDDLE adjacency are then kept partitioned by range (not bank-striped):
    // seg_off[s][m * (n_ranges+1) + r] is the entry offset inside row m where range r's ids begin,
    // so a pass streams only the segment it can use instead of filtering the whole list again.
    int n_ranges[2] = {1, 1};
    int range_words[2] = {0, 0};                      // bitmap words of one range (multiple of 4)
    int* seg_off[2] = {nullptr, nullptr};
    int hub_min_deg[2] = {0x7fffffff, 0x7fffffff};    // expansion ORs the bitmap from here on
    int probe_min_deg[2] = {0x7fffffff, 0x7fffffff};  // a bitmap exists from here on
    int n_hubs[2] = {0, 0};                           // bitmaps kept (both kinds)
    int probe_ratio = 2;                              // probe when deg(y) >= ratio * |hop2(x)|
    bool row_slots[2] = {false, false};               // slot bits present in the middle rows of side s
    // Business index: the business x business co-review relation as one bitmap row per business,
    // biz_index_words words each, and |hop2(b)| per business (biz_hop2, by id).  Rows AND columns
    // are business RANKS by degree (biz_rank[b], rank 0 = the most-reviewed business): row rank(b)
    // holds hop2(b) (businesses sharing a reviewer with b, b itself excluded).  The relation is
    // symmetric, so the kernel reads the bit of (b, b') at row max(rank b, rank b'), column min
    // (blp_score_index.cuh).  Built once per graph when the business side runs unranged and the
    // rows fit the cap (build_biz_index); the business side then scores every pair by testing N(u)
    // against it, with no grouping.  nullptr = the grouped path.  biz_radj = u_adj with every
    // business id replaced by its rank.
    unsigned* biz_index = nullptr;
    int* biz_hop2 = nullptr;
    int* biz_radj = nullptr;
    int* biz_rank = nullptr;
    int biz_index_words = 0;
    int64_t biz_index_bytes = 0;
    float biz_index_build_ms = 0.f;
    blp_score_stats_t stats[2] = {};
    cudaEvent_t ev[2][4] = {};   // per side: start, after grouping, after scoring, after the light kernel
    bool ev_light[2] = {false, false};
    int* d_counts[2] = {nullptr, nullptr};       // per side: work items, light items of the last call
    cudaStream_t side_stream = nullptr;          // the warp-per-group kernel runs beside the CTA kernel
    cudaEvent_t ev_fork[2] = {nullptr, nullptr};
    bool ev_recorded[2] = {false, false};
};

namespace blp {
// words of the shared-memory bitmap over n_side nodes (+1 sentinel bit), multiple of 4
inline int bitmap_words(int n_side) { return (int)((((long long)n_side + 1 + 31) / 32 + 3) & ~3LL); }
int build_hub_bitmaps(blp_graph* g, const int* u_deg_host, const int* b_deg_host);
// how many id-range passes side `n_side` needs on a device with `smem_optin` bytes per CTA
void range_plan(int n_side, int smem_optin, int forced, int* n_ranges, int* range_words);
constexpr int kMaxRanges = 255;
// partition the middle rows of every ranged side by id range and fill seg_off; `tmp` = device
// scratch of max(u_adj_len, b_adj_len) ints
int build_range_segments(blp_graph* g, int* tmp, cudaStream_t st);
int init_device_state(blp_graph* g, int device, const blp_tuning& tune);
void host_state_destroy(blp_graph* g);
void weight_lut(int32_t max_deg, std::vector<unsigned>& lut);
int radix_sort_u64(unsigned long long* keys, unsigned long long* tmp, long long n,
                   const std::vector<int>& shifts, cudaStream_t st, unsigned long long** sorted);
// out[i] = in[0] + ... + in[i-1] for n 32-bit counts, stream-ordered; with host_total the grand
// total is copied back (the stream is synchronised)
int exclusive_scan_u32(const unsigned* in, long long n, unsigned long long* out,
                       unsigned long long* host_total, cudaStream_t st);
void set_error(const std::string& msg);
int cuda_fail(cudaError_t e, const char* what, const char* file, int line);
blp_tuning read_tuning();
cudaMemPool_t acquire_scratch_pool(int device);
void release_scratch_pool(int device);
cudaError_t scratch_alloc(void** p, size_t bytes, cudaStream_t st);
// Raises `kernel`'s dynamic shared-memory opt-in on `device` (the current device) to at least
// `smem` -- never lowers it -- and, when ctas_per_sm != nullptr, returns how many CTAs of `threads`
// threads with `smem` bytes fit on one SM.  Every kernel whose dynamic shared memory may exceed the
// 48 KB default is configured here and nowhere else.
int kernel_ctas_per_sm(const void* kernel, int device, int threads, size_t smem, int* ctas_per_sm);
// stream-ordered scratch from the handle's own pool
inline cudaError_t pool_alloc(blp_graph* g, void** p, size_t bytes, cudaStream_t st) {
    return g->pool ? cudaMallocFromPoolAsync(p, bytes, g->pool, st) : cudaMallocAsync(p, bytes, st);
}

// Every entry point runs on the handle's device and leaves the caller's current device as it
// found it (a process driving several GPUs must not find its device switched by a library call).
struct DeviceGuard {
    int prev = -1;
    cudaError_t err = cudaSuccess;
    explicit DeviceGuard(int device) {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != device) err = cudaSetDevice(device);
        else prev = -1;   // nothing to restore
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
    DeviceGuard(const DeviceGuard&) = delete;
    DeviceGuard& operator=(const DeviceGuard&) = delete;
};
}  // namespace blp

#define BLP_ON_DEVICE(dev)                                                                    \
    blp::DeviceGuard device_guard__(dev);                                                     \
    if (device_guard__.err != cudaSuccess)                                                    \
        return blp::cuda_fail(device_guard__.err, "cudaSetDevice", __FILE__, __LINE__)

#define BLP_CUDA_TRY(expr)                                                     \
    do {                                                                       \
        cudaError_t e__ = (expr);                                              \
        if (e__ != cudaSuccess) return blp::cuda_fail(e__, #expr, __FILE__, __LINE__); \
    } while (0)

#endif  // BLP_INTERNAL_H_
