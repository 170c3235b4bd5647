// Grouping kernels: pairs -> work items (one item = one node whose hop-2 set is needed, with its
// pairs), and the split of the items between the two scoring kernels.
#ifndef BLP_SCORE_GROUP_CUH_
#define BLP_SCORE_GROUP_CUH_

#include <climits>

#include "blp_score_common.cuh"

namespace blp {

// ---------------------------------------------------------------------------------------------
// Grouping.  Every pair gets a key: the node whose hop-2 set it needs, or n_side when an id of
// the pair is not in the graph.  Two ways to turn keys into work items:
//   runs   -- the pairs already arrive grouped (examples.json stores them per user): every run
//             of equal keys is an item, the grouped order is the caller order, nothing moves;
//   sort   -- counting sort of the pair indices by key (any order in, e.g. the business side).
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ int group_key(int x, int y, int n_side, int n_mid,
                                         const int* __restrict__ g_deg,
                                         const int* __restrict__ m_deg) {
    bool ok = x >= 0 && x < n_side && y >= 0 && y < n_mid;
    if (ok) ok = (g_deg[x] > 0) && (m_deg[y] > 0);
    return ok ? x : n_side;   // similarity.py:52,59-60: any id not in the graph -> literal 0
}

// `cnt` (may be null): the group sizes are counted in the same pass when the sort mode is certain
// (the business side), which saves the counting sort's first pass over the keys
__global__ void k_group_keys(const int* __restrict__ gx, const int* __restrict__ gy, long long n,
                             int n_side, int n_mid, const int* __restrict__ g_deg,
                             const int* __restrict__ m_deg, int* __restrict__ keys,
                             unsigned* __restrict__ cnt) {
    long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    long long stride = (long long)gridDim.x * blockDim.x;
    for (; i < n; i += stride) {
        const int key = group_key(gx[i], gy[i], n_side, n_mid, g_deg, m_deg);
        keys[i] = key;
        if (cnt) atomicAdd(&cnt[key], 1u);
    }
}

constexpr int kRunCut = 4096;   // runs are cut at multiples of this, bounding the serial scan below

__device__ __forceinline__ bool run_starts_at(const int* __restrict__ keys, long long i) {
    return i == 0 || (i % kRunCut) == 0 || keys[i] != keys[i - 1];
}

__global__ void k_count_runs(const int* __restrict__ keys, long long n, unsigned* __restrict__ n_runs) {
    long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    long long stride = (long long)gridDim.x * blockDim.x;
    unsigned c = 0;
    for (; i < n; i += stride) c += run_starts_at(keys, i);
    c = __reduce_add_sync(kFull, c);
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(n_runs, c);
}

// Grouping mode, decided on the device so that the call never waits for the host:
// runs are used when they average >= 4 pairs (the business side forces sort mode).
__global__ void k_decide_mode(const unsigned* __restrict__ n_runs, long long n, int force,
                              int* __restrict__ mode) {
    *mode = force >= 0 ? force : (((long long)*n_runs * 4 <= n) ? MODE_RUNS : MODE_SORT);
}

// One CTA per kRunCut-sized segment of the pair list (runs never cross a segment boundary):
// every thread owns 16 consecutive positions, a block scan numbers the run starts, the item slots
// of the segment are claimed with one atomic, and a run's end is the next run's start.
__global__ void __launch_bounds__(256) k_runs_to_items(const int* __restrict__ mode,
                                                       const int* __restrict__ keys, long long n,
                                                       int* __restrict__ item_key,
                                                       int* __restrict__ item_start,
                                                       int* __restrict__ item_end,
                                                       int* __restrict__ n_items) {
    if (*mode != MODE_RUNS) return;
    static_assert(kRunCut == 256 * 16, "one thread owns 16 positions of a segment");
    __shared__ int s_warp[8];
    __shared__ int s_base;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const long long n_seg = (n + kRunCut - 1) / kRunCut;
    for (long long seg = blockIdx.x; seg < n_seg; seg += gridDim.x) {
        const long long seg_lo = seg * kRunCut, seg_hi = min(n, seg_lo + kRunCut);
        const long long lo = seg_lo + tid * 16;
        int k[17];
        k[0] = (lo > seg_lo && lo - 1 < seg_hi) ? keys[lo - 1] : INT_MIN;   // INT_MIN: forces a start
#pragma unroll
        for (int j = 0; j < 16; ++j) k[j + 1] = lo + j < seg_hi ? keys[lo + j] : INT_MIN;
        int mine = 0;
#pragma unroll
        for (int j = 0; j < 16; ++j) mine += (lo + j < seg_hi) && (k[j + 1] != k[j]);
        int inc = mine;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            int t = __shfl_up_sync(kFull, inc, d);
            if (lane >= d) inc += t;
        }
        if (lane == 31) s_warp[warp] = inc;
        __syncthreads();
        int before = inc - mine, total = 0;
#pragma unroll
        for (int w = 0; w < 8; ++w) {
            if (w < warp) before += s_warp[w];
            total += s_warp[w];
        }
        if (tid == 0) s_base = atomicAdd(n_items, total);
        __syncthreads();
        int slot = s_base + before;
        const int last = s_base + total - 1;
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            if (lo + j < seg_hi && k[j + 1] != k[j]) {
                item_key[slot] = k[j + 1];
                item_start[slot] = (int)(lo + j);
                if (slot > s_base) item_end[slot - 1] = (int)(lo + j);
                ++slot;
            }
        }
        if (tid == 0 && total > 0) item_end[last] = (int)seg_hi;
        __syncthreads();
    }
}

__global__ void k_group_count(const int* __restrict__ mode, const int* __restrict__ keys,
                              long long n, unsigned* __restrict__ cnt) {
    if (*mode != MODE_SORT) return;
    long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    long long stride = (long long)gridDim.x * blockDim.x;
    for (; i < n; i += stride) atomicAdd(&cnt[keys[i]], 1u);
}

// Exclusive scan of the group sizes, which also compacts the non-empty keys into items (in key
// order).  Three small launches -- per-tile sums, one CTA scanning the tile sums, per-tile apply --
// instead of one CTA walking all keys (84 us on C2's business side in round 1): a tile is 4096
// keys (1024 threads x 4).
constexpr int kScanTile = 4096;

// block-wide exclusive scan of (v, f) over 1024 threads; returns this thread's exclusive prefixes
// and the block totals (s_sum / s_flag: 32 entries each)
__device__ __forceinline__ void block_scan2(unsigned v, int f, unsigned* s_sum, int* s_flag, unsigned& ex_v,
                                            int& ex_f, unsigned& tot_v, int& tot_f) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned own_v = v;
    const int own_f = f;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const unsigned t = __shfl_up_sync(kFull, v, d);
        const int tf = __shfl_up_sync(kFull, f, d);
        if (lane >= d) {
            v += t;
            f += tf;
        }
    }
    if (lane == 31) {
        s_sum[warp] = v;
        s_flag[warp] = f;
    }
    __syncthreads();
    unsigned wv = s_sum[lane];
    int wf = s_flag[lane];
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const unsigned t = __shfl_up_sync(kFull, wv, d);
        const int tf = __shfl_up_sync(kFull, wf, d);
        if (lane >= d) {
            wv += t;
            wf += tf;
        }
    }
    tot_v = __shfl_sync(kFull, wv, 31);
    tot_f = __shfl_sync(kFull, wf, 31);
    unsigned wb = __shfl_sync(kFull, wv, max(warp, 1) - 1);
    int fb = __shfl_sync(kFull, wf, max(warp, 1) - 1);
    if (warp == 0) {
        wb = 0;
        fb = 0;
    }
    ex_v = wb + (v - own_v);
    ex_f = fb + (f - own_f);
    __syncthreads();   // s_sum / s_flag may be reused by the caller's next round
}

__global__ void __launch_bounds__(1024) k_group_tile_sums(const int* __restrict__ mode,
                                                          const unsigned* __restrict__ cnt, int n_keys,
                                                          unsigned* __restrict__ tile_sum,
                                                          int* __restrict__ tile_items) {
    if (*mode != MODE_SORT) return;
    __shared__ unsigned s_sum[32];
    __shared__ int s_flag[32];
    const int i0 = blockIdx.x * kScanTile + threadIdx.x * 4;
    unsigned v = 0;
    int f = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const unsigned c = i0 + k < n_keys ? cnt[i0 + k] : 0u;
        v += c;
        f += c > 0;
    }
    unsigned ex_v, tot_v;
    int ex_f, tot_f;
    block_scan2(v, f, s_sum, s_flag, ex_v, ex_f, tot_v, tot_f);
    if (threadIdx.x == 0) {
        tile_sum[blockIdx.x] = tot_v;
        tile_items[blockIdx.x] = tot_f;
    }
}

// one CTA: exclusive scan of the per-tile totals in place; the grand total of items -> n_items
__global__ void __launch_bounds__(1024) k_group_tile_scan(const int* __restrict__ mode,
                                                          unsigned* __restrict__ tile_sum,
                                                          int* __restrict__ tile_items, int n_tiles,
                                                          int* __restrict__ n_items) {
    if (*mode != MODE_SORT) return;
    __shared__ unsigned s_sum[32];
    __shared__ int s_flag[32];
    unsigned base_v = 0;   // carried identically by every thread (n < 2^31 pairs per call)
    int base_f = 0;
    for (int start = 0; start < n_tiles; start += 1024) {
        const int i = start + threadIdx.x;
        const unsigned v = i < n_tiles ? tile_sum[i] : 0u;
        const int f = i < n_tiles ? tile_items[i] : 0;
        unsigned ex_v, tot_v;
        int ex_f, tot_f;
        block_scan2(v, f, s_sum, s_flag, ex_v, ex_f, tot_v, tot_f);
        if (i < n_tiles) {
            tile_sum[i] = base_v + ex_v;
            tile_items[i] = base_f + ex_f;
        }
        base_v += tot_v;
        base_f += tot_f;
    }
    if (threadIdx.x == 0) *n_items = base_f;
}

__global__ void __launch_bounds__(1024) k_group_tile_apply(const int* __restrict__ mode,
                                                           const unsigned* __restrict__ cnt, int n_keys,
                                                           const unsigned* __restrict__ tile_sum,
                                                           const int* __restrict__ tile_items,
                                                           unsigned* __restrict__ grp_off,
                                                           int* __restrict__ item_key,
                                                           int* __restrict__ item_start,
                                                           int* __restrict__ item_end) {
    if (*mode != MODE_SORT) return;
    __shared__ unsigned s_sum[32];
    __shared__ int s_flag[32];
    const int i0 = blockIdx.x * kScanTile + threadIdx.x * 4;
    unsigned c[4];
    unsigned v = 0;
    int f = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        c[k] = i0 + k < n_keys ? cnt[i0 + k] : 0u;
        v += c[k];
        f += c[k] > 0;
    }
    unsigned ex_v, tot_v;
    int ex_f, tot_f;
    block_scan2(v, f, s_sum, s_flag, ex_v, ex_f, tot_v, tot_f);
    unsigned off = tile_sum[blockIdx.x] + ex_v;          // exclusive prefix of this thread
    int slot = tile_items[blockIdx.x] + ex_f;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        if (i0 + k < n_keys) {
            grp_off[i0 + k] = off;                       // doubles as the scatter cursor
            if (c[k] > 0) {
                item_key[slot] = i0 + k;
                item_start[slot] = (int)off;
                item_end[slot] = (int)(off + c[k]);
                ++slot;
            }
            off += c[k];
        }
    }
}

__global__ void k_group_scatter(const int* __restrict__ mode, const int* __restrict__ keys,
                                const int* __restrict__ gy, long long n,
                                unsigned* __restrict__ cursor, int2* __restrict__ pg,
                                int* __restrict__ inv) {
    if (*mode != MODE_SORT) return;
    long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    long long stride = (long long)gridDim.x * blockDim.x;
    for (; i < n; i += stride) {
        const unsigned pos = atomicAdd(&cursor[keys[i]], 1u);   // cursor starts at the group offset
        pg[pos] = make_int2((int)i, gy[i]);
        inv[i] = (int)pos;
    }
}

// Sort mode, second half: grouped-order records -> caller-order columns.  A gather through the
// inverse permutation: random 24-byte reads are far cheaper than the random 4/8-byte partial-
// sector writes the scoring kernel would otherwise issue (measured: 0.8 ms of 2.4 ms on C2).
__global__ void k_unpermute(const int* __restrict__ mode, const unsigned long long* __restrict__ rec,
                            const int* __restrict__ inv, long long n, int* __restrict__ cn,
                            int* __restrict__ uni, double* __restrict__ jac, double* __restrict__ aa) {
    if (*mode != MODE_SORT) return;
    long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    // two rows per trip: the two dependent chains (inverse index -> 24-byte record) overlap
    for (; i < n; i += 2 * stride) {
        const long long i1 = i + stride;
        const bool two = i1 < n;
        const unsigned long long* r0 = rec + 3ll * ld_once(inv + i);
        const unsigned long long* r1 = rec + 3ll * ld_once(inv + (two ? i1 : i));
        const unsigned long long c0 = ld_once(r0), c1 = ld_once(r1);
        unsigned long long j0 = 0, j1 = 0, a0 = 0, a1 = 0;
        if (jac) {
            j0 = ld_once(r0 + 1);
            j1 = ld_once(r1 + 1);
        }
        if (aa) {
            a0 = ld_once(r0 + 2);
            a1 = ld_once(r1 + 2);
        }
        if (cn) st_stream(cn + i, (int)(unsigned)c0);
        if (uni) st_stream(uni + i, (int)(unsigned)(c0 >> 32));
        if (jac) st_stream(jac + i, __longlong_as_double((long long)j0));
        if (aa) st_stream(aa + i, __longlong_as_double((long long)a0));
        if (two) {
            if (cn) st_stream(cn + i1, (int)(unsigned)c1);
            if (uni) st_stream(uni + i1, (int)(unsigned)(c1 >> 32));
            if (jac) st_stream(jac + i1, __longlong_as_double((long long)j1));
            if (aa) st_stream(aa + i1, __longlong_as_double((long long)a1));
        }
    }
}

// Items -> two lists of item indices (warp-per-group kernel / CTA kernel), any order.
enum { SC_N_ITEMS = 0, SC_HEAVY_WORK = 1, SC_N_RUNS = 2, SC_MODE = 3, SC_N_LIGHT = 4, SC_N_HEAVY = 5,
       SC_LIGHT_WORK = 6, SC_COUNT = 8 };
__global__ void k_split_items(int* __restrict__ scalars, const int* __restrict__ item_key,
                              const unsigned char* __restrict__ light, int n_side,
                              int* __restrict__ light_list, int* __restrict__ heavy_list) {
    const int n = scalars[SC_N_ITEMS];
    const int lane = threadIdx.x & 31;
    const int stride = gridDim.x * blockDim.x;
    for (int base = blockIdx.x * blockDim.x + threadIdx.x - lane; base < n; base += stride) {
        const int i = base + lane;
        int cls = -1;   // 0 CTA kernel, 1 warp-per-group kernel
        if (i < n) {
            const int key = item_key[i];
            cls = key < n_side ? light[key] : 0;
        }
        const unsigned lt = (1u << lane) - 1u;
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const unsigned m = __ballot_sync(kFull, cls == k);
            int b = 0;
            if (lane == 0 && m) b = atomicAdd(&scalars[k == 0 ? SC_N_HEAVY : SC_N_LIGHT], __popc(m));
            b = __shfl_sync(kFull, b, 0);
            int* dst = k == 0 ? heavy_list : light_list;
            if (cls == k) dst[b + __popc(m & lt)] = i;
        }
    }
}

}  // namespace blp

#endif  // BLP_SCORE_GROUP_CUH_
