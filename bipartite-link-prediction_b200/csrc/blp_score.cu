// Candidate-pair scoring kernels (sm_100a).
//
// One "side" of the reference's similarity.py is: build hop2(x) for every distinct grouping node
// x (users() loop A, similarity.py:24-33 / business() loop A', :67-78), then for every candidate
// pair (x, y) intersect hop2(x) with N(y) (loops C / C', :48-61 / :91-106) and derive
// common_neighbors, jaccard and adamic_adar (:108-126).  Both sides are the same computation
// with the two CSR directions swapped, so one set of kernels serves both:
//
//   hop2(x) = ( U_{m in N(x)} N(m) ) \ {x}        held in shared memory: a bitmap over the whole
//                                                 universe (k_score_side, one CTA per group) or a
//                                                 hash table + id list (k_score_light, one warp)
//   cn(x,y) = | { i in N(y) : i in hop2(x) } |     N(y) streamed with 128-bit loads -- or, when y
//                                                 has a bitmap of its own, hop2(x) probed into it
//
// Work distribution.  The user side, and the business side of a handle without a business index,
// take the GROUPED path: pairs are grouped by x (runs of an already grouped list, or a counting
// sort: k_group_*), the groups are split by size class, and two persistent grids pull their
// groups from atomic counters.  Inside a CTA of k_score_side both the expansion and the
// intersection phase walk a *set of adjacency lists* whose lengths span 1 .. >100k: the lists of
// a tile are cut into 512-id chunks, the chunk counts are prefix-summed in shared memory and warps
// take chunks round-robin, so a hub list is spread over the whole CTA while short lists cost one
// warp pass each (degree-bucketed scheduling without separate launches).  The business side of a
// handle WITH an index (hop2(b) of every business precomputed once per graph as a bitmap row:
// C1-C4) is one pass over the pairs in the caller's order, k_score_biz_indexed: a lane tests N(u)
// against row b, the warp walks the rare long N(u) together -- no grouping, no expansion, no
// un-permute.  Both paths end in the same epilogue (emit_pair).
//
// Layout of the translation unit:
//   blp_score_common.cuh  launch arguments (SideArgs), row-descriptor accessors, streaming loads,
//                         the shared epilogue
//   blp_score_group.cuh   pairs -> work items (runs / counting sort), light / heavy split
//   blp_score_light.cuh   k_score_light: one WARP per small group (hash-table hop-2 set), the
//                         per-node class flags and the hub x bitmap-node intersection tables
//   blp_score_index.cuh   the business index: its construction and the per-pair kernel
//   this file             k_score_side: one CTA per group (shared-memory bitmap), hub-bitmap
//                         construction, blp_score_pairs (grouping, split, both launches)
#include <algorithm>
#include <climits>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <vector>

#include "blp_internal.h"

#ifndef BLP_HUB_TMA
#define BLP_HUB_TMA 1   // 0: A/B build with the cp.async hub copy (and no async-proxy fences)
#endif

#include "blp_score_common.cuh"
#include "blp_score_group.cuh"
#include "blp_score_light.cuh"
#include "blp_score_index.cuh"

namespace blp {

// ---------------------------------------------------------------------------------------------
// The scoring kernel.
// ---------------------------------------------------------------------------------------------
struct TileSmem {
    unsigned long long row[kTile];     // packed row descriptor of every list of the tile
    unsigned long long aa[kTile];      // Q24.40 Adamic-Adar accumulators
    unsigned long long hub_bar;        // mbarrier the TMA bulk copy of a hub bitmap completes on
    int scan[kTile + 8];               // exclusive prefix of long-list chunk counts, [kTile] = total
    int coarse[32];                    // scan[8*i], contiguous: conflict-free first probe
    int next_chunk[4];                 // dynamic chunk dispensers, one per sweep kind (OP_*)
    int cn[kTile];
    int idx[kTile];                    // caller-order pair index
    int hub[kProbeCap];                // [0, kTile): hub-bitmap slots met in the current expansion
                                       // tile; hub-free group: hop2(x) as an id list (probe path)
    int wsum[32];
    int red[32];
    int item_next;
    int hop2cnt;                       // bits turned on during the expansion of this group
    int nhub;
    int list_on;                       // this group's expansion appends the ids it turns on to hub[]
    int list_n;                        // ids in the list
    int nprobe;                        // pairs of the current tile scored by probing
    unsigned char probe[kTile];        // their tile positions
};
static_assert(kProbeCap >= kTile && kTile <= 256, "hub[] doubles as the list; probe[] holds uint8");

// Exclusive scan of `v` over the first kTile threads into ts.scan[]; ts.scan[kTile] = total.
template <int NT>
__device__ __forceinline__ void tile_scan(TileSmem& ts, int v, int tid, int count) {
    const int lane = tid & 31, warp = tid >> 5;
#ifndef BLP_NO_SMALL_SCAN
    if (count <= 32) {
        // the common tile (a user's few businesses, a group's 32 pairs) lives in warp 0 alone:
        // one warp scan, one barrier
        if (warp == 0) {
            int inc = v;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                int t = __shfl_up_sync(kFull, inc, d);
                if (lane >= d) inc += t;
            }
            const int total = __shfl_sync(kFull, inc, 31);
            const int ex = inc - v;
            ts.scan[lane] = ex;
            const int c8 = __shfl_sync(kFull, ex, (lane & 3) * 8);
            ts.coarse[lane] = lane < 4 ? c8 : INT_MAX;
            if (lane == 0) ts.scan[kTile] = total;
            if (lane < 4) ts.next_chunk[lane] = NT / 32;   // chunks 0..NW-1 are dealt statically
        }
        __syncthreads();
        return;
    }
#endif
    int inc = v;
    if (tid < kTile) {
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            int t = __shfl_up_sync(kFull, inc, d);
            if (lane >= d) inc += t;
        }
        if (lane == 31) ts.wsum[warp] = inc;
    }
    __syncthreads();
    if (tid < kTile) {
        // prefix over the kTile/32 warp totals, computed redundantly by every warp
        int wv = lane < kTile / 32 ? ts.wsum[lane] : 0;
#pragma unroll
        for (int d = 1; d < kTile / 32; d <<= 1) {
            int t = __shfl_up_sync(kFull, wv, d);
            if (lane >= d) wv += t;
        }
        int base = __shfl_sync(kFull, wv, max(warp, 1) - 1);
        if (warp == 0) base = 0;
        const int ex = base + inc - v;
        ts.scan[tid] = ex;
        if ((tid & 7) == 0) ts.coarse[tid >> 3] = ex;
        if (tid == kTile - 1) ts.scan[kTile] = base + inc;
        if (tid < 4) ts.next_chunk[tid] = NT / 32;
    }
    __syncthreads();
}

// Which list owns chunk c?  Two 32-wide probes of the 257-entry prefix array (warp-uniform c).
__device__ __forceinline__ int find_list(const TileSmem& ts, int c, int lane) {
    int v = lane < kTile / 8 ? ts.coarse[lane] : INT_MAX;
    int kb = __popc(__ballot_sync(kFull, v <= c)) - 1;
    int v2 = lane < 8 ? ts.scan[kb * 8 + lane] : INT_MAX;
    return kb * 8 + __popc(__ballot_sync(kFull, v2 <= c)) - 1;
}

// The two things done to a streamed id.
//   OP_SET  expansion: set the id's bit.  A plain read filters ids whose bit is already there
//           (hub bitmaps and overlapping lists make that the common case); the rest go through
//           atomicOr, whose return value tells whether THIS thread turned the bit on -- summing
//           those gives |hop2| exactly, with no separate popcount pass over the bitmap.
//   OP_TEST membership test of the intersection phase (cnt = hits, acc = weighted hits).
enum { OP_SET = 0, OP_TEST = 2 };

template <int OP, bool RANGED>
__device__ __forceinline__ void touch(unsigned* bm, int id, unsigned wt, unsigned& cnt,
                                      unsigned long long& acc, int n_side, int lo, int range_bits) {
    if (RANGED) {
        // only ids of the current range [lo, lo + range_bits) have a bit in shared memory
        const unsigned rel = (unsigned)(id - lo);
        const bool in = rel < (unsigned)range_bits;
        volatile unsigned* w = bm + (rel >> 5);
        if (OP == OP_SET) {
            const unsigned bit = 1u << (rel & 31);
            if (in && id < n_side && !(*w & bit)) {
                const unsigned old = atomicOr(const_cast<unsigned*>(w), bit);
                cnt += !(old & bit);
            }
        } else if (in) {
            const unsigned hit = (*w >> (rel & 31)) & 1u;
            cnt += hit;
            acc += (unsigned long long)hit * (unsigned long long)wt;
        }
        return;
    }
    volatile unsigned* w = bm + (id >> 5);
    if (OP == OP_SET) {
        const unsigned bit = 1u << (id & 31);
        if (id < n_side && !(*w & bit)) {          // padding sentinels are never set
            const unsigned old = atomicOr(const_cast<unsigned*>(w), bit);
            cnt += !(old & bit);
        }
    } else {
        // branch-free: the weight rides in the stream next to the id, so a hit costs one
        // integer multiply-add (IMAD.WIDE) instead of a divergent 8-byte gather
        const unsigned hit = (*w >> (id & 31)) & 1u;
        cnt += hit;
        acc += (unsigned long long)hit * (unsigned long long)wt;
    }
}

template <int OP, bool RANGED>
__device__ __forceinline__ void touch4(unsigned* bm, int4 v, uint4 wt, unsigned& cnt,
                                       unsigned long long& acc, int n_side, int lo, int range_bits,
                                       TileSmem* list, int self) {
    if (OP == OP_SET) {
        // four probes first, then the atomics that are still needed, all in flight together
        const int id[4] = {v.x, v.y, v.z, v.w};
        unsigned rel[4], bit[4], old[4];
        bool need[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            rel[k] = RANGED ? (unsigned)(id[k] - lo) : (unsigned)id[k];
            bit[k] = 1u << (rel[k] & 31);
            need[k] = id[k] < n_side && (!RANGED || rel[k] < (unsigned)range_bits);
            old[k] = need[k] ? *(volatile unsigned*)(bm + (rel[k] >> 5)) : 0xffffffffu;
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            need[k] = need[k] && !(old[k] & bit[k]);
            if (need[k]) old[k] = atomicOr(bm + (rel[k] >> 5), bit[k]);
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const bool turned_on = need[k] && !(old[k] & bit[k]);
            cnt += turned_on;
            if (!RANGED && list && turned_on && id[k] != self)   // hop2(x) excludes x
                list->hub[atomicAdd(&list->list_n, 1)] = id[k];
        }
        return;
    }
    touch<OP, RANGED>(bm, v.x, wt.x, cnt, acc, n_side, lo, range_bits);
    touch<OP, RANGED>(bm, v.y, wt.y, cnt, acc, n_side, lo, range_bits);
    touch<OP, RANGED>(bm, v.z, wt.z, cnt, acc, n_side, lo, range_bits);
    touch<OP, RANGED>(bm, v.w, wt.w, cnt, acc, n_side, lo, range_bits);
}

// Walks the `count` adjacency lists described by ts.row[] (ts.scan[] already holds the chunk
// prefix of the long ones).  Short lists: 4 lanes per list, 8 lists per warp pass.  Long lists:
// 512-id chunks dealt round-robin to warps, so a hub list is spread over the whole CTA.
template <int NT, int OP, bool RANGED>
__device__ __forceinline__ unsigned sweep_tile(const SideArgs& a, unsigned* bm, TileSmem& ts,
                                               int count, int lane, int warp, int lo, int self,
                                               unsigned long long pol) {
    unsigned set_total = 0;   // OP_SET: bits this thread turned on
    TileSmem* const list = (OP == OP_SET && !RANGED && ts.list_on) ? &ts : nullptr;
    constexpr int NW = NT / 32;
    const int4* adj4 = reinterpret_cast<const int4*>(a.m_adj);
    const uint4* adjw4 = reinterpret_cast<const uint4*>(a.m_adjw);
    const int4 sent4 = make_int4(a.n_side, a.n_side, a.n_side, a.n_side);
    const uint4 zero4 = make_uint4(0u, 0u, 0u, 0u);
    // ---- short lists
    {
        const int sub = lane & 3, slot = lane >> 2;
        for (int base = warp * 8; base < count; base += NW * 8) {
            const int j = base + slot;
            const unsigned long long row = j < count ? ts.row[j] : 0ull;
            const int n4 = (row_deg(row) + 3) >> 2;
            const bool is_short = n4 > 0 && n4 <= kShortV4;
            const bool mine = is_short && sub < n4;
            if (!__any_sync(kFull, mine)) continue;
            unsigned cnt = 0;
            unsigned long long acc = 0ull;
            if (mine) {
                const long long at = row_first4(row) + sub;
                int4 v = ldg_stream(adj4 + at, pol);
                uint4 wt = OP == OP_TEST ? ldg_stream_u(adjw4 + at, pol) : zero4;
                touch4<OP, RANGED>(bm, v, wt, cnt, acc, a.n_side, lo, a.range_bits, list, self);
            }
            if (OP == OP_SET) set_total += cnt;
            if (OP == OP_TEST) {
                cnt += __shfl_xor_sync(kFull, cnt, 1);
                cnt += __shfl_xor_sync(kFull, cnt, 2);
                if (__any_sync(kFull, cnt > 0)) {
                    acc += __shfl_xor_sync(kFull, acc, 1);
                    acc += __shfl_xor_sync(kFull, acc, 2);
                }
                if (is_short && sub == 0) {
                    ts.cn[j] = (int)cnt;
                    ts.aa[j] = acc;
                }
            }
        }
    }
    // ---- probe pairs: one warp per pair, the hop-2 id list against the partner's bitmap
    if (OP == OP_TEST && !RANGED) {
        const int np = ts.nprobe;
        if (np > 0) {
            const int nl = ts.list_n;
            for (int q = warp; q < np; q += NW) {
                const int j = ts.probe[q];
                const unsigned* hb =
                    a.hub_bm + (size_t)(row_slot1(ts.row[j]) - 1) * (size_t)a.hub_words;
                unsigned cnt = 0;
                unsigned long long acc = 0ull;
                for (int i0 = lane; i0 < nl; i0 += 128) {
                    int w[4];
                    unsigned word[4];
#pragma unroll
                    for (int k = 0; k < 4; ++k)   // bit n_side is never on in a hub bitmap
                        w[k] = i0 + 32 * k < nl ? ts.hub[i0 + 32 * k] : a.n_side;
#pragma unroll
                    for (int k = 0; k < 4; ++k) word[k] = ldg_keep(hb + (w[k] >> 5), pol);
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        if ((word[k] >> (w[k] & 31)) & 1u) {
                            ++cnt;
                            acc += ldg_keep(a.node_wt + w[k], pol);
                        }
                }
                cnt = __reduce_add_sync(kFull, cnt);
                if (cnt > 0) {   // per-lane acc < 24 * 2^31: the two REDUX halves add it exactly
                    const unsigned lo16 = __reduce_add_sync(kFull, (unsigned)(acc & 0xffffull));
                    const unsigned hi = __reduce_add_sync(kFull, (unsigned)(acc >> 16));
                    acc = ((unsigned long long)hi << 16) + lo16;
                }
                if (lane == 0) {
                    ts.cn[j] = (int)cnt;
                    ts.aa[j] = cnt > 0 ? acc : 0ull;
                }
            }
        }
    }
    // ---- long lists
    const int total = ts.scan[kTile];
    // warp w starts on chunk w without asking; further chunks come from the shared-memory
    // dispenser (it starts at NW), which is only touched when there are more chunks than warps
    int c = warp;
    const bool dynamic = total > NW;
    while (c < total) {
        // claim the following chunk now: the dispenser's latency hides behind this chunk
        int c_next = total;
        if (dynamic && lane == 0) c_next = atomicAdd(&ts.next_chunk[OP], 1);
        const int j = find_list(ts, c, lane);
        const unsigned long long row = ts.row[j];
        const int off4 = (c - ts.scan[j]) * kChunkV4;
        const int n = min(kChunkV4, ((row_deg(row) + 3) >> 2) - off4);
        const long long at = row_first4(row) + off4;
        unsigned cnt = 0;
        unsigned long long acc = 0ull;
        // two halves of 256 ids: four 128-bit loads in flight per lane, half the registers
#pragma unroll
        for (int half = 0; half < kChunkV4 / 64; ++half) {
            if (64 * half < n) {
                int4 v[2];
                uint4 wt[2];
#pragma unroll
                for (int k = 0; k < 2; ++k) {
                    const int i = lane + 32 * (2 * half + k);
                    v[k] = i < n ? ldg_stream(adj4 + at + i, pol) : sent4;
                    wt[k] = (OP == OP_TEST && i < n) ? ldg_stream_u(adjw4 + at + i, pol) : zero4;
                }
#pragma unroll
                for (int k = 0; k < 2; ++k)
                    if (32 * (2 * half + k) < n)
                        touch4<OP, RANGED>(bm, v[k], wt[k], cnt, acc, a.n_side, lo, a.range_bits, list,
                                           self);
            }
        }
        if (OP == OP_SET) set_total += cnt;
        if (OP == OP_TEST) {
            const bool single = ((row_deg(row) + 3) >> 2) <= kChunkV4;   // whole list in this chunk
            if (single || __any_sync(kFull, cnt > 0)) {
                cnt = __reduce_add_sync(kFull, cnt);
                // per-lane acc < 16 * 2^31: two 32-bit warp reductions (REDUX) add it exactly
                const unsigned lo16 = __reduce_add_sync(kFull, (unsigned)(acc & 0xffffull));
                const unsigned hi = __reduce_add_sync(kFull, (unsigned)(acc >> 16));
                acc = ((unsigned long long)hi << 16) + lo16;
                if (lane == 0) {
                    if (single) {
                        ts.cn[j] = (int)cnt;
                        ts.aa[j] = acc;
                    } else {
                        atomicAdd(&ts.cn[j], (int)cnt);
                        atomicAdd(&ts.aa[j], acc);
                    }
                }
            }
        }
        c = dynamic ? __shfl_sync(kFull, c_next, 0) : total;
    }
    return set_total;
}

__device__ __forceinline__ int long_chunks(unsigned long long row) {
    const int n4 = (row_deg(row) + 3) >> 2;
    return n4 > kShortV4 ? (n4 + kChunkV4 - 1) / kChunkV4 : 0;
}

#ifdef BLP_PHASE_TIMING
__device__ unsigned long long g_phase_cycles[16];
#define BLP_TICK(slot)                                                        \
    do {                                                                      \
        if (tid == 0) {                                                       \
            long long now__ = clock64();                                      \
            atomicAdd(&g_phase_cycles[slot], (unsigned long long)(now__ - t_last)); \
            t_last = now__;                                                   \
        }                                                                     \
    } while (0)
#else
#define BLP_TICK(slot) do {} while (0)
#endif

#ifndef BLP_THREADS_PER_SM
#define BLP_THREADS_PER_SM 1024
#endif


// Descriptor of one work item (group) as the kernel carries it in registers.  The uniform part
// of the chain  item -> node -> (pair range, row)  is fetched for the NEXT group in two stages
// spread over the current group's phases, so it is off the critical path when the group starts;
// the first pair tile's gathers are issued at group start and parked in shared memory while the
// expansion runs.
struct GroupRegs {
    int item;                   // index into item_key, >= n_items when there is no group
    int x;                      // grouping node; n_side = the "not in graph" bucket
    int p0, p1;                 // pair range of the group in grouped order
    unsigned long long xrow;    // row descriptor of x
    int m;                      // this thread's neighbour of x in the first expansion tile, or -1
    unsigned long long rowx;    // expansion-side descriptor of m (0 when there is none)
};

__device__ __forceinline__ void stage4(const SideArgs& a, GroupRegs& g) {
    g.rowx = g.m >= 0 ? a.m_xrow[g.m] : 0ull;
}

__device__ __forceinline__ void stage3(const SideArgs& a, GroupRegs& g, int tid) {
    g.m = -1;
    if (g.x < a.n_side && tid < min(kTile, row_deg(g.xrow)))
        g.m = a.g_adj[row_first4(g.xrow) * 4 + tid];
}

__device__ __forceinline__ void stage1(const SideArgs& a, GroupRegs& g, int n_items) {
    g.x = a.n_side + 1;
    g.p0 = g.p1 = 0;
    if (g.item < n_items) {
        const int it = a.item_list ? a.item_list[g.item] : g.item;
        g.x = a.item_key[it];
        g.p0 = a.item_start[it];
        g.p1 = a.item_end[it];
    }
}
__device__ __forceinline__ void stage2(const SideArgs& a, GroupRegs& g) {
    g.xrow = g.x < a.n_side ? a.g_row[g.x] : 0ull;
}

template <int NT, bool RANGED, bool REC>
__global__ void __launch_bounds__(NT, (BLP_THREADS_PER_SM / NT) > 0 ? (BLP_THREADS_PER_SM / NT) : 1)
    k_score_side(SideArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    unsigned* bm = reinterpret_cast<unsigned*>(smem_raw);
    TileSmem& ts = *reinterpret_cast<TileSmem*>(smem_raw + (size_t)a.bm_words * 4);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int n_items = *a.n_items;
    if (*a.mode == MODE_RUNS) {   // kernel parameters are per-thread copies: patch them locally
        a.pg = nullptr;
    }
    const unsigned long long pol = l2_keep_policy();
    unsigned hub_phase = 0;   // parity of ts.hub_bar's current phase (uniform across the CTA)

#ifdef BLP_PHASE_TIMING
    long long t_last = clock64();
#endif
    int ahead = 0;   // thread 0: the claim that becomes the next group's item at the next group start
    if (tid == 0) {
        mbar_init(&ts.hub_bar, 1);
        ts.item_next = atomicAdd(a.work_counter, 1);
        ahead = atomicAdd(a.work_counter, 1);
        ts.nhub = 0;
        ts.hop2cnt = 0;
        ts.list_on = 0;
        ts.list_n = 0;
        ts.nprobe = 0;
    }
    {
        uint4* b4 = reinterpret_cast<uint4*>(bm);
        const int n4 = a.bm_words >> 2;
        for (int i = tid; i < n4; i += NT) b4[i] = make_uint4(0u, 0u, 0u, 0u);
    }
#if BLP_HUB_TMA
    fence_async_smem();   // the clear (and the barrier's init) before any bulk copy into the bitmap
#endif
    __syncthreads();
    GroupRegs cur;
    cur.item = ts.item_next;
    stage1(a, cur, n_items);
    stage2(a, cur);
    stage3(a, cur, tid);
    stage4(a, cur);

    while (cur.item < n_items) {
        BLP_TICK(0);
        // claim the next item now; its descriptor is fetched in stages below
        // work-queue claims run TWO groups ahead: the index published for the next group was
        // claimed during the previous group, so the global atomic's round trip (issued here for
        // the group after next) is never waited for
        const int claimed = ahead;
        if (tid == 0) ahead = atomicAdd(a.work_counter, 1);
        GroupRegs nxt;
        const int x = cur.x;
        const long long p0 = cur.p0, p1 = cur.p1;

        if (x >= a.n_side) {
            // pairs with an id that is not in the graph: every score is the literal 0
            for (long long k = p0 + tid; k < p1; k += NT) {
                int idx = a.pg ? a.pg[k].x : (int)k;
                emit_pair<REC>(a, k, idx, false, 0, 0, 0, 0, 0ull);
            }
            __syncthreads();                       // everyone is past reading ts.item_next
            if (tid == 0) ts.item_next = claimed;
            __syncthreads();
            nxt.item = ts.item_next;
            stage1(a, nxt, n_items);
            stage2(a, nxt);
            stage3(a, nxt, tid);
            stage4(a, nxt);
            cur = nxt;
            continue;
        }

        const unsigned long long xrow = cur.xrow;
        const int xdeg = row_deg(xrow);
        const int* xadj = a.g_adj + row_first4(xrow) * 4;
        if (tid == 0) ts.item_next = claimed;      // published by the first barrier below
        // gathers of the first pair tile: issued now, parked in shared memory after the hub pass
        unsigned long long park_row = 0ull;
        int park_idx = 0;
        if (tid < kTile && p0 + tid < p1) {
            const int2 iy = pair_at(a, p0 + tid);
            park_row = a.m_row[iy.y];
            park_idx = iy.x;
        }

        const int n_ranges = RANGED ? a.n_ranges : 1;
        for (int pass = 0; pass < n_ranges; ++pass) {
        const int lo = RANGED ? pass * a.range_bits : 0;
        // ---- phases 0+1: two-hop expansion, hop2(x) = U N(m) over m in N(x).
        // Hub lists arrive as precomputed bitmaps and are OR-ed with 128-bit loads by the thread
        // that owns the word (for the first tile this pass doubles as the clear); every other
        // list is walked id by id (OP_SET).  Both count the bits they turn on.
        for (int tb = 0; tb < xdeg; tb += kTile) {
            const int count = min(kTile, xdeg - tb);
            int nch = 0;
            int list_len = 0;
            if (tid < count) {
                const int m_id = tb == 0 ? cur.m : xadj[tb + tid];   // (the first tile's neighbour is in a register)
                unsigned long long row = (tb == 0 && pass == 0) ? cur.rowx : a.m_xrow[m_id];
                list_len = min(row_deg(row), kProbeCap + 1);
                if (row >> 63) {
                    const int h = atomicAdd(&ts.nhub, 1);
                    ts.hub[h] = (int)((row >> 24) & (unsigned long long)BLP_ROW_MAX_SLOTS);
                    ts.cn[h] = row_deg(row);   // ts.cn is idle during the expansion
                    row = 0ull;                // degree 0: skipped by both list walkers
                    list_len = kProbeCap + 1;
                } else if (RANGED) {
                    row = segment_row(a, row, m_id, pass);   // only this range's part of the list
                }
                ts.row[tid] = row;
                nch = long_chunks(row);
            }
            if (!RANGED && tb == 0 && warp == 0) {
                // probe path: keep hop2(x) as a list when x's whole expansion is this warp's, has
                // no hub and walks at most kProbeCap ids (published by tile_scan's barrier)
                const int walked = __reduce_add_sync(kFull, list_len);
                if (lane == 0)
                    ts.list_on = (a.node_wt != nullptr && xdeg <= 32 && walked <= kProbeCap) ? 1 : 0;
            }
            tile_scan<NT>(ts, nch, tid, count);
            if (pass == 0 && tb == 0) {            // stage 1 of the next group's descriptor
                nxt.item = ts.item_next;
                stage1(a, nxt, n_items);
            }
            BLP_TICK(1);
            int newbits = 0;
            {
                const int nhub = ts.nhub;
                uint4* b4 = reinterpret_cast<uint4*>(bm);
                const uint4* h4 = reinterpret_cast<const uint4*>(a.hub_bm);
                const int n4 = a.bm_words >> 2;   // bm_words is a multiple of 4
                const int hub4 = a.hub_words >> 2, lo4 = lo >> 7;
                int first_reg = 0;   // hubs [first_reg, nhub) go through registers
                // (the bitmap arrives all-zero: cleared at kernel start and after every group)
                if (nhub == 0) {
                    // nothing to OR, and no barrier needed before the list walk
                } else if (tb == 0 && !RANGED) {
                    // first hub of the first tile: ONE TMA bulk copy (cp.async.bulk, UBLKCP) of the
                    // hub's whole bitmap straight over the (all-zero) shared bitmap, issued by one
                    // thread and completing on an mbarrier -- no thread spends issue slots or
                    // registers on the 46 KB, and it turns on exactly deg(hub) bits.  The clear
                    // that precedes it was fenced for the async proxy where it was written.
#if BLP_HUB_TMA
                    if (tid == 0) {
                        const unsigned bytes = (unsigned)a.bm_words * 4u;
                        mbar_expect_tx(&ts.hub_bar, bytes);
                        bulk_copy_g2s(bm, h4 + (size_t)ts.hub[0] * hub4, bytes, &ts.hub_bar);
                        newbits += ts.cn[0];
                    }
                    first_reg = 1;
                    mbar_wait(&ts.hub_bar, hub_phase);   // every thread: the bytes have landed
                    hub_phase ^= 1u;
#else
                    // (A/B build: the Ampere-style copy, 16 bytes per cp.async, every thread issuing)
                    const uint4* src = h4 + (size_t)ts.hub[0] * hub4;
                    for (int i = tid; i < n4; i += NT) {
                        const unsigned dst = (unsigned)__cvta_generic_to_shared(b4 + i);
                        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src + i)
                                     : "memory");
                    }
                    asm volatile("cp.async.commit_group;" ::: "memory");
                    if (tid == 0) newbits += ts.cn[0];
                    first_reg = 1;
                    asm volatile("cp.async.wait_group 0;" ::: "memory");
                    (void)hub_phase;
#endif
                }
                if (nhub > first_reg) {
                    const bool fresh = false;   // words are valid (zero or earlier hubs / tiles)
                    // two independent 128-bit loads in flight per thread and hub
                    for (int i0 = tid; i0 < n4; i0 += 2 * NT) {
                        const int i1 = i0 + NT;
                        const bool ok1 = i1 < n4;
                        uint4 acc0 = fresh ? make_uint4(0u, 0u, 0u, 0u) : b4[i0];
                        uint4 acc1 = (fresh || !ok1) ? make_uint4(0u, 0u, 0u, 0u) : b4[i1];
                        newbits -= __popc(acc0.x) + __popc(acc0.y) + __popc(acc0.z) + __popc(acc0.w) +
                                   __popc(acc1.x) + __popc(acc1.y) + __popc(acc1.z) + __popc(acc1.w);
                        for (int h = first_reg; h < nhub; ++h) {
                            const uint4* src = h4 + (size_t)ts.hub[h] * hub4 + lo4;
                            const uint4 q0 = lo4 + i0 < hub4 ? ldg_keep(src + i0, pol)
                                                             : make_uint4(0u, 0u, 0u, 0u);
                            const uint4 q1 = (ok1 && lo4 + i1 < hub4) ? ldg_keep(src + i1, pol)
                                                                      : make_uint4(0u, 0u, 0u, 0u);
                            acc0.x |= q0.x;
                            acc0.y |= q0.y;
                            acc0.z |= q0.z;
                            acc0.w |= q0.w;
                            acc1.x |= q1.x;
                            acc1.y |= q1.y;
                            acc1.z |= q1.z;
                            acc1.w |= q1.w;
                        }
                        newbits += __popc(acc0.x) + __popc(acc0.y) + __popc(acc0.z) + __popc(acc0.w) +
                                   __popc(acc1.x) + __popc(acc1.y) + __popc(acc1.z) + __popc(acc1.w);
                        b4[i0] = acc0;
                        if (ok1) b4[i1] = acc1;
                    }
                }
            }
            if (pass == 0 && tb == 0 && tid < kTile) {
                // ts.idx / ts.aa are idle until phase 3: the first pair tile waits there
                ts.idx[tid] = park_idx;
                ts.aa[tid] = park_row;
            }
            if (ts.nhub > 0) {                // uniform: written before tile_scan's barrier
                __syncthreads();              // plain hub stores before the atomics of the walk
                if (tid == 0) ts.nhub = 0;
            }
            if (pass == 0 && tb == 0) stage2(a, nxt);
            BLP_TICK(2);
            newbits += (int)sweep_tile<NT, OP_SET, RANGED>(a, bm, ts, count, lane, warp, lo, x, pol);
            newbits = __reduce_add_sync(kFull, newbits);
            if (lane == 0 && newbits != 0) atomicAdd(&ts.hop2cnt, newbits);
            __syncthreads();
            if (pass == 0 && tb == 0) stage3(a, nxt, tid);
            BLP_TICK(3);
        }

        // ---- phase 2: x itself is in every N(m), so its bit is always on: |hop2(x)| = bits - 1
        // (with id ranges the count is complete once the last pass has expanded)
        const int hop2 = ts.hop2cnt - 1;
        const bool probing = !RANGED && ts.list_on;   // then ts.hub[0 .. hop2) lists hop2(x)
        if (tid == 0) {   // ordered before the tests by tile_scan's barriers
            const unsigned rel = (unsigned)(x - lo);
            if (!RANGED || rel < (unsigned)a.range_bits) bm[rel >> 5] &= ~(1u << (rel & 31));
        }
        BLP_TICK(5);

        // ---- phase 3: every pair (x, y) of the group: stream N(y), test, count, weigh
        for (long long tb = p0; tb < p1; tb += kTile) {
            const int count = (int)min((long long)kTile, p1 - tb);
            int nch = 0;
            if (tid < count) {
                const bool first = !RANGED && tb == p0 && pass == 0;
                unsigned long long row;
                if (first) {
                    row = ts.aa[tid];
                } else {
                    const int2 iy = pair_at(a, tb + tid);
                    row = a.m_row[iy.y];
                    ts.idx[tid] = iy.x;
                    if (RANGED) {
                        ts.hub[tid] = row_deg(row);              // deg(y) for the epilogue (hub[] is idle here)
                        row = segment_row(a, row, iy.y, pass);   // only this range's part of N(y)
                    }
                }
                ts.row[tid] = row;
                ts.cn[tid] = 0;
                ts.aa[tid] = 0ull;
                nch = long_chunks(row);
                if (probing && row_slot1(row) > 0 && (long long)a.probe_ratio * hop2 <= row_deg(row)) {
                    ts.probe[atomicAdd(&ts.nprobe, 1)] = (unsigned char)tid;
                    nch = 0;   // not streamed (a list this long is never on the short path)
                }
            }
            tile_scan<NT>(ts, nch, tid, count);
            if (pass == 0 && tb == p0) stage4(a, nxt);
            BLP_TICK(6);
            sweep_tile<NT, OP_TEST, RANGED>(a, bm, ts, count, lane, warp, lo, x, pol);
            __syncthreads();
            if (!RANGED && tid == 0) ts.nprobe = 0;   // next use is behind the barrier below
            BLP_TICK(7);
            // epilogue: one thread per pair of the tile
            bool final_pass = true;
            if (RANGED && tid < count) {
                // partial sums of earlier ranges wait in scratch; only the last pass emits
                if (pass > 0) {
                    ts.cn[tid] += a.acc_cn[tb + tid];
                    ts.aa[tid] += a.acc_aa[tb + tid];
                }
                final_pass = pass == n_ranges - 1;
                if (!final_pass) {
                    a.acc_cn[tb + tid] = ts.cn[tid];
                    a.acc_aa[tb + tid] = ts.aa[tid];
                }
            }
            if (tid < count && final_pass) {
                const int pdeg = RANGED ? ts.hub[tid] : row_deg(ts.row[tid]);
                emit_pair<REC>(a, tb + tid, ts.idx[tid], true, ts.cn[tid], hop2, xdeg, pdeg, ts.aa[tid]);
            }
            __syncthreads();
            BLP_TICK(8);
        }
        // leave the bitmap all-zero for the next group / pass (ordered by its tile_scan barrier)
        {
            uint4* b4 = reinterpret_cast<uint4*>(bm);
            const int n4 = a.bm_words >> 2;
            for (int i = tid; i < n4; i += NT) b4[i] = make_uint4(0u, 0u, 0u, 0u);
#if BLP_HUB_TMA
            fence_async_smem();   // ... before the next group's bulk copy may land on these words
#endif
        }
        }   // id-range passes
        if (tid == 0) {   // ordered before the next group's counting by its barriers
            ts.hop2cnt = 0;
            ts.list_n = 0;
        }
        cur = nxt;
    }
}


template <int NT, bool RANGED, bool REC>
static int launch_side(const SideArgs& a, int grid, size_t smem, cudaStream_t st) {
    // (the dynamic shared-memory opt-in covers this size: raise_smem_optin<>() ran just before)
    k_score_side<NT, RANGED, REC><<<grid, NT, smem, st>>>(a);
    BLP_CUDA_TRY(cudaGetLastError());
    return BLP_OK;
}

// The dynamic shared-memory opt-in is a property of (kernel, device) for the whole PROCESS, not of
// a graph handle: handles of different size share it.  It is kept in a process-wide table and only
// ever raised, so a small graph scored between two calls on a large one cannot lower it.
constexpr int kMaxDevices = 64;
static std::mutex g_optin_mutex;
template <int NT, bool RANGED, bool REC>
static int raise_smem_optin(int device, size_t smem) {
    static size_t granted[kMaxDevices] = {};
    std::lock_guard<std::mutex> lock(g_optin_mutex);
    if (device < 0 || device >= kMaxDevices || smem > granted[device]) {
        BLP_CUDA_TRY(cudaFuncSetAttribute(k_score_side<NT, RANGED, REC>,
                                          cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        if (device >= 0 && device < kMaxDevices) granted[device] = smem;
    }
    return BLP_OK;
}

template <int NT, bool RANGED, bool REC>
static int occupancy(size_t smem, int* ctas_per_sm) {
    BLP_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(
        ctas_per_sm, k_score_side<NT, RANGED, REC>, NT, smem));
    return BLP_OK;
}

// The bitmap must hold bits 0..n_side (the last one is the padding sentinel).  When that does not
// fit in one CTA's shared memory the id universe is cut into equal ranges and every group is
// processed once per range (BLP_RANGES forces a count, for tuning / tests).
void range_plan(int n_side, int smem_optin, int forced, int* n_ranges_out, int* range_words_out) {
    const int full_words = bitmap_words(n_side);
    const long long cap_words = (((long long)smem_optin - (long long)sizeof(TileSmem) - 256) / 4) & ~3LL;
    int n_ranges = (int)((full_words + cap_words - 1) / cap_words);
    n_ranges = std::max(n_ranges, forced);
    int range_words = full_words;
    if (n_ranges > 1) {
        range_words = (int)((((long long)full_words + n_ranges - 1) / n_ranges + 3) & ~3LL);
        n_ranges = (full_words + range_words - 1) / range_words;
    }
    *n_ranges_out = n_ranges;
    *range_words_out = range_words;
}

// One CTA per hub: write its neighbour list into its (already zeroed) bitmap.
__global__ void k_build_hub_bitmaps(const int* __restrict__ hub_nodes, int n_hubs,
                                    const unsigned long long* __restrict__ m_row,
                                    const int* __restrict__ m_adj, int bm_words,
                                    unsigned* __restrict__ hub_bm) {
    for (int h = blockIdx.x; h < n_hubs; h += gridDim.x) {
        const unsigned long long row = m_row[hub_nodes[h]];
        const int* adj = m_adj + row_first4(row) * 4;
        unsigned* bm = hub_bm + (size_t)h * bm_words;
        for (int i = threadIdx.x; i < row_deg(row); i += blockDim.x) {
            const int id = adj[i];
            atomicOr(bm + (id >> 5), 1u << (id & 31));
        }
    }
}

// Picks the hubs of both sides and builds their bitmaps on the device.
// Cost model (measured on C2, profiles/r01_notes.md): walking a list costs ~0.35 L1 wavefronts per
// id (two sweeps, bank-conflicted bitmap probes), OR-ing a bitmap costs bm_bytes/128 wavefronts,
// so by that model a list pays off as a bitmap from deg >= bm_bytes/45 on; measured on C2 with the
// final list walker (batched probes, counted atomics) the optimum sits at bm_bytes/30
// (user side: deg >= 1016 6.71 ms, >= 1500 6.50 ms, >= 2500 6.56 ms; business side flat).
int build_hub_bitmaps(blp_graph* g, const int* u_deg_host, const int* b_deg_host) {
    reserve_biz_index(g);   // first: with an index the business side needs no tables or flags
    for (int side = 0; side < 2; ++side) {
        const bool us = side == BLP_SIDE_USER;
        const int n_side = us ? g->n_users : g->n_biz;     // bitmap universe
        const int n_mid = us ? g->n_biz : g->n_users;      // hubs are middle nodes
        const int* mdeg = us ? b_deg_host : u_deg_host;
        const int words = bitmap_words(n_side);
        const long long bm_bytes = (long long)words * 4;
        // (round 2, with the hub copy done by TMA: C2 -- 46 KB bitmap -- 700..1000 flat and 3 % better
        // than 1525; C3 / C4 -- 200 KB bitmap, one CTA per SM -- 6667 better than 4500 and 3000)
        int min_deg = (int)std::max<long long>(64, bm_bytes <= 65536 ? bm_bytes / 50 : bm_bytes / 30);
        if (const char* e = getenv("BLP_HUB_MIN_DEG")) min_deg = atoi(e);   // tuning override
        // Bitmaps used only by the intersection's probe path start lower: a probe costs about as
        // much as a streamed id, and the path is taken when deg(y) >= kProbeRatio * |hop2(x)|
        // with |hop2(x)| <= kProbeCap, so a bitmap pays off from a few hundred ids on.
        int probe_deg = min_deg > 0 ? std::max(64, min_deg / 3) : 0;
        if (const char* e = getenv("BLP_PROBE_MIN_DEG")) probe_deg = atoi(e);   // 0 = path off
        // the slot field needs every first-entry index to fit BLP_ROW_FIRST4_BITS
        const long long mid_entries = us ? g->b_adj_len : g->u_adj_len;
        const bool slots_fit = mid_entries / 4 < (1LL << BLP_ROW_FIRST4_BITS);
        if (probe_deg <= 0 || !slots_fit) probe_deg = 0;
        else probe_deg = std::max(64, min_deg > 0 ? std::min(probe_deg, min_deg) : probe_deg);
        const int any_deg = probe_deg > 0 ? probe_deg : min_deg;   // a bitmap exists from here on
        std::vector<int> hubs;
        if (any_deg > 0)
            for (int m = 0; m < n_mid; ++m)
                if (mdeg[m] >= any_deg) hubs.push_back(m);
        // budget: at most BLP_ROW_MAX_SLOTS bitmaps and 2 GiB per side; keep the largest
        size_t cap = (size_t)std::min<long long>(BLP_ROW_MAX_SLOTS, (2LL << 30) / bm_bytes);
        if (hubs.size() > cap) {
            std::sort(hubs.begin(), hubs.end(), [&](int a, int b) { return mdeg[a] > mdeg[b]; });
            hubs.resize(cap);
            std::sort(hubs.begin(), hubs.end());
        }
        g->n_hubs[side] = (int)hubs.size();
        g->hub_min_deg[side] = min_deg > 0 ? min_deg : 0x7fffffff;
        g->probe_min_deg[side] = any_deg > 0 ? any_deg : 0x7fffffff;
        if (hubs.empty()) continue;
        const bool probing = probe_deg > 0;
        // expansion-side descriptors: a copy of the middle rows with the hubs' entries replaced
        const unsigned long long* d_mrow = (const unsigned long long*)(us ? g->b_row : g->u_row);
        std::vector<unsigned long long> xrow((size_t)n_mid);
        BLP_CUDA_TRY(cudaMemcpy(xrow.data(), d_mrow, sizeof(unsigned long long) * (size_t)n_mid,
                                cudaMemcpyDeviceToHost));
        // the middle rows themselves learn which of them has a bitmap (read by the intersection)
        std::vector<unsigned long long> mrow;
        if (probing) mrow = xrow;
        std::vector<int> or_nodes;   // the hubs the expansion ORs, in table-row order
        for (size_t h = 0; h < hubs.size(); ++h) {
            if (probing) mrow[hubs[h]] |= (unsigned long long)(h + 1) << BLP_ROW_SLOT_SHIFT;
            if (min_deg > 0 && mdeg[hubs[h]] >= min_deg) {   // the expansion ORs this one
                xrow[hubs[h]] = (1ull << 63) |
                                ((unsigned long long)or_nodes.size() << BLP_XROW_ORIDX_SHIFT) |
                                ((unsigned long long)h << 24) | (unsigned)mdeg[hubs[h]];
                or_nodes.push_back(hubs[h]);
            }
        }
        if (probing) {
            BLP_CUDA_TRY(cudaMemcpy(const_cast<unsigned long long*>(d_mrow), mrow.data(),
                                    sizeof(unsigned long long) * (size_t)n_mid,
                                    cudaMemcpyHostToDevice));
            // Q1.31 weight of every grouping-side node: a probe hit adds the weight of the id
            const int* gdeg = us ? u_deg_host : b_deg_host;
            std::vector<unsigned> lut;
            weight_lut(us ? g->max_udeg : g->max_bdeg, lut);
            std::vector<unsigned> wt((size_t)n_side + 1, 0u);
            for (int i = 0; i < n_side; ++i) wt[i] = lut[gdeg[i]];
            BLP_CUDA_TRY(cudaMalloc((void**)&g->node_wt[side], sizeof(unsigned) * wt.size()));
            BLP_CUDA_TRY(cudaMemcpy(g->node_wt[side], wt.data(), sizeof(unsigned) * wt.size(),
                                    cudaMemcpyHostToDevice));
            g->device_bytes += (int64_t)(sizeof(unsigned) * wt.size());
            g->row_slots[side] = true;
            g->probe_ratio = kProbeRatio;
            if (const char* e = getenv("BLP_PROBE_RATIO")) g->probe_ratio = std::max(1, atoi(e));
        }
        int* d_nodes = nullptr;
        const size_t bytes = hubs.size() * (size_t)bm_bytes;
        BLP_CUDA_TRY(cudaMalloc((void**)&g->xrow[side], sizeof(unsigned long long) * (size_t)n_mid));
        BLP_CUDA_TRY(cudaMemcpy(g->xrow[side], xrow.data(),
                                sizeof(unsigned long long) * (size_t)n_mid, cudaMemcpyHostToDevice));
        BLP_CUDA_TRY(cudaMalloc((void**)&g->hub_bm[side], bytes));
        BLP_CUDA_TRY(cudaMemset(g->hub_bm[side], 0, bytes));
        BLP_CUDA_TRY(cudaMalloc((void**)&d_nodes, sizeof(int) * hubs.size()));
        BLP_CUDA_TRY(cudaMemcpy(d_nodes, hubs.data(), sizeof(int) * hubs.size(),
                                cudaMemcpyHostToDevice));
        k_build_hub_bitmaps<<<(int)std::min<size_t>(hubs.size(), 4096), 256>>>(
            d_nodes, (int)hubs.size(),
            (const unsigned long long*)(us ? g->b_row : g->u_row), us ? g->b_adj : g->u_adj,
            words, g->hub_bm[side]);
        BLP_CUDA_TRY(cudaGetLastError());
        BLP_CUDA_TRY(cudaDeviceSynchronize());
        cudaFree(d_nodes);
        g->device_bytes += (int64_t)bytes + (int64_t)sizeof(unsigned long long) * n_mid;
        // hub x bitmap-node intersection tables (for one-hub groups in the warp-per-group kernel);
        // skipped when they would take more than ~2e9 probes to fill
        long long or_ids = 0;
        for (int m : or_nodes) or_ids += mdeg[m];
        const bool grouped = us || !g->biz_index;   // the tables serve the grouped path only
        if (grouped && probing && !or_nodes.empty() && or_ids * (long long)hubs.size() <= 2000000000LL) {
            const size_t cells = or_nodes.size() * hubs.size();
            int* d_or = nullptr;
            BLP_CUDA_TRY(cudaMalloc((void**)&d_or, sizeof(int) * or_nodes.size()));
            BLP_CUDA_TRY(cudaMemcpy(d_or, or_nodes.data(), sizeof(int) * or_nodes.size(),
                                    cudaMemcpyHostToDevice));
            BLP_CUDA_TRY(cudaMalloc((void**)&g->hubtab_cn[side], sizeof(int) * cells));
            BLP_CUDA_TRY(cudaMalloc((void**)&g->hubtab_aa[side], sizeof(unsigned long long) * cells));
            k_hub_tables<<<dim3((unsigned)hubs.size(), (unsigned)or_nodes.size()), 256>>>(
                d_or, (int)hubs.size(), d_mrow, us ? g->b_adj : g->u_adj, g->hub_bm[side], words,
                g->node_wt[side], g->hubtab_cn[side], g->hubtab_aa[side]);
            BLP_CUDA_TRY(cudaGetLastError());
            BLP_CUDA_TRY(cudaDeviceSynchronize());
            cudaFree(d_or);
            g->device_bytes += (int64_t)(cells * 12);
        }
    }
    // which grouping nodes qualify for the warp-per-group kernel (BLP_LIGHT=0 turns it off)
    const char* le = getenv("BLP_LIGHT");
    if (!le || atoi(le) != 0) {
        for (int side = 0; side < 2; ++side) {
            const bool us = side == BLP_SIDE_USER;
            const int n_side = us ? g->n_users : g->n_biz;
            if (n_side <= 0 || (!us && g->biz_index)) continue;
            const unsigned long long* g_row = (const unsigned long long*)(us ? g->u_row : g->b_row);
            const unsigned long long* m_row = (const unsigned long long*)(us ? g->b_row : g->u_row);
            BLP_CUDA_TRY(cudaMalloc((void**)&g->light[side], (size_t)n_side));
            const char* he = getenv("BLP_LIGHT_HUBS");   // BLP_LIGHT_HUBS=0: hub-free groups only
            const int max_hubs = (g->hubtab_cn[side] && !(he && atoi(he) == 0)) ? 1 : 0;
            k_flag_light<<<(n_side + 255) / 256, 256>>>(
                n_side, g_row, us ? g->u_adj : g->b_adj,
                g->xrow[side] ? (const unsigned long long*)g->xrow[side] : m_row, max_hubs,
                g->light[side]);
            BLP_CUDA_TRY(cudaGetLastError());
            g->device_bytes += n_side;
        }
        BLP_CUDA_TRY(cudaDeviceSynchronize());
    }
    return build_biz_index(g, b_deg_host);
}

}  // namespace blp

extern "C" int blp_score_pairs(blp_graph* g, int side, const int32_t* pair_u, const int32_t* pair_b,
                               int64_t n, int32_t* cn, int32_t* uni, double* jaccard,
                               double* adamic, int64_t* pa, int32_t* hop2_size, void* stream) {
    using namespace blp;
    if (!g || (side != BLP_SIDE_USER && side != BLP_SIDE_BUSINESS) || n < 0 ||
        (n > 0 && (!pair_u || !pair_b))) {
        set_error("blp_score_pairs: bad argument");
        return BLP_ERR_INVALID;
    }
    if (n >= (int64_t)INT_MAX) {
        set_error("blp_score_pairs: at most 2^31-2 pairs per call; split the pair list");
        return BLP_ERR_UNSUPPORTED;
    }
    BLP_ON_DEVICE(g->device);
    cudaStream_t st = (cudaStream_t)stream;
    blp_score_stats_t& stats = g->stats[side];
    stats = blp_score_stats_t{};
    stats.n_pairs = n;
    g->ev_recorded[side] = false;
    g->ev_light[side] = false;
    if (n == 0) return BLP_OK;

    const bool us = side == BLP_SIDE_USER;
    SideArgs a{};
    a.g_row = (const unsigned long long*)(us ? g->u_row : g->b_row);
    a.g_adj = us ? g->u_adj : g->b_adj;
    a.m_row = (const unsigned long long*)(us ? g->b_row : g->u_row);
    a.m_adj = us ? g->b_adj : g->u_adj;
    const int* g_deg = us ? g->u_deg : g->b_deg;
    const int* m_deg = us ? g->b_deg : g->u_deg;
    a.m_adjw = us ? g->b_adjw : g->u_adjw;
    a.m_xrow = g->xrow[side] ? (const unsigned long long*)g->xrow[side] : a.m_row;
    a.hub_bm = g->hub_bm[side];
    a.node_wt = g->row_slots[side] ? g->node_wt[side] : nullptr;
    a.probe_ratio = g->probe_ratio;
    a.hubtab_cn = g->hubtab_cn[side];
    a.hubtab_aa = g->hubtab_aa[side];
    a.hubtab_stride = g->n_hubs[side];
    a.n_side = us ? g->n_users : g->n_biz;
    const int n_mid = us ? g->n_biz : g->n_users;
    const int* gx = us ? pair_u : pair_b;
    const int* gy = us ? pair_b : pair_u;
    a.cn = cn;
    a.uni = uni;
    a.jac = jaccard;
    a.aa = adamic;
    a.pa = (long long*)pa;
    a.hop2 = hop2_size;
    if (!us && g->biz_index) return score_biz_indexed(g, a, pair_u, pair_b, n, st);

    // id-range passes: planned when the handle was created (range_plan), because the middle rows
    // of a ranged side are laid out partitioned by range
    const int full_words = bitmap_words(a.n_side);
    a.hub_words = full_words;
    const int n_ranges = g->n_ranges[side];
    const int range_words = g->range_words[side];
    const bool ranged = n_ranges > 1;
    if (ranged && !g->seg_off[side]) {
        set_error("blp_score_pairs: internal error: ranged side without range segments");
        return BLP_ERR_UNSUPPORTED;
    }
    a.seg_off = g->seg_off[side];
    a.seg_stride = n_ranges + 1;
    a.bm_words = range_words;
    a.range_bits = range_words * 32;
    a.n_ranges = n_ranges;
    const size_t smem = (size_t)a.bm_words * 4 + sizeof(TileSmem);
    if (smem > (size_t)g->max_smem_optin) {
        set_error("blp_score_pairs: internal error sizing the shared-memory bitmap");
        return BLP_ERR_UNSUPPORTED;
    }

    // ---- stream-ordered scratch + grouping
    const int n_keys = a.n_side + 1;
    std::vector<void*> scratch;
    // one stream-ordered block for all scratch of the call (an idle GPU would otherwise wait for
    // a dozen allocator calls before the first kernel): carved by a bump pointer, 256-byte aligned
    const size_t n_sz = (size_t)n, k_sz = (size_t)n_keys, i_sz = std::max(n_sz, k_sz);
    const size_t arena_bytes = 4 * n_sz + 20 * i_sz + 8 * k_sz + 12 * n_sz + 24 * n_sz +
                               (ranged ? 12 * n_sz : 0) + 8 * (k_sz / kScanTile + 1) + 64 * 256;
    unsigned char* arena = nullptr;
    size_t arena_used = 0;
    {
        cudaError_t e = pool_alloc(g, (void**)&arena, arena_bytes, st);
        if (e != cudaSuccess) return blp::cuda_fail(e, "cudaMallocFromPoolAsync(scratch)", __FILE__, __LINE__);
        scratch.push_back(arena);
    }
    auto alloc = [&](void** p, size_t bytes) -> cudaError_t {
        const size_t at = (arena_used + 255) & ~(size_t)255;
        if (at + bytes > arena_bytes) return cudaErrorMemoryAllocation;   // sizing bug, not OOM
        *p = arena + at;
        arena_used = at + bytes;
        return cudaSuccess;
    };
    auto release = [&]() {
        for (void* p : scratch) cudaFreeAsync(p, st);
        scratch.clear();
    };
#define BLP_TRY_SCRATCH(expr)                                                    \
    do {                                                                         \
        cudaError_t e__ = (expr);                                                \
        if (e__ != cudaSuccess) {                                                \
            release();                                                           \
            return blp::cuda_fail(e__, #expr, __FILE__, __LINE__);               \
        }                                                                        \
    } while (0)
    int *keys = nullptr, *scalars = nullptr, *inv = nullptr;
    int *item_key = nullptr, *item_start = nullptr, *item_end = nullptr;
    BLP_TRY_SCRATCH(alloc((void**)&keys, sizeof(int) * (size_t)n));
    // device-side scalars of the call, see the SC_* indices
    BLP_TRY_SCRATCH(alloc((void**)&scalars, sizeof(int) * SC_COUNT));
    BLP_TRY_SCRATCH(cudaMemsetAsync(scalars, 0, sizeof(int) * SC_COUNT, st));
    if (ranged) {
        BLP_TRY_SCRATCH(alloc((void**)&a.acc_cn, sizeof(int) * (size_t)n));
        BLP_TRY_SCRATCH(alloc((void**)&a.acc_aa, sizeof(unsigned long long) * (size_t)n));
    }

    // Pairs that already arrive grouped (the reference's examples.json stores them per user) need
    // no sort: the runs of equal keys are the work items when they average >= 4 pairs.  The
    // decision is taken on the device (k_decide_mode); the kernels of the mode not chosen exit at
    // once, so the call never waits for the host.
    int force = g->tune.grouping;   // (BLP_GROUPING=runs|sort, read at handle creation)
    if (!us && force < 0) force = MODE_SORT;   // a per-user list is never grouped by business
    unsigned* cnt = nullptr;
    if (force == MODE_SORT) {   // the mode is certain: the keys pass counts the group sizes as well
        BLP_TRY_SCRATCH(alloc((void**)&cnt, sizeof(unsigned) * (size_t)n_keys));
        BLP_TRY_SCRATCH(cudaMemsetAsync(cnt, 0, sizeof(unsigned) * (size_t)n_keys, st));
    }
    BLP_TRY_SCRATCH(cudaEventRecord(g->ev[side][0], st));
    const int gblocks = (int)std::min<long long>((n + 255) / 256, (long long)g->sm_count * 16);
    int launches = 1;
    k_group_keys<<<gblocks, 256, 0, st>>>(gx, gy, n, a.n_side, n_mid, g_deg, m_deg, keys, cnt);
    BLP_TRY_SCRATCH(cudaGetLastError());

    int* mode = scalars + 3;
    if (force < 0) {
        k_count_runs<<<gblocks, 256, 0, st>>>(keys, n, (unsigned*)(scalars + 2));
        BLP_TRY_SCRATCH(cudaGetLastError());
        ++launches;
    }
    k_decide_mode<<<1, 1, 0, st>>>((const unsigned*)(scalars + 2), n, force, mode);
    BLP_TRY_SCRATCH(cudaGetLastError());
    ++launches;
    const size_t n_items_max = force == MODE_SORT ? (size_t)n_keys : std::max((size_t)n_keys, (size_t)n);
    BLP_TRY_SCRATCH(alloc((void**)&item_key, sizeof(int) * n_items_max));
    BLP_TRY_SCRATCH(alloc((void**)&item_start, sizeof(int) * n_items_max));
    BLP_TRY_SCRATCH(alloc((void**)&item_end, sizeof(int) * n_items_max));
    if (force != MODE_SORT) {
        const int rblocks = (int)std::min<long long>((n + kRunCut - 1) / kRunCut,
                                                     (long long)g->sm_count * 8);
        k_runs_to_items<<<rblocks, 256, 0, st>>>(mode, keys, n, item_key, item_start, item_end,
                                                 scalars);
        BLP_TRY_SCRATCH(cudaGetLastError());
        ++launches;
    }
    if (force != MODE_RUNS) {
        unsigned* grp_off = nullptr;
        int2* pg = nullptr;
        const bool counted = cnt != nullptr;
        BLP_TRY_SCRATCH(alloc((void**)&inv, sizeof(int) * (size_t)n));
        // grouped-order result records + gather pass: only when the sort mode is certain (the
        // business side); a list whose mode is decided on the device writes its outputs directly
        if (force == MODE_SORT)
            BLP_TRY_SCRATCH(alloc((void**)&a.rec, sizeof(unsigned long long) * 3 * (size_t)n));
        if (!counted) BLP_TRY_SCRATCH(alloc((void**)&cnt, sizeof(unsigned) * (size_t)n_keys));
        BLP_TRY_SCRATCH(alloc((void**)&grp_off, sizeof(unsigned) * (size_t)n_keys));
        BLP_TRY_SCRATCH(alloc((void**)&pg, sizeof(int2) * (size_t)n));
        if (!counted) {
            BLP_TRY_SCRATCH(cudaMemsetAsync(cnt, 0, sizeof(unsigned) * (size_t)n_keys, st));
            k_group_count<<<gblocks, 256, 0, st>>>(mode, keys, n, cnt);
            BLP_TRY_SCRATCH(cudaGetLastError());
            ++launches;
        }
        const int n_tiles = (n_keys + kScanTile - 1) / kScanTile;
        unsigned* tile_sum = nullptr;
        int* tile_items = nullptr;
        BLP_TRY_SCRATCH(alloc((void**)&tile_sum, sizeof(unsigned) * (size_t)n_tiles));
        BLP_TRY_SCRATCH(alloc((void**)&tile_items, sizeof(int) * (size_t)n_tiles));
        k_group_tile_sums<<<n_tiles, 1024, 0, st>>>(mode, cnt, n_keys, tile_sum, tile_items);
        k_group_tile_scan<<<1, 1024, 0, st>>>(mode, tile_sum, tile_items, n_tiles, scalars);
        k_group_tile_apply<<<n_tiles, 1024, 0, st>>>(mode, cnt, n_keys, tile_sum, tile_items, grp_off,
                                                      item_key, item_start, item_end);
        BLP_TRY_SCRATCH(cudaGetLastError());
        k_group_scatter<<<gblocks, 256, 0, st>>>(mode, keys, gy, n, grp_off, pg, inv);
        BLP_TRY_SCRATCH(cudaGetLastError());
        launches += 4;
        a.pg = pg;
    }
    a.mode = mode;
    a.caller_y = gy;
    a.item_key = item_key;
    a.item_start = item_start;
    a.item_end = item_end;
    a.n_items = scalars;
    a.work_counter = scalars + 1;
    // light / heavy split of the work items: light groups go to the warp-per-group kernel
    const bool split = g->light[side] != nullptr;
    SideArgs la{};
    if (split) {
        int *light_list = nullptr, *heavy_list = nullptr;
        BLP_TRY_SCRATCH(alloc((void**)&light_list, sizeof(int) * n_items_max));
        BLP_TRY_SCRATCH(alloc((void**)&heavy_list, sizeof(int) * n_items_max));
        const int sblocks = (int)std::min<size_t>((n_items_max + 255) / 256, (size_t)g->sm_count * 8);
        k_split_items<<<sblocks, 256, 0, st>>>(scalars, item_key, g->light[side], a.n_side,
                                               light_list, heavy_list);
        BLP_TRY_SCRATCH(cudaGetLastError());
        ++launches;
        la = a;
        la.item_list = light_list;
        la.n_items = scalars + SC_N_LIGHT;
        la.work_counter = scalars + SC_LIGHT_WORK;
        a.item_list = heavy_list;
        a.n_items = scalars + SC_N_HEAVY;
    }
    BLP_TRY_SCRATCH(cudaEventRecord(g->ev[side][1], st));

    // ---- persistent scoring grid: as many CTAs per SM as the bitmap allows
    int per_sm = 0, nt = 0, rc = BLP_OK;
    const size_t budget = (size_t)g->max_smem_optin;
    const int nt_force = g->tune.nt;   // (BLP_NT, read at handle creation)
    if (nt_force == 256 || nt_force == 512 || nt_force == 1024) nt = nt_force;
    else if (smem * 4 + 4096 <= budget) nt = 256;
    else if (smem * 2 + 2048 <= budget) nt = 512;
    else nt = 1024;
    const int use_sms = std::max(1, g->sm_count - g->reserve_sms);
    const bool rec_mode = a.rec != nullptr;
    // the occupancy query and the shared-memory opt-in are done once per variant and size
    const int nt_i = nt == 256 ? 0 : (nt == 512 ? 1 : 2);
    int& occ_slot = g->occ_cache[nt_i][ranged ? 1 : 0][rec_mode ? 1 : 0];
    size_t& occ_smem = g->occ_smem[nt_i][ranged ? 1 : 0][rec_mode ? 1 : 0];
#define BLP_DISPATCH(NTV, RV)                                               \
    do {                                                                    \
        rc = rec_mode ? raise_smem_optin<NTV, RV, true>(g->device, smem)    \
                      : raise_smem_optin<NTV, RV, false>(g->device, smem);  \
        if (rc != BLP_OK) break;                                            \
        if (occ_slot > 0 && occ_smem == smem) {                             \
            per_sm = occ_slot;                                              \
        } else {                                                            \
            rc = rec_mode ? occupancy<NTV, RV, true>(smem, &per_sm)         \
                          : occupancy<NTV, RV, false>(smem, &per_sm);       \
            if (rc == BLP_OK) {                                             \
                occ_slot = per_sm;                                          \
                occ_smem = smem;                                            \
            }                                                               \
        }                                                                   \
        if (rc == BLP_OK && per_sm < 1) {                                   \
            set_error("blp_score_pairs: scoring kernel does not fit on an SM"); \
            rc = BLP_ERR_UNSUPPORTED;                                       \
        }                                                                   \
        if (rc == BLP_OK)                                                   \
            rc = rec_mode ? launch_side<NTV, RV, true>(a, per_sm * use_sms, smem, st)  \
                          : launch_side<NTV, RV, false>(a, per_sm * use_sms, smem, st); \
    } while (0)
    // The CTA kernel goes first and the warp-per-group kernel beside it on the handle's side
    // stream: both are persistent work-queue grids, so as the CTA kernel's blocks retire (its
    // groups are few and large, the tail is long) the small warp-per-group blocks fill the SMs.
    // BLP_LIGHT_STREAM=0 keeps both on the caller's stream.
    bool light_aside = false;
    if (split) {
        light_aside = g->side_stream != nullptr && g->tune.light_stream;
        if (light_aside) {
            BLP_TRY_SCRATCH(cudaEventRecord(g->ev_fork[side], st));
            BLP_TRY_SCRATCH(cudaStreamWaitEvent(g->side_stream, g->ev_fork[side], 0));
        }
    }
    if (nt == 256) {
        if (ranged) BLP_DISPATCH(256, true); else BLP_DISPATCH(256, false);
    } else if (nt == 512) {
        if (ranged) BLP_DISPATCH(512, true); else BLP_DISPATCH(512, false);
    } else {
        if (ranged) BLP_DISPATCH(1024, true); else BLP_DISPATCH(1024, false);
    }
#undef BLP_DISPATCH
    if (rc == BLP_OK && split) {
        cudaStream_t lst = light_aside ? g->side_stream : st;
        rc = rec_mode ? launch_light<kLightCap, kLightSlots, kLightWarps, true>(g, la, use_sms, lst)
                      : launch_light<kLightCap, kLightSlots, kLightWarps, false>(g, la, use_sms, lst);
        if (rc == BLP_OK) {
            ++launches;
            g->ev_light[side] = cudaEventRecord(g->ev[side][3], lst) == cudaSuccess;
            // join: everything behind this call on the caller's stream waits for the side stream
            if (light_aside && cudaStreamWaitEvent(st, g->ev[side][3], 0) != cudaSuccess)
                rc = blp::cuda_fail(cudaGetLastError(), "joining the side stream", __FILE__, __LINE__);
        }
        if (rc != BLP_OK && light_aside) cudaStreamSynchronize(g->side_stream);   // scratch is freed below
    }
    if (rc == BLP_OK && a.rec) {
        k_unpermute<<<gblocks, 256, 0, st>>>(a.mode, a.rec, inv, n, a.cn, a.uni, a.jac, a.aa);
        if (cudaGetLastError() != cudaSuccess) rc = BLP_ERR_CUDA;
        ++launches;
    }
    if (rc == BLP_OK) {
        // work-item counts of this call, for blp_score_stats (the scalars live in scratch)
        cudaMemcpyAsync(g->d_counts[side], scalars + SC_N_ITEMS, sizeof(int), cudaMemcpyDeviceToDevice, st);
        cudaMemcpyAsync(g->d_counts[side] + 1, scalars + SC_N_LIGHT, sizeof(int), cudaMemcpyDeviceToDevice, st);
        if (cudaEventRecord(g->ev[side][2], st) == cudaSuccess) g->ev_recorded[side] = true;
        stats.ctas = per_sm * use_sms;
        stats.threads_per_cta = nt;
        stats.smem_bytes = (int)smem;
        stats.kernel_launches = launches + 1;
        stats.range_passes = n_ranges;
    }
    release();
#undef BLP_TRY_SCRATCH
    return rc;
}

#ifdef BLP_PHASE_TIMING
extern "C" int blp_debug_phase_cycles(unsigned long long* host_out16, int reset) {
    BLP_CUDA_TRY(cudaDeviceSynchronize());
    BLP_CUDA_TRY(cudaMemcpyFromSymbol(host_out16, blp::g_phase_cycles, sizeof(unsigned long long) * 16));
    if (reset) {
        unsigned long long z[16] = {};
        BLP_CUDA_TRY(cudaMemcpyToSymbol(blp::g_phase_cycles, z, sizeof(z)));
    }
    return BLP_OK;
}
#endif
