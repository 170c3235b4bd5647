// The warp-per-group scoring kernel and what it needs from graph creation (part of blp_score.cu).
#ifndef BLP_SCORE_LIGHT_CUH_
#define BLP_SCORE_LIGHT_CUH_

#include "blp_score_common.cuh"

namespace blp {

// ---------------------------------------------------------------------------------------------
// Light groups: one WARP per group.
//
// Measured on C2 (tools/cost_model.py): 60 % of the CTA kernel's time is per-GROUP cost -- a
// chain of ~8 CTA barriers and ~6 dependent global round trips per group with only four groups in
// flight per SM (four 46 KB bitmaps) -- and about half of the groups are tiny: a user with a few
// small businesses whose expansion walks a few hundred ids.  Such a group (classified per node at
// graph creation: <= 32 middle nodes, none of them an OR-hub, <= CAP ids walked) needs no bitmap
// over the whole universe.  Here one warp owns it: hop2(x) goes into an open-addressing hash
// table in shared memory (and, in insertion order, into an id list), the partner lists are
// streamed against the table -- all lists of a 32-pair tile as ONE flattened index space, so that
// short lists cost no pass of their own and every lane has loads in flight -- and partners that
// have a bitmap are scored by probing it with the list.  No CTA barrier anywhere; the descriptor
// chain of the next group is fetched in stages behind the current group's phases.  The arithmetic
// is the same integer arithmetic as in k_score_side, so the outputs are bit-identical.
// A group with exactly ONE hub among its middle nodes qualifies as well: hop2(x) = N(h) + S' with
// S' = the ids of the other lists that are not in N(h); the table and the list hold S' only, a
// streamed id that misses the table is looked up in the hub's bitmap where it lies (L2), and for a
// partner y that has a bitmap itself |N(h) & N(y)| comes from a table precomputed at graph creation.
// (A larger-table "medium" instance with 8 groups in flight per SM was measured and is slower than
// the CTA kernel: one warp streaming a hub partner's list is too slow.)
// ---------------------------------------------------------------------------------------------
constexpr int kLightCap = 512, kLightSlots = 1024, kLightWarps = 8;
constexpr int kLightMinCtas = 4;   // __launch_bounds__ occupancy target of k_score_light
constexpr int kLightEmpty = -1;

template <int CAP, int SLOTS>
struct LightSmem {
    int table[SLOTS];
    int list[CAP];
    // per pair of the tile: hits and weighted hits.  The weight sum is kept as two 32-bit words
    // (low 24 bits / the rest) so that native 32-bit shared atomics add it exactly: a lane adds
    // its whole share of a pair at once (<= 32 adds per pair), and a pair has < 2^24 hits.
    unsigned aa_lo[32];
    unsigned aa_hi[32];
    int cn[32];
};

// The table is a set of 4-slot buckets (16 bytes, one 128-bit shared load).  A bucket fills from
// slot 0 upwards, so it is full exactly when its last slot is taken; only then does a search go on
// to the next bucket.  At the typical load (~0.2) a lookup is one load and four compares, with
// hardly any divergence between the lanes.
template <int SLOTS>
__device__ __forceinline__ unsigned light_bucket(int id) {
    static_assert((SLOTS & (SLOTS - 1)) == 0 && SLOTS >= 64, "power of two");
    return (((unsigned)id * 2654435761u) >> 8) & (unsigned)(SLOTS / 4 - 1);
}

template <int SLOTS>
__device__ __forceinline__ bool light_has(const int* table, int id) {
    unsigned b = light_bucket<SLOTS>(id);
    while (true) {
        const int4 v = reinterpret_cast<const int4*>(table)[b];
        if (v.x == id || v.y == id || v.z == id || v.w == id) return true;
        if (v.w == kLightEmpty) return false;   // bucket not full (the padding id ends here too)
        b = (b + 1) & (SLOTS / 4 - 1);
    }
}

// true when THIS call put the id into the table
template <int SLOTS>
__device__ __forceinline__ bool light_insert(int* table, int id) {
    unsigned b = light_bucket<SLOTS>(id);
    while (true) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int prev = atomicCAS(&table[4 * b + k], kLightEmpty, id);
            if (prev == kLightEmpty) return true;
            if (prev == id) return false;
        }
        b = (b + 1) & (SLOTS / 4 - 1);
    }
}

// expansion step for the four ids of one 128-bit load; new ids are appended to the list with one
// ballot per component (list_n is warp-uniform)
__device__ __forceinline__ bool hub_bit(const unsigned* hbm, int id, unsigned long long pol) {
    return (ldg_keep(hbm + (id >> 5), pol) >> (id & 31)) & 1u;
}

// hbm: bitmap of the group's single hub (null = none); ids already in it stay out of the table
template <int SLOTS>
__device__ __forceinline__ void light_expand4(int* table, int* list, int4 v, bool active, int x,
                                              int n_side, const unsigned* hbm, int& list_n, int lane,
                                              unsigned long long pol) {
    const int id[4] = {v.x, v.y, v.z, v.w};
    bool want[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) want[k] = active && id[k] < n_side && id[k] != x;
    if (hbm) {
        bool in_hub[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) in_hub[k] = want[k] && hub_bit(hbm, id[k], pol);   // four loads in flight
#pragma unroll
        for (int k = 0; k < 4; ++k) want[k] = want[k] && !in_hub[k];
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const bool fresh = want[k] && light_insert<SLOTS>(table, id[k]);
        const unsigned m = __ballot_sync(kFull, fresh);
        if (fresh) list[list_n + __popc(m & ((1u << lane) - 1u))] = id[k];
        list_n += __popc(m);
    }
}

template <int SLOTS>
__device__ __forceinline__ void light_test4(const int* table, int4 v, uint4 wt, int x,
                                            const unsigned* hbm, unsigned& cnt,
                                            unsigned long long& acc, unsigned long long pol) {
    const int id[4] = {v.x, v.y, v.z, v.w};
    const unsigned w[4] = {wt.x, wt.y, wt.z, wt.w};
    bool hit[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) hit[k] = light_has<SLOTS>(table, id[k]);
    if (hbm) {   // hop2(x) also holds N(h) \ {x}; bit n_side (the padding id) is never on
        bool in_hub[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) in_hub[k] = !hit[k] && id[k] != x && hub_bit(hbm, id[k], pol);
#pragma unroll
        for (int k = 0; k < 4; ++k) hit[k] = hit[k] || in_hub[k];
    }
#pragma unroll
    for (int k = 0; k < 4; ++k)
        if (hit[k]) {
            ++cnt;
            acc += w[k];
        }
}

// exact warp sum of per-lane weight sums (three 16/16/32-bit limbs, REDUX each)
__device__ __forceinline__ unsigned long long light_sum64(unsigned long long acc) {
    const unsigned l0 = __reduce_add_sync(kFull, (unsigned)(acc & 0xffffull));
    const unsigned l1 = __reduce_add_sync(kFull, (unsigned)((acc >> 16) & 0xffffull));
    const unsigned l2 = __reduce_add_sync(kFull, (unsigned)(acc >> 32));
    return ((unsigned long long)l2 << 32) + ((unsigned long long)l1 << 16) + l0;
}

__device__ __forceinline__ int warp_incl_scan(int v, int lane) {
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int t = __shfl_up_sync(kFull, v, d);
        if (lane >= d) v += t;
    }
    return v;
}

// Flattened lists: lane l holds the inclusive prefix of the lengths.  Which lane's list owns the
// flat index i (< total)?  = number of lanes whose inclusive prefix is <= i.
__device__ __forceinline__ int seg_search(int incl, int i) {
    int lo = 0;
#pragma unroll
    for (int s = 16; s >= 1; s >>= 1) {
        const int t = __shfl_sync(kFull, incl, lo + s - 1);
        if (t <= i) lo += s;
    }
    return lo;
}

// descriptor chain of one group, fetched in stages (every field warp-uniform except m / mrow)
struct LightRegs {
    int it;                     // item index, -1 = none
    int x;
    int p0, p1;
    unsigned long long xrow;
    int m;                      // lane < deg(x): this lane's middle node
    unsigned long long mrow;    // ... and its row
};
__device__ __forceinline__ void light_stage_a(const SideArgs& a, LightRegs& g, int c, int n_items) {
    g.it = c < n_items ? a.item_list[c] : -1;
}
__device__ __forceinline__ void light_stage_b(const SideArgs& a, LightRegs& g) {
    g.x = 0;
    g.p0 = g.p1 = 0;
    if (g.it >= 0) {
        g.x = a.item_key[g.it];
        g.p0 = a.item_start[g.it];
        g.p1 = a.item_end[g.it];
    }
}
__device__ __forceinline__ void light_stage_c(const SideArgs& a, LightRegs& g) {
    g.xrow = g.it >= 0 ? a.g_row[g.x] : 0ull;
}
__device__ __forceinline__ void light_stage_d(const SideArgs& a, LightRegs& g, int lane) {
    g.m = lane < row_deg(g.xrow) ? a.g_adj[row_first4(g.xrow) * 4 + lane] : -1;
}
__device__ __forceinline__ void light_stage_e(const SideArgs& a, LightRegs& g) {
    g.mrow = g.m >= 0 ? a.m_xrow[g.m] : 0ull;   // a hub's entry carries flag, slot and table row
}

template <int CAP, int SLOTS, int WARPS, bool REC>
__global__ void __launch_bounds__(WARPS * 32, kLightMinCtas) k_score_light(SideArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    typedef LightSmem<CAP, SLOTS> Smem;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    Smem& ls = reinterpret_cast<Smem*>(smem_raw)[warp];
    const int n_items = *a.n_items;
    if (*a.mode == MODE_RUNS) a.pg = nullptr;
    const unsigned long long pol = l2_keep_policy();
    const int4* adj4 = reinterpret_cast<const int4*>(a.m_adj);
    const uint4* adjw4 = reinterpret_cast<const uint4*>(a.m_adjw);
    const int4 sent4 = make_int4(a.n_side, a.n_side, a.n_side, a.n_side);
    const int4 empty4 = make_int4(kLightEmpty, kLightEmpty, kLightEmpty, kLightEmpty);
    {
        int4* t4 = reinterpret_cast<int4*>(ls.table);
        for (int i = lane; i < SLOTS / 4; i += 32) t4[i] = empty4;
    }
    __syncwarp();
    // two claims ahead: the index of the next group is known when the current one starts
    int c = 0, c1 = 0;
    if (lane == 0) {
        c = atomicAdd(a.work_counter, 1);
        c1 = atomicAdd(a.work_counter, 1);
    }
    c = __shfl_sync(kFull, c, 0);
    c1 = __shfl_sync(kFull, c1, 0);
    LightRegs cur;
    light_stage_a(a, cur, c, n_items);
    light_stage_b(a, cur);
    light_stage_c(a, cur);
    light_stage_d(a, cur, lane);
    light_stage_e(a, cur);
    while (c < n_items) {
        int c2 = 0;
        if (lane == 0) c2 = atomicAdd(a.work_counter, 1);
        LightRegs nxt;
        light_stage_a(a, nxt, c1, n_items);
        const int x = cur.x;
        const long long p0 = cur.p0, p1 = cur.p1;
        const int xdeg = row_deg(cur.xrow);   // 1..32 by the class flag
        // partners of the first pair tile: issued now, their rows after the expansion
        int2 iy0 = make_int2(0, 0);
        if (p0 + lane < p1) iy0 = pair_at(a, p0 + lane);
        // the group's hub, if it has one (at most one, by its class)
        const unsigned hub_lanes = __ballot_sync(kFull, (cur.mrow >> 63) != 0);
        const unsigned* hbm = nullptr;
        int hub_deg = 0, hub_tab = 0;
        if (hub_lanes) {
            const unsigned long long hr = __shfl_sync(kFull, cur.mrow, __ffs(hub_lanes) - 1);
            hbm = a.hub_bm + (size_t)((hr >> 24) & (unsigned long long)BLP_ROW_MAX_SLOTS) * (size_t)a.hub_words;
            hub_deg = row_deg(hr);
            hub_tab = (int)((hr >> BLP_XROW_ORIDX_SHIFT) & (unsigned long long)BLP_ROW_MAX_SLOTS) *
                      a.hubtab_stride;
        }
        // ---- expansion: the lists N(m), m in N(x), as one flattened space of 128-bit loads
        int list_n = 0;
        {
            const int mn4 = (cur.mrow >> 63) ? 0 : (row_deg(cur.mrow) + 3) >> 2;
            const long long mat = row_first4(cur.mrow);
            const int incl = warp_incl_scan(mn4, lane);
            const int excl = incl - mn4;
            const int total = __shfl_sync(kFull, incl, 31);
            for (int i0 = 0; i0 < total; i0 += 64) {
                int4 v[2];
                bool ok[2];
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const int i = i0 + 32 * h + lane;
                    ok[h] = i < total;
                    const int ii = ok[h] ? i : total - 1;
                    const int j = seg_search(incl, ii);
                    const int off = ii - __shfl_sync(kFull, excl, j);
                    const long long at = __shfl_sync(kFull, mat, j) + off;
                    v[h] = ok[h] ? ldg_stream(adj4 + at, pol) : sent4;
                }
#pragma unroll
                for (int h = 0; h < 2; ++h)
                    if (i0 + 32 * h < total)
                        light_expand4<SLOTS>(ls.table, ls.list, v[h], ok[h], x, a.n_side, hbm, list_n,
                                             lane, pol);
            }
        }
        __syncwarp();
        // x itself was never inserted; it is in N(h), and so is nothing else of the list
        const int hop2 = list_n + (hbm ? hub_deg - 1 : 0);
        light_stage_b(a, nxt);
        // ---- the pairs of the group, 32 at a time: lane l owns pair tb + l
        for (long long tb = p0; tb < p1; tb += 32) {
            const int count = (int)min(32ll, p1 - tb);
            unsigned long long row = 0ull;
            int idx = 0, py = -1;
            if (lane < count) {
                const int2 iy = tb == p0 ? iy0 : pair_at(a, tb + lane);
                row = a.m_row[iy.y];
                idx = iy.x;
                py = iy.y;
            }
            if (tb == p0) light_stage_c(a, nxt);
            const int pdeg = row_deg(row);
            const bool by_probe = lane < count && a.node_wt != nullptr && row_slot1(row) > 0 &&
                                  (long long)a.probe_ratio * list_n <= pdeg;
            ls.cn[lane] = 0;
            ls.aa_lo[lane] = 0u;
            ls.aa_hi[lane] = 0u;
            __syncwarp();
            unsigned my_cn = 0;
            unsigned long long my_aa = 0ull;
            // partners with a bitmap: the hop-2 list against the bitmap
            unsigned todo = __ballot_sync(kFull, by_probe);
            while (todo) {
                const int j = __ffs(todo) - 1;
                todo &= todo - 1;
                const unsigned long long r = __shfl_sync(kFull, row, j);
                const unsigned* hb = a.hub_bm + (size_t)(row_slot1(r) - 1) * (size_t)a.hub_words;
                unsigned cnt = 0;
                unsigned long long acc = 0ull;
                if (hbm && lane == 0) {
                    // the hub's share |N(h) & N(y)| from the table, minus x when x is in N(y)
                    const int t = hub_tab + row_slot1(r) - 1;
                    cnt = (unsigned)a.hubtab_cn[t];
                    acc = a.hubtab_aa[t];
                }
                if (hbm) {
                    const int yj = __shfl_sync(kFull, py, j);
                    const bool x_in = __any_sync(kFull, cur.m == yj);   // y in N(x)
                    if (x_in && lane == 0) {
                        cnt -= 1u;
                        acc -= (unsigned long long)ldg_keep(a.node_wt + x, pol);
                    }
                }
                for (int i0 = lane; i0 < list_n; i0 += 128) {
                    int w[4];
                    unsigned word[4];
#pragma unroll
                    for (int k = 0; k < 4; ++k)   // bit n_side is never on in a hub bitmap
                        w[k] = i0 + 32 * k < list_n ? ls.list[i0 + 32 * k] : a.n_side;
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
                if (cnt > 0) acc = light_sum64(acc);
                if (lane == j) {
                    my_cn = cnt;
                    my_aa = cnt > 0 ? acc : 0ull;
                }
            }
            // every other partner list, flattened: streamed against the table (and the hub's bitmap)
            if (hop2 > 0) {
                const int pn4 = (lane < count && !by_probe) ? (pdeg + 3) >> 2 : 0;
                const long long pat = row_first4(row);
                const int incl = warp_incl_scan(pn4, lane);
                const int excl = incl - pn4;
                const int total = __shfl_sync(kFull, incl, 31);
                int run_own = 0;
                unsigned run_cnt = 0;
                unsigned long long run_acc = 0ull;
                for (int i0 = 0; i0 < total; i0 += 64) {
                    int4 v[2];
                    uint4 wt[2];
                    int own[2];
                    bool ok[2];
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        const int i = i0 + 32 * h + lane;
                        ok[h] = i < total;
                        const int ii = ok[h] ? i : total - 1;
                        own[h] = seg_search(incl, ii);
                        const int off = ii - __shfl_sync(kFull, excl, own[h]);
                        const long long at = __shfl_sync(kFull, pat, own[h]) + off;
                        v[h] = ok[h] ? ldg_stream(adj4 + at, pol) : sent4;
                        wt[h] = ok[h] ? ldg_stream_u(adjw4 + at, pol) : make_uint4(0u, 0u, 0u, 0u);
                    }
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        if (ok[h]) {
                            // a lane meets the 128-bit words of one pair back to back: it keeps
                            // their sum in registers and adds it to the pair's totals once
                            if (own[h] != run_own) {
                                if (run_cnt > 0) {
                                    atomicAdd(&ls.cn[run_own], (int)run_cnt);
                                    atomicAdd(&ls.aa_lo[run_own], (unsigned)(run_acc & 0xffffffull));
                                    atomicAdd(&ls.aa_hi[run_own], (unsigned)(run_acc >> 24));
                                }
                                run_own = own[h];
                                run_cnt = 0;
                                run_acc = 0ull;
                            }
                            light_test4<SLOTS>(ls.table, v[h], wt[h], x, hbm, run_cnt, run_acc, pol);
                        }
                    }
                }
                if (run_cnt > 0) {
                    atomicAdd(&ls.cn[run_own], (int)run_cnt);
                    atomicAdd(&ls.aa_lo[run_own], (unsigned)(run_acc & 0xffffffull));
                    atomicAdd(&ls.aa_hi[run_own], (unsigned)(run_acc >> 24));
                }
                __syncwarp();
                if (!by_probe) {
                    my_cn = (unsigned)ls.cn[lane];
                    my_aa = ((unsigned long long)ls.aa_hi[lane] << 24) + ls.aa_lo[lane];
                }
            }
            if (tb == p0) light_stage_d(a, nxt, lane);
            // epilogue: the one every scoring kernel uses
            if (lane < count) emit_pair<REC>(a, tb + lane, idx, true, (int)my_cn, hop2, xdeg, pdeg, my_aa);
            __syncwarp();
        }
        if (p0 >= p1) {   // (never: an item has at least one pair)
            light_stage_c(a, nxt);
            light_stage_d(a, nxt, lane);
        }
        // leave the table empty for the next group
        if (list_n > 0) {
            int4* t4 = reinterpret_cast<int4*>(ls.table);
            for (int i = lane; i < SLOTS / 4; i += 32) t4[i] = empty4;
        }
        __syncwarp();
        light_stage_e(a, nxt);
        cur = nxt;
        c = c1;
        c1 = __shfl_sync(kFull, c2, 0);
    }
}

// Per node of the grouping side: can its group go to k_score_light?  (run once per graph)
// Yes when it has <= 32 middle nodes, at most one of them an OR-hub (and only if the hub tables
// exist), and the other lists together hold <= kLightCap ids.
__global__ void k_flag_light(int n_side, const unsigned long long* __restrict__ g_row,
                             const int* __restrict__ g_adj,
                             const unsigned long long* __restrict__ m_xrow, int max_hubs,
                             unsigned char* __restrict__ light) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    if (x >= n_side) return;
    const unsigned long long xr = g_row[x];
    const int d = row_deg(xr);
    bool ok = d >= 1 && d <= 32;
    long long walked = 0;
    int hubs = 0;
    if (ok) {
        const int* adj = g_adj + row_first4(xr) * 4;
        for (int i = 0; i < d; ++i) {
            const unsigned long long r = m_xrow[adj[i]];
            if (r >> 63) ++hubs;
            else walked += row_deg(r);
        }
    }
    light[x] = (ok && hubs <= max_hubs && walked <= kLightCap) ? 1 : 0;
}

// One CTA per (bitmap node y, OR-hub h): |N(h) & N(y)| and the Q1.31 weight sum over it.
__global__ void k_hub_tables(const int* __restrict__ or_nodes, int n_bm,
                             const unsigned long long* __restrict__ m_row,
                             const int* __restrict__ m_adj, const unsigned* __restrict__ hub_bm,
                             int bm_words, const unsigned* __restrict__ node_wt,
                             int* __restrict__ tab_cn, unsigned long long* __restrict__ tab_aa) {
    const int y = blockIdx.x, o = blockIdx.y;
    const unsigned long long row = m_row[or_nodes[o]];
    const int* adj = m_adj + row_first4(row) * 4;
    const unsigned* bm = hub_bm + (size_t)y * bm_words;
    const int padded = ((row_deg(row) + 3) >> 2) << 2;   // padding sits at the row's tail; its bit is never on
    unsigned cnt = 0;
    unsigned long long acc = 0ull;
    for (int i = threadIdx.x; i < padded; i += blockDim.x) {
        const int id = adj[i];   // the padding id's bit is never on
        if ((bm[id >> 5] >> (id & 31)) & 1u) {
            ++cnt;
            acc += node_wt[id];
        }
    }
    __shared__ unsigned s_cnt;
    __shared__ unsigned long long s_acc;
    if (threadIdx.x == 0) {
        s_cnt = 0;
        s_acc = 0ull;
    }
    __syncthreads();
    cnt = __reduce_add_sync(kFull, cnt);
    if (cnt > 0) {
        acc = light_sum64(acc);
        if ((threadIdx.x & 31) == 0) {
            atomicAdd(&s_cnt, cnt);
            atomicAdd(&s_acc, acc);
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        tab_cn[(size_t)o * n_bm + y] = (int)s_cnt;
        tab_aa[(size_t)o * n_bm + y] = s_acc;
    }
}

template <int CAP, int SLOTS, int WARPS, bool REC>
static int launch_light(blp_graph* g, const SideArgs& a, int use_sms, cudaStream_t st) {
    const size_t smem = sizeof(LightSmem<CAP, SLOTS>) * WARPS;
    int per_sm = 0;
    const int rc = kernel_ctas_per_sm((const void*)k_score_light<CAP, SLOTS, WARPS, REC>, g->device,
                                      WARPS * 32, smem, &per_sm);
    if (rc != BLP_OK) return rc;
    if (per_sm < 1) {
        set_error("blp_score_pairs: the warp-per-group kernel does not fit on an SM");
        return BLP_ERR_UNSUPPORTED;
    }
    k_score_light<CAP, SLOTS, WARPS, REC><<<per_sm * use_sms, WARPS * 32, smem, st>>>(a);
    BLP_CUDA_TRY(cudaGetLastError());
    return BLP_OK;
}

}  // namespace blp

#endif  // BLP_SCORE_LIGHT_CUH_
