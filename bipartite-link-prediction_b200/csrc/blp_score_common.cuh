// Shared by the scoring kernels (blp_score.cu and its .cuh parts): launch arguments, row
// descriptor accessors, streaming loads.  Not part of the ABI.
#ifndef BLP_SCORE_COMMON_CUH_
#define BLP_SCORE_COMMON_CUH_

#include "blp_internal.h"

namespace blp {


#ifndef BLP_TILE
#define BLP_TILE 256
#endif
constexpr int kTile = BLP_TILE;   // adjacency lists per scheduling tile (<= threads per CTA)
#ifndef BLP_CHUNK_V4
#define BLP_CHUNK_V4 128
#endif
constexpr int kChunkV4 = BLP_CHUNK_V4;   // int4 loads per chunk (at most 4 per lane): 512 ids
constexpr unsigned kFull = 0xffffffffu;

struct SideArgs {
    // grouping side x: rows x -> middle nodes m;   middle side: rows m -> nodes of x's side.
    // A row descriptor packs (first entry / 4) << 24 | degree: one 8-byte load locates a list.
    const unsigned long long* __restrict__ g_row;
    const int* __restrict__ g_adj;
    const unsigned long long* __restrict__ m_row;
    const int* __restrict__ m_adj;
    const unsigned* __restrict__ m_adjw;  // Q1.31 Adamic-Adar weight of every m_adj entry
    int n_side;                           // number of x-side nodes == sentinel id of m rows
    int bm_words;                         // bitmap words (covers bit n_side as well)
    // hub bitmaps: N(m) of every middle node with deg >= hub_min_deg, as bm_words-word bitmaps
    // m_xrow: row descriptors as seen by the expansion -- equal to m_row except that a hub's
    // entry is  1<<63 | bitmap slot << 24 | degree  (one gather tells list from bitmap)
    const unsigned long long* __restrict__ m_xrow;
    const unsigned* __restrict__ hub_bm;
    int hub_words;                        // words per hub bitmap (whole id universe)
    // probe path of the intersection: Q1.31 weight of every x-side node (null = path off)
    const unsigned* __restrict__ node_wt;
    int probe_ratio;
    // |N(h) & N(y)| and the weight sum over it for every OR-hub h (row) and bitmap node y (column):
    // lets the warp-per-group kernel take groups with ONE hub without touching the hub's bitmap
    const int* __restrict__ hubtab_cn;
    const unsigned long long* __restrict__ hubtab_aa;
    int hubtab_stride;
    // id-range passes: when the bitmap of the whole universe does not fit (or is not wanted) in
    // shared memory the group is processed n_ranges times, pass r covering ids
    // [r*range_bits, (r+1)*range_bits); partial cn / aa wait in scratch (grouped order)
    int range_bits;
    int n_ranges;
    // ranged sides: middle rows are partitioned by range; seg_off[m * seg_stride + r] = offset of
    // range r's first entry inside row m (seg_stride = n_ranges + 1)
    const int* __restrict__ seg_off;
    int seg_stride;
    int* acc_cn;
    unsigned long long* acc_aa;
    // grouping
    // work items: item i is the node item_key[i] (n_side = "not in graph") with the pairs
    // [item_start[i], item_end[i]) of the grouped order
    const int* __restrict__ item_key;
    const int* __restrict__ item_start;
    const int* __restrict__ item_end;
    const int* __restrict__ n_items;
    // with the light / heavy split (k_split_items) each scoring kernel walks its own list of item
    // indices: position i of the persistent loop is item item_list[i]; null = every item in order
    const int* __restrict__ item_list;
    const int2* __restrict__ pg;            // sort mode: (caller-order pair index, partner y) per
                                            // grouped position -- one 8-byte scattered store
    const int* __restrict__ mode;           // MODE_RUNS: grouped order == caller order, pg is
    const int* __restrict__ caller_y;       //            unused and the partners are caller_y
    int* work_counter;
    // sort mode only: results are first written as 24-byte records in GROUPED order (coalesced)
    // and brought to the caller's order by k_unpermute; null = write the outputs directly
    unsigned long long* rec;
    // outputs, caller order (any may be null)
    int* cn;
    int* uni;
    double* jac;
    double* aa;
    long long* pa;
    int* hop2;
};

// ---- L2 residency hints -------------------------------------------------------------------
// The graph (adjacency, weights, hub bitmaps, row descriptors) is what every group re-reads; the
// pair ids, the per-call scratch and the result columns stream through once.  Graph loads carry an
// L2 evict_last policy, the streams use evict-first loads / stores (ld/st.global.cs), so that the
// 0.5 GB of results per step do not push the graph out of L2 (BLP_L2_HINTS=0 compiles both away).
#ifndef BLP_L2_HINTS
#define BLP_L2_HINTS 1
#endif

__device__ __forceinline__ unsigned long long l2_keep_policy() {
    unsigned long long pol = 0ull;
#if BLP_L2_HINTS
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
#endif
    return pol;
}

__device__ __forceinline__ int4 ldg_stream(const int4* p, unsigned long long pol) {
    int4 r;
#if BLP_L2_HINTS
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.s32 {%0,%1,%2,%3}, [%4], %5;"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p), "l"(pol));
#else
    asm volatile("ld.global.nc.L1::no_allocate.v4.s32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
#endif
    return r;
}

__device__ __forceinline__ int row_deg(unsigned long long row) { return (int)(row & 0xffffffull); }
__device__ __forceinline__ long long row_first4(unsigned long long row) {
    return (long long)((row >> 24) & ((1ull << BLP_ROW_FIRST4_BITS) - 1));
}
// hub-bitmap slot + 1 of the node the row belongs to (0 = its list has no bitmap); bit 63 is the
// expansion-side hub flag of m_xrow and is not part of the field
__device__ __forceinline__ int row_slot1(unsigned long long row) {
    return (int)((row >> BLP_ROW_SLOT_SHIFT) & (unsigned long long)BLP_ROW_MAX_SLOTS);
}

__device__ __forceinline__ uint4 ldg_stream_u(const uint4* p, unsigned long long pol) {
    uint4 r;
#if BLP_L2_HINTS
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.u32 {%0,%1,%2,%3}, [%4], %5;"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p), "l"(pol));
#else
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
#endif
    return r;
}

// graph data through the read-only path with the keep-in-L2 policy (L1 allocation as usual)
__device__ __forceinline__ uint4 ldg_keep(const uint4* p, unsigned long long pol) {
#if BLP_L2_HINTS
    uint4 r;
    asm volatile("ld.global.nc.L2::cache_hint.v4.u32 {%0,%1,%2,%3}, [%4], %5;"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p), "l"(pol));
    return r;
#else
    return __ldg(p);
#endif
}
__device__ __forceinline__ unsigned ldg_keep(const unsigned* p, unsigned long long pol) {
#if BLP_L2_HINTS
    unsigned r;
    asm volatile("ld.global.nc.L2::cache_hint.u32 %0, [%1], %2;" : "=r"(r) : "l"(p), "l"(pol));
    return r;
#else
    return __ldg(p);
#endif
}

// streaming (evict-first) accessors for data that passes through once
template <typename T>
__device__ __forceinline__ void st_stream(T* p, T v) {
#if BLP_L2_HINTS
    __stcs(p, v);
#else
    *p = v;
#endif
}
template <typename T>
__device__ __forceinline__ T ld_once(const T* p) {
#if BLP_L2_HINTS
    return __ldcs(p);
#else
    return *p;
#endif
}

// ---- TMA bulk copy + mbarrier (sm_90+; the hub-bitmap copy of k_score_side) --------------------
__device__ __forceinline__ unsigned smem_u32(const void* p) {
    return (unsigned)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
// make generic-proxy shared-memory writes (and the barrier's init) visible to the async proxy
__device__ __forceinline__ void fence_async_smem() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
// one thread: global -> shared, `bytes` a multiple of 16, both addresses 16-byte aligned; the copy
// engine signals `bar` with the byte count when the data has landed
__device__ __forceinline__ void bulk_copy_g2s(void* dst_smem, const void* src, unsigned bytes,
                                              unsigned long long* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst_smem)), "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "BLP_MBAR_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra BLP_MBAR_DONE;\n"
        "bra BLP_MBAR_WAIT;\n"
        "BLP_MBAR_DONE:\n"
        "}" ::"r"(smem_u32(bar)), "r"(parity)
        : "memory");
}

// grouping mode, decided on the device (blp_score_group.cuh)
enum { MODE_SORT = 0, MODE_RUNS = 1 };

// (caller-order index, partner) of the pair at grouped position k
__device__ __forceinline__ int2 pair_at(const SideArgs& a, long long k) {
    return a.pg ? ld_once(a.pg + k) : make_int2((int)k, ld_once(a.caller_y + k));
}

// Descriptor of the part of row `row` (of middle node m) that holds the ids of range `pass`: the
// 16-byte aligned window around entries [s, e) of the row.  Entries of the window outside [s, e)
// belong to neighbouring ranges or are padding and fail the walker's range test.  The degree field
// is set so that (deg + 3) / 4 is the window's length in 128-bit words (0 = nothing to walk).
__device__ __forceinline__ unsigned long long segment_row(const SideArgs& a, unsigned long long row, int m,
                                                          int pass) {
    const int* so = a.seg_off + (size_t)m * a.seg_stride + pass;
    const int s = so[0], e = so[1];
    const long long f4 = row_first4(row) + (s >> 2);
    const int n4 = e > s ? ((e + 3) >> 2) - (s >> 2) : 0;
    return ((unsigned long long)f4 << 24) | (unsigned)(n4 << 2);
}

// The epilogue every scoring kernel shares: one pair's integer counts -> its result columns.
// c = |hop2(x) & N(y)|, aa_q = the Q1.31 weight sum over those ids, pdeg = deg(y), xdeg = deg(x).
// valid = false is the "id not in graph" bucket (similarity.py:52,59-60): every output, hop2
// included, is the literal 0.  REC: the record at grouped position k instead of the caller-order
// columns (pa and hop2 always go to the caller-order index idx).
template <bool REC>
__device__ __forceinline__ void emit_pair(const SideArgs& a, long long k, int idx, bool valid, int c,
                                          int hop2, int xdeg, int pdeg, unsigned long long aa_q) {
    int u = 0;
    double jv = 0.0, av = 0.0;
    long long pa = 0;
    if (valid) {
        u = hop2 + pdeg - c;   // |a| + |b| - |a & b|  (similarity.py:110)
        jv = __ddiv_rn((double)c, (double)u);
        av = (double)aa_q * (1.0 / (double)(1ull << BLP_AA_FRAC_BITS));
        pa = (long long)xdeg * (long long)pdeg;
    } else {
        c = 0;
        hop2 = 0;
    }
    // results stream out once (on the multi-GPU path into a peer's memory): evict-first
    if (REC) {
        unsigned long long* r = a.rec + 3 * k;
        st_stream(r, (unsigned long long)(unsigned)c | ((unsigned long long)(unsigned)u << 32));
        st_stream(r + 1, (unsigned long long)__double_as_longlong(jv));
        st_stream(r + 2, (unsigned long long)__double_as_longlong(av));
    } else {
        if (a.cn) st_stream(a.cn + idx, c);
        if (a.uni) st_stream(a.uni + idx, u);
        if (a.jac) st_stream(a.jac + idx, jv);
        if (a.aa) st_stream(a.aa + idx, av);
    }
    if (a.pa) st_stream(a.pa + idx, pa);
    if (a.hop2) st_stream(a.hop2 + idx, hop2);
}

constexpr int kShortV4 = 4;   // lists of <= 16 ids take the sub-warp path (4 lanes per list)
// Probe path.  A hop-2 set built from at most kProbeCap list entries and no hub bitmap is also
// kept as an id list (the atomicOr that turns a bit on appends the id).  A pair of that group
// whose partner y has a bitmap and deg(y) >= probe_ratio * |hop2(x)| is then scored by probing
// y's bitmap with the list -- |hop2(x)| global loads instead of streaming deg(y) ids + weights.
// On C2 this replaces ~45 % of all streamed ids by ~5 % as many probes (hub partners are drawn
// in proportion to their degree; two thirds of the users have no hub business and a small set).
constexpr int kProbeCap = 768;
constexpr int kProbeRatio = 2;   // default; BLP_PROBE_RATIO overrides it at graph creation

}  // namespace blp

#endif  // BLP_SCORE_COMMON_CUH_
