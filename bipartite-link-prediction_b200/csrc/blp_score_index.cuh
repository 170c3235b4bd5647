// Business index: the business side without grouping.
//
// For a pair (u, b) the business side needs |hop2(b) & N(u)|, its weight sum and |hop2(b)|.
// b' is in hop2(b) iff b' != b and b, b' share a reviewer -- a relation of the graph alone, the
// same on every call.  So it is built once per graph as one bitmap row per business (the
// co-review pattern of A^T A without its diagonal), and a call scores every pair in the caller's
// order by testing N(u) (4.8 ids on average on C2) against b's bits: no counting sort, no per-call
// expansion of hop2(b), no grouped-order records and no un-permute pass.  The index lives beside the
// graph for the handle's lifetime; it is read-only after the build.  The rows take
// n_biz^2 / 8 bytes (C2: 465 MB, C3 / C4: 4.5 GB), so a graph with too many businesses (C5) and a
// ranged business side keep the grouped path of k_score_side / k_score_light.
#ifndef BLP_SCORE_INDEX_CUH_
#define BLP_SCORE_INDEX_CUH_

#include <algorithm>
#include <chrono>
#include <vector>

#include "blp_score_common.cuh"
#include "blp_score_group.cuh"

namespace blp {

constexpr int kIndexBuildThreads = 512;
constexpr int kIndexScoreThreads = 256;   // a power of two (the long-list word search halves it)
// pairs with deg(u) <= this are scored by their own lane (C2: 96.6 % of the pairs); the longer
// lists by the whole CTA
constexpr int kIndexLaneDeg = 16;

// Rows and columns are kept in DEGREE-RANK order (rank 0 = the most-reviewed business): row
// rank(b) holds hop2(b), bit rank(b') of it stands for business b'.  The relation is symmetric and
// its diagonal is clear, so the bit of (b, b') is read at row max(rank b, rank b'), column min.
// The ids a pair tests are the businesses of N(u), and reviews are power-law distributed over
// businesses, so the tests gather in the low-rank columns: on C2 the 48 M tests of one call touch
// 5.8 M distinct 32-byte sectors (8.6 M when row b is read at column rank(b')), and the hottest
// 96 MiB of them answer 92 % of the tests (tools/biz_sectors.py).
// u_radj is u_adj with every business id replaced by its rank (padding stays the sentinel n_biz,
// whose bit is never set); the weights u_adjw stay parallel to it.
__global__ void k_rank_ids(const int* __restrict__ ids, long long n, const int* __restrict__ rank,
                           int sentinel, int* __restrict__ out) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n;
         i += (long long)gridDim.x * blockDim.x) {
        const int id = ids[i];
        out[i] = id == sentinel ? sentinel : rank[id];
    }
}

// One CTA per business (grid-stride): hop2(b) = U_{u in N(b)} N(u) \ {b} in a shared-memory bitmap
// over ranks.  Warps take the users of N(b) round-robin and walk their (ranked) lists id by id; the
// bitmap is then written to row rank(b) with 128-bit stores and its popcount is |hop2(b)|.  (The hub bitmaps of the
// business side are over ids, not ranks, so they are not used here: the whole build walks
// sum_u deg(u)^2 ids once per graph -- 205 M on C2.)
__global__ void __launch_bounds__(kIndexBuildThreads) k_build_biz_index(
    int n_biz, int words, const unsigned long long* __restrict__ b_row, const int* __restrict__ b_adj,
    const unsigned long long* __restrict__ u_row, const int* __restrict__ u_radj,
    const int* __restrict__ rank, unsigned* __restrict__ index, int* __restrict__ hop2) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    unsigned* bm = reinterpret_cast<unsigned*>(smem_raw);
    uint4* bm4 = reinterpret_cast<uint4*>(smem_raw);
    __shared__ int s_cnt;
    constexpr int NW = kIndexBuildThreads / 32;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int n4 = words >> 2;   // words is a multiple of 4
    for (int b = blockIdx.x; b < n_biz; b += gridDim.x) {
        for (int i = tid; i < n4; i += kIndexBuildThreads) bm4[i] = make_uint4(0u, 0u, 0u, 0u);
        if (tid == 0) s_cnt = 0;
        __syncthreads();
        const unsigned long long brow = b_row[b];
        const int bdeg = row_deg(brow);
        const int* users = b_adj + row_first4(brow) * 4;
        for (int j = warp; j < bdeg; j += NW) {
            const unsigned long long ur = u_row[users[j]];
            const int* ids = u_radj + row_first4(ur) * 4;
            for (int i = lane; i < row_deg(ur); i += 32) {
                const int r = ids[i];
                const unsigned bit = 1u << (r & 31);
                if (!(bm[r >> 5] & bit)) atomicOr(&bm[r >> 5], bit);
            }
        }
        __syncthreads();
        if (tid == 0 && bdeg > 0) {   // hop2(b) excludes b
            const int r = rank[b];
            bm[r >> 5] &= ~(1u << (r & 31));
        }
        __syncthreads();
        uint4* dst = reinterpret_cast<uint4*>(index + (size_t)rank[b] * words);
        int cnt = 0;
        for (int i = tid; i < n4; i += kIndexBuildThreads) {
            const uint4 v = bm4[i];
            cnt += __popc(v.x) + __popc(v.y) + __popc(v.z) + __popc(v.w);
            dst[i] = v;
        }
        cnt = __reduce_add_sync(kFull, cnt);
        if (lane == 0 && cnt) atomicAdd(&s_cnt, cnt);
        __syncthreads();
        if (tid == 0) hop2[b] = s_cnt;
        __syncthreads();   // the bitmap and s_cnt are cleared for the next business
    }
}

// Bit (rb, r) of the index: row max, column min.  Padding (r = the sentinel n_biz, weight 0) stays
// on the pair's own row rb at column n_biz, whose bit is never set: row n_biz does not exist.
__device__ __forceinline__ unsigned index_bit(const unsigned* index, int words, int n_biz, int rb, int r,
                                              unsigned long long pol) {
    const bool swap = r > rb && r < n_biz;
    const int row = swap ? r : rb, col = swap ? rb : r;
    return (ldg_keep(index + (size_t)row * (size_t)words + (col >> 5), pol) >> (col & 31)) & 1u;
}

// four ids of N(u) (as ranks) against business rank rb
__device__ __forceinline__ void index_test4(const unsigned* index, int words, int n_biz, int rb, int4 v,
                                            uint4 wt, unsigned& cnt, unsigned long long& acc,
                                            unsigned long long pol) {
    const unsigned h0 = index_bit(index, words, n_biz, rb, v.x, pol);
    const unsigned h1 = index_bit(index, words, n_biz, rb, v.y, pol);
    const unsigned h2 = index_bit(index, words, n_biz, rb, v.z, pol);
    const unsigned h3 = index_bit(index, words, n_biz, rb, v.w, pol);
    cnt += h0 + h1 + h2 + h3;
    acc += (unsigned long long)(h0 * wt.x) + (unsigned long long)(h1 * wt.y) +
           (unsigned long long)(h2 * wt.z) + (unsigned long long)(h3 * wt.w);
}

// One thread per pair, in the caller's order (x = business b, y = user u).  A lane scores its own
// pair when deg(u) <= kIndexLaneDeg.  The longer lists of the CTA's pairs are cut into their 128-bit
// words, laid end to end, and all threads of the CTA take those words round-robin, adding their hits
// to the pair's counters in shared memory (integer sums: the order does not matter).  Pairs come in
// runs of one user, so a user with thousands of businesses fills a whole warp with long lists: on
// one warp its run takes sum(deg) / 128 dependent load rounds (C2: up to 714), spread over the CTA
// an eighth of that.
__global__ void __launch_bounds__(kIndexScoreThreads) k_score_biz_indexed(
    SideArgs a, const int* __restrict__ pair_b, const int* __restrict__ pair_u, long long n, int n_mid,
    const int* __restrict__ b_deg, const int* __restrict__ u_deg, const int* __restrict__ u_radj,
    const unsigned* __restrict__ index, const int* __restrict__ hop2v, const int* __restrict__ rank,
    int words) {
    constexpr int NW = kIndexScoreThreads / 32;
    __shared__ int s_warp[NW];
    __shared__ int s_end[kIndexScoreThreads];   // end of each pair's long-list words (inclusive scan)
    __shared__ unsigned long long s_row[kIndexScoreThreads];
    __shared__ int s_rb[kIndexScoreThreads];
    __shared__ unsigned s_cnt[kIndexScoreThreads];
    __shared__ unsigned long long s_acc[kIndexScoreThreads];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const long long i = (long long)blockIdx.x * kIndexScoreThreads + tid;
    const unsigned long long pol = l2_keep_policy();
    const int4* adj4 = reinterpret_cast<const int4*>(u_radj);   // N(u) as ranks, beside u_adjw
    const uint4* adjw4 = reinterpret_cast<const uint4*>(a.m_adjw);
    const bool in = i < n;
    int b = 0, u = 0;
    if (in) {
        b = ld_once(pair_b + i);
        u = ld_once(pair_u + i);
    }
    const bool valid = in && group_key(b, u, a.n_side, n_mid, b_deg, u_deg) < a.n_side;
    unsigned long long urow = 0ull;
    int hop2 = 0, rb = 0;
    if (valid) {
        urow = a.m_row[u];
        hop2 = hop2v[b];
        rb = rank[b];
    }
    const int pdeg = row_deg(urow);   // 0 for an invalid pair: nothing to walk
    const int n_biz = a.n_side;
    const int n4 = (pdeg + 3) >> 2;
    const bool lng = pdeg > kIndexLaneDeg;
    int end = lng ? n4 : 0;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int t = __shfl_up_sync(kFull, end, d);
        if (lane >= d) end += t;
    }
    if (lane == 31) s_warp[warp] = end;
    s_row[tid] = urow;
    s_rb[tid] = rb;
    s_cnt[tid] = 0u;
    s_acc[tid] = 0ull;
    __syncthreads();
    int total = 0;
#pragma unroll
    for (int w = 0; w < NW; ++w) {
        if (w == warp) end += total;
        total += s_warp[w];
    }
    s_end[tid] = end;

    unsigned cnt = 0;
    unsigned long long acc = 0ull;
    if (!lng) {
        const long long f4 = row_first4(urow);
        for (int k = 0; k < n4; ++k)
            index_test4(index, words, n_biz, rb, ldg_stream(adj4 + f4 + k, pol), ldg_stream_u(adjw4 + f4 + k, pol),
                        cnt, acc, pol);
    }
    if (total > 0) {   // the same on every thread of the CTA
        __syncthreads();
        int cur = -1;
        unsigned c = 0;
        unsigned long long s = 0ull;
        for (int j = tid; j < total; j += kIndexScoreThreads) {
            int p = 0;   // the pair word j belongs to: the first with s_end[p] > j
#pragma unroll
            for (int step = kIndexScoreThreads / 2; step > 0; step >>= 1)
                if (s_end[p + step - 1] <= j) p += step;
            if (p != cur) {
                if (cur >= 0) {
                    atomicAdd(&s_cnt[cur], c);
                    atomicAdd(&s_acc[cur], s);
                }
                cur = p;
                c = 0;
                s = 0ull;
            }
            const unsigned long long r = s_row[p];
            const long long w4 = row_first4(r) + j - (s_end[p] - ((row_deg(r) + 3) >> 2));
            index_test4(index, words, n_biz, s_rb[p], ldg_stream(adj4 + w4, pol), ldg_stream_u(adjw4 + w4, pol),
                        c, s, pol);
        }
        if (cur >= 0) {
            atomicAdd(&s_cnt[cur], c);
            atomicAdd(&s_acc[cur], s);
        }
        __syncthreads();
        if (lng) {
            cnt = s_cnt[tid];
            acc = s_acc[tid];
        }
    }
    if (in) emit_pair<false>(a, i, (int)i, valid, (int)cnt, hop2, (valid && a.pa) ? b_deg[b] : 0, pdeg, acc);
}

// Decides whether the handle gets a business index and allocates it (before the hub tables and
// class flags, which the business side only needs without one).  Automatic: the business side runs
// unranged and the rows take at most min(1/16 of the device's memory, 8 GiB) and half of what is
// free -- C2 (465 MB), C3 and C4 (4.5 GB each) qualify on a B200, C5 (1M businesses: 125 GB) does
// not; the cap keeps a graph-lifetime structure from crowding out the per-call scratch of other
// handles.  An allocation that fails leaves the handle on the grouped path.
void reserve_biz_index(blp_graph* g) {
    const int mode = g->tune.biz_index;   // (BLP_BIZ_INDEX, read at handle creation)
    if (mode == 0 || g->n_ranges[BLP_SIDE_BUSINESS] != 1 || g->n_biz <= 0) return;
    const int words = bitmap_words(g->n_biz);
    const size_t bytes = (size_t)g->n_biz * (size_t)words * 4;
    if ((size_t)words * 4 > (size_t)g->max_smem_optin) return;   // the build's bitmap
    size_t free_b = 0, total_b = 0;
    if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) {
        (void)cudaGetLastError();
        return;
    }
    size_t cap = std::min<size_t>(total_b / 16, (size_t)8 << 30);
    if (g->tune.biz_index_cap > 0) cap = (size_t)g->tune.biz_index_cap;   // (BLP_BIZ_INDEX_MAX_MB)
    if (mode < 0 && (bytes > cap || bytes > free_b / 2)) return;
    if (cudaMalloc((void**)&g->biz_index, bytes) != cudaSuccess ||
        cudaMalloc((void**)&g->biz_hop2, sizeof(int) * (size_t)g->n_biz) != cudaSuccess ||
        cudaMalloc((void**)&g->biz_radj, sizeof(int) * (size_t)g->u_adj_len) != cudaSuccess ||
        cudaMalloc((void**)&g->biz_rank, sizeof(int) * (size_t)g->n_biz) != cudaSuccess) {
        (void)cudaGetLastError();
        cudaFree(g->biz_index);
        cudaFree(g->biz_hop2);
        cudaFree(g->biz_radj);
        cudaFree(g->biz_rank);
        g->biz_index = nullptr;
        g->biz_hop2 = g->biz_radj = g->biz_rank = nullptr;
        return;
    }
    g->biz_index_words = words;
    g->biz_index_bytes = (int64_t)bytes;
    g->device_bytes += (int64_t)bytes + (int64_t)sizeof(int) * (2 * (int64_t)g->n_biz + g->u_adj_len);
}

// Fills the reserved index: business ranks by degree (descending, ties by id, kept on the handle:
// the kernel reads rank(b) per pair), the ranked copy of the user rows, then the rows.
int build_biz_index(blp_graph* g, const int* b_deg_host) {
    if (!g->biz_index) return BLP_OK;
    const int n_biz = g->n_biz, words = g->biz_index_words;
    const auto t0 = std::chrono::steady_clock::now();
    std::vector<int> order((size_t)n_biz), rank((size_t)n_biz);
    for (int b = 0; b < n_biz; ++b) order[b] = b;
    std::stable_sort(order.begin(), order.end(), [&](int x, int y) { return b_deg_host[x] > b_deg_host[y]; });
    for (int r = 0; r < n_biz; ++r) rank[order[r]] = r;
    const size_t smem = (size_t)words * 4;
    const int rc = kernel_ctas_per_sm((const void*)k_build_biz_index, g->device, kIndexBuildThreads, smem, nullptr);
    if (rc != BLP_OK) return rc;
    cudaError_t e = cudaMemcpy(g->biz_rank, rank.data(), sizeof(int) * (size_t)n_biz, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) {
        k_rank_ids<<<g->sm_count * 8, 256>>>(g->u_adj, g->u_adj_len, g->biz_rank, n_biz, g->biz_radj);
        k_build_biz_index<<<std::min(n_biz, g->sm_count * 8), kIndexBuildThreads, smem>>>(
            n_biz, words, (const unsigned long long*)g->b_row, g->b_adj,
            (const unsigned long long*)g->u_row, g->biz_radj, g->biz_rank, g->biz_index, g->biz_hop2);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e != cudaSuccess) return blp::cuda_fail(e, "building the business index", __FILE__, __LINE__);
    g->biz_index_build_ms =
        std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
    return BLP_OK;
}

// The business side of blp_score_pairs on a handle with an index: one launch, caller order in
// and out.  Events 0 and 1 bracket nothing (no grouping), 1..2 the kernel.
int score_biz_indexed(blp_graph* g, const SideArgs& a, const int32_t* pair_u, const int32_t* pair_b,
                      int64_t n, cudaStream_t st) {
    blp_score_stats_t& stats = g->stats[BLP_SIDE_BUSINESS];
    const int grid = (int)((n + kIndexScoreThreads - 1) / kIndexScoreThreads);
    BLP_CUDA_TRY(cudaEventRecord(g->ev[BLP_SIDE_BUSINESS][0], st));
    BLP_CUDA_TRY(cudaEventRecord(g->ev[BLP_SIDE_BUSINESS][1], st));
    k_score_biz_indexed<<<grid, kIndexScoreThreads, 0, st>>>(a, pair_b, pair_u, n, g->n_users, g->b_deg,
                                                            g->u_deg, g->biz_radj, g->biz_index,
                                                            g->biz_hop2, g->biz_rank, g->biz_index_words);
    BLP_CUDA_TRY(cudaGetLastError());
    if (cudaEventRecord(g->ev[BLP_SIDE_BUSINESS][2], st) == cudaSuccess) g->ev_recorded[BLP_SIDE_BUSINESS] = true;
    stats.path = BLP_PATH_BIZ_INDEX;
    stats.ctas = grid;
    stats.threads_per_cta = kIndexScoreThreads;
    stats.smem_bytes = 0;
    stats.kernel_launches = 1;
    stats.range_passes = 1;
    return BLP_OK;
}

}  // namespace blp

#endif  // BLP_SCORE_INDEX_CUH_
