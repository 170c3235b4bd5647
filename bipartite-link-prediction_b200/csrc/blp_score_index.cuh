// Business index: the business side without grouping.
//
// For a pair (u, b) the business side needs |hop2(b) & N(u)|, its weight sum and |hop2(b)|.
// b' is in hop2(b) iff b' != b and b, b' share a reviewer -- a relation of the graph alone, the
// same on every call.  So it is built once per graph as one bitmap row per business (the
// co-review pattern of A^T A without its diagonal), and a call scores every pair in the caller's
// order by testing N(u) (4.8 ids on average on C2) against row b: no counting sort, no per-call
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

#ifndef BLP_BIZ_INDEX_KEEP
#define BLP_BIZ_INDEX_KEEP 1   // 0: index-row loads without the evict_last policy (A/B build)
#endif

namespace blp {

constexpr int kIndexBuildThreads = 512;
constexpr int kIndexScoreThreads = 256;
// pairs with deg(u) <= this are scored by their own lane (C2: 96.6 % of the pairs); the longer
// ones by the whole warp, 128 ids per pass
constexpr int kIndexLaneDeg = 16;

// Columns are kept in DEGREE-RANK order: bit rank(b') of a row stands for business b' (rank 0 =
// the most-reviewed business).  The ids a pair tests are the businesses of N(u), and reviews are
// power-law distributed over businesses, so most tests land in the first few hundred bits of a
// row: a few 32-byte sectors per row instead of one per id.  The rows themselves stay in id order.
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
// row is then written with 128-bit stores and its popcount is |hop2(b)|.  (The hub bitmaps of the
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
        uint4* dst = reinterpret_cast<uint4*>(index + (size_t)b * words);
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

__device__ __forceinline__ unsigned index_word(const unsigned* p, unsigned long long pol) {
#if BLP_BIZ_INDEX_KEEP
    return ldg_keep(p, pol);
#else
    (void)pol;
    return __ldg(p);
#endif
}

// four ids of N(u) (padding: the sentinel n_biz, whose bit is never set, weight 0) against row b
__device__ __forceinline__ void index_test4(const unsigned* row, int4 v, uint4 wt, unsigned& cnt,
                                            unsigned long long& acc, unsigned long long pol) {
    const unsigned w0 = index_word(row + (v.x >> 5), pol), w1 = index_word(row + (v.y >> 5), pol);
    const unsigned w2 = index_word(row + (v.z >> 5), pol), w3 = index_word(row + (v.w >> 5), pol);
    const unsigned h0 = (w0 >> (v.x & 31)) & 1u, h1 = (w1 >> (v.y & 31)) & 1u;
    const unsigned h2 = (w2 >> (v.z & 31)) & 1u, h3 = (w3 >> (v.w & 31)) & 1u;
    cnt += h0 + h1 + h2 + h3;
    acc += (unsigned long long)(h0 * wt.x) + (unsigned long long)(h1 * wt.y) +
           (unsigned long long)(h2 * wt.z) + (unsigned long long)(h3 * wt.w);
}

// One thread per pair, in the caller's order (x = business b, y = user u).  A lane scores its own
// pair when deg(u) <= kIndexLaneDeg; the warp then walks the longer lists of its 32 pairs together.
__global__ void __launch_bounds__(kIndexScoreThreads) k_score_biz_indexed(
    SideArgs a, const int* __restrict__ pair_b, const int* __restrict__ pair_u, long long n, int n_mid,
    const int* __restrict__ b_deg, const int* __restrict__ u_deg, const int* __restrict__ u_radj,
    const unsigned* __restrict__ index, const int* __restrict__ hop2v, int words) {
    const long long i = (long long)blockIdx.x * kIndexScoreThreads + threadIdx.x;
    const int lane = threadIdx.x & 31;
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
    int hop2 = 0;
    if (valid) {
        urow = a.m_row[u];
        hop2 = hop2v[b];
    }
    const int pdeg = row_deg(urow);
    const unsigned* row = index + (size_t)(valid ? b : 0) * (size_t)words;
    unsigned cnt = 0;
    unsigned long long acc = 0ull;
    const bool own = valid && pdeg <= kIndexLaneDeg;
    if (own) {
        const long long f4 = row_first4(urow);
        const int n4 = (pdeg + 3) >> 2;
        for (int k = 0; k < n4; ++k)
            index_test4(row, ldg_stream(adj4 + f4 + k, pol), ldg_stream_u(adjw4 + f4 + k, pol), cnt, acc,
                        pol);
    }
    unsigned todo = __ballot_sync(kFull, valid && !own);
    while (todo) {
        const int src = __ffs(todo) - 1;
        todo &= todo - 1;
        const unsigned long long r = __shfl_sync(kFull, urow, src);
        const unsigned* rb = index + (size_t)__shfl_sync(kFull, b, src) * (size_t)words;
        const long long f4 = row_first4(r);
        const int n4 = (row_deg(r) + 3) >> 2;
        unsigned c = 0;
        unsigned long long s = 0ull;
        for (int k = lane; k < n4; k += 32)
            index_test4(rb, ldg_stream(adj4 + f4 + k, pol), ldg_stream_u(adjw4 + f4 + k, pol), c, s, pol);
        c = __reduce_add_sync(kFull, c);
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) s += __shfl_xor_sync(kFull, s, d);
        if (lane == src) {
            cnt = c;
            acc = s;
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
        cudaMalloc((void**)&g->biz_radj, sizeof(int) * (size_t)g->u_adj_len) != cudaSuccess) {
        (void)cudaGetLastError();
        cudaFree(g->biz_index);
        cudaFree(g->biz_hop2);
        cudaFree(g->biz_radj);
        g->biz_index = nullptr;
        g->biz_hop2 = g->biz_radj = nullptr;
        return;
    }
    g->biz_index_words = words;
    g->biz_index_bytes = (int64_t)bytes;
    g->device_bytes += (int64_t)bytes + (int64_t)sizeof(int) * (g->n_biz + g->u_adj_len);
}

// Fills the reserved index: business ranks by degree (descending, ties by id), the ranked copy of
// the user rows, then the rows.
int build_biz_index(blp_graph* g, const int* b_deg_host) {
    if (!g->biz_index) return BLP_OK;
    const int n_biz = g->n_biz, words = g->biz_index_words;
    const auto t0 = std::chrono::steady_clock::now();
    std::vector<int> order((size_t)n_biz), rank((size_t)n_biz);
    for (int b = 0; b < n_biz; ++b) order[b] = b;
    std::stable_sort(order.begin(), order.end(), [&](int x, int y) { return b_deg_host[x] > b_deg_host[y]; });
    for (int r = 0; r < n_biz; ++r) rank[order[r]] = r;
    int* d_rank = nullptr;
    BLP_CUDA_TRY(cudaMalloc((void**)&d_rank, sizeof(int) * (size_t)n_biz));
    cudaError_t e = cudaMemcpy(d_rank, rank.data(), sizeof(int) * (size_t)n_biz, cudaMemcpyHostToDevice);
    const size_t smem = (size_t)words * 4;
    if (e == cudaSuccess && smem > 48 * 1024)
        e = cudaFuncSetAttribute(k_build_biz_index, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) {
        k_rank_ids<<<g->sm_count * 8, 256>>>(g->u_adj, g->u_adj_len, d_rank, n_biz, g->biz_radj);
        k_build_biz_index<<<std::min(n_biz, g->sm_count * 8), kIndexBuildThreads, smem>>>(
            n_biz, words, (const unsigned long long*)g->b_row, g->b_adj,
            (const unsigned long long*)g->u_row, g->biz_radj, d_rank, g->biz_index, g->biz_hop2);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    cudaFree(d_rank);
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
                                                            g->biz_hop2, g->biz_index_words);
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
