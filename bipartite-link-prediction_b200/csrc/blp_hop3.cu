// Candidate generation on the device (SURVEY.md section 8f, rank 2): for every given user the
// businesses at BFS distance exactly 3, i.e. what make_examples obtains from
// snap.GetNodesAtHop(G, u, 3, candidate_businesses, True) (dataset_maker.py:137-139):
//
//   hop2(u) = ( U_{b in N(u)} N(b) ) \ {u}          user bitmap
//   hop3(u) = ( U_{w in hop2(u)} N(w) ) \ N(u)      business bitmap in shared memory
//
// One CTA per user, pulled from an atomic counter.  The first call counts, the second writes the
// ids in ascending order at caller-provided offsets.  The user bitmap lives in shared memory when
// both bitmaps fit one CTA (C1-C4); for larger user universes (C5: 10 M users = 1.25 MB) every
// CTA owns a slice of a global scratch bitmap instead, kept all-zero between users by walking the
// same lists again (an undo pass touches only the words that were set, a clear would touch all).
#include <algorithm>
#include <climits>
#include <cstdio>

#include "blp_internal.h"

namespace blp {
namespace {

constexpr unsigned kAll = 0xffffffffu;

__device__ __forceinline__ int h3_deg(unsigned long long row) { return (int)(row & 0xffffffull); }
__device__ __forceinline__ const int* h3_list(const int* adj, unsigned long long row) {
    return adj + (long long)((row >> 24) & ((1ull << BLP_ROW_FIRST4_BITS) - 1)) * 4;
}

struct Hop3Args {
    const unsigned long long* __restrict__ u_row;
    const int* __restrict__ u_adj;
    const unsigned long long* __restrict__ b_row;
    const int* __restrict__ b_adj;
    int n_users, n_biz, uw, bw;            // bitmap words
    const int* __restrict__ users;
    long long n;
    long long* counts;                     // count pass
    const long long* offsets;              // fill pass
    int* out_biz;
    int* work_counter;
    unsigned* ubm_global;                  // null: user bitmap in shared memory; else [gridDim.x][uw]
};

template <bool FILL>
__global__ void __launch_bounds__(256) k_hop3(Hop3Args a) {
    extern __shared__ __align__(16) unsigned h3_smem[];
    // users at distance 2 / businesses at distance 3
    unsigned* ubm = a.ubm_global ? a.ubm_global + (size_t)blockIdx.x * (size_t)a.uw : h3_smem;
    unsigned* bbm = a.ubm_global ? h3_smem : h3_smem + a.uw;
    const int n_clear = a.ubm_global ? a.bw : a.uw + a.bw;   // (the global slice is kept clean)
    __shared__ int s_item;
    __shared__ int s_scan[9];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (;;) {
        __syncthreads();
        if (tid == 0) s_item = atomicAdd(a.work_counter, 1);
        __syncthreads();
        const long long it = s_item;
        if (it >= a.n) break;
        const int u = a.users[it];
        const bool ok = u >= 0 && u < a.n_users && h3_deg(a.u_row[u]) > 0;
        if (!ok) {
            if (!FILL && tid == 0) a.counts[it] = 0;
            continue;
        }
        for (int i = tid; i < n_clear; i += 256) h3_smem[i] = 0u;
        __syncthreads();
        const unsigned long long urow = a.u_row[u];
        const int* nu = h3_list(a.u_adj, urow);
        const int du = h3_deg(urow);
        // hop 2: one warp per business of u, lanes stride its user list
        for (int k = warp; k < du; k += 8) {
            const unsigned long long brow = a.b_row[nu[k]];
            const int* lst = h3_list(a.b_adj, brow);
            for (int j = lane; j < h3_deg(brow); j += 32) {
                const int w = lst[j];
                atomicOr(&ubm[w >> 5], 1u << (w & 31));
            }
        }
        __syncthreads();
        if (tid == 0) atomicAnd(&ubm[u >> 5], ~(1u << (u & 31)));   // distance 0, not 2
        __syncthreads();
        // hop 3: a warp takes 32 words of the user bitmap at a time; the users found in them are
        // dealt to the lanes round-robin (a warp-wide prefix over the popcounts numbers them), so
        // the lanes walk about equally many of the (short) business lists instead of one lane
        // getting a dense word and its neighbours an empty one
        for (int base = warp * 32; base < a.uw; base += 8 * 32) {
            const int i = base + lane;
            // (global slice: the bits were set by atomics in L2 -- read there, not from a stale L1 line)
            unsigned m = i < a.uw ? (a.ubm_global ? __ldcg(ubm + i) : ubm[i]) : 0u;
            const int c = __popc(m);
            int inc = c;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const int t = __shfl_up_sync(kAll, inc, d);
                if (lane >= d) inc += t;
            }
            const int total = __shfl_sync(kAll, inc, 31);
            if (total == 0) continue;
            const int excl = inc - c;
            for (int r0 = 0; r0 < total; r0 += 32) {     // uniform trip count: the shuffles need every lane
                const bool active = r0 + lane < total;
                const int r = active ? r0 + lane : total - 1;
                // the r-th user of the 32 words sits in the word of lane L = #{lanes : inc <= r}
                int L = 0;
#pragma unroll
                for (int sft = 16; sft >= 1; sft >>= 1) {
                    const int t = __shfl_sync(kAll, inc, L + sft - 1);
                    if (t <= r) L += sft;
                }
                unsigned mm = __shfl_sync(kAll, m, L);
                const int skip = r - __shfl_sync(kAll, excl, L);
                if (active) {
                    for (int q = 0; q < skip; ++q) mm &= mm - 1;
                    const int w = (base + L) * 32 + __ffs(mm) - 1;
                    const unsigned long long wrow = a.u_row[w];
                    const int* lst = h3_list(a.u_adj, wrow);
                    for (int j = 0; j < h3_deg(wrow); ++j) {
                        const int b = lst[j];
                        atomicOr(&bbm[b >> 5], 1u << (b & 31));
                    }
                }
            }
        }
        __syncthreads();
        if (a.ubm_global) {
            // undo: the same lists once more, zeroing the words they set (every set bit of a touched
            // word belongs to this user's hop-2 set), so the slice is all-zero for the next user
            for (int k = warp; k < du; k += 8) {
                const unsigned long long brow = a.b_row[nu[k]];
                const int* lst = h3_list(a.b_adj, brow);
                for (int j = lane; j < h3_deg(brow); j += 32) ubm[lst[j] >> 5] = 0u;
            }
        }
        for (int k = tid; k < du; k += 256) {             // distance 1, not 3
            const int b = nu[k];
            atomicAnd(&bbm[b >> 5], ~(1u << (b & 31)));
        }
        __syncthreads();
        // count / ascending write: per-thread contiguous word ranges keep the order
        const int per = (a.bw + 255) / 256;
        const int w0 = min(a.bw, tid * per), w1 = min(a.bw, w0 + per);
        int mine = 0;
        for (int i = w0; i < w1; ++i) mine += __popc(bbm[i]);
        int inc = mine;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            int t = __shfl_up_sync(kAll, inc, d);
            if (lane >= d) inc += t;
        }
        if (lane == 31) s_scan[warp] = inc;
        __syncthreads();
        int before = inc - mine, total = 0;
#pragma unroll
        for (int w = 0; w < 8; ++w) {
            if (w < warp) before += s_scan[w];
            total += s_scan[w];
        }
        if (!FILL) {
            if (tid == 0) a.counts[it] = total;
        } else {
            int* dst = a.out_biz + a.offsets[it] + before;
            for (int i = w0; i < w1; ++i) {
                unsigned m = bbm[i];
                while (m) {
                    *dst++ = i * 32 + __ffs(m) - 1;
                    m &= m - 1;
                }
            }
        }
    }
}

int launch_hop3(blp_graph* g, Hop3Args a, bool fill, cudaStream_t st) {
    a.u_row = (const unsigned long long*)g->u_row;
    a.u_adj = g->u_adj;
    a.b_row = (const unsigned long long*)g->b_row;
    a.b_adj = g->b_adj;
    a.n_users = g->n_users;
    a.n_biz = g->n_biz;
    a.uw = (g->n_users + 31) / 32;
    a.bw = (g->n_biz + 31) / 32;
    // both bitmaps in shared memory when they fit; else only the business bitmap, and the user
    // bitmap of every CTA in global scratch (BLP_HOP3_GLOBAL=1 forces that, for tests)
    size_t smem = sizeof(unsigned) * ((size_t)a.uw + a.bw);
    const bool global_users = g->tune.hop3_global || smem + 1024 > (size_t)g->max_smem_optin;
    if (global_users) smem = sizeof(unsigned) * (size_t)a.bw;
    if (smem + 1024 > (size_t)g->max_smem_optin) {
        set_error("blp_hop3: the business bitmap alone exceeds one CTA's shared memory");
        return BLP_ERR_UNSUPPORTED;
    }
    void (*const kernel)(Hop3Args) = fill ? k_hop3<true> : k_hop3<false>;
    int per_sm = 0;
    const int rc = kernel_ctas_per_sm((const void*)kernel, g->device, 256, smem, &per_sm);
    if (rc != BLP_OK) return rc;
    int* counter = nullptr;
    BLP_CUDA_TRY(pool_alloc(g, (void**)&counter, sizeof(int), st));
    BLP_CUDA_TRY(cudaMemsetAsync(counter, 0, sizeof(int), st));
    a.work_counter = counter;
    int grid = std::max(1, per_sm) * g->sm_count;
    if (global_users) {
        // at most 1 GiB of scratch bitmaps: fewer CTAs rather than more memory
        const size_t per_cta = sizeof(unsigned) * (size_t)a.uw;
        grid = (int)std::max<size_t>(1, std::min<size_t>((size_t)grid, ((size_t)1 << 30) / std::max<size_t>(per_cta, 1)));
        BLP_CUDA_TRY(pool_alloc(g, (void**)&a.ubm_global, per_cta * (size_t)grid, st));
        BLP_CUDA_TRY(cudaMemsetAsync(a.ubm_global, 0, per_cta * (size_t)grid, st));
    }
    kernel<<<grid, 256, smem, st>>>(a);
    if (a.ubm_global) cudaFreeAsync(a.ubm_global, st);
    BLP_CUDA_TRY(cudaGetLastError());
    cudaFreeAsync(counter, st);
    return BLP_OK;
}

}  // namespace
}  // namespace blp

extern "C" int blp_hop3_count(blp_graph* g, const int32_t* users, int64_t n, int64_t* counts,
                              void* stream) {
    if (!g || n < 0 || n >= INT_MAX || (n > 0 && (!users || !counts))) {
        blp::set_error("blp_hop3_count: bad argument");
        return BLP_ERR_INVALID;
    }
    if (n == 0) return BLP_OK;
    BLP_ON_DEVICE(g->device);
    blp::Hop3Args a{};
    a.users = users;
    a.n = n;
    a.counts = (long long*)counts;
    return blp::launch_hop3(g, a, false, (cudaStream_t)stream);
}

extern "C" int blp_hop3_fill(blp_graph* g, const int32_t* users, int64_t n, const int64_t* offsets,
                             int32_t* out_biz, void* stream) {
    if (!g || n < 0 || n >= INT_MAX || (n > 0 && (!users || !offsets || !out_biz))) {
        blp::set_error("blp_hop3_fill: bad argument");
        return BLP_ERR_INVALID;
    }
    if (n == 0) return BLP_OK;
    BLP_ON_DEVICE(g->device);
    blp::Hop3Args a{};
    a.users = users;
    a.n = n;
    a.offsets = (const long long*)offsets;
    a.out_biz = out_biz;
    return blp::launch_hop3(g, a, true, (cudaStream_t)stream);
}
