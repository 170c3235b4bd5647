// Graph construction on the device (SURVEY.md section 8f, rank 1: the step in front of the path).
// Replaces snap.LoadEdgeList(snap.PUNGraph, graph_file, 0, 1) (similarity.py:16).  Both create
// functions run the one builder here: blp_graph_create_device on edge arrays already in HBM,
// blp_graph_create after copying its host arrays to the device.
//
//   keys (u << 32 | b)  --LSD radix sort, 8 bits per pass, only the bits in use-->  sorted keys
//   --adjacent-difference flags + scan-->  distinct edges (duplicates collapse, SNAP TUNGraph)
//   --degrees, padded row offsets (scan)-->  user rows (from the sorted order), business rows
//   (atomic cursors)  --bank striping, sentinels, per-entry weights, row descriptors.
#include <algorithm>
#include <climits>
#include <cstdio>
#include <cstdlib>
#include <new>
#include <vector>

#include "blp_internal.h"

namespace blp {
namespace {

constexpr unsigned kFullMask = 0xffffffffu;
constexpr int kSortTile = 4096;   // keys per CTA per radix pass (256 threads x 16)

// ------------------------------------------------------------------------------------ scans
// Exclusive scan of n 32-bit counts into 64-bit offsets: per-4096 block sums, a single-CTA scan
// of the block sums, and a final pass.  `round4` pads every count to a multiple of four first.
__device__ __forceinline__ unsigned long long pad4(unsigned v, bool round4) {
    return round4 ? (((unsigned long long)v + 3ull) & ~3ull) : (unsigned long long)v;
}

__global__ void __launch_bounds__(256) k_scan_block_sums(const unsigned* __restrict__ in, long long n,
                                                         bool round4,
                                                         unsigned long long* __restrict__ sums) {
    __shared__ unsigned long long s_w[8];
    const long long lo = (long long)blockIdx.x * kSortTile + threadIdx.x * 16;
    unsigned long long v = 0;
#pragma unroll
    for (int j = 0; j < 16; ++j)
        if (lo + j < n) v += pad4(in[lo + j], round4);
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(kFullMask, v, d);
    if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long t = 0;
        for (int w = 0; w < 8; ++w) t += s_w[w];
        sums[blockIdx.x] = t;
    }
}

__global__ void __launch_bounds__(1024) k_scan_sums(unsigned long long* __restrict__ sums, int nb,
                                                    unsigned long long* __restrict__ total) {
    __shared__ unsigned long long s_w[32];
    __shared__ unsigned long long s_base;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) s_base = 0;
    __syncthreads();
    for (int start = 0; start < nb; start += 1024) {
        const int i = start + tid;
        const unsigned long long own = i < nb ? sums[i] : 0ull;
        unsigned long long v = own;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            unsigned long long t = __shfl_up_sync(kFullMask, v, d);
            if (lane >= d) v += t;
        }
        if (lane == 31) s_w[warp] = v;
        __syncthreads();
        unsigned long long wb = 0;
        for (int w = 0; w < warp; ++w) wb += s_w[w];
        const unsigned long long base = s_base;
        if (i < nb) sums[i] = base + wb + v - own;
        __syncthreads();
        if (tid == 1023) s_base = base + wb + v;
        __syncthreads();
    }
    if (tid == 0) *total = s_base;
}

__global__ void __launch_bounds__(256) k_scan_apply(const unsigned* __restrict__ in, long long n,
                                                    bool round4,
                                                    const unsigned long long* __restrict__ sums,
                                                    unsigned long long* __restrict__ out) {
    __shared__ unsigned long long s_w[8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long lo = (long long)blockIdx.x * kSortTile + threadIdx.x * 16;
    unsigned long long c[16], mine = 0;
#pragma unroll
    for (int j = 0; j < 16; ++j) {
        c[j] = lo + j < n ? pad4(in[lo + j], round4) : 0ull;
        mine += c[j];
    }
    unsigned long long inc = mine;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        unsigned long long t = __shfl_up_sync(kFullMask, inc, d);
        if (lane >= d) inc += t;
    }
    if (lane == 31) s_w[warp] = inc;
    __syncthreads();
    unsigned long long off = sums[blockIdx.x] + inc - mine;
    for (int w = 0; w < warp; ++w) off += s_w[w];
#pragma unroll
    for (int j = 0; j < 16; ++j) {
        if (lo + j < n) out[lo + j] = off;
        off += c[j];
    }
}

struct Scanner {
    cudaStream_t st;
    unsigned long long* sums = nullptr;
    unsigned long long* total = nullptr;
    long long cap = 0;
    int ensure(long long n) {
        const long long nb = (n + kSortTile - 1) / kSortTile;
        if (nb <= cap) return BLP_OK;
        if (sums) cudaFreeAsync(sums, st);
        BLP_CUDA_TRY(scratch_alloc((void**)&sums, sizeof(unsigned long long) * (size_t)(nb + 1), st));
        if (!total) BLP_CUDA_TRY(scratch_alloc((void**)&total, sizeof(unsigned long long), st));
        cap = nb;
        return BLP_OK;
    }
    // out[i] = sum of (padded) in[0..i);  *host_total = the grand total (synchronises the stream)
    int run(const unsigned* in, long long n, bool round4, unsigned long long* out,
            unsigned long long* host_total) {
        int rc = ensure(n);
        if (rc != BLP_OK) return rc;
        const int nb = (int)((n + kSortTile - 1) / kSortTile);
        k_scan_block_sums<<<nb, 256, 0, st>>>(in, n, round4, sums);
        k_scan_sums<<<1, 1024, 0, st>>>(sums, nb, total);
        k_scan_apply<<<nb, 256, 0, st>>>(in, n, round4, sums, out);
        BLP_CUDA_TRY(cudaGetLastError());
        if (host_total) {
            BLP_CUDA_TRY(cudaMemcpyAsync(host_total, total, sizeof(unsigned long long),
                                         cudaMemcpyDeviceToHost, st));
            BLP_CUDA_TRY(cudaStreamSynchronize(st));
        }
        return BLP_OK;
    }
    void release() {
        if (sums) cudaFreeAsync(sums, st);
        if (total) cudaFreeAsync(total, st);
        sums = total = nullptr;
    }
};

// ------------------------------------------------------------------------------------ radix sort
// One LSD pass over 8 bits.  k_radix_hist: per-tile digit histogram, stored digit-major
// ([digit][tile]) so that ONE exclusive scan over the whole matrix yields every (digit, tile)
// base.  k_radix_scatter: stable ranking inside the tile -- warps own consecutive strips, lanes
// rank equal digits with __match_any_sync, a per-warp running count keeps strip order.
__global__ void __launch_bounds__(256) k_radix_hist(const unsigned long long* __restrict__ keys,
                                                    long long n, int shift, int n_tiles,
                                                    unsigned* __restrict__ hist) {
    __shared__ unsigned s_h[256];
    s_h[threadIdx.x] = 0;
    __syncthreads();
    const long long lo = (long long)blockIdx.x * kSortTile;
    for (int j = threadIdx.x; j < kSortTile; j += 256)
        if (lo + j < n) atomicAdd(&s_h[(unsigned)(keys[lo + j] >> shift) & 255u], 1u);
    __syncthreads();
    hist[(size_t)threadIdx.x * n_tiles + blockIdx.x] = s_h[threadIdx.x];
}

__global__ void __launch_bounds__(256) k_radix_scatter(const unsigned long long* __restrict__ src,
                                                       unsigned long long* __restrict__ dst,
                                                       long long n, int shift, int n_tiles,
                                                       const unsigned long long* __restrict__ base) {
    __shared__ unsigned s_cnt[8][256];      // per warp: keys of each digit in the warp's strip
    __shared__ unsigned long long s_base[256];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const long long lo = (long long)blockIdx.x * kSortTile;
    for (int i = tid; i < 8 * 256; i += 256) (&s_cnt[0][0])[i] = 0;
    s_base[tid] = base[(size_t)tid * n_tiles + blockIdx.x];
    __syncthreads();
    // strip of warp w: keys [w*512, w*512+512) of the tile, read 32 at a time in order
    const long long strip = lo + warp * 512;
    unsigned long long key[16];
    unsigned rank[16];
#pragma unroll
    for (int r = 0; r < 16; ++r) {
        const long long i = strip + r * 32 + lane;
        const bool ok = i < n;
        key[r] = ok ? src[i] : 0ull;
        const unsigned digit = ok ? ((unsigned)(key[r] >> shift) & 255u) : 256u + lane;  // unique when absent
        const unsigned peers = __match_any_sync(kFullMask, digit);
        const unsigned before = __popc(peers & ((1u << lane) - 1u));
        unsigned seen = 0;
        if (ok) seen = s_cnt[warp][digit];
        rank[r] = seen + before;
        __syncwarp();
        if (ok && before == 0) s_cnt[warp][digit] = seen + __popc(peers);   // the leader adds the group
        __syncwarp();
    }
    __syncthreads();
    // exclusive prefix over the warps for every digit (thread = digit)
    {
        unsigned run = 0;
#pragma unroll
        for (int w = 0; w < 8; ++w) {
            const unsigned c = s_cnt[w][tid];
            s_cnt[w][tid] = run;
            run += c;
        }
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < 16; ++r) {
        const long long i = strip + r * 32 + lane;
        if (i < n) {
            const unsigned digit = (unsigned)(key[r] >> shift) & 255u;
            dst[s_base[digit] + s_cnt[warp][digit] + rank[r]] = key[r];
        }
    }
}

// ------------------------------------------------------------------------------------ build steps
__global__ void k_make_keys(const int* __restrict__ eu, const int* __restrict__ eb, long long n,
                            int n_users, int n_biz, unsigned long long* __restrict__ keys,
                            int* __restrict__ bad) {
    long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (; i < n; i += stride) {
        const int u = eu[i], b = eb[i];
        if (u < 0 || u >= n_users || b < 0 || b >= n_biz) {
            atomicMin(bad, (int)min(i, (long long)INT_MAX - 1));
            keys[i] = 0ull;
        } else {
            keys[i] = ((unsigned long long)(unsigned)u << 32) | (unsigned)b;
        }
    }
}

__global__ void k_unique_flags(const unsigned long long* __restrict__ keys, long long n,
                               unsigned* __restrict__ flag) {
    long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (; i < n; i += stride) flag[i] = (i == 0 || keys[i] != keys[i - 1]) ? 1u : 0u;
}

// distinct edges in sorted order + degree counts
__global__ void k_compact_edges(const unsigned long long* __restrict__ keys,
                                const unsigned* __restrict__ flag,
                                const unsigned long long* __restrict__ pos, long long n,
                                unsigned long long* __restrict__ edges, unsigned* __restrict__ u_deg,
                                unsigned* __restrict__ b_deg) {
    long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (; i < n; i += stride) {
        if (!flag[i]) continue;
        const unsigned long long k = keys[i];
        edges[pos[i]] = k;
        atomicAdd(&u_deg[(unsigned)(k >> 32)], 1u);
        atomicAdd(&b_deg[(unsigned)k], 1u);
    }
}

__global__ void k_fill(int* __restrict__ p, long long n, int v) {
    long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (; i < n; i += stride) p[i] = v;
}

// user rows straight from the sorted order; business rows through atomic cursors
__global__ void k_place_edges(const unsigned long long* __restrict__ edges, long long m,
                              const unsigned long long* __restrict__ u_first,
                              const unsigned long long* __restrict__ u_off,
                              const unsigned long long* __restrict__ b_off,
                              unsigned* __restrict__ b_cur, int* __restrict__ u_adj,
                              int* __restrict__ b_adj) {
    long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (; i < m; i += stride) {
        const unsigned u = (unsigned)(edges[i] >> 32), b = (unsigned)edges[i];
        u_adj[u_off[u] + ((unsigned long long)i - u_first[u])] = (int)b;
        b_adj[b_off[b] + atomicAdd(&b_cur[b], 1u)] = (int)u;
    }
}

__global__ void k_row_descriptors(const unsigned long long* __restrict__ off,
                                  const unsigned* __restrict__ deg, int n,
                                  unsigned long long* __restrict__ row, int* __restrict__ deg_out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        row[i] = ((off[i] >> 2) << 24) | (unsigned long long)deg[i];
        deg_out[i] = (int)deg[i];
    }
}

// Bank striping, one row per warp.  The kernels probe a shared-memory bitmap with one 32-bit load
// per id; word id>>5 lives in bank (id>>5)&31, so 32 random ids cost ~3 wavefronts instead of 1.
// Nothing in the algorithm needs a row in ascending order, so every row longer than the sub-warp
// path (16 ids) is permuted once here: the 32 ids that ONE load instruction touches (lane l reads
// component q of the int4 at index 32*block + l, i.e. slots 128*block + 4*l + q) are drawn from
// 32 different banks for as long as every bank still has ids left.  The ids are first bucketed by
// bank into `tmp`; id number r of bank b then goes to sequence position
//   e = sum_b' min(cnt[b'], r) + #{b' < b : cnt[b'] > r}
// (wave r holds one id of every bank that still has ids), and sequence position e of a full
// 128-slot block sits at slot 4*(e%32) + (e%128)/32 of that block -- the 32 ids one load
// instruction touches are 32 consecutive sequence positions.
__global__ void __launch_bounds__(256) k_bank_stripe(const unsigned long long* __restrict__ off,
                                                     const unsigned* __restrict__ deg, int n_rows,
                                                     int* __restrict__ adj, int* __restrict__ tmp,
                                                     int* __restrict__ next_row) {
    __shared__ int s_cnt[8][32], s_start[8][32], s_cur[8][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (;;) {
        int r = 0;
        if (lane == 0) r = atomicAdd(next_row, 1);
        r = __shfl_sync(kFullMask, r, 0);
        if (r >= n_rows) break;
        const int len = (int)deg[r];
        if (len <= 16) continue;
        int* row = adj + off[r];
        int* t = tmp + off[r];
        s_cnt[warp][lane] = 0;
        __syncwarp();
        for (int i = lane; i < len; i += 32) atomicAdd(&s_cnt[warp][(row[i] >> 5) & 31], 1);
        __syncwarp();
        const int c = s_cnt[warp][lane];
        int inc = c;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            int v = __shfl_up_sync(kFullMask, inc, d);
            if (lane >= d) inc += v;
        }
        s_start[warp][lane] = inc - c;
        s_cur[warp][lane] = inc - c;
        __syncwarp();
        for (int i = lane; i < len; i += 32) {
            const int id = row[i];
            t[atomicAdd(&s_cur[warp][(id >> 5) & 31], 1)] = id;
        }
        __syncwarp();
        const int full = (len / 128) * 128;
        for (int p = lane; p < len; p += 32) {
            const int id = t[p];
            const int b = (id >> 5) & 31;
            const int rk = p - s_start[warp][b];
            int e = 0;
#pragma unroll 8
            for (int bb = 0; bb < 32; ++bb) {
                const int cb = s_cnt[warp][bb];
                e += min(cb, rk) + ((bb < b && cb > rk) ? 1 : 0);
            }
            const int slot = e < full ? (e / 128) * 128 + 4 * (e % 32) + (e % 128) / 32 : e;
            row[slot] = id;
        }
        __syncwarp();
    }
}

__global__ void k_entry_weights(const int* __restrict__ adj, long long n_entries, int sentinel,
                                const unsigned* __restrict__ other_deg,
                                const unsigned* __restrict__ lut, unsigned* __restrict__ adjw) {
    long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (; i < n_entries; i += stride) {
        const int id = adj[i];
        adjw[i] = id == sentinel ? 0u : lut[other_deg[id]];
    }
}

int bits_for(unsigned v) {
    int b = 0;
    while (v) {
        ++b;
        v >>= 1;
    }
    return b ? b : 1;
}

}  // namespace

int exclusive_scan_u32(const unsigned* in, long long n, unsigned long long* out,
                       unsigned long long* host_total, cudaStream_t st) {
    if (n <= 0) {
        if (host_total) *host_total = 0;
        return BLP_OK;
    }
    Scanner scan;
    scan.st = st;
    const int rc = scan.run(in, n, false, out, host_total);
    scan.release();
    return rc;
}

// Sorts n 64-bit keys ascending on the bits named by `shifts` (8 bits from each shift, least
// significant group first).  `keys` and `tmp` are device buffers of n entries; the sorted keys
// end up where *sorted points (one of the two).  Stream-ordered, no host synchronisation.
int radix_sort_u64(unsigned long long* keys, unsigned long long* tmp, long long n,
                   const std::vector<int>& shifts, cudaStream_t st, unsigned long long** sorted) {
    *sorted = keys;
    if (n <= 1 || shifts.empty()) return BLP_OK;
    const int n_tiles = (int)((n + kSortTile - 1) / kSortTile);
    unsigned* hist = nullptr;
    unsigned long long* hbase = nullptr;
    BLP_CUDA_TRY(scratch_alloc((void**)&hist, sizeof(unsigned) * 256 * (size_t)n_tiles, st));
    cudaError_t e = scratch_alloc((void**)&hbase, sizeof(unsigned long long) * 256 * (size_t)n_tiles, st);
    if (e != cudaSuccess) {
        cudaFreeAsync(hist, st);
        return cuda_fail(e, "scratch_alloc(hbase)", __FILE__, __LINE__);
    }
    Scanner scan;
    scan.st = st;
    int rc = BLP_OK;
    for (int s : shifts) {
        k_radix_hist<<<n_tiles, 256, 0, st>>>(keys, n, s, n_tiles, hist);
        rc = scan.run(hist, 256LL * n_tiles, false, hbase, nullptr);
        if (rc != BLP_OK) break;
        k_radix_scatter<<<n_tiles, 256, 0, st>>>(keys, tmp, n, s, n_tiles, hbase);
        std::swap(keys, tmp);
    }
    if (rc == BLP_OK && cudaGetLastError() != cudaSuccess) rc = BLP_ERR_CUDA;
    scan.release();
    cudaFreeAsync(hist, st);
    cudaFreeAsync(hbase, st);
    *sorted = keys;
    return rc;
}
// ------------------------------------------------------------------------------------ graph.txt
// The text of graph.txt -- one "<user_id> <business_id>\n" per review (dataset_maker.py:197) -- is
// parsed where it will be used: the file's bytes go to the device as they are, a first pass
// counts the data lines of every 4 KB tile, a scan turns the counts into line numbers, and a
// second pass lets the thread that owns a line's first byte parse columns 0 and 1 (what
// snap.LoadEdgeList(PUNGraph, file, 0, 1) reads, similarity.py:16).  A data line is a line whose
// first non-blank character starts an integer; blank lines and comment lines are skipped, further
// columns ignored, "\r\n" accepted.
namespace {
constexpr int kParseTile = 4096;   // bytes per CTA: 256 threads x 16

__device__ __forceinline__ bool parse_blank(char c) { return c == ' ' || c == '\t' || c == '\r'; }
__device__ __forceinline__ bool parse_digit(char c) { return c >= '0' && c <= '9'; }

__device__ __forceinline__ bool data_line_at(const char* __restrict__ t, long long n, long long i) {
    if (i > 0 && t[i - 1] != '\n') return false;
    long long j = i;
    while (j < n && parse_blank(t[j])) ++j;
    if (j >= n) return false;
    const char c = t[j];
    if (c == '-' || c == '+') return j + 1 < n && parse_digit(t[j + 1]);
    return parse_digit(c);
}

// one whitespace-separated integer starting at or after j (never crosses the line's end)
__device__ __forceinline__ bool parse_int(const char* __restrict__ t, long long n, long long& j, long long& out) {
    while (j < n && parse_blank(t[j])) ++j;
    if (j >= n) return false;
    bool neg = false;
    if (t[j] == '-' || t[j] == '+') {
        neg = t[j] == '-';
        ++j;
    }
    if (j >= n || !parse_digit(t[j])) return false;
    long long v = 0;
    while (j < n && parse_digit(t[j])) {
        v = v * 10 + (t[j] - '0');
        ++j;
    }
    out = neg ? -v : v;
    return true;
}

__global__ void __launch_bounds__(256) k_parse_count(const char* __restrict__ t, long long n,
                                                     unsigned* __restrict__ tile_cnt) {
    __shared__ unsigned s_w[8];
    const long long lo = (long long)blockIdx.x * kParseTile + threadIdx.x * 16;
    unsigned c = 0;
#pragma unroll
    for (int j = 0; j < 16; ++j)
        if (lo + j < n) c += data_line_at(t, n, lo + j) ? 1u : 0u;
    c = __reduce_add_sync(kFullMask, c);
    if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned tot = 0;
        for (int w = 0; w < 8; ++w) tot += s_w[w];
        tile_cnt[blockIdx.x] = tot;
    }
}

__global__ void __launch_bounds__(256) k_parse_lines(const char* __restrict__ t, long long n,
                                                     const unsigned long long* __restrict__ tile_base,
                                                     long long n_lines, long long* __restrict__ col0,
                                                     long long* __restrict__ col1,
                                                     unsigned long long* __restrict__ bad_line) {
    __shared__ unsigned s_w[8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long lo = (long long)blockIdx.x * kParseTile + threadIdx.x * 16;
    unsigned mask = 0;
#pragma unroll
    for (int j = 0; j < 16; ++j)
        if (lo + j < n && data_line_at(t, n, lo + j)) mask |= 1u << j;
    const unsigned c = __popc(mask);
    unsigned inc = c;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const unsigned v = __shfl_up_sync(kFullMask, inc, d);
        if (lane >= d) inc += v;
    }
    if (lane == 31) s_w[warp] = inc;
    __syncthreads();
    unsigned long long line = tile_base[blockIdx.x] + inc - c;
    for (int w = 0; w < warp; ++w) line += s_w[w];
    while (mask) {
        const int j = __ffs(mask) - 1;
        mask &= mask - 1;
        long long at = lo + j, a = 0, b = 0;
        const bool ok = parse_int(t, n, at, a) && parse_int(t, n, at, b);
        if ((long long)line < n_lines) {
            col0[line] = a;
            col1[line] = b;
        }
        if (!ok) atomicMin(bad_line, line);
        ++line;
    }
}

int parse_tile_counts(const char* text, long long n_bytes, cudaStream_t st, unsigned** tile_cnt_out, int* n_tiles_out) {
    const long long n_tiles = (n_bytes + kParseTile - 1) / kParseTile;
    if (n_tiles >= (1LL << 31)) {
        set_error("edge list text too large (more than 8 TB)");
        return BLP_ERR_UNSUPPORTED;
    }
    unsigned* tile_cnt = nullptr;
    BLP_CUDA_TRY(scratch_alloc((void**)&tile_cnt, sizeof(unsigned) * (size_t)std::max<long long>(n_tiles, 1), st));
    if (n_tiles > 0) k_parse_count<<<(unsigned)n_tiles, 256, 0, st>>>(text, n_bytes, tile_cnt);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        cudaFreeAsync(tile_cnt, st);
        return cuda_fail(e, "k_parse_count", __FILE__, __LINE__);
    }
    *tile_cnt_out = tile_cnt;
    *n_tiles_out = (int)n_tiles;
    return BLP_OK;
}
}  // namespace

// ------------------------------------------------------------------------------------ id ranges
// One warp per row of a ranged side's middle adjacency: count the ids of every id range, write the
// exclusive prefix to seg_off[row][0..R] and move the ids so that range 0's come first, then range
// 1's, ... (order inside a range is free).  The padding at the row's tail (sentinel ids) is not
// touched and belongs to no segment.
namespace {
__global__ void __launch_bounds__(256) k_range_segments(const unsigned long long* __restrict__ row_desc,
                                                        int n_rows, int* __restrict__ adj,
                                                        int* __restrict__ tmp, int range_bits, int n_ranges,
                                                        int* __restrict__ seg_off, int* __restrict__ next_row) {
    __shared__ int s_cnt[8][kMaxRanges + 1], s_cur[8][kMaxRanges + 1];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (;;) {
        int r = 0;
        if (lane == 0) r = atomicAdd(next_row, 1);
        r = __shfl_sync(kFullMask, r, 0);
        if (r >= n_rows) break;
        const unsigned long long d = row_desc[r];
        const int len = (int)(d & 0xffffffull);
        const long long first = (long long)((d >> 24) & ((1ull << BLP_ROW_FIRST4_BITS) - 1)) * 4;
        int* row = adj + first;
        for (int k = lane; k <= n_ranges; k += 32) s_cnt[warp][k] = 0;
        __syncwarp();
        for (int i = lane; i < len; i += 32) atomicAdd(&s_cnt[warp][row[i] / range_bits + 1], 1);
        __syncwarp();
        if (lane == 0) {
            int run = 0;
            for (int k = 0; k <= n_ranges; ++k) {
                run += s_cnt[warp][k];
                s_cnt[warp][k] = run;      // exclusive prefix: s_cnt[k] = ids of ranges < k
                s_cur[warp][k] = run;
            }
        }
        __syncwarp();
        for (int k = lane; k <= n_ranges; k += 32) seg_off[(size_t)r * (n_ranges + 1) + k] = s_cnt[warp][k];
        if (len > 1) {
            int* t = tmp + first;
            for (int i = lane; i < len; i += 32) {
                const int id = row[i];
                t[atomicAdd(&s_cur[warp][id / range_bits], 1)] = id;
            }
            __syncwarp();
            for (int i = lane; i < len; i += 32) row[i] = t[i];
        }
        __syncwarp();
    }
}
}  // namespace

int build_range_segments(blp_graph* g, int* tmp, cudaStream_t st) {
    for (int side = 0; side < 2; ++side) {
        const int R = g->n_ranges[side];
        if (R <= 1) continue;
        if (R > kMaxRanges) {
            set_error("graph needs more id ranges than this build supports");
            return BLP_ERR_UNSUPPORTED;
        }
        const bool us = side == BLP_SIDE_USER;
        const int n_mid = us ? g->n_biz : g->n_users;
        int* adj = us ? g->b_adj : g->u_adj;
        const unsigned long long* rows = (const unsigned long long*)(us ? g->b_row : g->u_row);
        const size_t cells = (size_t)n_mid * (size_t)(R + 1);
        BLP_CUDA_TRY(cudaMalloc((void**)&g->seg_off[side], sizeof(int) * cells));
        g->device_bytes += (int64_t)(sizeof(int) * cells);
        int* counter = nullptr;
        BLP_CUDA_TRY(cudaMalloc((void**)&counter, sizeof(int)));
        BLP_CUDA_TRY(cudaMemsetAsync(counter, 0, sizeof(int), st));
        k_range_segments<<<g->sm_count * 4, 256, 0, st>>>(rows, n_mid, adj, tmp, g->range_words[side] * 32,
                                                          R, g->seg_off[side], counter);
        cudaError_t e = cudaGetLastError();
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        cudaFree(counter);
        if (e != cudaSuccess) return cuda_fail(e, "k_range_segments", __FILE__, __LINE__);
    }
    return BLP_OK;
}

}  // namespace blp

extern "C" int blp_edge_list_count(const char* text_dev, int64_t n_bytes, int64_t* n_lines_host, void* stream) {
    using namespace blp;
    if (!n_lines_host || n_bytes < 0 || (n_bytes > 0 && !text_dev)) {
        set_error("blp_edge_list_count: bad argument");
        return BLP_ERR_INVALID;
    }
    *n_lines_host = 0;
    if (n_bytes == 0) return BLP_OK;
    cudaStream_t st = (cudaStream_t)stream;
    unsigned* tile_cnt = nullptr;
    int n_tiles = 0;
    int rc = parse_tile_counts(text_dev, n_bytes, st, &tile_cnt, &n_tiles);
    if (rc != BLP_OK) return rc;
    Scanner scan;
    scan.st = st;
    unsigned long long* base = nullptr;
    unsigned long long total = 0;
    cudaError_t e = scratch_alloc((void**)&base, sizeof(unsigned long long) * (size_t)n_tiles, st);
    if (e == cudaSuccess) rc = scan.run(tile_cnt, n_tiles, false, base, &total);
    scan.release();
    cudaFreeAsync(tile_cnt, st);
    if (base) cudaFreeAsync(base, st);
    if (e != cudaSuccess) return cuda_fail(e, "scratch_alloc", __FILE__, __LINE__);
    if (rc != BLP_OK) return rc;
    *n_lines_host = (int64_t)total;
    return BLP_OK;
}

extern "C" int blp_edge_list_parse(const char* text_dev, int64_t n_bytes, int64_t n_lines, int64_t* col0_dev,
                                   int64_t* col1_dev, void* stream) {
    using namespace blp;
    if (n_bytes < 0 || n_lines < 0 || (n_bytes > 0 && !text_dev) || (n_lines > 0 && (!col0_dev || !col1_dev))) {
        set_error("blp_edge_list_parse: bad argument");
        return BLP_ERR_INVALID;
    }
    if (n_bytes == 0 || n_lines == 0) return BLP_OK;
    cudaStream_t st = (cudaStream_t)stream;
    unsigned* tile_cnt = nullptr;
    int n_tiles = 0;
    int rc = parse_tile_counts(text_dev, n_bytes, st, &tile_cnt, &n_tiles);
    if (rc != BLP_OK) return rc;
    Scanner scan;
    scan.st = st;
    unsigned long long *base = nullptr, *bad = nullptr;
    unsigned long long total = 0, bad_host = ~0ull;
    cudaError_t e = scratch_alloc((void**)&base, sizeof(unsigned long long) * (size_t)n_tiles, st);
    if (e == cudaSuccess) e = scratch_alloc((void**)&bad, sizeof(unsigned long long), st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(bad, &bad_host, sizeof(bad_host), cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) rc = scan.run(tile_cnt, n_tiles, false, base, &total);
    if (e == cudaSuccess && rc == BLP_OK && (int64_t)total == n_lines) {
        k_parse_lines<<<(unsigned)n_tiles, 256, 0, st>>>(text_dev, n_bytes, base, n_lines, (long long*)col0_dev,
                                                        (long long*)col1_dev, bad);
        e = cudaGetLastError();
        if (e == cudaSuccess) e = cudaMemcpyAsync(&bad_host, bad, sizeof(bad_host), cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    }
    scan.release();
    cudaFreeAsync(tile_cnt, st);
    if (base) cudaFreeAsync(base, st);
    if (bad) cudaFreeAsync(bad, st);
    if (e != cudaSuccess) return cuda_fail(e, "blp_edge_list_parse", __FILE__, __LINE__);
    if (rc != BLP_OK) return rc;
    if ((int64_t)total != n_lines) {
        set_error("blp_edge_list_parse: n_lines does not match blp_edge_list_count of this text");
        return BLP_ERR_INVALID;
    }
    if (bad_host != ~0ull) {
        char buf[128];
        snprintf(buf, sizeof(buf), "blp_edge_list_parse: data line %llu has fewer than two integer columns", bad_host);
        set_error(buf);
        return BLP_ERR_INVALID;
    }
    return BLP_OK;
}

namespace blp {
namespace {
// The argument checks of both create functions, in this order and before any CUDA call but the
// device count.
int check_create_args(const char* api, int32_t n_users, int32_t n_biz, int64_t n_edges,
                      const int32_t* edge_u, const int32_t* edge_b, int device, blp_graph** out) {
    if (!out) {
        set_error(std::string(api) + ": out is null");
        return BLP_ERR_INVALID;
    }
    *out = nullptr;
    if (n_users <= 0 || n_biz <= 0 || n_edges < 0 || (n_edges > 0 && (!edge_u || !edge_b))) {
        set_error(std::string(api) + ": need n_users>0, n_biz>0, n_edges>=0 and edge arrays");
        return BLP_ERR_INVALID;
    }
    int ndev = 0;
    int rc = blp_device_count(&ndev);
    if (rc != BLP_OK) return rc;
    if (device < 0 || device >= ndev) {
        set_error(std::string(api) + ": device index out of range");
        return BLP_ERR_INVALID;
    }
    return BLP_OK;
}

// The graph builder behind both create functions: edge arrays in device memory, run on `st` of
// the current device.  `api` names the entry point in error messages.
int build_graph(const char* api, int32_t n_users, int32_t n_biz, int64_t n_edges,
                const int32_t* edge_u_dev, const int32_t* edge_b_dev, int device, cudaStream_t st,
                blp_graph** out) {
    const long long n = n_edges;
    int sm_query = 0;
    if (cudaDeviceGetAttribute(&sm_query, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || sm_query <= 0)
        sm_query = 132;
    const int grid = sm_query * 8;

    blp_graph* g = new (std::nothrow) blp_graph();
    if (!g) {
        set_error(std::string(api) + ": host allocation failed");
        return BLP_ERR_OOM;
    }
    g->n_users = n_users;
    g->n_biz = n_biz;
    g->n_edges_in = n_edges;
    std::vector<void*> scratch;
    auto alloc = [&](void** p, size_t bytes) -> cudaError_t {
        cudaError_t e = scratch_alloc(p, bytes ? bytes : 16, st);
        if (e == cudaSuccess) scratch.push_back(*p);
        return e;
    };
    Scanner scan;
    scan.st = st;
    auto fail = [&](int code) {
        for (void* p : scratch) cudaFreeAsync(p, st);
        scan.release();
        std::string keep = blp_last_error();
        blp_graph_destroy(g);
        set_error(keep);
        return code;
    };
#define BLP_TRY_B(expr)                                                                   \
    do {                                                                                  \
        cudaError_t e__ = (expr);                                                         \
        if (e__ != cudaSuccess) return fail(cuda_fail(e__, #expr, __FILE__, __LINE__));   \
    } while (0)
#define BLP_RC_B(expr)                   \
    do {                                 \
        int rc__ = (expr);               \
        if (rc__ != BLP_OK) return fail(rc__); \
    } while (0)

    BLP_RC_B(init_device_state(g, device, read_tuning()));

    // ---- keys, validity
    unsigned long long *keys = nullptr, *keys2 = nullptr, *pos = nullptr, *edges = nullptr;
    unsigned* flag = nullptr;
    int* bad = nullptr;
    BLP_TRY_B(alloc((void**)&keys, sizeof(unsigned long long) * (size_t)n));
    BLP_TRY_B(alloc((void**)&keys2, sizeof(unsigned long long) * (size_t)n));
    BLP_TRY_B(alloc((void**)&bad, sizeof(int)));
    const int big = INT_MAX;
    BLP_TRY_B(cudaMemcpyAsync(bad, &big, sizeof(int), cudaMemcpyHostToDevice, st));
    if (n) k_make_keys<<<grid, 256, 0, st>>>(edge_u_dev, edge_b_dev, n, n_users, n_biz, keys, bad);
    int bad_host = INT_MAX;
    BLP_TRY_B(cudaMemcpyAsync(&bad_host, bad, sizeof(int), cudaMemcpyDeviceToHost, st));
    BLP_TRY_B(cudaStreamSynchronize(st));
    if (bad_host != INT_MAX) {
        char buf[160];
        snprintf(buf, sizeof(buf), "%s: edge %d outside [0,%d) x [0,%d)", api, bad_host, n_users,
                 n_biz);
        set_error(buf);
        return fail(BLP_ERR_RANGE);
    }

    // ---- LSD radix sort over the bits in use: business bits, then user bits
    {
        std::vector<int> shifts;
        for (int s = 0; s < bits_for((unsigned)n_biz); s += 8) shifts.push_back(s);
        for (int s = 0; s < bits_for((unsigned)n_users); s += 8) shifts.push_back(32 + s);
        unsigned long long* sorted = keys;
        BLP_RC_B(radix_sort_u64(keys, keys2, n, shifts, st, &sorted));
        if (sorted != keys) std::swap(keys, keys2);
    }

    // ---- distinct edges, degrees
    unsigned long long m = 0;
    unsigned *u_deg = nullptr, *b_deg = nullptr;
    BLP_TRY_B(alloc((void**)&u_deg, sizeof(unsigned) * (size_t)n_users));
    BLP_TRY_B(alloc((void**)&b_deg, sizeof(unsigned) * (size_t)n_biz));
    BLP_TRY_B(cudaMemsetAsync(u_deg, 0, sizeof(unsigned) * (size_t)n_users, st));
    BLP_TRY_B(cudaMemsetAsync(b_deg, 0, sizeof(unsigned) * (size_t)n_biz, st));
    if (n) {
        BLP_TRY_B(alloc((void**)&flag, sizeof(unsigned) * (size_t)n));
        BLP_TRY_B(alloc((void**)&pos, sizeof(unsigned long long) * (size_t)n));
        k_unique_flags<<<grid, 256, 0, st>>>(keys, n, flag);
        BLP_RC_B(scan.run(flag, n, false, pos, &m));
        BLP_TRY_B(alloc((void**)&edges, sizeof(unsigned long long) * (size_t)m));
        k_compact_edges<<<grid, 256, 0, st>>>(keys, flag, pos, n, edges, u_deg, b_deg);
        BLP_TRY_B(cudaGetLastError());
    }
    g->n_edges = (int64_t)m;

    // ---- offsets: first index in the sorted order (users), padded row offsets (both)
    unsigned long long *u_first = nullptr, *u_off = nullptr, *b_off = nullptr;
    unsigned long long u_len = 0, b_len = 0;
    BLP_TRY_B(alloc((void**)&u_first, sizeof(unsigned long long) * (size_t)n_users));
    BLP_TRY_B(alloc((void**)&u_off, sizeof(unsigned long long) * (size_t)n_users));
    BLP_TRY_B(alloc((void**)&b_off, sizeof(unsigned long long) * (size_t)n_biz));
    BLP_RC_B(scan.run(u_deg, n_users, false, u_first, nullptr));
    BLP_RC_B(scan.run(u_deg, n_users, true, u_off, &u_len));
    BLP_RC_B(scan.run(b_deg, n_biz, true, b_off, &b_len));

    // ---- degrees to the host: limits, weight table, hub selection
    std::vector<int> hu((size_t)n_users), hb((size_t)n_biz);
    BLP_TRY_B(cudaMemcpyAsync(hu.data(), u_deg, sizeof(int) * (size_t)n_users, cudaMemcpyDeviceToHost, st));
    BLP_TRY_B(cudaMemcpyAsync(hb.data(), b_deg, sizeof(int) * (size_t)n_biz, cudaMemcpyDeviceToHost, st));
    BLP_TRY_B(cudaStreamSynchronize(st));
    for (int d : hu) {
        g->n_users_in += d > 0;
        g->max_udeg = std::max(g->max_udeg, d);
    }
    for (int d : hb) {
        g->n_biz_in += d > 0;
        g->max_bdeg = std::max(g->max_bdeg, d);
    }
    if (u_len / 4 >= (1ull << BLP_ROW_FIRST4_BITS) || b_len / 4 >= (1ull << BLP_ROW_FIRST4_BITS) ||
        g->max_udeg >= (1 << 24) ||
        g->max_bdeg >= (1 << 24)) {
        set_error(std::string(api) + ": graph too large for the packed row descriptors");
        return fail(BLP_ERR_UNSUPPORTED);
    }

    // ---- persistent arrays of the handle
    auto keep = [&](void** p, size_t bytes) -> cudaError_t {
        cudaError_t e = cudaMalloc(p, bytes ? bytes : 16);
        if (e == cudaSuccess) g->device_bytes += (int64_t)bytes;
        return e;
    };
    int* tmp = nullptr;
    g->u_adj_len = (int64_t)u_len;
    g->b_adj_len = (int64_t)b_len;
    BLP_TRY_B(keep((void**)&g->u_adj, sizeof(int) * (size_t)u_len));
    BLP_TRY_B(keep((void**)&g->b_adj, sizeof(int) * (size_t)b_len));
    BLP_TRY_B(keep((void**)&g->u_adjw, sizeof(unsigned) * (size_t)u_len));
    BLP_TRY_B(keep((void**)&g->b_adjw, sizeof(unsigned) * (size_t)b_len));
    BLP_TRY_B(keep((void**)&g->u_row, sizeof(unsigned long long) * (size_t)n_users));
    BLP_TRY_B(keep((void**)&g->b_row, sizeof(unsigned long long) * (size_t)n_biz));
    BLP_TRY_B(keep((void**)&g->u_deg, sizeof(int) * (size_t)n_users));
    BLP_TRY_B(keep((void**)&g->b_deg, sizeof(int) * (size_t)n_biz));
    BLP_TRY_B(alloc((void**)&tmp, sizeof(int) * (size_t)std::max(u_len, b_len)));
    k_fill<<<grid, 256, 0, st>>>(g->u_adj, (long long)u_len, n_biz);     // padding sentinels
    k_fill<<<grid, 256, 0, st>>>(g->b_adj, (long long)b_len, n_users);
    unsigned* b_cur = nullptr;
    int* next_row = nullptr;
    BLP_TRY_B(alloc((void**)&b_cur, sizeof(unsigned) * (size_t)n_biz));
    BLP_TRY_B(alloc((void**)&next_row, sizeof(int) * 2));
    BLP_TRY_B(cudaMemsetAsync(b_cur, 0, sizeof(unsigned) * (size_t)n_biz, st));
    BLP_TRY_B(cudaMemsetAsync(next_row, 0, sizeof(int) * 2, st));
    if (m)
        k_place_edges<<<grid, 256, 0, st>>>(edges, (long long)m, u_first, u_off, b_off, b_cur,
                                            g->u_adj, g->b_adj);
    k_row_descriptors<<<(n_users + 255) / 256, 256, 0, st>>>(u_off, u_deg, n_users,
                                                             (unsigned long long*)g->u_row, g->u_deg);
    k_row_descriptors<<<(n_biz + 255) / 256, 256, 0, st>>>(b_off, b_deg, n_biz,
                                                           (unsigned long long*)g->b_row, g->b_deg);
    // a side that needs id-range passes gets its middle rows partitioned by range instead of
    // bank-striped: business rows serve the user side, user rows the business side
    if (g->n_ranges[1] == 1)
        k_bank_stripe<<<g->sm_count * 4, 256, 0, st>>>(u_off, u_deg, n_users, g->u_adj, tmp, next_row);
    if (g->n_ranges[0] == 1)
        k_bank_stripe<<<g->sm_count * 4, 256, 0, st>>>(b_off, b_deg, n_biz, g->b_adj, tmp, next_row + 1);
    BLP_TRY_B(cudaGetLastError());
    BLP_RC_B(build_range_segments(g, tmp, st));

    // ---- per-entry weights from a host-evaluated 1/ln(d) table
    {
        std::vector<unsigned> lut;
        weight_lut(std::max(g->max_udeg, g->max_bdeg), lut);
        unsigned* d_lut = nullptr;
        BLP_TRY_B(alloc((void**)&d_lut, sizeof(unsigned) * lut.size()));
        BLP_TRY_B(cudaMemcpyAsync(d_lut, lut.data(), sizeof(unsigned) * lut.size(),
                                  cudaMemcpyHostToDevice, st));
        // user rows name businesses, business rows name users
        k_entry_weights<<<grid, 256, 0, st>>>(g->u_adj, (long long)u_len, n_biz, b_deg, d_lut, g->u_adjw);
        k_entry_weights<<<grid, 256, 0, st>>>(g->b_adj, (long long)b_len, n_users, u_deg, d_lut, g->b_adjw);
        BLP_TRY_B(cudaGetLastError());
        BLP_TRY_B(cudaStreamSynchronize(st));   // lut (host vector) and scratch are done with
    }
    for (void* p : scratch) cudaFreeAsync(p, st);
    scratch.clear();
    scan.release();
    BLP_TRY_B(cudaStreamSynchronize(st));
    const int rc = build_hub_bitmaps(g, hu.data(), hb.data());
    if (rc != BLP_OK) return fail(rc);
#undef BLP_TRY_B
#undef BLP_RC_B
    *out = g;
    return BLP_OK;
}
}  // namespace
}  // namespace blp

extern "C" int blp_graph_create_device(int32_t n_users, int32_t n_biz, int64_t n_edges,
                                       const int32_t* edge_u_dev, const int32_t* edge_b_dev,
                                       int device, void* stream, blp_graph** out) {
    const char* api = "blp_graph_create_device";
    int rc = blp::check_create_args(api, n_users, n_biz, n_edges, edge_u_dev, edge_b_dev, device, out);
    if (rc != BLP_OK) return rc;
    BLP_ON_DEVICE(device);
    return blp::build_graph(api, n_users, n_biz, n_edges, edge_u_dev, edge_b_dev, device,
                            (cudaStream_t)stream, out);
}

extern "C" int blp_graph_create(int32_t n_users, int32_t n_biz, int64_t n_edges,
                                const int32_t* edge_u, const int32_t* edge_b, int device,
                                blp_graph** out) {
    const char* api = "blp_graph_create";
    int rc = blp::check_create_args(api, n_users, n_biz, n_edges, edge_u, edge_b, device, out);
    if (rc != BLP_OK) return rc;
    BLP_ON_DEVICE(device);
    // staged and built on the legacy default stream, so the build follows the caller's earlier work
    // on every blocking stream of the device
    const cudaStream_t st = cudaStreamLegacy;
    const size_t bytes = sizeof(int32_t) * (size_t)n_edges;
    int32_t *eu = nullptr, *eb = nullptr;
    cudaError_t e = cudaSuccess;
    if (n_edges > 0) {
        e = blp::scratch_alloc((void**)&eu, bytes, st);
        if (e == cudaSuccess) e = blp::scratch_alloc((void**)&eb, bytes, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(eu, edge_u, bytes, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(eb, edge_b, bytes, cudaMemcpyHostToDevice, st);
    }
    rc = e == cudaSuccess ? blp::build_graph(api, n_users, n_biz, n_edges, eu, eb, device, st, out)
                          : blp::cuda_fail(e, "staging the edge arrays", __FILE__, __LINE__);
    if (eu) cudaFreeAsync(eu, st);
    if (eb) cudaFreeAsync(eb, st);
    return rc;
}
