// The two JSON files of similarity.main on the device: examples.json in, score files out.
//
// Score-file writer (blp_json_scores_count / _fill): the bytes json.dumps writes for the nested
// dict similarity._emit builds, one warp per example user.  A user's text is
//     , "<u>": {"<b>": <v>, "<b>": <v>}
// (empty when none of its pairs is written); the document is "{" + the concatenation without its
// first two bytes + "}", or "{}".  The count call gives every user's byte length, the caller scans
// them and fills any range of users at its offsets, so a file of any size goes out in chunks cut
// at user boundaries.
//
// examples.json reader (blp_examples_count / _parse): the grammar json.dumps produces for
// {"<u>": {"<b>": int}} with any JSON whitespace between tokens, canonical decimal keys and int32
// values.  The text is uploaded as it is.  A first pass counts four bytes per 4 KB tile -- '"',
// '{', '}', ':' -- and the builder's scan turns them into counts before every tile; since keys
// hold only digits and '-', those give every byte's string parity and nesting depth.  A second
// pass lets the thread that owns a token's first byte check the token and the one after it: the
// grammar has depth 2, so (token kind, depth) is the state of a finite automaton and the whole
// document is valid exactly when every such transition is.  In a valid document the '{' and ':'
// counts before a key are its user and pair index.  Duplicate keys (json.load keeps the last
// value at the first position, which a columnar layout cannot express) are found by sorting a
// hash of (user, key) with the builder's radix sort and comparing the keys of every run of equal
// hashes exactly.  Anything outside the grammar is BLP_ERR_UNSUPPORTED with its byte offset.
#include <algorithm>
#include <cstdio>
#include <vector>

#include "blp_internal.h"

#define BLP_POW5_STORAGE static __device__
#include "blp_json_format.cuh"

namespace blp {
namespace {

constexpr unsigned kFullMask = 0xffffffffu;

// ------------------------------------------------------------------------------------ writer
struct ScoreCols {
    const int64_t* user_off;
    const int64_t* user_ids;
    const int64_t* biz_ids;
    const uint8_t* in_graph;
    const void* values;     // nullptr = only the out-of-graph zeros
    int kind;
};

__device__ __forceinline__ blp_json::Pow5Tables pow5_tables() {
    return blp_json::Pow5Tables{&blp_pow5_inv_split[0][0], &blp_pow5_split[0][0]};
}

// Text of pair i's value into buf; -1 when the pair is not written.
__device__ __forceinline__ int value_text(const ScoreCols& c, long long i, char* buf,
                                          const blp_json::Pow5Tables& t) {
    if (!c.in_graph[i]) {
        buf[0] = '0';   // similarity.py:59-60, 104-105: the literal int 0
        return 1;
    }
    if (!c.values) return -1;
    switch (c.kind) {
        case BLP_JSON_INT32: return blp_json::format_int64(((const int32_t*)c.values)[i], buf);
        case BLP_JSON_INT64: return blp_json::format_int64(((const long long*)c.values)[i], buf);
        case BLP_JSON_FLOAT64: return blp_json::format_double(((const double*)c.values)[i], buf, t);
        default: {   // BLP_JSON_FLOAT64_INT_ZERO
            const double v = ((const double*)c.values)[i];
            if (v == 0.0) {
                buf[0] = '0';
                return 1;
            }
            return blp_json::format_double(v, buf, t);
        }
    }
}

__global__ void __launch_bounds__(256) k_scores_count(ScoreCols c, long long n_users, int64_t* __restrict__ len) {
    const blp_json::Pow5Tables t = pow5_tables();
    const int lane = threadIdx.x & 31;
    const long long warps = (long long)gridDim.x * 8;
    for (long long u = blockIdx.x * 8LL + (threadIdx.x >> 5); u < n_users; u += warps) {
        const long long lo = c.user_off[u], hi = c.user_off[u + 1];
        long long bytes = 0, written = 0;
        for (long long i = lo + lane; i < hi; i += 32) {
            char buf[blp_json::kMaxDoubleChars];
            const int lv = value_text(c, i, buf, t);
            if (lv >= 0) {
                bytes += blp_json::format_int64(c.biz_ids[i], buf) + lv + 4;   // "<b>": <v>
                ++written;
            }
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            bytes += __shfl_xor_sync(kFullMask, bytes, d);
            written += __shfl_xor_sync(kFullMask, written, d);
        }
        if (lane == 0) {
            char ubuf[blp_json::kMaxIntChars];
            // , "<u>": {  entries joined by ", "  }
            len[u] = written ? blp_json::format_int64(c.user_ids[u], ubuf) + 7 + bytes + 2 * (written - 1) + 1 : 0;
        }
    }
}

__global__ void __launch_bounds__(256) k_scores_fill(ScoreCols c, const int64_t* __restrict__ text_off,
                                                     long long begin, long long end, char* __restrict__ out) {
    const blp_json::Pow5Tables t = pow5_tables();
    const int lane = threadIdx.x & 31;
    const long long warps = (long long)gridDim.x * 8;
    const long long base0 = text_off[begin];
    for (long long u = begin + blockIdx.x * 8LL + (threadIdx.x >> 5); u < end; u += warps) {
        char* base = out + (text_off[u] - base0);
        char ubuf[blp_json::kMaxIntChars];
        const int lu = blp_json::format_int64(c.user_ids[u], ubuf);
        char* body = base + lu + 7;
        const long long lo = c.user_off[u], hi = c.user_off[u + 1];
        long long cur = 0;
        bool any = false;
        for (long long b0 = lo; b0 < hi; b0 += 32) {
            const long long i = b0 + lane;
            char vbuf[blp_json::kMaxDoubleChars], kbuf[blp_json::kMaxIntChars];
            const int lv = i < hi ? value_text(c, i, vbuf, t) : -1;
            const unsigned ballot = __ballot_sync(kFullMask, lv >= 0);
            int lk = 0, sz = 0;
            bool sep = false;
            if (lv >= 0) {
                lk = blp_json::format_int64(c.biz_ids[i], kbuf);
                sep = any || lane != __ffs(ballot) - 1;   // ", " before all but the user's first entry
                sz = (sep ? 2 : 0) + lk + lv + 4;
            }
            int inc = sz;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const int v = __shfl_up_sync(kFullMask, inc, d);
                if (lane >= d) inc += v;
            }
            if (lv >= 0) {
                char* p = body + cur + (inc - sz);
                if (sep) {
                    *p++ = ',';
                    *p++ = ' ';
                }
                *p++ = '"';
                for (int k = 0; k < lk; ++k) *p++ = kbuf[k];
                *p++ = '"';
                *p++ = ':';
                *p++ = ' ';
                for (int k = 0; k < lv; ++k) *p++ = vbuf[k];
            }
            cur += __shfl_sync(kFullMask, inc, 31);
            any = any || ballot != 0u;
        }
        if (any && lane == 0) {
            char* p = base;
            *p++ = ',';
            *p++ = ' ';
            *p++ = '"';
            for (int k = 0; k < lu; ++k) *p++ = ubuf[k];
            *p++ = '"';
            *p++ = ':';
            *p++ = ' ';
            *p++ = '{';
            body[cur] = '}';
        }
    }
}

int check_score_args(const char* api, const int64_t* user_off, const int64_t* user_ids, int64_t n_users,
                     const int64_t* biz_ids, const uint8_t* in_graph, const void* values, int kind) {
    if (n_users < 0 || (n_users > 0 && (!user_off || !user_ids || !biz_ids || !in_graph)) ||
        (values && (kind < BLP_JSON_INT32 || kind > BLP_JSON_FLOAT64_INT_ZERO))) {
        set_error(std::string(api) + ": bad argument");
        return BLP_ERR_INVALID;
    }
    return BLP_OK;
}

unsigned warp_grid(long long n_items) {
    return (unsigned)std::min<long long>((n_items + 7) / 8, 1LL << 16);
}

// ------------------------------------------------------------------------------------ reader
constexpr int kTile = 4096;   // bytes per CTA: 256 threads x 16

enum Tok { T_LB = 0, T_RB, T_COLON, T_COMMA, T_STR, T_NUM, T_END, T_BAD };

__device__ __forceinline__ bool is_ws(char c) { return c == ' ' || c == '\t' || c == '\n' || c == '\r'; }
__device__ __forceinline__ bool is_num(char c) { return c == '-' || (c >= '0' && c <= '9'); }
__device__ __forceinline__ int classify(char c) {
    switch (c) {
        case '{': return T_LB;
        case '}': return T_RB;
        case ':': return T_COLON;
        case ',': return T_COMMA;
        case '"': return T_STR;
        default: return is_num(c) ? T_NUM : T_BAD;
    }
}

// the four counted bytes as 16-bit fields of one word (a tile holds at most 4096 of each)
__device__ __forceinline__ unsigned long long byte_fields(char c) {
    switch (c) {
        case '"': return 1ull;
        case '{': return 1ull << 16;
        case '}': return 1ull << 32;
        case ':': return 1ull << 48;
        default: return 0ull;
    }
}

__global__ void __launch_bounds__(256) k_ex_count(const char* __restrict__ t, long long n,
                                                  unsigned* __restrict__ cnt, int n_tiles) {
    __shared__ unsigned long long s_w[8];
    const long long lo = (long long)blockIdx.x * kTile + threadIdx.x * 16;
    unsigned long long f = 0;
#pragma unroll
    for (int j = 0; j < 16; ++j)
        if (lo + j < n) f += byte_fields(t[lo + j]);
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) f += __shfl_xor_sync(kFullMask, f, d);
    if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = f;
    __syncthreads();
    if (threadIdx.x < 4) {
        unsigned long long tot = 0;
        for (int w = 0; w < 8; ++w) tot += s_w[w];
        cnt[(size_t)threadIdx.x * n_tiles + blockIdx.x] = (unsigned)((tot >> (16 * threadIdx.x)) & 0xffffull);
    }
}

struct ExOut {
    bool write;             // false: validate only (blp_examples_count)
    long long n_users, n_pairs;
    int64_t* user_off;      // [n_users]; the last entry is set by the host
    int64_t* user_ids;
    int64_t* biz_ids;
    int32_t* labels;
    long long* user_pos;    // byte offset of every key (duplicate reports)
    long long* pair_pos;
    long long* pair_user;   // user index of every pair
};

// A key: "0" or -?[1-9][0-9]{0,17} between quotes starting at p; *end = one past the closing quote.
__device__ __forceinline__ bool parse_key(const char* __restrict__ t, long long n, long long p, long long* end,
                                          long long* key) {
    long long j = p + 1;
    const bool neg = j < n && t[j] == '-';
    if (neg) ++j;
    if (j >= n || t[j] < '0' || t[j] > '9') return false;
    long long v = 0;
    if (t[j] == '0') {
        if (neg) return false;   // "-0" is not the decimal text of an int64
        ++j;
    } else {
        int digits = 0;
        while (j < n && t[j] >= '0' && t[j] <= '9') {
            if (++digits > 18) return false;
            v = v * 10 + (t[j] - '0');
            ++j;
        }
    }
    if (j >= n || t[j] != '"') return false;
    *end = j + 1;
    *key = neg ? -v : v;
    return true;
}

// A JSON integer -?(0|[1-9][0-9]*) that fits int32, not followed by another number byte.
__device__ __forceinline__ bool parse_label(const char* __restrict__ t, long long n, long long p, long long* end,
                                            int* out) {
    long long j = p;
    const bool neg = t[j] == '-';
    if (neg) ++j;
    if (j >= n || t[j] < '0' || t[j] > '9') return false;
    long long v = 0;
    if (t[j] == '0') {
        ++j;
    } else {
        int digits = 0;
        while (j < n && t[j] >= '0' && t[j] <= '9') {
            if (++digits > 10) return false;
            v = v * 10 + (t[j] - '0');
            ++j;
        }
    }
    if (j < n && is_num(t[j])) return false;
    if (neg) v = -v;
    if (v < -2147483648LL || v > 2147483647LL) return false;
    *end = j;
    *out = (int)v;
    return true;
}

// Allowed successors of token `k` at nesting depth `d` (depth before the token), as a bit set of
// Tok values.  The grammar: { ( "u" : { ( "b" : int (, "b" : int)* )? } (, "u" : {...})* )? }
__device__ __forceinline__ unsigned successors(int k, long long d) {
    const unsigned LB = 1u << T_LB, RB = 1u << T_RB, CO = 1u << T_COLON, CM = 1u << T_COMMA,
                   ST = 1u << T_STR, NU = 1u << T_NUM, EN = 1u << T_END;
    if (d == 0) return k == T_LB ? (ST | RB) : 0u;
    if (d == 1) {
        switch (k) {
            case T_STR: return CO;        // user key
            case T_COLON: return LB;
            case T_LB: return ST | RB;    // a user's object
            case T_COMMA: return ST;
            case T_RB: return EN;         // end of the document
            default: return 0u;
        }
    }
    if (d == 2) {
        switch (k) {
            case T_STR: return CO;        // business key
            case T_COLON: return NU;
            case T_NUM: return CM | RB;
            case T_COMMA: return ST;
            case T_RB: return CM | RB;    // end of a user's object
            default: return 0u;
        }
    }
    return 0u;
}

__global__ void __launch_bounds__(256) k_ex_tokens(const char* __restrict__ t, long long n,
                                                   const unsigned long long* __restrict__ base, int n_tiles,
                                                   ExOut o, unsigned long long* __restrict__ err) {
    __shared__ unsigned long long s_w[8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long lo = (long long)blockIdx.x * kTile + threadIdx.x * 16;
    char b[16];
    unsigned long long f = 0;
#pragma unroll
    for (int j = 0; j < 16; ++j) {
        b[j] = lo + j < n ? t[lo + j] : ' ';
        f += byte_fields(b[j]);
    }
    unsigned long long inc = f;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const unsigned long long v = __shfl_up_sync(kFullMask, inc, d);
        if (lane >= d) inc += v;
    }
    if (lane == 31) s_w[warp] = inc;
    __syncthreads();
    unsigned long long before = inc - f;
    for (int w = 0; w < warp; ++w) before += s_w[w];
    long long q = (long long)base[blockIdx.x] + (long long)(before & 0xffffull);
    long long lb = (long long)base[(size_t)n_tiles + blockIdx.x] + (long long)((before >> 16) & 0xffffull);
    long long rb = (long long)base[(size_t)2 * n_tiles + blockIdx.x] + (long long)((before >> 32) & 0xffffull);
    long long col = (long long)base[(size_t)3 * n_tiles + blockIdx.x] + (long long)(before >> 48);
    for (int j = 0; j < 16 && lo + j < n; ++j) {
        const long long p = lo + j;
        const char c = b[j];
        const bool in_string = q & 1;   // inside a key, or at its closing quote
        if (!in_string && !is_ws(c) && !(is_num(c) && p > 0 && is_num(t[p - 1]))) {
            const int k = classify(c);
            const long long depth = lb - rb;
            long long end = p + 1, key = 0;
            int label = 0;
            bool ok = k != T_BAD;
            if (k == T_STR) ok = parse_key(t, n, p, &end, &key);
            else if (k == T_NUM) ok = parse_label(t, n, p, &end, &label);
            if (ok) {
                while (end < n && is_ws(t[end])) ++end;
                const int next = end < n ? classify(t[end]) : T_END;
                ok = (successors(k, depth) >> next) & 1u;
            }
            if (ok && k == T_STR && depth == 1) {
                const long long u = lb - 1;
                ok = u >= 0 && u < o.n_users;
                if (ok && o.write) {
                    o.user_ids[u] = key;
                    o.user_off[u] = col - lb + 1;
                    o.user_pos[u] = p;
                }
            } else if (ok && k == T_STR) {
                const long long i = col - lb + 1;
                ok = i >= 0 && i < o.n_pairs;
                if (ok && o.write) {
                    o.biz_ids[i] = key;
                    o.pair_pos[i] = p;
                    o.pair_user[i] = lb - 2;
                }
            } else if (ok && k == T_NUM) {
                const long long i = col - lb;
                ok = i >= 0 && i < o.n_pairs;
                if (ok && o.write && o.labels) o.labels[i] = label;
            }
            if (!ok) atomicMin(err, (unsigned long long)p);
        }
        q += c == '"';
        lb += c == '{';
        rb += c == '}';
        col += c == ':';
    }
}

__device__ __forceinline__ unsigned long long mix64(unsigned long long x) {   // splitmix64 finaliser
    x ^= x >> 30;
    x *= 0xbf58476d1ce4e5b9ull;
    x ^= x >> 27;
    x *= 0x94d049bb133111ebull;
    return x ^ (x >> 31);
}

// key of item i: a hash of (group, id) above the low `idx_bits` bits, which hold i
__global__ void k_dup_keys(const long long* __restrict__ group, const int64_t* __restrict__ id, long long n,
                           int idx_bits, unsigned long long* __restrict__ keys) {
    const unsigned long long low = (1ull << idx_bits) - 1ull;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const unsigned long long h = mix64((unsigned long long)id[i] + mix64(group ? (unsigned long long)group[i] + 1ull : 0ull));
        keys[i] = (h & ~low) | (unsigned long long)i;
    }
}

// Every run of equal hashes is compared exactly, all pairs (runs longer than one are rare); a true
// duplicate reports the byte offset of its later occurrence.
__global__ void k_dup_runs(const unsigned long long* __restrict__ keys, long long n, int idx_bits,
                           const long long* __restrict__ group, const int64_t* __restrict__ id,
                           const long long* __restrict__ pos, unsigned long long* __restrict__ err) {
    const unsigned long long low = (1ull << idx_bits) - 1ull;
    for (long long s = blockIdx.x * (long long)blockDim.x + threadIdx.x; s < n; s += (long long)gridDim.x * blockDim.x) {
        const unsigned long long h = keys[s] & ~low;
        if (s > 0 && (keys[s - 1] & ~low) == h) continue;    // not the start of a run
        long long e = s + 1;
        while (e < n && (keys[e] & ~low) == h) ++e;
        for (long long a = s; a < e; ++a) {
            const long long ia = (long long)(keys[a] & low);
            for (long long c = a + 1; c < e; ++c) {
                const long long ic = (long long)(keys[c] & low);
                if (id[ia] == id[ic] && (!group || group[ia] == group[ic]))
                    atomicMin(err, (unsigned long long)max(pos[ia], pos[ic]));
            }
        }
    }
}

int find_duplicates(const long long* group, const int64_t* id, const long long* pos, long long n,
                    unsigned long long* err, cudaStream_t st) {
    if (n <= 1) return BLP_OK;
    int idx_bits = 1;
    while ((1LL << idx_bits) < n) ++idx_bits;
    unsigned long long *keys = nullptr, *tmp = nullptr, *sorted = nullptr;
    BLP_CUDA_TRY(scratch_alloc((void**)&keys, sizeof(unsigned long long) * (size_t)n, st));
    cudaError_t e = scratch_alloc((void**)&tmp, sizeof(unsigned long long) * (size_t)n, st);
    int rc = BLP_OK;
    if (e == cudaSuccess) {
        const unsigned grid = (unsigned)std::min<long long>((n + 255) / 256, 1LL << 16);
        k_dup_keys<<<grid, 256, 0, st>>>(group, id, n, idx_bits, keys);
        std::vector<int> shifts;
        for (int s = idx_bits; s < 64; s += 8) shifts.push_back(s);
        rc = radix_sort_u64(keys, tmp, n, shifts, st, &sorted);
        if (rc == BLP_OK) k_dup_runs<<<grid, 256, 0, st>>>(sorted, n, idx_bits, group, id, pos, err);
        e = cudaGetLastError();
    }
    cudaFreeAsync(keys, st);
    if (tmp) cudaFreeAsync(tmp, st);
    if (e != cudaSuccess) return cuda_fail(e, "find_duplicates", __FILE__, __LINE__);
    return rc;
}

// Both reader calls: counts, the validating pass (writes when o carries outputs), and with
// outputs the duplicate checks.  *totals = {n_users, n_pairs} of the text.
int examples_run(const char* api, const char* text, long long n, ExOut o, long long totals[2], cudaStream_t st) {
    if (n == 0) {
        set_error(std::string(api) + ": empty text is not a JSON document");
        return BLP_ERR_UNSUPPORTED;
    }
    const long long n_tiles = (n + kTile - 1) / kTile;
    if (n_tiles >= (1LL << 31)) {
        set_error(std::string(api) + ": text too large (more than 8 TB)");
        return BLP_ERR_UNSUPPORTED;
    }
    unsigned* cnt = nullptr;
    unsigned long long *base = nullptr, *err = nullptr;
    unsigned long long err_host = ~0ull, tot[4] = {0, 0, 0, 0};
    int rc = BLP_OK;
    cudaError_t e = scratch_alloc((void**)&cnt, sizeof(unsigned) * 4 * (size_t)n_tiles, st);
    if (e == cudaSuccess) e = scratch_alloc((void**)&base, sizeof(unsigned long long) * 4 * (size_t)n_tiles, st);
    if (e == cudaSuccess) e = scratch_alloc((void**)&err, sizeof(unsigned long long), st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(err, &err_host, sizeof(err_host), cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) {
        k_ex_count<<<(unsigned)n_tiles, 256, 0, st>>>(text, n, cnt, (int)n_tiles);
        for (int f = 0; f < 4 && rc == BLP_OK; ++f)
            rc = exclusive_scan_u32(cnt + (size_t)f * n_tiles, n_tiles, base + (size_t)f * n_tiles, &tot[f], st);
    }
    // a valid document has one '{' per user plus the outer one and one ':' per user and per pair
    const long long n_users = (long long)tot[1] - 1, n_pairs = (long long)tot[3] - n_users;
    if (e == cudaSuccess && rc == BLP_OK && o.write && (n_users != o.n_users || n_pairs != o.n_pairs)) {
        set_error(std::string(api) + ": n_users / n_pairs do not match blp_examples_count of this text");
        rc = BLP_ERR_INVALID;
    }
    if (e == cudaSuccess && rc == BLP_OK) {
        if (!o.write) {
            o.n_users = n_users;
            o.n_pairs = n_pairs;
        }
        k_ex_tokens<<<(unsigned)n_tiles, 256, 0, st>>>(text, n, base, (int)n_tiles, o, err);
        e = cudaGetLastError();
        if (e == cudaSuccess) e = cudaMemcpyAsync(&err_host, err, sizeof(err_host), cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        if (e == cudaSuccess && err_host == ~0ull && tot[1] == 0) err_host = 0;   // no token at all
        if (e == cudaSuccess && err_host == ~0ull && o.write) {
            rc = find_duplicates(nullptr, o.user_ids, o.user_pos, o.n_users, err, st);
            if (rc == BLP_OK) rc = find_duplicates(o.pair_user, o.biz_ids, o.pair_pos, o.n_pairs, err, st);
            if (rc == BLP_OK) e = cudaMemcpyAsync(&err_host, err, sizeof(err_host), cudaMemcpyDeviceToHost, st);
            if (rc == BLP_OK && e == cudaSuccess) e = cudaStreamSynchronize(st);
        }
    }
    if (cnt) cudaFreeAsync(cnt, st);
    if (base) cudaFreeAsync(base, st);
    if (err) cudaFreeAsync(err, st);
    if (e != cudaSuccess) return cuda_fail(e, api, __FILE__, __LINE__);
    if (rc != BLP_OK) return rc;
    if (err_host != ~0ull) {
        char buf[160];
        snprintf(buf, sizeof(buf), "%s: outside the device grammar of examples.json at byte %llu", api, err_host);
        set_error(buf);
        return BLP_ERR_UNSUPPORTED;
    }
    totals[0] = n_users;
    totals[1] = n_pairs;
    return BLP_OK;
}

}  // namespace
}  // namespace blp

extern "C" int blp_json_scores_count(const int64_t* user_off, const int64_t* user_ids, int64_t n_users,
                                     const int64_t* biz_ids, const uint8_t* in_graph, const void* values,
                                     int kind, int64_t* lengths, void* stream) {
    using namespace blp;
    int rc = check_score_args("blp_json_scores_count", user_off, user_ids, n_users, biz_ids, in_graph, values, kind);
    if (rc != BLP_OK) return rc;
    if (n_users > 0 && !lengths) {
        set_error("blp_json_scores_count: lengths is null");
        return BLP_ERR_INVALID;
    }
    if (n_users == 0) return BLP_OK;
    cudaStream_t st = (cudaStream_t)stream;
    k_scores_count<<<warp_grid(n_users), 256, 0, st>>>(ScoreCols{user_off, user_ids, biz_ids, in_graph, values, kind},
                                                       n_users, lengths);
    BLP_CUDA_TRY(cudaGetLastError());
    return BLP_OK;
}

extern "C" int blp_json_scores_fill(const int64_t* user_off, const int64_t* user_ids, int64_t n_users,
                                    const int64_t* biz_ids, const uint8_t* in_graph, const void* values,
                                    int kind, const int64_t* text_off, int64_t user_begin, int64_t user_end,
                                    char* out, void* stream) {
    using namespace blp;
    int rc = check_score_args("blp_json_scores_fill", user_off, user_ids, n_users, biz_ids, in_graph, values, kind);
    if (rc != BLP_OK) return rc;
    if (user_begin < 0 || user_end < user_begin || user_end > n_users ||
        (user_end > user_begin && (!text_off || !out))) {
        set_error("blp_json_scores_fill: bad user range or null output");
        return BLP_ERR_INVALID;
    }
    if (user_end == user_begin) return BLP_OK;
    cudaStream_t st = (cudaStream_t)stream;
    k_scores_fill<<<warp_grid(user_end - user_begin), 256, 0, st>>>(
        ScoreCols{user_off, user_ids, biz_ids, in_graph, values, kind}, text_off, user_begin, user_end, out);
    BLP_CUDA_TRY(cudaGetLastError());
    return BLP_OK;
}

extern "C" int blp_examples_count(const char* text_dev, int64_t n_bytes, int64_t* n_users_host,
                                  int64_t* n_pairs_host, void* stream) {
    using namespace blp;
    if (!n_users_host || !n_pairs_host || n_bytes < 0 || (n_bytes > 0 && !text_dev)) {
        set_error("blp_examples_count: bad argument");
        return BLP_ERR_INVALID;
    }
    *n_users_host = *n_pairs_host = 0;
    ExOut o = {};
    long long totals[2] = {0, 0};
    const int rc = examples_run("blp_examples_count", text_dev, n_bytes, o, totals, (cudaStream_t)stream);
    if (rc != BLP_OK) return rc;
    *n_users_host = totals[0];
    *n_pairs_host = totals[1];
    return BLP_OK;
}

extern "C" int blp_examples_parse(const char* text_dev, int64_t n_bytes, int64_t n_users, int64_t n_pairs,
                                  int64_t* user_off, int64_t* user_ids, int64_t* biz_ids, int32_t* labels,
                                  void* stream) {
    using namespace blp;
    if (n_bytes < 0 || n_users < 0 || n_pairs < 0 || (n_bytes > 0 && !text_dev) || !user_off ||
        (n_users > 0 && !user_ids) || (n_pairs > 0 && !biz_ids)) {
        set_error("blp_examples_parse: bad argument");
        return BLP_ERR_INVALID;
    }
    cudaStream_t st = (cudaStream_t)stream;
    ExOut o = {};
    o.write = true;
    o.n_users = n_users;
    o.n_pairs = n_pairs;
    o.user_off = user_off;
    o.user_ids = user_ids;
    o.biz_ids = biz_ids;
    o.labels = labels;
    cudaError_t e = scratch_alloc((void**)&o.user_pos, sizeof(long long) * (size_t)std::max<int64_t>(n_users, 1), st);
    if (e == cudaSuccess) e = scratch_alloc((void**)&o.pair_pos, sizeof(long long) * (size_t)std::max<int64_t>(n_pairs, 1), st);
    if (e == cudaSuccess) e = scratch_alloc((void**)&o.pair_user, sizeof(long long) * (size_t)std::max<int64_t>(n_pairs, 1), st);
    long long totals[2] = {0, 0};
    int rc = BLP_OK;
    if (e == cudaSuccess) rc = examples_run("blp_examples_parse", text_dev, n_bytes, o, totals, st);
    const long long last = n_pairs;
    if (e == cudaSuccess && rc == BLP_OK) e = cudaMemcpyAsync(user_off + n_users, &last, sizeof(last), cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess && rc == BLP_OK) e = cudaStreamSynchronize(st);
    if (o.user_pos) cudaFreeAsync(o.user_pos, st);
    if (o.pair_pos) cudaFreeAsync(o.pair_pos, st);
    if (o.pair_user) cudaFreeAsync(o.pair_user, st);
    if (e != cudaSuccess) return cuda_fail(e, "blp_examples_parse", __FILE__, __LINE__);
    return rc;
}
