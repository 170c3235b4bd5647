// blp_score_pairs_host: the whole end-to-end step behind ONE C-ABI call with HOST buffers.
//
// The reference's scorer takes host data in and leaves host data behind (similarity.py:14-18
// loads examples.json, :61 / :106 dump the score dicts).  This entry point is that boundary for
// array-shaped callers: pair ids in host memory in, the nine result columns in host memory out,
// every copy inside the call.  The pipeline is built around the copy-back engine, because the
// device scores a step faster than the link carries its 56 bytes per pair back (C2: 560 MB at
// ~57 GB/s = 9.8 ms, kernels ~8 ms): the ids of the leading user-side slices go up first and are
// scored at once so that the D2H engine starts early, the remaining ids follow on an upload
// stream, then business-side and user-side slices take turns, each slice's copy-back overlapping
// the next slice's scoring.  Native on purpose: issuing ~100 launches and ~100 copies per step
// from Python costs more than a millisecond of host time during which the GPU starves.
#include <algorithm>
#include <cstdlib>
#include <vector>

#include "blp_internal.h"

struct blp_host_state {
    int64_t cap = 0;   // pairs the staging buffers hold
    int32_t* d_u = nullptr;
    int32_t* d_b = nullptr;
    void* d_out[9] = {};   // u_cn u_union u_jaccard u_adamic b_cn b_union b_jaccard b_adamic pa
    // one compute stream: the copy-back engine is the bottleneck, so slices should FINISH in order
    // as early as possible (two alternating streams were measured: slices then share the SMs, the
    // first results arrive later and the step gets slower); a grid's tail is filled by the
    // warp-per-group kernel that blp_score_pairs runs beside the CTA kernel
    cudaStream_t main[1] = {nullptr};
    cudaStream_t copy = nullptr, up = nullptr;
    std::vector<cudaEvent_t> events;
};

namespace blp {
namespace {
const int kElem[9] = {4, 4, 8, 8, 4, 4, 8, 8, 8};

void host_state_free(blp_host_state* h) {
    if (!h) return;
    cudaFree(h->d_u);
    cudaFree(h->d_b);
    for (void* p : h->d_out) cudaFree(p);
    for (cudaEvent_t e : h->events) cudaEventDestroy(e);
    for (cudaStream_t m : h->main)
        if (m) cudaStreamDestroy(m);
    if (h->copy) cudaStreamDestroy(h->copy);
    if (h->up) cudaStreamDestroy(h->up);
    delete h;
}

int host_state_reserve(blp_graph* g, int64_t n) {
    if (!g->host) {
        g->host = new blp_host_state();
        BLP_CUDA_TRY(cudaStreamCreateWithFlags(&g->host->main[0], cudaStreamNonBlocking));
        BLP_CUDA_TRY(cudaStreamCreateWithFlags(&g->host->copy, cudaStreamNonBlocking));
        BLP_CUDA_TRY(cudaStreamCreateWithFlags(&g->host->up, cudaStreamNonBlocking));
    }
    blp_host_state* h = g->host;
    if (n <= h->cap) return BLP_OK;
    cudaFree(h->d_u);
    cudaFree(h->d_b);
    for (void*& p : h->d_out) {
        cudaFree(p);
        p = nullptr;
    }
    h->d_u = h->d_b = nullptr;
    h->cap = 0;
    BLP_CUDA_TRY(cudaMalloc((void**)&h->d_u, sizeof(int32_t) * (size_t)n));
    BLP_CUDA_TRY(cudaMalloc((void**)&h->d_b, sizeof(int32_t) * (size_t)n));
    for (int k = 0; k < 9; ++k) BLP_CUDA_TRY(cudaMalloc(&h->d_out[k], (size_t)kElem[k] * (size_t)n));
    h->cap = n;
    return BLP_OK;
}
}  // namespace

void host_state_destroy(blp_graph* g) {
    host_state_free(g->host);
    g->host = nullptr;
}
}  // namespace blp

extern "C" int blp_score_pairs_host(blp_graph* g, const int32_t* pair_u, const int32_t* pair_b,
                                    int64_t n, int32_t* u_cn, int32_t* u_union, double* u_jaccard,
                                    double* u_adamic, int32_t* b_cn, int32_t* b_union,
                                    double* b_jaccard, double* b_adamic, int64_t* pa,
                                    int user_slices, int lead_slices, int biz_slices) {
    using namespace blp;
    void* h_out[9] = {u_cn, u_union, u_jaccard, u_adamic, b_cn, b_union, b_jaccard, b_adamic, pa};
    if (!g || n < 0 || (n > 0 && (!pair_u || !pair_b))) {
        set_error("blp_score_pairs_host: bad argument");
        return BLP_ERR_INVALID;
    }
    bool any = false;
    for (void* p : h_out) any = any || p != nullptr;
    if (n > 0 && !any) {
        set_error("blp_score_pairs_host: no output column given");
        return BLP_ERR_INVALID;
    }
    if (n == 0) return BLP_OK;
    BLP_ON_DEVICE(g->device);
    int rc = host_state_reserve(g, n);
    if (rc != BLP_OK) return rc;
    blp_host_state* h = g->host;

    // slice plan (defaults measured on C2 with the 48-byte result set, tools/e2e_time.py: 4/1/2 10.4 ms,
    // 5/1/2 10.5, 6/1/2 11.0, 8/1/2 11.9, 3/1/2 11.0, 4/1/1 10.9 -- every slice costs a grouping pass and a tail)
    const int64_t min_slice = 65536;
    const int max_slices = (int)std::max<int64_t>(1, n / min_slice);
    const int uc = std::max(1, std::min(user_slices > 0 ? user_slices : 4, max_slices));
    const int bc = std::max(1, std::min(biz_slices > 0 ? biz_slices : 2, max_slices));
    const int lead = std::max(0, std::min(lead_slices >= 0 ? lead_slices : 1, uc - 1));
    // equal user-side slices, bounds on multiples of four pairs (growing slices, a small first one
    // and larger later ones, measured slower on C2)
    auto ubound = [&](int c) {
        if (c >= uc) return n;
        return std::min<int64_t>(n, (int64_t)((double)n * ((double)c / uc)) / 4 * 4);
    };
    auto bbound = [&](int c) { return n * c / bc; };

    size_t ev_used = 0;
    auto next_event = [&](cudaEvent_t* out) -> cudaError_t {
        if (ev_used == h->events.size()) {
            cudaEvent_t e;
            cudaError_t err = cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
            if (err != cudaSuccess) return err;
            h->events.push_back(e);
        }
        *out = h->events[ev_used++];
        return cudaSuccess;
    };
    // everything queued by a failed call is drained before returning (buffers are the caller's)
#define BLP_TRY_H(expr)                                                     \
    do {                                                                    \
        cudaError_t e__ = (expr);                                           \
        if (e__ != cudaSuccess) {                                           \
            cudaDeviceSynchronize();                                        \
            return blp::cuda_fail(e__, #expr, __FILE__, __LINE__);          \
        }                                                                   \
    } while (0)
#define BLP_RC_H(expr)                 \
    do {                               \
        int r__ = (expr);              \
        if (r__ != BLP_OK) {           \
            cudaDeviceSynchronize();   \
            return r__;                \
        }                              \
    } while (0)

    const int64_t head = ubound(lead);
    cudaEvent_t ev_head, ev_up;
    BLP_TRY_H(next_event(&ev_head));
    BLP_TRY_H(next_event(&ev_up));
    if (head > 0) {
        BLP_TRY_H(cudaMemcpyAsync(h->d_u, pair_u, sizeof(int32_t) * (size_t)head,
                                  cudaMemcpyHostToDevice, h->main[0]));
        BLP_TRY_H(cudaMemcpyAsync(h->d_b, pair_b, sizeof(int32_t) * (size_t)head,
                                  cudaMemcpyHostToDevice, h->main[0]));
    }
    BLP_TRY_H(cudaEventRecord(ev_head, h->main[0]));
    BLP_TRY_H(cudaStreamWaitEvent(h->up, ev_head, 0));   // (keeps the head first on the link)
    if (head < n) {
        BLP_TRY_H(cudaMemcpyAsync(h->d_u + head, pair_u + head, sizeof(int32_t) * (size_t)(n - head),
                                  cudaMemcpyHostToDevice, h->up));
        BLP_TRY_H(cudaMemcpyAsync(h->d_b + head, pair_b + head, sizeof(int32_t) * (size_t)(n - head),
                                  cudaMemcpyHostToDevice, h->up));
    }
    BLP_TRY_H(cudaEventRecord(ev_up, h->up));

    auto copy_back = [&](cudaStream_t from, int first, int last, int64_t lo, int64_t hi) -> cudaError_t {
        cudaEvent_t ev;
        cudaError_t err = next_event(&ev);
        if (err == cudaSuccess) err = cudaEventRecord(ev, from);
        if (err == cudaSuccess) err = cudaStreamWaitEvent(h->copy, ev, 0);
        for (int k = first; k <= last && err == cudaSuccess; ++k)
            if (h_out[k])   // a null column is computed but not copied back
                err = cudaMemcpyAsync((char*)h_out[k] + (size_t)kElem[k] * (size_t)lo,
                                  (char*)h->d_out[k] + (size_t)kElem[k] * (size_t)lo,
                                  (size_t)kElem[k] * (size_t)(hi - lo), cudaMemcpyDeviceToHost, h->copy);
        return err;
    };
    auto at = [&](int k, int64_t lo) { return (void*)((char*)h->d_out[k] + (size_t)kElem[k] * (size_t)lo); };
    auto user_slice = [&](int c) -> int {
        const int64_t lo = ubound(c), hi = ubound(c + 1);
        if (hi <= lo) return BLP_OK;
        cudaStream_t st = h->main[0];
        int r = blp_score_pairs(g, BLP_SIDE_USER, h->d_u + lo, h->d_b + lo, hi - lo, (int32_t*)at(0, lo),
                                (int32_t*)at(1, lo), (double*)at(2, lo), (double*)at(3, lo),
                                (int64_t*)at(8, lo), nullptr, st);
        if (r != BLP_OK) return r;
        cudaError_t e = copy_back(st, 0, 3, lo, hi);
        if (e == cudaSuccess && h_out[8]) {   // pa travels with the user side (written by that kernel)
            e = cudaMemcpyAsync((char*)h_out[8] + 8 * (size_t)lo, (char*)h->d_out[8] + 8 * (size_t)lo,
                                8 * (size_t)(hi - lo), cudaMemcpyDeviceToHost, h->copy);
        }
        return e == cudaSuccess ? BLP_OK : blp::cuda_fail(e, "copy-back (user side)", __FILE__, __LINE__);
    };
    auto biz_slice = [&](int c) -> int {
        const int64_t lo = bbound(c), hi = bbound(c + 1);
        if (hi <= lo) return BLP_OK;
        cudaStream_t st = h->main[0];
        int r = blp_score_pairs(g, BLP_SIDE_BUSINESS, h->d_u + lo, h->d_b + lo, hi - lo,
                                (int32_t*)at(4, lo), (int32_t*)at(5, lo), (double*)at(6, lo),
                                (double*)at(7, lo), nullptr, nullptr, st);
        if (r != BLP_OK) return r;
        cudaError_t e = copy_back(st, 4, 7, lo, hi);
        return e == cudaSuccess ? BLP_OK : blp::cuda_fail(e, "copy-back (business side)", __FILE__, __LINE__);
    };

    for (int c = 0; c < lead; ++c) BLP_RC_H(user_slice(c));
    BLP_TRY_H(cudaStreamWaitEvent(h->main[0], ev_up, 0));
    // the remaining user slices with the business slices spread evenly between them
    const int rest = uc - lead;
    const int per = rest > 0 ? (rest + bc - 1) / bc : 0;
    int bi = 0;
    for (int i = 0; i < rest; ++i) {
        if (per > 0 && i % per == 0 && bi < bc) BLP_RC_H(biz_slice(bi++));
        BLP_RC_H(user_slice(lead + i));
    }
    while (bi < bc) BLP_RC_H(biz_slice(bi++));
    BLP_TRY_H(cudaStreamSynchronize(h->copy));
    BLP_TRY_H(cudaStreamSynchronize(h->main[0]));
    BLP_TRY_H(cudaStreamSynchronize(h->up));
#undef BLP_TRY_H
#undef BLP_RC_H
    return BLP_OK;
}
