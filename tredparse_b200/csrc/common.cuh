// common.cuh — context, error plumbing and device workspace shared by the libtredsw translation units.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <stdlib.h>
#include <vector>
#include <mutex>

#include "../../include/tredsw.h"

#define TREDSW_VERSION 100

void tredsw_set_error(const char *fmt, ...);

#define CUDA_TRY(expr)                                                                        \
    do {                                                                                      \
        cudaError_t _e = (expr);                                                              \
        if (_e != cudaSuccess) {                                                              \
            tredsw_set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, \
                             __LINE__);                                                       \
            return TREDSW_ERR_CUDA;                                                           \
        }                                                                                     \
    } while (0)

// A grow-only device buffer.
struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    int ensure(size_t bytes) {
        if (bytes <= cap) return TREDSW_OK;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = bytes + bytes / 4 + 256;
        CUDA_TRY(cudaMalloc(&p, want));
        cap = want;
        return TREDSW_OK;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <class T> T *as() { return reinterpret_cast<T *>(p); }
};

// A grow-only page-locked host buffer: staging for the small per-call tables and results of the host-pointer
// entry points.  A copy to or from PAGEABLE memory makes the driver block the calling thread until the stream
// reaches the copy — and other host threads' submissions with it — so several calls in flight on one GPU
// (cohort.HostPipeline) would serialise on it; copies through this buffer are truly asynchronous.
struct PinnedBuf {
    void *p = nullptr;
    size_t cap = 0;
    int ensure(size_t bytes) {
        if (bytes <= cap) return TREDSW_OK;
        if (p) cudaFreeHost(p);
        p = nullptr; cap = 0;
        size_t want = bytes + bytes / 4 + 256;
        CUDA_TRY(cudaHostAlloc(&p, want, cudaHostAllocDefault));
        cap = want;
        return TREDSW_OK;
    }
    void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
    template <class T> T *as() { return reinterpret_cast<T *>(p); }
};

struct tredsw_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    int sm_count = 0;
    size_t smem_optin = 0;
    // staging buffers (host-pointer mode)
    DevBuf d_q, d_qoff, d_t, d_toff, d_qidx, d_tidx, d_out, d_cigar, d_scratch, d_misc, d_fam,
        d_rfam, d_stats, d_work, d_prob, d_ipool, d_dpool, d_surface, d_marg, d_res, d_counter, d_tiles, d_pk, d_pe16, d_ftab,
        d_skip;   // strip-skip counters of the packed family kernel, accumulated over the context's calls
    PinnedBuf h_in, h_out, h_tab;
    // compute token (see DeviceToken): this context's "whole call finished" event, and the event the next
    // Smith-Waterman launch on this context has to wait for (consumed by tredsw_internal_classify)
    cudaEvent_t done_ev = nullptr, sw_end_ev = nullptr, wait_before_sw = nullptr;
    bool record_sw_end = false;
    std::mutex mu;
    long long launches = 0;
    bool timing = false;
    // events: 0/1 SW, 2/3 grid, 4/5 KDE, 6/7 whole pipeline, 8 call start (before the input copies), 9 results copied
    cudaEvent_t ev[10] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    bool ev_valid[10] = {false, false, false, false, false, false, false, false, false, false};
    void mark(int i) {            // record event i on the stream when timing is enabled
        if (!timing) return;
        if (!ev[i]) cudaEventCreate(&ev[i]);
        cudaEventRecord(ev[i], stream);
        ev_valid[i] = true;
    }
    ~tredsw_ctx();
};

static inline bool dev_ptrs(uint32_t flags) { return (flags & TREDSW_DEVICE_PTRS) != 0; }

// Host-buffer calls of several contexts on one GPU (cohort.HostPipeline) pass a per-device compute token: the
// persistent Smith-Waterman kernel of a call fills every SM's shared memory, so the short kernels that FINISH
// the previous call (KDE, grid, reductions) cannot be scheduled until it drains — every call in flight then
// completes at the same moment, all of them start their input copies together, and the GPU idles meanwhile
// (measured: tools/e2e_probe.py --timeline).  With the token, the SW launch of call B waits for the last kernel
// of call A and B's pre-filter / grouping kernels for the end of A's SW kernel; B's input copies overlap all of
// A, and completions stay staggered by one step.
struct DeviceToken {
    std::mutex mu;
    cudaEvent_t ev = nullptr;     // "done" event of the most recent host-buffer call on this device
    cudaEvent_t sw_end = nullptr; // ... and the end of its Smith-Waterman kernel
};
DeviceToken &tredsw_device_token(int device);

// Gather `n` small host tables into the page-locked buffer `buf` (each at a 256-byte aligned offset, returned
// in offs[]).  The buffer is rewritten only when its content would change, and then only after the stream has
// drained — an earlier enqueue-only call may still have a copy from it in flight — so repeated calls with the
// same tables (the normal case: one catalogue for a whole cohort) neither block nor race.
static inline int stage_small(tredsw_ctx *ctx, PinnedBuf &buf, const void *const *srcs, const size_t *sizes, int n,
                              size_t *offs) {
    size_t total = 0;
    for (int i = 0; i < n; ++i) { offs[i] = total; total += (sizes[i] + 255) & ~(size_t)255; }
    bool same = buf.p != nullptr && buf.cap >= total;
    if (same) {
        const unsigned char *b = static_cast<const unsigned char *>(buf.p);
        for (int i = 0; i < n && same; ++i) same = sizes[i] == 0 || memcmp(b + offs[i], srcs[i], sizes[i]) == 0;
    }
    if (same) return TREDSW_OK;
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    int rc = buf.ensure(total > 0 ? total : 256);
    if (rc) return rc;
    unsigned char *b = static_cast<unsigned char *>(buf.p);
    for (int i = 0; i < n; ++i) if (sizes[i]) memcpy(b + offs[i], srcs[i], sizes[i]);
    return TREDSW_OK;
}

// Copy helper: returns the device pointer to use for `host_or_dev`.
template <class T>
static inline int stage_in(tredsw_ctx *ctx, DevBuf &buf, const T *src, size_t n, uint32_t flags,
                           const T **out) {
    if (dev_ptrs(flags) || n == 0) { *out = src; if (n == 0 && !dev_ptrs(flags)) { int rc = buf.ensure(16); if (rc) return rc; *out = buf.as<T>(); } return TREDSW_OK; }
    int rc = buf.ensure(n * sizeof(T));
    if (rc) return rc;
    CUDA_TRY(cudaMemcpyAsync(buf.p, src, n * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
    *out = buf.as<T>();
    return TREDSW_OK;
}
