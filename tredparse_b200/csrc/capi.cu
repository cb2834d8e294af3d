// capi.cu — context management, error plumbing and the libssw.so-compatible legacy entry points.
#include "common.cuh"
#include <stdarg.h>

static thread_local char g_err[512] = "";

void tredsw_set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

DeviceToken &tredsw_device_token(int device) {
    static DeviceToken tok[64];
    return tok[(device >= 0 && device < 64) ? device : 0];
}

tredsw_ctx::~tredsw_ctx() {
    cudaSetDevice(device);
    if (done_ev) {
        DeviceToken &t = tredsw_device_token(device);
        std::lock_guard<std::mutex> lock(t.mu);
        if (t.ev == done_ev) { t.ev = nullptr; t.sw_end = nullptr; }
        cudaEventDestroy(done_ev);
        if (sw_end_ev) cudaEventDestroy(sw_end_ev);
    }
    DevBuf *all[] = {&d_q, &d_qoff, &d_t, &d_toff, &d_qidx, &d_tidx, &d_out, &d_cigar, &d_scratch, &d_misc,
                     &d_fam, &d_rfam, &d_stats, &d_work, &d_prob, &d_ipool, &d_dpool, &d_surface, &d_marg,
                     &d_res, &d_counter, &d_tiles, &d_pk, &d_pe16, &d_ftab, &d_skip};
    for (DevBuf *b : all) b->release();
    h_in.release(); h_out.release(); h_tab.release();
    for (int i = 0; i < 10; ++i) if (ev[i]) cudaEventDestroy(ev[i]);
    if (own_stream && stream) cudaStreamDestroy(stream);
}

namespace {
// 8 independent dependent-chains of packed DPX add-max per thread, all in registers
__global__ void __launch_bounds__(256) int_peak_kernel(unsigned *sink, int iters, unsigned seed) {
    unsigned a0 = seed + threadIdx.x, a1 = a0 * 3u, a2 = a0 * 5u, a3 = a0 * 7u, a4 = a0 * 11u, a5 = a0 * 13u,
             a6 = a0 * 17u, a7 = a0 * 19u;
    const unsigned b = 0xfffe0001u, c = 0x00030002u;
#pragma unroll 1
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            a0 = __viaddmax_s16x2_relu(a0, b, c); a1 = __viaddmax_s16x2_relu(a1, b, c);
            a2 = __viaddmax_s16x2_relu(a2, b, c); a3 = __viaddmax_s16x2_relu(a3, b, c);
            a4 = __viaddmax_s16x2_relu(a4, b, c); a5 = __viaddmax_s16x2_relu(a5, b, c);
            a6 = __viaddmax_s16x2_relu(a6, b, c); a7 = __viaddmax_s16x2_relu(a7, b, c);
        }
    }
    unsigned r = a0 ^ a1 ^ a2 ^ a3 ^ a4 ^ a5 ^ a6 ^ a7;
    if (r == 0x12345678u) sink[0] = r;     // never true in practice; keeps the chains alive
}
}  // namespace

extern "C" {

int tredsw_version(void) { return TREDSW_VERSION; }

const char *tredsw_last_error(void) { return g_err; }

int tredsw_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

tredsw_ctx *tredsw_create(int device, void *stream) {
    int n = tredsw_device_count();
    if (n <= 0) { tredsw_set_error("no CUDA device available (tredsw has no CPU fallback)"); return nullptr; }
    if (device < 0 || device >= n) { tredsw_set_error("device %d out of range (0..%d)", device, n - 1); return nullptr; }
    if (cudaSetDevice(device) != cudaSuccess) { tredsw_set_error("cudaSetDevice(%d) failed", device); return nullptr; }
    tredsw_ctx *ctx = new tredsw_ctx();
    ctx->device = device;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) {
        tredsw_set_error("cudaGetDeviceProperties failed"); delete ctx; return nullptr;
    }
    ctx->sm_count = prop.multiProcessorCount;
    ctx->smem_optin = prop.sharedMemPerBlockOptin;
    if (stream) { ctx->stream = (cudaStream_t)stream; ctx->own_stream = false; }
    else {
        if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) {
            tredsw_set_error("cudaStreamCreate failed"); delete ctx; return nullptr;
        }
        ctx->own_stream = true;
    }
    return ctx;
}

void tredsw_destroy(tredsw_ctx *ctx) { delete ctx; }

int tredsw_synchronize(tredsw_ctx *ctx) {
    if (!ctx) return TREDSW_ERR_ARG;
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return TREDSW_OK;
}

int tredsw_sm_count(tredsw_ctx *ctx) { return ctx ? ctx->sm_count : 0; }

int64_t tredsw_launch_count(tredsw_ctx *ctx) { return ctx ? ctx->launches : 0; }

int tredsw_strip_skip_stats(tredsw_ctx *ctx, int64_t *out) {
    if (!ctx || !out) { tredsw_set_error("bad arguments"); return TREDSW_ERR_ARG; }
    std::lock_guard<std::mutex> lock(ctx->mu);
    memset(out, 0, TREDSW_STRIP_SKIP_STATS * sizeof(int64_t));
    if (!ctx->d_skip.p) return TREDSW_OK;          // no packed-kernel call yet
    CUDA_TRY(cudaSetDevice(ctx->device));
    CUDA_TRY(cudaMemcpyAsync(out, ctx->d_skip.p, TREDSW_STRIP_SKIP_STATS * sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return TREDSW_OK;
}

int tredsw_enable_timing(tredsw_ctx *ctx, int on) {
    if (!ctx) return TREDSW_ERR_ARG;
    ctx->timing = on != 0;
    for (int i = 0; i < 10; ++i) ctx->ev_valid[i] = false;
    return TREDSW_OK;
}

int tredsw_get_timing(tredsw_ctx *ctx, float *ms4) {
    if (!ctx || !ms4) return TREDSW_ERR_ARG;
    CUDA_TRY(cudaSetDevice(ctx->device));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    const int pairs[4][2] = {{0, 1}, {2, 3}, {4, 5}, {6, 7}};
    for (int k = 0; k < 4; ++k) {
        ms4[k] = 0.f;
        if (ctx->ev_valid[pairs[k][0]] && ctx->ev_valid[pairs[k][1]])
            CUDA_TRY(cudaEventElapsedTime(&ms4[k], ctx->ev[pairs[k][0]], ctx->ev[pairs[k][1]]));
    }
    return TREDSW_OK;
}

// Device timestamps (ms since a process-wide reference event) of the last timed call's marks, for timelines of
// several contexts sharing one GPU: ms10[i] < 0 where mark i was not recorded.
int tredsw_get_timeline(tredsw_ctx *ctx, float *ms10) {
    if (!ctx || !ms10) return TREDSW_ERR_ARG;
    static std::mutex mu;
    static cudaEvent_t ref = nullptr;
    CUDA_TRY(cudaSetDevice(ctx->device));
    {
        std::lock_guard<std::mutex> lock(mu);
        if (!ref) {
            CUDA_TRY(cudaEventCreate(&ref));
            CUDA_TRY(cudaEventRecord(ref, ctx->stream));
            CUDA_TRY(cudaEventSynchronize(ref));
        }
    }
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    for (int k = 0; k < 10; ++k) {
        ms10[k] = -1.f;
        if (ctx->ev_valid[k] && cudaEventElapsedTime(&ms10[k], ref, ctx->ev[k]) != cudaSuccess) { cudaGetLastError(); ms10[k] = -1.f; }
    }
    return TREDSW_OK;
}

int tredsw_int_pipe_peak(tredsw_ctx *ctx, double *out) {
    if (!ctx || !out) return TREDSW_ERR_ARG;
    std::lock_guard<std::mutex> lock(ctx->mu);
    CUDA_TRY(cudaSetDevice(ctx->device));
    int rc;
    if ((rc = ctx->d_counter.ensure(256))) return rc;
    const int blocks = ctx->sm_count * 8, threads = 256, iters = 4096;
    cudaEvent_t e0, e1;
    CUDA_TRY(cudaEventCreate(&e0)); CUDA_TRY(cudaEventCreate(&e1));
    double best = 0.0;
    for (int rep = 0; rep < 5; ++rep) {
        CUDA_TRY(cudaEventRecord(e0, ctx->stream));
        int_peak_kernel<<<blocks, threads, 0, ctx->stream>>>(ctx->d_counter.as<unsigned>(), iters, 12345u + rep);
        CUDA_TRY(cudaEventRecord(e1, ctx->stream));
        CUDA_TRY(cudaEventSynchronize(e1));
        float ms = 0.f;
        CUDA_TRY(cudaEventElapsedTime(&ms, e0, e1));
        const double ops = (double)blocks * threads * (double)iters * 64.0;
        const double g = ops / (ms * 1e-3) / 1e9;
        if (rep > 0 && g > best) best = g;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    *out = best;
    return TREDSW_OK;
}

// ------------------------------------------------------------------------------------------------
// libssw.so drop-in (src/ssw.h:72-182).  One launch per ssw_align call: compatibility, not speed.
// ------------------------------------------------------------------------------------------------
struct _profile {
    const int8_t *read;
    int8_t mat25[25];
    int32_t readLen;
    int32_t n;
    int8_t score_size;
};

static tredsw_ctx *legacy_ctx() {
    static std::mutex mu;
    static tredsw_ctx *ctx = nullptr;
    std::lock_guard<std::mutex> lock(mu);
    if (!ctx) {
        int dev = 0;
        const char *e = getenv("TREDSW_DEVICE");
        if (e) dev = atoi(e);
        ctx = tredsw_create(dev, nullptr);
    }
    return ctx;
}

s_profile *ssw_init(const int8_t *read, const int32_t readLen, const int8_t *mat, const int32_t n,
                    const int8_t score_size) {
    if (!read || !mat || readLen < 0 || n < 1 || n > 5) { tredsw_set_error("ssw_init: unsupported arguments"); return nullptr; }
    s_profile *p = (s_profile *)calloc(1, sizeof(s_profile));
    if (!p) return nullptr;
    p->read = read; p->readLen = readLen; p->n = n; p->score_size = score_size;
    for (int t = 0; t < 5; ++t)
        for (int q = 0; q < 5; ++q) p->mat25[t * 5 + q] = (t < n && q < n) ? mat[t * n + q] : 0;
    return p;
}

void init_destroy(s_profile *p) { free(p); }

s_align *ssw_align(const s_profile *prof, const int8_t *ref, int32_t refLen, const uint8_t weight_gapO,
                   const uint8_t weight_gapE, const uint8_t flag, const uint16_t filters,
                   const int32_t filterd, const int32_t maskLen) {
    if (!prof || !ref || refLen < 0) { tredsw_set_error("ssw_align: bad arguments"); return nullptr; }
    tredsw_ctx *ctx = legacy_ctx();
    if (!ctx) return nullptr;
    int64_t qoff[2] = {0, prof->readLen}, toff[2] = {0, refLen};
    int32_t zero = 0, out[8];
    const int cap = 2 * (prof->readLen + refLen) + 8;
    uint32_t *cig = (uint32_t *)malloc((size_t)cap * sizeof(uint32_t));
    if (!cig) return nullptr;
    int bias = 0;
    for (int i = 0; i < 25; ++i) if (prof->mat25[i] < bias) bias = prof->mat25[i];
    bias = -bias;
    uint32_t fl = TREDSW_SCORE2;
    if (prof->score_size == 1) fl |= TREDSW_FORCE_WORD;
    // first pass without CIGAR decides the flag-dependent stages (src/ssw.c:836,853)
    if (flag == 0) fl |= TREDSW_NO_BEGIN;
    int rc = tredsw_align_pairs(ctx, prof->read, qoff, 1, ref, toff, 1, &zero, &zero, 1, prof->mat25,
                                weight_gapO, weight_gapE, fl, out, nullptr, 0);
    if (rc != TREDSW_OK) { free(cig); return nullptr; }
    if (prof->score_size == 0 && out[0] + bias >= 255) {
        // 8-bit-only profile overflowed: the reference gives up here (src/ssw.c:811-815)
        tredsw_set_error("ssw_align: score overflows the 8-bit profile; use score_size 2");
        free(cig); return nullptr;
    }
    s_align *r = (s_align *)calloc(1, sizeof(s_align));
    if (!r) { free(cig); return nullptr; }
    r->score1 = (uint16_t)out[0];
    r->ref_end1 = out[2];
    r->read_end1 = out[4];
    r->ref_begin1 = -1; r->read_begin1 = -1;
    if (maskLen >= 15) { r->score2 = (uint16_t)out[5]; r->ref_end2 = out[6]; }
    else { r->score2 = 0; r->ref_end2 = -1; }
    r->cigar = nullptr; r->cigarLen = 0;
    bool want_begin = !(flag == 0 || (flag == 2 && r->score1 < filters));
    if (!want_begin || out[0] <= 0) {
        if (out[0] <= 0 && want_begin) { r->ref_begin1 = -1; r->read_begin1 = 0; }
        free(cig); return r;
    }
    r->ref_begin1 = out[1]; r->read_begin1 = out[3];
    bool want_cigar = !((7 & flag) == 0 || ((2 & flag) != 0 && r->score1 < filters) ||
                        ((4 & flag) != 0 && (r->ref_end1 - r->ref_begin1 > filterd ||
                                             r->read_end1 - r->read_begin1 > filterd)));
    if (want_cigar) {
        rc = tredsw_align_pairs(ctx, prof->read, qoff, 1, ref, toff, 1, &zero, &zero, 1, prof->mat25,
                                weight_gapO, weight_gapE, fl | TREDSW_CIGAR, out, cig, cap);
        if (rc != TREDSW_OK || out[7] <= 0) { free(cig); free(r); return nullptr; }
        r->cigar = (uint32_t *)malloc((size_t)out[7] * sizeof(uint32_t));
        if (!r->cigar) { free(cig); free(r); return nullptr; }
        memcpy(r->cigar, cig, (size_t)out[7] * sizeof(uint32_t));
        r->cigarLen = out[7];
    }
    free(cig);
    return r;
}

void align_destroy(s_align *a) {
    if (!a) return;
    free(a->cigar);
    free(a);
}

char cigar_int_to_op(uint32_t cigar_int) {
    static const char ops[] = {'M', 'I', 'D', 'N', 'S', 'H', 'P', '=', 'X'};
    uint32_t code = cigar_int & 0xfu;
    return code < sizeof(ops) ? ops[code] : 'M';
}

uint32_t cigar_int_to_len(uint32_t cigar_int) { return cigar_int >> 4; }

}  // extern "C"
