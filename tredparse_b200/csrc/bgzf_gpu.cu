// bgzf_gpu.cu — BAM ingest on the GPU for a whole batch of (sample, locus) problems.
//
// The host ingest (ingest.cpp) spends ~85 % of a locus pass inflating BGZF blocks and the rest walking records; on
// real BAMs that made the product path ingest-bound by 10^2..10^3x against the genotyping kernels.  Here the host
// only reads COMPRESSED bytes (the BGZF blocks behind the BAI chunks of every requested window, each block once per
// sample) into page-locked memory; everything else runs on the device:
//
//   inflate_kernel        one warp per BGZF block: raw-DEFLATE decoder with its Huffman tables in shared memory
//                         (16-bit entries); the 32 lanes decode the same bits and share the copying (literals by
//                         lane 0, the bytes of a match dealt to the lanes); CRC-32 of the inflated block by 32 lanes;
//   walk (count, fill)    one warp per indexed fetch (the locus window, every alt region) follows the record chain
//                         of its BAI chunks exactly like tredsw_bam::fetch, through a 4 KB shared-memory window;
//   select                one thread per record: CIGAR span / clips, the read-selection rules of
//                         BamParser.parse (bam_parser.py:194-243), the pileup depth of BamDepth.region_depth
//                         (:404-411), the pair candidates of PEextractor (:316-369);
//   scans + scatter       ordered compaction (file order is the reference's order) into rbuf / roff / read_problem
//                         / names — the layout tredsw_genotype_batch consumes, already in device memory;
//   pair_*                pairing by query name through per-problem open-addressing tables (two smallest record
//                         indices per name = the reference's "first two records"), distances into pe_lens.
//
// A BAM without an index is read by a second front end, run_scan (tredsw_ingest_scan_run): one streaming pass per
// sample, slab by slab, that finds the record boundaries on the device and hands the records of every fetch to the
// same selection / compaction / pairing steps (select_and_pair) — see the scan_* bodies of ingest_device.cuh.
//
// A third front end, run_ref_tracts (tredsw_ref_tracts), scans a FASTA, plain text or BGZF, for the tracts of
// requested motifs with the same backend and the same staging (page-locked steps read by a host thread; BGZF blocks
// inflated by inflate_kernel): ref_tracts_device.cuh.
//
// The per-thread bodies live in ingest_device.cuh as __host__ __device__ functions; the pipeline below is written
// once against a small backend (allocate / copy / for_each / scan) with a CUDA implementation and a serial host
// implementation.  The host one is TEST INFRASTRUCTURE (tredsw_ingest_batch_emulate): it lets the CPU suite compare
// the device logic with the host reader bit for bit; the package never calls it.
//
// The host side the three front ends share: typed allocation (alloc_n, alloc_host_n), device buffers reused from step
// to step (Reused), a locus query's fetches (plan_fetches), a BGZF block's inflate job (block_desc), the thread that
// reads the next step while the device works (ReadAhead), and the body of every C entry point (run_entry).
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <fcntl.h>
#include <unistd.h>
#include <sys/stat.h>

#include <algorithm>
#include <cmath>
#include <map>
#include <memory>
#include <string>
#include <thread>
#include <vector>

#include "common.cuh"
#include "ingest_internal.h"
#include "ingest_device.cuh"
#include "ref_tracts_device.cuh"

namespace tredsw_gi {       // kernel name tags (they show up in profiler listings: for_each_kernel<tredsw_gi::SelectTag, ...>)
struct WalkCountTag; struct WalkFillTag; struct SelectTag; struct SummaryTag; struct CompactTag; struct EmitTag;
struct PairInsertTag; struct PairSecondTag; struct PairEvalTag; struct PairCountTag; struct PairScatterTag;
// the scan of an unindexed BAM
struct ScanCandidateTag; struct ScanRepairTag; struct ScanCountTag; struct ScanFillTag; struct ScanMatchTag; struct ScanKeepTag;
// its STR profile (in-repeat reads)
struct ScanIrrTag; struct ScanIrrFillTag;
// the reference tract scan
struct TractPackTag; struct TractRunsTag; struct TractChainsTag;
}
using namespace tredsw_gi;

namespace {

// ---------------------------------------------------------------------------------------------------------------
// kernels
// ---------------------------------------------------------------------------------------------------------------
constexpr int INFLATE_WARPS = 4, INFLATE_THREADS = 32 * INFLATE_WARPS;   // one warp per BGZF block; per CTA 4 x 3200 B of
                                                                         // Huffman tables + 4 KB of CRC tables
constexpr size_t INFLATE_SMEM = (size_t)INFLATE_WARPS * TAB_ENTRIES * sizeof(uint16_t) + 4 * 256 * sizeof(uint32_t);

__host__ __device__ inline void crc_tables(uint32_t *t, int i /* 0..255 */) {
    uint32_t c = (uint32_t)i;
    for (int k = 0; k < 8; ++k) c = (c & 1u) ? 0xedb88320u ^ (c >> 1) : c >> 1;
    t[i] = c;
}
__host__ __device__ inline void crc_tables_ext(uint32_t *t, int i) {    // after every t[0..255] is known
    uint32_t c = t[i];
    for (int k = 1; k < 4; ++k) { c = t[c & 0xffu] ^ (c >> 8); t[k * 256 + i] = c; }
}

// status: 0 ok, 1 the decoder refused the stream, 2 CRC-32 / length mismatch
__global__ void __launch_bounds__(INFLATE_THREADS, 8)
inflate_kernel(const uint8_t *comp, uint8_t *ibuf, const BlockDesc *blocks, int nblocks, uint8_t *status, int check_crc) {
    extern __shared__ __align__(16) unsigned char smem[];
    uint16_t *tabs = reinterpret_cast<uint16_t *>(smem);
    uint32_t *crct = reinterpret_cast<uint32_t *>(smem + (size_t)INFLATE_WARPS * TAB_ENTRIES * sizeof(uint16_t));
    for (int i = threadIdx.x; i < 256; i += blockDim.x) crc_tables(crct, i);
    __syncthreads();
    for (int i = threadIdx.x; i < 256; i += blockDim.x) crc_tables_ext(crct, i);
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.x * INFLATE_WARPS + warp;
    if (b >= nblocks) return;
    const BlockDesc d = blocks[b];
    uint8_t lens[320], sub_need[1 << LIT_ROOT];
    uint16_t sub_base[1 << LIT_ROOT];
    uint8_t st = 0;
    if (d.isize > 0) {
        const TabRef tr{tabs + warp, INFLATE_WARPS, lane == 0};
        if (!inflate_block<32>(comp + d.in_off, (int64_t)d.clen, ibuf + d.out_off, (int64_t)d.isize, tr, lens, sub_need, sub_base, lane)) st = 1;
        else if (check_crc && crc32_warp(crct, ibuf + d.out_off, (int64_t)d.isize, lane) != d.crc) st = 2;
    }
    if (lane == 0) status[b] = st;
}

template <class Tag, class F>
__global__ void for_each_kernel(int64_t n, F f) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) f(i);
}
// one warp per item: f(item, lane)
template <class Tag, class F>
__global__ void for_each_warp_kernel(int64_t n, F f) {
    const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (i < n) f(i, (int)(threadIdx.x & 31));
}

// one warp per item with WALK_WINDOW bytes of shared memory per warp: f(item, lane, window)
constexpr int WALK_WARPS = 4;
template <class Tag, class F>
__global__ void __launch_bounds__(32 * WALK_WARPS) for_each_warp_window_kernel(int64_t n, F f) {
    __shared__ __align__(16) uint32_t win[WALK_WARPS][WALK_WINDOW / 4 + 4];
    const int w = threadIdx.x >> 5;
    const int64_t i = (int64_t)blockIdx.x * WALK_WARPS + w;
    if (i < n) f(i, (int)(threadIdx.x & 31), win[w]);
}

// exclusive scan of uint32 -> uint32 (n + 1 outputs, out[n] = total), three phases over tiles of SCAN_TILE elements
constexpr int SCAN_THREADS = 256, SCAN_PER_THREAD = 8, SCAN_TILE = SCAN_THREADS * SCAN_PER_THREAD;
__device__ inline uint32_t block_exclusive_scan(uint32_t v, uint32_t *total) {     // SCAN_THREADS threads
    __shared__ uint32_t warp_sums[SCAN_THREADS / 32];
    __shared__ uint32_t block_total;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    uint32_t x = v;
    for (int o = 1; o < 32; o <<= 1) { const uint32_t y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
    if (lane == 31) warp_sums[wid] = x;
    __syncthreads();
    if (wid == 0) {
        uint32_t s = lane < SCAN_THREADS / 32 ? warp_sums[lane] : 0u;
        for (int o = 1; o < 32; o <<= 1) { const uint32_t y = __shfl_up_sync(0xffffffffu, s, o); if (lane >= o) s += y; }
        if (lane < SCAN_THREADS / 32) warp_sums[lane] = s;
        if (lane == SCAN_THREADS / 32 - 1) block_total = s;
    }
    __syncthreads();
    const uint32_t before = wid ? warp_sums[wid - 1] : 0u;
    *total = block_total;
    __syncthreads();
    return before + x - v;
}
__global__ void __launch_bounds__(SCAN_THREADS) scan_tile_sums_kernel(const uint32_t *in, int64_t n, uint32_t *tile_sums) {
    const int64_t base = (int64_t)blockIdx.x * SCAN_TILE + (int64_t)threadIdx.x * SCAN_PER_THREAD;
    uint32_t s = 0;
    for (int k = 0; k < SCAN_PER_THREAD; ++k) if (base + k < n) s += in[base + k];
    uint32_t total;
    block_exclusive_scan(s, &total);
    if (threadIdx.x == 0) tile_sums[blockIdx.x] = total;
}
__global__ void __launch_bounds__(SCAN_THREADS) scan_tiles_kernel(uint32_t *tile_sums, int64_t ntiles, uint32_t *grand) {
    uint32_t carry = 0;
    for (int64_t t0 = 0; t0 < ntiles; t0 += SCAN_THREADS) {
        const int64_t t = t0 + threadIdx.x;
        const uint32_t v = t < ntiles ? tile_sums[t] : 0u;
        uint32_t total;
        const uint32_t ex = block_exclusive_scan(v, &total);
        if (t < ntiles) tile_sums[t] = carry + ex;
        carry += total;
    }
    if (threadIdx.x == 0) *grand = carry;
}
__global__ void __launch_bounds__(SCAN_THREADS) scan_apply_kernel(const uint32_t *in, int64_t n, const uint32_t *tile_sums, uint32_t *out) {
    const int64_t base = (int64_t)blockIdx.x * SCAN_TILE + (int64_t)threadIdx.x * SCAN_PER_THREAD;
    uint32_t v[SCAN_PER_THREAD], s = 0;
    for (int k = 0; k < SCAN_PER_THREAD; ++k) { v[k] = base + k < n ? in[base + k] : 0u; s += v[k]; }
    uint32_t total;
    uint32_t run = tile_sums[blockIdx.x] + block_exclusive_scan(s, &total);
    for (int k = 0; k < SCAN_PER_THREAD; ++k) if (base + k < n) { out[base + k] = run; run += v[k]; }
}

// ---------------------------------------------------------------------------------------------------------------
// backends
// ---------------------------------------------------------------------------------------------------------------
// Page-locked host blocks are expensive to create (~0.3 ms per MB) and a batch needs a few tens of MB of them: freed
// blocks are kept and handed out again (best fit), so consecutive batches of a cohort allocate nothing.
struct PinnedPool {
    struct Block { void *p; size_t cap; bool used; };
    std::mutex mu;
    std::vector<Block> blocks;
    void *get(size_t bytes) {
        std::lock_guard<std::mutex> lock(mu);
        int best = -1;
        for (int i = 0; i < (int)blocks.size(); ++i)
            if (!blocks[i].used && blocks[i].cap >= bytes && (best < 0 || blocks[i].cap < blocks[best].cap)) best = i;
        if (best >= 0 && blocks[best].cap <= 4 * bytes + (1 << 16)) { blocks[best].used = true; return blocks[best].p; }
        void *p = nullptr;
        const size_t cap = bytes + bytes / 4 + 4096;
        if (cudaHostAlloc(&p, cap, cudaHostAllocDefault) != cudaSuccess) return nullptr;
        blocks.push_back(Block{p, cap, true});
        return p;
    }
    void put(void *p) {
        std::lock_guard<std::mutex> lock(mu);
        for (Block &b : blocks) if (b.p == p) { b.used = false; return; }
    }
};
PinnedPool &pinned_pool() { static PinnedPool *pool = new PinnedPool(); return *pool; }

struct CudaBackend {
    static constexpr bool on_device = true;
    cudaStream_t stream;
    std::vector<void *> dev, pinned;
    int rc = TREDSW_OK;
    long long launches = 0;                            // kernels launched by this batch
    bool fail(cudaError_t e, const char *what) {
        if (e == cudaSuccess) return false;
        if (rc == TREDSW_OK) { tredsw_set_error("%s failed: %s", what, cudaGetErrorString(e)); rc = TREDSW_ERR_CUDA; }
        return true;
    }
    // keep = true: a result buffer (lives until the batch is freed); otherwise an intermediate of the pipeline
    // (released as soon as the results are complete: the inflated stream alone is 8x the compressed bytes)
    std::vector<void *> dev_keep, pinned_keep;
    void *alloc(size_t bytes, bool keep = false) {     // device memory (with slack for the word-wise readers)
        void *p = nullptr;
        if (fail(cudaMallocAsync(&p, bytes + 64, stream), "cudaMallocAsync")) return nullptr;
        (keep ? dev_keep : dev).push_back(p);
        return p;
    }
    void *alloc_host(size_t bytes, bool keep = false) {   // page-locked host memory
        void *p = pinned_pool().get(bytes + 64);
        if (!p) { fail(cudaErrorMemoryAllocation, "cudaHostAlloc"); return nullptr; }
        (keep ? pinned_keep : pinned).push_back(p);
        return p;
    }
    bool quiesced = false;                             // the pipeline has run to its last synchronisation
    void release_intermediates() {                     // (after a synchronisation: nothing is in flight)
        for (void *p : dev) cudaFreeAsync(p, stream);
        dev.clear();
        for (void *p : pinned) pinned_pool().put(p);
        pinned.clear();
        quiesced = true;
    }
    void upload(void *dst, const void *src, size_t bytes) { if (bytes && dst) fail(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, stream), "cudaMemcpyAsync(H2D)"); }
    void download(void *dst, const void *src, size_t bytes) { if (bytes && dst) fail(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, stream), "cudaMemcpyAsync(D2H)"); }
    void copy(void *dst, const void *src, size_t bytes) { if (bytes && dst) fail(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, stream), "cudaMemcpyAsync(D2D)"); }
    void fill(void *dst, int byte, size_t bytes) { if (bytes && dst) fail(cudaMemsetAsync(dst, byte, bytes, stream), "cudaMemsetAsync"); }
    void sync() { fail(cudaStreamSynchronize(stream), "cudaStreamSynchronize"); }
    template <class Tag, class F> void for_each(int64_t n, F f) {
        if (n <= 0 || rc) return;
        for_each_kernel<Tag><<<(unsigned)((n + 127) / 128), 128, 0, stream>>>(n, f);
        ++launches;
        fail(cudaGetLastError(), "for_each launch");
    }
    template <class Tag, class F> void for_each_warp(int64_t n, F f) {
        if (n <= 0 || rc) return;
        for_each_warp_kernel<Tag><<<(unsigned)((n * 32 + 127) / 128), 128, 0, stream>>>(n, f);
        ++launches;
        fail(cudaGetLastError(), "for_each_warp launch");
    }
    template <class Tag, class F> void for_each_warp_window(int64_t n, F f) {
        if (n <= 0 || rc) return;
        for_each_warp_window_kernel<Tag><<<(unsigned)((n + WALK_WARPS - 1) / WALK_WARPS), 32 * WALK_WARPS, 0, stream>>>(n, f);
        ++launches;
        fail(cudaGetLastError(), "for_each_warp_window launch");
    }
    void inflate(const uint8_t *comp, uint8_t *ibuf, const BlockDesc *blocks, int nblocks, uint8_t *status, int check_crc) {
        if (nblocks <= 0 || rc) return;
        static bool attr_set[64] = {false};
        int devid = 0;
        cudaGetDevice(&devid);
        if (devid < 64 && !attr_set[devid]) {
            if (fail(cudaFuncSetAttribute(inflate_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)INFLATE_SMEM), "cudaFuncSetAttribute")) return;
            attr_set[devid] = true;
        }
        inflate_kernel<<<(nblocks + INFLATE_WARPS - 1) / INFLATE_WARPS, INFLATE_THREADS, INFLATE_SMEM, stream>>>(comp, ibuf, blocks, nblocks, status, check_crc);
        ++launches;
        fail(cudaGetLastError(), "inflate launch");
    }
    // out[0..n] = exclusive prefix sums of in[0..n)
    void scan(const uint32_t *in, int64_t n, uint32_t *out) {
        if (rc) return;
        if (n <= 0) { fill(out, 0, sizeof(uint32_t)); return; }
        const int64_t ntiles = (n + SCAN_TILE - 1) / SCAN_TILE;
        uint32_t *tiles = static_cast<uint32_t *>(alloc((size_t)ntiles * sizeof(uint32_t)));
        if (!tiles) return;
        scan_tile_sums_kernel<<<(unsigned)ntiles, SCAN_THREADS, 0, stream>>>(in, n, tiles);
        scan_tiles_kernel<<<1, SCAN_THREADS, 0, stream>>>(tiles, ntiles, out + n);
        scan_apply_kernel<<<(unsigned)ntiles, SCAN_THREADS, 0, stream>>>(in, n, tiles, out);
        launches += 3;
        fail(cudaGetLastError(), "scan launch");
    }
    void release() {
        for (void *p : dev) cudaFreeAsync(p, stream);
        for (void *p : dev_keep) cudaFreeAsync(p, stream);
        dev.clear(); dev_keep.clear();
        // a finished batch has nothing in flight (and its stream may be busy with the NEXT batch by now: waiting for it
        // would stall the thread that frees this one); an aborted one may still have copies into the pinned buffers
        if (!quiesced) cudaStreamSynchronize(stream);
        for (void *p : pinned) pinned_pool().put(p);
        for (void *p : pinned_keep) pinned_pool().put(p);
        pinned.clear(); pinned_keep.clear();
    }
};

struct HostBackend {                                   // serial emulation of the same pipeline (tests only)
    static constexpr bool on_device = false;
    std::vector<void *> mem;
    int rc = TREDSW_OK;
    std::vector<void *> mem_keep;
    void *alloc(size_t bytes, bool keep = false) {
        void *p = calloc(bytes + 64, 1);
        if (!p) { rc = TREDSW_ERR_ARG; tredsw_set_error("out of memory"); }
        (keep ? mem_keep : mem).push_back(p);
        return p;
    }
    void *alloc_host(size_t bytes, bool keep = false) { return alloc(bytes, keep); }
    void release_intermediates() { for (void *p : mem) free(p); mem.clear(); }
    void upload(void *dst, const void *src, size_t bytes) { if (bytes && dst) memcpy(dst, src, bytes); }
    void download(void *dst, const void *src, size_t bytes) { if (bytes && dst) memcpy(dst, src, bytes); }
    void copy(void *dst, const void *src, size_t bytes) { if (bytes && dst) memcpy(dst, src, bytes); }
    void fill(void *dst, int byte, size_t bytes) { if (bytes && dst) memset(dst, byte, bytes); }
    void sync() {}
    template <class Tag, class F> void for_each(int64_t n, F f) { for (int64_t i = 0; i < n && !rc; ++i) f(i); }
    template <class Tag, class F> void for_each_warp(int64_t n, F f) { for (int64_t i = 0; i < n && !rc; ++i) f(i, 0); }
    template <class Tag, class F> void for_each_warp_window(int64_t n, F f) { for (int64_t i = 0; i < n && !rc; ++i) f(i, 0, nullptr); }
    void inflate(const uint8_t *comp, uint8_t *ibuf, const BlockDesc *blocks, int nblocks, uint8_t *status, int check_crc) {
        std::vector<uint32_t> crct(1024);
        for (int i = 0; i < 256; ++i) crc_tables(crct.data(), i);
        for (int i = 0; i < 256; ++i) crc_tables_ext(crct.data(), i);
        std::vector<uint16_t> tabs(TAB_ENTRIES);
        uint8_t lens[320], sub_need[1 << LIT_ROOT];
        uint16_t sub_base[1 << LIT_ROOT];
        for (int b = 0; b < nblocks; ++b) {
            const BlockDesc &d = blocks[b];
            uint8_t st = 0;
            if (d.isize > 0) {
                const TabRef tr{tabs.data(), 1, true};
                if (!inflate_block<1>(comp + d.in_off, (int64_t)d.clen, ibuf + d.out_off, (int64_t)d.isize, tr, lens, sub_need, sub_base, 0)) st = 1;
                else if (check_crc) {                          // segmented like the 32 lanes of the device
                    uint32_t parts[32];
                    for (int l = 0; l < 32; ++l) {
                        int64_t sb, sl;
                        crc_segment<32>((int64_t)d.isize, l, &sb, &sl);
                        parts[l] = crc32_bytes(crct.data(), ibuf + d.out_off + sb, sl);
                    }
                    if (crc_fold_serial<32>(parts, (int64_t)d.isize) != d.crc) st = 2;
                }
            }
            status[b] = st;
        }
    }
    void scan(const uint32_t *in, int64_t n, uint32_t *out) { uint32_t s = 0; for (int64_t i = 0; i < n; ++i) { out[i] = s; s += in[i]; } out[n > 0 ? n : 0] = s; }
    void release() { for (void *p : mem) free(p); for (void *p : mem_keep) free(p); mem.clear(); mem_keep.clear(); }
};

// n elements of T, at least one (every buffer exists, so that an empty batch needs no special case)
template <class T, class B> T *alloc_n(B &be, int64_t n, bool keep = false) {
    void *p = be.alloc(sizeof(T) * (size_t)std::max<int64_t>(1, n), keep);
    return static_cast<T *>(p);
}
template <class T, class B> T *alloc_host_n(B &be, int64_t n, bool keep = false) {
    void *p = be.alloc_host(sizeof(T) * (size_t)std::max<int64_t>(1, n), keep);
    return static_cast<T *>(p);
}

// A device buffer reused from step to step (slab, FASTA step) that grows geometrically.  An outgrown block is not
// freed: it stays with the batch until release, because kernels in flight and the carry copy may still read it.
template <class T> struct Reused {
    T *p = nullptr;
    int64_t cap = 0;                                    // elements
    template <class B> T *get(B &be, int64_t n) {       // room for n elements (at least one)
        n = std::max<int64_t>(1, n);
        if (!p || n > cap) { cap = std::max(n, 2 * cap); p = alloc_n<T>(be, cap); }
        return p;
    }
    // get() for a buffer whose first `used` elements must survive the growth: they are copied into the new block
    template <class B> T *get_keeping(B &be, int64_t n, int64_t used) {
        T *old = p;
        get(be, n);
        if (p != old) be.copy(p, old, sizeof(T) * (size_t)used);
        return p;
    }
};

// A host thread that reads step k + 1 while the device works on step k; joined at the end of the step and on every
// return from the front end (an error return must not leave it writing into a released buffer).
struct ReadAhead {
    std::thread t;
    template <class... A> void start(A &&...a) { t = std::thread(std::forward<A>(a)...); }
    void join() { if (t.joinable()) t.join(); }
    ~ReadAhead() { join(); }
};

// Per-problem status of a batch (tredsw_ingest_view.status); a scan gives all its problems the status of the scan.
enum ProblemStatus : int32_t {
    PROBLEM_OK = 0,
    PROBLEM_STAGING = 1,        // the sample could not be staged: I/O, index, BGZF framing, contig out of range
    PROBLEM_INFLATE = 2,        // a block failed to inflate or its CRC-32 / length differs
    PROBLEM_CORRUPT = 3,        // corrupt or truncated records
    PROBLEM_UNSORTED = 4,       // (scan only) the file is not sorted by coordinate
};

struct ProblemSummary {         // device -> host after the selection pass
    uint32_t read0, nreads, base0, nbases, name0, name_bytes, pe0, npe;
};

}  // namespace

// ---------------------------------------------------------------------------------------------------------------
// the batch object
// ---------------------------------------------------------------------------------------------------------------
struct tredsw_ingest_batch {
    static constexpr bool keeps_backend = true;     // its device buffers are the view (run_entry)
    bool emulated = false;
    CudaBackend cuda;
    HostBackend host;
    int32_t nproblems = 0;
    std::vector<tredsw_locus_summary> summaries;
    std::vector<int32_t> status;                    // per problem: a ProblemStatus
    std::vector<tredsw_problem_span> spans;
    tredsw_ingest_view view;
    double ms_host_stage = 0, ms_total = 0, ms_marks[4] = {0, 0, 0, 0};
    long long n_blocks = 0, n_records = 0;
    long long comp_bytes = 0, inflated_bytes = 0;
    int64_t scan_stats[TREDSW_SCAN_NSTATS] = {0};   // tredsw_ingest_scan_stats
    bool irr_on = false;                            // the scan profiled in-repeat reads (tredsw_ingest_scan_irr)
    std::vector<IrrEntry> irr_entries;
    std::vector<char> irr_names;
    tredsw_irr_view irr_view;
    void reset(int32_t nq) {                        // nq problems, all ok, no evidence yet
        nproblems = nq;
        summaries.assign(nq, tredsw_locus_summary{});
        status.assign(nq, PROBLEM_OK);
        spans.assign(nq, tredsw_problem_span{});
        memset(&view, 0, sizeof(view));
    }
};
static_assert(sizeof(IrrEntry) == sizeof(tredsw_irr_entry), "IrrEntry mirrors tredsw_irr_entry");

namespace {

double now_ms() { timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6; }

// The BGZF framing of the block at h, `avail` bytes of which are at hand: 1 parsed, 0 the block is not all there,
// -1 not a valid block (*why says what is wrong or missing).
struct BgzfFrame { int xlen, bsize /* bytes of the whole block */, clen; uint32_t crc, isize; };
// The header alone (xlen, bsize, clen): the same results, with the block's end not needed.
int parse_bgzf_header(const uint8_t *h, int64_t avail, BgzfFrame *f, const char **why) {
    if (avail < 18) { *why = "truncated BGZF block header"; return 0; }
    if (h[0] != 31 || h[1] != 139 || !(h[3] & 4)) { *why = "not a BGZF block"; return -1; }
    f->xlen = h[10] | (h[11] << 8);
    if (12 + f->xlen > avail) { *why = "truncated BGZF block header"; return 0; }
    int bsize = -1;
    for (int off = 0; off + 4 <= f->xlen;) {
        const int slen = h[12 + off + 2] | (h[12 + off + 3] << 8);
        if (h[12 + off] == 66 && h[12 + off + 1] == 67 && off + 6 <= f->xlen) bsize = h[12 + off + 4] | (h[12 + off + 5] << 8);
        off += 4 + slen;
    }
    if (bsize < 0) { *why = "BGZF block without a BC field"; return -1; }
    f->clen = bsize - f->xlen - 19;
    if (f->clen < 0) { *why = "bad BGZF block size"; return -1; }
    f->bsize = bsize + 1;
    return 1;
}
int parse_bgzf_block(const uint8_t *h, int64_t avail, BgzfFrame *f, const char **why) {
    const int rc = parse_bgzf_header(h, avail, f, why);
    if (rc != 1) return rc;
    if (f->bsize > avail) { *why = "truncated BGZF block"; return 0; }
    memcpy(&f->crc, h + f->bsize - 8, 4); memcpy(&f->isize, h + f->bsize - 4, 4);
    if (f->isize > 65536) { *why = "BGZF block larger than 64 KiB"; return -1; }
    return 1;
}
// The inflate job of a parsed block that starts at in_off in the staging buffer and inflates to out_off.
BlockDesc block_desc(const BgzfFrame &f, int64_t in_off, int64_t out_off) {
    BlockDesc d;
    d.in_off = in_off + 12 + f.xlen; d.out_off = out_off;
    d.clen = (uint32_t)f.clen; d.isize = f.isize; d.crc = f.crc; d.pad_ = 0;
    return d;
}

int64_t pread_full(int fd, uint8_t *dst, int64_t n, int64_t off) {     // -> the bytes read (< n: end of file or error)
    int64_t got = 0;
    while (got < n) {
        const ssize_t k = pread(fd, dst + got, (size_t)(n - got), (off_t)(off + got));
        if (k <= 0) break;
        got += k;
    }
    return got;
}

// the windows of one locus (extract_locus_impl)
ProblemParams problem_params(const tredsw_locus_query &q) {
    ProblemParams pp;
    const int64_t start = q.repeat_start, end = q.repeat_end;
    pp.tid = q.tid; pp.span = q.span;
    pp.win_s = std::max<int64_t>(0, start - q.pad); pp.win_e = end + q.pad;
    pp.read_s = std::max<int64_t>(0, start - q.readlen); pp.read_e = end + q.readlen;
    pp.pe_s = std::max<int64_t>(start - q.pe_window, 0); pp.pe_e = end + q.pe_window;
    pp.tstart = start - q.flankmatch; pp.tend = end + q.flankmatch;
    return pp;
}

// The fetches of one locus query, in output order: its window (kind 0), then its alt regions whose contig is in
// [0, n_ref) (kind 1).  fetch(kind, tid, start, end), start clamped at 0.  False, and no fetch, when the locus's own
// contig is out of range.
template <class F> bool plan_fetches(const tredsw_locus_query &q, int32_t n_ref, ProblemParams *pp, F &&fetch) {
    if (q.tid < 0 || q.tid >= n_ref) return false;
    *pp = problem_params(q);
    auto add = [&](int kind, int32_t tid, int64_t s, int64_t e) { fetch(kind, tid, s < 0 ? 0 : s, e); };
    add(0, q.tid, std::min(pp->win_s, pp->pe_s), std::max(pp->win_e, pp->pe_e));
    for (int a = 0; a < q.n_alts && q.alts; ++a) {
        const int32_t atid = q.alts[3 * a], as = q.alts[3 * a + 1], ae = q.alts[3 * a + 2];
        if (atid >= 0 && atid < n_ref) add(1, atid, as, ae);
    }
    return true;
}

// One sample: the fetches of its problems (the locus window, then the alt regions), their BAI chunks, and the merged
// ranges of BGZF blocks behind them (every block is read and inflated once per sample).
struct SamplePlan {
    tredsw_bam *bam = nullptr;
    std::vector<int> problems;                      // batch-wide problem indices of this sample, in order
    struct PFetch { int problem, kind, tid; int64_t start, end; std::vector<std::pair<uint64_t, uint64_t>> chunks; };
    std::vector<PFetch> fetches;
    std::vector<std::pair<int64_t, int64_t>> ranges;   // merged [first block offset, last block offset]
    std::vector<int64_t> range_comp_off;               // where each range's bytes live in comp
    std::vector<int64_t> range_bytes;
    int64_t file_size = 0;
};

}  // namespace

// ---------------------------------------------------------------------------------------------------------------
// pipeline
// ---------------------------------------------------------------------------------------------------------------
template <class B>
int select_and_pair(B &be, tredsw_ingest_batch *out, const uint8_t *d_rbytes, const Fetch *d_fetches, const int64_t *d_rpos,
                    const int32_t *d_rfetch, const uint32_t *d_fbase, int64_t nrec, const std::vector<int32_t> &fetch_first,
                    const std::vector<ProblemParams> &params, const ProblemParams *d_params, ProblemCounts *d_counts,
                    bool want_names, double t_begin);

template <class B>
int run_pipeline(B &be, tredsw_ingest_batch *out, tredsw_bam *const *bams, const int32_t *sample_of,
                        const tredsw_locus_query *queries, int32_t nq, uint32_t flags) {
    const double t_begin = now_ms();
    const bool want_names = (flags & TREDSW_INGEST_NO_NAMES) == 0;
    const int check_crc = (flags & TREDSW_INGEST_NO_CRC) == 0;
    out->reset(nq);
    if (nq == 0) return TREDSW_OK;

    // ---- (1) plans per sample: fetches, chunks, merged block ranges --------------------------------------------
    int nsamples = 0;
    for (int i = 0; i < nq; ++i) { if (sample_of[i] < 0) { tredsw_set_error("negative sample index"); return TREDSW_ERR_ARG; } nsamples = std::max(nsamples, sample_of[i] + 1); }
    std::vector<SamplePlan> plans(nsamples);
    for (int i = 0; i < nq; ++i) {
        SamplePlan &sp = plans[sample_of[i]];
        sp.bam = bams[sample_of[i]];
        if (!sp.bam) { tredsw_set_error("null BAM handle for sample %d", sample_of[i]); return TREDSW_ERR_ARG; }
        if (sp.bam->is_stream()) { tredsw_set_error("%s is a stream: scan it (tredsw_ingest_scan_run)", sp.bam->path.c_str()); return TREDSW_ERR_UNSUPPORTED; }
        if (!sp.bam->has_index) { tredsw_set_error("%s has no index: scan it (tredsw_ingest_scan_run)", sp.bam->path.c_str()); return TREDSW_ERR_UNSUPPORTED; }
        sp.problems.push_back(i);
    }
    std::vector<ProblemParams> params(nq);
    // the samples are independent: their plans (index queries), reads (pread) and BGZF framing go to host threads
    const int nthreads = std::max(1, std::min({nsamples, (int)std::thread::hardware_concurrency(), 16}));
    auto parallel_samples = [&](auto &&body) {
        if (nthreads <= 1) { for (int s = 0; s < nsamples; ++s) body(s); return; }
        std::vector<std::thread> pool;
        for (int t = 0; t < nthreads; ++t) pool.emplace_back([&, t]() { for (int s = t; s < nsamples; s += nthreads) body(s); });
        for (auto &th : pool) th.join();
    };
    parallel_samples([&](int s) {
        SamplePlan &sp = plans[s];
        if (!sp.bam) return;
        const int fd = fileno(sp.bam->bgzf.fh);
        struct stat st;
        sp.file_size = fstat(fd, &st) == 0 ? (int64_t)st.st_size : 0;
        std::vector<std::pair<int64_t, int64_t>> raw;
        for (int p : sp.problems) {
            const bool planned = plan_fetches(queries[p], (int32_t)sp.bam->names.size(), &params[p],
                                              [&](int kind, int32_t tid, int64_t fs, int64_t fe) {
                SamplePlan::PFetch f;
                f.problem = p; f.kind = kind; f.tid = tid; f.start = fs; f.end = fe;
                f.chunks = sp.bam->chunks(tid, f.start, f.end);
                for (auto &c : f.chunks) {
                    const int64_t cb = (int64_t)(c.first >> 16);
                    int64_t ce = (int64_t)(c.second >> 16);
                    if ((c.second & 0xffff) == 0 && ce > cb) ce -= 1;       // the end block itself is not read: any offset
                                                                            // inside the previous block keeps it in range
                    raw.emplace_back(cb, ce);
                }
                sp.fetches.push_back(std::move(f));
            });
            if (!planned) out->status[p] = PROBLEM_STAGING;
        }
        std::sort(raw.begin(), raw.end());
        for (auto &r : raw) {
            if (!sp.ranges.empty() && r.first <= sp.ranges.back().second) sp.ranges.back().second = std::max(sp.ranges.back().second, r.second);
            else sp.ranges.push_back(r);
        }
    });
    // ---- (2) read the compressed bytes of every range into page-locked memory, parse the BGZF framing ----------
    int64_t comp_total = 0;
    for (SamplePlan &sp : plans) {
        for (auto &r : sp.ranges) {
            // `second` is an offset inside the last block wanted: that block ends at most 64 KiB later
            const int64_t bytes = std::max<int64_t>(0, std::min(sp.file_size, r.second + 65536 + 8) - r.first);
            sp.range_comp_off.push_back(comp_total);
            sp.range_bytes.push_back(bytes);
            comp_total += (bytes + 15) & ~(int64_t)15;
        }
    }
    uint8_t *h_comp = alloc_host_n<uint8_t>(be, comp_total + 16);
    if (be.rc) return be.rc;
    std::vector<Chunk> chunks;
    std::vector<Fetch> fetches;
    std::vector<int32_t> fetch_first(nq + 1, 0);
    // (offsets into ibuf are relative to the sample's first block until the samples are laid out one after the other)
    struct LoadedBlock { int64_t coffset; int64_t out_off; uint32_t isize; int64_t run_end; };
    std::vector<std::vector<LoadedBlock>> loaded(nsamples);
    std::vector<std::vector<BlockDesc>> sample_blocks(nsamples);
    std::vector<int64_t> sample_inflated(nsamples, 0);
    std::vector<const char *> sample_error(nsamples, nullptr);
    parallel_samples([&](int s) {
        SamplePlan &sp = plans[s];
        if (!sp.bam) return;
        const int fd = fileno(sp.bam->bgzf.fh);
        bool ok = true;
        const char *why = "";
        std::vector<LoadedBlock> &lb = loaded[s];
        int64_t cursor = 0;
        for (size_t r = 0; r < sp.ranges.size() && ok; ++r) {
            uint8_t *dst = h_comp + sp.range_comp_off[r];
            const int64_t got = pread_full(fd, dst, sp.range_bytes[r], sp.ranges[r].first);
            const size_t first_block = lb.size();
            int64_t o = 0;
            while (sp.ranges[r].first + o <= sp.ranges[r].second) {
                if (o == got) { if (got < sp.range_bytes[r]) { ok = false; why = "short read"; } break; }
                BgzfFrame fr;
                if (parse_bgzf_block(dst + o, got - o, &fr, &why) != 1) { ok = false; break; }
                sample_blocks[s].push_back(block_desc(fr, sp.range_comp_off[r] + o, cursor));
                lb.push_back(LoadedBlock{sp.ranges[r].first + o, cursor, fr.isize, 0});
                cursor += fr.isize;
                o += fr.bsize;
            }
            for (size_t k = first_block; k < lb.size(); ++k) lb[k].run_end = cursor;
        }
        sample_inflated[s] = cursor;
        if (!ok) sample_error[s] = why;
    });
    std::vector<BlockDesc> blocks;
    int64_t ibuf_total = 0;
    for (int s = 0; s < nsamples; ++s) {
        for (BlockDesc &d : sample_blocks[s]) { d.out_off += ibuf_total; blocks.push_back(d); }
        for (LoadedBlock &b : loaded[s]) { b.out_off += ibuf_total; b.run_end += ibuf_total; }
        ibuf_total += sample_inflated[s];
        if (sample_error[s]) {
            for (int p : plans[s].problems) if (!out->status[p]) out->status[p] = PROBLEM_STAGING;
            tredsw_set_error("%s: %s", plans[s].bam->path.c_str(), sample_error[s]);
        }
    }
    // fetches and chunks, problem-major (= output order): the window first, then the alt regions in order
    {
        std::vector<std::vector<const SamplePlan::PFetch *>> by_problem(nq);
        for (SamplePlan &sp : plans) for (auto &f : sp.fetches) by_problem[f.problem].push_back(&f);
        for (int p = 0; p < nq; ++p) {
            fetch_first[p] = (int32_t)fetches.size();
            if (out->status[p]) continue;
            const std::vector<LoadedBlock> &lb = loaded[sample_of[p]];
            auto find_block = [&](int64_t coff) -> const LoadedBlock * {       // last loaded block with coffset <= coff
                auto it = std::upper_bound(lb.begin(), lb.end(), coff, [](int64_t v, const LoadedBlock &b) { return v < b.coffset; });
                return it == lb.begin() ? nullptr : &*(it - 1);
            };
            for (const SamplePlan::PFetch *pf : by_problem[p]) {
                Fetch f;
                f.problem = p; f.kind = pf->kind; f.tid = pf->tid; f.start = pf->start; f.end = pf->end; f.pad_ = 0;
                f.chunk_begin = (int32_t)chunks.size();
                for (auto &c : pf->chunks) {
                    const LoadedBlock *b0 = find_block((int64_t)(c.first >> 16)), *b1 = find_block((int64_t)(c.second >> 16));
                    if (!b0 || b0->coffset != (int64_t)(c.first >> 16) || !b1) { out->status[p] = PROBLEM_STAGING; break; }
                    Chunk ch;
                    ch.begin = b0->out_off + std::min<int64_t>((int64_t)(c.first & 0xffff), b0->isize);
                    ch.end = b1->coffset == (int64_t)(c.second >> 16) ? b1->out_off + std::min<int64_t>((int64_t)(c.second & 0xffff), b1->isize)
                                                                     : b1->out_off + b1->isize;
                    ch.run_end = b0->run_end;
                    if (ch.end > ch.run_end) ch.end = ch.run_end;
                    chunks.push_back(ch);
                }
                f.chunk_end = (int32_t)chunks.size();
                fetches.push_back(f);
            }
        }
        fetch_first[nq] = (int32_t)fetches.size();
    }
    out->ms_host_stage = now_ms() - t_begin;
    out->n_blocks = (long long)blocks.size();
    out->comp_bytes = comp_total; out->inflated_bytes = ibuf_total;
    const int nblocks = (int)blocks.size(), nfetch = (int)fetches.size();

    // ---- (3) device: inflate ------------------------------------------------------------------------------------
    uint8_t *d_comp = alloc_n<uint8_t>(be, comp_total + 16);
    uint8_t *d_ibuf = alloc_n<uint8_t>(be, ibuf_total + 16);
    BlockDesc *d_blocks = alloc_n<BlockDesc>(be, nblocks);
    uint8_t *d_bstatus = alloc_n<uint8_t>(be, nblocks);
    uint8_t *h_bstatus = alloc_host_n<uint8_t>(be, nblocks);
    Chunk *d_chunks = alloc_n<Chunk>(be, (int64_t)chunks.size());
    Fetch *d_fetches = alloc_n<Fetch>(be, nfetch);
    ProblemParams *d_params = alloc_n<ProblemParams>(be, nq);
    ProblemCounts *d_counts = alloc_n<ProblemCounts>(be, nq);
    uint32_t *d_fcount = alloc_n<uint32_t>(be, nfetch + 1);
    uint32_t *d_fbase = alloc_n<uint32_t>(be, nfetch + 2);
    uint32_t *d_ferr = alloc_n<uint32_t>(be, nfetch + 1);
    uint32_t *h_fbase = alloc_host_n<uint32_t>(be, nfetch + 2);
    if (be.rc) return be.rc;
    be.upload(d_comp, h_comp, (size_t)comp_total);
    be.upload(d_blocks, blocks.data(), sizeof(BlockDesc) * (size_t)nblocks);
    be.upload(d_chunks, chunks.data(), sizeof(Chunk) * chunks.size());
    be.upload(d_fetches, fetches.data(), sizeof(Fetch) * (size_t)nfetch);
    be.upload(d_params, params.data(), sizeof(ProblemParams) * (size_t)nq);
    be.fill(d_counts, 0, sizeof(ProblemCounts) * (size_t)nq);
    be.inflate(d_comp, d_ibuf, d_blocks, nblocks, d_bstatus, check_crc);
    be.download(h_bstatus, d_bstatus, (size_t)nblocks);

    // ---- (4) record walk: count, then fill ------------------------------------------------------------------------
    {
        const uint8_t *ibuf = d_ibuf; const Fetch *fe = d_fetches; const Chunk *ch = d_chunks;
        uint32_t *fcount = d_fcount, *ferr = d_ferr;
        const int64_t ibuf_len = ((ibuf_total + 16) / 16) * 16;               // (allocated: ibuf_total + 16 + slack)
        be.template for_each_warp_window<WalkCountTag>(nfetch, [=] __host__ __device__(int64_t i, int lane, uint32_t *win) {
            uint32_t n = 0;
            const bool ok = walk_fetch_lanes(ibuf, ibuf_len, fe[i], ch, lane, win, [&](int64_t) { ++n; });
            if (lane == 0) { fcount[i] = n; ferr[i] = ok ? 0u : 1u; }
        });
    }
    be.scan(d_fcount, nfetch, d_fbase);
    be.download(h_fbase, d_fbase, sizeof(uint32_t) * (size_t)(nfetch + 1));
    uint32_t *h_ferr = alloc_host_n<uint32_t>(be, nfetch + 1);
    be.download(h_ferr, d_ferr, sizeof(uint32_t) * (size_t)nfetch);
    be.sync();                                                                                  // sync 1
    out->ms_marks[0] = now_ms() - t_begin;
    if (be.rc) return be.rc;
    {
        // blocks the decoder refused or whose CRC differs: the problems reading them are reported (the caller
        // falls back to the host reader for those samples, which has zlib behind it)
        bool any = false;
        for (int b = 0; b < nblocks; ++b) any = any || h_bstatus[b] != 0;
        if (any) {
            int b = 0;
            for (int s = 0; s < nsamples; ++s) {
                bool bad = false;
                for (size_t k = 0; k < loaded[s].size(); ++k, ++b) bad = bad || h_bstatus[b] != 0;
                if (bad) for (int p : plans[s].problems) if (!out->status[p]) out->status[p] = PROBLEM_INFLATE;
            }
        }
        for (int f = 0; f < nfetch; ++f) if (h_ferr[f] && !out->status[fetches[f].problem]) out->status[fetches[f].problem] = PROBLEM_CORRUPT;
    }
    const int64_t nrec = h_fbase[nfetch];
    out->n_records = nrec;
    int64_t *d_rpos = alloc_n<int64_t>(be, nrec);
    int32_t *d_rfetch = alloc_n<int32_t>(be, nrec);
    if (be.rc) return be.rc;
    {
        const uint8_t *ibuf = d_ibuf; const Fetch *fe = d_fetches; const Chunk *ch = d_chunks;
        const uint32_t *fbase = d_fbase;
        int64_t *rpos = d_rpos; int32_t *rfetch = d_rfetch;
        const int64_t ibuf_len = ((ibuf_total + 16) / 16) * 16;
        be.template for_each_warp_window<WalkFillTag>(nfetch, [=] __host__ __device__(int64_t i, int lane, uint32_t *win) {
            uint32_t k = fbase[i];                               // (a fetch flagged by the count pass yields the same prefix)
            const uint32_t stop = fbase[i + 1];
            walk_fetch_lanes(ibuf, ibuf_len, fe[i], ch, lane, win, [&](int64_t p) {
                if (k < stop && lane == 0) { rpos[k] = p; rfetch[k] = (int32_t)i; }
                ++k;
            });
        });
    }
    return select_and_pair(be, out, d_ibuf, d_fetches, d_rpos, d_rfetch, d_fbase, nrec, fetch_first, params, d_params,
                           d_counts, want_names, t_begin);
}

// Steps (5) to (7), shared by both front ends (the indexed walk above, the scan of an unindexed BAM below): per-record
// selection, ordered compaction, pairing by name, results.  rpos[i] is where record i starts in `rbytes`, rfetch[i] its
// fetch; the records are grouped by fetch (fetch f owns [fbase[f], fbase[f + 1])) and are in file order within a fetch.
template <class B>
int select_and_pair(B &be, tredsw_ingest_batch *out, const uint8_t *d_rbytes, const Fetch *d_fetches, const int64_t *d_rpos,
                    const int32_t *d_rfetch, const uint32_t *d_fbase, int64_t nrec, const std::vector<int32_t> &fetch_first,
                    const std::vector<ProblemParams> &params, const ProblemParams *d_params, ProblemCounts *d_counts,
                    bool want_names, double t_begin) {
    const int32_t nq = out->nproblems;
    const uint8_t *d_ibuf = d_rbytes;
    uint32_t *d_emit = alloc_n<uint32_t>(be, nrec + 1);
    uint32_t *d_bases = alloc_n<uint32_t>(be, nrec + 1);
    uint32_t *d_nameb = alloc_n<uint32_t>(be, nrec + 1);
    uint32_t *d_pe = alloc_n<uint32_t>(be, nrec + 1);
    uint32_t *d_semit = alloc_n<uint32_t>(be, nrec + 2);
    uint32_t *d_sbases = alloc_n<uint32_t>(be, nrec + 2);
    uint32_t *d_snameb = alloc_n<uint32_t>(be, nrec + 2);
    uint32_t *d_spe = alloc_n<uint32_t>(be, nrec + 2);
    Mate *d_mates = alloc_n<Mate>(be, nrec);
    int32_t *d_ffirst = alloc_n<int32_t>(be, nq + 1);
    ProblemSummary *d_psum = alloc_n<ProblemSummary>(be, nq);
    ProblemSummary *h_psum = alloc_host_n<ProblemSummary>(be, nq);
    ProblemCounts *h_counts = alloc_host_n<ProblemCounts>(be, nq);
    if (be.rc) return be.rc;
    be.upload(d_ffirst, fetch_first.data(), sizeof(int32_t) * (size_t)(nq + 1));
    {
        // ---- (5) per-record selection --------------------------------------------------------------------------------
        const uint8_t *ibuf = d_ibuf; const Fetch *fe = d_fetches;
        const int64_t *rpos = d_rpos; const int32_t *rfetch = d_rfetch;
        const ProblemParams *pp = d_params; ProblemCounts *pc = d_counts;
        uint32_t *emit = d_emit, *bases = d_bases, *nameb = d_nameb, *pe = d_pe;
        Mate *mates = d_mates;
        be.template for_each<SelectTag>(nrec, [=] __host__ __device__(int64_t i) {
            const Fetch &f = fe[rfetch[i]];
            const RecOut o = select_record(ibuf, rpos[i], f, pp[f.problem], &pc[f.problem], &mates[i]);
            emit[i] = o.emit; bases[i] = o.bases; nameb[i] = o.name_bytes; pe[i] = o.pe;
        });
    }
    be.scan(d_emit, nrec, d_semit);
    be.scan(d_bases, nrec, d_sbases);
    be.scan(d_nameb, nrec, d_snameb);
    be.scan(d_pe, nrec, d_spe);
    {
        const uint32_t *fbase = d_fbase, *semit = d_semit, *sbases = d_sbases, *snameb = d_snameb, *spe = d_spe;
        const int32_t *ffirst = d_ffirst;
        ProblemSummary *psum = d_psum;
        be.template for_each<SummaryTag>(nq, [=] __host__ __device__(int64_t p) {
            const uint32_t r0 = fbase[ffirst[p]], r1 = fbase[ffirst[p + 1]];
            ProblemSummary s;
            s.read0 = semit[r0]; s.nreads = semit[r1] - semit[r0];
            s.base0 = sbases[r0]; s.nbases = sbases[r1] - sbases[r0];
            s.name0 = snameb[r0]; s.name_bytes = snameb[r1] - snameb[r0];
            s.pe0 = spe[r0]; s.npe = spe[r1] - spe[r0];
            psum[p] = s;
        });
    }
    be.download(h_psum, d_psum, sizeof(ProblemSummary) * (size_t)nq);
    be.download(h_counts, d_counts, sizeof(ProblemCounts) * (size_t)nq);
    be.sync();                                                                                  // sync 2
    out->ms_marks[1] = now_ms() - t_begin;
    if (be.rc) return be.rc;
    const int64_t nreads = (int64_t)h_psum[nq - 1].read0 + h_psum[nq - 1].nreads;
    const int64_t nbases = (int64_t)h_psum[nq - 1].base0 + h_psum[nq - 1].nbases;
    const int64_t name_bytes = (int64_t)h_psum[nq - 1].name0 + h_psum[nq - 1].name_bytes;
    const int64_t npe = (int64_t)h_psum[nq - 1].pe0 + h_psum[nq - 1].npe;
    {
        // the scans are 32-bit: a batch whose selected bytes do not fit them (only a corrupt file gets there) is refused
        unsigned long long total64 = 0;
        for (int p = 0; p < nq; ++p) total64 += h_counts[p].bytes64;
        if (total64 != (unsigned long long)nbases + (unsigned long long)name_bytes || total64 >= (1ull << 31)) {
            tredsw_set_error("implausible amount of selected read data (%llu bytes): corrupt input?", total64);
            return TREDSW_ERR_IO;
        }
    }
    // per-problem pairing tables (power-of-two slots, load <= 1/2)
    std::vector<uint32_t> tab_off(nq + 1, 0), tab_mask(nq, 0);
    for (int p = 0; p < nq; ++p) {
        uint32_t sz = 8;
        while (sz < 2u * h_psum[p].npe) sz <<= 1;
        if (h_psum[p].npe == 0) sz = 0;
        tab_mask[p] = sz ? sz - 1 : 0;
        tab_off[p + 1] = tab_off[p] + sz;
        if (h_counts[p].error && !out->status[p]) out->status[p] = PROBLEM_CORRUPT;
    }
    const int64_t nslots = tab_off[nq];
    int8_t *d_rbuf = alloc_n<int8_t>(be, nbases + 16, true);
    int64_t *d_roff = alloc_n<int64_t>(be, nreads + 1, true);
    int32_t *d_rprob = alloc_n<int32_t>(be, nreads, true);
    char *d_names = want_names ? alloc_n<char>(be, name_bytes + 16) : nullptr;
    uint32_t *d_elist = alloc_n<uint32_t>(be, nreads);
    uint32_t *d_plist = alloc_n<uint32_t>(be, npe);
    uint32_t *d_tab = alloc_n<uint32_t>(be, 3 * std::max<int64_t>(1, nslots));     // rep, first, second
    uint32_t *d_taboff = alloc_n<uint32_t>(be, nq + 1);
    uint32_t *d_tabmask = alloc_n<uint32_t>(be, nq);
    uint32_t *d_slot = alloc_n<uint32_t>(be, npe);
    uint32_t *d_isg = alloc_n<uint32_t>(be, npe + 1);
    uint32_t *d_ist = alloc_n<uint32_t>(be, npe + 1);
    int32_t *d_pval = alloc_n<int32_t>(be, npe);
    uint32_t *d_sg = alloc_n<uint32_t>(be, npe + 2);
    uint32_t *d_st = alloc_n<uint32_t>(be, npe + 2);
    uint32_t *d_pcnt = alloc_n<uint32_t>(be, 2 * (int64_t)nq);
    uint32_t *h_pcnt = alloc_host_n<uint32_t>(be, 2 * (int64_t)nq);
    if (be.rc) return be.rc;
    be.upload(d_taboff, tab_off.data(), sizeof(uint32_t) * (size_t)(nq + 1));
    be.upload(d_tabmask, tab_mask.data(), sizeof(uint32_t) * (size_t)nq);
    be.fill(d_tab, 0xff, sizeof(uint32_t) * 3 * (size_t)nslots);
    be.fill(d_roff, 0, sizeof(int64_t));
    {
        // ---- (6) ordered compaction + scatter of the selected reads ------------------------------------------------
        const uint8_t *ibuf = d_ibuf; const Fetch *fe = d_fetches;
        const int64_t *rpos = d_rpos; const int32_t *rfetch = d_rfetch;
        const uint32_t *emit = d_emit, *bases = d_bases, *pe = d_pe, *semit = d_semit, *sbases = d_sbases, *snameb = d_snameb, *spe = d_spe;
        uint32_t *elist = d_elist, *plist = d_plist;
        int64_t *roff = d_roff; int32_t *rprob = d_rprob;
        be.template for_each<CompactTag>(nrec, [=] __host__ __device__(int64_t i) {
            if (emit[i]) {
                const uint32_t k = semit[i];
                elist[k] = (uint32_t)i;
                roff[k + 1] = (int64_t)sbases[i] + bases[i];
                rprob[k] = fe[rfetch[i]].problem;
            }
            if (pe[i]) plist[spe[i]] = (uint32_t)i;
        });
        int8_t *rbuf = d_rbuf; char *names = d_names;
        be.template for_each_warp<EmitTag>(nreads, [=] __host__ __device__(int64_t k, int lane) {
            const uint32_t i = elist[k];
            emit_read(ibuf, rpos[i], rbuf + sbases[i], names ? names + snameb[i] : nullptr, lane, B::on_device ? 32 : 1);
        });
        // ---- (7) pairing by name ---------------------------------------------------------------------------------------
        const ProblemParams *pp = d_params;
        const uint32_t *taboff = d_taboff, *tabmask = d_tabmask;
        uint32_t *rep = d_tab, *first = d_tab + nslots, *second = d_tab + 2 * nslots, *slot = d_slot;
        be.template for_each<PairInsertTag>(npe, [=] __host__ __device__(int64_t k) {
            const uint32_t i = plist[k];
            const int p = fe[rfetch[i]].problem;
            slot[k] = taboff[p] + pair_insert(ibuf, rpos, i, rep + taboff[p], first + taboff[p], tabmask[p]);
        });
        be.template for_each<PairSecondTag>(npe, [=] __host__ __device__(int64_t k) {
            const uint32_t i = plist[k], s = slot[k];
            if (first[s] != i) atomic_min_u32(&second[s], i);
        });
        const Mate *mates = d_mates;
        uint32_t *isg = d_isg, *ist = d_ist; int32_t *pval = d_pval;
        be.template for_each<PairEvalTag>(npe, [=] __host__ __device__(int64_t k) {
            const uint32_t i = plist[k], s = slot[k];
            int kind = 0; int32_t tlen = 0;
            if (first[s] == i && second[s] != EMPTY) kind = pair_eval(mates[i], mates[second[s]], pp[fe[rfetch[i]].problem], &tlen);
            isg[k] = kind == 1; ist[k] = kind == 2; pval[k] = tlen;
        });
    }
    be.scan(d_isg, npe, d_sg);
    be.scan(d_ist, npe, d_st);
    {
        const ProblemSummary *psum = d_psum; const uint32_t *sg = d_sg, *st = d_st; uint32_t *pcnt = d_pcnt;
        be.template for_each<PairCountTag>(nq, [=] __host__ __device__(int64_t p) {
            const uint32_t a = psum[p].pe0, b = a + psum[p].npe;
            pcnt[2 * p] = sg[b] - sg[a]; pcnt[2 * p + 1] = st[b] - st[a];
        });
    }
    be.download(h_pcnt, d_pcnt, sizeof(uint32_t) * 2 * (size_t)nq);
    be.sync();                                                                                  // sync 3
    out->ms_marks[2] = now_ms() - t_begin;
    if (be.rc) return be.rc;
    std::vector<int64_t> pe_off(2 * (size_t)nq);
    int64_t n_pe_lens = 0;
    for (int p = 0; p < nq; ++p) {
        pe_off[2 * p] = n_pe_lens; n_pe_lens += h_pcnt[2 * p];
        pe_off[2 * p + 1] = n_pe_lens; n_pe_lens += h_pcnt[2 * p + 1];
    }
    int32_t *d_pelens = alloc_n<int32_t>(be, n_pe_lens, true);
    int64_t *d_peoff = alloc_n<int64_t>(be, 2 * (int64_t)nq);
    int8_t *h_rbuf = alloc_host_n<int8_t>(be, nbases + 16, true);
    int64_t *h_roff = alloc_host_n<int64_t>(be, nreads + 1, true);
    int32_t *h_pelens = alloc_host_n<int32_t>(be, n_pe_lens, true);
    char *h_names = want_names ? alloc_host_n<char>(be, name_bytes + 16, true) : nullptr;
    if (be.rc) return be.rc;
    be.upload(d_peoff, pe_off.data(), sizeof(int64_t) * 2 * (size_t)nq);
    {
        const Fetch *fe = d_fetches; const int32_t *rfetch = d_rfetch; const uint32_t *plist = d_plist;
        const ProblemSummary *psum = d_psum;
        const uint32_t *isg = d_isg, *ist = d_ist, *sg = d_sg, *st = d_st; const int32_t *pval = d_pval;
        const int64_t *peoff = d_peoff; int32_t *pelens = d_pelens;
        be.template for_each<PairScatterTag>(npe, [=] __host__ __device__(int64_t k) {
            const int p = fe[rfetch[plist[k]]].problem;
            const uint32_t a = psum[p].pe0;
            if (isg[k]) pelens[peoff[2 * p] + (sg[k] - sg[a])] = pval[k];
            if (ist[k]) pelens[peoff[2 * p + 1] + (st[k] - st[a])] = pval[k];
        });
    }
    be.download(h_rbuf, d_rbuf, (size_t)nbases);
    be.download(h_roff, d_roff, sizeof(int64_t) * (size_t)(nreads + 1));
    be.download(h_pelens, d_pelens, sizeof(int32_t) * (size_t)n_pe_lens);
    if (want_names) be.download(h_names, d_names, (size_t)name_bytes);
    be.sync();                                                                                  // sync 4
    out->ms_marks[3] = now_ms() - t_begin;
    if (be.rc) return be.rc;

    for (int p = 0; p < nq; ++p) {
        tredsw_locus_summary &s = out->summaries[p];
        tredsw_problem_span &sp = out->spans[p];
        s.nreads = (int32_t)h_psum[p].nreads; s.nbases = h_psum[p].nbases; s.name_bytes = h_psum[p].name_bytes;
        s.n_unmapped = h_counts[p].n_unmapped;
        s.n_global = (int32_t)h_pcnt[2 * p]; s.n_target = (int32_t)h_pcnt[2 * p + 1];
        s.depth = (double)h_counts[p].depth_sum * 1.0 / (double)(params[p].win_e - params[p].win_s + 1);
        s.overflow = 0;
        sp.read0 = h_psum[p].read0; sp.base0 = h_psum[p].base0; sp.name0 = h_psum[p].name0;
        sp.off_global = pe_off[2 * p]; sp.off_target = pe_off[2 * p + 1];
        if (out->status[p]) { s.depth = 0; }
    }
    tredsw_ingest_view &v = out->view;
    v.nproblems = nq; v.nreads = (int32_t)nreads; v.nbases = nbases; v.name_bytes = want_names ? name_bytes : 0; v.n_pe_lens = n_pe_lens;
    v.d_rbuf = d_rbuf; v.d_roff = d_roff; v.d_read_problem = d_rprob; v.d_pe_lens = d_pelens;
    v.h_rbuf = h_rbuf; v.h_roff = h_roff; v.h_pe_lens = h_pelens; v.h_names = h_names;
    v.summaries = out->summaries.data(); v.spans = out->spans.data(); v.status = out->status.data();
    v.n_blocks = out->n_blocks; v.n_records = out->n_records; v.comp_bytes = out->comp_bytes; v.inflated_bytes = out->inflated_bytes;
    be.release_intermediates();            // compressed bytes, inflated stream, record arrays, tables: only results stay
    out->ms_total = now_ms() - t_begin;
    v.ms_host_stage = out->ms_host_stage; v.ms_total = out->ms_total;
    for (int k = 0; k < 4; ++k) v.ms_marks[k] = out->ms_marks[k];
    return TREDSW_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// the scan of a BAM without an index: one streaming pass per sample (ingest_device.cuh: record boundaries, matching)
// ---------------------------------------------------------------------------------------------------------------
namespace {

constexpr int64_t SCAN_DEFAULT_SLAB = 128ll << 20;     // compressed bytes per slab when the caller passes 0
constexpr int64_t SCAN_MIN_SLAB = 65536;               // a slab holds at least one whole BGZF block
constexpr int64_t SCAN_MAX_INFLATED = 1ll << 30;       // inflated bytes per slab: its record offsets are scanned in 32 bits

struct ScanSlab {                   // the compressed bytes of one slab (page-locked) and their BGZF framing
    uint8_t *comp = nullptr;
    std::vector<BlockDesc> blocks;  // in_off into comp, out_off from the slab's first inflated byte
    int64_t begin = 0, next = 0, inflated = 0;
    int64_t got = 0;                // bytes in comp (the whole blocks end at next - begin)
    const char *why = nullptr;      // I/O or framing error
    double ms = 0;                  // host time: read + framing
};

// Where the slabs come from.  A file is read with pread at absolute offsets; its size caps the slab and tells a block
// cut by the end of the file.  A stream is read strictly in order with read(), its size unknown: a slab starts with the
// bytes the slab before it read past its last whole block (the first slab: what the handle buffered while it read the
// header and the read length), and the end of the input is read() returning 0.
struct ScanSource {
    int fd = -1;
    bool stream = false;
    int64_t file_size = 0;                  // file
    bool eof = false;                       // stream: read() returned 0
    const uint8_t *head = nullptr;          // stream: the first slab's leading bytes
    int64_t head_len = 0;
};

// Reads up to `want` bytes from `off` and frames the whole blocks among them.  A block cut by the end of the read is
// left to the next slab (`next` is its offset); one cut by the end of the input is an error.  prev: the slab before
// (a stream's next slab starts with its unframed tail).
void read_slab(ScanSource *src, int64_t off, int64_t want, const ScanSlab *prev, ScanSlab *sl) {
    const double t0 = now_ms();
    sl->blocks.clear(); sl->begin = sl->next = off; sl->inflated = 0; sl->why = nullptr;
    int64_t got = 0;
    if (!src->stream) {
        const int64_t n = std::max<int64_t>(0, std::min(want, src->file_size - off));
        got = pread_full(src->fd, sl->comp, n, off);
        if (got < n) sl->why = "short read";
    } else {
        const uint8_t *lead = prev ? prev->comp + (prev->next - prev->begin) : src->head;
        got = prev ? prev->got - (prev->next - prev->begin) : src->head_len;
        if (got > 0) memcpy(sl->comp, lead, (size_t)got);
        while (got < want && !src->eof) {
            const ssize_t k = read(src->fd, sl->comp + got, (size_t)(want - got));
            if (k > 0) got += k;
            else if (k == 0) src->eof = true;
            else if (errno != EINTR) { sl->why = "read failed"; break; }
        }
    }
    sl->got = got;
    const bool at_end = src->stream ? src->eof : off + got >= src->file_size;
    int64_t o = 0;
    while (!sl->why && o < got) {
        BgzfFrame fr;
        const char *why = nullptr;
        const int rc = parse_bgzf_block(sl->comp + o, got - o, &fr, &why);
        if (rc < 0 || (rc == 0 && at_end)) { sl->why = why; break; }
        if (rc == 0 || (sl->inflated + fr.isize > SCAN_MAX_INFLATED && !sl->blocks.empty())) break;
        sl->blocks.push_back(block_desc(fr, o, sl->inflated));
        sl->inflated += fr.isize;
        o += fr.bsize;
    }
    sl->next = off + o;
    sl->ms = now_ms() - t0;
}

struct ScanBuffers {                // the device buffers of the slab loop, reused from slab to slab
    Reused<uint8_t> ibuf[2];        // the carry + the slab's inflated blocks (alternating: the carry is copied across)
    Reused<uint8_t> comp, bstatus;
    Reused<BlockDesc> blocks;
    Reused<ScanBlock> sblk;
    Reused<int64_t> cand, land, first, recpos, epos;
    Reused<uint32_t> rcnt, rbase, nm, kb, ebase, kbase;
    Reused<int32_t> efetch;
    Reused<uint32_t> iflag, inb, ibase, inbase;     // the STR profile
    Reused<IrrEntry> ient;
    Reused<char> iname;
    Reused<uint8_t> kept;           // the kept-record stream of the whole scan (grows with its contents)
};

}  // namespace

namespace { void irr_join(tredsw_ingest_batch *out, const unsigned long long *st); }

// Verification and repair of a slab's record starts (DESIGN §4.4.1): h_first[b], the true first record of block b,
// from the known start s0 of block 0.  Returns the next carry's start, or SCAN_BAD (corrupt records); *repaired counts
// the blocks walked again.  The result means nothing after a backend error (be.rc).
template <class B>
int64_t verify_record_starts(B &be, uint8_t *s, int64_t len, ScanBlock *blk, int64_t *cand, int64_t *land, int64_t *stop,
                             const std::vector<ScanBlock> &sblk, const std::vector<int64_t> &h_cand,
                             std::vector<int64_t> &h_land, std::vector<int64_t> &h_first, int64_t s0, int64_t *repaired) {
    const int nb = (int)sblk.size();
    int64_t tf = s0;
    for (int b = 0; b < nb && tf != SCAN_BAD;) {
        h_first[b] = tf;
        if (scan_agrees(sblk[b], h_cand[b], tf)) {
            if (tf >= sblk[b].begin && tf < sblk[b].end) tf = h_land[b];
            ++b;
            continue;
        }
        const int b0 = b; const int64_t t0 = tf;
        be.template for_each<ScanRepairTag>(1, [=] __host__ __device__(int64_t) { *stop = scan_repair_run(s, len, blk, cand, nb, b0, t0, land); });
        int64_t h_stop = 0;
        be.download(&h_stop, stop, sizeof(int64_t));
        be.sync();
        if (be.rc) return SCAN_BAD;
        be.download(h_land.data() + b0, land + b0, sizeof(int64_t) * (size_t)(h_stop - b0));
        be.sync();
        for (int k = b0 + 1; k < (int)h_stop; ++k) h_first[k] = h_land[k - 1];
        *repaired += h_stop - b0;
        tf = h_land[h_stop - 1];
        b = (int)h_stop;
    }
    return tf;
}

template <class B>
int run_scan(B &be, tredsw_ingest_batch *out, tredsw_bam *bam, const tredsw_locus_query *queries, int32_t nq,
             const int32_t *depth_regions, int32_t n_depth, double *depth_out, int64_t slab_bytes, uint32_t flags,
             const tredsw_irr_params *irr) {
    const double t_begin = now_ms();
    const bool want_names = (flags & TREDSW_INGEST_NO_NAMES) == 0;
    const int check_crc = (flags & TREDSW_INGEST_NO_CRC) == 0;
    constexpr int NL = B::on_device ? 32 : 1;
    out->reset(nq);
    const int32_t n_ref = (int32_t)bam->names.size();

    // ---- (1) the fetches (problem-major, like run_pipeline), then the depth regions; their elementary segments -----
    std::vector<ProblemParams> params(nq);
    std::vector<Fetch> fetches;
    std::vector<int32_t> fetch_first(nq + 1, 0);
    std::vector<int32_t> id_tid;
    std::vector<int64_t> id_start, id_end;
    auto add_id = [&](int32_t tid, int64_t s, int64_t e) { id_tid.push_back(tid); id_start.push_back(s < 0 ? 0 : s); id_end.push_back(e); };
    for (int p = 0; p < nq; ++p) {
        fetch_first[p] = (int32_t)fetches.size();
        const bool planned = plan_fetches(queries[p], n_ref, &params[p], [&](int kind, int32_t tid, int64_t s, int64_t e) {
            Fetch f;
            f.problem = p; f.kind = kind; f.tid = tid; f.start = s; f.end = e;
            f.chunk_begin = f.chunk_end = 0; f.pad_ = 0;
            fetches.push_back(f);
            add_id(tid, s, e);
        });
        if (!planned) out->status[p] = PROBLEM_STAGING;
    }
    fetch_first[nq] = (int32_t)fetches.size();
    const int32_t nfetch = (int32_t)fetches.size();
    for (int d = 0; d < n_depth; ++d) {
        const int32_t tid = depth_regions[3 * d], s = depth_regions[3 * d + 1], e = depth_regions[3 * d + 2];
        if (tid < 0 || tid >= n_ref) { tredsw_set_error("depth region %d: contig id %d out of range", d, tid); return TREDSW_ERR_ARG; }
        if (e < s) { tredsw_set_error("depth region %d is empty", d); return TREDSW_ERR_ARG; }
        add_id(tid, s, e);
    }
    const int nids = (int)id_tid.size();
    std::vector<int32_t> tid_x0(n_ref + 1, 0), seg_f0, seg_ids;
    std::vector<int64_t> xs, id_lo(nids), id_hi(nids);
    for (int i = 0; i < nids; ++i) {                        // the interval every fetch is listed on (MatchTables)
        id_lo[i] = id_start[i] < id_end[i] ? id_start[i] : id_end[i] - 1;
        id_hi[i] = id_start[i] < id_end[i] ? id_end[i] : id_end[i];
    }
    {
        std::vector<std::vector<int64_t>> pts(n_ref);
        for (int i = 0; i < nids; ++i) { pts[id_tid[i]].push_back(id_lo[i]); pts[id_tid[i]].push_back(id_hi[i]); }
        for (int t = 0; t < n_ref; ++t) {
            std::sort(pts[t].begin(), pts[t].end());
            pts[t].erase(std::unique(pts[t].begin(), pts[t].end()), pts[t].end());
            tid_x0[t] = (int32_t)xs.size();
            xs.insert(xs.end(), pts[t].begin(), pts[t].end());
        }
        tid_x0[n_ref] = (int32_t)xs.size();
        std::vector<std::vector<int32_t>> lists(xs.size());
        for (int i = 0; i < nids; ++i) {
            const auto b0 = xs.begin() + tid_x0[id_tid[i]], b1 = xs.begin() + tid_x0[id_tid[i] + 1];
            const int j0 = (int)(std::lower_bound(b0, b1, id_lo[i]) - xs.begin()), j1 = (int)(std::lower_bound(b0, b1, id_hi[i]) - xs.begin());
            for (int j = j0; j < j1; ++j) lists[j].push_back(i);
        }
        seg_f0.assign(xs.size() + 1, 0);
        for (size_t j = 0; j < xs.size(); ++j) { seg_f0[j + 1] = seg_f0[j] + (int32_t)lists[j].size(); seg_ids.insert(seg_ids.end(), lists[j].begin(), lists[j].end()); }
    }
    int32_t *d_tid_x0 = alloc_n<int32_t>(be, n_ref + 1);
    int64_t *d_xs = alloc_n<int64_t>(be, (int64_t)xs.size());
    int32_t *d_seg_f0 = alloc_n<int32_t>(be, (int64_t)seg_f0.size());
    int32_t *d_seg_ids = alloc_n<int32_t>(be, (int64_t)seg_ids.size());
    int64_t *d_id_start = alloc_n<int64_t>(be, 3 * (int64_t)std::max(1, nids));     // start, end, lo
    unsigned long long *d_depth = alloc_n<unsigned long long>(be, n_depth);
    uint32_t *d_err = alloc_n<uint32_t>(be, 2);
    int64_t *d_small = alloc_n<int64_t>(be, 2);     // last record's order key; repair stop
    // the STR profile: counters over the whole scan; per slab the IRR flags / name bytes, their scans, the entries
    out->irr_on = irr != nullptr;
    const IrrParams ip = irr ? IrrParams{irr->min_period, irr->max_period, irr->purity_num, irr->purity_den, irr->min_read_len}
                             : IrrParams{0, 0, 0, 1, 0};
    unsigned long long *d_irr_stats = irr ? alloc_n<unsigned long long>(be, IRR_NSTATS) : nullptr;
    if (be.rc) return be.rc;
    if (irr) be.fill(d_irr_stats, 0, sizeof(unsigned long long) * IRR_NSTATS);
    be.upload(d_tid_x0, tid_x0.data(), sizeof(int32_t) * tid_x0.size());
    be.upload(d_xs, xs.data(), sizeof(int64_t) * xs.size());
    be.upload(d_seg_f0, seg_f0.data(), sizeof(int32_t) * seg_f0.size());
    be.upload(d_seg_ids, seg_ids.data(), sizeof(int32_t) * seg_ids.size());
    be.upload(d_id_start, id_start.data(), sizeof(int64_t) * (size_t)nids);
    be.upload(d_id_start + nids, id_end.data(), sizeof(int64_t) * (size_t)nids);
    be.upload(d_id_start + 2 * nids, id_lo.data(), sizeof(int64_t) * (size_t)nids);
    be.fill(d_depth, 0, sizeof(unsigned long long) * (size_t)std::max(1, n_depth));
    be.fill(d_err, 0, sizeof(uint32_t) * 2);
    const MatchTables mt{d_tid_x0, d_xs, d_seg_f0, d_seg_ids, d_id_start + 2 * nids, d_id_start, d_id_start + nids, n_ref, nfetch};

    // ---- (2) slab by slab: read (the next slab on a host thread), inflate, record boundaries, match, keep ------------
    ScanSource src;
    int64_t want;
    if (!bam->is_stream()) {
        src.fd = fileno(bam->bgzf.fh);
        struct stat st;
        src.file_size = fstat(src.fd, &st) == 0 ? (int64_t)st.st_size : 0;
        want = std::max(std::min(slab_bytes > 0 ? slab_bytes : SCAN_DEFAULT_SLAB, src.file_size), SCAN_MIN_SLAB);
    } else {
        tredsw_bam::Bgzf &z = bam->bgzf;
        const int64_t at = (int64_t)(bam->first_record >> 16) - z.sbase;
        src.fd = z.sfd; src.stream = true; src.eof = z.seof;
        src.head = z.sbuf.data() + at; src.head_len = (int64_t)z.sbuf.size() - at;
        want = std::max({slab_bytes > 0 ? slab_bytes : SCAN_DEFAULT_SLAB, SCAN_MIN_SLAB, src.head_len});
    }
    ScanSlab slabs[2];
    for (ScanSlab &sl : slabs) sl.comp = alloc_host_n<uint8_t>(be, want + 64);
    if (be.rc) return be.rc;
    ScanBuffers buf;
    std::vector<int32_t> ent_fetch;         // (record, fetch) entries of the whole file, in file order
    std::vector<int64_t> ent_pos;           // where the record is in the kept-record stream
    int64_t kept_total = 0, carry_len = 0, carry_at = 0, prev_key = INT64_MIN;
    int64_t s0 = (int64_t)(bam->first_record & 0xffff);
    int32_t status = PROBLEM_OK;
    int64_t *stats = out->scan_stats;
    ReadAhead reader;
    bam->consumed = bam->is_stream();
    read_slab(&src, (int64_t)(bam->first_record >> 16), want, nullptr, &slabs[0]);
    if (src.stream) { bam->bgzf.sbuf = std::vector<unsigned char>(); src.head = nullptr; }
    for (int cur = 0;; cur ^= 1) {
        ScanSlab &sl = slabs[cur];
        stats[6] += (int64_t)(sl.ms * 1e3);
        if (sl.why) { status = PROBLEM_STAGING; tredsw_set_error("%s: %s", bam->path.c_str(), sl.why); break; }
        const int nb = (int)sl.blocks.size();
        if (nb == 0) break;                                                  // end of file
        const bool more = src.stream ? !(src.eof && sl.next == sl.begin + sl.got) : sl.next < src.file_size;
        if (more) reader.start(read_slab, &src, sl.next, want, &slabs[cur], &slabs[cur ^ 1]);
        else { slabs[cur ^ 1].blocks.clear(); slabs[cur ^ 1].why = nullptr; slabs[cur ^ 1].ms = 0; }
        const double t_dev = now_ms();
        const int64_t len = carry_len + sl.inflated;
        uint8_t *s = buf.ibuf[cur].get(be, len + 64);
        if (be.rc) return be.rc;
        be.copy(s, buf.ibuf[cur ^ 1].p + carry_at, (size_t)carry_len);
        std::vector<ScanBlock> sblk(nb);
        for (int b = 0; b < nb; ++b) {
            sl.blocks[b].out_off += carry_len;
            sblk[b].begin = b ? sl.blocks[b].out_off : 0;
            sblk[b].end = sl.blocks[b].out_off + sl.blocks[b].isize;
        }
        // inflate; candidates and landings
        uint8_t *comp = buf.comp.get(be, sl.next - sl.begin + 64);
        BlockDesc *blocks = buf.blocks.get(be, nb);
        uint8_t *bstatus = buf.bstatus.get(be, nb);
        ScanBlock *blk = buf.sblk.get(be, nb);
        int64_t *cand = buf.cand.get(be, nb);
        int64_t *land = buf.land.get(be, nb);
        if (be.rc) return be.rc;
        be.upload(comp, sl.comp, (size_t)(sl.next - sl.begin));
        be.upload(blocks, sl.blocks.data(), sizeof(BlockDesc) * nb);
        be.upload(blk, sblk.data(), sizeof(ScanBlock) * nb);
        be.inflate(comp, s, blocks, nb, bstatus, check_crc);
        {
            const int64_t first0 = s0;
            be.template for_each_warp<ScanCandidateTag>(nb, [=] __host__ __device__(int64_t b, int lane) {
                const int64_t c = b == 0 ? first0 : scan_find_candidate<NL>(s, len, blk[b].begin, blk[b].end, n_ref, lane);
                if (lane == 0) { cand[b] = c; land[b] = c < 0 ? c : scan_chain(s, len, c, blk[b].end); }
            });
        }
        std::vector<uint8_t> h_bstatus(nb);
        std::vector<int64_t> h_cand(nb), h_land(nb), h_first(nb);
        be.download(h_bstatus.data(), bstatus, (size_t)nb);
        be.download(h_cand.data(), cand, sizeof(int64_t) * nb);
        be.download(h_land.data(), land, sizeof(int64_t) * nb);
        be.sync();
        if (be.rc) return be.rc;
        if (std::any_of(h_bstatus.begin(), h_bstatus.end(), [](uint8_t v) { return v != 0; })) { status = PROBLEM_INFLATE; tredsw_set_error("%s: a BGZF block failed to inflate", bam->path.c_str()); break; }
        const int64_t tf = verify_record_starts(be, s, len, blk, cand, land, d_small + 1, sblk, h_cand, h_land, h_first, s0, &stats[3]);
        if (be.rc) return be.rc;
        if (tf == SCAN_BAD) { status = PROBLEM_CORRUPT; tredsw_set_error("%s: corrupt BAM records (implausible block_size)", bam->path.c_str()); break; }
        // the records that start in every block, in file order
        int64_t *first = buf.first.get(be, nb);
        uint32_t *rcnt = buf.rcnt.get(be, nb + 1);
        uint32_t *rbase = buf.rbase.get(be, nb + 2);
        if (be.rc) return be.rc;
        be.upload(first, h_first.data(), sizeof(int64_t) * nb);
        be.template for_each<ScanCountTag>(nb, [=] __host__ __device__(int64_t b) {
            uint32_t n = 0;
            scan_block_records(s, len, first[b], blk[b].end, [&](int64_t) { ++n; });
            rcnt[b] = n;
        });
        be.scan(rcnt, nb, rbase);
        uint32_t h_nrec = 0;
        be.download(&h_nrec, rbase + nb, sizeof(uint32_t));
        be.sync();
        if (be.rc) return be.rc;
        const int64_t nrec = h_nrec;
        int64_t *recpos = buf.recpos.get(be, nrec);
        uint32_t *nm = buf.nm.get(be, nrec + 1);
        uint32_t *kb = buf.kb.get(be, nrec + 1);
        uint32_t *ebase = buf.ebase.get(be, nrec + 2);
        uint32_t *kbase = buf.kbase.get(be, nrec + 2);
        if (be.rc) return be.rc;
        {
            const int64_t pk = prev_key;
            int64_t *last = d_small;
            uint32_t *err = d_err;
            unsigned long long *depth = d_depth;
            be.template for_each<ScanFillTag>(nb, [=] __host__ __device__(int64_t b) {
                uint32_t k = rbase[b];
                scan_block_records(s, len, first[b], blk[b].end, [&](int64_t p) { recpos[k++] = p; });
            });
            be.template for_each<ScanMatchTag>(nrec, [=] __host__ __device__(int64_t i) {
                const uint32_t n = scan_record(s, recpos, i, pk, mt, depth, err);
                nm[i] = n;
                kb[i] = n ? 4u + (uint32_t)ld_i32(s, recpos[i]) : 0u;
                if (i == nrec - 1) *last = order_key(ld_i32(s, recpos[i] + 4), ld_i32(s, recpos[i] + 8));
            });
        }
        be.scan(nm, nrec, ebase);
        be.scan(kb, nrec, kbase);
        // the profile: classify every record (one thread each), IRR flags and name bytes -> their exclusive scans
        uint32_t *iflag = nullptr, *inb = nullptr, *ibase = nullptr, *inbase = nullptr;
        uint32_t h_itot[2] = {0, 0};
        if (irr) {
            iflag = buf.iflag.get(be, nrec + 1);
            inb = buf.inb.get(be, nrec + 1);
            ibase = buf.ibase.get(be, nrec + 2);
            inbase = buf.inbase.get(be, nrec + 2);
            if (be.rc) return be.rc;
            unsigned long long *ist = d_irr_stats;
            be.template for_each<ScanIrrTag>(nrec, [=] __host__ __device__(int64_t i) {
                uint64_t motif; RecFields r;
                const int per = scan_irr_record(s, recpos[i], ip, ist, &motif, &r);
                iflag[i] = per ? 1u : 0u;
                inb[i] = per && r.l_name > 1 ? (uint32_t)(r.l_name - 1) : 0u;
            });
            be.scan(iflag, nrec, ibase);
            be.scan(inb, nrec, inbase);
            be.download(&h_itot[0], ibase + nrec, sizeof(uint32_t));
            be.download(&h_itot[1], inbase + nrec, sizeof(uint32_t));
        }
        uint32_t h_tot[2] = {0, 0}, h_err = 0;
        int64_t h_last = prev_key;
        be.download(&h_tot[0], ebase + nrec, sizeof(uint32_t));
        be.download(&h_tot[1], kbase + nrec, sizeof(uint32_t));
        be.download(&h_err, d_err, sizeof(uint32_t));
        if (nrec) be.download(&h_last, d_small, sizeof(int64_t));
        be.sync();
        if (be.rc) return be.rc;
        if (h_err & SCAN_ERR_RECORD) { status = PROBLEM_CORRUPT; tredsw_set_error("%s: corrupt BAM record", bam->path.c_str()); break; }
        if (h_err & SCAN_ERR_ORDER) { status = PROBLEM_UNSORTED; tredsw_set_error("%s is not sorted by coordinate", bam->path.c_str()); break; }
        // the slab's IRR entries and names, appended to the host lists (IRRs are rare: the join by name is host work)
        if (h_itot[0]) {
            const int64_t nirr = h_itot[0], nnb = h_itot[1];
            IrrEntry *ient = buf.ient.get(be, nirr);
            char *iname = buf.iname.get(be, nnb + 1);
            if (be.rc) return be.rc;
            unsigned long long *ist = d_irr_stats;
            be.template for_each<ScanIrrFillTag>(nrec, [=] __host__ __device__(int64_t i) {
                if (!iflag[i]) return;
                const int64_t p = recpos[i];
                const RecFields r = parse_record(s, p);
                IrrEntry e;
                e.period = irr_classify(PackedSeq{s + record_seq(p, r)}, r.l_seq, ip, &e.motif);
                bool unparsed;
                e.mq = aux_mq(s, record_aux(p, r), p + 4 + (int64_t)ld_i32(s, p), &unparsed);
                if (unparsed) atomic_add_u64(&ist[IRR_UNPARSED_AUX], 1ull);
                e.tid = r.tid; e.pos = r.pos; e.next_tid = r.next_tid; e.next_pos = r.next_pos;
                e.flag = r.flag; e.mapq = s[p + 13];
                e.name_off = inbase[i]; e.name_len = (int32_t)inb[i]; e.mate = -1;
                ient[ibase[i]] = e;
                for (uint32_t k = 0; k < inb[i]; ++k) iname[inbase[i] + k] = (char)s[p + 36 + k];
            });
            const size_t e0 = out->irr_entries.size(), n0 = out->irr_names.size();
            out->irr_entries.resize(e0 + (size_t)nirr);
            out->irr_names.resize(n0 + (size_t)nnb);
            be.download(out->irr_entries.data() + e0, ient, sizeof(IrrEntry) * (size_t)nirr);
            be.download(out->irr_names.data() + n0, iname, (size_t)nnb);
            be.sync();
            if (be.rc) return be.rc;
            for (size_t k = e0; k < out->irr_entries.size(); ++k) out->irr_entries[k].name_off += (int64_t)n0;
        }
        // copy the kept records once into the kept-record stream; one (fetch, position) entry per (record, fetch)
        const int64_t nent = h_tot[0], kbytes = h_tot[1];
        if (nent) {
            uint8_t *kept = buf.kept.get_keeping(be, kept_total + kbytes + 64, kept_total) + kept_total;
            int32_t *efetch = buf.efetch.get(be, nent);
            int64_t *epos = buf.epos.get(be, nent);
            if (be.rc) return be.rc;
            const int64_t k0 = kept_total;
            be.template for_each_warp<ScanKeepTag>(nrec, [=] __host__ __device__(int64_t i, int lane) {
                if (!nm[i]) return;
                const int64_t p = recpos[i];
                const uint32_t nbytes = kb[i], at = kbase[i];
                for (uint32_t k = (uint32_t)lane; k < nbytes; k += NL) kept[at + k] = s[p + k];
                if (lane) return;
                const RecFields r = parse_record(s, p);
                uint32_t e = ebase[i];
                scan_matches(mt, r.tid, r.pos, record_fetch_end(r), [&](int32_t id) {
                    if (id < mt.nfetch) { efetch[e] = id; epos[e] = k0 + at; ++e; }
                });
            });
            const size_t e0 = ent_fetch.size();
            ent_fetch.resize(e0 + nent); ent_pos.resize(e0 + nent);
            be.download(ent_fetch.data() + e0, efetch, sizeof(int32_t) * (size_t)nent);
            be.download(ent_pos.data() + e0, epos, sizeof(int64_t) * (size_t)nent);
            be.sync();
            if (be.rc) return be.rc;
            kept_total += kbytes;
        }
        prev_key = h_last;
        carry_at = tf; carry_len = len - tf; s0 = 0;
        stats[0] += 1; stats[1] += nb; stats[2] += nrec;
        stats[4] += sl.next - sl.begin; stats[5] += sl.inflated;
        stats[7] += (int64_t)((now_ms() - t_dev) * 1e3);
        reader.join();
    }
    reader.join();
    if (!status && carry_len > 0) { status = PROBLEM_CORRUPT; tredsw_set_error("%s ends inside a BAM record", bam->path.c_str()); }
    stats[9] = status;
    if (irr) {
        unsigned long long h_ist[IRR_NSTATS];
        be.download(h_ist, d_irr_stats, sizeof(h_ist));
        be.sync();
        if (be.rc) return be.rc;
        if (status) { out->irr_entries.clear(); out->irr_names.clear(); memset(h_ist, 0, sizeof(h_ist)); }
        irr_join(out, h_ist);
    }

    // ---- (3) depth regions; the entries grouped by fetch (stable counting sort: file order within a fetch) ----------
    std::vector<unsigned long long> h_depth((size_t)std::max(1, n_depth));
    be.download(h_depth.data(), d_depth, sizeof(unsigned long long) * (size_t)std::max(1, n_depth));
    be.sync();
    if (be.rc) return be.rc;
    for (int d = 0; d < n_depth; ++d)
        depth_out[d] = status ? NAN : (double)h_depth[d] * 1.0 / (double)(depth_regions[3 * d + 2] - depth_regions[3 * d + 1] + 1);
    if (status) {
        for (int p = 0; p < nq; ++p) if (!out->status[p]) out->status[p] = status;
        ent_fetch.clear(); ent_pos.clear();
    }
    const int64_t nrec = (int64_t)ent_fetch.size();
    if (nrec >= (1ll << 32)) { tredsw_set_error("too many selected records"); return TREDSW_ERR_IO; }
    std::vector<uint32_t> fbase(nfetch + 2, 0);
    for (int32_t f : ent_fetch) ++fbase[f + 1];
    for (int f = 0; f < nfetch; ++f) fbase[f + 1] += fbase[f];
    std::vector<int64_t> rpos((size_t)std::max<int64_t>(1, nrec));
    std::vector<int32_t> rfetch((size_t)std::max<int64_t>(1, nrec));
    {
        std::vector<uint32_t> at(fbase.begin(), fbase.begin() + nfetch + 1);
        for (int64_t e = 0; e < nrec; ++e) { const uint32_t k = at[ent_fetch[e]]++; rpos[k] = ent_pos[e]; rfetch[k] = ent_fetch[e]; }
    }
    out->n_blocks = stats[1]; out->n_records = stats[2];
    out->comp_bytes = stats[4]; out->inflated_bytes = stats[5];
    out->ms_host_stage = stats[6] * 1e-3;
    out->ms_marks[0] = now_ms() - t_begin;
    if (nq == 0) {
        be.release_intermediates();
        out->ms_total = now_ms() - t_begin;
        stats[8] = (int64_t)(out->ms_total * 1e3);
        tredsw_ingest_view &v = out->view;
        v.n_blocks = out->n_blocks; v.n_records = out->n_records; v.comp_bytes = out->comp_bytes; v.inflated_bytes = out->inflated_bytes;
        v.ms_host_stage = out->ms_host_stage; v.ms_total = out->ms_total; v.ms_marks[0] = out->ms_marks[0];
        return TREDSW_OK;
    }
    Fetch *d_fetches = alloc_n<Fetch>(be, nfetch);
    ProblemParams *d_params = alloc_n<ProblemParams>(be, nq);
    ProblemCounts *d_counts = alloc_n<ProblemCounts>(be, nq);
    int64_t *d_rpos = alloc_n<int64_t>(be, (int64_t)rpos.size());
    int32_t *d_rfetch = alloc_n<int32_t>(be, (int64_t)rfetch.size());
    uint32_t *d_fbase = alloc_n<uint32_t>(be, (int64_t)fbase.size());
    const uint8_t *d_kept = buf.kept.get(be, 64);   // (a scan that kept nothing still hands over a buffer)
    if (be.rc) return be.rc;
    be.upload(d_fetches, fetches.data(), sizeof(Fetch) * (size_t)nfetch);
    be.upload(d_params, params.data(), sizeof(ProblemParams) * (size_t)nq);
    be.fill(d_counts, 0, sizeof(ProblemCounts) * (size_t)nq);
    be.upload(d_rpos, rpos.data(), sizeof(int64_t) * (size_t)nrec);
    be.upload(d_rfetch, rfetch.data(), sizeof(int32_t) * (size_t)nrec);
    be.upload(d_fbase, fbase.data(), sizeof(uint32_t) * fbase.size());
    const int rc = select_and_pair(be, out, d_kept, d_fetches, d_rpos, d_rfetch, d_fbase, nrec,
                                   fetch_first, params, d_params, d_counts, want_names, t_begin);
    stats[8] = (int64_t)(out->ms_total * 1e3);
    return rc;
}

namespace {
// The mates among the IRR entries: the records of one name with segment flags 0x40 and 0x80 (the first of each, in
// file order), and the profile's counters.  An anchored IRR without an MQ tag (paired, mate mapped and not an IRR)
// is counted in anchors_without_mq.
void irr_join(tredsw_ingest_batch *out, const unsigned long long *st) {
    std::vector<IrrEntry> &e = out->irr_entries;
    const char *names = out->irr_names.data();
    std::unordered_map<std::string, std::pair<int32_t, int32_t>> seg;     // name -> (first 0x40 entry, first 0x80 entry)
    seg.reserve(e.size());
    for (size_t k = 0; k < e.size(); ++k) {
        const int f = e[k].flag & 0xc0;
        if (f != 0x40 && f != 0x80) continue;
        auto it = seg.emplace(std::string(names + e[k].name_off, (size_t)e[k].name_len), std::make_pair(-1, -1)).first;
        int32_t &slot = f == 0x40 ? it->second.first : it->second.second;
        if (slot < 0) slot = (int32_t)k;
    }
    for (auto &kv : seg)
        if (kv.second.first >= 0 && kv.second.second >= 0) { e[kv.second.first].mate = kv.second.second; e[kv.second.second].mate = kv.second.first; }
    tredsw_irr_view &v = out->irr_view;
    memset(&v, 0, sizeof(v));
    v.n_entries = (int64_t)e.size();
    v.entries = reinterpret_cast<const tredsw_irr_entry *>(e.data());
    v.names = names; v.name_bytes = (int64_t)out->irr_names.size();
    v.records_considered = (int64_t)st[IRR_CONSIDERED]; v.irr_records = (int64_t)e.size();
    v.depth_bases = (int64_t)st[IRR_DEPTH_BASES]; v.max_l_seq = (int64_t)st[IRR_MAX_LSEQ];
    v.unparsed_aux = (int64_t)st[IRR_UNPARSED_AUX];
    for (const IrrEntry &x : e)
        v.anchors_without_mq += (x.flag & 1) && !(x.flag & 8) && x.next_tid >= 0 && x.mate < 0 && x.mq < 0;
}

bool irr_params_ok(const tredsw_irr_params *p) {
    if (!p) return true;
    if (p->min_period < 2 || p->min_period > p->max_period || p->max_period > 20 || p->purity_num <= 0 ||
        p->purity_num > p->purity_den || p->purity_den > 1000 || p->min_read_len < 2 * p->max_period) {
        tredsw_set_error("IRR parameters out of range (2 <= min_period <= max_period <= 20, 0 < num <= den <= 1000, "
                         "min_read_len >= 2 max_period)");
        return false;
    }
    return true;
}

// (once per device) keep freed blocks in the stream-ordered pool: the buffers of consecutive batches have similar sizes
void keep_pool(int device) {
    static bool pool_set[64] = {false};
    if (device < 64 && !pool_set[device]) {
        cudaMemPool_t pool;
        if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
            unsigned long long thr = ~0ull;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
        }
        pool_set[device] = true;
    }
}

// The body of every C entry point of this file: a new result R filled by run(backend, result).  With a context it runs
// on the context's device and stream under its lock, and its kernel launches are added to ctx->launches; without one
// (nullptr: the test emulations) it runs on the host backend.  An exception is TREDSW_ERR_IO named after `what`.  A
// failed run releases its backend; a successful one too, unless R::keeps_backend (an ingest batch's device buffers
// are its view).  On success *out owns the result.
template <class R, class Run>
int run_entry(tredsw_ctx *ctx, const char *what, R **out, Run &&run) {
    *out = nullptr;
    std::unique_lock<std::mutex> lock;
    if (ctx) {
        lock = std::unique_lock<std::mutex>(ctx->mu);
        CUDA_TRY(cudaSetDevice(ctx->device));
        keep_pool(ctx->device);
    }
    std::unique_ptr<R> r(new R());
    r->emulated = !ctx;
    r->cuda.stream = ctx ? ctx->stream : nullptr;
    auto go = [&](auto &be) {
        int rc;
        try { rc = run(be, r.get()); }
        catch (const std::exception &e) { tredsw_set_error("%s: %s", what, e.what()); rc = TREDSW_ERR_IO; }
        if (ctx) ctx->launches += r->cuda.launches;
        if (rc || !R::keeps_backend) be.release();
        return rc;
    };
    const int rc = ctx ? go(r->cuda) : go(r->host);
    if (rc) return rc;
    *out = r.release();
    return TREDSW_OK;
}
}  // namespace

extern "C" {

int tredsw_ingest_scan_run(tredsw_ctx *ctx, tredsw_bam *bam, const tredsw_locus_query *queries, int32_t nqueries,
                           const int32_t *depth_regions, int32_t n_depth, double *depth_out, int64_t slab_bytes,
                           uint32_t flags, tredsw_ingest_batch **out) {
    return tredsw_ingest_scan_run_ex(ctx, bam, queries, nqueries, depth_regions, n_depth, depth_out, slab_bytes, flags, nullptr, out);
}

int tredsw_ingest_scan_run_ex(tredsw_ctx *ctx, tredsw_bam *bam, const tredsw_locus_query *queries, int32_t nqueries,
                              const int32_t *depth_regions, int32_t n_depth, double *depth_out, int64_t slab_bytes,
                              uint32_t flags, const tredsw_irr_params *irr, tredsw_ingest_batch **out) {
    if (!ctx || !bam || !out || nqueries < 0 || (nqueries > 0 && !queries) || n_depth < 0 ||
        (n_depth > 0 && (!depth_regions || !depth_out)) || slab_bytes < 0) { tredsw_set_error("bad arguments"); return TREDSW_ERR_ARG; }
    if (!irr_params_ok(irr)) return TREDSW_ERR_ARG;
    *out = nullptr;
    if (bam->consumed) { tredsw_set_error("%s: stream already consumed", bam->path.c_str()); return TREDSW_ERR_ARG; }
    return run_entry(ctx, "tredsw_ingest_scan_run", out, [&](auto &be, tredsw_ingest_batch *b) {
        return run_scan(be, b, bam, queries, nqueries, depth_regions, n_depth, depth_out, slab_bytes, flags, irr);
    });
}

// TEST INFRASTRUCTURE: tredsw_ingest_scan_run with every kernel body run serially on the host.  Not used by the package.
int tredsw_ingest_scan_emulate(tredsw_bam *bam, const tredsw_locus_query *queries, int32_t nqueries,
                               const int32_t *depth_regions, int32_t n_depth, double *depth_out, int64_t slab_bytes,
                               uint32_t flags, tredsw_ingest_batch **out) {
    return tredsw_ingest_scan_emulate_ex(bam, queries, nqueries, depth_regions, n_depth, depth_out, slab_bytes, flags, nullptr, out);
}

int tredsw_ingest_scan_emulate_ex(tredsw_bam *bam, const tredsw_locus_query *queries, int32_t nqueries,
                                  const int32_t *depth_regions, int32_t n_depth, double *depth_out, int64_t slab_bytes,
                                  uint32_t flags, const tredsw_irr_params *irr, tredsw_ingest_batch **out) {
    if (!bam || !out || nqueries < 0 || (nqueries > 0 && !queries) || n_depth < 0 ||
        (n_depth > 0 && (!depth_regions || !depth_out)) || slab_bytes < 0) { tredsw_set_error("bad arguments"); return TREDSW_ERR_ARG; }
    if (!irr_params_ok(irr)) return TREDSW_ERR_ARG;
    *out = nullptr;
    if (bam->consumed) { tredsw_set_error("%s: stream already consumed", bam->path.c_str()); return TREDSW_ERR_ARG; }
    return run_entry(nullptr, "tredsw_ingest_scan_emulate", out, [&](auto &be, tredsw_ingest_batch *b) {
        return run_scan(be, b, bam, queries, nqueries, depth_regions, n_depth, depth_out, slab_bytes, flags, irr);
    });
}

int tredsw_ingest_scan_irr(const tredsw_ingest_batch *b, tredsw_irr_view *v) {
    if (!b || !v) { tredsw_set_error("bad arguments"); return TREDSW_ERR_ARG; }
    if (!b->irr_on) { tredsw_set_error("the scan did not profile in-repeat reads (tredsw_ingest_scan_run_ex with irr)"); return TREDSW_ERR_ARG; }
    *v = b->irr_view;
    return TREDSW_OK;
}

// The IRR classifier on its own (test hook, host execution of the device code)
int tredsw_irr_classify_host(const int8_t *codes, int32_t len, const tredsw_irr_params *p, int32_t *period, uint64_t *motif) {
    if (!p || !period || !motif || len < 0 || (len > 0 && !codes)) { tredsw_set_error("bad arguments"); return TREDSW_ERR_ARG; }
    if (!irr_params_ok(p)) return TREDSW_ERR_ARG;
    const IrrParams ip{p->min_period, p->max_period, p->purity_num, p->purity_den, p->min_read_len};
    *period = irr_classify(CodeSeq{codes}, len, ip, motif);
    return TREDSW_OK;
}

int tredsw_ingest_scan_stats(const tredsw_ingest_batch *b, int64_t *stats) {
    if (!b || !stats) { tredsw_set_error("bad arguments"); return TREDSW_ERR_ARG; }
    memcpy(stats, b->scan_stats, sizeof(b->scan_stats));
    return TREDSW_OK;
}

int tredsw_ingest_batch_run(tredsw_ctx *ctx, tredsw_bam *const *bams, const int32_t *sample_of,
                            const tredsw_locus_query *queries, int32_t nqueries, uint32_t flags, tredsw_ingest_batch **out) {
    if (!ctx || !out || nqueries < 0 || (nqueries > 0 && (!bams || !sample_of || !queries))) { tredsw_set_error("bad arguments"); return TREDSW_ERR_ARG; }
    return run_entry(ctx, "tredsw_ingest_batch_run", out, [&](auto &be, tredsw_ingest_batch *b) {
        return run_pipeline(be, b, bams, sample_of, queries, nqueries, flags);
    });
}

// TEST INFRASTRUCTURE: the same pipeline with every kernel body run serially on the host (no CUDA calls).  The
// "device" pointers of the view are host pointers.  Not used by the package.
int tredsw_ingest_batch_emulate(tredsw_bam *const *bams, const int32_t *sample_of, const tredsw_locus_query *queries,
                                int32_t nqueries, uint32_t flags, tredsw_ingest_batch **out) {
    if (!out || nqueries < 0 || (nqueries > 0 && (!bams || !sample_of || !queries))) { tredsw_set_error("bad arguments"); return TREDSW_ERR_ARG; }
    return run_entry(nullptr, "tredsw_ingest_batch_emulate", out, [&](auto &be, tredsw_ingest_batch *b) {
        return run_pipeline(be, b, bams, sample_of, queries, nqueries, flags);
    });
}

int tredsw_ingest_batch_view(const tredsw_ingest_batch *b, tredsw_ingest_view *view) {
    if (!b || !view) { tredsw_set_error("bad arguments"); return TREDSW_ERR_ARG; }
    *view = b->view;
    return TREDSW_OK;
}

void tredsw_ingest_batch_free(tredsw_ingest_batch *b) {
    if (!b) return;
    if (b->emulated) b->host.release(); else b->cuda.release();
    delete b;
}

// The block decoder on its own (test hook, host execution of the device code): 0 iff `in` inflates to out_len bytes.
int tredsw_inflate_raw_device_code(const uint8_t *in, int64_t in_len, uint8_t *out, int64_t out_len) {
    std::vector<uint8_t> padded((size_t)in_len + 4 + 32, 0);  // the bit reader loads whole words, up to 16 bytes behind a corrupt stream
    if (in_len > 0) memcpy(padded.data() + 4, in, (size_t)in_len);
    std::vector<uint16_t> tabs(TAB_ENTRIES);
    uint8_t lens[320], sub_need[1 << LIT_ROOT];
    uint16_t sub_base[1 << LIT_ROOT];
    // (offset 4 + a caller-chosen misalignment would also work: the reader handles any start address)
    return inflate_block<1>(padded.data() + 4, in_len, out, out_len, TabRef{tabs.data(), 1, true}, lens, sub_need, sub_base, 0) ? 0 : 1;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------------------
// the reference tract scan: every tract of the requested motifs in a FASTA, plain text or BGZF (ref_tracts_device.cuh)
// ---------------------------------------------------------------------------------------------------------------
struct tredsw_tracts {
    static constexpr bool keeps_backend = false;    // the results are host memory: the backend is released by run_entry
    bool emulated = false;
    CudaBackend cuda;
    HostBackend host;
    std::vector<TractOut> tracts;
    std::vector<int32_t> segments;                  // per tract: its chain's segments (1: a pure tract)
    std::vector<double> read_ms, device_ms;
    tredsw_tracts_view view;
};
static_assert(sizeof(TractOut) == sizeof(tredsw_tract), "TractOut mirrors tredsw_tract");

namespace {

constexpr int64_t TRACT_DEFAULT_STEP = 256ll << 20;    // bytes of FASTA text per step when the caller passes 0

int64_t fai_text_bytes(const tredsw_fai_entry &c) {     // bytes from a contig's first base to its last
    if (c.length <= 0) return 0;
    const int64_t last = c.length - 1;
    return last / c.line_bases * c.line_width + last % c.line_bases + 1;
}

// One block of a BGZF FASTA, from the walk of its headers: compressed offset and size, inflated offset and size.  The
// .fai of a bgzipped FASTA gives inflated offsets (samtools writes it so); the .gzi is not read.
struct TractBlock { int64_t coff, uoff; int32_t bsize; uint32_t isize; };

struct TractStep {                  // contigs [c0, c1) of the call; of a BGZF file, the blocks [b0, b1) that hold them
    int32_t c0 = 0, c1 = 0, b0 = 0, b1 = 0;
    int64_t bytes = 0;              // text handed to the kernels: the contigs' text, or the inflated blocks [b0, b1)
    int64_t comp_bytes = 0;         // BGZF: the compressed blocks [b0, b1)
    uint8_t *buf = nullptr;         // page-locked: the text, or the compressed blocks
    std::vector<BlockDesc> blocks;  // BGZF: in_off into buf, out_off from block b0's first inflated byte
    const char *why = nullptr;      // I/O or framing error
    int64_t at = -1;                // the file offset of the block it concerns, where there is one
    double ms = 0;                  // host read time
};

void read_tract_step(int fd, const tredsw_fai_entry *cs, TractStep *st) {
    const double t0 = now_ms();
    st->why = nullptr;
    int64_t at = 0;
    for (int32_t c = st->c0; c < st->c1 && !st->why; ++c) {
        const int64_t n = fai_text_bytes(cs[c]);
        if (pread_full(fd, st->buf + at, n, cs[c].offset) < n) st->why = "the file is shorter than its index says";
        at += n;
    }
    st->ms = now_ms() - t0;
}

// A BGZF step: its compressed blocks in one read, each framed again and checked against the walk.
void read_bgzf_step(int fd, const TractBlock *tb, TractStep *st) {
    const double t0 = now_ms();
    st->why = nullptr; st->at = -1;
    st->blocks.clear();
    const int64_t c0 = st->b1 > st->b0 ? tb[st->b0].coff : 0, n = st->comp_bytes;
    const int64_t got = pread_full(fd, st->buf, n, c0);
    if (got < n) { st->why = "the file is shorter than its BGZF blocks"; st->at = c0 + got; }
    for (int32_t b = st->b0; b < st->b1 && !st->why; ++b) {
        const int64_t o = tb[b].coff - c0;
        BgzfFrame fr;
        const char *why = nullptr;
        if (parse_bgzf_block(st->buf + o, n - o, &fr, &why) != 1 || fr.bsize != tb[b].bsize || fr.isize != tb[b].isize) {
            st->why = why ? why : "the BGZF framing differs from the block walk (the file changed)";
            st->at = tb[b].coff;
            break;
        }
        st->blocks.push_back(block_desc(fr, o, tb[b].uoff - tb[st->b0].uoff));
    }
    st->ms = now_ms() - t0;
}

// The block table of a BGZF file: one pass over the block headers, BSIZE from each header and ISIZE from each block's
// last 4 bytes (one read per block: a block's ISIZE and the next block's header).  TREDSW_ERR_IO names the offset of a
// block that is truncated or not BGZF (a plain gzip file fails here).
int walk_bgzf(int fd, const char *path, std::vector<TractBlock> *tb) {
    struct stat sb;
    if (fstat(fd, &sb) != 0) { tredsw_set_error("%s: cannot stat: %s", path, strerror(errno)); return TREDSW_ERR_IO; }
    const int64_t size = (int64_t)sb.st_size;
    auto fail = [&](const char *why, int64_t at) {
        tredsw_set_error("%s: %s at offset %lld", path, why, (long long)at);
        return TREDSW_ERR_IO;
    };
    std::vector<uint8_t> h(4 + 64);                     // [ISIZE of the block before | the header of the block at o]
    int64_t o = 0, u = 0, n = pread_full(fd, h.data() + 4, std::min<int64_t>(64, size), 0);
    while (o < size) {
        const int64_t need = n >= 12 ? 12 + (h[4 + 10] | (h[4 + 11] << 8)) : 18;     // extra subfields beyond BC
        if (need > n && o + n < size) {
            h.resize((size_t)(4 + need));
            n = pread_full(fd, h.data() + 4, std::min(need, size - o), o);
        }
        BgzfFrame fr;
        const char *why = nullptr;
        if (parse_bgzf_header(h.data() + 4, n, &fr, &why) != 1) return fail(why, o);
        const int64_t e = o + fr.bsize;
        if (e > size) return fail("truncated BGZF block", o);
        const int64_t want = 4 + std::min<int64_t>(64, size - e);
        if (h.size() < 4 + 64) h.resize(4 + 64);
        if (pread_full(fd, h.data(), want, e - 4) < want) return fail("short read", o);
        uint32_t isize;
        memcpy(&isize, h.data(), 4);
        if (isize > 65536) return fail("BGZF block larger than 64 KiB", o);
        tb->push_back(TractBlock{o, u, fr.bsize, isize});
        u += isize;
        o = e;
        n = want - 4;
    }
    return TREDSW_OK;
}

// The blocks of every step of a BGZF file: from the block holding the step's first text byte to the one holding its
// last (a block two steps share is read and inflated by both).  An index that reaches past the inflated end is
// TREDSW_ERR_IO before anything is read.
int plan_bgzf_steps(const char *path, const std::vector<TractBlock> &tb, const tredsw_fai_entry *cs,
                    std::vector<TractStep> &steps) {
    const int64_t total = tb.empty() ? 0 : tb.back().uoff + tb.back().isize;
    auto block_of = [&](int64_t x) {                    // the last block starting at or before x (a non-empty one)
        return (int32_t)(std::upper_bound(tb.begin(), tb.end(), x, [](int64_t v, const TractBlock &b) { return v < b.uoff; })
                         - tb.begin()) - 1;
    };
    for (TractStep &st : steps) {
        int64_t lo = -1, hi = -1;                       // the step's first and last text byte
        for (int32_t c = st.c0; c < st.c1; ++c) {
            const int64_t n = fai_text_bytes(cs[c]);
            if (!n) continue;
            if (cs[c].offset + n > total) {
                tredsw_set_error("%s: contig %d ends at inflated byte %lld, past the end of the inflated text (%lld "
                                 "bytes): the index does not fit the file", path, c, (long long)(cs[c].offset + n),
                                 (long long)total);
                return TREDSW_ERR_IO;
            }
            lo = lo < 0 ? cs[c].offset : std::min(lo, cs[c].offset);
            hi = std::max(hi, cs[c].offset + n - 1);
        }
        st.bytes = st.comp_bytes = 0;
        st.b0 = st.b1 = 0;
        if (lo < 0) continue;                           // empty contigs only
        st.b0 = block_of(lo);
        st.b1 = block_of(hi) + 1;
        const TractBlock &f = tb[st.b0], &l = tb[st.b1 - 1];
        st.bytes = l.uoff + l.isize - f.uoff;
        st.comp_bytes = l.coff + l.bsize - f.coff;
    }
    return TREDSW_OK;
}

template <class B>
int run_ref_tracts(B &be, tredsw_tracts *out, const char *path, const tredsw_fai_entry *cs, int32_t nc,
                   const tredsw_motif *ms, int32_t nm, const tredsw_tract_params &prm, const TractChain &ch) {
    const double t_begin = now_ms();
    // the requested codes by period, ascending
    std::vector<std::pair<int32_t, uint64_t>> mv;
    for (int32_t i = 0; i < nm; ++i) mv.emplace_back(ms[i].period, ms[i].code);
    std::sort(mv.begin(), mv.end());
    mv.erase(std::unique(mv.begin(), mv.end()), mv.end());
    std::vector<int32_t> periods, mfirst;
    std::vector<uint64_t> mcodes;
    for (const auto &m : mv) {
        if (periods.empty() || periods.back() != m.first) { periods.push_back(m.first); mfirst.push_back((int32_t)mcodes.size()); }
        mcodes.push_back(m.second);
    }
    mfirst.push_back((int32_t)mcodes.size());
    const int32_t nper = (int32_t)periods.size();
    // steps: consecutive contigs under the byte budget (a larger contig alone)
    const int64_t budget = prm.step_bytes > 0 ? prm.step_bytes : TRACT_DEFAULT_STEP;
    std::vector<TractStep> steps;
    int64_t max_bytes = 0, bases = 0;
    for (int32_t c = 0; c < nc && nper; ++c) {
        const int64_t n = fai_text_bytes(cs[c]);
        bases += cs[c].length;
        if (steps.empty() || (steps.back().bytes + n > budget && steps.back().c1 > steps.back().c0)) {
            steps.push_back(TractStep());
            steps.back().c0 = c;
        }
        steps.back().c1 = c + 1;
        steps.back().bytes += n;
        max_bytes = std::max(max_bytes, steps.back().bytes);
    }
    const int fd = steps.empty() ? -1 : open(path, O_RDONLY);
    if (!steps.empty() && fd < 0) { tredsw_set_error("%s: cannot open: %s", path, strerror(errno)); return TREDSW_ERR_IO; }
    struct Close { int fd; ~Close() { if (fd >= 0) close(fd); } } close_fd{fd};
    // the format, from the file: gzip magic -> BGZF (its blocks inflated on the device), anything else -> text
    uint8_t magic[2] = {0, 0};
    const bool bgzf = fd >= 0 && pread_full(fd, magic, 2, 0) == 2 && magic[0] == 31 && magic[1] == 139;
    std::vector<TractBlock> tb;
    if (bgzf) {
        int rc = walk_bgzf(fd, path, &tb);
        if (!rc) rc = plan_bgzf_steps(path, tb, cs, steps);
        if (rc) return rc;
        max_bytes = 0;
        for (const TractStep &st : steps) max_bytes = std::max(max_bytes, st.comp_bytes);
    }
    uint8_t *pinned[2] = {nullptr, nullptr};
    for (uint8_t *&p : pinned) if (!steps.empty()) p = alloc_host_n<uint8_t>(be, max_bytes + 64);
    int32_t *d_per = alloc_n<int32_t>(be, 2 * nper + 1);
    uint64_t *d_codes = alloc_n<uint64_t>(be, (int64_t)mcodes.size());
    unsigned long long *d_small = alloc_n<unsigned long long>(be, 3);
    if (be.rc) return be.rc;
    be.upload(d_per, periods.data(), sizeof(int32_t) * (size_t)nper);
    be.upload(d_per + nper, mfirst.data(), sizeof(int32_t) * (size_t)(nper + 1));
    be.upload(d_codes, mcodes.data(), sizeof(uint64_t) * mcodes.size());
    const TractQuery q{d_per, d_per + nper, d_codes, nper, prm.min_units, (int64_t)prm.min_len};
    struct {                                            // device buffers reused from step to step
        Reused<uint8_t> text, comp, bstatus;
        Reused<uint64_t> code;
        Reused<uint32_t> valid;
        Reused<TractContig> cs;
        Reused<BlockDesc> blocks;
        Reused<TractOut> out;
        Reused<int32_t> segs;                           // with chains: per tract, its segments
    } buf;
    const bool chained = ch.max_interrupt > 0;
    buf.out.get(be, 65536);
    if (chained) buf.segs.get(be, 65536);
    int64_t invalid = 0, bytes = 0, comp_bytes = 0, nblocks = 0;
    auto read_step = [&](TractStep *st) { if (bgzf) read_bgzf_step(fd, tb.data(), st); else read_tract_step(fd, cs, st); };
    ReadAhead reader;
    if (!steps.empty()) { steps[0].buf = pinned[0]; read_step(&steps[0]); }
    for (size_t k = 0; k < steps.size(); ++k) {
        TractStep &st = steps[k];
        if (st.why && st.at >= 0) { tredsw_set_error("%s: %s at offset %lld", path, st.why, (long long)st.at); return TREDSW_ERR_IO; }
        if (st.why) { tredsw_set_error("%s: %s", path, st.why); return TREDSW_ERR_IO; }
        if (k + 1 < steps.size()) {
            steps[k + 1].buf = pinned[(k + 1) & 1];
            reader.start(read_step, &steps[k + 1]);
        }
        const double t_dev = now_ms();
        // the step's contigs: text and word offsets
        const int ncs = st.c1 - st.c0;
        std::vector<TractContig> tc(ncs);
        int64_t text_at = 0, words = 0;
        for (int i = 0; i < ncs; ++i) {
            const tredsw_fai_entry &f = cs[st.c0 + i];
            if (bgzf) text_at = f.length > 0 ? f.offset - tb[st.b0].uoff : 0;      // (header lines are never addressed)
            tc[i] = TractContig{f.length, text_at, words, f.line_bases, f.line_width, st.c0 + i, 0};
            text_at += fai_text_bytes(f);
            words += tract_words(f.length);
        }
        uint8_t *text = buf.text.get(be, st.bytes + 64);
        uint64_t *code = buf.code.get(be, words);
        uint32_t *valid = buf.valid.get(be, words);
        TractContig *dcs = buf.cs.get(be, ncs);
        if (be.rc) return be.rc;
        const int nb = (int)st.blocks.size();
        std::vector<uint8_t> h_bstatus(nb);
        uint8_t *bstatus = nullptr;
        if (bgzf) {                                     // the step's blocks, inflated into its text buffer
            uint8_t *comp = buf.comp.get(be, st.comp_bytes + 64);
            BlockDesc *blocks = buf.blocks.get(be, nb);
            bstatus = buf.bstatus.get(be, nb);
            if (be.rc) return be.rc;
            be.upload(comp, st.buf, (size_t)st.comp_bytes);
            be.upload(blocks, st.blocks.data(), sizeof(BlockDesc) * (size_t)nb);
            be.inflate(comp, text, blocks, nb, bstatus, 1);
        } else {
            be.upload(text, st.buf, (size_t)st.bytes);
        }
        be.upload(dcs, tc.data(), sizeof(TractContig) * (size_t)ncs);
        be.fill(d_small, 0, sizeof(unsigned long long) * 3);
        unsigned long long *cnt = d_small, *inval = d_small + 1, *err = d_small + 2;
        be.template for_each<TractPackTag>(words, [=] __host__ __device__(int64_t w) {
            const TractContig c = dcs[tract_contig_of(dcs, ncs, w)];
            bool bad = false;
            const int n = tract_pack_word(text, c, w - c.word0, &code[w], &valid[w], &bad);
            warp_add_u64(inval, (uint32_t)n);
            if (bad) atomic_add_u64(err, 1ull);
        });
        // the runs of every period, one thread per (word, period); more tracts than room: run again with room for all
        unsigned long long h_small[3] = {0, 0, 0};
        for (int pass = 0; pass < 2; ++pass) {
            const unsigned long long cap = (unsigned long long)buf.out.cap;
            TractOut *tout = buf.out.p;
            if (chained) {                              // interrupted tracts: replaces the pure runs
                int32_t *tsegs = buf.segs.p;
                be.template for_each<TractChainsTag>(words * nper, [=] __host__ __device__(int64_t i) {
                    const int64_t w = i / q.nper;
                    const TractContig &c = dcs[tract_contig_of(dcs, ncs, w)];
                    tract_chains(code, valid, c, w - c.word0, (int)(i - w * q.nper), q, ch, tout, tsegs, cnt, cap);
                });
            } else {
                be.template for_each<TractRunsTag>(words * nper, [=] __host__ __device__(int64_t i) {
                    const int64_t w = i / q.nper;
                    const TractContig &c = dcs[tract_contig_of(dcs, ncs, w)];
                    tract_runs(code, valid, c, w - c.word0, (int)(i - w * q.nper), q, tout, cnt, cap);
                });
            }
            be.download(h_small, d_small, sizeof(h_small));
            if (pass == 0) be.download(h_bstatus.data(), bstatus, (size_t)nb);
            be.sync();
            if (be.rc) return be.rc;
            for (int b = 0; b < nb; ++b)
                if (h_bstatus[b]) {
                    tredsw_set_error("%s: the BGZF block at offset %lld %s", path, (long long)tb[st.b0 + b].coff,
                                     h_bstatus[b] == 1 ? "does not inflate" : "fails its CRC-32 / length check");
                    return TREDSW_ERR_IO;
                }
            if (h_small[2]) { tredsw_set_error("%s: a base position holds a line break or a header: the index does not fit the file", path); return TREDSW_ERR_IO; }
            if (h_small[0] <= cap) break;
            if (pass) { tredsw_set_error("tract count changed between passes"); return TREDSW_ERR_CUDA; }
            buf.out.cap = (int64_t)(h_small[0] + h_small[0] / 4 + 1024);      // room for all, not geometric
            buf.out.p = alloc_n<TractOut>(be, buf.out.cap);
            if (chained) { buf.segs.cap = buf.out.cap; buf.segs.p = alloc_n<int32_t>(be, buf.segs.cap); }
            be.fill(cnt, 0, sizeof(unsigned long long));
            if (be.rc) return be.rc;
        }
        const size_t t0 = out->tracts.size();
        out->tracts.resize(t0 + (size_t)h_small[0]);
        be.download(out->tracts.data() + t0, buf.out.p, sizeof(TractOut) * (size_t)h_small[0]);
        out->segments.resize(t0 + (size_t)h_small[0], 1);
        if (chained) be.download(out->segments.data() + t0, buf.segs.p, sizeof(int32_t) * (size_t)h_small[0]);
        be.sync();
        if (be.rc) return be.rc;
        invalid += (int64_t)h_small[1];
        bytes += st.bytes;
        comp_bytes += st.comp_bytes;
        nblocks += nb;
        out->read_ms.push_back(st.ms);
        out->device_ms.push_back(now_ms() - t_dev);
        reader.join();
    }
    auto before = [](const TractOut &x, const TractOut &y) {
        return x.contig != y.contig ? x.contig < y.contig : x.start != y.start ? x.start < y.start : x.period < y.period;
    };
    if (!chained) {
        std::sort(out->tracts.begin(), out->tracts.end(), before);
    } else {                                            // the tracts and their segment counts, in one order
        std::vector<size_t> ord(out->tracts.size());
        for (size_t i = 0; i < ord.size(); ++i) ord[i] = i;
        std::sort(ord.begin(), ord.end(), [&](size_t x, size_t y) { return before(out->tracts[x], out->tracts[y]); });
        std::vector<TractOut> t(ord.size());
        std::vector<int32_t> sg(ord.size());
        for (size_t i = 0; i < ord.size(); ++i) { t[i] = out->tracts[ord[i]]; sg[i] = out->segments[ord[i]]; }
        out->tracts.swap(t);
        out->segments.swap(sg);
    }
    be.release_intermediates();
    tredsw_tracts_view &v = out->view;
    memset(&v, 0, sizeof(v));
    v.n_tracts = (int64_t)out->tracts.size();
    v.tracts = reinterpret_cast<const tredsw_tract *>(out->tracts.data());
    v.steps = (int64_t)out->read_ms.size(); v.bytes = bytes; v.bases = bases; v.invalid_bases = invalid;
    v.step_read_ms = out->read_ms.data(); v.step_device_ms = out->device_ms.data();
    v.ms_total = now_ms() - t_begin;
    v.comp_bytes = comp_bytes; v.blocks = nblocks;
    v.segments = out->segments.data();
    return TREDSW_OK;
}

bool tract_args_ok(const char *path, const tredsw_fai_entry *cs, int32_t nc, const tredsw_motif *ms, int32_t nm,
                   const tredsw_tract_params *p, tredsw_tracts **out) {
    if (!path || !out || !p || nc < 0 || nm < 0 || (nc && !cs) || (nm && !ms)) { tredsw_set_error("bad arguments"); return false; }
    if (p->min_units < 2 || p->min_len < 0 || p->step_bytes < 0) {
        tredsw_set_error("tract parameters out of range (min_units >= 2, min_len >= 0, step_bytes >= 0)");
        return false;
    }
    for (int32_t i = 0; i < nm; ++i)
        if (ms[i].period < 2 || ms[i].period > 20 || ms[i].code >> (2 * ms[i].period)) {
            tredsw_set_error("motif %d: period %d / code %llu out of range (2 <= period <= 20, code < 4^period)", i,
                             ms[i].period, (unsigned long long)ms[i].code);
            return false;
        }
    for (int32_t c = 0; c < nc; ++c)
        if (cs[c].length < 0 || cs[c].offset < 0 || (cs[c].length > 0 && (cs[c].line_bases <= 0 || cs[c].line_width < cs[c].line_bases))) {
            tredsw_set_error("contig %d: bad index entry (length %lld, offset %lld, line %d bases / %d bytes)", c,
                             (long long)cs[c].length, (long long)cs[c].offset, cs[c].line_bases, cs[c].line_width);
            return false;
        }
    return true;
}

// the chaining parameters of a call: NULL -> off; out of range -> false
bool tract_chain_ok(const tredsw_tract_chain *c, TractChain *ch) {
    *ch = TractChain{0, 1, 1};
    if (!c) return true;
    if (c->max_interrupt < 0 || c->max_interrupt > 20 || c->purity_num <= 0 || c->purity_num > c->purity_den ||
        c->purity_den > 1000) {
        tredsw_set_error("chain parameters out of range (0 <= max_interrupt <= 20, 0 < purity_num <= purity_den <= 1000): "
                         "%d, %d / %d", c->max_interrupt, c->purity_num, c->purity_den);
        return false;
    }
    *ch = TractChain{c->max_interrupt, c->purity_num, c->purity_den};
    return true;
}

}  // namespace

extern "C" {

int tredsw_ref_tracts_ex(tredsw_ctx *ctx, const char *fasta_path, const tredsw_fai_entry *contigs, int32_t ncontigs,
                         const tredsw_motif *motifs, int32_t nmotifs, const tredsw_tract_params *params,
                         const tredsw_tract_chain *chain, tredsw_tracts **result) {
    TractChain ch;
    if (!ctx) { tredsw_set_error("bad arguments"); return TREDSW_ERR_ARG; }
    if (!tract_args_ok(fasta_path, contigs, ncontigs, motifs, nmotifs, params, result) || !tract_chain_ok(chain, &ch))
        return TREDSW_ERR_ARG;
    return run_entry(ctx, "tredsw_ref_tracts", result, [&](auto &be, tredsw_tracts *r) {
        return run_ref_tracts(be, r, fasta_path, contigs, ncontigs, motifs, nmotifs, *params, ch);
    });
}

// TEST INFRASTRUCTURE: tredsw_ref_tracts_ex with every kernel body run serially on the host.  Not used by the package.
int tredsw_ref_tracts_emulate_ex(tredsw_ctx *, const char *fasta_path, const tredsw_fai_entry *contigs,
                                 int32_t ncontigs, const tredsw_motif *motifs, int32_t nmotifs,
                                 const tredsw_tract_params *params, const tredsw_tract_chain *chain,
                                 tredsw_tracts **result) {
    TractChain ch;
    if (!tract_args_ok(fasta_path, contigs, ncontigs, motifs, nmotifs, params, result) || !tract_chain_ok(chain, &ch))
        return TREDSW_ERR_ARG;
    return run_entry(nullptr, "tredsw_ref_tracts_emulate", result, [&](auto &be, tredsw_tracts *r) {
        return run_ref_tracts(be, r, fasta_path, contigs, ncontigs, motifs, nmotifs, *params, ch);
    });
}

int tredsw_ref_tracts(tredsw_ctx *ctx, const char *fasta_path, const tredsw_fai_entry *contigs, int32_t ncontigs,
                      const tredsw_motif *motifs, int32_t nmotifs, const tredsw_tract_params *params,
                      tredsw_tracts **result) {
    if (!ctx) { tredsw_set_error("bad arguments"); return TREDSW_ERR_ARG; }
    if (!tract_args_ok(fasta_path, contigs, ncontigs, motifs, nmotifs, params, result)) return TREDSW_ERR_ARG;
    return run_entry(ctx, "tredsw_ref_tracts", result, [&](auto &be, tredsw_tracts *r) {
        return run_ref_tracts(be, r, fasta_path, contigs, ncontigs, motifs, nmotifs, *params, TractChain{0, 1, 1});
    });
}

// TEST INFRASTRUCTURE: tredsw_ref_tracts with every kernel body run serially on the host.  Not used by the package.
int tredsw_ref_tracts_emulate(tredsw_ctx *, const char *fasta_path, const tredsw_fai_entry *contigs, int32_t ncontigs,
                              const tredsw_motif *motifs, int32_t nmotifs, const tredsw_tract_params *params,
                              tredsw_tracts **result) {
    if (!tract_args_ok(fasta_path, contigs, ncontigs, motifs, nmotifs, params, result)) return TREDSW_ERR_ARG;
    return run_entry(nullptr, "tredsw_ref_tracts_emulate", result, [&](auto &be, tredsw_tracts *r) {
        return run_ref_tracts(be, r, fasta_path, contigs, ncontigs, motifs, nmotifs, *params, TractChain{0, 1, 1});
    });
}

int tredsw_ref_tracts_view(const tredsw_tracts *r, tredsw_tracts_view *v) {
    if (!r || !v) { tredsw_set_error("bad arguments"); return TREDSW_ERR_ARG; }
    *v = r->view;
    return TREDSW_OK;
}

void tredsw_ref_tracts_free(tredsw_tracts *r) { delete r; }

}  // extern "C"
