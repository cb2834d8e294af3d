// ingest_device.cuh — per-thread bodies of the GPU BAM ingest (bgzf_gpu.cu): raw-DEFLATE decoding of one BGZF
// block, CRC-32, the BAM record walk of one indexed fetch, per-record selection (reads for Smith-Waterman, pileup
// depth, pair candidates), pairing by query name, and the scatter of the selected reads into the flat buffers
// tredsw_genotype_batch consumes.
//
// Replaces the three pysam passes per locus of the reference — BamParser.parse selection
// (tredparse/bam_parser.py:194-243), PEextractor (:316-369), BamDepth.region_depth (:404-411) — and is, item by
// item, the same rule set as the host reader in ingest.cpp (`extract_locus_impl`, `tredsw_bam::fetch`,
// `read_record`), which the tests use as its oracle.
//
// Every body is `__host__ __device__` and touches memory only through plain loads / stores and the atomic wrappers
// below: the kernels of bgzf_gpu.cu call them with one thread (or one warp: NL = 32 lanes, `lane`) per item, and a
// serial host loop over the same bodies with NL = 1 (tredsw_ingest_batch_emulate: test infrastructure) lets the CPU
// suite check the device logic bit for bit.  Only the warp-level plumbing (shuffles of the CRC tree, the shared-memory
// window of the record walk) is device-only; the GPU tests cover it against the same oracle.
#pragma once
#include <stdint.h>
#include <string.h>

#if defined(__CUDACC__)
#define TG_HD __host__ __device__ __forceinline__
#else
#define TG_HD inline
#endif

// (statistics hooks of an offline tool; empty in the library)
#ifndef TG_STAT_LIT
#define TG_STAT_LIT()
#define TG_STAT_MATCH(len, dist)
#define TG_STAT_DBLOCK()
#endif

namespace tredsw_gi {

// ---- memory helpers ----------------------------------------------------------------------------------------------
TG_HD uint32_t atomic_cas_u32(uint32_t *p, uint32_t cmp, uint32_t val) {
#if defined(__CUDA_ARCH__)
    return atomicCAS(p, cmp, val);
#else
    const uint32_t old = *p; if (old == cmp) *p = val; return old;
#endif
}
TG_HD void atomic_min_u32(uint32_t *p, uint32_t val) {
#if defined(__CUDA_ARCH__)
    atomicMin(p, val);
#else
    if (val < *p) *p = val;
#endif
}
TG_HD void atomic_add_u64(unsigned long long *p, unsigned long long val) {
#if defined(__CUDA_ARCH__)
    atomicAdd(p, val);
#else
    *p += val;
#endif
}
TG_HD void atomic_add_i32(int32_t *p, int32_t val) {
#if defined(__CUDA_ARCH__)
    atomicAdd(p, val);
#else
    *p += val;
#endif
}
TG_HD void atomic_or_u32(uint32_t *p, uint32_t val) {
#if defined(__CUDA_ARCH__)
    atomicOr(p, val);
#else
    *p |= val;
#endif
}

// little-endian 32-bit load at an arbitrary byte offset (the device needs aligned accesses: two words + funnel shift;
// every buffer read this way is allocated with >= 8 bytes of slack behind its end)
TG_HD uint32_t ld_u32(const uint8_t *base, int64_t off) {
#if defined(__CUDA_ARCH__)
    const uint8_t *p = base + off;
    const uintptr_t a = reinterpret_cast<uintptr_t>(p);
    const uint32_t *w = reinterpret_cast<const uint32_t *>(a & ~(uintptr_t)3);
    const unsigned sh = (unsigned)(a & 3u) * 8u;
    const uint32_t lo = w[0];
    if (sh == 0) return lo;
    return __funnelshift_r(lo, w[1], sh);
#else
    uint32_t v; memcpy(&v, base + off, 4); return v;
#endif
}
TG_HD int32_t ld_i32(const uint8_t *base, int64_t off) { return (int32_t)ld_u32(base, off); }
TG_HD uint32_t ld_u16(const uint8_t *base, int64_t off) { return (uint32_t)base[off] | ((uint32_t)base[off + 1] << 8); }

// ---- raw DEFLATE (RFC 1951), one warp (device) / one thread (host) per BGZF block -------------------------------------
// Huffman tables of 16-bit entries, reached through a strided reference: stride 1 on the host, the warp count of the
// CTA on the device (entry i of warp w at [i * stride + w] in shared memory; the lanes of a warp read the same entry).
//   entry: bits 0..3 code bits to consume (sub-table pointer: index bits of the sub-table), bits 4..6 kind,
//          bits 7..15 payload (literal byte, length / distance / code-length symbol, sub-table offset / 2)
struct TabRef {
    uint16_t *p; int stride;
    bool writer;                // the lanes that share a table all compute its entries; one of them stores them
    TG_HD uint32_t get(uint32_t i) const { return p[(size_t)i * stride]; }
    TG_HD void set(uint32_t i, uint32_t v) const { if (writer) p[(size_t)i * stride] = (uint16_t)v; }
};
enum : uint32_t { K_INVALID = 0, K_LITERAL = 1, K_LENGTH = 2, K_END = 3, K_SUB = 4, K_SYMBOL = 5 };
constexpr int LIT_ROOT = 9, DIST_ROOT = 6, PRE_ROOT = 7;
// worst-case table sizes of a complete code (zlib's ENOUGH: 852 for 286 symbols / 9 root bits, 592 for 30 / 6)
constexpr int LIT_CAP = 864, DIST_CAP = 608, PRE_CAP = 128;
constexpr int TAB_ENTRIES = LIT_CAP + DIST_CAP + PRE_CAP;          // 16-bit entries per thread: 3200 bytes

TG_HD uint32_t mk_entry(uint32_t kind, uint32_t payload, uint32_t bits) { return bits | (kind << 4) | (payload << 7); }

// which: 0 literal / length alphabet, 1 distance alphabet, 2 code-length alphabet
TG_HD bool build_table(const uint8_t *lens, int nsyms, int which, const TabRef &tab, int root_bits, int cap,
                       uint8_t *sub_need /* 1 << root_bits bytes of scratch */, uint16_t *sub_base /* likewise, 16-bit */) {
    int count[16];
    for (int l = 0; l < 16; ++l) count[l] = 0;
    for (int s = 0; s < nsyms; ++s) { if (lens[s] > 15) return false; ++count[lens[s]]; }
    count[0] = 0;
    int left = 1;                                     // over-subscribed codes are rejected, incomplete ones allowed
    for (int l = 1; l <= 15; ++l) { left <<= 1; left -= count[l]; if (left < 0) return false; }
    uint32_t first_code[16];
    uint32_t code = 0;
    first_code[0] = 0;
    for (int l = 1; l <= 15; ++l) { code = (code + (uint32_t)count[l - 1]) << 1; first_code[l] = code; }
    const int root_size = 1 << root_bits;
    for (int i = 0; i < root_size; ++i) { tab.set(i, 0); sub_need[i] = 0; }
    auto reversed = [](uint32_t c, int l) -> uint32_t {
#if defined(__CUDA_ARCH__)
        return __brev(c) >> (32 - l);
#else
        uint32_t r = 0; for (int b = 0; b < l; ++b) { r = (r << 1) | (c & 1u); c >>= 1; } return r;
#endif
    };
    // pass 1: longest code behind every root prefix
    uint32_t next_code[16];
    for (int l = 0; l < 16; ++l) next_code[l] = first_code[l];
    for (int s = 0; s < nsyms; ++s) {
        const int l = lens[s];
        if (l <= root_bits) { if (l) ++next_code[l]; continue; }
        const uint32_t r = reversed(next_code[l]++, l);
        const uint32_t prefix = r & (uint32_t)(root_size - 1);
        if (l - root_bits > sub_need[prefix]) sub_need[prefix] = (uint8_t)(l - root_bits);
    }
    int top = root_size;
    for (int prefix = 0; prefix < root_size; ++prefix) {
        if (!sub_need[prefix]) continue;
        const int size = 1 << sub_need[prefix];
        if (top + size > cap) return false;
        tab.set(prefix, mk_entry(K_SUB, (uint32_t)top >> 1, sub_need[prefix]));    // (top is even: sizes are powers of two)
        sub_base[prefix] = (uint16_t)top;
        for (int i = 0; i < size; ++i) tab.set(top + i, 0);
        top += size;
    }
    // pass 2: fill
    for (int l = 0; l < 16; ++l) next_code[l] = first_code[l];
    for (int s = 0; s < nsyms; ++s) {
        const int l = lens[s];
        if (!l) continue;
        const uint32_t r = reversed(next_code[l]++, l);
        uint32_t kind, payload;
        if (which == 0) {
            if (s < 256) { kind = K_LITERAL; payload = (uint32_t)s; }
            else if (s == 256) { kind = K_END; payload = 0; }
            else if (s <= 285) { kind = K_LENGTH; payload = (uint32_t)(s - 257); }
            else { kind = K_INVALID; payload = 0; }              // 286, 287: never valid in a stream
        } else if (which == 1) {
            if (s < 30) { kind = K_SYMBOL; payload = (uint32_t)s; } else { kind = K_INVALID; payload = 0; }
        } else { kind = K_SYMBOL; payload = (uint32_t)s; }
        if (l <= root_bits) {
            const uint32_t e = kind == K_INVALID ? 0u : mk_entry(kind, payload, (uint32_t)l);
            for (uint32_t i = r; i < (uint32_t)root_size; i += 1u << l) tab.set(i, e);
        } else {
            const uint32_t prefix = r & (uint32_t)(root_size - 1);
            if (!sub_need[prefix]) return false;
            const uint32_t base = sub_base[prefix], sub_bits = sub_need[prefix], rem = (uint32_t)(l - root_bits);
            const uint32_t e = kind == K_INVALID ? 0u : mk_entry(kind, payload, rem);
            for (uint32_t i = r >> root_bits; i < (1u << sub_bits); i += 1u << rem) tab.set(base + i, e);
        }
    }
    return true;
}

// LSB-first bit reader over aligned 32-bit words (the compressed bytes may start at any address).  A valid stream
// reads at most 7 bytes behind the end of its input; a corrupt one is stopped by overrun() at the next symbol, by
// when it may have read up to 16 bytes behind it — the buffers are allocated with that slack; the bytes are never used
struct BitReader {
    const uint32_t *w0, *w, *wlimit;
    uint64_t buf; int cnt; int mis;
    TG_HD void init(const uint8_t *in, int64_t in_len) {
        const uintptr_t a = reinterpret_cast<uintptr_t>(in);
        mis = (int)(a & 3u);
        w0 = reinterpret_cast<const uint32_t *>(a - (uintptr_t)mis);
        w = w0;
        wlimit = w0 + (in_len + mis + 3) / 4 + 2;
        buf = (uint64_t)(*w++) >> (8 * mis);
        cnt = 32 - 8 * mis;
    }
    TG_HD void refill() { if (cnt <= 32) { buf |= (uint64_t)(*w++) << cnt; cnt += 32; } }      // >= 33 bits afterwards
    TG_HD uint32_t peek(int n) const { return (uint32_t)buf & ((1u << n) - 1u); }              // n <= 16
    TG_HD void drop(int n) { buf >>= n; cnt -= n; }
    TG_HD uint32_t take(int n) { const uint32_t v = peek(n); drop(n); return v; }
    TG_HD int64_t bytes_consumed() const {                // whole bytes of the input the decoder has moved past
        const int64_t bits = (int64_t)(w - w0) * 32 - 8 * mis - cnt;
        return (bits + 7) / 8;
    }
    TG_HD bool overrun() const { return w > wlimit; }
};

// Barrier + memory ordering among the NL lanes that decode one block together (a warp on the device, nothing on the host)
template <int NL> TG_HD void lanes_sync() {
#if defined(__CUDA_ARCH__)
    if (NL > 1) __syncwarp();
#endif
}
// a byte the lanes of this warp wrote earlier (read past the non-coherent L1)
TG_HD uint8_t ld_written(const uint8_t *p) {
#if defined(__CUDA_ARCH__)
    return __ldcg(p);
#else
    return *p;
#endif
}

// Inflate the raw DEFLATE stream in[0, in_len) to exactly out_len bytes.  `tabs` holds TAB_ENTRIES entries
// (literal / length table, distance table, code-length table); lens / sub_need are per-thread scratch.
// NL lanes (1 on the host, the 32 lanes of a warp on the device) decode ONE block together: the Huffman decoding is
// inherently serial, so every lane runs it redundantly on the same bits (uniform control flow, broadcast loads: free
// in SIMT) — what the lanes share is the copying: lane 0 stores the literals, and the bytes of a match (or a stored
// block) are dealt to the lanes, so that a match costs one memory round trip whatever its length.  An overlapping
// match (distance < length) is a repetition of its first `distance` bytes, which lie before the match: every byte
// of it can be fetched independently.
template <int NL>
TG_HD bool inflate_block(const uint8_t *in, int64_t in_len, uint8_t *out, int64_t out_len, const TabRef &tabs,
                         uint8_t *lens /* 320 */, uint8_t *sub_need /* 512 */, uint16_t *sub_base /* 512 */, int lane) {
    const TabRef lit = tabs, dist = TabRef{tabs.p + (size_t)LIT_CAP * tabs.stride, tabs.stride, tabs.writer},
                 pre = TabRef{tabs.p + (size_t)(LIT_CAP + DIST_CAP) * tabs.stride, tabs.stride, tabs.writer};
    BitReader br;
    br.init(in, in_len);
    int64_t op = 0;
    for (;;) {
        br.refill();
        const uint32_t bfinal = br.take(1), btype = br.take(2);
        if (btype == 0) {
            // stored: skip to the byte boundary, LEN / NLEN, then raw bytes straight from the input
            br.drop(br.cnt & 7);
            br.refill();
            const uint32_t len = br.take(16);
            br.refill();
            const uint32_t nlen = br.take(16);
            if ((len ^ 0xffffu) != nlen) return false;
            const int64_t at = br.bytes_consumed();             // (the bit position is a byte boundary here)
            if (at + (int64_t)len > in_len || (int64_t)len > out_len - op) return false;
            for (uint32_t i = (uint32_t)lane; i < len; i += NL) out[op + i] = in[at + i];
            op += len;
            br.init(in + at + len, in_len - at - len);
            // (init re-bases the byte accounting: keep `in` consistent with it)
            in += at + len; in_len -= at + len;
        } else if (btype == 1 || btype == 2) {
            int nlit, ndist;
            if (btype == 1) {
                for (int i = 0; i < 144; ++i) lens[i] = 8;
                for (int i = 144; i < 256; ++i) lens[i] = 9;
                for (int i = 256; i < 280; ++i) lens[i] = 7;
                for (int i = 280; i < 288; ++i) lens[i] = 8;
                for (int i = 288; i < 320; ++i) lens[i] = 5;
                nlit = 288; ndist = 32;
            } else {
                nlit = (int)br.take(5) + 257; ndist = (int)br.take(5) + 1;
                const int npre = (int)br.take(4) + 4;
                if (nlit > 286 || ndist > 30) return false;
                uint8_t plens[19];
                for (int i = 0; i < 19; ++i) plens[i] = 0;
                for (int i = 0; i < npre; ++i) {
                    br.refill();
                    // order of the code-length code lengths: 16 17 18 0 8 7 9 6 10 5 11 4 12 3 13 2 14 1 15
                    int o;
                    if (i < 3) o = 16 + i;
                    else if (i == 3) o = 0;
                    else if ((i & 1) == 0) o = 8 + ((i - 4) >> 1);          // i = 4, 6, 8 ... -> 8, 9, 10, ...
                    else o = 7 - ((i - 5) >> 1);                            // i = 5, 7, 9 ... -> 7, 6, 5, ...
                    plens[o] = (uint8_t)br.take(3);
                }
                lanes_sync<NL>();                                  // nobody still reads the previous block's tables
                if (!build_table(plens, 19, 2, pre, PRE_ROOT, PRE_CAP, sub_need, sub_base)) return false;
                lanes_sync<NL>();
                int i = 0;
                while (i < nlit + ndist) {
                    if (br.overrun()) return false;
                    br.refill();
                    const uint32_t e = pre.get(br.peek(PRE_ROOT));
                    if (((e >> 4) & 7u) != K_SYMBOL) return false;
                    br.drop((int)(e & 15u));
                    const uint32_t sym = e >> 7;
                    if (sym < 16) { lens[i++] = (uint8_t)sym; continue; }
                    int rep; uint8_t v = 0;
                    if (sym == 16) { if (i == 0) return false; v = lens[i - 1]; rep = 3 + (int)br.take(2); }
                    else if (sym == 17) rep = 3 + (int)br.take(3);
                    else rep = 11 + (int)br.take(7);
                    if (i + rep > nlit + ndist) return false;
                    while (rep--) lens[i++] = v;
                }
                if (lens[256] == 0) return false;                 // no end-of-block code
                // distance lengths behind a fixed offset (288), the gaps zeroed
                for (int k = ndist - 1; k >= 0; --k) lens[288 + k] = lens[nlit + k];
                for (int k = nlit; k < 288; ++k) lens[k] = 0;
                for (int k = 288 + ndist; k < 320; ++k) lens[k] = 0;
                nlit = 288; ndist = 32;
            }
            TG_STAT_DBLOCK();
            lanes_sync<NL>();
            if (!build_table(lens, nlit, 0, lit, LIT_ROOT, LIT_CAP, sub_need, sub_base)) return false;
            if (!build_table(lens + 288, ndist, 1, dist, DIST_ROOT, DIST_CAP, sub_need, sub_base)) return false;
            lanes_sync<NL>();                                      // the tables are visible to every lane
            for (;;) {
                if (br.overrun()) return false;
                br.refill();                                      // >= 33 bits: code 15 + extra 5
                uint32_t e = lit.get(br.peek(LIT_ROOT));
                if (((e >> 4) & 7u) == K_SUB) {
                    br.drop(LIT_ROOT);
                    e = lit.get(((e >> 7) << 1) + br.peek((int)(e & 15u)));
                }
                br.drop((int)(e & 15u));
                const uint32_t kind = (e >> 4) & 7u, pay = e >> 7;
                if (kind == K_LITERAL) {
                    if (op >= out_len) return false;
                    if (lane == 0) out[op] = (uint8_t)pay;
                    ++op;
                    TG_STAT_LIT();
                    continue;
                }
                if (kind == K_END) break;
                if (kind != K_LENGTH) return false;
                uint32_t length;
                if (pay < 8) length = 3 + pay;
                else if (pay == 28) length = 258;
                else { const int eb = (int)(pay >> 2) - 1; length = ((4 + (pay & 3u)) << eb) + 3 + br.take(eb); }
                br.refill();                                      // code 15 + extra 13
                uint32_t d = dist.get(br.peek(DIST_ROOT));
                if (((d >> 4) & 7u) == K_SUB) {
                    br.drop(DIST_ROOT);
                    d = dist.get(((d >> 7) << 1) + br.peek((int)(d & 15u)));
                }
                if (((d >> 4) & 7u) != K_SYMBOL) return false;
                br.drop((int)(d & 15u));
                const uint32_t ds = d >> 7;
                uint32_t distance;
                if (ds < 4) distance = 1 + ds;
                else { const int eb = (int)(ds >> 1) - 1; distance = ((2 + (ds & 1u)) << eb) + 1 + br.take(eb); }
                if ((int64_t)distance > op || (int64_t)length > out_len - op) return false;
                TG_STAT_MATCH(length, distance);
                uint8_t *dst = out + op;
                const uint8_t *src = dst - distance;
                lanes_sync<NL>();                                  // the bytes before `op` are visible to every lane
                for (uint32_t k = (uint32_t)lane; k < length; k += NL)
                    dst[k] = ld_written(src + (k < distance ? k : k % distance));
                op += length;
            }
        } else {
            return false;
        }
        if (bfinal) break;
    }
    lanes_sync<NL>();
    return op == out_len && br.bytes_consumed() <= in_len;
}

// CRC-32 (IEEE, reflected, as in gzip) by four tables; `t` points to 4 x 256 words
TG_HD uint32_t crc32_bytes(const uint32_t *t, const uint8_t *p, int64_t n) {
    uint32_t c = 0xffffffffu;
    int64_t i = 0;
    for (; i < n && (reinterpret_cast<uintptr_t>(p + i) & 3u); ++i) c = t[(c ^ p[i]) & 0xffu] ^ (c >> 8);
    for (; i + 4 <= n; i += 4) {
        c ^= *reinterpret_cast<const uint32_t *>(p + i);
        c = t[768 + (c & 0xffu)] ^ t[512 + ((c >> 8) & 0xffu)] ^ t[256 + ((c >> 16) & 0xffu)] ^ t[c >> 24];
    }
    for (; i < n; ++i) c = t[(c ^ p[i]) & 0xffu] ^ (c >> 8);
    return c ^ 0xffffffffu;
}

// CRC-32 of a block by NL lanes: every lane takes a contiguous segment (lane 0 the first n - (NL-1) * (n / NL) bytes,
// the others n / NL bytes each), and the segment CRCs are combined with zlib's crc32_combine identity
//     crc(A || B) = x^(8 |B|) * crc(A) + crc(B)     (polynomials over GF(2) modulo the CRC polynomial, reflected)
// in a tree: at level k the right-hand operand of every pair is 2^k whole segments long.
TG_HD uint32_t crc_multmodp(uint32_t a, uint32_t b) {          // a != 0
    uint32_t m = 1u << 31, p = 0;
    for (;;) {
        if (a & m) { p ^= b; if ((a & (m - 1u)) == 0) break; }
        m >>= 1;
        b = (b & 1u) ? (b >> 1) ^ 0xedb88320u : b >> 1;
    }
    return p;
}
TG_HD uint32_t crc_x8n_modp(uint64_t n) {                     // x^(8 n)
    uint32_t sq = 0x40000000u;                                  // x^1
    for (int k = 0; k < 3; ++k) sq = crc_multmodp(sq, sq);      // x^8
    uint32_t p = 1u << 31;                                      // x^0
    while (n) { if (n & 1u) p = crc_multmodp(sq, p); n >>= 1; if (n) sq = crc_multmodp(sq, sq); }
    return p;
}
template <int NL>
TG_HD void crc_segment(int64_t n, int lane, int64_t *begin, int64_t *len) {
    const int64_t L = n / NL, first = n - (NL - 1) * L;
    *begin = lane == 0 ? 0 : first + (int64_t)(lane - 1) * L;
    *len = lane == 0 ? first : L;
}
// serial form of the tree (host / tests): parts[i] = CRC of lane i's segment
template <int NL>
TG_HD uint32_t crc_fold_serial(uint32_t *parts, int64_t n) {
    uint32_t op = crc_x8n_modp((uint64_t)(n / NL));
    for (int s = 1; s < NL; s <<= 1) {
        for (int i = 0; i + s < NL; i += 2 * s) parts[i] = crc_multmodp(op, parts[i]) ^ parts[i + s];
        op = crc_multmodp(op, op);
    }
    return parts[0];
}
#if defined(__CUDACC__)
__device__ __forceinline__ uint32_t crc32_warp(const uint32_t *t, const uint8_t *p, int64_t n, int lane) {
    int64_t b, len;
    crc_segment<32>(n, lane, &b, &len);
    uint32_t c = crc32_bytes(t, p + b, len);
    uint32_t op = crc_x8n_modp((uint64_t)(n / 32));
#pragma unroll
    for (int s = 1; s < 32; s <<= 1) {
        const uint32_t q = __shfl_down_sync(0xffffffffu, c, s);
        if ((lane & (2 * s - 1)) == 0) c = crc_multmodp(op, c) ^ q;
        op = crc_multmodp(op, op);
    }
    return __shfl_sync(0xffffffffu, c, 0);
}
#endif

// ---- batch description (host-built, read-only on the device) ----------------------------------------------------------
struct BlockDesc {              // one BGZF block of the batch
    int64_t in_off;             // compressed payload (raw DEFLATE) in the staging buffer
    int64_t out_off;            // inflated bytes in ibuf; consecutive file blocks are contiguous
    uint32_t clen, isize, crc, pad_;
};
struct Chunk {                  // one merged BAI chunk of a fetch, as positions in ibuf
    int64_t begin, end;         // records are read while position < end
    int64_t run_end;            // end of the contiguous run of loaded blocks the chunk lies in
};
struct Fetch {                  // one indexed region query (tredsw_bam::fetch)
    int32_t problem;            // owning (sample, locus) problem
    int32_t kind;               // 0: the locus window, 1: an alt region
    int32_t tid;
    int32_t chunk_begin, chunk_end;
    int32_t pad_;
    int64_t start, end;         // [start, end) on tid
};
struct ProblemParams {          // windows of one locus (extract_locus_impl)
    int32_t tid, span;
    int64_t win_s, win_e, read_s, read_e, pe_s, pe_e, tstart, tend;
};
struct ProblemCounts {          // accumulated by the record kernel
    unsigned long long depth_sum;
    unsigned long long bytes64; // selected bases + name bytes in 64 bits: guards the 32-bit scans against a wrap
    int32_t n_unmapped;
    uint32_t error;             // bit 0 walk (record chain), bit 1 record fields
};
constexpr int32_t MAX_SELECTED_READ = 1 << 20;      // a "read" longer than this is a corrupt record, not evidence

enum : uint32_t { ERR_WALK = 1u, ERR_RECORD = 2u };

// ---- record walk of one fetch ----------------------------------------------------------------------------------------
// Follows the record chain of every chunk of the fetch exactly like tredsw_bam::fetch (ingest_internal.h) and calls
// sink(position) for every record that fetch would parse and hand to its overlap test.  Returns false when the chain
// leaves the loaded bytes or a block_size is implausible (corrupt file / index): the caller flags the problem.
// The chain is one dependent load per record, and the inflated bytes of a batch do not fit the L2: read through
// `Reader`, which on the device is a 4 KB window of the record stream in shared memory that the 32 lanes of a warp
// refill together (one memory round trip per ~12 records instead of one per record); every lane follows the chain
// redundantly on the same bytes (uniform control flow).  On the host the reader loads directly.
struct DirectReader {
    const uint8_t *ibuf;
    TG_HD void head(int64_t p, int32_t *bs, int32_t *tid, int32_t *pos) { *bs = ld_i32(ibuf, p); *tid = ld_i32(ibuf, p + 4); *pos = ld_i32(ibuf, p + 8); }
};
constexpr int WALK_WINDOW = 4096;                    // bytes per warp
#if defined(__CUDACC__)
struct WindowReader {
    const uint8_t *ibuf; int64_t ibuf_len;           // (allocated length, a multiple of 16)
    uint32_t *win; int lane; int64_t base;
    __device__ __forceinline__ void refill(int64_t p) {
        base = p & ~(int64_t)15;
        __syncwarp();
#pragma unroll
        for (int k = 0; k < WALK_WINDOW / 512; ++k) {
            const int64_t a = base + 16 * (lane + 32 * k);
            uint4 v = make_uint4(0u, 0u, 0u, 0u);
            if (a + 16 <= ibuf_len) v = *reinterpret_cast<const uint4 *>(ibuf + a);
            reinterpret_cast<uint4 *>(win)[lane + 32 * k] = v;
        }
        __syncwarp();
    }
    __device__ __forceinline__ uint32_t word(int64_t p) const {      // 32 bits at byte p (inside the window)
        const int o = (int)(p - base);
        const uint32_t lo = win[o >> 2];
        const unsigned sh = (unsigned)(o & 3) * 8u;
        return sh ? __funnelshift_r(lo, win[(o >> 2) + 1], sh) : lo;
    }
    __device__ __forceinline__ void head(int64_t p, int32_t *bs, int32_t *tid, int32_t *pos) {
        if (p < base || p + 16 > base + WALK_WINDOW) refill(p);
        *bs = (int32_t)word(p); *tid = (int32_t)word(p + 4); *pos = (int32_t)word(p + 8);
    }
};
#endif

template <class Reader, class Sink>
TG_HD bool walk_fetch(Reader &rd, const Fetch &f, const Chunk *chunks, Sink &&sink) {
    for (int c = f.chunk_begin; c < f.chunk_end; ++c) {
        int64_t p = chunks[c].begin;
        const int64_t end = chunks[c].end, run_end = chunks[c].run_end;
        while (p < end) {
            if (p + 12 > run_end) return false;
            int32_t bs, tid, pos;
            rd.head(p, &bs, &tid, &pos);
            if (bs < 32 || bs > (64 << 20) || p + 4 + (int64_t)bs > run_end) return false;
            const int64_t here = p;
            p += 4 + (int64_t)bs;
            if (tid != f.tid) { if (tid >= 0 && tid < f.tid) continue; return true; }
            if ((int64_t)pos >= f.end) return true;
            sink(here);
        }
    }
    return true;
}
// one warp (device) / one thread (host) per fetch; `win`: WALK_WINDOW bytes of shared memory of this warp
template <class Sink>
TG_HD bool walk_fetch_lanes(const uint8_t *ibuf, int64_t ibuf_len, const Fetch &f, const Chunk *chunks, int lane,
                            uint32_t *win, Sink &&sink) {
#if defined(__CUDA_ARCH__)
    WindowReader rd{ibuf, ibuf_len, win, lane, (int64_t)-(1ll << 40)};
    return walk_fetch(rd, f, chunks, sink);
#else
    (void)ibuf_len; (void)lane; (void)win;
    DirectReader rd{ibuf};
    return walk_fetch(rd, f, chunks, sink);
#endif
}

// ---- one record ----------------------------------------------------------------------------------------------------
struct RecOut {                 // per walked record
    uint32_t emit;              // 1: the read goes to Smith-Waterman
    uint32_t bases;             // l_seq when emitted
    uint32_t name_bytes;        // bytes of its NUL-terminated name when emitted
    uint32_t pe;                // 1: candidate of the pair extractor
};
struct Mate { int32_t pos, ref_end, qstart, qend, l_seq, reverse; };

struct RecFields {
    int32_t tid, pos, l_name, n_cigar, flag, l_seq, next_tid, next_pos;
    int32_t ref_len, qstart, qend;
    bool has_cigar, ok;
};
TG_HD RecFields parse_record(const uint8_t *ibuf, int64_t p) {
    RecFields r;
    const int32_t bs = ld_i32(ibuf, p);
    const int64_t d = p + 4;
    r.tid = ld_i32(ibuf, d); r.pos = ld_i32(ibuf, d + 4);
    r.l_name = ibuf[d + 8];
    r.n_cigar = (int32_t)ld_u16(ibuf, d + 12);
    r.flag = (int32_t)ld_u16(ibuf, d + 14);
    r.l_seq = ld_i32(ibuf, d + 16); r.next_tid = ld_i32(ibuf, d + 20); r.next_pos = ld_i32(ibuf, d + 24);
    r.ok = !(r.l_seq < 0 || 32LL + r.l_name + 4LL * r.n_cigar + ((int64_t)r.l_seq + 1) / 2 + r.l_seq > (int64_t)bs);
    r.ref_len = 0; r.has_cigar = r.n_cigar > 0; r.qstart = 0; r.qend = r.l_seq;
    if (!r.ok) return r;
    const int64_t cg = d + 32 + r.l_name;
    int qs = 0, qe = r.l_seq;
    bool lead = true;
    for (int k = 0; k < r.n_cigar; ++k) {
        const uint32_t c = ld_u32(ibuf, cg + 4 * k);
        const int op = (int)(c & 15u), len = (int)(c >> 4);
        if (op == 0 || op == 2 || op == 3 || op == 7 || op == 8) r.ref_len += len;       // M D N = X
        if (lead) { if (op == 4) qs += len; else if (op != 5) lead = false; }
    }
    for (int k = r.n_cigar - 1; k >= 0; --k) {
        const uint32_t c = ld_u32(ibuf, cg + 4 * k);
        const int op = (int)(c & 15u), len = (int)(c >> 4);
        if (op == 4) qe -= len; else if (op != 5) break;
    }
    r.qstart = qs; r.qend = qe;
    return r;
}

// the per-record rules of extract_locus_impl (main window) and of its alt-region loop
TG_HD RecOut select_record(const uint8_t *ibuf, int64_t p, const Fetch &f, const ProblemParams &q, ProblemCounts *cnt,
                           Mate *mate) {
    RecOut o; o.emit = 0; o.bases = 0; o.name_bytes = 0; o.pe = 0;
    const RecFields r = parse_record(ibuf, p);
    if (!r.ok) { atomic_or_u32(&cnt->error, ERR_RECORD); return o; }
    int64_t rend = (int64_t)r.pos + r.ref_len;
    const bool unmapped = (r.flag & 4) != 0;
    if (unmapped || !r.has_cigar || rend <= r.pos) rend = (int64_t)r.pos + 1;
    if (!(r.pos < f.end && rend > f.start)) return o;               // fetch's own overlap test
    bool emit = false;
    if (f.kind == 0) {
        if (r.pos < q.win_e && rend > q.win_s) {
            if (unmapped) { atomic_add_i32(&cnt->n_unmapped, 1); emit = true; }
            else if (r.pos >= q.read_s && r.pos <= q.read_e) emit = true;
            if (!(r.flag & (4 | 256 | 512 | 1024)) && r.has_cigar) atomic_add_u64(&cnt->depth_sum, (unsigned long long)r.ref_len);
        }
        if (r.pos < q.pe_e && rend > q.pe_s && (r.flag & 1) && !unmapped && !(r.flag & 1024)) {
            o.pe = 1;
            mate->pos = r.pos; mate->ref_end = (!r.has_cigar) ? -1 : r.pos + r.ref_len;
            mate->qstart = r.qstart; mate->qend = r.qend; mate->l_seq = r.l_seq; mate->reverse = (r.flag & 16) != 0;
        }
    } else {
        emit = r.next_tid == q.tid && (int64_t)r.next_pos >= q.win_s && (int64_t)r.next_pos <= q.win_e;
    }
    if (emit && r.l_seq > MAX_SELECTED_READ) { atomic_or_u32(&cnt->error, ERR_RECORD); emit = false; }
    if (emit) {
        o.emit = 1; o.bases = (uint32_t)r.l_seq; o.name_bytes = (uint32_t)(r.l_name > 0 ? r.l_name : 1);
        atomic_add_u64(&cnt->bytes64, (unsigned long long)o.bases + o.name_bytes);
    }
    return o;
}

// base codes of an emitted read (A,C,G,T,N -> 0..4 from the 4-bit "=ACMGRSVTWYHKDBN") and its NUL-terminated name
TG_HD int8_t nib_code(uint32_t nib) {
    // {4, 0, 1, 4, 2, 4, 4, 4, 3, 4, ...}: only 1, 2, 4, 8 are bases
    return nib == 1 ? 0 : nib == 2 ? 1 : nib == 4 ? 2 : nib == 8 ? 3 : 4;
}
TG_HD void emit_read(const uint8_t *ibuf, int64_t p, int8_t *rbuf_at, char *name_at, int lane, int nlanes) {
    const int64_t d = p + 4;
    const int l_name = ibuf[d + 8];
    const int n_cigar = (int)ld_u16(ibuf, d + 12);
    const int l_seq = ld_i32(ibuf, d + 16);
    const uint8_t *seq = ibuf + d + 32 + l_name + 4 * (int64_t)n_cigar;
    for (int i = lane; i < l_seq; i += nlanes) rbuf_at[i] = nib_code((seq[i >> 1] >> ((i & 1) ? 0 : 4)) & 15u);
    if (name_at) {
        const int n = l_name > 0 ? l_name - 1 : 0;
        for (int i = lane; i < n; i += nlanes) name_at[i] = (char)ibuf[d + 32 + i];
        if (lane == 0) name_at[n] = 0;
    }
}

// ---- pairing by query name (PEextractor, bam_parser.py:316-369; ingest.cpp: slot / pairs / npair) -----------------------
// Per problem an open-addressing table in global memory: rep = record that claimed the slot (its name is the key),
// first / second = the two smallest record indices carrying that name.
constexpr uint32_t EMPTY = 0xffffffffu;
TG_HD int name_len(const uint8_t *ibuf, int64_t p) { const int l = ibuf[p + 12]; return l > 0 ? l - 1 : 0; }
TG_HD bool same_name(const uint8_t *ibuf, int64_t pa, int64_t pb) {
    const int la = name_len(ibuf, pa), lb = name_len(ibuf, pb);
    if (la != lb) return false;
    for (int i = 0; i < la; ++i) if (ibuf[pa + 36 + i] != ibuf[pb + 36 + i]) return false;
    // (std::string keys built with assign(ptr, n): embedded NULs are part of the key on the host path as well)
    return true;
}
TG_HD uint32_t name_hash(const uint8_t *ibuf, int64_t p) {
    const int n = name_len(ibuf, p);
    uint32_t h = 2166136261u;
    for (int i = 0; i < n; ++i) { h ^= ibuf[p + 36 + i]; h *= 16777619u; }
    h ^= h >> 15; h *= 0x2c1b3c6du; h ^= h >> 12;
    return h;
}
// step 1: find / claim the slot of record i (index into the walked-record arrays), note the smallest index per name
TG_HD uint32_t pair_insert(const uint8_t *ibuf, const int64_t *rec_pos, uint32_t i, uint32_t *rep, uint32_t *first,
                           uint32_t mask) {
    const int64_t p = rec_pos[i];
    uint32_t s = name_hash(ibuf, p) & mask;
    for (;;) {
        const uint32_t old = atomic_cas_u32(&rep[s], EMPTY, i);
        if (old == EMPTY || old == i || same_name(ibuf, rec_pos[old], p)) break;
        s = (s + 1) & mask;
    }
    atomic_min_u32(&first[s], i);
    return s;
}
// step 3: the pair whose first record is x and second y -> 0 none, 1 global, 2 target; *tlen its distance
TG_HD int pair_eval(const Mate &x, const Mate &y, const ProblemParams &q, int32_t *tlen_out) {
    if (!(!x.reverse && y.reverse)) return 0;
    int64_t s = x.pos, e = y.ref_end;
    if (x.qstart > 0) s -= x.qstart;
    if (y.qend < y.l_seq) e += y.l_seq - y.qend;
    const int64_t tlen = e - s;
    if (tlen >= q.span) return 0;
    *tlen_out = (int32_t)tlen;
    return (x.pos < q.tstart && y.ref_end > q.tend) ? 2 : 1;
}

// ---- scan of a BAM without an index (tredsw_ingest_scan_run) ---------------------------------------------------------
// A slab of the file is inflated into one stream: the carry (the bytes of the last record of the previous slab that was
// not complete there) followed by the slab's blocks.  Nothing says where a record starts inside a block, so:
//   1. candidate: the first offset of every block where a record header passes a strict predicate, and so do the next
//      two records of the chain it starts (one warp per block, 32 offsets per step);
//   2. landing: from its candidate, the chain (block_size only) to the first record at or after the block's end;
//   3. the true start of block 0 is known (after the header / the carry); wherever a block's landing equals the next
//      block's candidate, that candidate is a true record start, by induction.  Where they differ, the landing is the
//      true start and the chain is walked again from it (scan_repair_run, on the few such blocks).
// Every record position the later steps use therefore comes from a chain that starts at a known record.
constexpr int64_t SCAN_NONE = -1;           // no candidate in the block
constexpr int64_t SCAN_BAD = -2;            // the chain met an implausible block_size: corrupt records
struct ScanBlock { int64_t begin, end; };   // a block's bytes in the slab stream (block 0 includes the carry)

// strict record predicate at p (offsets relative to the stream s[0, len)); *bs: its block_size
TG_HD bool scan_plausible(const uint8_t *s, int64_t len, int64_t p, int32_t n_ref, int32_t *bs) {
    if (p + 36 > len) return false;
    const int32_t b = ld_i32(s, p), tid = ld_i32(s, p + 4), pos = ld_i32(s, p + 8), l_seq = ld_i32(s, p + 20);
    const int32_t next_tid = ld_i32(s, p + 24);
    const int l_name = s[p + 12];
    const int n_cigar = (int)ld_u16(s, p + 16);
    if (b < 33 || b > (64 << 20)) return false;
    if (tid < -1 || tid >= n_ref || next_tid < -1 || next_tid >= n_ref || pos < -1) return false;
    if (l_name < 1 || l_seq < 0 || p + 36 + l_name > len || s[p + 35 + l_name] != 0) return false;
    if (32LL + l_name + 4LL * n_cigar + ((int64_t)l_seq + 1) / 2 + l_seq > (int64_t)b) return false;
    *bs = b;
    return true;
}
// p passes the predicate, and so do the next two records of its chain as far as they lie in the stream
TG_HD bool scan_candidate_ok(const uint8_t *s, int64_t len, int64_t p, int32_t n_ref) {
    for (int k = 0; k < 3; ++k) {
        if (k > 0 && p + 36 > len) return true;
        int32_t bs;
        if (!scan_plausible(s, len, p, n_ref, &bs)) return false;
        p += 4 + (int64_t)bs;
    }
    return true;
}
// first offset of [begin, end) that passes scan_candidate_ok, or SCAN_NONE; NL lanes test NL consecutive offsets a step
template <int NL>
TG_HD int64_t scan_find_candidate(const uint8_t *s, int64_t len, int64_t begin, int64_t end, int32_t n_ref, int lane) {
    for (int64_t o0 = begin; o0 < end; o0 += NL) {
        const int64_t o = o0 + lane;
        const bool ok = o < end && scan_candidate_ok(s, len, o, n_ref);
#if defined(__CUDA_ARCH__)
        const uint32_t m = __ballot_sync(0xffffffffu, ok);
        if (m) return o0 + __ffs(m) - 1;
#else
        if (ok) return o;
#endif
    }
    return SCAN_NONE;
}
// Follows the chain from the record at p to the first record at or after `end`.  Stops early at a record that is not
// complete in the stream (it is carried into the next slab) and returns its start; SCAN_BAD at an implausible size.
TG_HD int64_t scan_chain(const uint8_t *s, int64_t len, int64_t p, int64_t end) {
    while (p < end) {
        if (p + 4 > len) return p;
        const int32_t bs = ld_i32(s, p);
        if (bs < 32 || bs > (64 << 20)) return SCAN_BAD;
        if (p + 4 + (int64_t)bs > len) return p;
        p += 4 + (int64_t)bs;
    }
    return p;
}
// Where the chain entering block b at `tf` stands relative to the block's candidate: true when the block needs no walk
// from tf (no record starts in it, or its candidate is tf and so its landing is right).
TG_HD bool scan_agrees(const ScanBlock &blk, int64_t cand, int64_t tf) {
    return tf < blk.begin || tf >= blk.end || cand == tf;
}
// The repair of a run of blocks whose candidates were wrong: walk from the true start tf of block b on, block after
// block, until the chain agrees with a block's candidate again.  land[k] receives the true landing of every block
// walked; returns the first block not walked.
TG_HD int scan_repair_run(const uint8_t *s, int64_t len, const ScanBlock *blk, const int64_t *cand, int nblocks, int b,
                          int64_t tf, int64_t *land) {
    for (;;) {
        tf = scan_chain(s, len, tf, blk[b].end);
        land[b] = tf;
        ++b;
        if (b >= nblocks || tf == SCAN_BAD || scan_agrees(blk[b], cand[b], tf)) return b;
    }
}
// records that start in a block: from its true first record, while they start before the block's end and are complete
template <class F>
TG_HD void scan_block_records(const uint8_t *s, int64_t len, int64_t p, int64_t end, F &&f) {
    while (p < end && p + 4 <= len) {
        const int64_t next = p + 4 + (int64_t)ld_i32(s, p);
        if (next > len) return;
        f(p);
        p = next;
    }
}

// Records -> fetches.  A record [pos, rend) belongs to a fetch [start, end) of its contig when pos < end and
// rend > start (tredsw_bam::fetch).  The fetches of a scan (locus windows, alt regions, then depth regions: ids >=
// nfetch) are cut, per contig, into elementary segments between consecutive fetch boundaries; segment j =
// [xs[j], xs[j + 1]) lists the fetches that cover it.  A record meets every fetch that covers a segment it overlaps; a
// fetch is reported once, at the first such segment (the record's first segment, or the one where the fetch starts).
// (A fetch with end <= start holds the records that contain [end - 1, start + 1): it is listed on [end - 1, end) and
// the rule above is checked for every fetch reported.)
struct MatchTables {
    const int32_t *tid_x0;      // n_ref + 1: contig t owns xs[tid_x0[t], tid_x0[t + 1])
    const int64_t *xs;          // segment boundaries
    const int32_t *seg_f0;      // segment j lists seg_ids[seg_f0[j], seg_f0[j + 1])
    const int32_t *seg_ids;
    const int64_t *id_lo;       // first boundary of every fetch / depth region in xs
    const int64_t *id_start, *id_end;
    int32_t n_ref, nfetch;
};
template <class F>
TG_HD void scan_matches(const MatchTables &m, int32_t tid, int64_t pos, int64_t rend, F &&f) {
    if (tid < 0 || tid >= m.n_ref) return;
    const int k0 = m.tid_x0[tid], k1 = m.tid_x0[tid + 1];
    int lo = k0, hi = k1;                                   // first boundary > pos
    while (lo < hi) { const int mid = (lo + hi) >> 1; if (m.xs[mid] <= pos) lo = mid + 1; else hi = mid; }
    const int j0 = lo > k0 ? lo - 1 : k0;
    for (int j = j0; j < k1 - 1 && m.xs[j] < rend; ++j)
        for (int e = m.seg_f0[j]; e < m.seg_f0[j + 1]; ++e) {
            const int32_t id = m.seg_ids[e];
            if ((j == j0 || m.id_lo[id] >= m.xs[j]) && pos < m.id_end[id] && rend > m.id_start[id]) f(id);
        }
}
// the overlap interval of a record as tredsw_bam::fetch tests it
TG_HD int64_t record_fetch_end(const RecFields &r) {
    int64_t rend = (int64_t)r.pos + r.ref_len;
    if ((r.flag & 4) || !r.has_cigar || rend <= r.pos) rend = (int64_t)r.pos + 1;
    return rend;
}
TG_HD int64_t order_key(int32_t tid, int32_t pos) {         // coordinate order: unmapped records (tid -1) last
    return ((int64_t)(tid < 0 ? 0x7fffffff : tid) << 32) + ((int64_t)pos + 1);
}
enum : uint32_t { SCAN_ERR_RECORD = 1u, SCAN_ERR_ORDER = 2u };
// per record: matched fetches (depth regions are summed here, with the pileup filter of select_record), order check
TG_HD uint32_t scan_record(const uint8_t *s, const int64_t *rec_pos, int64_t i, int64_t prev_key, const MatchTables &m,
                           unsigned long long *depth_sum, uint32_t *err) {
    const int64_t p = rec_pos[i];
    const RecFields r = parse_record(s, p);
    if (!r.ok) { atomic_or_u32(err, SCAN_ERR_RECORD); return 0; }
    const int64_t before = i ? order_key(ld_i32(s, rec_pos[i - 1] + 4), ld_i32(s, rec_pos[i - 1] + 8)) : prev_key;
    if (order_key(r.tid, r.pos) < before) atomic_or_u32(err, SCAN_ERR_ORDER);
    uint32_t n = 0;
    const bool counted = !(r.flag & (4 | 256 | 512 | 1024)) && r.has_cigar;
    scan_matches(m, r.tid, r.pos, record_fetch_end(r), [&](int32_t id) {
        if (id < m.nfetch) ++n;
        else if (counted) atomic_add_u64(&depth_sum[id - m.nfetch], (unsigned long long)r.ref_len);
    });
    return n;
}

// ---- in-repeat reads: the STR profile of a scan (tredsw_ingest_scan_run_ex, DESIGN §4.5) ---------------------------
// A read is an in-repeat read (IRR) when, for some period k in [min_period, max_period], the bases k apart agree (N
// never agrees) on at least num / den of its L - k comparisons; the smallest such k is its period.  Its motif is the
// per-phase majority base, reduced to its primitive root (a root of one base is a homopolymer: not an IRR), in the
// canonical form: the smallest rotation of the root and of its reverse complement, 2 bits a base, first base in the
// most significant bits.  All integer arithmetic: the kernel, the host hook and the Python oracle agree bit for bit.
struct IrrParams { int32_t min_period, max_period, num, den, min_read_len; };
struct IrrEntry {               // one IRR record (tredsw_irr_entry)
    int32_t tid, pos, next_tid, next_pos;
    int32_t flag, mapq, mq, period;     // mq: the MQ:i tag, -1 without one
    uint64_t motif;
    int64_t name_off;
    int32_t name_len, mate;             // mate: filled by the host join (index of the mate's entry, -1 none)
};
enum : int { IRR_CONSIDERED = 0, IRR_DEPTH_BASES = 1, IRR_MAX_LSEQ = 2, IRR_UNPARSED_AUX = 3, IRR_NSTATS = 4 };
constexpr uint32_t IRR_SKIP_FLAGS = 0x100u | 0x200u | 0x400u | 0x800u;      // secondary, QC fail, duplicate, supplementary

struct PackedSeq {              // base i of a record's 4-bit sequence as a code 0..4 (A C G T, anything else N)
    const uint8_t *p;
    TG_HD int operator()(int i) const { return nib_code((p[i >> 1] >> ((i & 1) ? 0 : 4)) & 15u); }
};
struct CodeSeq {                // a sequence of codes (the host test hook)
    const int8_t *p;
    TG_HD int operator()(int i) const { const int c = p[i]; return (c >= 0 && c < 4) ? c : 4; }
};

TG_HD int popc64(uint64_t x) {
#if defined(__CUDA_ARCH__)
    return __popcll(x);
#else
    return __builtin_popcountll(x);
#endif
}

// -> the period of the IRR (0: not one); *motif its canonical motif
template <class Seq>
TG_HD int irr_classify(const Seq &sq, int L, const IrrParams &pr, uint64_t *motif) {
    *motif = 0;
    if (L < pr.min_read_len) return 0;                  // (min_read_len >= 2 max_period: L - k >= k for every k)
    // Prefilter: the first W <= 64 bases as 2-bit codes (base i at bits 2i) and their N flags (bit 2i).  The
    // disagreements of period k among the first W - k comparisons are counted at once (shift, xor, popcount); they are
    // a subset of the read's, so more than the allowance rejects k exactly.  Most reads are rejected here at every k
    // from one pass over 32 bytes instead of per-period walks over the sequence.
    const int W = L < 64 ? L : 64;
    unsigned __int128 codes = 0, nflag = 0;
    for (int i = 0; i < W; ++i) {
        const int a = sq(i);
        if (a == 4) nflag |= (unsigned __int128)1 << (2 * i);
        else codes |= (unsigned __int128)a << (2 * i);
    }
    const unsigned __int128 low = ((unsigned __int128)0x5555555555555555ull << 64) | 0x5555555555555555ull;
    int P = 0;
    for (int k = pr.min_period; k <= pr.max_period; ++k) {
        const int n = L - k;
        const int64_t need = ((int64_t)pr.num * n + pr.den - 1) / pr.den;    // ceil(num n / den) agreements
        const int64_t allow = n - need;                  // disagreements a passing read can have: exact early exit
        {
            const unsigned __int128 d = codes ^ (codes >> (2 * k));
            const unsigned __int128 window = ((unsigned __int128)1 << (2 * (W - k))) - 1;      // comparisons i < W - k
            const unsigned __int128 mis = (d | (d >> 1) | nflag | (nflag >> (2 * k))) & low & window;
            if (popc64((uint64_t)mis) + popc64((uint64_t)(mis >> 64)) > allow) continue;
        }
        int64_t miss = 0;
        int i = 0;
        for (; i < n; ++i) {
            const int a = sq(i);
            if ((a == 4 || a != sq(i + k)) && ++miss > allow) break;
        }
        if (i == n) { P = k; break; }
    }
    if (!P) return 0;
    uint64_t cons = 0;                                  // phase j's majority base at bits 2j
    for (int j = 0; j < P; ++j) {
        int c0 = 0, c1 = 0, c2 = 0, c3 = 0;
        for (int i = j; i < L; i += P) {
            const int a = sq(i);
            c0 += a == 0; c1 += a == 1; c2 += a == 2; c3 += a == 3;
        }
        int best = 0, bc = c0;                          // ties: the smallest code; all N: A
        if (c1 > bc) { best = 1; bc = c1; }
        if (c2 > bc) { best = 2; bc = c2; }
        if (c3 > bc) { best = 3; }
        cons |= (uint64_t)best << (2 * j);
    }
    int d = P;                                          // primitive root: the smallest period that divides P
    for (int e = 1; e < P; ++e) {
        if (P % e) continue;
        bool rep = true;
        for (int i = e; i < P && rep; ++i) rep = ((cons >> (2 * i)) & 3u) == ((cons >> (2 * (i - e))) & 3u);
        if (rep) { d = e; break; }
    }
    if (d == 1) return 0;                               // homopolymer
    uint64_t f = 0, r = 0;
    for (int i = 0; i < d; ++i) f = (f << 2) | ((cons >> (2 * i)) & 3u);
    for (int i = d - 1; i >= 0; --i) r = (r << 2) | (3u - ((cons >> (2 * i)) & 3u));
    const uint64_t mask = (1ull << (2 * d)) - 1ull;
    uint64_t best = f < r ? f : r;
    for (int t = 1; t < d; ++t) {                       // the other rotations, one base to the left at a time
        f = ((f << 2) | (f >> (2 * d - 2))) & mask;
        r = ((r << 2) | (r >> (2 * d - 2))) & mask;
        if (f < best) best = f;
        if (r < best) best = r;
    }
    *motif = best;
    return d;
}

// The MQ tag of the aux area [a, end): its value (negative values read as 0), -1 when there is none.  Only the integer
// types c C s S i I count; A Z H B f fields are skipped.  An area the walk cannot parse (a field running past the end,
// an unknown type) is "no MQ" and sets *unparsed.
TG_HD int32_t aux_mq(const uint8_t *s, int64_t a, int64_t end, bool *unparsed) {
    *unparsed = false;
    while (a < end) {
        if (a + 3 > end) { *unparsed = true; return -1; }
        const bool mq = s[a] == 'M' && s[a + 1] == 'Q';
        const uint8_t t = s[a + 2];
        a += 3;
        int size = 0;
        if (t == 'A' || t == 'c' || t == 'C') size = 1;
        else if (t == 's' || t == 'S') size = 2;
        else if (t == 'i' || t == 'I' || t == 'f') size = 4;
        if (size) {
            if (a + size > end) { *unparsed = true; return -1; }
            if (mq && t != 'A' && t != 'f') {
                int64_t v;
                if (t == 'c') v = (int8_t)s[a];
                else if (t == 'C') v = s[a];
                else if (t == 's') v = (int16_t)ld_u16(s, a);
                else if (t == 'S') v = ld_u16(s, a);
                else if (t == 'i') v = ld_i32(s, a);
                else v = ld_u32(s, a);
                return v < 0 ? 0 : v > 0x7fffffff ? 0x7fffffff : (int32_t)v;
            }
            a += size;
        } else if (t == 'Z' || t == 'H') {
            while (a < end && s[a] != 0) ++a;
            if (a >= end) { *unparsed = true; return -1; }
            ++a;
        } else if (t == 'B') {
            if (a + 5 > end) { *unparsed = true; return -1; }
            const uint8_t st = s[a];
            const int es = (st == 'c' || st == 'C') ? 1 : (st == 's' || st == 'S') ? 2 : (st == 'i' || st == 'I' || st == 'f') ? 4 : 0;
            const int64_t cnt = ld_u32(s, a + 1);
            if (!es || a + 5 + cnt * es > end) { *unparsed = true; return -1; }
            a += 5 + cnt * es;
        } else {
            *unparsed = true; return -1;
        }
    }
    return -1;
}

// where a record's sequence and aux area lie (it passed parse_record)
TG_HD int64_t record_seq(int64_t p, const RecFields &r) { return p + 36 + r.l_name + 4 * (int64_t)r.n_cigar; }
TG_HD int64_t record_aux(int64_t p, const RecFields &r) { return record_seq(p, r) + ((int64_t)r.l_seq + 1) / 2 + r.l_seq; }

// sum / max over the lanes that call it together, one atomic per warp (every record of a slab adds its depth bases)
TG_HD void warp_add_u64(unsigned long long *p, uint32_t v) {
#if defined(__CUDA_ARCH__)
    const unsigned m = __activemask();
    const uint32_t t = __reduce_add_sync(m, v);
    if ((threadIdx.x & 31u) == (unsigned)(__ffs(m) - 1) && t) atomicAdd(p, (unsigned long long)t);
#else
    *p += v;
#endif
}
TG_HD void warp_max_u64(unsigned long long *p, uint32_t v) {
#if defined(__CUDA_ARCH__)
    const unsigned m = __activemask();
    const uint32_t t = __reduce_max_sync(m, v);
    if ((threadIdx.x & 31u) == (unsigned)(__ffs(m) - 1) && t) atomicMax(p, (unsigned long long)t);
#else
    if (v > *p) *p = v;
#endif
}

// per record of a scan: the profile's counters; -> its IRR period (0: not an IRR) and motif
TG_HD int scan_irr_record(const uint8_t *s, int64_t p, const IrrParams &pr, unsigned long long *stats, uint64_t *motif,
                          RecFields *fields) {
    const RecFields r = parse_record(s, p);
    *fields = r;
    const bool primary = r.ok && !(r.flag & IRR_SKIP_FLAGS);
    const bool considered = primary && r.l_seq >= pr.min_read_len;
    warp_add_u64(&stats[IRR_CONSIDERED], considered ? 1u : 0u);
    warp_add_u64(&stats[IRR_DEPTH_BASES], primary && !(r.flag & 4) ? (uint32_t)r.l_seq : 0u);
    warp_max_u64(&stats[IRR_MAX_LSEQ], primary ? (uint32_t)r.l_seq : 0u);
    *motif = 0;
    if (!considered) return 0;
    return irr_classify(PackedSeq{s + record_seq(p, r)}, r.l_seq, pr, motif);
}

}  // namespace tredsw_gi
