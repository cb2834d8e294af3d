// ref_tracts_device.cuh — per-thread bodies of the reference tract scan (tredsw_ref_tracts, bgzf_gpu.cu; DESIGN §4.5):
// every tract of a requested motif in a plain-text FASTA.
//
// For a period k, a tract comes from a maximal stretch [a, b) of bases in ACGTacgt (compared case-insensitively; N,
// IUPAC codes and anything else break it) with s[j] == s[j + k] for every j in [a, b - k): it is [a, a + c k) with
// c = floor((b - a) / k) copies of the unit s[a, a + k).  It is kept when the unit's primitive root has period k, c >=
// min_units (>= 2), c k >= min_len and the unit's canonical code (canonical_root, shared with the IRR classifier) is
// requested for k.  With c >= 2 such a stretch is exactly a maximal run [a, e) of agreements s[j] == s[j + k] (both
// bases valid), b = e + k, which is what the kernels find.
//
// Like the ingest bodies, everything is __host__ __device__: the kernels run it one thread per item and the serial
// host backend (tredsw_ref_tracts_emulate, test infrastructure) runs the same code.
#pragma once
#include "ingest_device.cuh"
#if defined(__CUDACC__)
#include <cooperative_groups.h>
#endif

namespace tredsw_gi {

struct TractContig {            // one contig of a step
    int64_t length;             // bases
    int64_t text;               // its first base's byte in the step's text buffer
    int64_t word0;              // its first word in the step's code / valid arrays (ceil(length / 32) words)
    int32_t lb, lw;             // bases and bytes of a full line (.fai)
    int32_t id, pad_;           // index among the call's contigs
};
struct TractOut { int64_t start, length; uint64_t code; int32_t contig, period; };     // mirrors tredsw_tract
constexpr uint32_t TRACT_ERR_TEXT = 1u;                 // a base position holds '\n', '\r' or '>'

// a FASTA byte -> 0..3 (A C G T, either case), 4 any other base, -1 a byte no base position may hold
TG_HD int fasta_code(uint8_t c) {
    switch (c | 0x20) {
        case 'a': return 0;
        case 'c': return 1;
        case 'g': return 2;
        case 't': return 3;
        default: return (c == '\n' || c == '\r' || c == '>') ? -1 : 4;
    }
}

// the step contig holding word w (contig c's words are [word0, word0 + ceil(length / 32)))
TG_HD int tract_contig_of(const TractContig *cs, int nc, int64_t w) {
    int lo = 0, hi = nc - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (cs[mid].word0 <= w) lo = mid; else hi = mid - 1;
    }
    return lo;
}

TG_HD int64_t tract_words(int64_t length) { return (length + 31) >> 5; }

// Pack: bases [32 lw, 32 lw + 32) of contig c -> 2-bit codes (base i at bits 2 (i mod 32)) and a valid mask (bit
// i mod 32: the base is one of ACGTacgt).  -> the number of invalid bases; *bad when a position holds a line break or
// a header: the index does not describe the file.
TG_HD int tract_pack_word(const uint8_t *text, const TractContig &c, int64_t lw, uint64_t *code, uint32_t *valid, bool *bad) {
    const int64_t i0 = lw << 5;
    const int n = (int)((c.length - i0) < 32 ? (c.length - i0) : 32);
    int64_t line = i0 / c.lb;
    int col = (int)(i0 - line * c.lb);
    uint64_t cw = 0;
    uint32_t vw = 0;
    int invalid = 0;
    for (int i = 0; i < n; ++i) {
        const int x = fasta_code(text[c.text + line * c.lw + col]);
        if (x < 0) *bad = true;
        if (x >= 0 && x < 4) { cw |= (uint64_t)x << (2 * i); vw |= 1u << i; }
        else ++invalid;
        if (++col == c.lb) { col = 0; ++line; }
    }
    *code = cw; *valid = vw;
    return invalid;
}

// the even bits of x, packed into 32 bits
TG_HD uint32_t compress_even(uint64_t x) {
    x &= 0x5555555555555555ull;
    x = (x | (x >> 1)) & 0x3333333333333333ull;
    x = (x | (x >> 2)) & 0x0f0f0f0f0f0f0f0full;
    x = (x | (x >> 4)) & 0x00ff00ff00ff00ffull;
    x = (x | (x >> 8)) & 0x0000ffff0000ffffull;
    x = (x | (x >> 16)) & 0x00000000ffffffffull;
    return (uint32_t)x;
}

// bit j: s[i] == s[i + k] with both bases valid, i = 32 lw + j, for word lw of a contig of nw words (0 past its end)
TG_HD uint32_t tract_agree(const uint64_t *code, const uint32_t *valid, int64_t word0, int64_t nw, int64_t lw, int k) {
    if (lw >= nw) return 0;
    const uint64_t lo = code[word0 + lw], hi = lw + 1 < nw ? code[word0 + lw + 1] : 0;
    const uint32_t vlo = valid[word0 + lw], vhi = lw + 1 < nw ? valid[word0 + lw + 1] : 0;
    const uint64_t x = lo ^ ((lo >> (2 * k)) | (hi << (64 - 2 * k)));      // 2 <= k <= 20
    return compress_even(~(x | (x >> 1))) & vlo & ((vlo >> k) | (vhi << (32 - k)));
}

TG_HD int ctz32(uint32_t x) {
#if defined(__CUDA_ARCH__)
    return __ffs((int)x) - 1;
#else
    return __builtin_ctz(x);
#endif
}

// appends t (and, with segs, its segment count m at the same index) at a unique index below cap through a
// warp-aggregated counter; the count keeps going past cap, so the caller sees an overflow and runs again with room
// for all
TG_HD void tract_emit(TractOut *out, unsigned long long *count, unsigned long long cap, const TractOut &t,
                      int32_t *segs = nullptr, int32_t m = 1) {
#if defined(__CUDA_ARCH__)
    namespace cg = cooperative_groups;
    const cg::coalesced_group g = cg::coalesced_threads();
    unsigned long long base = 0;
    if (g.thread_rank() == 0) base = atomicAdd(count, (unsigned long long)g.size());
    const unsigned long long at = g.shfl(base, 0) + g.thread_rank();
#else
    const unsigned long long at = (*count)++;
#endif
    if (at < cap) {
        out[at] = t;
        if (segs) segs[at] = m;
    }
}

struct TractQuery {             // what a step looks for
    const int32_t *periods;     // the distinct requested periods
    const int32_t *mfirst;      // codes of periods[p]: mcodes[mfirst[p] .. mfirst[p + 1]), ascending
    const uint64_t *mcodes;
    int32_t nper, min_units;
    int64_t min_len;
};

// The tracts of period q.periods[p] whose agreement run starts in word lw of contig c: each run start walks forward
// word by word to the run's end.
TG_HD void tract_runs(const uint64_t *code, const uint32_t *valid, const TractContig &c, int64_t lw, int p,
                      const TractQuery &q, TractOut *out, unsigned long long *count, unsigned long long cap) {
    const int k = q.periods[p];
    const int64_t nw = tract_words(c.length);
    const uint32_t A = tract_agree(code, valid, c.word0, nw, lw, k);
    if (!A) return;
    const uint32_t carry = lw > 0 ? tract_agree(code, valid, c.word0, nw, lw - 1, k) >> 31 : 0u;
    uint32_t starts = A & ~((A << 1) | carry);
    while (starts) {
        const int j = ctz32(starts);
        starts &= starts - 1;
        const int64_t a = (lw << 5) + j;
        int64_t e;
        const uint32_t z = ~A & (~0u << j);
        if (z) e = (lw << 5) + ctz32(z);
        else {
            int64_t v = lw + 1;
            uint32_t B;
            while ((B = tract_agree(code, valid, c.word0, nw, v, k)) == ~0u) ++v;
            e = (v << 5) + ctz32(~B);
        }
        const int64_t copies = (e + k - a) / k, len = copies * k;
        if (copies < q.min_units || len < q.min_len) continue;
        const int64_t w = a >> 5;
        const int off = (int)(a & 31);
        uint64_t unit = code[c.word0 + w] >> (2 * off);
        if (off && w + 1 < nw) unit |= code[c.word0 + w + 1] << (64 - 2 * off);
        unit &= (1ull << (2 * k)) - 1ull;
        uint64_t canon;
        if (canonical_root(unit, k, &canon) != k) continue;
        int lo = q.mfirst[p], hi = q.mfirst[p + 1];
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (q.mcodes[mid] < canon) lo = mid + 1; else hi = mid;
        }
        if (lo == q.mfirst[p + 1] || q.mcodes[lo] != canon) continue;
        tract_emit(out, count, cap, TractOut{a, len, canon, c.id, k});
    }
}

// ---- interrupted tracts (tredsw_tract_chain; DESIGN §4.5.1) ----------------------------------------------------
// With ag(j) the agreement bit above, a run is a maximal [a, e) of agreements (its bases [a, e + k)) and a segment a
// run with e - a >= k.  A segment S = [a, e) links to T = [a', e'), the next segment after it, when both have root
// period k and one canonical code, a' - (e + k) <= g (a deletion gives 0 or less) and the bases [e + k, a') are all
// in ACGTacgt.  A chain is a maximal sequence of links S1 -> ... -> Sm; it gives the tract [a1, a1 + c k),
// c = floor((em + k - a1) / k), of S1's code and m segments when A den >= num C, C = em - a1 and A the agreements in
// [a1, em); a chain with m >= 2 that fails this falls back to its segments, each judged alone.  Kept tracts pass the
// pure rule's filters.  g <= 20 bounds every look-back and look-ahead to 2 k + g + 1 <= 61 positions.
struct TractChain { int32_t max_interrupt, num, den; };

TG_HD int clz64(uint64_t x) {
#if defined(__CUDA_ARCH__)
    return __clzll((long long)x);
#else
    return __builtin_clzll(x);
#endif
}

// bit i: ag(pos + i), i < 64, for a contig of nw words (0 before its first base and past its end)
TG_HD uint64_t tract_agree64(const uint64_t *code, const uint32_t *valid, int64_t word0, int64_t nw, int64_t pos, int k) {
    const int64_t w = pos >= 0 ? pos >> 5 : -((31 - pos) >> 5);
    const int off = (int)(pos - (w << 5));
    uint32_t x[3];
    for (int i = 0; i < 3; ++i) x[i] = w + i >= 0 ? tract_agree(code, valid, word0, nw, w + i, k) : 0u;
    const uint64_t lo = (uint64_t)x[0] | ((uint64_t)x[1] << 32);
    return off ? (lo >> off) | ((uint64_t)x[2] << (64 - off)) : lo;
}

// the first j >= a with ag(j) == 0
TG_HD int64_t tract_run_end(const uint64_t *code, const uint32_t *valid, int64_t word0, int64_t nw, int64_t a, int k) {
    int64_t v = a >> 5;
    uint32_t z = ~tract_agree(code, valid, word0, nw, v, k) & (~0u << (a & 31));
    while (!z) z = ~tract_agree(code, valid, word0, nw, ++v, k);
    return (v << 5) + ctz32(z);
}

// whether every base of [x, y), y - x <= 32, of the contig is in ACGTacgt (true when y <= x)
TG_HD bool tract_valid_span(const uint32_t *valid, int64_t word0, int64_t nw, int64_t x, int64_t y) {
    if (y <= x) return true;
    const int64_t w = x >> 5;
    const int off = (int)(x & 31), n = (int)(y - x);
    uint64_t v = valid[word0 + w];
    if (w + 1 < nw) v |= (uint64_t)valid[word0 + w + 1] << 32;
    const uint64_t m = (1ull << n) - 1ull;
    return ((v >> off) & m) == m;
}

// the canonical code of the k bases from a when their primitive root has period k, else ~0
TG_HD uint64_t tract_code_at(const uint64_t *code, int64_t word0, int64_t nw, int64_t a, int k) {
    const int64_t w = a >> 5;
    const int off = (int)(a & 31);
    uint64_t unit = code[word0 + w] >> (2 * off);
    if (off && w + 1 < nw) unit |= code[word0 + w + 1] << (64 - 2 * off);
    unit &= (1ull << (2 * k)) - 1ull;
    uint64_t canon;
    return canonical_root(unit, k, &canon) == k ? canon : ~0ull;
}

// The segment S of the chain ending at e (code canon) links to the next segment T: -> T's start a' and, in *gap_agree,
// the agreements in [e, a'); -1 when S ends its chain.
TG_HD int64_t tract_link(const uint64_t *code, const uint32_t *valid, int64_t word0, int64_t nw, int64_t e, int k,
                         int g, uint64_t canon, int *gap_agree) {
    const int n = 2 * k + g;                            // positions [e, e + 2k + g): a' <= e + k + g, then k agreements
    const uint64_t M = tract_agree64(code, valid, word0, nw, e, k) & ((1ull << n) - 1ull);
    uint64_t F = M;                                     // bit i: ag at [i, i + k)
    for (int t = 1; t < k; ++t) F &= M >> t;
    const uint64_t cand = M & ~(M << 1) & F & ((2ull << (k + g)) - 1ull);      // run starts at e + i, i <= k + g
    if (!cand) return -1;
    const int i = (uint32_t)cand ? ctz32((uint32_t)cand) : 32 + ctz32((uint32_t)(cand >> 32));
    const int64_t a2 = e + i;
    if (!tract_valid_span(valid, word0, nw, e + k, a2) || tract_code_at(code, word0, nw, a2, k) != canon) return -1;
    *gap_agree = popc64(M & ((1ull << i) - 1ull));
    return a2;
}

// whether the segment at a (code canon) is linked to from the segment before it: the nearest earlier segment
// [aP, eP) with eP >= a - k - g, when there is one
TG_HD bool tract_linked_back(const uint64_t *code, const uint32_t *valid, int64_t word0, int64_t nw, int64_t a, int k,
                             int g, uint64_t canon) {
    const int n = 2 * k + g + 1;                        // positions [a - n, a): eP - 1 >= a - k - g - 1, then k agreements
    const int64_t lo = a - n;
    const uint64_t M = tract_agree64(code, valid, word0, nw, lo, k) & ((1ull << n) - 1ull);
    uint64_t K = M;                                     // bit i: ag at [i - k + 1, i]
    for (int t = 1; t < k; ++t) K &= M << t;
    const uint64_t cand = M & ~(M >> 1) & K & (~0ull << k);     // run ends eP = lo + i + 1 >= a - k - g (bit n - 1,
    if (!cand) return false;                                    // position a - 1, is 0: a starts a run)
    const int64_t eP = lo + (63 - clz64(cand)) + 1;
    return tract_valid_span(valid, word0, nw, eP + k, a) && tract_code_at(code, word0, nw, eP - k, k) == canon;
}

// The tracts of period q.periods[p] of the chains (tract_chains) whose first segment starts in word lw of contig c:
// each run start that begins a segment of a requested code and is not linked to from the segment before it walks its
// chain forward, hopping each interruption with tract_link, and emits the chain or, when it fails purity, its segments.
TG_HD void tract_chains(const uint64_t *code, const uint32_t *valid, const TractContig &c, int64_t lw, int p,
                        const TractQuery &q, const TractChain &ch, TractOut *out, int32_t *segs,
                        unsigned long long *count, unsigned long long cap) {
    const int k = q.periods[p], g = ch.max_interrupt;
    const int64_t nw = tract_words(c.length);
    const uint32_t A = tract_agree(code, valid, c.word0, nw, lw, k);
    if (!A) return;
    const uint32_t carry = lw > 0 ? tract_agree(code, valid, c.word0, nw, lw - 1, k) >> 31 : 0u;
    uint32_t starts = A & ~((A << 1) | carry);
    const uint64_t km = (1ull << k) - 1ull;
    while (starts) {
        const int j = ctz32(starts);
        starts &= starts - 1;
        const int64_t a = (lw << 5) + j;
        // a segment (k agreements from a) of a requested code, first of its chain
        const uint64_t f = j + k <= 32 ? (uint64_t)(A >> j) : tract_agree64(code, valid, c.word0, nw, a, k);
        if ((f & km) != km) continue;
        const uint64_t canon = tract_code_at(code, c.word0, nw, a, k);
        if (canon == ~0ull) continue;
        int lo = q.mfirst[p], hi = q.mfirst[p + 1];
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (q.mcodes[mid] < canon) lo = mid + 1; else hi = mid;
        }
        if (lo == q.mfirst[p + 1] || q.mcodes[lo] != canon) continue;
        if (tract_linked_back(code, valid, c.word0, nw, a, k, g, canon)) continue;
        // the chain: its last segment's end em, its segments m and its agreements
        int64_t em = tract_run_end(code, valid, c.word0, nw, a, k), agree = em - a;
        int32_t m = 1;
        int gap;
        for (int64_t a2; (a2 = tract_link(code, valid, c.word0, nw, em, k, g, canon, &gap)) >= 0; ++m) {
            em = tract_run_end(code, valid, c.word0, nw, a2, k);
            agree += gap + (em - a2);
        }
        auto emit = [&](int64_t s, int64_t e, int32_t nseg) {
            const int64_t copies = (e + k - s) / k;
            if (copies >= q.min_units && copies * k >= q.min_len)
                tract_emit(out, count, cap, TractOut{s, copies * k, canon, c.id, k}, segs, nseg);
        };
        if (agree * ch.den >= (int64_t)ch.num * (em - a)) { emit(a, em, m); continue; }
        // failed purity (m >= 2: a single segment agrees throughout): its segments, each alone
        for (int64_t s = a;;) {
            const int64_t e = tract_run_end(code, valid, c.word0, nw, s, k);
            emit(s, e, 1);
            if ((s = tract_link(code, valid, c.word0, nw, e, k, g, canon, &gap)) < 0) break;
        }
    }
}

}  // namespace tredsw_gi
