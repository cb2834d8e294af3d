// sw_family.cu — the production Smith-Waterman path: every read of a locus against the whole template
// family of that locus (prefix + repeat*u + suffix and reverse complements, u = 1..max_units), with the
// reference's post-filter, classification and per-read arg-max fused in.
//
// Replaces, for a whole batch of (sample, locus) problems, the loop
//     for read: for (units, target, ssw) in db: ssw.align(...) ; classify ; max(res)
// of tredparse/bam_parser.py:123-182 over src/ssw_wrap.py:177-227 over src/ssw.c:780-871.
//
// Stage 0 (prefilter_kernel): an exact q-gram bound drops the reads that cannot reach min_score against
//   any template of their family (about half of a locus window) before any DP is done.
//
// Mapping of the DP (classify_kernel): one warp = 32 surviving reads of the same family, one thread = one
// read; persistent single-warp CTAs pull such items from a counter.  Every lane walks the same template
// columns at the same time, so template bases are warp-uniform; query bases are per lane.  Reads that the
// pre-filter shows to have candidates on one strand only run two per thread (64 per warp), see phase 1.
//
// Phase 1 (scores of all 2*max_units templates), all packed int16x2 = forward template | reverse complement
// of one read, or read a | read b on one strand:
//   * the templates of a family are nested — prefix + repeat*u is a prefix of prefix + repeat*(u+1) — so
//     the main DP (prefix + repeat*max_units) runs once, in 12-column strips held in registers (previous-
//     row H and running F per column), two query rows in flight; the H/E column between strips lives in
//     this CTA's global scratch slot (L2), requested two iterations ahead;
//   * the suffix of every template is NOT recomputed: a backward DP of the read against the suffix block
//     (suffix_pass, once per read) yields "potentials" A[j], B[j] with which the best score inside the
//     suffix block of template u is max_j(H_u(j-1) + A[j], E_u(j) + B[j]) — two add-max per row and unit,
//     hooked into the main strips where a unit ends.
//   ssw's outputs only depend on column maxima / first-maximum positions, so this is exact.
// Phase 2 (positions, rounds over candidates in the reference's arg-max order: score desc, units asc,
//   forward before reverse complement): the running main maximum after every unit tells which strip (or
//   the suffix block) holds the end cell; that strip is recomputed warp-uniformly with per-column keys
//   H << 8 | 255 - row (locate_packed); the begin cell comes from a reverse pass per lane — a diagonal walk
//   when no gap is affordable, else a scalar sweep banded by the gap budget; then the reference's filter +
//   tag rules.  The first candidate that yields a tag is the read's result — the same result as classifying
//   all 2*max_units alignments and taking max(key=(score, -units)).
#include "internal.cuh"
#include "sw_sweep.cuh"
#include <type_traits>
#include <algorithm>
#include <vector>
#ifdef TREDSW_DEBUG
#include <assert.h>
#endif

namespace {

constexpr int FAM_W2 = 16;         // strip width of the scalar phase-2 sweeps
constexpr int FLANK = 18;          // flank length of the fast path (all catalogue loci)
// Strand class of a read that reaches the DP, from the q-gram pre-filter: templates of both strands may score
// >= 30, or only forward / only reverse-complement ones.  Only families of the packed kernel get the single-strand
// classes; two single-strand reads share a lane there (read a | read b as s16x2 halves).
constexpr int CLASS_BOTH = 0, CLASS_FWD = 1, CLASS_RC = 2, NCLASS = 3;

struct FamilySmem {
    int8_t prefix[32], suffix[32], repeat[32];
    int Lp, Ls, P, U, clip;
};

struct ClassifyParams {
    const int8_t *rbuf; const int64_t *roff;
    const int32_t *order;          // read indices grouped by (family, strand class): group f * NCLASS + class
    const int32_t *grp_start;      // [ngroups+1] offsets into order
    const int32_t *chunk_start;    // [ngroups+1] offsets into the item (warp-chunk) list, groups in grp_perm order
    const int32_t *grp_perm;       // [ngroups] groups sorted by period: CTAs that run at the same time mostly
                                   // share one instantiation of the strip loops (instruction cache)
    const tredsw_family *families;
    int ngroups;
    int go, ge;
    int max_rows;
    int allow_fast;                // scores fit the 8-bit boundary column (max_read_len * match < 256)
    int match;                     // largest entry of the substitution matrix (band bounds)
    int max_u;                     // largest max_units of the batch (stride of score_buf)
    uint16_t *score_buf;           // [CTAs][2*max_u][32] per-template scores (u8 in the fast kernel)
    uint32_t *pot_buf;             // [CTAs][max_rows+2][32] suffix potentials of the CTA's current item
    uint32_t *gbnd_buf;            // [CTAs][nslots][max_rows+2][32] boundary column entering every main strip
    int nslots;
    uint32_t one;                  // == 1, opaque to the compiler: keeps x = Hdiag * one + S an IMAD (FMA pipe)
    int32_t *counter;              // [2] work counters (generic, fast), zeroed before the launches
    int32_t *out;
    unsigned long long *stats;     // 4 counters
    int strip_skip;                // phase1_packed stops at the fixed point of the strip boundary
    unsigned long long *skip_stats;  // [TREDSW_STRIP_SKIP_STATS] context counters (tredsw_strip_skip_stats)
};

__constant__ int8_t c_fmat25[25];

// Base codes of one read, one byte per base at an arbitrary byte address: the unaligned head byte by byte, the body
// with 16-byte loads (LDG.128), then the tail — f(j, code) is called for j = 0..m-1 in order.
template <class F>
__device__ __forceinline__ void for_each_base(const int8_t *s, int m, F f) {
    int j = 0;
    const int head = min(m, (int)((16u - (unsigned)(reinterpret_cast<uintptr_t>(s) & 15u)) & 15u));
    for (; j < head; ++j) f(j, (int)s[j]);
    for (; j + 16 <= m; j += 16) {
        const uint4 w = __ldg(reinterpret_cast<const uint4 *>(s + j));
        const uint32_t v[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
        for (int k = 0; k < 16; ++k) f(j + k, (int)(int8_t)((v[k >> 2] >> ((k & 3) * 8)) & 0xffu));
    }
    for (; j < m; ++j) f(j, (int)s[j]);
}


__device__ __forceinline__ int fam_code(const FamilySmem &F, int u, int strand, int n, int i) {
    int k = strand ? (n - 1 - i) : i;
    int c;
    if (k < F.Lp) c = F.prefix[k];
    else if (k < F.Lp + F.P * u) c = F.repeat[(k - F.Lp) % F.P];
    else c = F.suffix[k - F.Lp - F.P * u];
    return strand ? (c < 4 ? 3 - c : c) : c;
}

// ---------------------------------------------------------------------------------------------------
// Phase 1, generic: one scalar sweep per template.  Any flank length / period.  Used when the family
// does not fit the packed fast path, and as an on-device cross-check of it.
// ---------------------------------------------------------------------------------------------------
__device__ void phase1_generic(const FamilySmem &F, const SwLut *lut, const uint8_t *codes, int lane,
                               int m, int m_warp, uint32_t *bnd, uint16_t *scores, int go, int ge,
                               unsigned long long &cells) {
    auto rc = [&](int j) { return j < m ? (int)codes[j * 32 + lane] : SW_CODE_GHOST; };
    for (int rank = 0; rank < 2 * F.U; ++rank) {
        const int u = rank / 2 + 1, s = rank & 1;
        const int n = F.Lp + F.Ls + F.P * u;
        auto cc = [&](int i) { return fam_code(F, u, s, n, i); };
        int dc, dr;
        int score = sw_sweep<FAM_W2, 0, false>(m, m, n, rc, cc, lut, bnd + lane, 32, go, ge, 0, &dc, &dr, nullptr);
        scores[rank * 32 + lane] = (uint16_t)min(score, 65535);
        cells += (unsigned long long)m * n;
    }
}

// ---------------------------------------------------------------------------------------------------
// Phase 1, fast: nested strips, two half-strands packed as s16x2.
// Requires Lp == Ls == FLANK and scores < 256 (8-bit boundary column).
// An item's lanes hold either one read with the forward template in the low half and the reverse
// complement in the high half ("both" class), or two reads a | b on the same strand (the pre-filter
// proved the other strand of each has no candidate): the half-strands (sa, sb) are warp-uniform.
// The query side of a row is the PAIR CODE qa * 6 + qb of the two halves' base codes (qa == qb for
// "both" items); the score tables have one row per pair code.
// Boundary word per row and lane: H_a | H_b << 8 | E_a << 16 | E_b << 24.
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t sel2(int ta, int tb) {   // PRMT selector: sign-extended bytes -> s16x2
    return (uint32_t)ta | ((uint32_t)(8 | ta) << 4) | ((uint32_t)tb << 8) | ((uint32_t)(8 | tb) << 12);
}
constexpr int NPAIR = 36;                         // pair codes (6 query codes per half)
constexpr int PAIR_GHOST = SW_CODE_GHOST * 7;     // pair code of a row past the end of both halves
// own base code of half h (0: a, 1: b) of a pair code; for "both" items (code 7q) either decode gives q
__device__ __forceinline__ int pair_half(int code, int h) { return h ? code % 6 : code / 6; }

// template bases on strand s (1 = reverse complement: prefix' = rc(suffix), repeat' = rc(repeat), suffix' = rc(prefix))
__device__ __forceinline__ int comp_code(int c) { return c < 4 ? 3 - c : c; }
__device__ __forceinline__ int pre_base(const FamilySmem &F, int s, int c) { return s ? comp_code(F.suffix[FLANK - 1 - c]) : F.prefix[c]; }
__device__ __forceinline__ int rep_base(const FamilySmem &F, int s, int c) { return s ? comp_code(F.repeat[F.P - 1 - c]) : F.repeat[c]; }
__device__ __forceinline__ int suf_base(const FamilySmem &F, int s, int c) { return s ? comp_code(F.prefix[FLANK - 1 - c]) : F.suffix[c]; }

// One DP cell for both strands (packed s16x2), all operands in registers.  Four integer-pipe instructions:
//     E~ = E + go, F~ = F + go (gap states stored biased by the opening cost, never clamped: E~ >= H >= 0)
//     S  = substitution score + go (table), so that x = Hdiag + S >= 0 in both halves and the add cannot
//          borrow across them: it is issued as an IMAD (x = Hdiag * one + S) on the otherwise idle FMA pipe
//     y  = max(x, E~, F~)                       VIMNMX3
//     H  = max(y - go, 0)                       VIADDMNMX.RELU
//     E~ = max(E~ - ge, H), F~ likewise         VIADDMNMX x 2
// which is H = max(0, Hdiag + s, E, F), E' = max(E - ge, H - go), F' = max(F - ge, H - go).
#define PACKED_CELL(HD, E, S, C, HOUT)                                                        \
    {                                                                                         \
        const uint32_t x_ = HD * one + S;                                                     \
        const uint32_t y_ = __vimax3_s16x2(x_, E, Fv[C]);                                     \
        HOUT = __viaddmax_s16x2_relu(y_, mgo2, mgo2);   /* (third operand: any value <= 0) */ \
        HD = Hrow[C];                                                                         \
        Hrow[C] = HOUT;                                                                       \
        E = __viaddmax_s16x2(E, mge2, HOUT);                                                  \
        Fv[C] = __viaddmax_s16x2(Fv[C], mge2, HOUT);                                          \
    }

constexpr int STAB_PAD = 20;       // words per query-code row of the score table: >= the widest strip (FLANK), a
                                   // multiple of 4 (16-byte rows for LDS.128) and an odd number of 16-byte groups, so
                                   // that 8 consecutive rows start in all 8 bank groups (vector loads of lanes on
                                   // different rows conflict as little as the row count allows)

// Columns per main strip: K whole repeat units, about 12 columns.  Measured on B200 (period 3): 30 columns
// 9.29 ms, 24: 9.06, 18: 8.94, 12: 8.66 per 11,520-problem step — the fully unrolled two-row loop body must
// stay well inside the 6 KB L0 instruction cache; the extra boundary traffic of narrow strips is cheap.
__host__ __device__ constexpr int strip_units(int P) { return P >= 12 ? 1 : 12 / P; }
// The strip loops are instantiated per period PI; a family whose period is G * PI (G = 2, 4) runs through the
// PI instantiation with "sub-units" of PI columns — the hooks of every G-th sub-unit are its real units.
// Fewer distinct loop bodies run at the same time (25 of the 30 catalogue loci have period 3, three more 6
// or 12): they compete for the instruction cache, see DESIGN.md.
__host__ __device__ constexpr int instance_period(int P) { return P == 6 ? 3 : P; }

// One pass over all query rows of a strip of NC template columns made of K = NC / PER units of PER
// columns (previous-row H and running F of every strip column in registers).  Two rows are in flight per
// iteration, skewed by one column (row j at column s, row j+1 at column s-1): two independent dependency
// chains for the scheduler.  Substitution scores of both halves come from a per-strip table in shared
// memory indexed by the pair code (row, per lane) and the strip column (uniform): vector LDS on the
// otherwise idle LSU pipe instead of one PRMT per cell on the saturated integer pipe.
//
//   seg[u]  running maximum of H over the columns of unit u (all rows)
//   mu[u]   (HOOK) best score of any path that leaves unit u's last column into the template's SUFFIX
//           block, by the suffix potentials of this read (see suffix_pass): for every row j
//               mu[u] = max(mu[u], H(j-1, last) + A[j], E(j, last -> next) + B[j])
//           — 2 add-max per row and unit instead of a forked DP over the suffix columns.
//   bin     (HAS_IN) boundary column entering the strip, bout (HAS_OUT) the one leaving it: H | E~ << 16 as
//           bytes per half, one word per row and lane in this CTA's global scratch (L1/L2 resident,
//           requested one iteration ahead); every strip keeps its own slot, phase 2 restarts from them
//   pot     suffix potentials of this warp's reads in global scratch, one word per row and lane
//   diff    (HAS_IN and HAS_OUT) OR of bout ^ bin over the lane's rows: 0 when the strip left exactly the column it
//           received, so that every later strip of the same table would repeat it (phase1_packed's fixed point)
template <int NC, int PER, bool HAS_IN, bool HAS_OUT, bool HOOK>
__device__ __forceinline__ void strip_pass(const uint32_t *stab, const uint8_t *codes, int lane, int m, int rows2,
                                           const uint32_t *bin, uint32_t *bout, const uint32_t *pot,
                                           uint32_t (&seg)[NC / PER], uint32_t (&mu)[NC / PER], uint32_t mgo2,
                                           uint32_t mge2, uint32_t one, uint32_t &diff) {
    constexpr int K = NC / PER;
    static_assert(K * PER == NC, "strip = whole units");
    constexpr int NG = (NC + 3) / 4;
    uint32_t Hrow[NC], Fv[NC], pend[K];
#pragma unroll
    for (int c = 0; c < NC; ++c) { Hrow[c] = 0; Fv[c] = 0; }
#pragma unroll
    for (int u = 0; u < K; ++u) pend[u] = 0;
    uint32_t hin_prev = 0;
    auto code_at = [&](int j) { return j < m ? (int)codes[j * 32 + lane] : PAIR_GHOST; };
    auto row_of = [&](int code) { return reinterpret_cast<const uint4 *>(stab + code * STAB_PAD); };
    // software pipeline: shared-memory operands of row j are requested one iteration ahead, the global ones
    // (boundary column, potentials: L2 latency) two iterations ahead
    const uint4 *rowA = row_of(code_at(0)), *rowB = row_of(code_at(1));
    uint4 gA = rowA[0], gB = rowB[0];
    uint32_t bA = 0, bB = 0, pA = 0, pB = 0, bA2 = 0, bB2 = 0, pA2 = 0, pB2 = 0;
    const int j1 = min(2, rows2 - 2);
    if (HAS_IN) { bA = bin[lane]; bB = bin[32 + lane]; bA2 = bin[j1 * 32 + lane]; bB2 = bin[(j1 + 1) * 32 + lane]; }
    if (HOOK) { pA = pot[lane]; pB = pot[32 + lane]; pA2 = pot[j1 * 32 + lane]; pB2 = pot[(j1 + 1) * 32 + lane]; }
    int codeA2 = code_at(2), codeB2 = code_at(3);
    for (int j = 0; j < rows2; j += 2) {
        uint32_t hinA = 0, eA = 0, hinB = 0, eB = 0;
        if (HAS_IN) {
            hinA = sw_prmt(bA, 0, 0x4140); eA = sw_prmt(bA, 0, 0x4342);     // bytes -> s16x2 halves
            hinB = sw_prmt(bB, 0, 0x4140); eB = sw_prmt(bB, 0, 0x4342);
        }
        uint32_t potHA = 0, potEA = 0, potHB = 0, potEB = 0;
        if (HOOK) {                                                          // signed bytes -> s16x2 halves
            potHA = sw_prmt(pA, 0, 0x9180); potEA = sw_prmt(pA, 0, 0xb3a2);
            potHB = sw_prmt(pB, 0, 0x9180); potEB = sw_prmt(pB, 0, 0xb3a2);
        }
        // requests for the rows after next (indices clamped; unused past the end)
        const int jn = min(j + 4, rows2 - 2);
        const uint4 *rowA2 = row_of(codeA2), *rowB2 = row_of(codeB2);
        uint32_t bA3 = 0, bB3 = 0, pA3 = 0, pB3 = 0;
        if (HAS_IN) { bA3 = bin[jn * 32 + lane]; bB3 = bin[(jn + 1) * 32 + lane]; }
        if (HOOK) { pA3 = pot[jn * 32 + lane]; pB3 = pot[(jn + 1) * 32 + lane]; }
        const int codeA3 = code_at(j + 4), codeB3 = code_at(j + 5);
        uint32_t sA[NG * 4], sB[NG * 4];
        sA[0] = gA.x; sA[1] = gA.y; sA[2] = gA.z; sA[3] = gA.w;
        sB[0] = gB.x; sB[1] = gB.y; sB[2] = gB.z; sB[3] = gB.w;
        uint32_t hdA = hin_prev, hdB = hinA;
        hin_prev = hinB;
        uint32_t hA = 0, hB = 0;
#pragma unroll
        for (int s = 0; s <= NC; ++s) {
            // table groups are requested one group (4 columns) ahead of their use
            if ((s & 3) == 0 && s / 4 + 1 < NG) {
                const uint4 a = rowA[s / 4 + 1];
                sA[s + 4] = a.x; sA[s + 5] = a.y; sA[s + 6] = a.z; sA[s + 7] = a.w;
            }
            if (s >= 1 && ((s - 1) & 3) == 0 && (s - 1) / 4 + 1 < NG) {
                const uint4 b = rowB[(s - 1) / 4 + 1];
                sB[s + 3] = b.x; sB[s + 4] = b.y; sB[s + 5] = b.z; sB[s + 6] = b.w;
            }
            if (s == NC - 4 || (NC < 4 && s == 0)) { gA = rowA2[0]; gB = rowB2[0]; }   // first group of the next rows
            if (s < NC) {
                PACKED_CELL(hdA, eA, sA[s], s, hA)
                const int u = s / PER, i = s % PER;
                // running maxima: the 2*PER cells a unit sees per iteration are folded pairwise (VIMNMX3)
                if (i == 0) pend[u] = hA; else seg[u] = __vimax3_s16x2(seg[u], pend[u], hA);
                if (HOOK && i == PER - 1) {          // hdA = H(j-1, s) now, eA = E entering column s+1
                    mu[u] = __viaddmax_s16x2(hdA, potHA, mu[u]);
                    mu[u] = __viaddmax_s16x2(eA, potEA, mu[u]);
                }
                if (HAS_OUT && s == NC - 1) {
                    const uint32_t w = sw_prmt(hA, eA, 0x6420);
                    bout[j * 32 + lane] = w;
                    if (HAS_IN) diff |= w ^ bA;                          // bA: row j's entering word
                }
            }
            if (s >= 1) {
                PACKED_CELL(hdB, eB, sB[s - 1], s - 1, hB)
                const int u = (s - 1) / PER, i = (s - 1) % PER;
                if (i == PER - 1) seg[u] = __vimax3_s16x2(seg[u], pend[u], hB); else pend[u] = hB;
                if (HOOK && i == PER - 1) {
                    mu[u] = __viaddmax_s16x2(hdB, potHB, mu[u]);
                    mu[u] = __viaddmax_s16x2(eB, potEB, mu[u]);
                }
                if (HAS_OUT && s - 1 == NC - 1) {
                    const uint32_t w = sw_prmt(hB, eB, 0x6420);
                    bout[(j + 1) * 32 + lane] = w;
                    if (HAS_IN) diff |= w ^ bB;
                }
            }
        }
        rowA = rowA2; rowB = rowB2; codeA2 = codeA3; codeB2 = codeB3;
        bA = bA2; bB = bB2; bA2 = bA3; bB2 = bB3; pA = pA2; pB = pB2; pA2 = pA3; pB2 = pB3;
    }
}

// Suffix potentials: the DP of the read against the template's SUFFIX block, run backwards (rows from the
// last query base up, columns from the last suffix base to the first), both halves packed.
//   G(j,c)  = best score of a path that STARTS with the aligned pair (j, c) and ends anywhere
//   GH(j,c) = best score still to gain after the pair (j, c) (>= 0: the path may stop there)
//   GE(j,c) = best score still to gain for a path that is in a template-axis gap at (j, c)
//     GH(j,c) = max(0, G(j+1,c+1), max(GE(j,c+1), GF(j+1,c)) - go)      G(j,c) = s(j,c) + GH(j,c)
//     GE(j,c) = max(GH(j,c), GE(j,c+1) - ge)                             GF(j,c) = max(GH(j,c), GF(j+1,c) - ge)
// Every cell of the forward DP over the suffix block of template u is, in the (max,+) sense, a linear
// function of the H/E column entering the block plus the paths that start inside the block, so
//     max H over the suffix block of template u = max(fresh, max_j H_u(j-1,last)+A[j], max_j E_u(j)+B[j])
// with A[j] = G(j,0), B[j] = GE(j,0) and fresh = max G — none of which depends on u.
// pot[j] = A_a | A_b << 8 | (B_a - go) << 16 | (B_b - go) << 24 (signed bytes; 0x80 = -128 on ghost rows).
template <int NC>
__device__ __forceinline__ void suffix_pass(const uint32_t *stab, const uint8_t *codes, int lane, int m, int rows2,
                                            uint32_t *pot, uint32_t &fresh, uint32_t mgo2, uint32_t mge2) {
    // (the forward cells keep E biased by +go, so the stored E potential is B - go)
    constexpr int NG = (NC + 3) / 4;
    uint32_t Grow[NC], Fv[NC];
#pragma unroll
    for (int c = 0; c < NC; ++c) { Grow[c] = 0; Fv[c] = 0; }
    // r = reversed row index; table columns are stored reversed as well (column 0 = last suffix base)
    auto code_at = [&](int r) { const int j = rows2 - 1 - r; return (j >= 0 && j < m) ? (int)codes[j * 32 + lane] : PAIR_GHOST; };
    auto row_of = [&](int code) { return reinterpret_cast<const uint4 *>(stab + code * STAB_PAD); };
    uint32_t f0 = 0, f1 = 0;
#define SUFFIX_CELL(GD, E, S, C, GOUT)                                                        \
    {                                                                                         \
        const uint32_t t_ = __vmaxs2(E, Fv[C]);                                               \
        const uint32_t gh_ = __viaddmax_s16x2_relu(t_, mgo2, GD);  /* max(t-go, G diag, 0) */ \
        GD = Grow[C];                                                                         \
        GOUT = __vadd2(gh_, S);                                                               \
        Grow[C] = GOUT;                                                                       \
        E = __viaddmax_s16x2(E, mge2, gh_);                                                   \
        Fv[C] = __viaddmax_s16x2(Fv[C], mge2, gh_);                                           \
    }
    for (int r = 0; r < rows2; r += 2) {
        const uint4 *rowA = row_of(code_at(r)), *rowB = row_of(code_at(r + 1));
        uint32_t sA[NG * 4], sB[NG * 4];
#pragma unroll
        for (int g = 0; g < NG; ++g) {
            const uint4 a = rowA[g], b = rowB[g];
            sA[4 * g] = a.x; sA[4 * g + 1] = a.y; sA[4 * g + 2] = a.z; sA[4 * g + 3] = a.w;
            sB[4 * g] = b.x; sB[4 * g + 1] = b.y; sB[4 * g + 2] = b.z; sB[4 * g + 3] = b.w;
        }
        uint32_t gdA = 0, gdB = 0, eA = 0, eB = 0, gA = 0, gB = 0;
#pragma unroll
        for (int s = 0; s <= NC; ++s) {
            if (s < NC) { SUFFIX_CELL(gdA, eA, sA[s], s, gA) f0 = __vmaxs2(f0, gA); }
            if (s >= 1) { SUFFIX_CELL(gdB, eB, sB[s - 1], s - 1, gB) f1 = __vmaxs2(f1, gB); }
        }
        const int jA = rows2 - 1 - r, jB = jA - 1;
        pot[jA * 32 + lane] = jA < m ? sw_prmt(gA, __vadd2(eA, mgo2), 0x6420) : 0x80808080u;
        pot[jB * 32 + lane] = jB < m ? sw_prmt(gB, __vadd2(eB, mgo2), 0x6420) : 0x80808080u;
    }
#undef SUFFIX_CELL
    fresh = __vimax3_s16x2(f0, f1, 0u);
}

// score table of one strip: stab[qa * 6 + qb][c] = s16x2( score(qa, half-a column c), score(qb, half-b column c) )
// (NROWS == NPAIR, rows by pair code), or stab[q][c] = s16x2( score(q, a column c), score(q, b column c) ) (NROWS == 6)
template <int NROWS>
__device__ __forceinline__ void build_stab(uint32_t *stab, const SwLut *lut, int lane, int ncols,
                                           const uint32_t *colsel /* smem, per column PRMT selector */,
                                           uint32_t bias2 = 0u /* added to both halves (PACKED_CELL: go) */) {
    static_assert(NROWS == NPAIR || NROWS == 6, "rows by pair code or by single code");
    for (int i = lane; i < NROWS * STAB_PAD; i += 32) {
        const int q = i / STAB_PAD, c = i % STAB_PAD;
        const int qa = NROWS == NPAIR ? q / 6 : q, qb = NROWS == NPAIR ? q % 6 : q;
        uint32_t v = 0u;
        if (c < ncols) {
            const uint32_t lo = sw_prmt(lut->w0[qa], lut->w1[qa], colsel[c]), hi = sw_prmt(lut->w0[qb], lut->w1[qb], colsel[c]);
            v = __vadd2(sw_prmt(lo, hi, 0x7610), bias2);
        }
        stab[i] = v;
    }
}

// Phase-2 strip: the same packed DP over one strip, but recording WHERE the maxima are.
//   colkey[c] = max over rows of (H << 8 | 255 - row), per strand half (unsigned compare): the column
//               maximum and the smallest row attaining it — what ssw.c's end_ref / end_read need.
//   row_code  row of `stab` for query row j of this lane (ghost row past the end)
//   bin       this lane's boundary column entering the strip (lane offset folded in, 32-word row stride)
//   bout      (CAPTURE) the H/E column leaving unit `kstar` of the strip = the column entering the
//             suffix block of this lane's winning template
// Control flow is uniform across the warp; only addresses and the captured unit differ per lane.
template <int NC, int PER, bool CAPTURE, class RowCode>
__device__ __forceinline__ void strip_locate(const uint32_t *stab, RowCode row_code, int rows2,
                                             const uint32_t *bin, uint32_t *bout, int kstar,
                                             uint32_t (&colkey)[NC], uint32_t mgo2, uint32_t mge2, uint32_t one) {
    constexpr int NG = (NC + 3) / 4;
    uint32_t Hrow[NC], Fv[NC];
#pragma unroll
    for (int c = 0; c < NC; ++c) { Hrow[c] = 0; Fv[c] = 0; colkey[c] = 0; }
    uint32_t hin_prev = 0;
    auto row_of = [&](int code) { return reinterpret_cast<const uint4 *>(stab + code * STAB_PAD); };
    uint32_t bA = bin[0], bB = bin[32];
    // capture without branches: unit k's leaving H / E~ are ANDed with an all-ones mask only for k == kstar
    constexpr int KU = CAPTURE ? NC / PER : 1;
    uint32_t kmask[KU];
#pragma unroll
    for (int k = 0; k < KU; ++k) kmask[k] = (CAPTURE && k == kstar) ? 0xffffffffu : 0u;
    for (int j = 0; j < rows2; j += 2) {
        uint32_t capHA = 0, capEA = 0, capHB = 0, capEB = 0;
        const uint32_t hinA = sw_prmt(bA, 0, 0x4140), hinB = sw_prmt(bB, 0, 0x4140);
        uint32_t eA = sw_prmt(bA, 0, 0x4342), eB = sw_prmt(bB, 0, 0x4342);
        const int jn = min(j + 2, rows2 - 2);
        bA = bin[jn * 32]; bB = bin[(jn + 1) * 32];
        const uint4 *rowA = row_of(row_code(j)), *rowB = row_of(row_code(j + 1));
        uint32_t sA[NG * 4], sB[NG * 4];
#pragma unroll
        for (int g = 0; g < NG; ++g) {
            const uint4 a = rowA[g], b = rowB[g];
            sA[4 * g] = a.x; sA[4 * g + 1] = a.y; sA[4 * g + 2] = a.z; sA[4 * g + 3] = a.w;
            sB[4 * g] = b.x; sB[4 * g + 1] = b.y; sB[4 * g + 2] = b.z; sB[4 * g + 3] = b.w;
        }
        const uint32_t rcA = 0x00010001u * (uint32_t)(255 - j), rcB = rcA - 0x00010001u;
        uint32_t hdA = hin_prev, hdB = hinA;
        hin_prev = hinB;
        uint32_t hA = 0, hB = 0, keyA_prev = 0;
#pragma unroll
        for (int s = 0; s <= NC; ++s) {
            uint32_t keyA = 0;
            if (s < NC) {
                PACKED_CELL(hdA, eA, sA[s], s, hA)
                keyA = hA * 256u + rcA;                          // IMAD on the FMA pipe: H < 256 per half
                if (CAPTURE && s % PER == PER - 1) { capHA |= hA & kmask[s / PER]; capEA |= eA & kmask[s / PER]; }
            }
            if (s >= 1) {
                PACKED_CELL(hdB, eB, sB[s - 1], s - 1, hB)
                const uint32_t keyB = hB * 256u + rcB;
                colkey[s - 1] = __vimax3_u16x2(colkey[s - 1], keyA_prev, keyB);
                if (CAPTURE && (s - 1) % PER == PER - 1) { capHB |= hB & kmask[(s - 1) / PER]; capEB |= eB & kmask[(s - 1) / PER]; }
            }
            keyA_prev = keyA;
        }
        if (CAPTURE) { bout[j * 32] = sw_prmt(capHA, capEA, 0x6420); bout[(j + 1) * 32] = sw_prmt(capHB, capEB, 0x6420); }
    }
}

// Exact end coordinates (ssw.c's end_ref, end_read) of every lane's current candidate (units u, score cs) in
// half `half` of the lane (the candidate's strand in a "both" item, the read in a pair item), warp-uniform.  Only
// that half of the packed pass is read: its rows are the read's own, whatever the other half holds.  end_ref is the first template column whose maximum equals cs.  Phase 1 kept the
// running maximum of the main columns after every unit (runs[]): if some unit u_main <= u is the first whose
// running maximum equals cs, the column lies in that unit's own columns (never in the first FLANK columns:
// cs >= 30 > FLANK * match) — recompute the main strip holding it from its stored entering boundary and read
// the answer off per-column keys.  Otherwise it lies in the suffix block of template u: recompute the strip
// holding unit u, capture the boundary column leaving unit u, then run the suffix block from it.
template <int P>
__device__ __noinline__ void locate_packed(const FamilySmem &F, const SwLut *lut, uint32_t *stab, uint32_t *stab2,
                                           uint32_t *colsel, bool &suffix_table_ready, const uint8_t *codes, int lane,
                                           int m, int m_warp, uint32_t *bnd, const uint32_t *gbnd, int R, int go, int ge,
                                           uint32_t one, int G, int cs, int u, int u_main, int half, int sa, int sb,
                                           int last_slot, int *end_ref, int *end_read, unsigned long long &cells) {
    constexpr int K = strip_units(P);
    constexpr int NC = P * K;
    const uint32_t mgo2 = (uint32_t)((-go) & 0xffff) | ((uint32_t)((-go) & 0xffff) << 16);
    const uint32_t mge2 = (uint32_t)((-ge) & 0xffff) | ((uint32_t)((-ge) & 0xffff) << 16);
    const uint32_t go2 = (uint32_t)go * 0x00010001u;
    const int rows2 = (m_warp + 1) & ~1;
    const int su = G * (u_main > 0 ? u_main : u) - 1;        // last sub-unit of the unit of interest (idle lanes: u = 1)
    const int tstar = su / K, kstar = su % K;                // (K is a multiple of G: units do not straddle strips)
    // Phase 1 stopped after writing slot last_slot when the strips reached their fixed point: every later strip
    // enters with that same column.  The running main maximum does not grow in a skipped strip, so u_main (the
    // first unit attaining cs) never lies in one — only the suffix case reads an aliased slot.
#ifdef TREDSW_DEBUG
    assert(u_main <= 0 || tstar < last_slot);
#endif
    const int sh = half ? 16 : 0;
    int found_col = -1, found_row = 0;
    {
        // main strip tstar (the repeat table of phase 1 stays in shared memory).  Every lane restarts from its
        // own strip's stored boundary column: stage it into shared memory first — 2 x rows independent,
        // sector-sized loads per lane in flight at once instead of an L2 round trip per row pair in the loop.
        {
            const uint32_t *src = gbnd + (size_t)min(tstar, last_slot) * R * 32 + lane;
            for (int j = 0; j < rows2; ++j) bnd[j * 32 + lane] = src[j * 32];
        }
        uint32_t colkey[NC];
        // (pair-code rows: the main table of phase 1 is still in shared memory)
        auto pair_row = [&](int j) { return j < m ? (int)codes[j * 32 + lane] : PAIR_GHOST; };
        strip_locate<NC, P, true>(stab, pair_row, rows2, bnd + lane, bnd + lane, u_main > 0 ? -1 : kstar, colkey,
                                  mgo2, mge2, one);
        if (u_main > 0) {
#pragma unroll
            for (int c = NC - 1; c >= 0; --c) {
                const uint32_t k16 = (colkey[c] >> sh) & 0xffffu;
                if (c / P <= kstar && c / P > kstar - G && (int)(k16 >> 8) == cs) { found_col = FLANK + (tstar * K) * P + c; found_row = 255 - (int)(k16 & 0xffu); }
            }
        }
    }
    __syncwarp();
    cells += (unsigned long long)m * 2ull * (unsigned long long)NC;
    if (__any_sync(0xffffffffu, u_main <= 0 && cs < 0x7fff)) {
        // suffix block of every lane's own template, entered through the captured boundary
        if (!suffix_table_ready) {
            if (lane < FLANK) colsel[lane] = sel2(suf_base(F, sa, lane), suf_base(F, sb, lane));
            __syncwarp();
            build_stab<6>(stab2, lut, lane, FLANK, colsel, go2);
            __syncwarp();
            suffix_table_ready = true;
        }
        uint32_t colkey[FLANK];
        // (rows by this half's own code: a 6-row table suffices, as only this half is read)
        auto own_row = [&](int j) { return j < m ? pair_half(codes[j * 32 + lane], half) : SW_CODE_GHOST; };
        strip_locate<FLANK, FLANK, false>(stab2, own_row, rows2, bnd + lane, nullptr, 0, colkey, mgo2, mge2, one);
        if (u_main <= 0) {
#pragma unroll
            for (int c = FLANK - 1; c >= 0; --c) {
                const uint32_t k16 = (colkey[c] >> sh) & 0xffffu;
                if ((int)(k16 >> 8) == cs) { found_col = FLANK + u * F.P + c; found_row = 255 - (int)(k16 & 0xffu); }
            }
        }
        __syncwarp();
        cells += (unsigned long long)m * 2ull * (unsigned long long)FLANK;
    }
    *end_ref = found_col; *end_read = found_row;
}

// Returns the index of the last boundary slot written (warp-uniform); *planned = main strips of the full plan;
// *lane_conv = main strips this lane needed: the first strip that left the lane's own column unchanged (its outputs
// depend on that column alone, so the lane stays at the fixed point), or the strips run when it never got there.
template <int P>
__device__ __noinline__ int phase1_packed(const FamilySmem &F, const SwLut *lut, uint32_t *stab, uint32_t *colsel,
                                          const uint8_t *codes, int lane, int m, int m_warp, uint32_t *pot,
                                          uint32_t *gbnd, int R, uint8_t *scores, uint8_t *runs, int go, int ge,
                                          uint32_t one, int G, int sa, int sb, bool skip, int *planned, int *lane_conv,
                                          unsigned long long &cells, unsigned long long &skipped_cells) {
    constexpr int K = strip_units(P);
    constexpr int NC = P * K;
    static_assert(NC <= STAB_PAD && FLANK <= STAB_PAD, "strip wider than the score table");
    const uint32_t mgo2 = (uint32_t)((-go) & 0xffff) | ((uint32_t)((-go) & 0xffff) << 16);
    const uint32_t mge2 = (uint32_t)((-ge) & 0xffff) | ((uint32_t)((-ge) & 0xffff) << 16);
    const uint32_t go2 = (uint32_t)go * 0x00010001u;
    const int rows2 = (m_warp + 1) & ~1;
    // ---- suffix potentials (table columns reversed: column c' = suffix base FLANK-1-c') ---------------
    if (lane < FLANK) colsel[lane] = sel2(suf_base(F, sa, FLANK - 1 - lane), suf_base(F, sb, FLANK - 1 - lane));
    __syncwarp();
    build_stab<NPAIR>(stab, lut, lane, FLANK, colsel);
    __syncwarp();
    uint32_t fresh = 0;
    suffix_pass<FLANK>(stab, codes, lane, m, rows2, pot, fresh, mgo2, mge2);
    __syncwarp();
    // ---- strip 0: the FLANK prefix columns -----------------------------------------------------------
    if (lane < FLANK) colsel[lane] = sel2(pre_base(F, sa, lane), pre_base(F, sb, lane));
    __syncwarp();
    build_stab<NPAIR>(stab, lut, lane, FLANK, colsel, go2);
    __syncwarp();
    uint32_t run;                   // running maximum over the main columns so far, per half
    {
        uint32_t seg0[1] = {0u}, mu0[1] = {0u}, unused = 0u;
        strip_pass<FLANK, FLANK, false, true, false>(stab, codes, lane, m, rows2, nullptr, gbnd, pot, seg0, mu0, mgo2, mge2,
                                                     one, unused);
        run = seg0[0];
    }
    __syncwarp();
    // ---- main strips: K repeat units each; the suffix of every template is folded in by the potentials --
    for (int c = lane; c < NC; c += 32) colsel[c] = sel2(rep_base(F, sa, c % F.P), rep_base(F, sb, c % F.P));
    __syncwarp();
    build_stab<NPAIR>(stab, lut, lane, NC, colsel, go2);
    __syncwarp();
    // scores and running main maxima of the template with sub-units su (when su ends a real unit)
    auto put = [&](int su, uint32_t mu_u) {
        if (su % G == 0 && su <= F.U * G) {
            const int ur = su / G - 1;                              // 0-based real unit
            const uint32_t best = __vimax3_s16x2(run, mu_u, fresh);
            // slot 2 * ur + h: half h of the lane (strand h of a "both" item's read, read h of a pair item)
            scores[(2 * ur + 0) * 32 + lane] = (uint8_t)(best & 0xffu);
            scores[(2 * ur + 1) * 32 + lane] = (uint8_t)((best >> 16) & 0xffu);
            runs[(2 * ur + 0) * 32 + lane] = (uint8_t)(run & 0xffu);          // running maximum of the main columns
            runs[(2 * ur + 1) * 32 + lane] = (uint8_t)((run >> 16) & 0xffu);
        }
    };
    // Every main strip runs the same table and potentials, so its outputs (seg, mu, leaving column) are a function
    // of its entering column alone.  A strip that leaves exactly the column it received (every row, both halves, all
    // lanes) is therefore repeated verbatim by every later strip: the running maximum stays `run`, unit u of a later
    // strip scores max(run, mu[u], fresh), and every later boundary slot equals the one just written.  The loop
    // stops there; phase 2 reads that slot for any later strip (locate_packed's last_slot).
    const int nplan = (F.U * G + K - 1) / K;                        // main strips of the full nested plan
    int nstrips = 0, conv = 0;
    for (int u0 = 0; u0 < F.U * G; u0 += K) {                       // u0, u: sub-units of P columns
        uint32_t seg[K], mu[K], diff = 0u;
#pragma unroll
        for (int u = 0; u < K; ++u) { seg[u] = 0; mu[u] = 0; }
        // (slot t of the scratch = boundary entering main strip t; the strip writes slot t+1)
        strip_pass<NC, P, true, true, true>(stab, codes, lane, m, rows2, gbnd + (size_t)nstrips * R * 32,
                                            gbnd + (size_t)(nstrips + 1) * R * 32, pot, seg, mu, mgo2, mge2, one, diff);
        ++nstrips;
        if (conv == 0 && diff == 0u) conv = nstrips;
#pragma unroll
        for (int u = 0; u < K; ++u) {
            run = __vmaxs2(run, seg[u]);
            put(u0 + u + 1, mu[u]);                                 // (sub-units completed)
        }
        if (skip && __all_sync(0xffffffffu, diff == 0u)) {
            for (int v0 = u0 + K; v0 < F.U * G; v0 += K) {
#pragma unroll
                for (int u = 0; u < K; ++u) put(v0 + u + 1, mu[u]);
            }
            break;
        }
    }
    // (cells: the full plan, whether or not strips were skipped — the executed-cell statistic keeps its meaning;
    //  the skipped ones are counted apart)
    cells += (unsigned long long)m * 2ull * (unsigned long long)(2 * FLANK + nplan * NC);
    skipped_cells += (unsigned long long)m * 2ull * (unsigned long long)((nplan - nstrips) * NC);
    *planned = nplan;
    *lane_conv = conv ? conv : nstrips;
    return nstrips;                 // the last boundary slot written
}

// ---------------------------------------------------------------------------------------------------
// FAST = true : every family with 18-bp flanks, period <= 12 and scores < 256 (packed phase 1, u8 scores)
// FAST = false: everything else (scalar phase 1, u16 scores)
// Persistent: one warp per CTA, CTAs pull items (32 reads of one family, or 64 single-strand reads of one family
// and strand, two per lane) from a counter; both kernels walk the same item list and skip the items of the other
// kernel.
template <bool FAST>
__global__ void __launch_bounds__(32) classify_kernel(ClassifyParams p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ SwLut lut;
    __shared__ FamilySmem F;
    // stab: rows by pair code (phase 1, and the main strips of phase 2); stab2: rows by one half's own code (the
    // suffix block of phase 2, which reads one half at a time)
    __shared__ __align__(16) uint32_t stab[NPAIR * STAB_PAD], stab2[6 * STAB_PAD];
    __shared__ uint32_t colsel[STAB_PAD];
    // (shared memory: the reads as codes [rows][32], the score table and ONE boundary column [rows][32] for
    //  phase 2, whose scalar sweeps walk it with dependent load -> compute -> store chains that must not pay
    //  L2 latency per row; per-template scores, suffix potentials and the per-strip boundary columns of
    //  phase 1 live in this CTA's slot of the global scratch, streamed with one-iteration-ahead requests)
    typedef typename std::conditional<FAST, uint8_t, uint16_t>::type score_t;
    const int lane = threadIdx.x;
    const int R = p.max_rows + 2;                                                  // + ghost row of the 2-row loop
    uint32_t *bnd = reinterpret_cast<uint32_t *>(smem_raw);                        // [R][32] phase-2 boundary column
    uint8_t *codes = reinterpret_cast<uint8_t *>(bnd + (size_t)R * 32);            // [R][32]
    // per-CTA slot of 2*max_u*32 u16-sized elements: generic kernel = u16 scores; packed kernel = u8 scores in
    // the first half, u8 running main maxima (runs) in the second
    unsigned char *slot = reinterpret_cast<unsigned char *>(p.score_buf) + (size_t)blockIdx.x * (2 * p.max_u) * 32 * sizeof(uint16_t);
    score_t *scores = reinterpret_cast<score_t *>(slot);                           // [2U][32]
    uint8_t *runs = slot + (size_t)(2 * p.max_u) * 32;                             // [2U][32] (packed kernel only)
    // suffix potentials [R][32]: phase 1 only, so in the packed kernel they live in the shared-memory column that
    // phase 2 later uses for its boundary staging (LDS instead of an L2 round trip per row pair and strip)
    uint32_t *pot = FAST ? bnd : p.pot_buf + (size_t)blockIdx.x * R * 32;
    uint32_t *gbnd = p.gbnd_buf + (size_t)blockIdx.x * (p.nslots + 1) * R * 32;    // [nslots + 1][R][32]
    const uint32_t one = p.one;
    __shared__ unsigned long long skip_acc[TREDSW_STRIP_SKIP_STATS];   // this CTA's share, added up at the end
    for (int i = lane; i < TREDSW_STRIP_SKIP_STATS; i += 32) skip_acc[i] = 0ull;
    sw_build_lut(&lut, c_fmat25, lane, 32);
    const int nitems = p.chunk_start[p.ngroups];
    unsigned long long alg = 0, cells1 = 0, cells2 = 0, cells_skipped = 0;
    unsigned nal = 0;

    for (;;) {
        __syncwarp();
        int item = 0;
        if (lane == 0) item = atomicAdd(p.counter + (FAST ? 1 : 0), 1);
        item = __shfl_sync(0xffffffffu, item, 0);
        if (item >= nitems) break;
        // item -> (family, strand class) group (binary search over chunk_start)
        int lo = 0, hi = p.ngroups;
        while (hi - lo > 1) {
            int mid = (lo + hi) >> 1;
            if (p.chunk_start[mid] <= item) lo = mid; else hi = mid;
        }
        const int grp = p.grp_perm[lo], f = grp / NCLASS, cls = grp % NCLASS;
        {
            const tredsw_family &g = p.families[f];
            F.prefix[lane] = g.prefix[lane]; F.suffix[lane] = g.suffix[lane]; F.repeat[lane] = g.repeat[lane];
            if (lane == 0) { F.Lp = g.prefix_len; F.Ls = g.suffix_len; F.P = g.period; F.U = g.max_units; F.clip = g.clip; }
        }
        __syncwarp();
        const bool fast_shape = p.allow_fast && (F.Lp == FLANK && F.Ls == FLANK && F.P >= 1 && F.P <= 12);
        if (fast_shape != FAST) continue;

        // The lane's reads: one read of a "both" item, or reads 2*lane and 2*lane+1 of a pair item's 64 (read h in
        // half h; a missing partner is a ghost of length 0).  Half-strands (sa, sb) of the item: (fwd, rc) for
        // "both", (fwd, fwd) or (rc, rc) for a pair item.
        const bool pair = FAST && cls != CLASS_BOTH;
        const int sa = cls == CLASS_RC ? 1 : 0, sb = cls == CLASS_FWD ? 0 : 1;
        const int idx0 = p.grp_start[grp] + (pair ? 64 * (item - p.chunk_start[lo]) + 2 * lane : 32 * (item - p.chunk_start[lo]) + lane);
        int r0 = -1, r1 = -1, m0 = 0, m1 = 0;
        const bool valid0 = idx0 < p.grp_start[grp + 1], valid1 = pair && idx0 + 1 < p.grp_start[grp + 1];
        if (valid0) { r0 = p.order[idx0]; m0 = (int)(p.roff[r0 + 1] - p.roff[r0]); }
        if (valid1) { r1 = p.order[idx0 + 1]; m1 = (int)(p.roff[r1 + 1] - p.roff[r1]); }
        const bool too_long0 = m0 > p.max_rows, too_long1 = m1 > p.max_rows;
        if (too_long0) m0 = 0;
        if (too_long1) m1 = 0;
        auto clampc = [](int c) { return (c < 0 || c > 4) ? 4 : c; };
        // codes: plain base codes in the generic kernel, pair codes qa * 6 + qb (ghost past each read's end) in the
        // packed one — 7q for a "both" item, whose halves share the read
        const int m_lane = max(m0, m1);
        if (!pair) {
            if (m0 > 0) for_each_base(p.rbuf + p.roff[r0], m0, [&](int j, int c) { codes[j * 32 + lane] = (uint8_t)((FAST ? 7 : 1) * clampc(c)); });
        } else {
            if (m0 > 0) for_each_base(p.rbuf + p.roff[r0], m0, [&](int j, int c) { codes[j * 32 + lane] = (uint8_t)(6 * clampc(c) + SW_CODE_GHOST); });
            for (int j = m0; j < m_lane; ++j) codes[j * 32 + lane] = (uint8_t)PAIR_GHOST;
            if (m1 > 0) for_each_base(p.rbuf + p.roff[r1], m1, [&](int j, int c) { codes[j * 32 + lane] += (uint8_t)(clampc(c) - SW_CODE_GHOST); });
        }
        const int m_warp = __reduce_max_sync(0xffffffffu, m_lane);
        __syncwarp();

        int last_slot = 0;              // last boundary slot phase 1 wrote (packed kernel)
        if constexpr (!FAST) {
            phase1_generic(F, &lut, codes, lane, m0, m_warp, bnd, scores, p.go, p.ge, cells1);
        } else {
            const int pi = instance_period(F.P);
            int planned = 0, conv = 0;
            switch (pi) {
#define PCASE(PP) case PP: last_slot = phase1_packed<PP>(F, &lut, stab, colsel, codes, lane, m_lane, m_warp, pot, gbnd, R, scores, runs, p.go, p.ge, one, F.P / PP, sa, sb, p.strip_skip != 0, &planned, &conv, cells1, cells_skipped); break;
                PCASE(1) PCASE(2) PCASE(3) PCASE(4) PCASE(5) PCASE(7) PCASE(8) PCASE(9) PCASE(10) PCASE(11) PCASE(12)
#undef PCASE
            }
            if (lane == 0) {            // per instance period: planned / skipped main strips, items, items without a skip
                unsigned long long *a = skip_acc + 1 + 4 * (pi - 1);
                a[0] += (unsigned long long)planned; a[1] += (unsigned long long)(planned - last_slot);
                a[2] += 1ull; a[3] += last_slot == planned ? 1ull : 0ull;
            }
            // per lane holding a read: the strips of the plan, those its warp skipped, and those it could skip on its
            // own (the bound that no grouping of reads into items can beat)
            const bool busy = m_lane > 0;
            const unsigned lane_planned = __reduce_add_sync(0xffffffffu, busy ? (unsigned)planned : 0u);
            const unsigned lane_skipped = __reduce_add_sync(0xffffffffu, busy ? (unsigned)(planned - last_slot) : 0u);
            const unsigned lane_skippable = __reduce_add_sync(0xffffffffu, busy ? (unsigned)(planned - conv) : 0u);
            if (lane == 0) {
                unsigned long long *b = skip_acc + 1 + 4 * 12 + 3 * (pi - 1);
                b[0] += lane_planned; b[1] += lane_skipped; b[2] += lane_skippable;
            }
        }
        __syncwarp();

        // ---- Phase 2, once per read of the lane: walk candidates in arg-max order until one yields a tag ----------
        bool suffix_table_ready = false;
        for (int h = 0; h < (pair ? 2 : 1); ++h) {
            const bool valid = h ? valid1 : valid0, too_long = h ? too_long1 : too_long0;
            const int r = h ? r1 : r0, m = h ? m1 : m0;
            const int own_strand = h ? sb : sa;        // (pair items: the strand of this read's templates)
            int tag = TREDSW_TAG_NONE, best_u = 0, best_score = -1, rb = -1, re = -1, qb = -1, qe = -1, best_rank = -1;
            const bool active = valid && m > 0;
            // next candidate after (last_score, last_rank) in the reference's arg-max order.  Score slot of rank
            // 2(u-1) + s: the rank itself in a "both" item; in a pair item only the read's own strand was computed,
            // in half h — every template of the other strand scores below 30 (q-gram bound) and is never a candidate
            auto pick = [&](int last_score, int last_rank, int &cs, int &cr) {
                cs = -1; cr = -1;
                if (!active) return;
                for (int rank = 0; rank < 2 * F.U; ++rank) {
                    if (pair && (rank & 1) != own_strand) continue;
                    const int sc = scores[(pair ? (rank & ~1) | h : rank) * 32 + lane];
                    const int n = F.Lp + F.Ls + F.P * (rank / 2 + 1);
                    const int min_len = min(m, n) / 2;
                    if (sc < max(min_len, 30)) continue;
                    if (sc > last_score || (sc == last_score && rank <= last_rank)) continue;   // already tried
                    if (sc > cs) { cs = sc; cr = rank; }
                }
            };
            int cs, cr;
            pick(0x7fffffff, -1, cs, cr);
            // Rounds: every lane that still has a candidate evaluates it — end coordinates from one warp-uniform
            // packed pass (locate_packed), begin coordinates and the tag per lane — until all lanes are settled.
            // Almost every read settles in the first round.
            const int max_units_eff = F.clip ? (m + F.P - 1) / F.P : F.U;
            auto own_code = [&](int j) { return FAST ? pair_half(codes[j * 32 + lane], h) : (int)codes[j * 32 + lane]; };
            while (__any_sync(0xffffffffu, cr >= 0)) {
                const bool pending = cr >= 0;
                const int u = pending ? cr / 2 + 1 : 1, s = pending ? (cr & 1) : 0;
                const int half = pair ? h : s;
                int fast_end_ref = -1, fast_end_read = 0;
                if constexpr (FAST) {
                    if (FLANK * p.match < 30) {
                        int u_main = 0;                      // first unit whose running main maximum equals cs
                        if (pending) for (int k = 1; k <= u; ++k) if ((int)runs[(2 * (k - 1) + half) * 32 + lane] == cs) { u_main = k; break; }
                        switch (instance_period(F.P)) {
#define PCASE(PP) case PP: locate_packed<PP>(F, &lut, stab, stab2, colsel, suffix_table_ready, codes, lane, m, m_warp, bnd, gbnd, R, p.go, p.ge, one, F.P / PP, pending ? cs : 0x7fff, u, u_main, half, sa, sb, last_slot, &fast_end_ref, &fast_end_read, cells2); break;
                            PCASE(1) PCASE(2) PCASE(3) PCASE(4) PCASE(5) PCASE(7) PCASE(8) PCASE(9) PCASE(10) PCASE(11) PCASE(12)
#undef PCASE
                        }
                        if (!pending) fast_end_ref = -1;
                    }
                }
                if (pending) {
                    const int n = F.Lp + F.Ls + F.P * u;
                    auto cc_f = [&](int i) { return fam_code(F, u, s, n, i); };
                    int end_ref = fast_end_ref, end_read = fast_end_read;
                    if (end_ref < 0) {
                        // (generic kernel, or a scoring scheme outside the packed pass's preconditions)
                        // Exact banding (sw_sweep.cuh): a path ending with score cs drifts at most `drift` diagonals
                        // from the diagonal it starts on.  Forward: it starts at some (i0, j0) with i0 <= n - need,
                        // j0 <= m - need, where need = ceil(cs / match) aligned pairs are indispensable.
                        const int drift = sw_max_drift(cs, m, n, p.match, p.go, p.ge);
                        const int need = (cs + p.match - 1) / p.match;
                        sw_sweep<FAM_W2, 1, false>(m, m, n, own_code, cc_f, &lut, bnd + lane, 32, p.go, p.ge, cs, &end_ref, &end_read,
                                                   nullptr, -(m - need) - drift, (n - need) + drift, &cells2);
                    }
                    bool settled = false;
                    if (end_ref >= 0) {      // (always: the score was produced by this very template)
                        // Reverse: only a path leaving the corner (end_ref, end_read) can reach cs (Appendix A); it
                        // lives in the (end_read+1) x (end_ref+1) rectangle, which bounds its aligned pairs and
                        // therefore how far it can drift from the corner's diagonal.
                        const int rdrift = sw_max_drift(cs, end_read + 1, end_ref + 1, p.match, p.go, p.ge);
                        int ci = -1, rj = 0;
                        if (rdrift == 0) {   // no gap affordable: walk the diagonal
                            const int lim = min(end_read, end_ref) + 1;
                            int hs = 0;
                            for (int k = 0; k < lim; ++k) {
                                const int qc = own_code(end_read - k);
                                const int sc = (int)sw_prmt(lut.w0[qc], lut.w1[qc], sw_sel32(fam_code(F, u, s, n, end_ref - k)));
                                hs = max(0, hs + sc);
                                if (hs == cs) { ci = rj = k; break; }
                            }
                            cells2 += (unsigned long long)lim;
                        }
                        if (ci < 0) {
                            auto rc_r = [&](int j) { return own_code(end_read - j); };
                            auto cc_r = [&](int i) { return fam_code(F, u, s, n, end_ref - i); };
                            sw_sweep<FAM_W2, 1, false>(end_read + 1, end_read + 1, end_ref + 1, rc_r, cc_r, &lut, bnd + lane, 32,
                                                       p.go, p.ge, cs, &ci, &rj, nullptr, -rdrift, rdrift, &cells2);
                        }
                        const int c_rb = end_ref - ci, c_qb = end_read - rj;
                        const int t = sw_classify(cs, c_rb, end_ref, c_qb, end_read, m, n, u, F.P, max_units_eff);
                        if (t != TREDSW_TAG_NONE) {
                            tag = t; best_u = u; best_score = cs; rb = c_rb; re = end_ref; qb = c_qb; qe = end_read;
                            best_rank = cr;
                            settled = true;
                        }
                    }
                    if (settled) cr = -1;
                    else { const int ls = cs, lr = cr; pick(ls, lr, cs, cr); }
                }
                __syncwarp();
            }
            if (valid) {
                int32_t *o = p.out + (int64_t)r * 8;
                o[0] = too_long ? -1 : tag; o[1] = best_u; o[2] = best_score; o[3] = rb; o[4] = re; o[5] = qb; o[6] = qe;
                o[7] = best_rank;
            }
            if (p.stats && active) {
                unsigned long long sum_n = 0;
                for (int u = 1; u <= F.U; ++u) sum_n += 2ull * (unsigned long long)(F.Lp + F.Ls + F.P * u);
                alg += (unsigned long long)m * sum_n;
                nal += (unsigned)(2 * F.U);
            }
        }
    }
    if (p.stats) {
        unsigned long long c1 = cells1, c2 = cells2, na = nal;
        for (int d = 16; d > 0; d >>= 1) {
            alg += __shfl_down_sync(0xffffffffu, alg, d);
            c1 += __shfl_down_sync(0xffffffffu, c1, d);
            c2 += __shfl_down_sync(0xffffffffu, c2, d);
            na += __shfl_down_sync(0xffffffffu, na, d);
        }
        if (lane == 0) {
            atomicAdd(&p.stats[0], alg); atomicAdd(&p.stats[1], c1); atomicAdd(&p.stats[2], c2);
            atomicAdd(&p.stats[3], na);
        }
    }
    if (FAST) {
        for (int d = 16; d > 0; d >>= 1) cells_skipped += __shfl_down_sync(0xffffffffu, cells_skipped, d);
        if (lane == 0) skip_acc[0] = cells_skipped;
        __syncwarp();
        for (int i = lane; i < TREDSW_STRIP_SKIP_STATS; i += 32)
            if (skip_acc[i]) atomicAdd(&p.skip_stats[i], skip_acc[i]);
    }
}

// ---- grouping of reads by family on the device (counting sort) ------------------------------------
// ---- exact q-gram pre-filter --------------------------------------------------------------------------
// About half of the reads fetched around a locus (bam_parser.py:206-214 takes everything in the window)
// cannot pass min_score = max(min_len, 30) (bam_parser.py:134) against any template: they lie in the
// flanking genome.  q-gram lemma for this scoring: an alignment with score S >= 30 has M matches, X
// mismatches and g gap runs with M - b X - go g >= 30; its matches form at most X + g + Z + 1 exact runs
// (Z = aligned N bases, which score 0), and a run of length r shares r - q + 1 q-grams with the template:
//     shared q-grams >= 30 + X (b - (q-1)) + g (go - (q-1)) - (q-1)(Z + 1) >= 30 - (q-1)(Z + 1)
// for q - 1 <= min(b, go).  So a read with fewer than 30 - (q-1)(#N + 1) positions whose q-gram occurs in
// ANY template of the family (on either strand) has no candidate at all: it is given the "no tag" record here
// and never reaches the Smith-Waterman kernel.  Exact — no alignment is lost (parity tests cover it).
// The same bound per strand gives the read's strand class: when only one strand reaches the threshold, no
// template of the other strand can score min_score, so that strand can never be a candidate (pick() skips scores
// below max(min_len, 30)) and the packed kernel computes the read on one strand only, two reads per lane.
//
// Convergence key.  A lane's main strips reach their fixed point (phase1_packed) about one strip after the template
// columns have passed the read's own repeat stretch, so the q-grams of the read that occur in the pure repeat (repeat^k,
// either strand) predict the strips the read needs: min(nplan, ceil((hits + q - 1) / NC) + 1), NC = strip columns.
// Reads are grouped by (family, strand class, predicted strips), so that the reads of an item stop at about the same
// strip instead of all waiting for the one with the longest repeat stretch.
struct QgramInfo {
    int q;                         // 0: filter off for this family (N in the templates)
    int min_score;
    int pair;                      // single-strand classes allowed (packed-kernel family, pairing not switched off)
    int nplan;                     // main strips of the packed plan; 0: reads keep predicted strips 0 (no ordering)
    int nc;                        // columns per main strip
};
// per family: 4096 six-mers x 2 bits (forward / reverse-complement templates), then the same for the pure repeat
constexpr int QTAB_WORDS = 256;

// eff_bin[r] = (f * NCLASS + strand class) * nb + nb - 1 - predicted strips (the bins of a group in descending
// predicted strips), -2 when the read has no candidate, -1 when it has no family
__global__ void prefilter_kernel(const int8_t *rbuf, const int64_t *roff, int nreads, const int32_t *read_family,
                                 int nfam, const tredsw_family *families, const uint32_t *qtab, const QgramInfo *qinfo,
                                 int nb, int32_t *eff_bin, unsigned long long *stats) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long alg = 0; unsigned nal = 0;
    if (r < nreads) {
        int f = read_family[r], cls = CLASS_BOTH, strips = 0;
        if (f < 0 || f >= nfam) f = -1;
        if (f >= 0 && qinfo[f].q > 0) {
            const int q = qinfo[f].q;
            const uint32_t mask = (1u << (2 * q)) - 1u;
            const uint32_t *tab = qtab + (size_t)f * 2 * QTAB_WORDS, *rtab = tab + QTAB_WORDS;
            const int8_t *s = rbuf + roff[r];
            const int m = (int)(roff[r + 1] - roff[r]);
            uint32_t code = 0; int run = 0, nN = 0, hf = 0, hr = 0, rf = 0, rr = 0;
            for_each_base(s, m, [&](int, int c) {
                if (c < 0 || c > 3) { ++nN; run = 0; return; }
                code = ((code << 2) | (uint32_t)c) & mask;
                if (++run >= q) {
                    const uint32_t sh = (code & 15u) * 2u;
                    const uint32_t e = (tab[code >> 4] >> sh) & 3u, er = (rtab[code >> 4] >> sh) & 3u;
                    hf += e & 1u; hr += e >> 1;
                    rf += er & 1u; rr += er >> 1;
                }
            });
            const int thr = qinfo[f].min_score - (q - 1) * (nN + 1);
            if (hf < thr && hr < thr) {
                if (stats) {
                    const tredsw_family &g = families[f];
                    unsigned long long sum_n = 0;
                    for (int u = 1; u <= g.max_units; ++u) sum_n += 2ull * (unsigned long long)(g.prefix_len + g.suffix_len + g.period * u);
                    alg = (unsigned long long)m * sum_n; nal = 2u * (unsigned)g.max_units;
                }
                f = -2;
            } else if (qinfo[f].pair && (hf < thr || hr < thr)) {
                cls = hf >= thr ? CLASS_FWD : CLASS_RC;
            }
            if (f >= 0 && qinfo[f].nplan > 0) {
                const int key = cls == CLASS_FWD ? rf : cls == CLASS_RC ? rr : max(rf, rr);
                strips = min(qinfo[f].nplan, (key + q - 1 + qinfo[f].nc - 1) / qinfo[f].nc + 1);
            }
        }
        eff_bin[r] = f >= 0 ? (f * NCLASS + cls) * nb + nb - 1 - strips : f;
    }
    if (stats) {
        for (int d = 16; d > 0; d >>= 1) { alg += __shfl_down_sync(0xffffffffu, alg, d); nal += __shfl_down_sync(0xffffffffu, nal, d); }
        if ((threadIdx.x & 31) == 0 && alg) { atomicAdd(&stats[0], alg); atomicAdd(&stats[3], (unsigned long long)nal); }
    }
}

// Counting sort of the reads into bins (group, predicted strips), nb bins per (family, strand class) group.
// (reads arrive grouped by problem, so the lanes of a warp mostly share one bin: the atomics are aggregated per warp
//  and distinct bin — one atomic instead of up to 32 on the same counter)
__global__ void fam_count_kernel(const int32_t *read_bin, int nreads, int nbins, int32_t *count) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    int f = r < nreads ? read_bin[r] : -1;
    if (f >= nbins) f = -1;
    const unsigned peers = __match_any_sync(0xffffffffu, f);
    if (f >= 0 && (threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&count[f], __popc(peers));
}
constexpr int SCAN_THREADS = 1024;
// exclusive prefix sums of load(0..n-1), handed to store(i, sum); returns the total (one block of SCAN_THREADS)
template <class Load, class Store>
__device__ int block_exclusive_scan(int n, Load load, Store store, int *warp_sums) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int carry = 0;
    for (int base = 0; base < n; base += SCAN_THREADS) {
        const int i = base + threadIdx.x;
        const int v = i < n ? load(i) : 0;
        int x = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const int y = __shfl_up_sync(0xffffffffu, x, d); if (lane >= d) x += y; }
        if (lane == 31) warp_sums[warp] = x;
        __syncthreads();
        if (warp == 0) {
            int w = warp_sums[lane];
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) { const int y = __shfl_up_sync(0xffffffffu, w, d); if (lane >= d) w += y; }
            warp_sums[lane] = w;
        }
        __syncthreads();
        if (i < n) store(i, carry + (warp ? warp_sums[warp - 1] : 0) + x - v);
        carry += warp_sums[31];
        __syncthreads();
    }
    return carry;
}
// An item holds 32 reads of a "both" group, 64 of a single-strand group (two per lane).
__host__ __device__ constexpr int item_reads(int grp) { return grp % NCLASS == CLASS_BOTH ? 32 : 64; }
// one block of SCAN_THREADS: cursor[bin] := start of the bin, grp_start[g] = start of group g's first bin, and
// chunk_start (items, groups in perm order).  A group that fits one item gains nothing from the order of its reads:
// fam_scatter_kernel sends all its reads to its last bin, in arrival order, so its cursor is the group's start.
__global__ void __launch_bounds__(SCAN_THREADS) fam_scan_kernel(const int32_t *count, int ngroups, int nb,
                                                                 const int32_t *perm, int32_t *grp_start,
                                                                 int32_t *chunk_start, int32_t *cursor) {
    __shared__ int warp_sums[32];
    const int total = block_exclusive_scan(ngroups * nb, [&](int i) { return count[i]; },
                                           [&](int i, int v) { cursor[i] = v; }, warp_sums);
    for (int g = threadIdx.x; g < ngroups; g += SCAN_THREADS) grp_start[g] = cursor[g * nb];
    if (threadIdx.x == 0) grp_start[ngroups] = total;
    __syncthreads();
    for (int g = threadIdx.x; g < ngroups; g += SCAN_THREADS)
        if (grp_start[g + 1] - grp_start[g] <= item_reads(g)) cursor[g * nb + nb - 1] = grp_start[g];
    const int items = block_exclusive_scan(ngroups, [&](int i) {
        const int g = perm[i], per = item_reads(g);
        return (grp_start[g + 1] - grp_start[g] + per - 1) / per; }, [&](int i, int v) { chunk_start[i] = v; }, warp_sums);
    if (threadIdx.x == 0) chunk_start[ngroups] = items;
}
__global__ void fam_scatter_kernel(const int32_t *read_bin, int nreads, int nbins, int nb, const int32_t *grp_start,
                                   int32_t *cursor, int32_t *order, int32_t *out) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31;
    int f = r < nreads ? read_bin[r] : -1;
    if (f >= nbins) f = -1;
    if (f >= 0) {
        const int g = f / nb;
        if (grp_start[g + 1] - grp_start[g] <= item_reads(g)) f = g * nb + nb - 1;
    }
    const unsigned peers = __match_any_sync(0xffffffffu, f);
    const int leader = __ffs(peers) - 1;
    int base = 0;
    if (f >= 0 && lane == leader) base = atomicAdd(&cursor[f], __popc(peers));
    base = __shfl_sync(0xffffffffu, base, leader);
    if (r < nreads) {
        if (f >= 0) order[base + __popc(peers & ((1u << lane) - 1u))] = r;
        else if (f == -2) {      // pre-filtered: the record of a read without candidates
            int32_t *o = out + (int64_t)r * 8; o[0] = TREDSW_TAG_NONE; o[1] = 0; o[2] = o[3] = o[4] = o[5] = o[6] = o[7] = -1;
        } else { int32_t *o = out + (int64_t)r * 8; o[0] = -1; o[1] = o[2] = o[3] = o[4] = o[5] = o[6] = o[7] = -1; }
    }
}

template <bool FAST>
int launch_classify(tredsw_ctx *ctx, const ClassifyParams &p, int nctas, size_t smem) {
    classify_kernel<FAST><<<nctas, 32, smem, ctx->stream>>>(p);
    CUDA_TRY(cudaGetLastError());
    ctx->launches += 1;
    return TREDSW_OK;
}

// static shared memory of the classify kernels (score tables, LUT, family): the 48 KB a block gets without opting in
// bounds static + dynamic bytes together
int classify_static_smem(size_t *out) {
    cudaFuncAttributes fa{}, ga{};
    CUDA_TRY(cudaFuncGetAttributes(&fa, classify_kernel<true>));
    CUDA_TRY(cudaFuncGetAttributes(&ga, classify_kernel<false>));
    *out = std::max(fa.sharedSizeBytes, ga.sharedSizeBytes);
    return TREDSW_OK;
}

// resident CTAs per SM of the persistent kernels (registers / shared memory), times the SM count
int persistent_ctas(tredsw_ctx *ctx, size_t smem, size_t static_smem, bool need_fast, bool need_generic, int *out) {
    int a = 0, b = 0;
    if (smem + static_smem > 48 * 1024) {
        CUDA_TRY(cudaFuncSetAttribute(classify_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        CUDA_TRY(cudaFuncSetAttribute(classify_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    }
    if (need_fast) CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&a, classify_kernel<true>, 32, smem));
    if (need_generic) CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, classify_kernel<false>, 32, smem));
    int per_sm = need_fast ? a : b;          // the packed kernel is the one that matters when both run
    static const int env_cap = [] { const char *e = getenv("TREDSW_CTAS_PER_SM"); return e ? atoi(e) : 0; }();
    // measured on B200 (profiles/): beyond 8 resident warps per SM the strip loops of the concurrently running
    // phases no longer fit the instruction caches (L0 6 KB / L1.5 32 KB) and throughput drops
    const int cap = env_cap > 0 ? env_cap : 8;
    if (per_sm > cap) per_sm = cap;
    if (per_sm < 1) per_sm = 1;
    // Leave a few CTA slots of the GPU empty (spread over the SMs by the block scheduler): the short kernels that
    // finish the PREVIOUS call of a pipeline (KDE, grid, reductions: up to ~35 KB of shared memory per block)
    // need a place to run while this persistent kernel holds everything else, or that call — and the input copy
    // of the one after it — waits for this kernel to drain (tools/e2e_probe.py --timeline).
    static const int env_free = [] { const char *e = getenv("TREDSW_FREE_SLOTS"); return e ? atoi(e) : -1; }();
    int free_slots = env_free >= 0 ? env_free : 0;
    if (free_slots > per_sm * ctx->sm_count / 2) free_slots = per_sm * ctx->sm_count / 2;
    *out = per_sm * ctx->sm_count - free_slots;
    return TREDSW_OK;
}

// packed plan of a family: main strips and columns per strip (0 strips: the family runs the generic kernel)
void packed_plan(const tredsw_family &g, bool allow_fast, int *nplan, int *nc) {
    *nplan = 0; *nc = 0;
    if (!(allow_fast && g.prefix_len == FLANK && g.suffix_len == FLANK && g.period >= 1 && g.period <= 12)) return;
    const int pi = instance_period(g.period), k = strip_units(pi);
    *nplan = (g.max_units * (g.period / pi) + k - 1) / k;
    *nc = pi * k;
}

}  // namespace

// bins per (family, strand class) group of the read order: predicted strips 0..nplan of the longest packed plan
int tredsw_classify_bins(const tredsw_family *h_families, int nfamilies) {
    int nb = 1;
    for (int f = 0; f < nfamilies; ++f) {
        const tredsw_family &g = h_families[f];
        if (g.period < 1 || g.period > 12 || g.max_units < 1 || g.max_units > 4096) continue;
        int nplan, nc;
        packed_plan(g, true, &nplan, &nc);
        nb = std::max(nb, nplan + 1);
    }
    return nb;
}

size_t tredsw_classify_work_words(const tredsw_family *h_families, int nfamilies, int nreads) {
    const size_t ngroups = (size_t)NCLASS * nfamilies, nbins = ngroups * tredsw_classify_bins(h_families, nfamilies);
    return 2 * nbins + 2 * (ngroups + 1) + (size_t)nreads;
}

int tredsw_internal_classify(tredsw_ctx *ctx, const int8_t *d_rbuf, const int64_t *d_roff, int nreads,
                             const int32_t *d_read_family, const tredsw_family *d_families,
                             const tredsw_family *h_families, int nfamilies, int max_m,
                             const int8_t *mat25, int gap_open, int gap_extend, int32_t *d_work, int32_t *d_out,
                             unsigned long long *d_stats) {
    int max_u = 0, nslots = 1; bool need_fast = false, need_generic = false; int max_match = 0;
    for (int i = 0; i < 25; ++i) if (mat25[i] > max_match) max_match = mat25[i];
    int min_mat = 0;
    for (int i = 0; i < 25; ++i) if (mat25[i] < min_mat) min_mat = mat25[i];
    // packed kernel: scores fit a byte, suffix potentials fit a signed byte, biased scores stay >= 0
    const bool allow_fast = (long long)max_m * max_match < 256 && FLANK * max_match <= 120 && gap_open + min_mat >= 0 &&
                            gap_open >= 0 && gap_open <= 100 && gap_extend >= 0;
    for (int f = 0; f < nfamilies; ++f) {
        const tredsw_family &g = h_families[f];
        if (g.prefix_len < 1 || g.prefix_len > 32 || g.suffix_len < 1 || g.suffix_len > 32 || g.period < 1 ||
            g.period > 32 || g.max_units < 1 || g.max_units > 4096) { tredsw_set_error("family %d out of range", f); return TREDSW_ERR_ARG; }
        if (g.max_units > max_u) max_u = g.max_units;
        bool fast = allow_fast && g.prefix_len == FLANK && g.suffix_len == FLANK && g.period <= 12;
        if (fast) {
            need_fast = true;
            int nplan, nc;
            packed_plan(g, allow_fast, &nplan, &nc);
            if (nplan + 1 > nslots) nslots = nplan + 1;
        } else need_generic = true;
    }
    const int max_rows = max_m > 0 ? max_m : 1;
    const size_t rows_alloc = (size_t)max_rows + 2;
    const size_t smem = rows_alloc * 32 * 4 + rows_alloc * 32 + 64;
    size_t static_smem = 0;
    int rc;
    if ((rc = classify_static_smem(&static_smem))) return rc;
    if (smem + static_smem > ctx->smem_optin) {
        tredsw_set_error("reads too long for shared memory (%zu B)", smem + static_smem);
        return TREDSW_ERR_UNSUPPORTED;
    }
    ClassifyParams p{};
    p.rbuf = d_rbuf; p.roff = d_roff; p.families = d_families; p.out = d_out;
    const int ngroups = NCLASS * nfamilies;
    // read order: bins of predicted strips per group (one bin when the order is switched off; read on every call, so
    // that one process can compare both modes).  d_work is sized for tredsw_classify_bins bins per group.
    const bool conv_order = getenv("TREDSW_NO_CONVERGENCE_ORDER") == nullptr;
    const int nb = conv_order ? tredsw_classify_bins(h_families, nfamilies) : 1, nbins = ngroups * nb;
    int32_t *w = d_work;
    int32_t *d_count = w, *d_grp_start = w + nbins, *d_chunk_start = d_grp_start + ngroups + 1,
            *d_cursor = d_chunk_start + ngroups + 1, *d_order = d_cursor + nbins;
    CUDA_TRY(cudaMemsetAsync(d_count, 0, nbins * sizeof(int32_t), ctx->stream));
    const int tb = 256, nblk = (nreads + tb - 1) / tb;
    p.order = d_order; p.grp_start = d_grp_start; p.chunk_start = d_chunk_start;
    p.ngroups = ngroups; p.go = gap_open; p.ge = gap_extend; p.max_rows = max_rows;
    p.allow_fast = allow_fast ? 1 : 0;
    p.match = max_match > 0 ? max_match : 1;
    p.stats = d_stats;
    // (read on every call, so that one process can compare both modes)
    p.strip_skip = getenv("TREDSW_NO_STRIP_SKIP") == nullptr ? 1 : 0;
    if (!ctx->d_skip.p) {
        if ((rc = ctx->d_skip.ensure(TREDSW_STRIP_SKIP_STATS * sizeof(unsigned long long)))) return rc;
        CUDA_TRY(cudaMemsetAsync(ctx->d_skip.p, 0, TREDSW_STRIP_SKIP_STATS * sizeof(unsigned long long), ctx->stream));
    }
    p.skip_stats = ctx->d_skip.as<unsigned long long>();
    const int nitems_bound = nreads / 32 + ngroups + 1;
    int nctas = 0;
    if ((rc = persistent_ctas(ctx, smem, static_smem, need_fast, need_generic, &nctas))) return rc;
    if (nctas > nitems_bound) nctas = nitems_bound;
    // per-CTA scratch: scores [2*max_u][32] u16, potentials [rows][32] u32, then the two work counters
    const size_t score_bytes = (size_t)nctas * 2 * max_u * 32 * sizeof(uint16_t);
    const size_t pot_bytes = (size_t)nctas * rows_alloc * 32 * sizeof(uint32_t);
    const size_t gbnd_bytes = pot_bytes * (nslots + 1);
    const size_t perm_bytes = (((size_t)ngroups * sizeof(int32_t)) + 15) & ~(size_t)15;
    const size_t qtab_bytes = (size_t)nfamilies * 2 * QTAB_WORDS * sizeof(uint32_t);
    const size_t qinfo_bytes = (((size_t)nfamilies * sizeof(QgramInfo)) + 15) & ~(size_t)15;
    const size_t eff_bytes = (((size_t)nreads * sizeof(int32_t)) + 15) & ~(size_t)15;
    if ((rc = ctx->d_scratch.ensure(score_bytes + pot_bytes + gbnd_bytes + 16 + perm_bytes + qtab_bytes + qinfo_bytes + eff_bytes))) return rc;
    p.score_buf = ctx->d_scratch.as<uint16_t>();
    p.pot_buf = reinterpret_cast<uint32_t *>(ctx->d_scratch.as<unsigned char>() + score_bytes);
    p.gbnd_buf = reinterpret_cast<uint32_t *>(ctx->d_scratch.as<unsigned char>() + score_bytes + pot_bytes);
    p.nslots = nslots; p.one = 1u;
    p.counter = reinterpret_cast<int32_t *>(ctx->d_scratch.as<unsigned char>() + score_bytes + pot_bytes + gbnd_bytes);
    p.max_u = max_u;
    int32_t *d_perm = p.counter + 4;
    std::vector<int32_t> h_perm;
    {   // Item order: families grouped by loop instantiation (measured: mixing instantiations on an SM costs far
        // more than any order could gain — they compete for the instruction cache), the groups with the fewest
        // families first: their items run cold code and are the slowest, so they must not form the tail of the
        // launch; the big uniform group (period 3 for the catalogue) finishes it with short, even items.  The strand
        // classes of a family stay together, in class order, inside its instantiation's run.
        std::vector<int32_t> perm(ngroups);
        int group_size[33] = {0};
        for (int f = 0; f < nfamilies; ++f) ++group_size[instance_period(h_families[f].period)];
        for (int g = 0; g < ngroups; ++g) perm[g] = g;
        std::stable_sort(perm.begin(), perm.end(), [&](int a, int b) {
            const int pa = instance_period(h_families[a / NCLASS].period), pb = instance_period(h_families[b / NCLASS].period);
            if (group_size[pa] != group_size[pb]) return group_size[pa] < group_size[pb];
            return pa < pb; });
        h_perm.swap(perm);
    }
    p.grp_perm = d_perm;
    // q-gram pre-filter tables: per family 4096 x 2 bits (q-grams of all forward / all reverse-complement templates),
    // then 4096 x 2 bits for the pure repeat (convergence key)
    uint32_t *d_qtab = reinterpret_cast<uint32_t *>(reinterpret_cast<unsigned char *>(d_perm) + perm_bytes);
    QgramInfo *d_qinfo = reinterpret_cast<QgramInfo *>(reinterpret_cast<unsigned char *>(d_qtab) + qtab_bytes);
    int32_t *d_eff = reinterpret_cast<int32_t *>(reinterpret_cast<unsigned char *>(d_qinfo) + qinfo_bytes);
    {
        // q - 1 <= min(mismatch penalty, gap open); only for match == 1 and N scoring <= 0 everywhere
        int max_off = -128; bool n_ok = true, diag_ok = true;
        for (int i = 0; i < 5; ++i) for (int j = 0; j < 5; ++j) {
            const int v = mat25[i * 5 + j];
            if (i == 4 || j == 4) { if (v > 0) n_ok = false; }
            else if (i == j) { if (v != 1) diag_ok = false; }
            else if (v > max_off) max_off = v;
        }
        const int b_minus = -max_off;
        int q = 6;
        if (q > b_minus + 1) q = b_minus + 1;
        if (q > gap_open + 1) q = gap_open + 1;
        static const bool env_off = getenv("TREDSW_NO_PREFILTER") != nullptr;
        const bool usable = n_ok && diag_ok && q >= 4 && !env_off;
        // (read on every call, so that one process can compare both modes)
        const bool pairing = getenv("TREDSW_NO_STRAND_PAIRING") == nullptr;
        std::vector<uint32_t> tab((size_t)nfamilies * 2 * QTAB_WORDS, 0u);
        std::vector<QgramInfo> info(nfamilies);
        std::vector<int8_t> t;
        const uint32_t mask = (1u << (2 * q)) - 1u;
        // N in a template (GCN / NGC motifs) scores 0 against every base: such a pair neither breaks the score nor
        // earns it.  Count it as "compatible": runs of compatible pairs are broken by mismatches and gaps only, so the
        // same bound holds for q-grams compared with N as a wildcard — every q-gram of t with N's is expanded to the
        // concrete q-grams it is compatible with.  False when a q-gram holds too many N.
        auto add_grams = [&](uint32_t *tf) {
            const int n = (int)t.size();
            for (int i = 0; i + q <= n; ++i) {
                    // forward q-gram t[i..i+q) and the reverse complement's q-gram that covers the same bases
                    int npos[8], nn = 0;
                    uint32_t cf = 0, cr = 0;
                    for (int k = 0; k < q; ++k) {
                        const int c = t[i + k];
                        const bool isn = c < 0 || c > 3;
                        if (isn && nn < 8) npos[nn] = k;
                        if (isn) ++nn;
                        cf |= (uint32_t)(isn ? 0 : c) << (2 * (q - 1 - k));
                        cr |= (uint32_t)(isn ? 0 : 3 - c) << (2 * k);       // position k of the forward gram = q-1-k from the right
                    }
                    if (nn > 4) return false;
                    for (uint32_t e = 0; e < (1u << (2 * nn)); ++e) {       // all fillings of the N positions
                        uint32_t xf = cf, xr = cr;
                        for (int z = 0; z < nn; ++z) {
                            const uint32_t b = (e >> (2 * z)) & 3u;
                            xf |= b << (2 * (q - 1 - npos[z]));
                            xr |= (3u - b) << (2 * npos[z]);
                        }
                        xf &= mask; xr &= mask;
                        tf[xf >> 4] |= 1u << ((xf & 15u) * 2u);
                        tf[xr >> 4] |= 2u << ((xr & 15u) * 2u);
                    }
            }
            return true;
        };
        for (int f = 0; f < nfamilies; ++f) {
            const tredsw_family &g = h_families[f];
            info[f].q = usable ? q : 0;
            info[f].min_score = 30;                         // bam_parser.py:134: min_score = max(min_len, 30)
            info[f].pair = pairing && allow_fast && g.prefix_len == FLANK && g.suffix_len == FLANK && g.period <= 12;
            packed_plan(g, allow_fast && conv_order, &info[f].nplan, &info[f].nc);
            if (!info[f].q) continue;
            bool ok = true;
            // every q-gram of a template with u >= u0 units already occurs in the template with u0 units
            const int u0 = (q - 1 + g.period - 1) / g.period + 1;
            uint32_t *tf = tab.data() + (size_t)f * 2 * QTAB_WORDS;
            for (int u = 1; ok && u <= std::min(g.max_units, u0 + 1); ++u) {
                t.clear();
                for (int i = 0; i < g.prefix_len; ++i) t.push_back(g.prefix[i]);
                for (int k = 0; k < u; ++k) for (int i = 0; i < g.period; ++i) t.push_back(g.repeat[i]);
                for (int i = 0; i < g.suffix_len; ++i) t.push_back(g.suffix[i]);
                ok = add_grams(tf);
            }
            // the pure repeat repeat^(u0 + 1): every q-gram of any run of the repeat
            t.clear();
            for (int k = 0; k <= u0; ++k) for (int i = 0; i < g.period; ++i) t.push_back(g.repeat[i]);
            if (ok && info[f].nplan) ok = add_grams(tf + QTAB_WORDS);
            if (!ok) info[f].q = 0;
        }
        // perm | qtab | qinfo through the page-locked table staging (see stage_small): no pageable copy sits
        // between the input transfer and the kernels of a call
        const void *srcs[4] = {h_perm.data(), tab.data(), info.data(), mat25};
        const size_t sizes[4] = {(size_t)ngroups * sizeof(int32_t), qtab_bytes, (size_t)nfamilies * sizeof(QgramInfo), 25};
        size_t offs[4];
        if ((rc = stage_small(ctx, ctx->h_tab, srcs, sizes, 4, offs))) return rc;
        const unsigned char *ht = ctx->h_tab.as<unsigned char>();
        CUDA_TRY(cudaMemcpyToSymbolAsync(c_fmat25, ht + offs[3], 25, 0, cudaMemcpyHostToDevice, ctx->stream));
        CUDA_TRY(cudaMemcpyAsync(d_perm, ht + offs[0], sizes[0], cudaMemcpyHostToDevice, ctx->stream));
        CUDA_TRY(cudaMemcpyAsync(d_qtab, ht + offs[1], sizes[1], cudaMemcpyHostToDevice, ctx->stream));
        CUDA_TRY(cudaMemcpyAsync(d_qinfo, ht + offs[2], sizes[2], cudaMemcpyHostToDevice, ctx->stream));
    }
    ctx->mark(0);
    prefilter_kernel<<<nblk, tb, 0, ctx->stream>>>(d_rbuf, d_roff, nreads, d_read_family, nfamilies, d_families, d_qtab,
                                                   d_qinfo, nb, d_eff, d_stats);
    fam_count_kernel<<<nblk, tb, 0, ctx->stream>>>(d_eff, nreads, nbins, d_count);
    fam_scan_kernel<<<1, SCAN_THREADS, 0, ctx->stream>>>(d_count, ngroups, nb, d_perm, d_grp_start, d_chunk_start,
                                                         d_cursor);
    fam_scatter_kernel<<<nblk, tb, 0, ctx->stream>>>(d_eff, nreads, nbins, nb, d_grp_start, d_cursor, d_order, p.out);
    CUDA_TRY(cudaGetLastError());
    ctx->launches += 4;
    CUDA_TRY(cudaMemsetAsync(p.counter, 0, 2 * sizeof(int32_t), ctx->stream));
    if (ctx->wait_before_sw) {            // compute token of the host-buffer pipeline (common.cuh: DeviceToken)
        CUDA_TRY(cudaStreamWaitEvent(ctx->stream, ctx->wait_before_sw, 0));
        ctx->wait_before_sw = nullptr;
    }
    if (need_generic) { if ((rc = launch_classify<false>(ctx, p, nctas, smem))) return rc; }
    if (need_fast) { if ((rc = launch_classify<true>(ctx, p, nctas, smem))) return rc; }
    if (ctx->record_sw_end && ctx->sw_end_ev) {
        CUDA_TRY(cudaEventRecord(ctx->sw_end_ev, ctx->stream));
        ctx->record_sw_end = false;
    }
    ctx->mark(1);
    return TREDSW_OK;
}

extern "C" int tredsw_classify_reads(tredsw_ctx *ctx, const int8_t *rbuf, const int64_t *roff, int32_t nreads,
                                     const int32_t *read_family, const tredsw_family *families,
                                     int32_t nfamilies, const int8_t *mat25, int gap_open, int gap_extend,
                                     uint32_t flags, int32_t *out, int64_t *stats) {
    if (!ctx) { tredsw_set_error("null context"); return TREDSW_ERR_ARG; }
    if (nreads < 0 || nfamilies <= 0 || !families || !mat25 || !out) { tredsw_set_error("bad arguments"); return TREDSW_ERR_ARG; }
    if (nreads == 0) return TREDSW_OK;
    if (dev_ptrs(flags)) { tredsw_set_error("tredsw_classify_reads takes host buffers; device-resident batches go through tredsw_genotype_batch"); return TREDSW_ERR_UNSUPPORTED; }
    std::lock_guard<std::mutex> lock(ctx->mu);
    CUDA_TRY(cudaSetDevice(ctx->device));
    int max_m = 0;
    for (int i = 0; i < nreads; ++i) { int l = (int)(roff[i + 1] - roff[i]); if (l > max_m) max_m = l; }
    int rc;
    const int8_t *d_rbuf; const int64_t *d_roff; const int32_t *d_rfam; const tredsw_family *d_fam;
    if ((rc = stage_in(ctx, ctx->d_q, rbuf, (size_t)roff[nreads], flags, &d_rbuf))) return rc;
    if ((rc = stage_in(ctx, ctx->d_qoff, roff, (size_t)nreads + 1, flags, &d_roff))) return rc;
    if ((rc = stage_in(ctx, ctx->d_rfam, read_family, (size_t)nreads, flags, &d_rfam))) return rc;
    if ((rc = stage_in(ctx, ctx->d_fam, families, (size_t)nfamilies, flags, &d_fam))) return rc;
    if ((rc = ctx->d_out.ensure((size_t)nreads * 8 * sizeof(int32_t)))) return rc;
    if ((rc = ctx->d_work.ensure(tredsw_classify_work_words(families, nfamilies, nreads) * sizeof(int32_t)))) return rc;
    if ((rc = ctx->d_stats.ensure(4 * sizeof(unsigned long long)))) return rc;
    CUDA_TRY(cudaMemsetAsync(ctx->d_stats.p, 0, 4 * sizeof(unsigned long long), ctx->stream));
    if ((rc = tredsw_internal_classify(ctx, d_rbuf, d_roff, nreads, d_rfam, d_fam, families, nfamilies, max_m, mat25,
                                       gap_open, gap_extend, ctx->d_work.as<int32_t>(), ctx->d_out.as<int32_t>(),
                                       stats ? ctx->d_stats.as<unsigned long long>() : nullptr))) return rc;
    CUDA_TRY(cudaMemcpyAsync(out, ctx->d_out.p, (size_t)nreads * 8 * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    if (stats) CUDA_TRY(cudaMemcpyAsync(stats, ctx->d_stats.p, 4 * sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return TREDSW_OK;
}
