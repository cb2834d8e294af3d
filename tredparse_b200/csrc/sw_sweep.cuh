// sw_sweep.cuh — scalar (one thread = one alignment) affine-gap local-alignment sweeps.
//
// These device functions are the position-exact building block of both the generic pairs kernel
// (sw_pairs.cu) and the second phase of the family kernel (sw_family.cu).  They evaluate the plain
// Gotoh recurrence that src/ssw.c's striped kernels are value-equivalent to (SURVEY.md Appendix A, Q4):
//
//     H[i][j]   = max(0, H[i-1][j-1] + s(t[i], q[j]), E[i][j], F[i][j])
//     E[i+1][j] = max(0, E[i][j] - ge, H[i][j] - go)        F[i][j+1] = max(0, F[i][j] - ge, H[i][j] - go)
//
// Layout: a thread walks the template in strips of W columns held in registers (previous-row H and the
// running F of each strip column), streaming the query rows; the H/E column leaving a strip goes
// through a per-thread boundary column in scratch memory (one 32-bit word per row: H | E << 16).
// Substitution scores come from one PRMT per cell: the query base selects a 2-word LUT (the matrix
// column of that base as int8 bytes), the template base is a byte selector with sign replication.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

// Codes: 0..3 = A,C,G,T ; 4 = N ; 5 = ghost (query side: score 0 against everything; template side:
// "dead" column scoring -128 so that nothing can start or improve there).
#define SW_CODE_GHOST 5

struct SwLut {
    uint32_t w0[6];   // bytes [t=0..3] = mat[t][q]
    uint32_t w1[6];   // byte0 = mat[4][q], byte1 = 0x80 (dead column)
};

// Build the LUT from a 5x5 int8 matrix (row = template code, column = query code).
__device__ __forceinline__ void sw_build_lut(SwLut *lut, const int8_t *mat25, int tid, int nthreads) {
    for (int q = tid; q < 6; q += nthreads) {
        uint32_t w0 = 0, w1 = 0x00008000u;
        if (q < 5) {
            for (int t = 0; t < 4; ++t) w0 |= (uint32_t)(uint8_t)mat25[t * 5 + q] << (8 * t);
            w1 |= (uint32_t)(uint8_t)mat25[4 * 5 + q];
        }
        lut->w0[q] = w0;
        lut->w1[q] = w1;
    }
}

// PRMT with the full selector semantics (bit 3 of a selector nibble replicates the sign of the selected
// byte).  The __byte_perm() intrinsic masks the selector with 0x7777, which loses exactly that bit.
__device__ __forceinline__ uint32_t sw_prmt(uint32_t a, uint32_t b, uint32_t sel) {
    uint32_t d;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
    return d;
}

// byte selector producing a sign-extended 32-bit score for template code t (0..5)
__device__ __forceinline__ uint32_t sw_sel32(int t) { return 0x8880u + 0x1111u * (uint32_t)t; }

// MODE 0: maximum score over the whole matrix (optionally per-column maxima to colmax_out).
// MODE 1: locate `target`: the first strip that holds a cell equal to target ends the sweep; among such
//         cells the smallest column, then the smallest row (< m_real) is returned (out_col/out_row);
//         out_col < 0 when the value never occurs.
//
// Band [dlo, dhi] on the diagonal offset d = column - row (pass SW_NO_BAND for none): rows whose cells in
// a strip all lie outside the band are skipped and read as zero.  This is exact for MODE 1 whenever every
// path that can end with score == target is known to stay inside the band (a skipped cell only removes
// paths, so no cell can exceed its true value and a cell equal to target is still reached by a real
// path): see sw_band_* below for the bounds used.
#define SW_NO_BAND_LO (-0x3fffffff)
#define SW_NO_BAND_HI (0x3fffffff)

template <int W, int MODE, bool COLMAX, class RowCode, class ColCode>
__device__ __forceinline__ int sw_sweep(int m_real, int m_rows, int n, RowCode rowcode, ColCode colcode,
                                        const SwLut *lut, uint32_t *bnd, int stride, int go, int ge,
                                        int target, int *out_col, int *out_row, int32_t *colmax_out,
                                        int dlo = SW_NO_BAND_LO, int dhi = SW_NO_BAND_HI,
                                        unsigned long long *visited = nullptr) {
    static_assert(W <= 32, "hit columns of a row are kept as a 32-bit mask");
    int mx = 0;
    int best_col = 0x7fffffff, best_row = 0;
    const int mge = -ge;
    int jlo_prev = 0, jhi_prev = 0;            // rows the previous strip wrote to the boundary column
    for (int c0 = 0; c0 < n; c0 += W) {
        uint32_t sel[W];
        int Hrow[W], F[W], cm[W];
#pragma unroll
        for (int c = 0; c < W; ++c) {
            int code = (c0 + c < n) ? colcode(c0 + c) : SW_CODE_GHOST;
            sel[c] = sw_sel32(code);
            Hrow[c] = 0; F[c] = 0; cm[c] = 0;
        }
        const bool first = (c0 == 0);
        const bool last = (c0 + W >= n);
        // rows of this strip that intersect the band: d = c - j in [dlo, dhi] for some c in [c0, c0+W)
        const int jlo = max(0, c0 - dhi);
        const int jhi = min(m_rows, c0 + W - dlo);         // exclusive; c0 + W - 1 - dlo inclusive
        int hin_prev = 0;
        if (!first && jlo > 0 && jlo - 1 >= jlo_prev && jlo - 1 < jhi_prev)
            hin_prev = (int)(bnd[(size_t)(jlo - 1) * stride] & 0xffffu);
        // One DP cell of column c: hd = H diagonal in, H(above) read from / H written to Hrow[c], e = E along the row.
        auto cell = [&](int &hd, int &e, int c, uint32_t w0, uint32_t w1) {
            const int s = (int)sw_prmt(w0, w1, sel[c]);
            const int t = max(e, F[c]);
            const int h = __viaddmax_s32_relu(hd, s, t);
            hd = Hrow[c];
            Hrow[c] = h;
            const int hgo = h - go;
            e = __viaddmax_s32_relu(e, mge, hgo);
            F[c] = __viaddmax_s32_relu(F[c], mge, hgo);
            return h;
        };
        auto entering = [&](int j, int &hin, int &e) {
            hin = 0; e = 0;
            if (!first && j >= jlo_prev && j < jhi_prev) {
                const uint32_t b = bnd[(size_t)j * stride];
                hin = (int)(b & 0xffffu);
                e = (int)(b >> 16);
            }
        };
        // Rows in pairs, two dependency chains in flight: row j at column s while row j+1 is at column s-1 (row j+1's
        // cell needs row j's cell of the same column, done one step earlier).  Same cells as one row at a time; the hit
        // rule is kept: per row the smallest hit column, rows in order, a later row only wins with a smaller column.
        int j = jlo;
        for (; j + 1 < jhi; j += 2) {
            int hinA, eA, hinB, eB;
            entering(j, hinA, eA);
            entering(j + 1, hinB, eB);
            const int codeA = rowcode(j), codeB = rowcode(j + 1);
            const uint32_t w0A = lut->w0[codeA], w1A = lut->w1[codeA], w0B = lut->w0[codeB], w1B = lut->w1[codeB];
            int hdA = hin_prev, hdB = hinA;
            hin_prev = hinB;
            int hA = 0, hB = 0;
            uint32_t hitA = 0u, hitB = 0u;           // hit columns of each row (bit c)
#pragma unroll
            for (int s = 0; s <= W; ++s) {
                if (s < W) {
                    hA = cell(hdA, eA, s, w0A, w1A);
                    if (MODE == 1) hitA |= (hA == target) ? (1u << s) : 0u;
                    else if (COLMAX) cm[s] = max(cm[s], hA);
                    else mx = max(mx, hA);
                }
                if (s >= 1) {
                    hB = cell(hdB, eB, s - 1, w0B, w1B);
                    if (MODE == 1) hitB |= (hB == target) ? (1u << (s - 1)) : 0u;
                    else if (COLMAX) cm[s - 1] = max(cm[s - 1], hB);
                    else mx = max(mx, hB);
                }
            }
            if (!last) {
                bnd[(size_t)j * stride] = (uint32_t)hA | ((uint32_t)eA << 16);
                bnd[(size_t)(j + 1) * stride] = (uint32_t)hB | ((uint32_t)eB << 16);
            }
            if (MODE == 1) {
                if (hitA && j < m_real && c0 + __ffs(hitA) - 1 < best_col) { best_col = c0 + __ffs(hitA) - 1; best_row = j; }
                if (hitB && j + 1 < m_real && c0 + __ffs(hitB) - 1 < best_col) { best_col = c0 + __ffs(hitB) - 1; best_row = j + 1; }
            }
        }
        for (; j < jhi; ++j) {                       // the last row of an odd count
            int hin = 0, e = 0;
            if (!first && j >= jlo_prev && j < jhi_prev) {
                uint32_t b = bnd[(size_t)j * stride];
                hin = (int)(b & 0xffffu);
                e = (int)(b >> 16);
            }
            const int code = rowcode(j);
            const uint32_t w0 = lut->w0[code], w1 = lut->w1[code];
            int hd = hin_prev;
            hin_prev = hin;
            int h = 0;
            bool hit = false;
#pragma unroll
            for (int c = 0; c < W; ++c) {
                const int s = (int)sw_prmt(w0, w1, sel[c]);
                const int t = max(e, F[c]);
                h = __viaddmax_s32_relu(hd, s, t);
                hd = Hrow[c];
                Hrow[c] = h;
                const int hgo = h - go;
                e = __viaddmax_s32_relu(e, mge, hgo);
                F[c] = __viaddmax_s32_relu(F[c], mge, hgo);
                if (MODE == 1) hit |= (h == target);
                else if (COLMAX) cm[c] = max(cm[c], h);
                else mx = max(mx, h);
            }
            if (!last) bnd[(size_t)j * stride] = (uint32_t)h | ((uint32_t)e << 16);
            if (MODE == 1 && hit && j < m_real) {
#pragma unroll
                for (int c = 0; c < W; ++c) {
                    if (Hrow[c] == target && c0 + c < best_col) { best_col = c0 + c; best_row = j; }
                }
            }
        }
        jlo_prev = jlo; jhi_prev = jhi;
        if (visited && jhi > jlo) *visited += (unsigned long long)(jhi - jlo) * W;
        if (MODE == 0 && COLMAX) {
#pragma unroll
            for (int c = 0; c < W; ++c) {
                if (c0 + c < n) { colmax_out[c0 + c] = cm[c]; mx = max(mx, cm[c]); }
            }
        }
        if (MODE == 1 && best_col != 0x7fffffff) break;
    }
    if (MODE == 1) {
        *out_col = (best_col == 0x7fffffff) ? -1 : best_col;
        *out_row = best_row;
    }
    return mx;
}

// Largest diagonal deviation a path can afford and still END with score `target`: every aligned pair
// scores at most `match`, a path uses at most min(m, n) pairs, and drifting d diagonals costs at least
// go + (d - 1) * ge.  (d < 0: no drift possible beyond 0.)
__device__ __forceinline__ int sw_max_drift(int target, int m, int n, int match, int go, int ge) {
    const int slack = min(m, n) * match - target - go;     // budget left for gap extension after one opening
    if (slack < 0) return 0;
    return ge > 0 ? 1 + slack / ge : 0x3ffffff;
}

// Post-filter (src/ssw_wrap.py:213-220) + classification (tredparse/bam_parser.py:133-168).
__device__ __forceinline__ int sw_classify(int score, int rb, int re, int qb, int qe, int m, int n, int u,
                                           int period, int max_units_eff) {
    const int FLANKMATCH = 9;
    int min_len = min(m, n) / 2;
    int min_score = max(min_len, 30);
    if (!(score >= min_score && (qe - qb + 1) >= min_len)) return TREDSW_TAG_NONE;
    bool prefix_read = rb < FLANKMATCH;
    bool suffix_read = re > n - FLANKMATCH - 1;
    int aL = rb, aR = n - re - 1, bL = qb, bR = m - qe - 1;
    int hang = min(min(aR + bL, aL + bR), min(aL + aR, bL + bR));
    if (hang >= FLANKMATCH) return TREDSW_TAG_HANG;
    if (prefix_read) return suffix_read ? TREDSW_TAG_FULL : TREDSW_TAG_PREF;
    if (suffix_read) return TREDSW_TAG_POST;
    if (u >= max_units_eff - 1 && u * period <= m) return TREDSW_TAG_REPT;
    return TREDSW_TAG_NONE;
}
