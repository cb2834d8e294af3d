// grid.cu — the (h1, h2) log-likelihood surface of IntegratedCaller and its reductions, FP64.
//
// Replaces the double loop of tredparse/models.py:260-273 (evaluate_spanning / evaluate_partial /
// evaluate_rept / PEMaxLikModel.evaluate at every candidate pair) and the reductions of
// models.py:277-302, 304-317, 342-368 (max, arg-max with key (ml, -h1), exp-normalised marginals, the sparse
// joint posterior, PP sums).
//
// The reference materialises length-1000 probability vectors per candidate allele and takes the log of whole
// vectors at every grid point; only the entries at the observed keys are ever used.  Here a point is evaluated
// from the closed forms of SURVEY.md Appendix B:
//   PS(h)[k]  spanning pdf (models.py:149-168, quirks Q6/Q7)     PT(h)[k] partial pdf (:170-180, Q8)
//   alpha     mixing weights (:182-190)                           R(h)[x]  rolled PE pdf (:441-458)
// and a sum of logarithms  sum_k c_k log(max(v_k, eps))  is taken as the logarithm of the running PRODUCT of the
// v_k (flushed every 64 factors: v_k >= eps = e^-10 keeps 64 factors above e^-640) plus log(eps) times the
// number of floored factors — one FP64 log per term and point instead of one per observed key (rounding
// differs from the reference's sum by ~1e-16 relative; the parity bar is 1e-9).
//
// THE SURFACE IS NOT MATERIALISED (unless the caller asks for it).  What the caller of the reference gets are
// the call, the marginals P_h1 / P_h2, the sparse joint P_h1h2 and the PP sums; so:
//   * small surfaces (<= 512 points, every haploid problem) are cut into work items of 256 points — one warp per
//     item, whatever the mix of sizes — that park the ml values in the problem's scratch slot (L1/L2); one warp
//     per problem then reduces and emits;
//   * large surfaces: row-structured.  A warp owns rows (one h1), its lanes walk the columns (h2) in chunks of
//     256; everything that depends on h1 only is hoisted out of the columns.  Where the longer allele lies
//     beyond every observed key, the partial clamp and the read length (column index >= fam, the MID region)
//     the spanning and partial terms depend on h1 only; where it is also shifted past the KDE support
//     (>= fa2, the FAR region) so does the paired-end term; the repeat-only term is a function of
//     dsum = max(h1-L,1) + max(h2-L,1) everywhere.  With per-row tables {c12(h1), pe(h1)} and rept[dsum] a far
//     point is  ml = (c12 + rept[dsum]) + pe  — on a --fullsearch / long-expansion grid > 90 % of the points —
//     and its weight exp(ml - max) = exp(c12 + pe - max) * exp(rept[dsum]): one multiply with a per-row factor
//     and a tabulated exp(rept) (rept lies in [-100, 0], so neither factor can overflow).
//     Pass A (rows_eval) evaluates the near / mid points into the scratch slot — the paired-end term of 8 columns
//     per lane at once, pair lengths outer: 8 independent product chains fed by one uniform and 8 coalesced loads
//     — and finds the maximum and the arg-max (Q10); pass B (grid_rows_reduce_kernel) accumulates row sums, column
//     sums (registers -> shared memory -> per-CTA partials, summed by the last CTA of the problem in rank order:
//     deterministic), the PP sums and emits the joint-posterior entries >= e^-10.
// Four launches per call: classify | {point items, table setup} | {small reductions, pass A} | pass B.
// DRAM traffic is the near-region scratch (a few % of the surface, L2-resident) plus the tables.
#include "internal.cuh"
#include "kde.cuh"
#include <math.h>

namespace {

constexpr int SPAN = 1000;
constexpr int NSTEP = 37;
constexpr int DEV = 18;
constexpr long long SMALL_LIMIT = 512;    // <= : point items + one warp for the reductions
constexpr int ITEM_POINTS = 256;          // points per work item of a small surface (8 per lane)
constexpr int ITEM_MAX = 12;              // items per small surface (an item strides when there are more chunks)
constexpr int NC_MAX = 32;                // CTAs per large surface (rows are dealt round-robin in groups of 8)
constexpr int CHUNK = 256;                // columns per chunk: 8 per lane
constexpr int FILL_SPLIT = 8;             // blocks per large surface filling its tables
constexpr int PE_BLOCK = 64;              // factors per flush of the paired-end product

// per large surface: constants, thresholds, table layout (written by the classify / setup kernels)
struct BigInfo {
    long long off;               // table arena offset (doubles)
    double lgamma_k1;            // lgamma(n_rept + 1)
    double sig_mp;               // sigma(max_partial)
    int tmin;                    // smallest pair length >= MINPE (after numpy's negative-index wrap); INT_MAX if none
    int fam, fa2;                // first column of the mid / far region
    int ok;                      // row / rept / sigma tables present
    int npe;                     // paired-end operand tables present (= n_target)
    int sorted;                  // both candidate lists non-decreasing: rows skip the h1 > h2 columns wholesale
    int nd;                      // entries of rept[] / erept[]
    int hrep;                    // a far allele (the largest h2)
    int mx1;                     // largest h1
    int nc;                      // CTA slots allocated for this surface
    int nce;                     // CTAs actually working on it (chosen once the number of large surfaces is known)
    int nb1, nb2;                // length of the sorted base part of the h1 / h2 list (duplicates live beyond it)
    int patho_mode;              // the PP predicate for h1 <= h2: 0 = by column (h2), 1 = by row (h1)
    int far_arith;               // the far columns are an arithmetic sequence above the read length:
    int far_d0, far_step;        //   max(h2s[col] - L, 1) = far_d0 + far_step * (col - fa2)  (no list load per point)
    int has_dup;                 // a candidate occurs twice (Q9)
    int h2_arith, h2_a0, h2_step; // the whole h2 list is h2_a0 + h2_step * col (step > 0): lower bounds need no search
    unsigned int done_b;         // CTAs of pass B that have finished
};

struct GridParams {
    const tredsw_grid_problem *prob;
    const int32_t *ipool;
    const double *dpool;
    double *surface;             // per-problem slots (off_surface): scratch, or the full surface when materialise
    double *marg;
    tredsw_grid_result *res;
    double small_value, log_small;
    int nproblems;
    int materialise;             // write every point (and -inf where h1 > h2) into the surface slots
    int tables;                  // best table tier a large surface may take: 0 full, 1 without PE operands, 2 none
    BigInfo *big;                // [nproblems]
    int *lists;                  // [0] number of large surfaces, [1 + i] their problem indices
    int *items;                  // point items of the small surfaces: (problem, chunk, nitems) triples
    int *row_items;              // work items of the row kernels: (problem, CTA rank) pairs
    unsigned int *counters;      // [0] items, [1] work cursor pass A, [2] work cursor pass B, [3] item cursor, [4] row items
    double *ftab;                // table arena
    long long ftab_cap;
    unsigned long long *fcursor; // [0] arena cursor, [1] overflow flag
    tredsw_posterior *post;      // sparse joint-posterior entries (optional)
    long long post_cap;
    unsigned long long *post_cursor;
    int nblk_small;              // horizontally fused launches: blocks [0, nblk_small) work on the small surfaces
    int target_ctas;             // CTAs the row kernels should spread the large surfaces over
};

// table layout of one large surface, in doubles from BigInfo.off
struct Tab {
    long long colpart, partial, pa, dup, rows, sig1, sig2, rept, erept, R1, R2, end;
};
__host__ __device__ inline Tab tab_layout(int n1, int n2, int nd, int npe, int nc, bool with_tables) {
    Tab t;
    long long o = 0;
    t.colpart = o; o += (long long)nc * n2;                  // pass B: column sums of each CTA
    t.partial = o; o += (long long)nc * 4;                   // pass B: {sum_all, sum_path, sum_dup} of each CTA
    t.pa = o; o += (long long)nc * 4;                        // pass A: {max ml, arg key, points} of each CTA
    t.dup = o; o += ((long long)n1 + n2 + 1) / 2;            // int32 flags, two per double
    t.rows = o; if (with_tables) o += 3LL * n1;              // {c12, pe_far, f} per row
    t.sig1 = o; if (with_tables) o += n1;
    t.sig2 = o; if (with_tables) o += n2;
    t.rept = o; if (with_tables) o += nd;                    // repeat-only term per dsum
    t.erept = o; if (with_tables) o += nd;                   // exp of it
    t.R1 = o; if (with_tables) o += (long long)npe * n1;     // 0.5 * rolled pdf of h1 at pair length t
    t.R2 = o; if (with_tables) o += (long long)npe * n2;     // 0.5 * rolled pdf of h2 (stride fa2)
    t.end = (o + 1) & ~1LL;
    return t;
}

__device__ __forceinline__ double sigma_h(const tredsw_grid_problem &P, int h) {
    double z = __dadd_rn(P.stutter_a, __dmul_rn(P.stutter_w2, (double)(h / P.period)));
    z = __dadd_rn(__dadd_rn(z, P.stutter_c3), P.stutter_c4);
    return 1.0 / (1.0 + exp(-1.0 * z));
}

// spanning pdf of allele h at key k given sig = sigma(h)
__device__ __forceinline__ double pdf_span(const double *step, int h, double sig, int k) {
    if (k < 0 || k >= SPAN) return 0.0;
    int idx;
    if (h + DEV + 1 <= SPAN) {
        idx = k - h + DEV;                      // also covers the low-end clip (h < 18): tail of p
    } else {
        if (k < h - DEV) return 0.0;            // high-end clip copies the *tail* of p as well (Q6)
        idx = k - (SPAN - NSTEP);
    }
    if (idx < 0 || idx >= NSTEP) return 0.0;
    return idx == DEV ? (1.0 - sig) : __dmul_rn(step[idx], sig);
}

__device__ __forceinline__ double pdf_part(const double *step, int hc, double sig_c, double c, int k) {
    const double v = (k < hc) ? c : 0.0;
    return __dadd_rn(v, __dmul_rn(c, pdf_span(step, hc, sig_c, k)));
}

__device__ __forceinline__ double pe_roll(const double *pdf, int h, int ref, int minpe, int x, double eps) {
    if (x < minpe) return eps;
    const int y = x + h - ref;
    if (y < 0 || y >= SPAN) return eps;
    return pdf[y];
}

// sum_k c_k log(v_k) as the log of a running product; every factor lies in (eps, 1], so 64 of them stay above
// e^-640.  The explicit intrinsics keep the compiler from contracting differently in different call sites: the
// table-driven and the direct evaluation of a point have to give the same bits.
struct LogProd {
    double acc, prod;
    int room;
    __device__ __forceinline__ LogProd() : acc(0.0), prod(1.0), room(64) {}
    __device__ __forceinline__ void flush() {
        if (room != 64) { acc = __dadd_rn(acc, log(prod)); prod = 1.0; room = 64; }
    }
    __device__ __forceinline__ void mul(double v) {
        prod = __dmul_rn(prod, v);
        if (--room == 0) flush();
    }
    __device__ __forceinline__ void mulc(double v, int c) {
        if (c > 4) acc = __dadd_rn(acc, __dmul_rn((double)c, log(v)));
        else for (int q = 0; q < c; ++q) mul(v);
    }
    __device__ __forceinline__ double done() { flush(); return acc; }
};

// ---- the four terms of one point -------------------------------------------------------------------------
// sg1 / sg2: sigma(h1) / sigma(h2) when the caller has them (row / column tables), negative = compute on
// first use.  A key farther than 18 from both alleles sees 0 -> floored to eps.
__device__ __forceinline__ double term_span(const tredsw_grid_problem &P, const GridParams &g, int h1, int h2,
                                            double sg1, double sg2) {
    if (P.n_span <= 0) return 0.0;
    const int32_t *skey = g.ipool + P.off_span, *scnt = skey + P.n_span;
    const double *step = g.dpool + P.off_step;
    const double eps = g.small_value;
    const int t2 = P.readlen - 18;
    const int s1 = max(0, t2 - h1), s2 = max(0, t2 - h2);
    const double a = (s1 + s2) ? (double)s1 * 1.0 / (double)(s1 + s2) : 0.5;
    const double b = 1.0 - a;
    const int lo = min(h1, h2) - DEV, hi = max(h1, h2) + DEV;
    LogProd lp;
    int nfloor = 0;
    for (int i = 0; i < P.n_span; ++i) {
        const int k = skey[i], c = scnt[i];
        if (k < lo || k > hi) { nfloor += c; continue; }
        if (sg1 < 0.0) sg1 = sigma_h(P, h1);
        if (sg2 < 0.0) sg2 = sigma_h(P, h2);
        const double v = __dadd_rn(__dmul_rn(a, pdf_span(step, h1, sg1, k)), __dmul_rn(b, pdf_span(step, h2, sg2, k)));
        if (v <= eps) { nfloor += c; continue; }
        lp.mulc(v, c);
    }
    return __dadd_rn(lp.done(), __dmul_rn((double)nfloor, g.log_small));
}

// sgc1 / sgc2: sigma of the alleles clamped to max_partial (negative = compute on first use).
// With A <= B the clamped alleles, a partial key k sees (models.py:170-180: c [k < hc] + c PS(hc)[k])
//   k < A-18        : alpha_A c_A + alpha_B c_B         (below both, no stutter mass)            "bulk"
//   A+18 < k < B-18 : alpha_A 0   + alpha_B c_B         (past A altogether, still below B)       "between"
//   k > B+18        : 0                                  -> floored
// and only the keys within 18 of A or B need the stutter pdf.  Same products and sums as the plain formula.
__device__ __forceinline__ double term_part(const tredsw_grid_problem &P, const GridParams &g, int h1, int h2,
                                            double sgc1, double sgc2, double sig_mp) {
    if (P.n_part <= 0) return 0.0;
    const int32_t *pkey = g.ipool + P.off_part, *pcnt = pkey + P.n_part;
    const double *step = g.dpool + P.off_step;
    const double eps = g.small_value;
    const int t1 = P.readlen - 9;
    const int s1 = min(h1, t1), s2 = min(h2, t1);
    const double a = (s1 + s2) ? (double)s1 * 1.0 / (double)(s1 + s2) : 0.5;
    const double b = 1.0 - a;
    const int hc1 = min(h1, P.max_partial), hc2 = min(h2, P.max_partial);
    const double c1 = 1.0 / (double)(hc1 + 1), c2 = 1.0 / (double)(hc2 + 1);
    const int A = min(hc1, hc2), B = max(hc1, hc2);
    const double v_bulk = __dadd_rn(__dmul_rn(a, c1), __dmul_rn(b, c2));   // p1 = c1 + c1 * 0, p2 = c2 + c2 * 0
    // between: the smaller clamped allele contributes 0, the larger its plateau
    const double v_btw = hc1 <= hc2 ? __dadd_rn(__dmul_rn(a, 0.0), __dmul_rn(b, c2)) : __dadd_rn(__dmul_rn(a, c1), __dmul_rn(b, 0.0));
    LogProd lp;
    int nfloor = 0, nbulk = 0, nbtw = 0;
    for (int i = 0; i < P.n_part; ++i) {
        const int k = pkey[i], c = pcnt[i];
        if (k < A - DEV) { nbulk += c; continue; }
        if (k > B + DEV) { nfloor += c; continue; }
        if (k > A + DEV && k < B - DEV) { nbtw += c; continue; }
        if (sgc1 < 0.0) sgc1 = hc1 == P.max_partial ? sig_mp : sigma_h(P, hc1);
        if (sgc2 < 0.0) sgc2 = hc2 == P.max_partial ? sig_mp : sigma_h(P, hc2);
        const double v = __dadd_rn(__dmul_rn(a, pdf_part(step, hc1, sgc1, c1, k)), __dmul_rn(b, pdf_part(step, hc2, sgc2, c2, k)));
        if (v <= eps) { nfloor += c; continue; }
        lp.mulc(v, c);
    }
    double acc = lp.done();
    if (nbulk) {
        if (v_bulk <= eps) nfloor += nbulk;
        else acc = __dadd_rn(acc, __dmul_rn((double)nbulk, log(v_bulk)));
    }
    if (nbtw) {
        if (v_btw <= eps) nfloor += nbtw;
        else acc = __dadd_rn(acc, __dmul_rn((double)nbtw, log(v_btw)));
    }
    return __dadd_rn(acc, __dmul_rn((double)nfloor, g.log_small));
}

// repeat-only reads: Poisson (scipy: exp(xlogy(k, mu) - gammaln(k + 1) - mu)); dsum = max(h1-L,1) + max(h2-L,1)
__device__ __forceinline__ double term_rept(const tredsw_grid_problem &P, int dsum, double lgamma_k1) {
    const double mu = (double)dsum * P.half_depth / (double)P.readlen;
    const double kk = (double)P.n_rept;
    const double xl = (P.n_rept == 0) ? 0.0 : __dmul_rn(kk, log(mu));
    const double pk = __dsub_rn(__dsub_rn(xl, lgamma_k1), mu);
    // log(max(exp(pk), e^-100)): log(exp(pk)) is pk to within an ulp of the pmf (~1e-16 absolute on a term
    // of magnitude 0.1..100, far inside the 1e-9 relative bar)
    return pk > -100.0 ? pk : -100.0;
}

// paired-end term: sum_t log(max(.5 R(h1)[x_t] + .5 R(h2)[x_t], eps)) as the log of the product of the floored
// mixtures, flushed every PE_BLOCK pairs (64 factors >= e^-10 stay above e^-640); the row kernels evaluate the
// same blocks from tabulated halves, 8 columns at a time
__device__ __forceinline__ double term_pe(const tredsw_grid_problem &P, const GridParams &g, int h1, int h2, int tmin) {
    if (!P.run_pe) return 0.0;
    const double eps = g.small_value;
    const double *pdf = g.dpool + P.off_pdf;
    const int32_t *tl = g.ipool + P.off_target;
    double acc = 0.0;
    const long long off1 = (long long)h1 - P.pe_ref, off2 = (long long)h2 - P.pe_ref;
    if (tmin == 0x7fffffff || (tmin + off1 >= SPAN && tmin + off2 >= SPAN)) {
        // every pair length is below MINPE or shifted past the end of the support: every factor is eps
        // (.5 eps + .5 eps); the same blocks of products as below, without touching the pdf
        for (int t0 = 0; t0 < P.n_target; t0 += PE_BLOCK) {
            double prod = 1.0;
            const int t1 = min(t0 + PE_BLOCK, P.n_target);
            for (int i = t0; i < t1; ++i) prod = __dmul_rn(prod, eps);
            acc = __dadd_rn(acc, log(prod));
        }
        return acc;
    }
    for (int t0 = 0; t0 < P.n_target; t0 += PE_BLOCK) {
        double prod = 1.0;
        const int t1 = min(t0 + PE_BLOCK, P.n_target);
        for (int i = t0; i < t1; ++i) {
            int x = tl[i];
            if (x < 0) x += SPAN;               // numpy negative-index wrap (models.py:473)
            const double r1 = pe_roll(pdf, h1, P.pe_ref, P.pe_minpe, x, eps);
            const double r2 = pe_roll(pdf, h2, P.pe_ref, P.pe_minpe, x, eps);
            prod = __dmul_rn(prod, fmax(__dadd_rn(__dmul_rn(0.5, r1), __dmul_rn(0.5, r2)), eps));
        }
        acc = __dadd_rn(acc, log(prod));
    }
    return acc;
}

struct ProblemConsts {
    double lgamma_k1;      // lgamma(n_rept + 1) of the Poisson term
    double sig_mp;         // sigma(max_partial): the stutter probability of every allele clamped to max_partial
    int tmin;              // smallest pair length >= MINPE (after numpy's negative-index wrap); INT_MAX if none
};

__device__ __forceinline__ double point_ml(const tredsw_grid_problem &P, const GridParams &g, int h1, int h2,
                                           const ProblemConsts &T) {
    double ml = term_span(P, g, h1, h2, -1.0, -1.0);
    ml = __dadd_rn(ml, term_part(P, g, h1, h2, -1.0, -1.0, T.sig_mp));
    ml = __dadd_rn(ml, term_rept(P, max(h1 - P.readlen, 1) + max(h2 - P.readlen, 1), T.lgamma_k1));
    ml = __dadd_rn(ml, term_pe(P, g, h1, h2, T.tmin));
    return ml;
}

// PP predicate of a point (models.py:351-364) on alleles in bp (h >= 0): floor(h / K) >= c  <=>  h >= c K;
// floor(h / K) <= c  <=>  h < (c + 1) K
__device__ __forceinline__ bool pathological_h(const tredsw_grid_problem &P, int hlo, int hhi) {
    if (P.expansion) return (P.recessive ? hlo : hhi) >= P.cutoff_risk * P.period;
    return (P.recessive ? hhi : hlo) < (P.cutoff_risk + 1) * P.period;
}

// A candidate list is a sorted base part [0, nb) followed by an ascending extension (models.py:250-257; with
// --fullsearch the whole list is ascending and nb = n).  An extension entry repeating a base value is the
// second occurrence of that allele (Q9): its points are evaluated and counted again in the marginals and the
// PP sums, but the joint posterior is a dict keyed by (h1, h2) and holds them once.
__device__ __forceinline__ int base_len(const int32_t *hs, int n, int lane) {       // warp-cooperative
    int nb = n;
    for (int i = 1 + lane; i < n; i += 32) if (hs[i] <= hs[i - 1]) { nb = min(nb, i); break; }
    return __reduce_min_sync(0xffffffffu, nb);
}
__device__ __forceinline__ bool is_second_occurrence(const int32_t *hs, int nb, int i) {
    if (i < nb) return false;
    const int v = hs[i];
    if (nb == 0 || v > hs[nb - 1]) return false;
    for (int j = 0; j < nb; ++j) if (hs[j] == v) return true;
    return false;
}

__device__ __forceinline__ void emit_joint(const GridParams &g, int pi, int u1, int u2, double w) {
    if (!g.post) return;
    const unsigned long long at = atomicAdd(g.post_cursor, 1ULL);
    if ((long long)at < g.post_cap) {
        tredsw_posterior e;
        e.problem = pi; e.kind = TREDSW_POST_JOINT; e.a = u1; e.b = u2; e.p = w;
        g.post[at] = e;
    }
}

__device__ __forceinline__ ProblemConsts problem_consts(const tredsw_grid_problem &P, const GridParams &g, int lane) {
    ProblemConsts T;
    T.lgamma_k1 = lgamma((double)P.n_rept + 1.0);
    T.sig_mp = sigma_h(P, P.max_partial);
    int tmin = 0x7fffffff;
    if (P.run_pe) {
        const int32_t *tl = g.ipool + P.off_target;
        for (int i = lane; i < P.n_target; i += 32) { int x = tl[i]; if (x < 0) x += SPAN; if (x >= P.pe_minpe && x < tmin) tmin = x; }
        tmin = __reduce_min_sync(0xffffffffu, tmin);
    }
    T.tmin = tmin;
    return T;
}

// ==========================================================================================================
// K1  classify: one warp per problem.  Small surfaces (<= 512 points, every haploid problem) are cut into work
//     items of 256 points; large ones are registered for the row kernels and get their table space.
// ==========================================================================================================
__global__ void __launch_bounds__(256) grid_classify_kernel(GridParams g) {
    const int lane = threadIdx.x & 31;
    const int pi = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (pi >= g.nproblems) return;
    const tredsw_grid_problem &P = g.prob[pi];
    const int n1 = P.n_h1, n2 = P.n_h2;
    const long long total = n2 > 0 ? (long long)n1 * n2 : 0;
    if (P.ploidy == 1 || total <= SMALL_LIMIT) {
        // the stutter probability of every candidate, once per problem instead of up to four times per point;
        // parked in the marginal slots (P_h1 / P_h2 are written by the reduction, after the points are done)
        {
            const int32_t *a1 = g.ipool + P.off_h1, *a2 = g.ipool + P.off_h2;
            double *ph1 = g.marg + P.off_ph1, *ph2 = g.marg + P.off_ph2;
            for (int i = lane; i < n1; i += 32) ph1[i] = sigma_h(P, a1[i]);
            if (P.ploidy != 1) for (int i = lane; i < n2; i += 32) ph2[i] = sigma_h(P, a2[i]);
        }
        if (lane == 0 && total > 0) {
            const int chunks = (int)((total + ITEM_POINTS - 1) / ITEM_POINTS);
            const int n = min(chunks, ITEM_MAX);
            const unsigned at = atomicAdd(&g.counters[0], (unsigned)n);
            for (int i = 0; i < n; ++i) { g.items[3 * (at + i)] = pi; g.items[3 * (at + i) + 1] = i; g.items[3 * (at + i) + 2] = n; }
        }
        return;
    }
    const int32_t *h1s = g.ipool + P.off_h1, *h2s = g.ipool + P.off_h2;
    int mx1 = -0x7fffffff, mx2 = -0x7fffffff;
    for (int i = lane; i < n1; i += 32) mx1 = max(mx1, h1s[i]);
    for (int i = lane; i < n2; i += 32) mx2 = max(mx2, h2s[i]);
    mx1 = __reduce_max_sync(0xffffffffu, mx1); mx2 = __reduce_max_sync(0xffffffffu, mx2);
    const int nb1 = base_len(h1s, n1, lane), nb2 = base_len(h2s, n2, lane);
    if (lane == 0) {
        BigInfo B;
        memset(&B, 0, sizeof(B));
        B.mx1 = mx1; B.hrep = mx2; B.nb1 = nb1; B.nb2 = nb2;
        B.nd = max(mx1 - P.readlen, 1) + max(mx2 - P.readlen, 1) - 1;
        B.nc = min(NC_MAX, max(1, (n1 + 7) / 8)); B.nce = B.nc;
        // for h1 <= h2: expansion-dominant and contraction-recessive look at the longer allele (column),
        // expansion-recessive and contraction-dominant at the shorter one (row)
        B.patho_mode = (P.expansion != 0) == (P.recessive != 0) ? 1 : 0;
        const int npe = (P.run_pe && P.n_target > 0) ? P.n_target : 0;
        const Tab full = tab_layout(n1, n2, B.nd, npe, B.nc, true), nope = tab_layout(n1, n2, B.nd, 0, B.nc, true),
                  bare = tab_layout(n1, n2, B.nd, 0, B.nc, false);
        // the reduction scratch is mandatory; the tables are taken when the arena has room for them (and the
        // caller allows that tier)
        bool fail = false;
        unsigned long long off = 0;
        if (g.tables == 0) off = atomicAdd(&g.fcursor[0], (unsigned long long)full.end);
        if (g.tables == 0 && (long long)(off + full.end) <= g.ftab_cap) { B.ok = 1; B.npe = npe; }
        else {
            if (g.tables <= 1) off = atomicAdd(&g.fcursor[0], (unsigned long long)nope.end);
            if (g.tables <= 1 && (long long)(off + nope.end) <= g.ftab_cap) { B.ok = 1; B.npe = 0; }
            else {
                off = atomicAdd(&g.fcursor[0], (unsigned long long)bare.end);
                if ((long long)(off + bare.end) > g.ftab_cap) { fail = true; atomicExch(&g.fcursor[1], 1ULL); off = 0; }
            }
        }
        B.off = (long long)off;
        g.big[pi] = B;
        if (!fail) { const int slot = atomicAdd(&g.lists[0], 1); g.lists[1 + slot] = pi; }
        else {
            tredsw_grid_result r;
            memset(&r, 0, sizeof(r));
            r.arg_i1 = r.arg_i2 = -1; r.n_points = -1;
            g.res[pi] = r;
        }
    }
}

// ---- small surfaces, part 1: one warp per item evaluates its points into the scratch slot ---------------------
// (items come from an atomic cursor: their cost varies by two orders of magnitude)
__device__ __forceinline__ void small_points(const GridParams &g) {
    const int lane = threadIdx.x & 31;
    const unsigned nitems = g.counters[0];
    for (;;) {
        unsigned it = 0;
        if (lane == 0) it = atomicAdd(&g.counters[3], 1u);
        it = __shfl_sync(0xffffffffu, it, 0);
        if (it >= nitems) break;
        const int pi = g.items[3 * it], chunk0 = g.items[3 * it + 1], stride = g.items[3 * it + 2];
        const tredsw_grid_problem &P = g.prob[pi];
        const int n2 = P.n_h2;
        const long long total = (long long)P.n_h1 * n2;
        const int32_t *h1s = g.ipool + P.off_h1, *h2s = g.ipool + P.off_h2;
        const double *sg1s = g.marg + P.off_ph1, *sg2s = g.marg + P.off_ph2;
        const bool haploid = P.ploidy == 1;
        const ProblemConsts T = problem_consts(P, g, lane);
        double *surf = g.surface + P.off_surface;
        for (long long c0 = (long long)chunk0 * ITEM_POINTS; c0 < total; c0 += (long long)stride * ITEM_POINTS)
            for (int q = lane; q < ITEM_POINTS; q += 32) {
                const long long t = c0 + q;
                if (t >= total) break;
                const int i1 = (int)(t / n2), i2 = (int)(t - (long long)i1 * n2);
                const int h1 = h1s[i1];
                const int h2 = haploid ? h1 : h2s[i2];
                double ml = -INFINITY;
                if (h1 <= h2) {
                    const double s1 = sg1s[i1], s2 = haploid ? s1 : sg2s[i2];
                    const double sc1 = h1 >= P.max_partial ? T.sig_mp : s1, sc2 = h2 >= P.max_partial ? T.sig_mp : s2;
                    ml = term_span(P, g, h1, h2, s1, s2);
                    ml = __dadd_rn(ml, term_part(P, g, h1, h2, sc1, sc2, T.sig_mp));
                    ml = __dadd_rn(ml, term_rept(P, max(h1 - P.readlen, 1) + max(h2 - P.readlen, 1), T.lgamma_k1));
                    ml = __dadd_rn(ml, term_pe(P, g, h1, h2, T.tmin));
                }
                surf[t] = ml;
            }
    }
}

// ---- small surfaces, part 2: one warp per problem reduces its scratch slot ------------------------------------
__device__ __forceinline__ void small_reduce(const GridParams &g, int first_warp, int nwarps) {
    const int lane = threadIdx.x & 31;
    for (int pi = first_warp; pi < g.nproblems; pi += nwarps) {
        const tredsw_grid_problem &P = g.prob[pi];
        const int n1 = P.n_h1, n2 = P.n_h2;
        const long long total = n2 > 0 ? (long long)n1 * n2 : 0;
        const bool haploid = P.ploidy == 1;
        if (!haploid && total > SMALL_LIMIT) continue;
        const int32_t *h1s = g.ipool + P.off_h1, *h2s = g.ipool + P.off_h2;
        const double *surf = g.surface + P.off_surface;
        double best_ml = -INFINITY;
        int best_h1 = 0x7fffffff, cnt = 0;
        long long best_t = 0x7fffffffffffffffLL;
        for (long long t = lane; t < total; t += 32) {
            const double ml = surf[t];
            if (ml == -INFINITY) continue;
            ++cnt;
            const int h1 = h1s[t / n2];
            if (ml > best_ml || (ml == best_ml && (h1 < best_h1 || (h1 == best_h1 && t < best_t)))) { best_ml = ml; best_h1 = h1; best_t = t; }
        }
        for (int d = 16; d > 0; d >>= 1) {
            const double oml = __shfl_xor_sync(0xffffffffu, best_ml, d);
            const int oh = __shfl_xor_sync(0xffffffffu, best_h1, d);
            const long long ot = __shfl_xor_sync(0xffffffffu, best_t, d);
            if (oml > best_ml || (oml == best_ml && (oh < best_h1 || (oh == best_h1 && ot < best_t)))) { best_ml = oml; best_h1 = oh; best_t = ot; }
            cnt += __shfl_xor_sync(0xffffffffu, cnt, d);
        }
        double *ph1 = g.marg + P.off_ph1, *ph2 = g.marg + P.off_ph2;
        for (int i2 = lane; i2 < n2; i2 += 32) ph2[i2] = 0.0;
        const int nb1 = cnt ? base_len(h1s, n1, lane) : n1;
        const int nb2 = (cnt && !haploid) ? base_len(h2s, n2, lane) : n2;
        double sum_all = 0.0, sum_path = 0.0, sum_uniq = 0.0;
        const double eps = g.small_value;
        if (haploid) {
            // one point per candidate (h2 = h1): lanes over the candidates
            double acc = 0.0, accp = 0.0, accu = 0.0;
            for (int i1 = lane; i1 < n1; i1 += 32) {
                const double ml = surf[i1];
                const int h1 = h1s[i1];
                const double w = exp(ml - best_ml);
                ph1[i1] = w; acc += w;
                if (pathological_h(P, h1, h1)) accp += w;
                if (!is_second_occurrence(h1s, nb1, i1)) {
                    accu += w;
                    if (w >= eps) emit_joint(g, pi, h1 / P.period, h1 / P.period, w);
                }
            }
            for (int d = 16; d > 0; d >>= 1) {
                acc += __shfl_xor_sync(0xffffffffu, acc, d);
                accp += __shfl_xor_sync(0xffffffffu, accp, d);
                accu += __shfl_xor_sync(0xffffffffu, accu, d);
            }
            sum_all = acc; sum_path = accp; sum_uniq = accu;
            if (lane == 0 && n2 > 0) ph2[0] = acc;
        } else
        for (int i1 = 0; i1 < n1; ++i1) {
            const int h1 = h1s[i1];
            const bool dup1 = is_second_occurrence(h1s, nb1, i1);
            double acc = 0.0, accp = 0.0, accu = 0.0;
            for (int i2 = lane; i2 < n2; i2 += 32) {           // column i2 always belongs to lane i2 % 32: the plain
                const double ml = surf[(long long)i1 * n2 + i2];   // read-modify-write of ph2 is race-free and ordered
                if (ml == -INFINITY) continue;
                const double w = exp(ml - best_ml);
                const int h2 = haploid ? h1 : h2s[i2];
                acc += w; ph2[i2] += w;
                if (pathological_h(P, h1, h2)) accp += w;            // (evaluated points have h1 <= h2)
                if (!(dup1 || (!haploid && is_second_occurrence(h2s, nb2, i2)))) {
                    accu += w;
                    if (w >= eps) emit_joint(g, pi, h1 / P.period, h2 / P.period, w);
                }
            }
            for (int d = 16; d > 0; d >>= 1) {
                acc += __shfl_down_sync(0xffffffffu, acc, d);
                accp += __shfl_down_sync(0xffffffffu, accp, d);
                accu += __shfl_down_sync(0xffffffffu, accu, d);
            }
            if (lane == 0) { ph1[i1] = acc; sum_all += acc; sum_path += accp; sum_uniq += accu; }
        }
        if (lane == 0) {
            tredsw_grid_result r;
            r.max_ml = best_ml; r.sum_all = sum_all; r.sum_path = sum_path; r.sum_uniq = sum_uniq;
            r.arg_i1 = cnt ? (int)(best_t / n2) : -1;
            r.arg_i2 = cnt ? (int)(best_t % n2) : -1;
            r.n_points = cnt; r.pad = 0;
            g.res[pi] = r;
        }
    }
}

// ==========================================================================================================
// large surfaces
// ==========================================================================================================
// block-wide max of an int (256 threads); every thread gets the result
__device__ __forceinline__ int block_max_int(int v, int *s8) {
    v = __reduce_max_sync(0xffffffffu, v);
    __syncthreads();                                   // s8 may still be read from the previous call
    if ((threadIdx.x & 31) == 0) s8[threadIdx.x >> 5] = v;
    __syncthreads();
    int r = s8[0];
#pragma unroll
    for (int w = 1; w < 8; ++w) r = max(r, s8[w]);
    return r;
}

// FILL_SPLIT blocks per large surface: each derives the thresholds (cheap, block-parallel scans — no block waits
// for another), part 0 publishes them, all fill their share of the tables.
__device__ __forceinline__ void big_setup(const GridParams &g, int first_block, int nblocks) {
    __shared__ int s8[8];
    const int nbig = g.lists[0];
    const int tid = threadIdx.x;
    for (int kk = first_block; kk < nbig * FILL_SPLIT; kk += nblocks) {
        const int pi = g.lists[1 + kk / FILL_SPLIT], part = kk % FILL_SPLIT;
        const tredsw_grid_problem &P = g.prob[pi];
        BigInfo &B = g.big[pi];
        const int n1 = P.n_h1, n2 = P.n_h2;
        const int32_t *h1s = g.ipool + P.off_h1, *h2s = g.ipool + P.off_h2;
        const int32_t *skey = g.ipool + P.off_span, *tl = g.ipool + P.off_target;
        int ks = -1000000, ntmin = -0x7fffffff, unsorted = 0;
        for (int i = tid; i < P.n_span; i += 256) ks = max(ks, skey[i]);
        if (P.run_pe)
            for (int i = tid; i < P.n_target; i += 256) { int x = tl[i]; if (x < 0) x += SPAN; if (x >= P.pe_minpe) ntmin = max(ntmin, -x); }
        for (int i = tid + 1; i < n1; i += 256) if (h1s[i - 1] > h1s[i]) unsorted = 1;
        for (int i = tid + 1; i < n2; i += 256) if (h2s[i - 1] > h2s[i]) unsorted = 1;
        ks = block_max_int(ks, s8); ntmin = block_max_int(ntmin, s8); unsorted = block_max_int(unsorted, s8);
        const int tmin = ntmin == -0x7fffffff ? 0x7fffffff : -ntmin;
        const int t1 = P.readlen - 9;
        // h2 >= H1: no spanning key within 18, partial clamp and mixing weights saturated, h2 > readlen
        const int H1 = max(max(ks + DEV + 1, P.max_partial), max(t1, P.readlen + 1));
        // h2 >= H2: every pair length >= MINPE is shifted past the support as well
        long long H2 = H1;
        if (P.run_pe && tmin != 0x7fffffff) H2 = max((long long)H1, (long long)P.pe_ref + SPAN - tmin);
        int l1 = -1, l2 = -1;                          // last column below H1 / H2
        for (int i = tid; i < n2; i += 256) { const int h = h2s[i]; if (h < H1) l1 = max(l1, i); if (h < H2) l2 = max(l2, i); }
        l1 = block_max_int(l1, s8); l2 = block_max_int(l2, s8);
        const int fam = B.ok ? l1 + 1 : n2, fa2 = B.ok ? l2 + 1 : n2;
        const double lgk = lgamma((double)P.n_rept + 1.0), sig_mp = sigma_h(P, P.max_partial);
        int notarith = 0, anydup = 0;
        const int fstep = fa2 + 1 < n2 ? h2s[fa2 + 1] - h2s[fa2] : 0, fd0 = fa2 < n2 ? h2s[fa2] - P.readlen : 1;
        for (int i = fa2 + tid; i < n2; i += 256) if (h2s[i] != h2s[fa2] + (i - fa2) * fstep) notarith = 1;
        if (fd0 < 1) notarith = 1;
        for (int i = tid; i < n1 + n2; i += 256)
            if (i < n1 ? is_second_occurrence(h1s, B.nb1, i) : is_second_occurrence(h2s, B.nb2, i - n1)) anydup = 1;
        int notall = 0;
        const int astep = n2 > 1 ? h2s[1] - h2s[0] : 1;
        for (int i = tid; i < n2; i += 256) if (h2s[i] != h2s[0] + i * astep) notall = 1;
        if (astep <= 0) notall = 1;
        notarith = block_max_int(notarith, s8); anydup = block_max_int(anydup, s8); notall = block_max_int(notall, s8);
        if (part == 0 && tid == 0) {
            B.far_arith = notarith ? 0 : 1; B.far_d0 = fd0; B.far_step = fstep; B.has_dup = anydup;
            B.h2_arith = notall ? 0 : 1; B.h2_a0 = h2s[0]; B.h2_step = astep;
            B.lgamma_k1 = lgk; B.sig_mp = sig_mp; B.tmin = tmin; B.fam = fam; B.fa2 = fa2; B.sorted = unsorted ? 0 : 1;
            // few large surfaces: many CTAs each (latency); many: few CTAs each, so that a warp keeps its column
            // registers over many rows (throughput)
            B.nce = max(1, min(B.nc, (g.target_ctas + nbig - 1) / nbig));
            const unsigned at = atomicAdd(&g.counters[4], (unsigned)B.nce);
            for (int r = 0; r < B.nce; ++r) { g.row_items[2 * (at + r)] = pi; g.row_items[2 * (at + r) + 1] = r; }
        }
        const Tab tb = tab_layout(n1, n2, B.nd, B.npe, B.nc, B.ok != 0);
        double *tab = g.ftab + B.off;
        int32_t *dup = reinterpret_cast<int32_t *>(tab + tb.dup);
        for (int e = part * 256 + tid; e < n1 + n2; e += 256 * FILL_SPLIT)
            dup[e] = e < n1 ? (int)is_second_occurrence(h1s, B.nb1, e) : (int)is_second_occurrence(h2s, B.nb2, e - n1);
        if (!B.ok) continue;
        const int hrep = B.hrep, npe = B.npe, nd = B.nd;
        const double *pdf = g.dpool + P.off_pdf;
        const long long o_s2 = n1, o_rows = o_s2 + n2, o_rept = o_rows + n1, o_R1 = o_rept + nd,
                        o_R2 = o_R1 + (long long)npe * n1, n_all = o_R2 + (long long)npe * fa2;
        for (long long e = part * 256 + tid; e < n_all; e += 256 * FILL_SPLIT) {
            if (e < o_s2) tab[tb.sig1 + e] = sigma_h(P, h1s[e]);
            else if (e < o_rows) tab[tb.sig2 + (e - o_s2)] = sigma_h(P, h2s[e - o_s2]);
            else if (e < o_rept) {
                const int i1 = (int)(e - o_rows), h1 = h1s[i1];
                const int hc1 = min(h1, P.max_partial);
                const double s1 = sigma_h(P, h1), sc1 = hc1 == P.max_partial ? sig_mp : s1;
                // (for a far column the second allele's sigma is never used: every key is farther than 18 from it;
                //  sig_mp is the clamped one)
                tab[tb.rows + 3LL * i1] = __dadd_rn(term_span(P, g, h1, hrep, s1, 0.5), term_part(P, g, h1, hrep, sc1, sig_mp, sig_mp));
                tab[tb.rows + 3LL * i1 + 1] = term_pe(P, g, h1, hrep, tmin);
                tab[tb.rows + 3LL * i1 + 2] = 0.0;
            } else if (e < o_R1) {
                const int d = (int)(e - o_rept);
                const double r = term_rept(P, d + 2, lgk);
                tab[tb.rept + d] = r;
                tab[tb.erept + d] = exp(r);
            } else {
                // halved operands of the two-dimensional paired-end term (0.5 * what pe_roll returns: exact)
                long long idx = e - o_R1;
                const bool first = e < o_R2;
                if (!first) idx = e - o_R2;
                const int width = first ? n1 : fa2;
                const int t = (int)(idx / width), i = (int)(idx - (long long)t * width);
                int x = tl[t];
                if (x < 0) x += SPAN;
                tab[(first ? tb.R1 : tb.R2) + idx] = __dmul_rn(0.5, pe_roll(pdf, first ? h1s[i] : h2s[i], P.pe_ref, P.pe_minpe, x, g.small_value));
            }
        }
    }
}

// K2 = { point items of the small surfaces | table setup of the large ones }
__global__ void __launch_bounds__(256, 3) grid_points_setup_kernel(GridParams g) {
    if ((int)blockIdx.x < g.nblk_small) small_points(g);
    else big_setup(g, blockIdx.x - g.nblk_small, gridDim.x - g.nblk_small);
}

struct RowTables {
    const double *rows, *sig1, *sig2, *rept, *erept, *R1, *R2;
    const int32_t *dup;
    double *colpart, *partial, *pa;
};
__device__ __forceinline__ RowTables row_tables(const GridParams &g, const BigInfo &B, int n1, int n2) {
    const Tab tb = tab_layout(n1, n2, B.nd, B.npe, B.nc, B.ok != 0);
    double *tab = g.ftab + B.off;
    RowTables r;
    r.rows = tab + tb.rows; r.sig1 = tab + tb.sig1; r.sig2 = tab + tb.sig2; r.rept = tab + tb.rept; r.erept = tab + tb.erept;
    r.R1 = tab + tb.R1; r.R2 = tab + tb.R2; r.dup = reinterpret_cast<const int32_t *>(tab + tb.dup);
    r.colpart = tab + tb.colpart; r.partial = tab + tb.partial; r.pa = tab + tb.pa;
    return r;
}

struct Best {                       // running arg-max with the reference's tie rule (ml, -h1, evaluation order): Q10
    double ml;
    unsigned long long key;         // h1 << 40 | row-major index
    __device__ __forceinline__ void take(double m, int h1, long long idx) {
        if (m >= ml) {
            const unsigned long long k = ((unsigned long long)h1 << 40) | (unsigned long long)idx;
            if (m > ml || k < key) { ml = m; key = k; }
        }
    }
    __device__ __forceinline__ void merge(double m, unsigned long long k) {
        if (m > ml || (m == ml && k < key)) { ml = m; key = k; }
    }
};

// Pass A: near / mid points into the scratch slot; maximum, arg-max and point count of this CTA's rows.
// Work item = (surface, CTA rank c < nce): the row groups g = c, c + nce, ... of 8 rows (one per warp); items are
// taken from an atomic cursor, rank-major, so the ranks holding the expensive near rows start first.
// A warp walks one row at a time, left to right: column groups of 32 with near / mid columns go through
// mixed_batch<NJ> (NJ = 4, 2, 1 groups at a time: the paired-end products of NJ columns per lane run as NJ
// independent chains over the pair lengths, fed by one uniform and NJ coalesced loads per length), the far
// columns through a loop of two additions per point.
struct RowCtx {
    const tredsw_grid_problem *P;
    const GridParams *g;
    const int32_t *h2s;
    double *surf;                 // row base
    const double *rept_row;       // rept + max(h1 - L, 1) - 2
    const double *R1row, *R2, *sig2;
    double c12, pe_far, sg1, sgc1, eps;
    int h1, i1, n1, n2, L, fam, fa2, npe, ok, c0, tmin;
    long long rowbase;
    bool mat, strict;
};

template <int NJ>
__device__ __forceinline__ void mixed_batch(const RowCtx &x, const ProblemConsts &T, int gb, int lane, Best &best, int &cnt) {
    const tredsw_grid_problem &P = *x.P;
    double pe[NJ];
    int col[NJ];
#pragma unroll
    for (int q = 0; q < NJ; ++q) { col[q] = 32 * (gb + q) + lane; pe[q] = 0.0; }
    if (x.ok && x.npe > 0) {
        int cj[NJ];
#pragma unroll
        for (int q = 0; q < NJ; ++q) cj[q] = min(col[q], x.fa2 - 1);
        for (int t0 = 0; t0 < x.npe; t0 += PE_BLOCK) {
            double prod[NJ];
#pragma unroll
            for (int q = 0; q < NJ; ++q) prod[q] = 1.0;
            const int t1 = min(t0 + PE_BLOCK, x.npe);
#pragma unroll 2
            for (int t = t0; t < t1; ++t) {
                const double r1 = x.R1row[(long long)t * x.n1];
                const double *r2p = x.R2 + (long long)t * x.fa2;
#pragma unroll
                for (int q = 0; q < NJ; ++q) prod[q] = __dmul_rn(prod[q], fmax(__dadd_rn(r1, r2p[cj[q]]), x.eps));
            }
#pragma unroll
            for (int q = 0; q < NJ; ++q) pe[q] = __dadd_rn(pe[q], log(prod[q]));
        }
    }
#pragma unroll
    for (int q = 0; q < NJ; ++q) {
        const int c = col[q];
        if (c >= x.n2) continue;
        const int h2 = x.h2s[c];
        double ml = -INFINITY;
        if (x.h1 <= h2) {
            if (x.ok) {
                const double rp = x.rept_row[max(h2 - x.L, 1)];
                if (c >= x.fa2) ml = __dadd_rn(__dadd_rn(x.c12, rp), x.pe_far);
                else {
                    const double pej = x.npe > 0 ? pe[q] : term_pe(P, *x.g, x.h1, h2, x.tmin);
                    if (c >= x.fam) ml = __dadd_rn(__dadd_rn(x.c12, rp), pej);
                    else {
                        const double sg2 = x.sig2[c];
                        const double sgc2 = min(h2, P.max_partial) == P.max_partial ? T.sig_mp : sg2;
                        ml = __dadd_rn(term_span(P, *x.g, x.h1, h2, x.sg1, sg2), term_part(P, *x.g, x.h1, h2, x.sgc1, sgc2, T.sig_mp));
                        ml = __dadd_rn(__dadd_rn(ml, rp), pej);
                    }
                }
            } else {
                ml = point_ml(P, *x.g, x.h1, h2, T);
            }
            if (x.strict) { if (ml > best.ml) { best.ml = ml; best.key = ((unsigned long long)x.h1 << 40) | (unsigned long long)(x.rowbase + c); } }
            else best.take(ml, x.h1, x.rowbase + c);
            ++cnt;
            if (!(x.ok && c >= x.fa2) || x.mat) x.surf[c] = ml;
        } else if (x.mat) x.surf[c] = ml;
    }
}

__device__ __forceinline__ void rows_eval(const GridParams &g) {
    __shared__ double s_ml[8];
    __shared__ unsigned long long s_key[8];
    __shared__ int s_cnt[8];
    __shared__ unsigned s_item;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    for (;;) {
        __syncthreads();
        if (tid == 0) s_item = atomicAdd(&g.counters[1], 1u);
        __syncthreads();
        const unsigned item = s_item;
        if (item >= g.counters[4]) break;
        const int pi = g.row_items[2 * item], c = g.row_items[2 * item + 1];
        const BigInfo &B = g.big[pi];
        const int nc = B.nce;
        if (c >= nc) continue;
        const tredsw_grid_problem &P = g.prob[pi];
        const int n1 = P.n_h1, n2 = P.n_h2, L = P.readlen;
        const int32_t *h1s = g.ipool + P.off_h1, *h2s = g.ipool + P.off_h2;
        double *surf = g.surface + P.off_surface, *ph1 = g.marg + P.off_ph1;
        const RowTables R = row_tables(g, B, n1, n2);
        ProblemConsts T;
        T.lgamma_k1 = B.lgamma_k1; T.sig_mp = B.sig_mp; T.tmin = B.tmin;
        RowCtx x;
        x.P = &P; x.g = &g; x.h2s = h2s; x.R2 = R.R2; x.sig2 = R.sig2; x.eps = g.small_value;
        x.n1 = n1; x.n2 = n2; x.L = L; x.fam = B.fam; x.fa2 = B.fa2; x.npe = B.npe; x.ok = B.ok; x.tmin = B.tmin;
        x.mat = g.materialise != 0; x.strict = B.sorted != 0;
        const bool sorted = B.sorted != 0, arith = B.far_arith != 0 && B.ok;
        const int ngroups = (n2 + 31) >> 5;
        const int g_mid_end = B.ok ? (min(B.fa2, n2) + 31) >> 5 : ngroups;     // groups [.., g_mid_end) hold near / mid columns
        Best best{-INFINITY, ~0ULL};
        int cnt = 0;
        for (int grp = c; grp * 8 < n1; grp += nc) {
            const int i1 = grp * 8 + warp;
            if (i1 >= n1) continue;
            if (lane == 0) ph1[i1] = 0.0;
            const int h1 = h1s[i1];
            x.h1 = h1; x.i1 = i1; x.rowbase = (long long)i1 * n2; x.surf = surf + x.rowbase;
            x.c12 = 0.0; x.pe_far = 0.0; x.sg1 = -1.0; x.sgc1 = -1.0;
            x.rept_row = R.rept + (max(h1 - L, 1) - 2);
            x.R1row = R.R1 + i1;
            if (B.ok) {
                x.c12 = R.rows[3LL * i1]; x.pe_far = R.rows[3LL * i1 + 1]; x.sg1 = R.sig1[i1];
                x.sgc1 = min(h1, P.max_partial) == P.max_partial ? T.sig_mp : x.sg1;
            }
            // first column the row evaluates (sorted lists: lower bound of h1)
            int c0 = 0;
            if (B.h2_arith) c0 = min(n2, max(0, (h1 - B.h2_a0 + B.h2_step - 1) / B.h2_step));
            else if (sorted) {
                int lo = 0, hi = n2;
                while (lo < hi) { const int mid = (lo + hi) >> 1; if (h2s[mid] < h1) lo = mid + 1; else hi = mid; }
                c0 = lo;
            }
            x.c0 = c0;
            if (x.mat) for (int col = lane; col < c0; col += 32) x.surf[col] = -INFINITY;
            int gb = c0 >> 5;
            while (gb < g_mid_end) {
                const int left = g_mid_end - gb;
                if (left >= 4) { mixed_batch<4>(x, T, gb, lane, best, cnt); gb += 4; }
                else if (left >= 2) { mixed_batch<2>(x, T, gb, lane, best, cnt); gb += 2; }
                else { mixed_batch<1>(x, T, gb, lane, best, cnt); gb += 1; }
            }
            // far columns: two additions per point
            const double c12 = x.c12, pe_far = x.pe_far;
            const double *rr = x.rept_row;
            const unsigned long long keybase = ((unsigned long long)h1 << 40) | (unsigned long long)x.rowbase;
            const bool mat = x.mat, strict = x.strict;
            if (arith && strict && !mat) {
                // sorted lists, arithmetic far columns: every column from max(32 gb, c0) on is evaluated, its table
                // index is linear in the column — one load, two additions and a compare per point
                const int cf = max(32 * gb, c0);
                const int step32 = 32 * B.far_step;
                const double *pp = rr + (B.far_d0 + B.far_step * (cf + lane - B.fa2));
                double bm = best.ml;
                int bc = -1;
                int col = cf + lane;
                for (; col + 96 < n2; col += 128, pp += 4 * step32) {
                    const double v0 = pp[0], v1 = pp[step32], v2 = pp[2 * step32], v3 = pp[3 * step32];
                    const double m0 = __dadd_rn(__dadd_rn(c12, v0), pe_far), m1 = __dadd_rn(__dadd_rn(c12, v1), pe_far);
                    const double m2 = __dadd_rn(__dadd_rn(c12, v2), pe_far), m3 = __dadd_rn(__dadd_rn(c12, v3), pe_far);
                    if (m0 > bm) { bm = m0; bc = col; }
                    if (m1 > bm) { bm = m1; bc = col + 32; }
                    if (m2 > bm) { bm = m2; bc = col + 64; }
                    if (m3 > bm) { bm = m3; bc = col + 96; }
                }
                for (; col < n2; col += 32, pp += step32) {
                    const double m0 = __dadd_rn(__dadd_rn(c12, pp[0]), pe_far);
                    if (m0 > bm) { bm = m0; bc = col; }
                }
                if (bc >= 0) { best.ml = bm; best.key = keybase + (unsigned)bc; }
                if (cf + lane < n2) cnt += (n2 - 1 - cf - lane) / 32 + 1;
            } else
            for (; gb < ngroups; gb += 4) {
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int col = 32 * (gb + q) + lane;
                    if (col >= n2) continue;
                    int d2;
                    bool valid;
                    if (arith) { d2 = B.far_d0 + B.far_step * (col - B.fa2); valid = h1 <= L + d2; }      // (h2 = L + d2 there)
                    else { const int h2 = h2s[col]; d2 = max(h2 - L, 1); valid = h1 <= h2; }
                    double ml = -INFINITY;
                    if (valid) {
                        ml = __dadd_rn(__dadd_rn(c12, rr[d2]), pe_far);
                        if (strict) { if (ml > best.ml) { best.ml = ml; best.key = keybase + (unsigned)col; } }
                        else best.take(ml, h1, x.rowbase + col);
                        ++cnt;
                    }
                    if (mat) x.surf[col] = ml;
                }
            }
        }
        for (int d = 16; d > 0; d >>= 1) {
            best.merge(__shfl_xor_sync(0xffffffffu, best.ml, d), __shfl_xor_sync(0xffffffffu, best.key, d));
            cnt += __shfl_xor_sync(0xffffffffu, cnt, d);
        }
        if (lane == 0) { s_ml[warp] = best.ml; s_key[warp] = best.key; s_cnt[warp] = cnt; }
        __syncthreads();
        if (tid == 0) {
            Best b{s_ml[0], s_key[0]};
            int n = s_cnt[0];
#pragma unroll
            for (int w = 1; w < 8; ++w) { b.merge(s_ml[w], s_key[w]); n += s_cnt[w]; }
            R.pa[4LL * c] = b.ml;
            R.pa[4LL * c + 1] = __longlong_as_double((long long)b.key);
            R.pa[4LL * c + 2] = (double)n;
        }
    }
}

// K3 = { reductions of the small surfaces | pass A of the large ones }
__global__ void __launch_bounds__(256, 2) grid_reduce_eval_kernel(GridParams g) {
    const int nrows_blocks = (int)gridDim.x - g.nblk_small;       // the row blocks come first: they are the long pole
    if ((int)blockIdx.x >= nrows_blocks) small_reduce(g, (blockIdx.x - nrows_blocks) * 8 + (threadIdx.x >> 5), g.nblk_small * 8);
    else rows_eval(g);
}

// K4  pass B: weights exp(ml - max) of every point -> row sums (P_h1), column sums (P_h2), PP sums, joint entries.
// A far point costs a multiply (per-row factor x tabulated exp of the repeat-only term) and two additions.
// Column sums: registers (8 columns per lane over the warp's rows) -> shared memory (8 warps, in warp order) ->
// this CTA's slice of colpart; the last CTA of a surface to finish adds the slices in rank order.
__global__ void __launch_bounds__(256, 3) grid_rows_reduce_kernel(GridParams g) {
    __shared__ double s_col[8][CHUNK];
    __shared__ double s_sum[8][3];
    __shared__ int s_last;
    __shared__ unsigned s_item;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    for (;;) {
        __syncthreads();
        if (tid == 0) s_item = atomicAdd(&g.counters[2], 1u);
        __syncthreads();
        const unsigned item = s_item;
        if (item >= g.counters[4]) break;
        const int pi = g.row_items[2 * item], c = g.row_items[2 * item + 1];
        BigInfo &B = g.big[pi];
        const int nc = B.nce;
        if (c >= nc) continue;
        const tredsw_grid_problem &P = g.prob[pi];
        const int n1 = P.n_h1, n2 = P.n_h2, L = P.readlen, K = P.period;
        const int32_t *h1s = g.ipool + P.off_h1, *h2s = g.ipool + P.off_h2;
        const double *surf = g.surface + P.off_surface;
        double *ph1 = g.marg + P.off_ph1, *ph2 = g.marg + P.off_ph2;
        const RowTables R = row_tables(g, B, n1, n2);
        double *rows_w = const_cast<double *>(R.rows);
        const int ok = B.ok, fa2 = B.fa2, sorted = B.sorted, prow_mode = B.patho_mode, has_dup = B.has_dup;
        const double eps = g.small_value;
        // the surface maximum: pass A's per-CTA results in rank order
        Best top{-INFINITY, ~0ULL};
        long long npoints = 0;
        for (int r = 0; r < nc; ++r) {
            top.merge(R.pa[4LL * r], (unsigned long long)__double_as_longlong(R.pa[4LL * r + 1]));
            npoints += (long long)R.pa[4LL * r + 2];
        }
        const double M = npoints ? top.ml : INFINITY;
        // per-row factor of the far weights
        if (ok)
            for (int g0 = c; g0 * 8 < n1; g0 += 32 * nc) {            // lane r: the r-th row of this warp
                const int i1 = (g0 + lane * nc) * 8 + warp;
                if (i1 < n1) rows_w[3LL * i1 + 2] = exp(__dadd_rn(R.rows[3LL * i1], R.rows[3LL * i1 + 1]) - M);
            }
        __syncwarp();
        // PP predicate as thresholds on the allele in bp (pathological_h)
        const int pp_thr = P.expansion ? P.cutoff_risk * K : (P.cutoff_risk + 1) * K;
        const bool pp_ge = P.expansion != 0;
        double sum_all = 0.0, sum_path = 0.0, sum_dup = 0.0;          // lane 0 of every warp
        for (int cb = 0; cb < n2; cb += CHUNK) {
            const int cend = min(cb + CHUNK, n2);
            const int jmax = (cend - cb + 31) >> 5;
            const int h2_last = sorted ? h2s[cend - 1] : 0x7fffffff;
            const bool all_far = ok && cb >= fa2;
            int h2v[8], dh2[8], dup2 = 0, pcol = 0;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int col = cb + lane + 32 * j;
                h2v[j] = col < cend ? h2s[col] : -0x40000000;
                dh2[j] = max(h2v[j] - L, 1);
                if (col < cend) {
                    if (has_dup && R.dup[n1 + col]) dup2 |= 1 << j;
                    // column mode: the PP predicate looks at the longer allele only
                    if (!prow_mode && (pp_ge ? h2v[j] >= pp_thr : h2v[j] < pp_thr)) pcol |= 1 << j;
                }
            }
            const int h2_first = h2s[cb];
            const bool full_chunk = cend - cb == CHUNK;
            double colacc[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) colacc[j] = 0.0;
            for (int grp = c; grp * 8 < n1; grp += nc) {
                const int i1 = grp * 8 + warp;
                if (i1 >= n1) continue;
                const int h1 = h1s[i1];
                if (h2_last < h1) continue;
                const int dh1 = max(h1 - L, 1) - 2;
                const bool dup1 = has_dup && R.dup[i1] != 0;
                const bool prow = prow_mode && (pp_ge ? h1 >= pp_thr : h1 < pp_thr);
                const long long row = (long long)i1 * n2;
                const double f = ok ? R.rows[3LL * i1 + 2] : 0.0;
                // a far weight is f * exp(rept) <= f: below e^-10 none of them enters the joint posterior
                const bool may_emit = g.post != nullptr && !dup1 && f >= eps;
                double racc = 0.0, raccp = 0.0, raccd = 0.0;
                if (all_far && full_chunk && sorted && h1 <= h2_first && !dup1 && dup2 == 0 && !may_emit) {
                    // the common case of a long-expansion grid: 8 valid far columns, nothing to test
                    const double *er = R.erept + dh1;
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const double w = f * er[dh2[j]];
                        colacc[j] += w; racc += w;
                        if ((pcol >> j) & 1) raccp += w;
                    }
                } else if (all_far && !dup1 && dup2 == 0 && !may_emit) {
                    const double *er = R.erept + dh1;
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        if (h1 > h2v[j]) continue;                        // not evaluated, or past the chunk
                        const double w = f * er[dh2[j]];
                        colacc[j] += w; racc += w;
                        if ((pcol >> j) & 1) raccp += w;
                    }
                } else if (all_far) {
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        if (j >= jmax) break;
                        if (h1 > h2v[j]) continue;
                        const double w = f * R.erept[dh1 + dh2[j]];
                        colacc[j] += w; racc += w;
                        if ((pcol >> j) & 1) raccp += w;
                        if (dup1 || ((dup2 >> j) & 1)) raccd += w;
                        else if (may_emit && w >= eps) emit_joint(g, pi, h1 / K, h2v[j] / K, w);
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        if (j >= jmax) break;
                        if (h1 > h2v[j]) continue;
                        const int col = cb + lane + 32 * j;
                        double w;
                        if (ok && col >= fa2) w = f * R.erept[dh1 + dh2[j]];
                        else {
                            const double d = surf[row + col] - M;
                            w = d < -746.0 ? 0.0 : exp(d);
                        }
                        colacc[j] += w; racc += w;
                        if ((pcol >> j) & 1) raccp += w;
                        if (dup1 || ((dup2 >> j) & 1)) raccd += w;
                        else if (w >= eps) emit_joint(g, pi, h1 / K, h2v[j] / K, w);
                    }
                }
                if (__any_sync(0xffffffffu, racc != 0.0)) {
                    for (int d = 16; d > 0; d >>= 1) {
                        racc += __shfl_down_sync(0xffffffffu, racc, d);
                        raccp += __shfl_down_sync(0xffffffffu, raccp, d);
                        raccd += __shfl_down_sync(0xffffffffu, raccd, d);
                    }
                    if (lane == 0) { ph1[i1] += racc; sum_all += racc; sum_path += prow ? racc : raccp; sum_dup += raccd; }
                }
            }
#pragma unroll
            for (int j = 0; j < 8; ++j) s_col[warp][lane + 32 * j] = colacc[j];
            __syncthreads();
            double cs = 0.0;
#pragma unroll
            for (int w = 0; w < 8; ++w) cs += s_col[w][tid];
            if (cb + tid < n2) R.colpart[(long long)c * n2 + cb + tid] = cs;
            __syncthreads();
        }
        if (lane == 0) { s_sum[warp][0] = sum_all; s_sum[warp][1] = sum_path; s_sum[warp][2] = sum_dup; }
        __syncthreads();
        if (tid == 0) {
            double a = 0.0, p = 0.0, u = 0.0;
            for (int w = 0; w < 8; ++w) { a += s_sum[w][0]; p += s_sum[w][1]; u += s_sum[w][2]; }
            R.partial[4LL * c] = a; R.partial[4LL * c + 1] = p; R.partial[4LL * c + 2] = u;
            __threadfence();
            s_last = (atomicAdd(&B.done_b, 1u) == (unsigned)(nc - 1));
        }
        __syncthreads();
        if (s_last) {
            __threadfence();
            for (int x = tid; x < n2; x += 256) {
                double acc = 0.0;
                for (int r = 0; r < nc; ++r) acc += __ldcg(R.colpart + (long long)r * n2 + x);
                ph2[x] = acc;
            }
            if (tid == 0) {
                double a = 0.0, p = 0.0, u = 0.0;
                for (int r = 0; r < nc; ++r) { a += __ldcg(R.partial + 4LL * r); p += __ldcg(R.partial + 4LL * r + 1); u += __ldcg(R.partial + 4LL * r + 2); }
                tredsw_grid_result r;
                r.max_ml = npoints ? top.ml : -INFINITY; r.sum_all = a; r.sum_path = p; r.sum_uniq = a - u;
                const long long idx = (long long)(top.key & ((1ULL << 40) - 1));
                r.arg_i1 = npoints ? (int)(idx / n2) : -1;
                r.arg_i2 = npoints ? (int)(idx % n2) : -1;
                r.n_points = (int)npoints; r.pad = 0;
                g.res[pi] = r;
            }
        }
    }
}

// ---- KDE of paired-end lengths (models.py:428-435): see kde.cuh ---------------------------------------
__global__ void __launch_bounds__(KDE_THREADS) pe_kde_kernel(const int32_t *lens, const int64_t *off, int nproblems,
                                                      double *pdf_out) {
    for (int pi = blockIdx.x; pi < nproblems; pi += gridDim.x)
        kde_block(lens + off[pi], (int)(off[pi + 1] - off[pi]), pdf_out + (int64_t)pi * SPAN);
}

}  // namespace

// TREDSW_GRID_TABLES=nope | none: large surfaces evaluate the paired-end term point by point, or every term (the
// tiers a full arena falls back to; same results).  Read on every call.
int tredsw_internal_grid_tables(int *tables) {
    *tables = 0;
    if (const char *tier = getenv("TREDSW_GRID_TABLES")) {
        if (strcmp(tier, "nope") == 0) *tables = 1;
        else if (strcmp(tier, "none") == 0) *tables = 2;
        else { tredsw_set_error("TREDSW_GRID_TABLES must be nope or none, not '%s'", tier); return TREDSW_ERR_ARG; }
    }
    return TREDSW_OK;
}

// device-side bookkeeping area of one grid call, at the start of ctx->d_ftab
struct GridArea {
    size_t big_bytes, ctr_off, list_off, item_off, row_off, tab_off;
};
static GridArea grid_area(int nproblems) {
    GridArea a;
    a.big_bytes = (((size_t)nproblems * sizeof(BigInfo)) + 255) & ~(size_t)255;
    a.ctr_off = a.big_bytes;                                                         // fcursor[2] | counters[8] | lists[0]
    a.list_off = a.ctr_off + 48;
    a.item_off = (a.list_off + ((size_t)nproblems + 1) * sizeof(int) + 255) & ~(size_t)255;
    a.row_off = (a.item_off + (size_t)nproblems * ITEM_MAX * 3 * sizeof(int) + 255) & ~(size_t)255;
    a.tab_off = (a.row_off + (size_t)nproblems * NC_MAX * 2 * sizeof(int) + 255) & ~(size_t)255;
    return a;
}

int tredsw_internal_grid(tredsw_ctx *ctx, const tredsw_grid_problem *d_prob, int nproblems,
                         const int32_t *d_ipool, const double *d_dpool, double *d_surface, double *d_marg,
                         tredsw_grid_result *d_res, long long points_hint, int materialise,
                         tredsw_posterior *d_post, long long post_cap, unsigned long long *d_post_cursor,
                         unsigned long long **d_overflow_flag, int tables) {
    GridParams g{};
    g.prob = d_prob; g.ipool = d_ipool; g.dpool = d_dpool; g.surface = d_surface; g.marg = d_marg; g.res = d_res;
    g.small_value = exp(-10.0);
    g.log_small = log(g.small_value);
    g.nproblems = nproblems; g.materialise = materialise; g.tables = tables;
    g.post = d_post; g.post_cap = post_cap; g.post_cursor = d_post_cursor;
    int rc;
    ctx->mark(2);
    const GridArea ar = grid_area(nproblems);
    // table arena, in doubles: 128 MB serve ~250 long-expansion surfaces; a cohort searched with --fullsearch has
    // one large surface per problem, ~(100 + n_target) doubles of tables and reduction scratch per candidate
    // allele each.  A surface that finds the arena short of its tables is evaluated point by point (slower, same
    // result); one that cannot even get its reduction scratch is reported through the overflow flag and the
    // call is repeated with a larger arena.
    long long cap = 16LL << 20;
    if (points_hint > SMALL_LIMIT) {
        const long long side = (long long)ceil(sqrt((double)points_hint));
        const long long want = (long long)nproblems * 160 * side;
        if (want > cap) cap = want < (1LL << 30) ? want : (1LL << 30);
    }
    const long long have = ((long long)ctx->d_ftab.cap - (long long)ar.tab_off) / (long long)sizeof(double);
    if (have > cap) cap = have;
    if (ctx->d_ftab.ensure(ar.tab_off + (size_t)cap * sizeof(double)) != TREDSW_OK) {
        cudaGetLastError();                                            // not enough memory for the big arena
        cap = 16LL << 20;
        if ((rc = ctx->d_ftab.ensure(ar.tab_off + (size_t)cap * sizeof(double)))) return rc;
    }
    unsigned char *base = ctx->d_ftab.as<unsigned char>();
    g.big = reinterpret_cast<BigInfo *>(base);
    g.fcursor = reinterpret_cast<unsigned long long *>(base + ar.ctr_off);
    g.counters = reinterpret_cast<unsigned int *>(base + ar.ctr_off + 16);
    g.lists = reinterpret_cast<int *>(base + ar.list_off);
    g.items = reinterpret_cast<int *>(base + ar.item_off);
    g.row_items = reinterpret_cast<int *>(base + ar.row_off);
    g.ftab = reinterpret_cast<double *>(base + ar.tab_off);
    g.ftab_cap = cap;
    if (d_overflow_flag) *d_overflow_flag = g.fcursor;                 // [0] doubles needed, [1] overflow
    CUDA_TRY(cudaMemsetAsync(base + ar.ctr_off, 0, 48 + sizeof(int), ctx->stream));   // cursors, counters, lists[0]
    grid_classify_kernel<<<(nproblems + 7) / 8, 256, 0, ctx->stream>>>(g);
    // fused launches: a share of the blocks serves the small surfaces, the rest the large ones
    const int per_sm = 8;
    int nsmall = (nproblems + 7) / 8;
    if (nsmall > ctx->sm_count * per_sm / 2) nsmall = ctx->sm_count * per_sm / 2;
    g.nblk_small = nsmall;
    g.target_ctas = ctx->sm_count * 6;
    grid_points_setup_kernel<<<nsmall + ctx->sm_count * per_sm / 2, 256, 0, ctx->stream>>>(g);
    grid_reduce_eval_kernel<<<nsmall + ctx->sm_count * 4, 256, 0, ctx->stream>>>(g);
    grid_rows_reduce_kernel<<<ctx->sm_count * 4, 256, 0, ctx->stream>>>(g);
    CUDA_TRY(cudaGetLastError());
    ctx->mark(3);
    ctx->launches += 4;
    return TREDSW_OK;
}

extern "C" int tredsw_likelihood_grid(tredsw_ctx *ctx, const tredsw_grid_problem *problems, int32_t nproblems,
                                      const int32_t *ipool, int64_t n_ipool, const double *dpool,
                                      int64_t n_dpool, double *surface, int64_t n_surface, double *marg,
                                      int64_t n_marg, tredsw_grid_result *results, uint32_t flags) {
    if (!ctx) { tredsw_set_error("null context"); return TREDSW_ERR_ARG; }
    if (nproblems < 0 || !problems || !results) { tredsw_set_error("bad arguments"); return TREDSW_ERR_ARG; }
    if (nproblems == 0) return TREDSW_OK;
    const bool dev = dev_ptrs(flags);
    if (dev && !surface) { tredsw_set_error("device mode needs the surface buffer (it is the kernels' scratch)"); return TREDSW_ERR_ARG; }
    int tables, rc;
    if ((rc = tredsw_internal_grid_tables(&tables))) return rc;
    std::lock_guard<std::mutex> lock(ctx->mu);
    CUDA_TRY(cudaSetDevice(ctx->device));
    // host mode: the surface is materialised iff the caller wants it back; device mode: unless TREDSW_GRID_NO_SURFACE
    const int materialise = dev ? ((flags & TREDSW_GRID_NO_SURFACE) ? 0 : 1) : ((surface && n_surface > 0) ? 1 : 0);
    GridParams g{};
    long long max_points = 0;
    if (!dev) {
        for (int i = 0; i < nproblems; ++i) {
            const tredsw_grid_problem &P = problems[i];
            if (P.n_h1 < 0 || P.n_h2 < 0 || P.period < 1 || P.readlen < 1 ||
                P.off_surface + (long long)P.n_h1 * P.n_h2 > n_surface || P.off_ph1 + P.n_h1 > n_marg ||
                P.off_ph2 + P.n_h2 > n_marg) { tredsw_set_error("grid problem %d out of range", i); return TREDSW_ERR_ARG; }
            long long t = (long long)P.n_h1 * P.n_h2;
            if (t > max_points) max_points = t;
        }
    } else {
        max_points = n_surface;   // upper bound
    }
    if ((rc = stage_in(ctx, ctx->d_prob, problems, (size_t)nproblems, flags, &g.prob))) return rc;
    if ((rc = stage_in(ctx, ctx->d_ipool, ipool, (size_t)n_ipool, flags, &g.ipool))) return rc;
    if ((rc = stage_in(ctx, ctx->d_dpool, dpool, (size_t)n_dpool, flags, &g.dpool))) return rc;
    if (dev) { g.surface = surface; g.marg = marg; g.res = results; }
    else {
        if ((rc = ctx->d_surface.ensure((size_t)(n_surface > 0 ? n_surface : 1) * sizeof(double)))) return rc;
        if ((rc = ctx->d_marg.ensure((size_t)(n_marg > 0 ? n_marg : 1) * sizeof(double)))) return rc;
        if ((rc = ctx->d_res.ensure((size_t)nproblems * sizeof(tredsw_grid_result)))) return rc;
        g.surface = ctx->d_surface.as<double>(); g.marg = ctx->d_marg.as<double>();
        g.res = ctx->d_res.as<tredsw_grid_result>();
    }
    for (int attempt = 0; attempt < 2; ++attempt) {
        unsigned long long *d_flag = nullptr;
        if ((rc = tredsw_internal_grid(ctx, g.prob, nproblems, g.ipool, g.dpool, g.surface, g.marg, g.res, max_points,
                                       materialise, nullptr, 0, nullptr, &d_flag, tables))) return rc;
        if (dev) return TREDSW_OK;
        unsigned long long h_flag[2] = {0, 0};
        CUDA_TRY(cudaMemcpyAsync(h_flag, d_flag, sizeof(h_flag), cudaMemcpyDeviceToHost, ctx->stream));
        CUDA_TRY(cudaStreamSynchronize(ctx->stream));
        if (!h_flag[1]) break;
        if (attempt == 1) { tredsw_set_error("likelihood table arena overflow (%llu doubles needed)", h_flag[0]); return TREDSW_ERR_UNSUPPORTED; }
        if ((rc = ctx->d_ftab.ensure(grid_area(nproblems).tab_off + (size_t)(h_flag[0] + h_flag[0] / 8) * sizeof(double)))) return rc;
    }
    if (surface && n_surface > 0)
        CUDA_TRY(cudaMemcpyAsync(surface, g.surface, (size_t)n_surface * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    if (marg && n_marg > 0)
        CUDA_TRY(cudaMemcpyAsync(marg, g.marg, (size_t)n_marg * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(results, g.res, (size_t)nproblems * sizeof(tredsw_grid_result), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return TREDSW_OK;
}

extern "C" int tredsw_pe_kde(tredsw_ctx *ctx, const int32_t *lens, const int64_t *off, int32_t nproblems,
                             double *pdf_out, uint32_t flags) {
    if (!ctx) { tredsw_set_error("null context"); return TREDSW_ERR_ARG; }
    if (nproblems < 0 || !off || !pdf_out) { tredsw_set_error("bad arguments"); return TREDSW_ERR_ARG; }
    if (nproblems == 0) return TREDSW_OK;
    std::lock_guard<std::mutex> lock(ctx->mu);
    CUDA_TRY(cudaSetDevice(ctx->device));
    const int32_t *d_lens; const int64_t *d_off; double *d_out;
    int rc;
    if (dev_ptrs(flags)) { d_lens = lens; d_off = off; d_out = pdf_out; }
    else {
        if ((rc = stage_in(ctx, ctx->d_ipool, lens, (size_t)off[nproblems], flags, &d_lens))) return rc;
        if ((rc = stage_in(ctx, ctx->d_qoff, off, (size_t)nproblems + 1, flags, &d_off))) return rc;
        if ((rc = ctx->d_dpool.ensure((size_t)nproblems * SPAN * sizeof(double)))) return rc;
        d_out = ctx->d_dpool.as<double>();
    }
    int gb = nproblems > ctx->sm_count * 8 ? ctx->sm_count * 8 : nproblems;
    pe_kde_kernel<<<gb, KDE_THREADS, 0, ctx->stream>>>(d_lens, d_off, nproblems, d_out);
    CUDA_TRY(cudaGetLastError());
    ctx->launches += 1;
    if (!dev_ptrs(flags)) {
        CUDA_TRY(cudaMemcpyAsync(pdf_out, d_out, (size_t)nproblems * SPAN * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    }
    return TREDSW_OK;
}
