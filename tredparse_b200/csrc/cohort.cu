// cohort.cu — whole (sample, locus) problems on the device: the per-locus loop body of
// tredparse/tred.py:225-275 for a cohort shard, minus BAM I/O.
//
//   reads --sw_family--> (tag, h) per read            bam_parser.py:123-182
//         --tally-----> FULL / PREF(+POST) / REPT histograms per problem      bam_parser.py:259-268, 256
//         --plan------> observed keys, run_pe, candidate lists (Q9 duplicates kept)   models.py:224-257, 399-403
//         --kde-------> normalised pair-length pdf per problem                 models.py:428-435
//         --grid------> log-likelihood surface + max / arg-max / marginals / PP sums  models.py:260-302
//         --finalize--> alleles, CI (Q11), PP, label                          models.py:287-290, 319-392, 406-413
//
// No host round trip between the stages; one problem = one thread in the bookkeeping kernels.
#include "internal.cuh"
#include "kde.cuh"

namespace {

constexpr int FLANKMATCH = 9;
constexpr int NSTEP = 37;

struct CohortDev {
    const tredsw_problem *problems;
    const tredsw_family *families;
    const tredsw_locus *loci;
    const int32_t *read_problem;
    const int32_t *read_out;     // nreads x 8
    int nreads, nproblems;
    int HU;                      // histogram units capacity (bins 0..HU)
    int KC;                      // key capacity per problem
    int HL;                      // candidate-list capacity per problem
    int32_t *hist;               // nproblems x 3 x (HU+1)
    int32_t *ipool;              // [pe_lens copy | per-problem slots]
    int64_t slot_base;           // offset of the first slot in ipool
    double *dpool;               // [nproblems x 1000 pdf | nfamilies x 37 step]
    int64_t step_base;
    tredsw_grid_problem *gp;
    int32_t *nbase;              // nproblems x 2: length of the sorted "base" part of h1 / h2 lists
    double *marg;                // nproblems x 2 x HL
    unsigned long long *counters;// [0] surface arena cursor, [1] overflow flag, [2] points
    long long surface_cap;
    int maxinsert, fullsearch;
    double w0, w1, w2, w3, w4, gc, score;
    const int32_t *read_name;    // name ids (norepeatpairs) or NULL
    int32_t *read_rw;            // read_out, writable (REPT-pair removal rewrites tags)
    int8_t *drop;                // nreads flags: read removed with its REPT pair
    int norepeatpairs;
    tredsw_posterior *post;      // sparse posterior entries (optional)
    long long post_cap;
    unsigned long long *post_cursor;
    double small_value;
};

__global__ void read_family_kernel(const int32_t *read_problem, const tredsw_problem *problems, int nreads,
                                   int nproblems, int32_t *read_family) {
    int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r < nreads) {
        int p = read_problem[r];
        read_family[r] = (p >= 0 && p < nproblems) ? problems[p].family : -1;
    }
}

// compact transfer formats -> regular device layouts (tredsw_cohort.input_flags)
__global__ void unpack_reads4_kernel(const uint32_t *packed, int64_t nwords, uint32_t *out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nwords) return;
    const uint32_t w = packed[i];                       // 8 bases
    out[2 * i] = (w & 0xfu) | ((w >> 4) & 0xfu) << 8 | ((w >> 8) & 0xfu) << 16 | ((w >> 12) & 0xfu) << 24;
    out[2 * i + 1] = ((w >> 16) & 0xfu) | ((w >> 20) & 0xfu) << 8 | ((w >> 24) & 0xfu) << 16 | ((w >> 28) & 0xfu) << 24;
}
__global__ void widen_i16_kernel(const int16_t *in, int64_t n, int32_t *out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (int32_t)in[i];
}

// remove_pairs_of_rept (bam_parser.py:270-287): a name carried by more than one REPT read of a problem is
// removed from the evidence altogether — every read of that name that made it into `details` (any tag but HANG).
// Reads of a problem are contiguous, so each read scans its problem's neighbourhood (~10^2 reads).  Clip families
// skip this (bam_parser.py:248: `if not (self.repeatpairs or self.clip)`).
__global__ void rept_pairs_mark_kernel(CohortDev c) {
    int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= c.nreads) return;
    c.drop[r] = 0;
    const int tag = c.read_out[(int64_t)r * 8];
    const int p = c.read_problem[r];
    if (tag <= 0 || tag == TREDSW_TAG_HANG || p < 0 || p >= c.nproblems) return;
    if (c.families[c.problems[p].family].clip) return;
    const int name = c.read_name[r];
    int n_rept = 0;
    for (int j = r; j >= 0 && c.read_problem[j] == p; --j)
        if (c.read_name[j] == name && c.read_out[(int64_t)j * 8] == TREDSW_TAG_REPT) ++n_rept;
    for (int j = r + 1; j < c.nreads && c.read_problem[j] == p; ++j)
        if (c.read_name[j] == name && c.read_out[(int64_t)j * 8] == TREDSW_TAG_REPT) ++n_rept;
    if (n_rept > 1) c.drop[r] = 1;
}
__global__ void rept_pairs_apply_kernel(CohortDev c) {
    int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r < c.nreads && c.drop[r]) c.read_rw[(int64_t)r * 8] = TREDSW_TAG_REPT_PAIR;
}

__global__ void tally_kernel(CohortDev c) {
    int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= c.nreads) return;
    const int32_t *o = c.read_out + (int64_t)r * 8;
    const int tag = o[0], h = o[1];
    const int p = c.read_problem[r];
    if (p < 0 || p >= c.nproblems || tag <= 0 || tag == TREDSW_TAG_HANG || tag == TREDSW_TAG_REPT_PAIR || h < 0 || h > c.HU) return;
    // PREF and POST share one histogram (bam_parser.py:77)
    const int which = tag == TREDSW_TAG_FULL ? 0 : (tag == TREDSW_TAG_REPT ? 2 : 1);
    atomicAdd(&c.hist[((int64_t)p * 3 + which) * (c.HU + 1) + h], 1);
}

// One warp per problem: histogram bins -> observed keys (ordered compaction by ballot), run_pe, candidate lists.
__global__ void __launch_bounds__(256) plan_kernel(CohortDev c) {
    const int lane = threadIdx.x & 31;
    const int p = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (p >= c.nproblems) return;
    const tredsw_problem pr = c.problems[p];
    const tredsw_locus L = c.loci[pr.family];
    const int P = L.period;
    const int t2 = L.readlen - 2 * FLANKMATCH, t3 = L.readlen - 3 * FLANKMATCH;
    const int32_t *hf = c.hist + ((int64_t)p * 3 + 0) * (c.HU + 1);
    const int32_t *hp = hf + (c.HU + 1), *hr = hp + (c.HU + 1);
    int32_t *slot = c.ipool + c.slot_base + (int64_t)p * (4 * c.KC + 2 * c.HL);
    int32_t *skey = slot, *scnt = slot + c.KC, *pkey = slot + 2 * c.KC, *pcnt = slot + 3 * c.KC;
    int32_t *h1s = slot + 4 * c.KC, *h2s = h1s + c.HL;
    const unsigned lt = (1u << lane) - 1u;
    int ns = 0, np_ = 0, max_full = 0, max_partial = 0, n_rept = 0;
    for (int k0 = 0; k0 <= c.HU; k0 += 32) {
        const int k = k0 + lane;
        const int f = k <= c.HU ? hf[k] : 0, q = k <= c.HU ? hp[k] : 0, r = k <= c.HU ? hr[k] : 0;
        const unsigned mf = __ballot_sync(0xffffffffu, f > 0), mq = __ballot_sync(0xffffffffu, q > 0);
        const int pf = ns + __popc(mf & lt), pq = np_ + __popc(mq & lt);
        if (f > 0 && pf < c.KC) { skey[pf] = k * P; scnt[pf] = f; }
        if (q > 0 && pq < c.KC) { pkey[pq] = k * P; pcnt[pq] = q; }
        if (mf) max_full = (k0 + 31 - __clz(mf)) * P;
        if (mq) max_partial = (k0 + 31 - __clz(mq)) * P;
        ns = min(ns + __popc(mf), c.KC); np_ = min(np_ + __popc(mq), c.KC);
        n_rept += __reduce_add_sync(0xffffffffu, r);
    }
    __syncwarp();
    // counts directly after the keys (keys[n] then counts[n]); the two regions may overlap: read, then write
    {
        int vs[8], vp[8];                                    // KC <= 256 (checked by the caller)
#pragma unroll
        for (int j = 0; j < 8; ++j) { const int i = lane + 32 * j; vs[j] = i < ns ? scnt[i] : 0; vp[j] = i < np_ ? pcnt[i] : 0; }
        __syncwarp();
#pragma unroll
        for (int j = 0; j < 8; ++j) { const int i = lane + 32 * j; if (i < ns) skey[ns + i] = vs[j]; if (i < np_) pkey[np_ + i] = vp[j]; }
        __syncwarp();
    }
    int above = 0;
    for (int i = lane; i < np_; i += 32) if (pkey[i] > max_full + P) above += pkey[np_ + i];
    above = __reduce_add_sync(0xffffffffu, above);
    const bool has_pe = pr.n_global >= 100 && pr.n_target >= 5;
    const bool run_pe = max_partial >= t3 && above > 1 && has_pe;
    int mp_model = t2;
    if (np_ > 0 && max_partial > mp_model) mp_model = max_partial;
    // base = sorted(set(span keys) U {max_partial}), built by lane 0 (<= KC entries)
    int nb = 0;
    if (lane == 0) {
        bool placed = (np_ == 0);
        for (int i = 0; i < ns; ++i) {
            const int k = skey[i];
            if (!placed && max_partial < k) { h1s[nb++] = max_partial; placed = true; }
            if (!placed && max_partial == k) placed = true;
            h1s[nb++] = k;
        }
        if (!placed) h1s[nb++] = max_partial;
    }
    nb = __shfl_sync(0xffffffffu, nb, 0);
    __syncwarp();
    int n1 = 0, n2 = 0, nb1 = 0, nb2 = 0;
    if (nb > 0) {
        if (c.fullsearch) {
            n1 = min(c.maxinsert, c.HL);
            for (int i = lane; i < n1; i += 32) { h1s[i] = P * (i + 1); h2s[i] = P * (i + 1); }
            n2 = n1; nb1 = n1; nb2 = n2;
        } else {
            const bool ext1 = (max_full == 0), ext2 = (n_rept > 0 || run_pe);
            for (int i = lane; i < nb; i += 32) h2s[i] = h1s[i];
            // extension: max_partial + P, max_partial + 2P, ..., P * maxinsert
            const int next = max(0, c.maxinsert - max_partial / P);
            const int e1 = ext1 ? min(next, c.HL - nb) : 0, e2 = ext2 ? min(next, c.HL - nb) : 0;
            for (int j = lane; j < e1; j += 32) h1s[nb + j] = max_partial + P * (j + 1);
            for (int j = lane; j < e2; j += 32) h2s[nb + j] = max_partial + P * (j + 1);
            n1 = nb + e1; n2 = nb + e2; nb1 = nb; nb2 = nb;
        }
        if (pr.ploidy == 1) { n2 = 1; nb2 = 1; }
    }
    if (lane != 0) return;
    tredsw_grid_problem g;
    memset(&g, 0, sizeof(g));
    g.period = P; g.readlen = L.readlen; g.ploidy = pr.ploidy; g.n_rept = n_rept;
    g.max_partial = mp_model; g.run_pe = run_pe ? 1 : 0; g.pe_ref = L.pe_ref; g.pe_minpe = L.pe_minpe;
    g.n_span = ns; g.n_part = np_; g.n_target = run_pe ? pr.n_target : 0;
    g.expansion = L.expansion; g.recessive = L.recessive; g.cutoff_risk = L.cutoff_risk;
    g.half_depth = pr.depth / 2;
    g.stutter_a = c.w0 + c.w1 * (double)P; g.stutter_w2 = c.w2; g.stutter_c3 = c.w3 * c.gc; g.stutter_c4 = c.w4 * c.score;
    g.off_span = skey - c.ipool; g.off_part = pkey - c.ipool; g.off_target = pr.off_target;
    g.off_h1 = h1s - c.ipool; g.off_h2 = h2s - c.ipool;
    g.off_pdf = run_pe ? (int64_t)p * KDE_SPAN : -1;
    g.off_step = c.step_base + (int64_t)pr.family * NSTEP;
    g.off_ph1 = (int64_t)p * 2 * c.HL; g.off_ph2 = g.off_ph1 + c.HL;
    g.n_h1 = n1; g.n_h2 = n2;
    const long long need = (long long)n1 * n2;
    long long off = 0;
    if (need > 0) {
        off = (long long)atomicAdd(&c.counters[0], (unsigned long long)need);
        if (off + need > c.surface_cap) { atomicExch(&c.counters[1], 1ull); g.n_h1 = 0; g.n_h2 = -1; off = 0; }   // n_h2 = -1 marks the overflow
    }
    g.off_surface = off;
    c.gp[p] = g;
    c.nbase[2 * p] = nb1; c.nbase[2 * p + 1] = nb2;
}

__global__ void __launch_bounds__(KDE_THREADS) cohort_kde_kernel(CohortDev c, const int32_t *pe_lens) {
    for (int p = blockIdx.x; p < c.nproblems; p += gridDim.x) {
        if (!c.gp[p].run_pe) continue;          // block-uniform
        const tredsw_problem pr = c.problems[p];
        kde_block(pe_lens + pr.off_global, pr.n_global, c.dpool + (int64_t)p * KDE_SPAN);
    }
}

// 95% interval over the merged, sorted keys of a marginal (models.py:319-340) and its sparsified form
// (models.py:304-317), by one warp.  The candidate list is a sorted base part [0, nb) followed by an ascending
// extension [nb, n); equal keys are one key of the reference's defaultdict (their weights add up); entries outside
// [ulo, uhi] never became keys (an h1 above every h2, an h2 below every h1: no evaluated point uses them).
// cum(x) = sum of the weights of the keys <= x is evaluated by the whole warp; the interval ends are the smallest
// keys with cum > 2.5 % / 97.5 % of the total — found by bisection in each sorted part, no serial merge.
struct Marginal {
    const int32_t *hs;
    const double *w;
    int n, nb, ulo, uhi;
    __device__ __forceinline__ bool used(int h) const { return h >= ulo && h <= uhi; }
    __device__ __forceinline__ double cum(int x, int lane) const {
        double a = 0.0;
        for (int i = lane; i < n; i += 32) { const int h = hs[i]; if (h <= x && used(h)) a += w[i]; }
        for (int d = 16; d > 0; d >>= 1) a += __shfl_xor_sync(0xffffffffu, a, d);
        return a;
    }
    // smallest used key of the sorted part [a, b) with cum(key) > thr; INT_MAX when there is none
    __device__ __forceinline__ int first_above(int a, int b, double thr, int lane) const {
        int lo = a, hi = b;
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (cum(hs[mid], lane) > thr) hi = mid; else lo = mid + 1;
        }
        return (lo < b && used(hs[lo])) ? hs[lo] : 0x7fffffff;
    }
};

__device__ void ci_of(const CohortDev &c, int p, int kind, int period, const Marginal &m, int lane, int &lo, int &hi) {
    const double total = m.cum(0x7fffffff, lane);
    int last = -0x7fffffff;
    for (int i = lane; i < m.n; i += 32) if (m.used(m.hs[i])) last = max(last, m.hs[i]);
    last = __reduce_max_sync(0xffffffffu, last);
    lo = 0; hi = 0;
    if (last != -0x7fffffff) {
        const int l = min(m.first_above(0, m.nb, .025 * total, lane), m.first_above(m.nb, m.n, .025 * total, lane));
        const int h = min(m.first_above(0, m.nb, .975 * total, lane), m.first_above(m.nb, m.n, .975 * total, lane));
        lo = l == 0x7fffffff ? 0 : l;
        hi = h == 0x7fffffff ? last : h;
    }
    if (!c.post) return;
    for (int i = lane; i < m.n; i += 32) {
        const int key = m.hs[i];
        if (!m.used(key)) continue;
        double v = m.w[i];
        if (i >= m.nb) {
            bool second = false;                                   // already a key of the base part?
            if (m.nb > 0 && key <= m.hs[m.nb - 1]) for (int j = 0; j < m.nb; ++j) if (m.hs[j] == key) second = true;
            if (second) continue;
        } else {
            int a = m.nb, b = m.n;                                 // the same key among the extension
            while (a < b) { const int mid = (a + b) >> 1; if (m.hs[mid] < key) a = mid + 1; else b = mid; }
            if (a < m.n && m.hs[a] == key) v += m.w[a];
        }
        if (v >= c.small_value) {
            const unsigned long long at = atomicAdd(c.post_cursor, 1ULL);
            if ((long long)at < c.post_cap) {
                tredsw_posterior e;
                e.problem = p; e.kind = kind; e.a = key / period; e.b = 0; e.p = v / total;
                c.post[at] = e;
            }
        }
    }
}

// one warp per problem
__global__ void __launch_bounds__(256) finalize_kernel(CohortDev c, const tredsw_grid_result *res, tredsw_call *calls) {
    const int lane = threadIdx.x & 31;
    const int p = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (p >= c.nproblems) return;
    const tredsw_grid_problem g = c.gp[p];
    const tredsw_locus L = c.loci[c.problems[p].family];
    const int32_t *hf = c.hist + ((int64_t)p * 3 + 0) * (c.HU + 1);
    tredsw_call out;
    memset(&out, 0, sizeof(out));
    int fdp = 0, pdp = 0;
    for (int k = lane; k <= c.HU; k += 32) { fdp += hf[k]; pdp += hf[(c.HU + 1) + k]; }
    out.fdp = __reduce_add_sync(0xffffffffu, fdp); out.pdp = __reduce_add_sync(0xffffffffu, pdp);
    out.rdp = g.n_rept; out.run_pe = g.run_pe;
    int a1 = -1, a2 = -1;
    if (g.n_h1 == 0 || res[p].n_points <= 0) {
        out.allele1 = out.allele2 = -1;
        out.ci[0] = out.ci[1] = out.ci[2] = out.ci[3] = -1;
        out.pp = -1; out.lik = -1; out.n_points = (g.n_h2 < 0 || res[p].n_points < 0) ? -1 : 0;   // -1: an arena overflowed
    } else {
        const tredsw_grid_result r = res[p];
        const int32_t *h1s = c.ipool + g.off_h1, *h2s = c.ipool + g.off_h2;
        const int h1 = h1s[r.arg_i1];
        const int h2 = g.ploidy == 1 ? h1 : h2s[r.arg_i2];
        a1 = min(h1, h2) / g.period; a2 = max(h1, h2) / g.period;
        out.allele1 = a1; out.allele2 = a2;
        out.pp = fmin(1.0, r.sum_path / r.sum_all);
        out.lik = r.max_ml; out.n_points = r.n_points;
        const double *ph1 = c.marg + g.off_ph1, *ph2 = c.marg + g.off_ph2;
        int lo1, hi1, lo2, hi2;
        if (g.ploidy == 1) {
            const Marginal m{h1s, ph1, g.n_h1, c.nbase[2 * p], -0x7fffffff, 0x7fffffff};
            ci_of(c, p, TREDSW_POST_H1, g.period, m, lane, lo1, hi1);
            if (c.post) ci_of(c, p, TREDSW_POST_H2, g.period, m, lane, lo2, hi2);      // h2 = h1: the same marginal
            lo2 = lo1; hi2 = hi1;
        } else {
            int mx2 = -0x7fffffff, mn1 = 0x7fffffff;
            for (int i = lane; i < g.n_h2; i += 32) mx2 = max(mx2, h2s[i]);
            for (int i = lane; i < g.n_h1; i += 32) mn1 = min(mn1, h1s[i]);
            mx2 = __reduce_max_sync(0xffffffffu, mx2); mn1 = __reduce_min_sync(0xffffffffu, mn1);
            const Marginal m1{h1s, ph1, g.n_h1, c.nbase[2 * p], -0x7fffffff, mx2};
            const Marginal m2{h2s, ph2, g.n_h2, c.nbase[2 * p + 1], mn1, 0x7fffffff};
            ci_of(c, p, TREDSW_POST_H1, g.period, m1, lane, lo1, hi1);
            ci_of(c, p, TREDSW_POST_H2, g.period, m2, lane, lo2, hi2);
        }
        out.ci[0] = lo1 / g.period; out.ci[1] = hi1 / g.period; out.ci[2] = lo2 / g.period; out.ci[3] = hi2 / g.period;
        if (lane == 0) {
            atomicAdd(&c.counters[2], (unsigned long long)r.n_points);
            if (c.post) {                                    // divisor of this problem's joint entries
                const unsigned long long at = atomicAdd(c.post_cursor, 1ULL);
                if ((long long)at < c.post_cap) {
                    tredsw_posterior e;
                    e.problem = p; e.kind = TREDSW_POST_JOINT_TOTAL; e.a = 0; e.b = 0; e.p = r.sum_uniq;
                    c.post[at] = e;
                }
            }
        }
    }
    if (lane != 0) return;
    // label (models.py:370-392)
    int label = (a1 != -1) ? 0 : 3;
    if (L.expansion) {
        const int crit = L.recessive ? a1 : a2;
        if (L.cutoff_prerisk <= crit && crit < L.cutoff_risk) label = 1;
        else if (crit >= L.cutoff_risk) label = 2;
    } else {
        const int crit = L.recessive ? a2 : a1;
        if (L.cutoff_prerisk <= crit && crit < L.cutoff_risk) label = 1;
        else if (0 < crit && crit <= L.cutoff_risk) label = 2;
    }
    out.label = label;
    calls[p] = out;
}

}  // namespace

extern "C" int tredsw_genotype_batch(tredsw_ctx *ctx, const tredsw_cohort *c, uint32_t flags, tredsw_call *calls,
                                     int32_t *read_out, int32_t *hist, int32_t hist_units, int64_t *stats) {
    return tredsw_genotype_batch_ex(ctx, c, flags, calls, read_out, hist, hist_units, stats, nullptr, 0, nullptr);
}

extern "C" int tredsw_genotype_batch_ex(tredsw_ctx *ctx, const tredsw_cohort *c, uint32_t flags, tredsw_call *calls,
                                        int32_t *read_out, int32_t *hist, int32_t hist_units, int64_t *stats,
                                        tredsw_posterior *post, int64_t post_cap, int64_t *n_post) {
    if (!ctx || !c || !calls) { tredsw_set_error("null argument"); return TREDSW_ERR_ARG; }
    if (post && (post_cap <= 0 || !n_post)) { tredsw_set_error("post needs post_cap > 0 and n_post"); return TREDSW_ERR_ARG; }
    if (c->norepeatpairs && c->nreads > 0 && !c->read_name) { tredsw_set_error("norepeatpairs needs read_name"); return TREDSW_ERR_ARG; }
    if (c->nproblems <= 0 || c->nreads < 0 || c->nfamilies <= 0 || !c->families || !c->loci || !c->step_pmf ||
        c->max_read_len <= 0 || c->maxinsert < 1) { tredsw_set_error("bad cohort descriptor"); return TREDSW_ERR_ARG; }
    int grid_tables;
    if (int rc0 = tredsw_internal_grid_tables(&grid_tables)) return rc0;
    const bool dev = dev_ptrs(flags);
    // TREDSW_DEVICE_INPUTS: the bulk evidence (rbuf, roff, read_problem, pe_lens) already lies in device memory — e.g.
    // where tredsw_ingest_batch_run left it — while `problems`, `read_name` and every output are host buffers that
    // travel through the page-locked staging of the host mode (the call returns when the outputs are valid)
    const bool dev_in = dev || (flags & TREDSW_DEVICE_INPUTS) != 0;
    if (!dev_in && c->nreads > 0) {
        // host buffers can be checked: a read longer than max_read_len would be skipped by the kernels (their row
        // buffers are sized by it), i.e. silently lose evidence
        if (!c->roff || !c->rbuf || !c->read_problem || !c->problems) { tredsw_set_error("null input buffer"); return TREDSW_ERR_ARG; }
        int64_t longest = 0;
        for (int32_t i = 0; i < c->nreads; ++i) { const int64_t l = c->roff[i + 1] - c->roff[i]; longest = l > longest ? l : longest; }
        if (longest > c->max_read_len) {
            tredsw_set_error("a read of %lld bases exceeds max_read_len = %d", (long long)longest, c->max_read_len);
            return TREDSW_ERR_ARG;
        }
    }
    std::lock_guard<std::mutex> lock(ctx->mu);
    CUDA_TRY(cudaSetDevice(ctx->device));
    ctx->mark(8);
    ctx->wait_before_sw = nullptr; ctx->record_sw_end = false;
    const int nr = c->nreads, np_ = c->nproblems, nf = c->nfamilies;
    int max_u = 0, min_period = 1 << 30;
    for (int f = 0; f < nf; ++f) {
        if (c->families[f].max_units > max_u) max_u = c->families[f].max_units;
        if (c->loci[f].period < min_period) min_period = c->loci[f].period;
    }
    const int HU = max_u;
    if (hist && hist_units != HU) { tredsw_set_error("hist_units must equal the largest max_units (%d)", HU); return TREDSW_ERR_ARG; }
    const int KC = HU + 2;
    if (KC > 256) { tredsw_set_error("max_units %d too large (<= 254)", HU); return TREDSW_ERR_UNSUPPORTED; }
    const int HL = c->maxinsert + KC + 2;
    int rc;
    // ---- inputs ------------------------------------------------------------------------------------
    const int8_t *d_rbuf = c->rbuf; const int64_t *d_roff = c->roff; const int32_t *d_rp = c->read_problem;
    const tredsw_problem *d_prob = c->problems;
    const int32_t *d_rname = c->read_name;
    const tredsw_family *d_fam; const tredsw_locus *d_loci;
    const bool packed4 = (c->input_flags & TREDSW_IN_READS_PACKED4) != 0, pe16 = (c->input_flags & TREDSW_IN_PE_LENS_I16) != 0;
    if (dev_in && c->n_bases <= 0 && nr > 0 && (packed4 || !dev)) { tredsw_set_error("n_bases is required for reads in device memory"); return TREDSW_ERR_ARG; }
    const int64_t nbases = nr > 0 ? (dev_in ? c->n_bases : c->roff[nr]) : 0;
    const uint32_t *unpack_src = nullptr; int64_t unpack_words = 0;
    const int16_t *widen_src = nullptr;
    if (packed4 && nr > 0) {
        // rbuf holds nibbles: bring the packed words to the device, expand into the byte-per-base buffer
        const int64_t nwords = (nbases + 7) / 8;
        const uint32_t *d_pk = reinterpret_cast<const uint32_t *>(c->rbuf);
        if (!dev_in) {
            if ((rc = ctx->d_pk.ensure((size_t)nwords * 4))) return rc;
            CUDA_TRY(cudaMemcpyAsync(ctx->d_pk.p, c->rbuf, (size_t)(nbases + 1) / 2, cudaMemcpyHostToDevice, ctx->stream));
            d_pk = ctx->d_pk.as<uint32_t>();
        }
        if ((rc = ctx->d_q.ensure((size_t)nwords * 8))) return rc;
        unpack_src = d_pk; unpack_words = nwords;            // launched below, once every input copy is queued
        d_rbuf = ctx->d_q.as<int8_t>();
    }
    if (!dev_in && nr > 0) {
        if (!packed4 && (rc = stage_in(ctx, ctx->d_q, c->rbuf, (size_t)c->roff[nr], 0u, &d_rbuf))) return rc;
        if ((rc = stage_in(ctx, ctx->d_qoff, c->roff, (size_t)nr + 1, 0u, &d_roff))) return rc;
        if ((rc = stage_in(ctx, ctx->d_qidx, c->read_problem, (size_t)nr, 0u, &d_rp))) return rc;
    }
    // (name ids and problem records are made by host code in either mode)
    if (!dev && nr > 0 && c->norepeatpairs && (rc = stage_in(ctx, ctx->d_tidx, c->read_name, (size_t)nr, 0u, &d_rname))) return rc;
    if (!dev && (rc = stage_in(ctx, ctx->d_prob, c->problems, (size_t)np_, 0u, &d_prob))) return rc;
    // the small per-call tables (always host pointers) travel through the context's page-locked staging buffer
    const size_t b_step = (size_t)nf * NSTEP * sizeof(double);
    size_t hoff[3];
    {
        const void *srcs[3] = {c->families, c->loci, c->step_pmf};
        const size_t sizes[3] = {(size_t)nf * sizeof(tredsw_family), (size_t)nf * sizeof(tredsw_locus), b_step};
        if ((rc = stage_small(ctx, ctx->h_in, srcs, sizes, 3, hoff))) return rc;
    }
    const unsigned char *hin = ctx->h_in.as<unsigned char>();
    const size_t b_fam = hoff[1], b_loci = hoff[2] - hoff[1];
    if ((rc = stage_in(ctx, ctx->d_fam, reinterpret_cast<const tredsw_family *>(hin), (size_t)nf, 0u, &d_fam))) return rc;
    if ((rc = stage_in(ctx, ctx->d_t, reinterpret_cast<const tredsw_locus *>(hin + b_fam), (size_t)nf, 0u, &d_loci))) return rc;
    // ---- arenas ------------------------------------------------------------------------------------
    const int64_t slot_ints = 4 * (int64_t)KC + 2 * (int64_t)HL;
    const int64_t n_ipool = c->n_pe_lens + (int64_t)np_ * slot_ints;
    if ((rc = ctx->d_ipool.ensure((size_t)n_ipool * sizeof(int32_t)))) return rc;
    int32_t *d_ipool = ctx->d_ipool.as<int32_t>();
    if (c->n_pe_lens > 0 && pe16) {
        const int16_t *d16 = reinterpret_cast<const int16_t *>(c->pe_lens);
        if (!dev_in) {
            if ((rc = ctx->d_pe16.ensure((size_t)c->n_pe_lens * sizeof(int16_t)))) return rc;
            CUDA_TRY(cudaMemcpyAsync(ctx->d_pe16.p, c->pe_lens, (size_t)c->n_pe_lens * sizeof(int16_t), cudaMemcpyHostToDevice, ctx->stream));
            d16 = ctx->d_pe16.as<int16_t>();
        }
        widen_src = d16;
    } else if (c->n_pe_lens > 0)
        CUDA_TRY(cudaMemcpyAsync(d_ipool, c->pe_lens, (size_t)c->n_pe_lens * sizeof(int32_t),
                                 dev_in ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, ctx->stream));

    const int64_t n_dpool = (int64_t)np_ * KDE_SPAN + (int64_t)nf * NSTEP;
    if ((rc = ctx->d_dpool.ensure((size_t)n_dpool * sizeof(double)))) return rc;
    double *d_dpool = ctx->d_dpool.as<double>();
    CUDA_TRY(cudaMemcpyAsync(d_dpool + (int64_t)np_ * KDE_SPAN, hin + b_fam + b_loci, b_step,
                             cudaMemcpyHostToDevice, ctx->stream));
    // ---- compute token (common.cuh: DeviceToken) ---------------------------------------------------------
    // Every input copy of this call is queued by now and runs while earlier calls compute.  The kernels follow
    // in two steps: the expansion / pre-filter / grouping kernels wait until the previous call's Smith-Waterman
    // kernel has ended (they then share the GPU with that call's short finishing kernels instead of slowing its
    // SW kernel down), and this call's SW kernel waits until the previous call has finished altogether.
    DeviceToken &token = tredsw_device_token(ctx->device);
    std::unique_lock<std::mutex> token_lock(token.mu, std::defer_lock);
    static const bool no_token = getenv("TREDSW_NO_TOKEN") != nullptr;
    if (!dev && !no_token) {
        if (!ctx->done_ev) CUDA_TRY(cudaEventCreateWithFlags(&ctx->done_ev, cudaEventDisableTiming));
        if (!ctx->sw_end_ev) CUDA_TRY(cudaEventCreateWithFlags(&ctx->sw_end_ev, cudaEventDisableTiming));
        token_lock.lock();
        if (token.ev && token.ev != ctx->done_ev) {
            ctx->wait_before_sw = token.ev;
            if (token.sw_end) CUDA_TRY(cudaStreamWaitEvent(ctx->stream, token.sw_end, 0));
        }
        ctx->record_sw_end = true;
    }
    if (unpack_src) {
        unpack_reads4_kernel<<<(unsigned)((unpack_words + 255) / 256), 256, 0, ctx->stream>>>(unpack_src, unpack_words, ctx->d_q.as<uint32_t>());
        ctx->launches += 1;
    }
    if (widen_src) {
        widen_i16_kernel<<<(unsigned)((c->n_pe_lens + 255) / 256), 256, 0, ctx->stream>>>(widen_src, c->n_pe_lens, d_ipool);
        ctx->launches += 1;
    }
    // surface arena: default search needs <= (#base) x (#ext) points per problem; start generous, grow on overflow
    long long per_problem = c->fullsearch ? (long long)c->maxinsert * c->maxinsert : 16LL * HL;
    long long surface_cap = (long long)np_ * per_problem;
    if ((size_t)surface_cap * sizeof(double) < ctx->d_surface.cap) surface_cap = (long long)(ctx->d_surface.cap / sizeof(double));
    if ((rc = ctx->d_surface.ensure((size_t)surface_cap * sizeof(double)))) return rc;
    if ((rc = ctx->d_marg.ensure((size_t)np_ * 2 * HL * sizeof(double)))) return rc;
    if ((rc = ctx->d_res.ensure((size_t)np_ * sizeof(tredsw_grid_result)))) return rc;
    // misc: gp[np] | nbase[2np] | hist | read_family[nr] | read_out[nr*8] | calls[np] | counters
    const size_t sz_gp = (size_t)np_ * sizeof(tredsw_grid_problem);
    const size_t sz_hist = (size_t)np_ * 3 * (HU + 1) * sizeof(int32_t);
    size_t off = 0;
    auto carve = [&](size_t bytes) { size_t o = off; off += (bytes + 255) / 256 * 256; return o; };
    const size_t o_gp = carve(sz_gp), o_nb = carve((size_t)np_ * 2 * sizeof(int32_t)), o_hist = carve(sz_hist),
                 o_rf = carve((size_t)(nr + 1) * sizeof(int32_t)), o_ro = carve((size_t)(nr + 1) * 8 * sizeof(int32_t)),
                 o_calls = carve((size_t)np_ * sizeof(tredsw_call)), o_cnt = carve(8 * sizeof(unsigned long long)),
                 o_stats = carve(4 * sizeof(unsigned long long)), o_drop = carve((size_t)nr + 1);
    if ((rc = ctx->d_misc.ensure(off))) return rc;
    unsigned char *mb = ctx->d_misc.as<unsigned char>();
    if ((rc = ctx->d_work.ensure((tredsw_classify_work_words(c->families, nf, nr) + 1) * sizeof(int32_t)))) return rc;
    CohortDev cd{};
    cd.problems = d_prob; cd.families = d_fam; cd.loci = d_loci; cd.read_problem = d_rp;
    cd.nreads = nr; cd.nproblems = np_; cd.HU = HU; cd.KC = KC; cd.HL = HL;
    cd.hist = (dev && hist) ? hist : reinterpret_cast<int32_t *>(mb + o_hist);
    cd.ipool = d_ipool; cd.slot_base = c->n_pe_lens;
    cd.dpool = d_dpool; cd.step_base = (int64_t)np_ * KDE_SPAN;
    cd.gp = reinterpret_cast<tredsw_grid_problem *>(mb + o_gp);
    cd.nbase = reinterpret_cast<int32_t *>(mb + o_nb);
    cd.marg = ctx->d_marg.as<double>();
    cd.counters = reinterpret_cast<unsigned long long *>(mb + o_cnt);
    cd.surface_cap = surface_cap;
    cd.maxinsert = c->maxinsert; cd.fullsearch = c->fullsearch;
    cd.w0 = c->stutter_w[0]; cd.w1 = c->stutter_w[1]; cd.w2 = c->stutter_w[2]; cd.w3 = c->stutter_w[3]; cd.w4 = c->stutter_w[4];
    cd.gc = c->gc; cd.score = c->score;
    cd.small_value = exp(-10.0);
    cd.norepeatpairs = c->norepeatpairs; cd.read_name = d_rname;
    cd.drop = reinterpret_cast<int8_t *>(mb + o_drop);
    // sparse posteriors: device arena of post_cap entries; counters[3] is its cursor
    tredsw_posterior *d_post = nullptr;
    if (post) {
        if (dev) d_post = post;
        else { if ((rc = ctx->d_cigar.ensure((size_t)post_cap * sizeof(tredsw_posterior)))) return rc; d_post = ctx->d_cigar.as<tredsw_posterior>(); }
    }
    cd.post = d_post; cd.post_cap = post_cap; cd.post_cursor = cd.counters + 3;
    int32_t *d_read_family = reinterpret_cast<int32_t *>(mb + o_rf);
    int32_t *d_read_out = (dev && read_out) ? read_out : reinterpret_cast<int32_t *>(mb + o_ro);
    cd.read_out = d_read_out; cd.read_rw = d_read_out;
    tredsw_call *d_calls = dev ? calls : reinterpret_cast<tredsw_call *>(mb + o_calls);
    unsigned long long *d_stats = reinterpret_cast<unsigned long long *>(mb + o_stats);
    CUDA_TRY(cudaMemsetAsync(cd.hist, 0, sz_hist, ctx->stream));
    CUDA_TRY(cudaMemsetAsync(cd.counters, 0, 8 * sizeof(unsigned long long), ctx->stream));
    CUDA_TRY(cudaMemsetAsync(d_stats, 0, 4 * sizeof(unsigned long long), ctx->stream));
    // ---- pipeline ----------------------------------------------------------------------------------
    const int tb = 256;
    ctx->mark(6);
    if (nr > 0) {
        ctx->launches += 2;
        read_family_kernel<<<(nr + tb - 1) / tb, tb, 0, ctx->stream>>>(d_rp, d_prob, nr, np_, d_read_family);
        if ((rc = tredsw_internal_classify(ctx, d_rbuf, d_roff, nr, d_read_family, d_fam, c->families, nf,
                                           c->max_read_len, c->mat25, c->gap_open, c->gap_extend,
                                           ctx->d_work.as<int32_t>(), d_read_out, stats ? d_stats : nullptr))) return rc;
        if (c->norepeatpairs) {
            rept_pairs_mark_kernel<<<(nr + tb - 1) / tb, tb, 0, ctx->stream>>>(cd);
            rept_pairs_apply_kernel<<<(nr + tb - 1) / tb, tb, 0, ctx->stream>>>(cd);
            ctx->launches += 2;
        }
        tally_kernel<<<(nr + tb - 1) / tb, tb, 0, ctx->stream>>>(cd);
    }
    plan_kernel<<<(np_ + 7) / 8, 256, 0, ctx->stream>>>(cd);
    ctx->mark(4);
    // one block per problem (most exit at once: only problems with run_pe need the KDE); the hardware block
    // scheduler balances the sparse, uneven survivors better than a strided loop would
    cohort_kde_kernel<<<np_, KDE_THREADS, 0, ctx->stream>>>(cd, d_ipool);
    ctx->mark(5);
    CUDA_TRY(cudaGetLastError());
    ctx->launches += 3;
    unsigned long long *d_tab_flag = nullptr;
    if ((rc = tredsw_internal_grid(ctx, cd.gp, np_, d_ipool, d_dpool, ctx->d_surface.as<double>(), cd.marg,
                                   ctx->d_res.as<tredsw_grid_result>(), c->fullsearch ? per_problem : 4LL * HL, 0,
                                   d_post, post_cap, cd.post_cursor, &d_tab_flag, grid_tables))) return rc;
    finalize_kernel<<<(np_ + 7) / 8, 256, 0, ctx->stream>>>(cd, ctx->d_res.as<tredsw_grid_result>(), d_calls);
    CUDA_TRY(cudaGetLastError());
    ctx->mark(7);
    if (token_lock.owns_lock()) {
        if (ctx->record_sw_end) {                            // nr == 0: no SW launch recorded it
            CUDA_TRY(cudaEventRecord(ctx->sw_end_ev, ctx->stream));
            ctx->record_sw_end = false;
        }
        ctx->wait_before_sw = nullptr;
        CUDA_TRY(cudaEventRecord(ctx->done_ev, ctx->stream));
        token.ev = ctx->done_ev; token.sw_end = ctx->sw_end_ev;
        token_lock.unlock();
    }
    // ---- outputs -----------------------------------------------------------------------------------
    // calls and counters come back through the page-locked staging buffer (see PinnedBuf); the optional bulky
    // per-read / histogram outputs go straight to the caller's memory
    const size_t b_calls = ((size_t)np_ * sizeof(tredsw_call) + 255) & ~(size_t)255;
    if ((rc = ctx->h_out.ensure(b_calls + 14 * sizeof(unsigned long long)))) return rc;
    unsigned char *hout = ctx->h_out.as<unsigned char>();
    unsigned long long *h_cnt = reinterpret_cast<unsigned long long *>(hout + b_calls), *h_st = h_cnt + 8, *h_tab = h_cnt + 12;
    if (dev && post) CUDA_TRY(cudaMemcpyAsync(n_post, cd.post_cursor, sizeof(int64_t), cudaMemcpyDeviceToDevice, ctx->stream));
    if (!dev) {
        CUDA_TRY(cudaMemcpyAsync(hout, d_calls, (size_t)np_ * sizeof(tredsw_call), cudaMemcpyDeviceToHost, ctx->stream));
        if (read_out && nr > 0)
            CUDA_TRY(cudaMemcpyAsync(read_out, d_read_out, (size_t)nr * 8 * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
        if (hist) CUDA_TRY(cudaMemcpyAsync(hist, cd.hist, sz_hist, cudaMemcpyDeviceToHost, ctx->stream));
    }
    ctx->mark(9);
    if (stats || !dev) {
        CUDA_TRY(cudaMemcpyAsync(h_cnt, cd.counters, 8 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
        if (stats) CUDA_TRY(cudaMemcpyAsync(h_st, d_stats, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
        CUDA_TRY(cudaMemcpyAsync(h_tab, d_tab_flag, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
        CUDA_TRY(cudaStreamSynchronize(ctx->stream));
        if (!dev) memcpy(calls, hout, (size_t)np_ * sizeof(tredsw_call));
        if (!dev && post) {
            *n_post = (int64_t)h_cnt[3];
            const size_t n = (size_t)(h_cnt[3] < (unsigned long long)post_cap ? h_cnt[3] : (unsigned long long)post_cap);
            if (n) {
                CUDA_TRY(cudaMemcpyAsync(post, d_post, n * sizeof(tredsw_posterior), cudaMemcpyDeviceToHost, ctx->stream));
                CUDA_TRY(cudaStreamSynchronize(ctx->stream));
            }
        }
        if (stats) {
            for (int i = 0; i < 4; ++i) stats[i] = (int64_t)h_st[i];
            stats[4] = (int64_t)h_cnt[2]; stats[5] = (int64_t)h_cnt[1]; stats[6] = (int64_t)h_cnt[0]; stats[7] = 0;
        }
        if (h_cnt[1]) {
            // the surface arena was too small for this batch: grow it for the next call and report
            ctx->d_surface.ensure((size_t)(h_cnt[0] + h_cnt[0] / 4) * sizeof(double));
            tredsw_set_error("likelihood surface arena overflow (%llu points needed); call again", h_cnt[0]);
            return TREDSW_ERR_UNSUPPORTED;
        }
        if (h_tab[1]) {
            // likewise the table / reduction-scratch arena of the large surfaces (grid.cu)
            ctx->d_ftab.ensure(ctx->d_ftab.cap + (size_t)(h_tab[0] + h_tab[0] / 4) * sizeof(double));
            tredsw_set_error("likelihood table arena overflow (%llu doubles needed); call again", h_tab[0]);
            return TREDSW_ERR_UNSUPPORTED;
        }
    }
    return TREDSW_OK;
}
