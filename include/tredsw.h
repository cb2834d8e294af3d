/*
 * tredsw.h — C ABI of libtredsw.so, the sm_100a CUDA replacement for tredparse's native layer.
 *
 * Two groups of entry points:
 *
 *  (A) the six symbols of the reference's libssw.so, with identical signatures and the identical
 *      s_align layout, so that the reference's own ctypes binding (src/ssw_wrap.py:69-83,274-280)
 *      binds to this library unmodified;
 *  (B) the batched entry points the hot path actually uses (one call = all reads x all templates of
 *      many (sample, locus) problems; one call = many likelihood grids).
 *
 * All pointers are plain C pointers.  Unless TREDSW_DEVICE_PTRS is set in `flags` they are HOST
 * pointers and the call performs its own host<->device copies on the context's stream and returns
 * after the results are in the output buffers.  With TREDSW_DEVICE_PTRS every buffer pointer is a
 * device pointer on the context's device, nothing is copied and the call only enqueues work on the
 * stream (the caller synchronises).  No entry point prints or exits; errors are returned as negative
 * codes and described by tredsw_last_error().  There is no CPU fallback: without a usable CUDA
 * device every compute entry point fails with TREDSW_ERR_CUDA.
 *
 * Citations are into the reference tree (/root/reference at build time).
 */
#ifndef TREDSW_H
#define TREDSW_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------------------------------------
 * (A) libssw.so drop-in — replaces src/ssw.c behind src/ssw.h:72-182
 * ---------------------------------------------------------------------------------------------- */
struct _profile;
typedef struct _profile s_profile;

/* src/ssw.h:42-52 (== CAlignRes, src/ssw_wrap.py:43-51); 40 bytes on LP64 */
typedef struct {
    uint16_t score1;
    uint16_t score2;
    int32_t ref_begin1;
    int32_t ref_end1;
    int32_t read_begin1;
    int32_t read_end1;
    int32_t ref_end2;
    uint32_t *cigar;
    int32_t cigarLen;
} s_align;

/* src/ssw.h:72 / src/ssw.c:751-772.  `read` and `mat` are borrowed (must outlive the profile).
 * Only n <= 5 (nucleotide matrices) is supported; otherwise NULL. */
s_profile *ssw_init(const int8_t *read, const int32_t readLen, const int8_t *mat, const int32_t n,
                    const int8_t score_size);
/* src/ssw.h:77 / src/ssw.c:774-778 */
void init_destroy(s_profile *p);
/* src/ssw.h:112-120 / src/ssw.c:780-871.  One GPU launch per call — the compatibility path, not the
 * fast one.  Returns NULL on error (never exits, never prints). */
s_align *ssw_align(const s_profile *prof, const int8_t *ref, int32_t refLen, const uint8_t weight_gapO,
                   const uint8_t weight_gapE, const uint8_t flag, const uint16_t filters,
                   const int32_t filterd, const int32_t maskLen);
/* src/ssw.h:125 / src/ssw.c:873-876 */
void align_destroy(s_align *a);
/* src/ssw.h:176,182 / src/ssw.c:878-904 */
char cigar_int_to_op(uint32_t cigar_int);
uint32_t cigar_int_to_len(uint32_t cigar_int);

/* ------------------------------------------------------------------------------------------------
 * (B) batched API
 * ---------------------------------------------------------------------------------------------- */
#define TREDSW_OK 0
#define TREDSW_ERR_CUDA (-1)     /* CUDA runtime / driver error, or no device */
#define TREDSW_ERR_ARG (-2)      /* invalid argument */
#define TREDSW_ERR_UNSUPPORTED (-3)
#define TREDSW_ERR_IO (-4)       /* BAM ingest: truncated / corrupt file, read error (never partial evidence) */

#define TREDSW_DEVICE_PTRS 1u    /* all buffer arguments are device pointers; enqueue only */
#define TREDSW_DEVICE_INPUTS 64u /* tredsw_genotype_batch[_ex]: rbuf, roff, read_problem and pe_lens are device pointers
                                    (e.g. a tredsw_ingest_view); `problems`, `read_name` and all outputs are host
                                    buffers; tredsw_cohort.n_bases is required; returns with the outputs valid */
#define TREDSW_SCORE2 2u         /* also produce score2 / ref_end2 exactly like ssw.c (ghost rows) */
#define TREDSW_NO_BEGIN 4u       /* skip the reverse pass (ref_begin/query_begin = -1), flag==0 of ssw_align */
#define TREDSW_CIGAR 8u          /* also produce CIGARs (banded_sw restatement) */
#define TREDSW_FORCE_WORD 16u    /* behave like ssw_init(score_size=1): 16-bit kernel conventions only */
#define TREDSW_GRID_NO_SURFACE 32u /* tredsw_likelihood_grid with device pointers: `surface` is scratch only */

typedef struct tredsw_ctx tredsw_ctx;

int tredsw_version(void);
int tredsw_device_count(void);
const char *tredsw_last_error(void);            /* thread-local, never NULL */

/* One context per (host thread, GPU).  stream == NULL: the context creates its own non-blocking
 * stream; otherwise `stream` is a cudaStream_t the caller owns (e.g. torch's current stream). */
tredsw_ctx *tredsw_create(int device, void *stream);
void tredsw_destroy(tredsw_ctx *ctx);
int tredsw_synchronize(tredsw_ctx *ctx);
int tredsw_sm_count(tredsw_ctx *ctx);
/* Kernels launched through this context so far (bench.py's gpu_launches claim). */
int64_t tredsw_launch_count(tredsw_ctx *ctx);
/* Main strips of the packed family kernel skipped at the fixed point of their boundary column (DESIGN.md §4.1),
 * summed over every call on this context so far; synchronises the stream.  out (TREDSW_STRIP_SKIP_STATS x int64):
 * [0] skipped phase-1 cell updates (stats[1] of tredsw_classify_reads counts them as planned), then for each loop
 * instantiation period p = 1..12 at [1 + 4 (p - 1)]: main strips planned, main strips skipped, warp items, items
 * that skipped nothing; then at [49 + 3 (p - 1)], summed over the lanes that hold a read: main strips planned, main
 * strips their warp skipped, and main strips the lane could skip on its own (from the first strip that leaves the
 * lane's own column unchanged: the bound that no grouping of reads into items can beat).  TREDSW_NO_STRIP_SKIP set
 * in the environment turns the skipping off (read on every call). */
#define TREDSW_STRIP_SKIP_STATS 85
int tredsw_strip_skip_stats(tredsw_ctx *ctx, int64_t *out);
/* Stage timing with CUDA events on the context's stream: enable, run calls, then read the device time
 * of the LAST call's stages in ms: [0] Smith-Waterman classify kernels, [1] likelihood grid (surface +
 * reduce), [2] KDE, [3] whole call.  Reading synchronises the stream. */
int tredsw_enable_timing(tredsw_ctx *ctx, int on);
int tredsw_get_timing(tredsw_ctx *ctx, float *ms4);
/* Device timestamps of the last timed call on this context, in ms since a process-wide reference event (the first
 * call of this function records it): [0/1] SW start/end, [2/3] grid, [4/5] KDE, [6] inputs on the device,
 * [7] calls final, [8] call start, [9] results copied; -1 where a mark was not recorded.  Lets a caller line up
 * the calls of several contexts that share one GPU (tools/e2e_probe.py). */
int tredsw_get_timeline(tredsw_ctx *ctx, float *ms10);
/* Measured integer-pipe peak of this GPU: a register-resident VIADDMNMX.S16x2 loop with 8 independent
 * chains per thread on every SM; returns giga lane-instructions per second (one 32-bit lane executing
 * one packed DPX instruction = 1).  The roofline denominator of the Smith-Waterman kernel. */
int tredsw_int_pipe_peak(tredsw_ctx *ctx, double *giga_lane_instr_per_s);

/* Tags of a classified read (tredparse/bam_parser.py:157-168). */
enum { TREDSW_TAG_NONE = 0, TREDSW_TAG_FULL = 1, TREDSW_TAG_PREF = 2, TREDSW_TAG_POST = 3,
       TREDSW_TAG_REPT = 4, TREDSW_TAG_HANG = 5,
       TREDSW_TAG_REPT_PAIR = 6 /* tredsw_genotype_batch + norepeatpairs: a read removed with its REPT pair */ };

/* Generic batch of independent (query, template) alignments == a batch of
 * ssw_init -> ssw_align(flag=1) -> destroy calls (src/ssw_wrap.py:186-224).
 * Sequences are int8 codes 0..4 (A,C,G,T,N) in flat buffers with offset arrays (nq+1 / nt+1 entries).
 * mat25 is the 5x5 substitution matrix of src/ssw_wrap.py:154-167 (row = template code, col = query
 * code).  out: npairs x 8 int32 = score, ref_begin, ref_end, query_begin, query_end, score2,
 * ref_end2, cigar_len.  cigar_out (TREDSW_CIGAR): npairs x cigar_cap uint32 words (len<<4|op). */
int tredsw_align_pairs(tredsw_ctx *ctx, const int8_t *qbuf, const int64_t *qoff, int32_t nq,
                       const int8_t *tbuf, const int64_t *toff, int32_t nt, const int32_t *qidx,
                       const int32_t *tidx, int64_t npairs, const int8_t *mat25, int gap_open,
                       int gap_extend, uint32_t flags, int32_t *out, uint32_t *cigar_out,
                       int32_t cigar_cap);

/* A locus' template family (tredparse/bam_parser.py:84-100): templates prefix + repeat*u + suffix and
 * their reverse complements for u = 1..max_units. */
typedef struct {
    int8_t prefix[32];          /* codes; prefix_len <= 32 */
    int8_t suffix[32];
    int8_t repeat[32];          /* period <= 32 */
    int32_t prefix_len;
    int32_t suffix_len;
    int32_t period;
    int32_t max_units;          /* ceil(READLEN / period) (bam_parser.py:73) */
    int32_t clip;               /* bam_parser.py:154-155: per-read max_units when clipped reads are used */
    int32_t reserved[3];
} tredsw_family;

/* The production path: every read against every template of its family, post-filter, classification
 * and per-read arg-max fused (== BamParser._parseReadSW for a whole batch; bam_parser.py:123-182,
 * src/ssw_wrap.py:213-220).  Reads are int8 codes, grouped by problem: read r belongs to family
 * read_family[r].
 * out: nreads x 8 int32 = tag, h (units), score, ref_begin, ref_end, query_begin, query_end, rank
 * (rank = DB index of the winning template: 2*(units-1) + strand; -1 when tag == NONE).
 * stats (optional, 4 x int64): [0] algorithmic forward cells (sum len(read)*len(template)),
 * [1] executed forward cell updates, [2] executed second-phase cell updates, [3] alignments. */
int tredsw_classify_reads(tredsw_ctx *ctx, const int8_t *rbuf, const int64_t *roff, int32_t nreads,
                          const int32_t *read_family, const tredsw_family *families, int32_t nfamilies,
                          const int8_t *mat25, int gap_open, int gap_extend, uint32_t flags,
                          int32_t *out, int64_t *stats);

/* One likelihood problem (tredparse/models.py:223-302 + 394-415); see SURVEY.md Appendix B. */
typedef struct {
    int32_t period;             /* K */
    int32_t readlen;            /* L */
    int32_t ploidy;
    int32_t n_rept;             /* U */
    int32_t max_partial;        /* mp (already raised to the largest partial key, models.py:241-242) */
    int32_t run_pe;
    int32_t pe_ref;             /* ref = repeat_end - repeat_start + 1 */
    int32_t pe_minpe;
    int32_t n_span;             /* K_s observed spanning keys */
    int32_t n_part;             /* K_p observed partial keys */
    int32_t n_target;           /* n_t target pair lengths */
    int32_t n_h1;               /* candidate lists (bp), in reference order, duplicates kept (Q9) */
    int32_t n_h2;
    int32_t expansion;          /* PP rule: models.py:351-364 */
    int32_t recessive;
    int32_t cutoff_risk;
    double half_depth;          /* D */
    double stutter_a;           /* w0 + w1*K            logistic stutter model, models.py:79-84,156:  */
    double stutter_w2;          /* w2                   z = ((a + w2*(h // K)) + c3) + c4,             */
    double stutter_c3;          /* w3 * gc              sigma = 1 / (1 + exp(-z))                      */
    double stutter_c4;          /* w4 * score */
    /* offsets into the shared arrays below */
    int64_t off_span;           /* ipool: n_span keys (bp) followed by n_span counts */
    int64_t off_part;           /* ipool: n_part keys (bp) followed by n_part counts */
    int64_t off_target;
    int64_t off_h1;
    int64_t off_h2;
    int64_t off_pdf;            /* 1000 doubles (normalised KDE), -1 when no PE model */
    int64_t off_step;           /* 37 doubles: step PMF of this period */
    int64_t off_surface;        /* n_h1*n_h2 doubles in `surface` (row-major, -inf where h1 > h2) */
    int64_t off_ph1;            /* n_h1 doubles in `marg` */
    int64_t off_ph2;            /* n_h2 doubles in `marg` */
} tredsw_grid_problem;

/* Per-problem reductions. */
typedef struct {
    double max_ml;              /* lik of the call */
    double sum_all;             /* sum exp(ml - max_ml) over evaluated points (duplicates counted, Q9) */
    double sum_path;            /* same over pathological points */
    int32_t arg_i1;             /* indices into the h1/h2 candidate lists of the call (Q10) */
    int32_t arg_i2;
    int32_t n_points;           /* -1: the table arena was too small for this surface (call again) */
    int32_t pad;
    double sum_uniq;            /* sum_all without the second occurrences of duplicated candidates (Q9) = the
                                   total of the joint posterior dict P_h1h2 (models.py:285,304-317) */
} tredsw_grid_result;

/* One entry of a sparsified posterior (models.py:304-317: entries below e^-10 are dropped, the rest divided
 * by the full total).  a / b are alleles in repeat units.  JOINT entries carry the un-normalised weight
 * exp(ml - max ml); the JOINT_TOTAL entry of the same problem carries their divisor. */
typedef struct {
    int32_t problem;
    int32_t kind;               /* TREDSW_POST_* */
    int32_t a, b;               /* P_h1: a = h1; P_h2: a = h2; joint: (a, b) = (h1, h2) */
    double p;
} tredsw_posterior;
enum { TREDSW_POST_H1 = 1, TREDSW_POST_H2 = 2, TREDSW_POST_JOINT = 3, TREDSW_POST_JOINT_TOTAL = 4 };

/* Evaluate the log-likelihood surface of `nproblems` problems and reduce it.
 * ipool: int32 pool holding, per problem, the observed spanning / partial keys and counts, the target
 * pair lengths (already wrapped into 0..999 like a numpy index) and the h1 / h2 candidate lists;
 * dpool: double pool holding the KDE pdfs (1000 each) and step PMFs (37 each);
 * surface / marg: output pools.  The reductions do not need the surface: it is materialised (every point,
 * -inf where h1 > h2) only when asked for — host mode: `surface` non-NULL; device mode: unless
 * TREDSW_GRID_NO_SURFACE (the buffer is then scratch for the near-allele part of large surfaces).
 * For ploidy 1 the caller passes n_h2 = 1 and the kernel evaluates h2 = h1 (models.py:261). */
int tredsw_likelihood_grid(tredsw_ctx *ctx, const tredsw_grid_problem *problems, int32_t nproblems,
                           const int32_t *ipool, int64_t n_ipool, const double *dpool, int64_t n_dpool,
                           double *surface, int64_t n_surface, double *marg, int64_t n_marg,
                           tredsw_grid_result *results, uint32_t flags);

/* Gaussian KDE of paired-end lengths on the grid 0..999, normalised to sum 1
 * (tredparse/models.py:428-435: scipy gaussian_kde with Scott's factor, pdf / pdf.sum()).
 * lens: int32 pool, off: nproblems+1 offsets; pdf_out: nproblems x 1000 doubles. */
int tredsw_pe_kde(tredsw_ctx *ctx, const int32_t *lens, const int64_t *off, int32_t nproblems,
                  double *pdf_out, uint32_t flags);


/* ------------------------------------------------------------------------------------------------
 * Whole (sample, locus) problems in one call: reads -> Smith-Waterman + classification -> tallies ->
 * candidate ranges -> KDE -> likelihood grid -> call / CI / PP / label, everything on the device.
 * == the body of tred.run's per-locus loop (tredparse/tred.py:225-275) for a whole cohort shard,
 * minus BAM I/O.  --useclippedreads: set tredsw_family.clip (per-read max_units, bam_parser.py:154-155);
 * --norepeatpairs: set tredsw_cohort.norepeatpairs and pass read_name (bam_parser.py:248-249,270-287).
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
    int32_t family;             /* index into families / loci */
    int32_t ploidy;             /* 1 or 2 (bam_parser.py:58-61) */
    int32_t n_global;           /* global pair lengths (KDE input) */
    int32_t n_target;           /* spanning pair lengths */
    int64_t off_global;         /* offsets into pe_lens */
    int64_t off_target;
    double depth;               /* mean depth of the locus window */
} tredsw_problem;

typedef struct {                /* model-side constants of a locus (meta.py:103-129, models.py:114-118) */
    int32_t period;
    int32_t readlen;
    int32_t pe_ref;             /* repeat_end - repeat_start + 1 */
    int32_t pe_minpe;           /* bam_parser.py:361 */
    int32_t expansion;
    int32_t recessive;
    int32_t cutoff_prerisk;
    int32_t cutoff_risk;
} tredsw_locus;

typedef struct {
    const int8_t *rbuf;         /* read codes, flat */
    const int64_t *roff;        /* nreads + 1 */
    const int32_t *read_problem;/* nreads: owning problem of each read */
    const tredsw_problem *problems;
    const int32_t *pe_lens;     /* pooled pair lengths */
    int64_t n_pe_lens;
    int32_t nreads;
    int32_t nproblems;
    int32_t max_read_len;       /* upper bound on read length (required; checked against roff for host buffers —
                                   with TREDSW_DEVICE_PTRS a longer read is skipped: it gets the "no tag" record) */
    int32_t nfamilies;
    /* the following three are always HOST pointers (small, shape decisions are made on the host) */
    const tredsw_family *families;
    const tredsw_locus *loci;
    const double *step_pmf;     /* nfamilies x 37 */
    double stutter_w[5];        /* logistic weights, models.py:79-84 */
    double gc, score;           /* models.py:106 */
    int32_t maxinsert;
    int32_t fullsearch;
    int8_t mat25[25];
    int8_t pad_[3];
    int32_t gap_open, gap_extend;
    uint32_t input_flags;       /* TREDSW_IN_* below: compact transfer formats, expanded on the device */
    int32_t norepeatpairs;      /* 1: drop every read whose name occurs on more than one REPT read of its problem
                                   (remove_pairs_of_rept, bam_parser.py:270-287; ignored for clip families, :248) */
    int64_t n_bases;            /* total bases in rbuf (= roff[nreads]); required with TREDSW_DEVICE_PTRS + PACKED4 */
    const int32_t *read_name;   /* nreads name ids (equal id within a problem = same query name); needed only
                                   with norepeatpairs, may be NULL otherwise */
} tredsw_cohort;

/* tredsw_cohort.input_flags — halve the host->device bytes of a call; the buffers are expanded into the
 * regular layouts by two small kernels right after the copy (everything downstream is unchanged): */
#define TREDSW_IN_READS_PACKED4 1u   /* rbuf holds two base codes per byte: base i in bits 4*(i&1).. of byte i>>1 */
#define TREDSW_IN_PE_LENS_I16 2u     /* pe_lens points to int16_t values (pair lengths kept are < 1000) */

/* The transfer formats on the host side: base codes (one per byte) -> TREDSW_IN_READS_PACKED4, int32 lengths ->
 * TREDSW_IN_PE_LENS_I16.  `out` holds (n + 1) / 2 bytes / n values; `threads` host threads share the packing. */
int tredsw_pack_reads4(const int8_t *codes, int64_t n, uint8_t *out, int threads);
int tredsw_narrow_i16(const int32_t *in, int64_t n, int16_t *out, int threads);

typedef struct {
    int32_t allele1, allele2;   /* units, sorted; -1/-1 when there is no evidence */
    int32_t ci[4];              /* h1_lo, h1_hi, h2_lo, h2_hi (units); -1 when missing */
    int32_t label;              /* 0 ok, 1 prerisk, 2 risk, 3 missing */
    int32_t n_points;
    int32_t fdp, pdp, rdp;      /* FULL / PREF(+POST) / REPT read counts */
    int32_t run_pe;
    double pp;                  /* -1 when missing */
    double lik;
} tredsw_call;

/* buffers in `c`, `calls`, `read_out` (optional, nreads x 8 like tredsw_classify_reads) and `hist`
 * (optional, nproblems x 3 x (hist_units+1) int32: FULL, PREF, REPT histograms by units) are host or
 * device pointers according to `flags`.  stats (optional, host, 8 x int64): [0..3] as in
 * tredsw_classify_reads, [4] grid points evaluated, [5] surface arena overflow (0 = ok). */
int tredsw_genotype_batch(tredsw_ctx *ctx, const tredsw_cohort *c, uint32_t flags, tredsw_call *calls,
                          int32_t *read_out, int32_t *hist, int32_t hist_units, int64_t *stats);

/* The same, also returning the sparsified posteriors P_h1 / P_h2 / P_h1h2 the reference writes into its JSON
 * (models.py:292-294,304-317) as one flat list of entries in no particular order.  `post` (host or device
 * according to `flags`) holds post_cap entries; *n_post (same memory space, 64-bit) receives the number of
 * entries produced — when it exceeds post_cap the list is truncated and the call should be repeated with a
 * larger buffer. */
int tredsw_genotype_batch_ex(tredsw_ctx *ctx, const tredsw_cohort *c, uint32_t flags, tredsw_call *calls,
                             int32_t *read_out, int32_t *hist, int32_t hist_units, int64_t *stats,
                             tredsw_posterior *post, int64_t post_cap, int64_t *n_post);

/* ------------------------------------------------------------------------------------------------
 * (C) native BAM ingest (host code, zlib) — replaces the three pysam passes per locus of the reference:
 * read selection (tredparse/bam_parser.py:194-243), PEextractor (:316-369) and BamDepth.region_depth
 * (:404-411) with one indexed pass that writes base codes, pair distances and depth into caller-owned
 * (e.g. pinned) buffers in the layout tredsw_genotype_batch consumes.
 * ---------------------------------------------------------------------------------------------- */
typedef struct tredsw_bam tredsw_bam;

typedef struct {
    int32_t tid;                /* contig of the locus (tredsw_bam_tid) */
    int32_t repeat_start, repeat_end;
    int32_t readlen;            /* READLEN: mapped reads must start within +-READLEN of the repeat */
    int32_t pad;                /* parse / depth window: +-pad around the repeat (SPAN = 1000) */
    int32_t pe_window;          /* pair window: +-pe_window (DNAPE_ELONGATE = 10000) */
    int32_t flankmatch;         /* FLANKMATCH = 9: a pair is "target" if it spans the repeat by more than this */
    int32_t span;               /* pairs with distance >= span are dropped (SPAN = 1000) */
    int32_t n_alts;             /* alternative (mis-mapping) regions: reads there whose mate lies in the window */
    int32_t reserved_;
    const int32_t *alts;        /* n_alts x (tid, start, end) */
} tredsw_locus_query;

typedef struct {
    int32_t nreads;             /* reads selected (also counted when a buffer overflowed) */
    int32_t n_unmapped;
    int32_t n_global, n_target; /* pair distances written to global_lens / target_lens */
    int64_t nbases;             /* roff[nreads] */
    int64_t name_bytes;         /* NUL-separated read names written to `names` */
    double depth;               /* mean pileup depth of the +-pad window */
    int32_t overflow;           /* 1: some buffer was too small; counts above tell the sizes needed */
    int32_t reserved_;
} tredsw_locus_summary;

/* bai_path NULL: <bam>.bai, then <bam without extension>.bai.  NULL + tredsw_last_error() on failure. */
tredsw_bam *tredsw_bam_open(const char *bam_path, const char *bai_path);
/* A second, independent handle on the same BAM for another host thread (handles are not thread-safe): own file
 * descriptor and inflate state, the parsed index shared with `bam`.  Close each clone with tredsw_bam_close. */
tredsw_bam *tredsw_bam_clone(tredsw_bam *bam);
void tredsw_bam_close(tredsw_bam *bam);
int32_t tredsw_bam_nref(tredsw_bam *bam);
/* contig `tid` of the binary reference dictionary: its length (-1: no such contig); its name, NUL-terminated and cut to
 * cap - 1 bytes, into name when name is not NULL */
int64_t tredsw_bam_ref(tredsw_bam *bam, int32_t tid, char *name, int64_t cap);
int32_t tredsw_bam_tid(tredsw_bam *bam, const char *contig);     /* -1 when unknown */
/* signature of the reference dictionary (names + lengths, in order): equal signatures = equal contig numbering */
uint64_t tredsw_bam_header_signature(tredsw_bam *bam);
/* names may be NULL (not wanted).  Reads are written in the reference's order: window reads in file
 * order, then the alt-region reads. */
int tredsw_bam_extract_locus(tredsw_bam *bam, const tredsw_locus_query *q, int8_t *rbuf, int64_t rbuf_cap,
                             int64_t *roff, int32_t reads_cap, int32_t *global_lens, int32_t global_cap,
                             int32_t *target_lens, int32_t target_cap, char *names, int64_t names_cap,
                             tredsw_locus_summary *out);

/* BGZF blocks inflated so far by the library's own DEFLATE decoder (csrc/inflate_fast.h, every block CRC-checked)
 * and by zlib (the fallback for streams the decoder refuses). */
void tredsw_bam_inflate_stats(tredsw_bam *bam, int64_t *own_blocks, int64_t *zlib_blocks);
/* The decoder on its own (test hook): 0 iff the raw DEFLATE stream `in` inflates to exactly out_len bytes. */
int tredsw_inflate_raw(const uint8_t *in, int64_t in_len, uint8_t *out, int64_t out_len);
/* BamDepth.region_depth (tredparse/bam_parser.py:404-411): sum of pileup column depths over the reads
 * overlapping [start, end) / (end - start + 1); feeds half_depth of the repeat-only term and the chrY depth of
 * the gender inference (bam_parser.py:413-429). */
int tredsw_bam_region_depth(tredsw_bam *bam, int32_t tid, int64_t start, int64_t end, double *depth);
/* BamReadLen.readlen (tredparse/bam_parser.py:372-391): longest (and optionally shortest) query among the
 * first first_n + 1 records of the file. */
int tredsw_bam_read_length(tredsw_bam *bam, int32_t first_n, int32_t *max_out, int32_t *min_out);

/* ------------------------------------------------------------------------------------------------
 * (D) BAM ingest on the GPU for a whole batch of (sample, locus) problems (csrc/bgzf_gpu.cu): the host reads only
 * the COMPRESSED BGZF blocks behind the BAI chunks of the requested windows; raw-DEFLATE decoding (one thread per
 * block, CRC-32 checked), the record walk, read selection (tredparse/bam_parser.py:194-243), PEextractor
 * (:316-369, pairing by query name) and the pileup depth (:404-411) run on the device and leave rbuf / roff /
 * read_problem / pe_lens in device memory in the layout of tredsw_cohort (TREDSW_DEVICE_PTRS) — same reads,
 * order, pair lists and depth as tredsw_bam_extract_locus query by query.
 * ---------------------------------------------------------------------------------------------- */
typedef struct tredsw_ingest_batch tredsw_ingest_batch;

#define TREDSW_INGEST_NO_NAMES 1u    /* do not collect read names */
#define TREDSW_INGEST_NO_CRC 2u      /* skip the CRC-32 check of the inflated blocks */

typedef struct {                /* where problem p's share of the flat buffers starts */
    int64_t read0, base0, name0;
    int64_t off_global, off_target;   /* into pe_lens: n_global values, then n_target values */
} tredsw_problem_span;

typedef struct {
    int32_t nproblems, nreads;
    int64_t nbases, name_bytes, n_pe_lens;
    /* device memory, valid until tredsw_ingest_batch_free */
    const int8_t *d_rbuf; const int64_t *d_roff; const int32_t *d_read_problem; const int32_t *d_pe_lens;
    /* page-locked host copies of the same */
    const int8_t *h_rbuf; const int64_t *h_roff; const int32_t *h_pe_lens; const char *h_names;
    const tredsw_locus_summary *summaries;   /* per problem: counts and depth as tredsw_bam_extract_locus reports them */
    const tredsw_problem_span *spans;
    const int32_t *status;      /* per problem: 0 ok; 1 its sample could not be staged (I/O, index, BGZF framing), 2 a block
                                   failed to inflate or its CRC-32 differs, 3 corrupt records, 4 (scan only) the file is not
                                   sorted by coordinate — no evidence is reported for such a problem: read it with
                                   tredsw_bam_extract_locus (which has zlib behind it) or the Python reader */
    int64_t n_blocks, n_records, comp_bytes, inflated_bytes;
    double ms_host_stage, ms_total;   /* host time: compressed bytes staged; whole call */
    double ms_marks[4];         /* host time at the four synchronisation points: blocks inflated + records counted,
                                   records selected, pairs formed, results copied */
} tredsw_ingest_view;

/* queries[i] belongs to bams[sample_of[i]]; problems are numbered like the queries.  The handles are only read
 * (index, file descriptor with pread): one handle may serve several batches, but not from two threads at once. */
int tredsw_ingest_batch_run(tredsw_ctx *ctx, tredsw_bam *const *bams, const int32_t *sample_of,
                            const tredsw_locus_query *queries, int32_t nqueries, uint32_t flags,
                            tredsw_ingest_batch **out);
int tredsw_ingest_batch_view(const tredsw_ingest_batch *batch, tredsw_ingest_view *view);
void tredsw_ingest_batch_free(tredsw_ingest_batch *batch);
/* TEST INFRASTRUCTURE: the same pipeline with every kernel body executed serially on the host (the bodies are
 * __host__ __device__, csrc/ingest_device.cuh), so that the CPU test-suite can compare the device logic with the
 * host reader bit for bit.  The d_* pointers of its view are host pointers.  The package never calls it. */
int tredsw_ingest_batch_emulate(tredsw_bam *const *bams, const int32_t *sample_of, const tredsw_locus_query *queries,
                                int32_t nqueries, uint32_t flags, tredsw_ingest_batch **out);
int tredsw_inflate_raw_device_code(const uint8_t *in, int64_t in_len, uint8_t *out, int64_t out_len);

/* BAMs without an index.  tredsw_bam_open_unindexed reads the header and leaves the BGZF stream open without looking
 * for an index: tredsw_bam_tid, tredsw_bam_header_signature, tredsw_bam_read_length and tredsw_bam_clone work on the
 * handle; tredsw_bam_extract_locus, tredsw_bam_region_depth and tredsw_ingest_batch_run refuse it with
 * TREDSW_ERR_UNSUPPORTED.  NULL + tredsw_last_error() on failure. */
tredsw_bam *tredsw_bam_open_unindexed(const char *bam_path);
/* One sample in ONE streaming pass over the whole file (csrc/bgzf_gpu.cu, run_scan): the host reads the file after
 * the header slab by slab (slab_bytes compressed bytes a step, 0 = 128 MiB; at least 64 KiB), the device inflates
 * every block, finds the record boundaries without an index (a candidate per block, verified by chaining from the
 * known first record), keeps the records that overlap a fetch of `queries` (locus windows and alt regions) and sums
 * the depth of `depth_regions` (n_depth x (tid, start, end); depth_out[d] = what tredsw_bam_region_depth returns for
 * region d, NaN when the scan failed).  On a stream handle the slabs are read in order with read() (a slab of slab_bytes
 * is not capped by a size) and the end of the input is read() returning 0.  The result is an ordinary batch (tredsw_ingest_batch_view / _free), with the
 * same evidence as tredsw_ingest_batch_run on an indexed copy, problem by problem.  Its status is per scan: every
 * problem gets 1 (I/O, BGZF framing), 2 (a block failed to inflate), 3 (corrupt or truncated records) or 4 (the file is
 * not sorted by coordinate: tid non-decreasing with -1 last, pos non-decreasing within a tid). */
/* A BAM read strictly in order with read(): a pipe, a FIFO, a socket, or stdin when bam_path is "-" (a regular file works
 * too, read the same way).  No seek, no size.  The handle parses the header from the bytes it has read and keeps every
 * byte from the block of the first record on; tredsw_bam_read_length reads the first records ahead and answers from
 * them.  tredsw_bam_tid, tredsw_bam_header_signature and tredsw_bam_header_text work on it; tredsw_bam_clone,
 * tredsw_bam_extract_locus, tredsw_bam_region_depth and tredsw_ingest_batch_run refuse it (TREDSW_ERR_UNSUPPORTED).  The
 * stream can be scanned ONCE (tredsw_ingest_scan_run / _emulate): a second scan, or a read length after the scan, is
 * TREDSW_ERR_ARG.  NULL + tredsw_last_error() on failure. */
tredsw_bam *tredsw_bam_open_stream(const char *bam_path);
/* The SAM header text of any handle: copies at most cap - 1 bytes and a NUL into buf (buf may be NULL); returns the
 * length of the whole text. */
int64_t tredsw_bam_header_text(tredsw_bam *bam, char *buf, int64_t cap);
int tredsw_ingest_scan_run(tredsw_ctx *ctx, tredsw_bam *bam, const tredsw_locus_query *queries, int32_t nqueries,
                           const int32_t *depth_regions, int32_t n_depth, double *depth_out, int64_t slab_bytes,
                           uint32_t flags, tredsw_ingest_batch **out);
/* TEST INFRASTRUCTURE: the same with every kernel body run serially on the host.  The package never calls it. */
int tredsw_ingest_scan_emulate(tredsw_bam *bam, const tredsw_locus_query *queries, int32_t nqueries,
                               const int32_t *depth_regions, int32_t n_depth, double *depth_out, int64_t slab_bytes,
                               uint32_t flags, tredsw_ingest_batch **out);
/* Statistics of a scan (zeros for a batch of tredsw_ingest_batch_run), TREDSW_SCAN_NSTATS values: [0] slabs, [1] BGZF
 * blocks, [2] records scanned, [3] blocks whose candidate record start was wrong and that were walked again, [4]
 * compressed bytes, [5] inflated bytes, [6] host time reading and framing the slabs (us, summed over slabs; the read of
 * slab k + 1 overlaps the device work on slab k), [7] time of the device work on the slabs (us, summed), [8] whole call
 * (us), [9] status of the scan (the per-problem code above; 0 ok). */
#define TREDSW_SCAN_NSTATS 10
int tredsw_ingest_scan_stats(const tredsw_ingest_batch *batch, int64_t *stats);

/* The STR profile of a scan: in-repeat reads (IRRs), found in the same streaming pass (DESIGN §4.5).  Records
 * considered are the primary ones (flags 0x100, 0x200, 0x400, 0x800 unset), mapped or not, with l_seq >= min_read_len.
 * A read s of length L is an IRR of period k when, of the L - k positions i with s[i] == s[i + k] (N never equal), at
 * least purity_num / purity_den agree (m * den >= num * (L - k)); its period is the smallest such k in
 * [min_period, max_period].  Its motif: the majority base of every phase (ties: the smallest of A < C < G < T; an
 * all-N phase: A), reduced to its primitive root (a root of one base is a homopolymer: not an IRR), in canonical
 * form (the smallest rotation of the root and of its reverse complement), 2 bits a base, first base most significant.
 * Valid parameters: 2 <= min_period <= max_period <= 20, 0 < purity_num <= purity_den <= 1000, min_read_len >=
 * 2 max_period; anything else is TREDSW_ERR_ARG. */
typedef struct { int32_t min_period, max_period, purity_num, purity_den, min_read_len; } tredsw_irr_params;
typedef struct {                /* one IRR record, in file order */
    int32_t tid, pos, next_tid, next_pos;
    int32_t flag, mapq, mq, period;   /* mq: the record's MQ tag (integer types c C s S i I), -1 without one */
    uint64_t motif;             /* canonical motif, `period` bases of 2 bits */
    int64_t name_off;           /* its name: name_len bytes (no NUL) at names + name_off */
    int32_t name_len, mate;     /* mate: the entry with the same name and the other segment flag (0x40 / 0x80), -1 none */
} tredsw_irr_entry;
typedef struct {                /* host arrays, valid until tredsw_ingest_batch_free; a failed scan (status 1-4) has no
                                   entries and every counter 0 */
    int64_t n_entries;
    const tredsw_irr_entry *entries;
    const char *names; int64_t name_bytes;
    int64_t records_considered, irr_records;
    int64_t depth_bases;        /* sum of l_seq over primary, mapped, non-duplicate, non-QC-fail records */
    int64_t max_l_seq;          /* over the primary records */
    int64_t anchors_without_mq; /* IRRs that are paired (0x1), whose mate is mapped (0x8 unset, next_tid >= 0) and not
                                   an IRR, and that carry no MQ tag */
    int64_t unparsed_aux;       /* IRR records whose aux area could not be parsed (taken as without MQ) */
} tredsw_irr_view;
/* tredsw_ingest_scan_run / _emulate with an IRR profile: irr = NULL is exactly those calls; nqueries = 0 and no depth
 * regions with irr set is a profile-only scan.  The profile's kernels do not change the evidence, depths or
 * statistics of the scan. */
int tredsw_ingest_scan_run_ex(tredsw_ctx *ctx, tredsw_bam *bam, const tredsw_locus_query *queries, int32_t nqueries,
                              const int32_t *depth_regions, int32_t n_depth, double *depth_out, int64_t slab_bytes,
                              uint32_t flags, const tredsw_irr_params *irr, tredsw_ingest_batch **out);
/* TEST INFRASTRUCTURE: the same with every kernel body run serially on the host.  The package never calls it. */
int tredsw_ingest_scan_emulate_ex(tredsw_bam *bam, const tredsw_locus_query *queries, int32_t nqueries,
                                  const int32_t *depth_regions, int32_t n_depth, double *depth_out, int64_t slab_bytes,
                                  uint32_t flags, const tredsw_irr_params *irr, tredsw_ingest_batch **out);
/* The profile of a batch scanned with irr set (TREDSW_ERR_ARG otherwise). */
int tredsw_ingest_scan_irr(const tredsw_ingest_batch *batch, tredsw_irr_view *view);
/* Test hook: the classifier body on the host.  codes: 0..3 = A C G T, anything else N.  *period = 0: not an IRR. */
int tredsw_irr_classify_host(const int8_t *codes, int32_t len, const tredsw_irr_params *params, int32_t *period,
                             uint64_t *motif);

#ifdef __cplusplus
}
#endif
#endif /* TREDSW_H */
