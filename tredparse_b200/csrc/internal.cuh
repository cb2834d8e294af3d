// internal.cuh — enqueue-only building blocks shared between the public entry points (device pointers in,
// work queued on ctx->stream, no synchronisation).
#pragma once
#include "common.cuh"

// Smith-Waterman + classification of every read against its family (sw_family.cu).
// h_families: host copy (shape decisions); d_* : device buffers.  d_work needs tredsw_classify_work_words int32:
// counts and cursors per bin (family, strand class, predicted strips), offsets per (family, strand class), the read
// order.  d_stats: 4 x u64 or NULL (must be zeroed by the caller).
int tredsw_classify_bins(const tredsw_family *h_families, int nfamilies);
size_t tredsw_classify_work_words(const tredsw_family *h_families, int nfamilies, int nreads);
int tredsw_internal_classify(tredsw_ctx *ctx, const int8_t *d_rbuf, const int64_t *d_roff, int nreads,
                             const int32_t *d_read_family, const tredsw_family *d_families,
                             const tredsw_family *h_families, int nfamilies, int max_read_len,
                             const int8_t *h_mat25, int go, int ge, int32_t *d_work, int32_t *d_out,
                             unsigned long long *d_stats);

// Likelihood surface + reductions (grid.cu).  points_hint (largest surface of the batch, or an upper bound)
// sizes the table arena.  d_surface: per-problem slots (scratch; the full surface when `materialise`).
// d_post / post_cap / d_post_cursor: optional arena for the sparse joint-posterior entries.
// *d_overflow_flag receives a device pointer to {doubles needed, overflow flag} of the table arena.
int tredsw_internal_grid(tredsw_ctx *ctx, const tredsw_grid_problem *d_prob, int nproblems,
                         const int32_t *d_ipool, const double *d_dpool, double *d_surface, double *d_marg,
                         tredsw_grid_result *d_res, long long points_hint, int materialise,
                         tredsw_posterior *d_post, long long post_cap, unsigned long long *d_post_cursor,
                         unsigned long long **d_overflow_flag, int tables);
// TREDSW_GRID_TABLES -> the best table tier a large likelihood surface may take (0 full, 1 without the paired-end
// operands, 2 none); an unknown value is an argument error.  Parsed by the public entry points before they launch.
int tredsw_internal_grid_tables(int *tables);
