/* pasio_b200.h -- C ABI of the B200-native Pasio segmentation hot path.
 *
 * The reference (autosome-ru/pasio v1.1.3) is pure Python and has NO FFI of its own:
 * its boundary for this path is three duck-typed Python protocols (reducer, splitter,
 * scorer; SURVEY.md 8b).  This header is the boundary a maintainer would bind instead
 * (ctypes stub shown in INTEGRATION.md); every entry point names the reference code
 * it replaces (paths under /root/reference/src/pasio/).
 *
 * Conventions: plain C symbols, plain pointers and sizes, no torch types.  Every
 * function returns 0 on success or a negative pasio_status; pasio_last_error() gives
 * the message.  All pointers are HOST pointers unless the name says `_device`; host
 * buffers may be pageable or pinned (pinned is faster).  The caller owns every buffer.
 * A context owns one CUDA stream and is not re-entrant.  No function falls back to
 * the CPU: without a usable sm_100 device pasio_ctx_create fails.
 */
#ifndef PASIO_B200_H
#define PASIO_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct pasio_ctx pasio_ctx;

typedef enum pasio_status {
    PASIO_OK = 0,
    PASIO_E_CUDA = -1,            /* CUDA runtime error (message has the detail)            */
    PASIO_E_ARG = -2,             /* malformed argument                                     */
    PASIO_E_COUNTS = -3,          /* negative count / empty contig   -> AssertionError
                                     (log_marginal_likelyhood.py:30-34)                      */
    PASIO_E_CANDIDATES = -4,      /* candidates not 0..n strictly ascending -> AssertionError
                                     (log_marginal_likelyhood.py:36-40)                      */
    PASIO_E_TABLE_TOO_SHORT = -5, /* a look-up table is shorter than the largest argument;
                                     pasio_table_need() says how long they must be          */
    PASIO_E_STATE = -6,           /* call out of order (no contig / no tables / ...)         */
    PASIO_E_TOO_LARGE = -7,       /* contig >= 2^31-1 nt, total count >= 2^31, or window
                                     larger than one CTA's shared memory                    */
    PASIO_E_NOMEM = -8
} pasio_status;

/* Table ids for pasio_table_upload / pasio_table_need. */
enum { PASIO_TAB_LOG = 0,          /* Lg[k] = log(k + beta)      cached_log.py:9  (LogComputer)            */
       PASIO_TAB_LGAMMA = 1,       /* G[k]  = gammaln(k)         cached_log.py:36 (LogGammaComputer())     */
       PASIO_TAB_LGAMMA_ALPHA = 2  /* Ga[k] = gammaln(k + alpha) cached_log.py:36 (shift=alpha)            */ };

/* split_constraints of default_splitters.py:52-59 */
enum { PASIO_CONSTRAINT_NONE = 0, PASIO_CONSTRAINT_ZEROS = 1, PASIO_CONSTRAINT_CONSTANTS = 2 };

/* tuning switches of pasio_set_tuning (results never depend on them; they exist for A/B parity
 * tests and measurements) */
enum { PASIO_TUNE_WINDOW_PRUNE = 0,   /* 1: window DP bounds far columns (default), 0: every cell evaluated */
       PASIO_TUNE_WINDOW_PHASES = 1,  /* 1: windows whose candidates all survived already are skipped      */
       PASIO_TUNE_EXACT_PRUNE = 2,    /* 1: whole-contig exact DP bounds far columns (csrc/exact_pruned.cu) */
       PASIO_TUNE_EXACT_LAG = 3,      /* far columns start this many 128-row blocks behind the diagonal (3 .. 5, default 5) */
       PASIO_TUNE_EXACT_RING = 4,     /* 1 (default): self scores in an L2-resident ring of 64 row blocks; 0: one slab per row block
                                         while that fits 2 GB (measured slower: the slabs fall out of L2) */
       PASIO_TUNE_LOGFAC_EXACT = 5,   /* 1 (default): logfac_cumsum summed sequentially like np.cumsum (bit-identical LMM column);
                                         0: three-pass parallel scan (1e-9 relative, faster on dense coverage) */
       PASIO_TUNE_WINDOW_SPECULATE = 6, /* 1 (default): window DP first resolves a 32-row block assuming every row's arg-max is the
                                         row before it (true for nearly all rows of the later rounds), verifies, and falls
                                         back to the ordinary chain where the assumption fails */
       PASIO_TUNE_UPLOAD_NARROW = 7,  /* 1 (default): large uploads send counts packed to uint8, uint16 or int32 (whatever every count of
                                         a 4 MB slice fits): host threads pack them into page-locked slices, a kernel widens them on
                                         arrival; a slice holding a negative count or one >= 2^31 goes up as it is.  0: plain copies;
                                         k in 2..24 (tests): uint8 if the slice fits k bits, uint16 k + 3, int32 k + 6, else plain */
       PASIO_TUNE_LOGFAC_EAGER = 8,   /* 1: pasio_contig_load_round also forms the sequential log-factorial sums, chunk by chunk on a
                                         side stream behind the upload (set it when log_marginal_likelyhoods() / the LMM column
                                         will be asked for: the 30 ms sum of a chr1-sized contig is then done when the upload is).
                                         0 (default): on demand, or pasio_logfac_prefetch */
       PASIO_TUNE_EXACT_NBLOCK = 9,   /* the exact DP hands the first n column blocks in front of the far columns (blocks b - lag + 1 ..
                                         of row block b) to worker CTAs, which evaluate them exhaustively; the diagonal sweeps the
                                         remaining lag - n blocks itself.  0 .. lag - 2, default 3 (with lag 5: a band of two blocks) */
       PASIO_TUNE_WINDOW_CERTIFY = 10, /* 1 (default): in rounds after one that removed under 1 % of its candidates, window DP first
                                         checks every large window for "every candidate survives" in one parallel pass and resumes
                                         the ordinary pipeline at the first block that fails; 2: in every round; 0: never */
       PASIO_TUNE_REG_EXACT = 11,     /* whole-list DP of pasio_square_split_regularized: 1 (default): one CTA for short
                                         candidate lists, a kernel on every SM for long ones (the threshold is
                                         REG_EXACT_MIN_CANDIDATES in csrc/api.cu); 0: always one CTA; 2: always every SM */
       PASIO_TUNE_COUNT = 12 };

/* ---- context ------------------------------------------------------------------------ */
int pasio_ctx_create(int device, pasio_ctx **out);
int pasio_ctx_destroy(pasio_ctx *ctx);
const char *pasio_last_error(const pasio_ctx *ctx);   /* never NULL; ctx may be NULL */
int pasio_abi_version(void);

/* ---- scorer parameters and tables ---------------------------------------------------
 * Replaces ScorerFactory.__init__ (log_marginal_likelyhood.py:6-16) and the LogComputer /
 * LogGammaComputer tables (cached_log.py:5-56).  The VALUES are produced on the host by
 * the same numpy/scipy calls the reference makes, so they are bit-identical to what the
 * reference would look up or compute; the device only gathers from them.
 * alpha_is_int mirrors log_marginal_likelyhood.py:9-12,19.  segment_creation_cost is
 * alpha*log(beta) - gammaln(alpha) (:62) evaluated by the host. */
int pasio_set_params(pasio_ctx *ctx, int alpha_is_int, double alpha, double beta,
                     double segment_creation_cost);
int pasio_table_upload(pasio_ctx *ctx, int table_id, const double *values, int64_t n);
/* After PASIO_E_TABLE_TOO_SHORT: minimum lengths (entries) the three tables need. */
int pasio_table_need(const pasio_ctx *ctx, int64_t *n_log, int64_t *n_lgamma, int64_t *n_lgamma_alpha);

/* ---- contig(s) ----------------------------------------------------------------------
 * Replaces LogMarginalLikelyhoodComputer.__init__'s np.cumsum (log_marginal_likelyhood.py:57)
 * and the change-point test of NotConstantReducer (constants_reducer.py:16-17), done once
 * per contig instead of once per window.  counts: int64[n] >= 0.
 * n_contigs > 1 loads a batch: contig c is counts[offsets[c] .. offsets[c+1]) and is
 * segmented independently (process_bedgraph.py:69: one segments_with_scores per contig);
 * offsets has n_contigs+1 entries, offsets[0]=0.  Pass offsets=NULL for one contig.
 * Candidates are reset to "all positions" (segmentation.py:8). */
int pasio_contig_load(pasio_ctx *ctx, const int64_t *counts, int64_t n,
                      const int64_t *offsets, int64_t n_contigs);
/* Same, from run-length intervals (the bedgraph form, process_bedgraph.py:46-60):
 * run r covers [starts[r], starts[r+1]) with value values[r]; starts has n_runs+1 entries. */
int pasio_contig_load_rle(pasio_ctx *ctx, const int64_t *starts, const int64_t *values,
                          int64_t n_runs, const int64_t *offsets, int64_t n_contigs);
/* pasio_contig_load of ONE contig fused with the first pasio_round (all positions are candidates): the counts go
 * up in 256 MB chunks on a copy stream while the chunks that have arrived are scanned and their windows run, so the
 * host-to-device copy hides the scan and the first round (segments_with_scores, segmentation.py:5-20, always starts
 * from np.arange(len(counts) + 1): segmentation.py:8).  Results and state are those of pasio_contig_load followed by
 * pasio_round.  PASIO_E_TABLE_TOO_SHORT: the contig IS loaded, no round was completed -- upload longer tables
 * (pasio_table_need) and call pasio_round. */
int pasio_contig_load_round(pasio_ctx *ctx, const int64_t *counts, int64_t n, int64_t window_size,
                            int64_t window_shift, int constraint, int64_t *n_in, int64_t *n_out, int64_t *cells);

/* Same as pasio_contig_load with the counts already resident in device memory (no copy is made;
 * the caller keeps d_counts alive and unmodified until the next load). */
int pasio_contig_load_device(pasio_ctx *ctx, const int64_t *d_counts_device, int64_t n,
                             const int64_t *offsets, int64_t n_contigs);
int pasio_contig_info(const pasio_ctx *ctx, int64_t *n, int64_t *total_count, int64_t *n_contigs);
/* cumsum[candidates] as the reference scorer exposes it (log_marginal_likelyhood.py:57). */
int pasio_cumsum_at(pasio_ctx *ctx, const int64_t *positions, int64_t m, int64_t *out);

/* ---- candidates ---------------------------------------------------------------------
 * positions are in the concatenated coordinate space of the loaded batch (contig c starts
 * at offsets[c]); contig boundaries are always candidates.  cands=NULL: all positions. */
int pasio_candidates_set(pasio_ctx *ctx, const int64_t *cands, int64_t m);
int pasio_candidates_count(const pasio_ctx *ctx, int64_t *m);
int pasio_candidates_download(pasio_ctx *ctx, int64_t *out, int64_t capacity, int64_t *m);

/* NotZeroReducer / NotConstantReducer applied to the whole contig as one slice (constants_reducer.py:5-21):
 * zeros: if every count is 0 only the two ends survive, else nothing changes; constants: a candidate p
 * survives when counts[p-1] != counts[p], both ends always survive.  Single-contig contexts only.
 * The current candidates are replaced by the survivors. */
int pasio_filter_candidates(pasio_ctx *ctx, int constraint, int64_t *n_in, int64_t *n_out);

/* ---- one sliding-window round -------------------------------------------------------
 * Replaces SlidingWindowReducer.reduce_candidate_list (sliding_window_reducer.py:21-29)
 * with base reducer [NotConstantReducer|NotZeroReducer +] SquareSplitter
 * (constants_reducer.py:5-21, square_splitter.py:67-109, dto/sliding_window.py:9-15):
 * every window of the round is one DP, all windows run in one launch, survivors are
 * united and compacted on the device.  Candidates stay device-resident.
 * n_in / n_out: candidate counts before / after (round_reducer.py:21: the round loop's
 * fixed-point test is n_in == n_out because the new list is a subset).
 * cells: DP (i,j) cells evaluated in this round. */
int pasio_round(pasio_ctx *ctx, int64_t window_size, int64_t window_shift, int constraint,
                int64_t *n_in, int64_t *n_out, int64_t *cells);
/* Of the most recent pasio_round: algorithmic cells, and how many of them the kernel proved irrelevant
 * with the exact far-column bound (csrc/window_dp.cu) instead of evaluating them.  After
 * pasio_square_split: the same two numbers for the whole-contig DP. */
int pasio_round_stats(const pasio_ctx *ctx, int64_t *cells, int64_t *cells_skipped);
/* Of the most recent pasio_round or pasio_square_split_batch (PASIO_TUNE_WINDOW_CERTIFY): windows in which every
 * candidate was proven a survivor up front, windows whose check failed, and the rows those failed checks still proved
 * (summed; the DP resumed after them). */
int pasio_round_certify_stats(const pasio_ctx *ctx, int64_t *passed, int64_t *fell_back, int64_t *resume_rows_sum);
/* The task list of the exact DP's worker CTAs (host only, no context, nothing is launched): for a candidate list of
 * n_candidates entries, lag and nblock as in PASIO_TUNE_EXACT_LAG / PASIO_TUNE_EXACT_NBLOCK, the tasks in the order the
 * worker CTAs pull them, as (row block, kind, slice) triples -- kind 0: S (self scores of the block, slice = quarter),
 * 1: F (far columns, bounded), 2: N (the column blocks in front of the band, exhaustive), 3: R (records of the finished
 * block, then done_block).  *n_tasks receives their number; PASIO_E_ARG when cap (in triples) is too small.  The flag
 * waits of the kernel are deadlock-free because every task only waits for tasks earlier in this list or for the
 * diagonal: tests/test_exact_task_plan.py checks that ordering for many shapes without a GPU. */
int pasio_exact_task_plan(int64_t n_candidates, int lag, int nblock, int32_t *triples, int64_t cap, int64_t *n_tasks);
/* Bytes the most recent pasio_contig_load_round put on the PCIe link (counts travel as uint16 or int32 where they fit,
 * PASIO_TUNE_UPLOAD_NARROW): n when every slice fitted 8 bits, 8 * n with plain copies. */
int pasio_upload_stats(const pasio_ctx *ctx, int64_t *wire_bytes);
/* Switch a kernel variant on or off (PASIO_TUNE_*).  Every variant returns identical results
 * (the bounds are exact); defaults come from PASIO_WD_PRUNE / PASIO_WD_PHASES / PASIO_XD_PRUNE /
 * PASIO_XD_LAG in the environment. */
int pasio_set_tuning(pasio_ctx *ctx, int key, int value);
/* RoundReducer.reduce_candidate_list (round_reducer.py:10-31): rounds until fixed point or
 * max_rounds (<=0: len(counts)).  Stops with PASIO_E_TABLE_TOO_SHORT when tables must grow
 * (state is kept; call again after uploading longer tables).
 * sizes (optional, capacity sizes_cap) receives the candidate count before each round run. */
int pasio_rounds(pasio_ctx *ctx, int64_t window_size, int64_t window_shift, int constraint,
                 int64_t max_rounds, int64_t *rounds_done, int64_t *n_out, int64_t *cells,
                 int64_t *sizes, int64_t sizes_cap);
/* Penalties of the window DP: while a term is set, pasio_round, pasio_rounds and pasio_contig_load_round run every
 * window through SquareSplitter.split_with_normalizations (square_splitter.py:29-65, reached from
 * sliding_window_reducer.py:10-18 when the window's base splitter is regularised) instead of
 * split_without_normalizations; per cell, in that order,
 *   t = self_score + P_i - split_number_penalty[num_splits_i] (+ first_column_refund for i = 0) - length_penalty[L_j - L_i],
 * first arg-max, num_splits_j = prev_j ? num_splits[prev_j] + 1 : 0, positions and split numbers local to the window.
 * The tables are those of pasio_square_split_regularized (square_splitter.py:46-54): split_number_penalty[k] =
 * multiplier * function(k + 1), at least as many entries as the largest window has candidates (PASIO_E_ARG otherwise);
 * length_penalty[len] = multiplier * function(len), as long as the log table (a round that needs more returns
 * PASIO_E_TABLE_TOO_SHORT with pasio_table_need's log entry); first_column_refund = multiplier * function(1).  NULL
 * switches a term off, both NULL clear the penalties; after an error both terms are off.  The tables are copied; pasio_square_split, the exact DP
 * with its own tables and the scoring entry points do not use them. */
int pasio_set_penalties(pasio_ctx *ctx, const double *split_number_penalty, int64_t n_split_number_penalty,
                        double first_column_refund, const double *length_penalty, int64_t n_length_penalty);

/* ---- exact DP -----------------------------------------------------------------------
 * Replaces SquareSplitter.split_without_normalizations + collect_split_points
 * (square_splitter.py:67-109) over the CURRENT candidates of a single-contig context.
 * out_splits (capacity cap) receives split positions; score = prefix_scores[-1].
 * prefix_scores / previous_splits (optional, N entries each) expose the DP arrays. */
int pasio_square_split(pasio_ctx *ctx, int64_t *out_splits, int64_t cap, int64_t *n_splits,
                       double *score, double *prefix_scores, int64_t *previous_splits);
/* The same DP for every contig of a loaded batch (any n_contigs >= 1), each over its own slice of the CURRENT
 * candidates, contigs independent of each other (the reference segments them one by one): the candidates are replaced
 * by the union of the contigs' split points, which holds every contig boundary.  Lists of at most
 * window_dp_max_candidates (8 192 on a B200) run together as whole-list windows of the window DP, longer lists through
 * the whole-chip DP one after another.  n_out: the new candidate count; cells / cells_skipped: summed over all contigs,
 * as pasio_round_stats reports them afterwards.  No score is returned (there is one per contig; pasio_segment_scores
 * gives the parts).  Errors, all raised before anything changes: PASIO_E_TABLE_TOO_SHORT (the tables must cover the
 * longest contig and its total count; grow them and call again), PASIO_E_TOO_LARGE (a contig's own total count + alpha
 * reaches 2^31; the message names the contig -- the batch's sum may exceed it), PASIO_E_STATE (no contig / params). */
int pasio_square_split_batch(pasio_ctx *ctx, int64_t *n_out, int64_t *cells, int64_t *cells_skipped);
/* SquareSplitter.split_with_normalizations (square_splitter.py:29-65) for element-wise penalty functions: per cell
 *   t = self_score + P_i - split_number_penalty[num_splits_i] (+ first_column_refund for i = 0) - length_penalty[L_j - L_i],
 * in that order, first arg-max, num_splits_j = prev_j ? num_splits[prev_j] + 1 : 0.  The caller builds the tables with
 * the reference's own expressions: length_penalty[len] = multiplier * function(len) for len = 0 .. contig length,
 * split_number_penalty[k] = multiplier * function(k + 1) for k = 0 .. candidates - 1, first_column_refund =
 * multiplier * function(1) (square_splitter.py:46-54); NULL switches a term off.  Other arguments as pasio_square_split. */
int pasio_square_split_regularized(pasio_ctx *ctx, const double *length_penalty, int64_t n_length_penalty,
                                   const double *split_number_penalty, int64_t n_split_number_penalty,
                                   double first_column_refund, int64_t *out_splits, int64_t cap, int64_t *n_splits,
                                   double *score, double *prefix_scores, int64_t *previous_splits);
/* LogMarginalLikelyhood*AlphaComputer.all_suffixes_self_score(stop)
 * (log_marginal_likelyhood.py:105-115, :121-132) over the current candidates:
 * out[0..stop). */
int pasio_suffix_scores(pasio_ctx *ctx, int64_t stop, double *out);

/* ---- per-segment outputs ------------------------------------------------------------
 * Replaces scores(), mean_counts(), log_marginal_likelyhoods(), total_sum_logfac()
 * (log_marginal_likelyhood.py:64-83) and NopSplitter.split (nop_splitter.py:15-18) over
 * the CURRENT candidates taken as the final split points (m candidates -> m-1 segments;
 * in a batch, the segment count is still m-1 because boundaries are shared).
 * Any output pointer may be NULL.  logfac_cumsum has m entries. */
int pasio_segment_scores(pasio_ctx *ctx, double *scores, int64_t *segment_counts,
                         double *mean_counts, double *logfac_cumsum, int64_t capacity,
                         int64_t *n_segments);

/* NopSplitter.split's total (nop_splitter.py:15-18: np.sum(scorer.scores())) over the current candidates, on the
 * device and in numpy's own summation order -- pairwise: blocks of <= 128 elements with 8 running sums, halves split
 * at multiples of 8 (numpy/core/src/umath/loops_utils.h.src, *_pairwise_sum) -- so the float64 result is the one
 * np.sum gives on the downloaded scores (checked against numpy 2.3.5), without a host pass over 8 bytes/segment. */
int pasio_segment_scores_sum(pasio_ctx *ctx, double *total);

/* log_marginal_likelyhoods() (log_marginal_likelyhood.py:76-78) over the current candidates, formed on the
 * device: lmm[k] = score[k] - (logfac_cumsum[k+1] - logfac_cumsum[k]), same two roundings as numpy.
 * sum_logfac = total_sum_logfac() (:64-65).  lmm has m-1 entries. */
int pasio_segment_lmm(pasio_ctx *ctx, double *lmm, int64_t capacity, double *sum_logfac);
/* Start computing the log-factorial prefix sums of the loaded batch (what pasio_segment_lmm and the logfac_cumsum output
 * of pasio_segment_scores need) on a side stream, so that the sequential sum (one thread per contig) runs beside the
 * rounds instead of after them.  Optional: the consumers compute the sums themselves when nothing was prefetched. */
int pasio_logfac_prefetch(pasio_ctx *ctx);

/* ---- pinned host buffers --------------------------------------------------------------------------
 * Page-locked host memory for callers that want full-rate PCIe copies (any host pointer works, pinned
 * is faster).  Plain cudaHostAlloc / cudaFreeHost behind a C symbol so a binding needs no CUDA headers. */
int pasio_host_alloc(int64_t bytes, void **out);
int pasio_host_free(void *ptr);

/* Groups parsed intervals into contigs and builds each contig's run lengths / values (interval_groups and the
 * accumulation loop of parse_bedgraph_stream, process_bedgraph.py:26-60; gap filling and --split-at-gaps as there).
 * run_len / run_val: capacity 2n; group_line[g] = first line of group g, group_run[g] = its first run
 * (n_groups + 1 entries).  Returns the number of groups. */
int64_t pasio_bedgraph_runs(const int64_t *starts, const int64_t *stops, const int64_t *counts,
                            const uint8_t *new_chrom, int64_t n, int split_at_gaps, int64_t *run_len,
                            int64_t *run_val, int64_t *group_line, int64_t *group_run, int64_t *n_runs);

/* ---- bedgraph text in / segment text out (host C++, csrc/textio.cpp) --------------------------------
 * pasio_bedgraph_parse replaces BedgraphInterval.from_string / each_in_stream (dto/intervals.py:16-39):
 * whitespace-separated `chrom start stop count` lines, blank lines skipped, a count that is not an integer
 * literal is read as float and truncated.  Per interval it returns start, stop, count and the byte range of
 * the chromosome token inside buf; new_chrom[i] = 1 where the token differs from the previous interval's
 * (the consecutive grouping of process_bedgraph.py:33).  On a malformed line returns PASIO_E_ARG with
 * *n_out = 0-based line number.  pasio_format_segments replaces the %-formatting of
 * process_bedgraph.py:71-89: mode 0 `chrom\tstart\tstop\tmean`, 1 `chrom\tstart\tstop`,
 * 2 `chrom\tstart\tstop\tmean\tlength\tlmm`; returns bytes written or a negative value if cap is too small. */
int64_t pasio_bedgraph_count_lines(const char *buf, int64_t len);
int pasio_bedgraph_parse(const char *buf, int64_t len, int64_t cap, int64_t *starts, int64_t *stops,
                         int64_t *counts, int64_t *name_off, int32_t *name_len, uint8_t *new_chrom,
                         int64_t *n_out, int64_t *float_counts);
int64_t pasio_format_segments(const char *chrom, int64_t offset, const int64_t *splits, int64_t n_splits,
                              const double *means, const double *lmm, int mode, char *out, int64_t cap);

/* pasio_format_segments for a batch of contigs segmented as one super-contig (splits hold every contig boundary):
 * first_split[c] = index of contig c's first split point (n_contigs + 1 entries), shift[c] = what to add to its
 * positions, names[name_off[c] .. name_off[c+1]) = its name.  Same lines as per-contig calls, in contig order. */
int64_t pasio_format_segments_batch(const char *names, const int64_t *name_off, const int64_t *shift,
                                    const int64_t *first_split, int64_t n_contigs, const int64_t *splits,
                                    const double *means, const double *lmm, int mode, char *out, int64_t cap);


/* ---- measurement hooks (bench.py / profiles) ------------------------------------------
 * Device time (ms, CUDA events on the context's stream) and launch count accumulated per
 * kernel family since the last reset: 0 scan, 1 window DP, 2 compaction+prepass,
 * 3 exact DP, 4 scoring, 5 H2D, 6 D2H. */
int pasio_timing_reset(pasio_ctx *ctx, int enable);
/* The context's cudaStream_t (as void*), so a caller can bracket calls with its own CUDA events. */
void *pasio_stream(pasio_ctx *ctx);
/* FP64-pipe micro-benchmark (independent DFMA chains on every SM): measured FP64 instructions/s,
 * the denominator of the DP roofline (MEASURED_PEAKS.json has no FP64 entry). */
int pasio_fp64_peak(pasio_ctx *ctx, double *instr_per_sec);
int pasio_timing_get(pasio_ctx *ctx, int family, double *ms, int64_t *launches);

#ifdef __cplusplus
}
#endif
#endif /* PASIO_B200_H */
