// Internal declarations shared by the CUDA translation units of libpasio_b200.so.
// sm_100a only; no other architecture is targeted.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <string>
#include <vector>

#include "../../include/pasio_b200.h"

typedef long long i64;
typedef unsigned long long u64;

#define PASIO_ABI_VERSION 1

// Grow-only device buffer.
struct DevBuf {
    void *p = nullptr;
    size_t bytes = 0;
    template <typename T> T *as() const { return reinterpret_cast<T *>(p); }
};

enum TimingFamily { TF_SCAN = 0, TF_WINDOW_DP = 1, TF_COMPACT = 2, TF_EXACT_DP = 3, TF_SCORE = 4,
                    TF_H2D = 5, TF_D2H = 6, TF_COUNT = 7 };

struct TimedSpan { int family; cudaEvent_t a, b; };

struct pasio_ctx {
    int device = 0;
    int sm_count = 0;
    int smem_optin = 0;          // max dynamic shared memory per block (opt-in)
    cudaStream_t stream = nullptr;
    cudaStream_t stream2 = nullptr;      // side stream: the warp-per-window kernels run beside the CTA-per-window kernel
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    cudaStream_t stream_copy = nullptr;  // host->device chunks of pasio_contig_load_round
    cudaStream_t stream_lx = nullptr;    // log-factorial sums prefetched beside the rounds (pasio_logfac_prefetch)
    cudaEvent_t ev_lx0 = nullptr, ev_lx1 = nullptr;
    bool logfac_eager = false;     // the pending sums were formed chunk by chunk behind the upload: verdict still to be read
    bool logfac_pending = false;         // the prefetch is in flight: consumers wait for ev_lx1 first
    std::vector<cudaEvent_t> chunk_events;
    void *stage[3] = {nullptr, nullptr, nullptr};   // page-locked staging ring for uploads from pageable memory
    cudaEvent_t stage_free[3] = {nullptr, nullptr, nullptr};
    bool stage_used[3] = {false, false, false};
    int stage_next = 0;
    // narrowed upload (api.cu: NarrowUpload): per host thread two page-locked slices and two device slices of int32
    void *nstage_host = nullptr;
    void *nstage_dev = nullptr;
    std::vector<cudaEvent_t> nstage_free;
    int nstage_threads = 0;
    i64 last_wire_bytes = 0;       // bytes the last pasio_contig_load_round put on the PCIe link
    std::string err;

    // scorer parameters (log_marginal_likelyhood.py:6-16,62)
    bool have_params = false;
    int alpha_is_int = 1;
    i64 alpha_int = 1;
    double alpha = 1.0, beta = 1.0, pen = 0.0;

    // look-up tables (cached_log.py), device copies
    DevBuf tab[3];
    i64 ntab[3] = {0, 0, 0};
    i64 need[3] = {0, 0, 0};

    // loaded batch ("super-contig": contigs concatenated, boundaries forced)
    bool have_contig = false;
    i64 n = 0;                   // total nt
    i64 total = 0;               // total count
    i64 max_count = 0;           // largest count
    bool logfac_ready = false;   // the log-factorial prefix sums of the loaded contig are computed (logfac_full, or lxPos / lxSum)
    bool logfac_is_exact = false;
    i64 n_contigs = 0;
    std::vector<int32_t> h_bounds;   // n_contigs+1 boundary positions (host copy)
    DevBuf counts;               // int64[n]
    bool counts_borrowed = false; // counts.p belongs to the caller (pasio_contig_load_device)
    DevBuf cg;                   // int64[n+1] exclusive prefix sums, cg[0]=0
    DevBuf cpbits;               // uint32 bitmap over positions 0..n : counts[p-1]!=counts[p]
    DevBuf keepbits;             // uint32 bitmap over positions 0..n : survivors of a round
    DevBuf bounds;               // int32[n_contigs+1]
    DevBuf brank;                // int32[n_contigs+1] index of each boundary in the candidate list

    // candidates (positions, int32, ascending); implicit_all: cand[q] == q
    bool implicit_all = true;
    DevBuf cand[2];
    DevBuf candC[2];             // int64 prefix sums at the candidates (cg[cand[k]]), written with the list
    int cur = 0;
    i64 m = 0;

    // per-round window table for batches (n_contigs > 1)
    DevBuf win_st, win_en;
    DevBuf win_flags;            // per window of the round (index relative to w_begin): 1 once a phase-1 window of the CTA kernel is done (others start at 1)
    DevBuf win_small, win_medium, win_large;  // per-round work lists of window numbers (small / medium: warp per window, large: CTA per window)
    i64 n_small = 0, n_medium = 0, n_large = 0;
    i64 n_large_p1 = 0;          // win_large[0 .. n_large_p1) are phase-1 windows, the rest (filled from the back of the nwin-long buffer) phase 2
    std::vector<int32_t> h_win_st, h_win_en, h_brank;

    // scratch
    DevBuf blocksum, tilestate, scalars, dpL, dpC, dpP, dpPrev, dpPart, dpPartArg, dpMark, dpJump, fscan, logfac_full;
    DevBuf xpRing, xpRec, xpTasks, regLR, regNR;

    // penalties of the rounds (pasio_set_penalties): NR[k] split-number, LR[len] length table, first-column refund
    bool pen_num = false, pen_len = false;
    DevBuf penNR, penLR;
    i64 n_pen_nr = 0, n_pen_lr = 0;
    double pen_refund = 0.0;
    DevBuf lxPos, lxSum, lxFirst, lxState;    // logfac_exact.cu: positions / running sums of the non-zero log-factorial terms, first term per contig
    i64 lx_terms = 0;
    i64 scan_tiles_done = 0;     // tiles of the loaded contig already scanned (pasio_contig_load_round scans chunk by chunk)   // exact_pruned.cu: self-score ring, column-block records, task list

    // tuning switches (pasio_set_tuning; defaults from the PASIO_WD_* / PASIO_XD_* environment variables)
    int tune[PASIO_TUNE_COUNT];
    i64 *h_scalars = nullptr;    // pinned, 20 entries

    i64 last_cells = 0, last_cells_skipped = 0;   // of the most recent round
    i64 last_certify[3] = {0, 0, 0};              // of the most recent round: windows passed, fell back, rows proven before falling back
    i64 prev_round_in = 0, prev_round_out = 0;    // candidates before / after the previous round on the current candidates (0: none)
    std::vector<i64> pw_leaf_start;      // leaf boundaries of numpy's pairwise sum for pw_n elements (pasio_segment_scores_sum)
    i64 pw_n = -1;
    std::vector<double> pw_leaf_sum;

    // timing
    bool timing = false;
    std::vector<TimedSpan> spans;
    std::vector<cudaEvent_t> event_pool;
    double fam_ms[TF_COUNT] = {0};
    i64 fam_launches[TF_COUNT] = {0};
};

int pasio_fail(pasio_ctx *ctx, int code, const char *fmt, ...);
int pasio_reserve(pasio_ctx *ctx, DevBuf &b, size_t bytes);   // grow-only; returns status

#define CUDA_TRY(ctx, call)                                                                     \
    do {                                                                                        \
        cudaError_t e__ = (call);                                                               \
        if (e__ != cudaSuccess)                                                                 \
            return pasio_fail((ctx), PASIO_E_CUDA, "%s failed: %s (%s:%d)", #call,              \
                              cudaGetErrorString(e__), __FILE__, __LINE__);                     \
    } while (0)

#define PASIO_TRY(call)                    \
    do {                                   \
        int rc__ = (call);                 \
        if (rc__ != PASIO_OK) return rc__; \
    } while (0)

// RAII-less timing helpers: record an event pair around a family of launches.
struct TimingScope {
    pasio_ctx *ctx;
    int idx;
    cudaStream_t on;
    TimingScope(pasio_ctx *c, int family, i64 launches = 1, cudaStream_t stream = nullptr);
    ~TimingScope();
};

// ---- launchers implemented in the kernel translation units (all asynchronous on ctx->stream) ----

// scan.cu
int launch_scan_counts(pasio_ctx *ctx);                       // counts -> cg, cpbits, validation, total
int launch_scan_prepare(pasio_ctx *ctx, i64 *n_tiles, i64 *tile_elems);   // the same in pieces: reset the tile states ...
int launch_scan_tiles(pasio_ctx *ctx, i64 tiles);             // ... then the next `tiles` tiles, in order
int launch_expand_rle(pasio_ctx *ctx, const i64 *d_starts, const i64 *d_values, i64 n_runs);
int launch_logfac_scan(pasio_ctx *ctx, double *d_out, cudaStream_t stream = nullptr);   // float64 prefix sums of G[counts+1], n+1 entries

// compact.cu
int launch_compact_keepbits(pasio_ctx *ctx, int slot, i64 *h_count);  // keepbits -> cand[slot] (sorted positions) + candC[slot]; syncs
int launch_boundary_ranks(pasio_ctx *ctx);                    // brank from current candidates
// classify_constraint >= 0: also sort the windows into ctx->win_small / win_large (n_small, n_large) for launch_window_dp
int launch_window_prepass(pasio_ctx *ctx, i64 nwin, int wsize, int wshift, i64 *h_max_span, i64 *h_max_cnt,
                          int classify_constraint = -1, i64 w_begin = 0);  // windows [w_begin, w_begin + nwin); syncs
// most candidates the warp-per-window kernels take (small / medium class), shared by K4 (window_dp.cu) and K8
// (window_dp_reg.cu) because the prepass sorts the windows for both
constexpr int WD_SMALL_MAX_CANDIDATES = 160, WD_MEDIUM_MAX_CANDIDATES = 512;
int small_window_max_candidates();                           // window_dp.cu: most candidates the warp-per-window kernels take
int medium_window_max_candidates();
int launch_validate_candidates(pasio_ctx *ctx, i64 *h_bad);   // syncs
int launch_filter_candidates(pasio_ctx *ctx, int constraint);  // current candidates -> keepbits

// window_dp.cu
int launch_window_dp(pasio_ctx *ctx, i64 nwin, int wsize, int wshift, int constraint, i64 w_begin = 0,
                     bool keep_cell_counters = false);   // windows [w_begin, w_begin + nwin)
int window_dp_max_candidates(pasio_ctx *ctx);

// window_dp_reg.cu: the same round with the penalties of pasio_set_penalties (needs the classified prepass lists)
int launch_window_dp_reg(pasio_ctx *ctx, i64 nwin, int wsize, int wshift, int constraint, bool keep_cell_counters = false);
int window_dp_reg_max_candidates(pasio_ctx *ctx);

// exact_dp.cu
int launch_exact_dp(pasio_ctx *ctx, i64 N);                   // over ctx->dpL/dpC -> dpP/dpPrev
int launch_exact_dp_pruned(pasio_ctx *ctx, i64 N, int lag);
int launch_regularized_dp(pasio_ctx *ctx, i64 N, const double *d_lr, const double *d_nr, double add0);   // regularized_dp.cu   // exact_pruned.cu: the same result, far columns bounded
int launch_gather_candidates(pasio_ctx *ctx);                 // current candidates -> dpL/dpC (rebased)
int launch_backtrace_mark(pasio_ctx *ctx, i64 N);             // dpPrev -> keepbits (positions on the optimal path)
int launch_suffix_row(pasio_ctx *ctx, i64 stop, double *d_out);

// score.cu
int launch_segment_scores(pasio_ctx *ctx, double *d_scores, i64 *d_segcounts, double *d_means);
int launch_pairwise_leaves(pasio_ctx *ctx, const double *d_values, const i64 *d_leaf_start, i64 n_leaves, double *d_leaf_sum);
int launch_gather_i64(pasio_ctx *ctx, const i64 *d_src, const int32_t *d_idx32, const i64 *d_idx64, i64 m, i64 *d_out);
int launch_gather_f64_at_cands(pasio_ctx *ctx, const double *d_src, double *d_out);
int launch_lmm(pasio_ctx *ctx, const double *d_scores, const double *d_logfac_full, double *d_lmm);

// logfac_exact.cu: logfac_cumsum with the reference's sequential rounding
int launch_logfac_exact(pasio_ctx *ctx, cudaStream_t stream = nullptr);
int launch_logfac_exact_begin(pasio_ctx *ctx, cudaStream_t stream);                  // the same chunk by chunk behind an upload ...
int launch_logfac_exact_chunk(pasio_ctx *ctx, i64 p0, i64 p1, cudaStream_t stream);   // ... positions [p0, p1) ...
int logfac_exact_chunks_result(pasio_ctx *ctx, bool *usable);                        // ... and, after the stream finished, the verdict
int launch_lmm_exact(pasio_ctx *ctx, const double *d_scores, double *d_lmm);
int launch_logfac_at_candidates_exact(pasio_ctx *ctx, double *d_out);
int logfac_exact_total(pasio_ctx *ctx, double *h_out);

static inline const int32_t *cur_cand(const pasio_ctx *ctx) {
    return ctx->implicit_all ? nullptr : ctx->cand[ctx->cur].as<int32_t>();
}
static inline const i64 *cur_cand_cg(const pasio_ctx *ctx) {
    return ctx->implicit_all ? nullptr : ctx->candC[ctx->cur].as<i64>();
}

// Window geometry of dto/sliding_window.py:9-15 over candidate indices: either the closed form
// for one contig or a host-built table for a batch (windows never span contigs).
struct WinGeom {
    const int32_t *st_tab;
    const int32_t *en_tab;
    i64 m;
    int wsize, wshift;
};
WinGeom make_geom(const pasio_ctx *ctx, int wsize, int wshift);

// ---- device helpers -------------------------------------------------------------------------
#ifdef __CUDACC__
__device__ __forceinline__ void window_range(const WinGeom &g, i64 w, i64 &st, i64 &en) {
    if (g.st_tab) {
        st = __ldg(g.st_tab + w);
        en = __ldg(g.en_tab + w);
    } else {
        st = w * g.wshift;                       // range(0, len-1, shift)
        en = min(st + (i64)g.wsize + 1, g.m);    // stop = min(start + size + 1, len)
    }
}
// Exact int32 (0 <= v < 2^31) -> double with one DADD on the FP64 pipe instead of a
// quarter-rate I2F conversion: 2^52 + v is representable, so the subtraction is exact.
__device__ __forceinline__ double u32_to_double(int v) {
    return __dsub_rn(__hiloint2double(0x43300000, v), 4503599627370496.0);
}
__device__ __forceinline__ bool bit_test(const uint32_t *__restrict__ bits, i64 p) {
    return (__ldg(bits + (p >> 5)) >> (p & 31)) & 1u;
}
#endif
