// K4: all windows of one sliding-window round: one launch per size class (a CTA per large window, a warp per
// small / medium window; the prepass in compact.cu sorts the windows).
//
// Replaces, per window, the chain
//   SlidingWindowReducer.reduce_candidates_in_window   splitters/sliding_window_reducer.py:10-18
//   -> NotConstantReducer / NotZeroReducer              splitters/constants_reducer.py:5-21
//   -> SquareSplitter.split_without_normalizations      splitters/square_splitter.py:67-100
//   -> collect_split_points                              splitters/square_splitter.py:102-109
//   -> set.update(...)                                   splitters/sliding_window_reducer.py:25
// (paths under /root/reference/src/pasio/).  In the flat formulation (SURVEY 7.4) a window needs
// only two integer vectors: positions L and global prefix sums C of its candidates, re-based to
// the window's first candidate exactly like counts[start:stop] / candidates - start.
//
// Per CTA: (A) warp-ballot stream compaction of the window's candidates (constraint filter)
// into shared memory, (B) the DP in 32-row block steps (dp_core.cuh) -- plain sweeps, or, for explicit
// candidate lists, pruned and software-pipelined steps (far_pass below), (C) back-trace by pointer
// doubling and an atomicOr scatter of the survivors into the position bitmap.
// CTAs are persistent and pull windows from an atomic counter (window cost varies as N^2); phase-2
// windows whose candidates all survived already are skipped (see window_dp_kernel).
#include "dp_core.cuh"
#include "bound.cuh"
#include <cstdio>
#include <cstdlib>

namespace {

constexpr int WD_THREADS = 256;
constexpr int WD_WARPS = WD_THREADS / 32;
constexpr int WD_FARW = WD_WARPS - 1;   // pruned path: warps 1..7 bound / evaluate columns while warp 0 runs the dependent chain
constexpr int NEAR_Q = 4;               // pruned path: the nearest 32 columns are swept as 4 chunks of 8
constexpr int PR_CB = 32;               // far columns are first bounded in blocks of 32 ...
constexpr int PR_FB = 8;                // ... and the surviving blocks again in sub-blocks of 8
constexpr int PR_MIN_N = 256;           // windows up to this many candidates are not worth bounding
constexpr int PR_DENSE = 28;            // a block with this many surviving 4 x 8 rectangles (of 32) is swept whole

// Development-only phase timers (make PROF=1): cycles seen by thread 0 (warp 0: chain side) and thread 32
// (warp 1: far side) of every CTA, summed per phase.
#ifdef PASIO_WD_PROF
__device__ unsigned long long g_wd_prof[16];
struct ProfAcc { long long t0; long long a0, a1, a2, a3, a4, a5, a6, a7; };
#define PROF_DECL ProfAcc prof = {clock64(), 0, 0, 0, 0, 0, 0, 0, 0}
// the clock read is made dependent on a shared-memory load: BAR.SYNC does not block at issue, only at the next
// consumer, so a bare clock64() after __syncthreads() would charge the wait to the following phase
__device__ __forceinline__ long long prof_clock()
{
    unsigned dummy;
    long long t;
    asm volatile("ld.volatile.shared.u32 %0, [%1];" : "=r"(dummy) : "r"(0u) : "memory");
    asm volatile("mov.u64 %0, %%clock64;" : "=l"(t) : "r"(dummy) : "memory");
    return t;
}
#define PROF_T(i) do { const long long t1__ = prof_clock(); prof.a##i += t1__ - prof.t0; prof.t0 = t1__; } while (0)
#define PROF_FLUSH do { if (threadIdx.x == 0 || threadIdx.x == 32) { unsigned long long *g__ = g_wd_prof + (threadIdx.x ? 8 : 0); \
    atomicAdd(g__ + 0, (unsigned long long)prof.a0); atomicAdd(g__ + 1, (unsigned long long)prof.a1); \
    atomicAdd(g__ + 2, (unsigned long long)prof.a2); atomicAdd(g__ + 3, (unsigned long long)prof.a3); \
    atomicAdd(g__ + 4, (unsigned long long)prof.a4); atomicAdd(g__ + 5, (unsigned long long)prof.a5); \
    atomicAdd(g__ + 6, (unsigned long long)prof.a6); atomicAdd(g__ + 7, (unsigned long long)prof.a7); } \
    prof.a0 = prof.a1 = prof.a2 = prof.a3 = prof.a4 = prof.a5 = prof.a6 = prof.a7 = 0; } while (0)
#define PROF_ARGS , ProfAcc &prof
#define PROF_PASS , prof
#else
#define PROF_DECL
#define PROF_T(i) do { } while (0)
#define PROF_FLUSH do { } while (0)
#define PROF_ARGS
#define PROF_PASS
#endif

struct WinDpParams {
    WinGeom geom;
    i64 nwin;
    const int32_t *cand;        // nullptr: all positions
    const i64 *cg;
    const i64 *cgc;             // cg at the candidates (cgc[q] == cg[cand[q]]); nullptr with all positions
    const uint32_t *cpbits;
    uint32_t *keepbits;
    const double *gtab;
    const double *ltab;
    int constraint;
    int alpha_int;
    double alpha;
    double pen;
    int cap;                    // max candidates in a window
    u64 *cells;                 // algorithmic cells N(N-1)/2
    u64 *cells_skipped;         // cells proven irrelevant by the far-column bound (0 without pruning)
    unsigned *work_counter;
    const int32_t *list;        // window numbers to process (nwin of them); nullptr: w_begin .. w_begin+nwin-1
    i64 w_begin;
    // two phases (CTA kernel): list[0 .. n_p1) first; the other nwin - n_p1 windows (stored from the END of the
    // list_len-long list backwards) start once all of phase 1 is done and are skipped if every one of their candidates
    // already survived
    i64 n_p1, list_len;
    unsigned char *done_flags;  // [list_len], index = window number - w_begin
    int p1_stride;
    int skip_covered;           // 0: phase-2 windows neither wait nor get skipped (experiments)
    int speculate;              // CTA kernel: try block_chain_speculative first (PASIO_TUNE_WINDOW_SPECULATE)
    int certify;                // CTA kernel: check every pruned window for "every candidate survives" first (certify_window)
    u64 *certify_stats;         // [0] windows that passed the check, [1] windows that fell back, [2] sum of their proven rows
    int n_lg;                   // warp-per-window kernels with the log table in shared memory: entries copied
};

__host__ __device__ inline size_t window_smem_bytes(int cap)
{
    const size_t capr = (size_t)((cap + 31) & ~31);
    return capr * 16                // sCol (L, C, P)
           + NEAR_Q * 32 * 8        // sPartV
           + DP_JB * DP_JB * 8      // sTri            (back-trace: sMark lives here, needs capr <= 8192)
           + NEAR_Q * 32 * 4        // sPartA
           + 24 * 4                 // sMisc (+ the list counters)
           + capr * 2               // sPrev
           + (capr / PR_CB) * sizeof(CoarseRec)   // sCoarse  (back-trace: sJump lives here, capr*2 bytes)
           + 2 * 32 * sizeof(float4)              // sRow: the 32 rows being bounded (lower bound, C, L as floats), two blocks
           + capr * 2                             // sList: fine rectangles that survived both bounds (< PR_DENSE per block)
           + 2 * ((capr / PR_CB) * 2 + 16)        // sDense: blocks to sweep whole; sSurv: blocks that survived level 1
           + 2 * WD_FARW * 32 * (8 + 4)           // sFarV, sFarA: per-warp far results of the 32 rows, double-buffered
           + 8 * 8;                 // sScal
}

__device__ __forceinline__ int2 col_lc(const ColRec *sCol, int i)      // (L, C) only: P of that column may be in flight
{
    return *reinterpret_cast<const int2 *>(sCol + i);
}

// ---- exact pruning of far columns (branch and bound) -----------------------------------------
// For rows j in [j0, j1] and columns i in [i0, i1] every cell value
//     t_ij = F(u_ij, len_ij) + P_i ,  F(u, len) = G[u (+alpha)] - s*Lg[len],  u_ij = C_j - C_i,  len_ij = L_j - L_i
// satisfies, for ANY real a, b (the "tilt"),
//     t_ij - LB_j = [P_i + a*C_i + b*L_i] + [F(u_ij, len_ij) + a*u_ij + b*len_ij] - [LB_j + a*C_j + b*L_j]
//                <= max_i [P_i + a*C_i + b*L_i]  +  max_box [F(u, len) + a*u + b*len]  -  min_j [LB_j + a*C_j + b*L_j]
// where the box is [C_j0 - C_i1, C_j1 - C_i0] x [L_j0 - L_i1, L_j1 - L_i0].  F + a*u + b*len is convex in u for fixed
// len (lgamma is convex, the rest is linear) and convex in len for fixed u (-s*log(len + beta) with s >= 0), so
// its maximum over the box is at one of the 4 corners.  With a, b fitted to the block's own P (least squares: along
// an optimal path P is close to linear in (C, L)) the first bracket hardly varies and the bound is tight to second
// order; without the tilt it is loose by the block's whole range of P.  If the right-hand side (plus delta, which
// covers table and rounding errors: 2^-44 of the window's largest magnitudes, > 50x the worst case, < 1e-6 in
// absolute terms) is negative, no cell of the rectangle reaches the lower bound LB_j of its row's maximum: it can
// hold neither the arg-max nor a tie, so skipping it leaves P, prev and the back-trace bit-identical.
// LB_j is the value of the "split at every candidate" path from the last finished row to row j -- a feasible
// segmentation, hence a lower bound of the maximum, and in the later rounds (where nearly every candidate
// survives) the maximum itself.  It needs no result of the block that is being chained at the moment, so the far
// pass of block k+1 runs on warps 1..7 WHILE warp 0 resolves the dependent chain of block k.  The path value is
// formed with parallel sums and lowered by delta_path (2^-39 of the largest magnitudes: at most 76 roundings of
// partial sums below 64x that magnitude separate it from the sequentially rounded value the chain produces).
// Two levels: 32 rows x 32 columns first (one lane per rectangle), the survivors again as 4 rows x 8 columns
// (one warp per surviving rectangle); what survives both is evaluated exactly, cell by cell, in the reference's
// operation order.
// Lower bounds for the 32 rows of the block starting at jb, by one warp (lane = row), while the block before it
// (rows [jbp, jb), jbp = jb - 32) is still to be chained; everything before row jbp is final.
//   sRow[r] = (lb, C, L, -) as floats: the far pass takes min_r (lb_r + a*C_r + b*L_r) in float and subtracts a
//   rigorous bound of the float error, 2^-20 * (max|lb| + |a|*C_max + |b|*L_max)  (sRowStat = max |lb|).
template <bool AI>
__device__ __forceinline__ void compute_row_lb(int jbp, int jb, int N, const ColRec *sCol, float4 *sRow, double *sRowStat,
                                               double delta_path, double pen,
                                               const double *__restrict__ gtab, const double *__restrict__ ltab,
                                               int alpha_int, double alpha)
{
    const int lane = threadIdx.x & 31;
    const int jrow = min(jb + lane, N - 1);
    const int2 me = col_lc(sCol, jrow);                     // (L, C)
    const RowConst<AI> rme = make_row<AI>(me.y, me.x, alpha_int, alpha);
    const int jp = jbp + lane;                              // a row of the block in flight
    const int2 pm = col_lc(sCol, jp), pb = col_lc(sCol, jp - 1), before = col_lc(sCol, jrow - 1);
    const RowConst<AI> rp = make_row<AI>(pm.y, pm.x, alpha_int, alpha);
    const double wp = self_score<AI>(pb.y, pb.x, rp, gtab, ltab) + pen;          // w(m-1, m) + pen, m in [jbp, jb)
    double run = self_score<AI>(before.y, before.x, rme, gtab, ltab) + (lane ? pen : 0.0);   // w(j-1, j) [+ pen of the previous row]
    const double tot_prev = warp_sum(wp);
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const double o = __shfl_up_sync(0xffffffffu, run, d);
        if (lane >= d) run += o;
    }
    double path = (sCol[jbp - 1].P + tot_prev) + run - delta_path;
    if (!(fabs(path) < 1e30)) path = -INFINITY;             // NaN / inf / beyond float range: no information
    float lbf = (float)path;                                // overflow gives -inf: no information, still valid
    sRow[lane] = make_float4(lbf, (float)me.y, (float)me.x, 0.f);
    double ab = (jb + lane < N && path > -1e300) ? fabs(path) : 0.0;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) ab = fmax(ab, __shfl_xor_sync(0xffffffffu, ab, off));
    if (lane == 0) *sRowStat = ab;
}

// min over rows [r0, r1] of lb_r + a*C_r + b*L_r, as a rigorous lower bound (float arithmetic minus its error bound)
__device__ __forceinline__ double tilted_row_min(const float4 *sRow, int r0, int r1, double a, double b, double lbabs,
                                                 int c_max, int l_max)
{
    const float af = (float)a, bf = (float)b;
    float m = INFINITY;
#pragma unroll 4
    for (int r = r0; r <= r1; ++r) {
        const float4 rr = sRow[r];
        m = fminf(m, fmaf(af, rr.y, fmaf(bf, rr.z, rr.x)));
    }
    const double err = (lbabs + fabs(a) * (double)c_max + fabs(b) * (double)l_max) * 9.5367431640625e-07;   // 2^-20
    return (double)m - err;
}

// Far columns [1, 1 + 32*nfar) of the 32-row block starting at row jb, run by warps 1..7 while warp 0 chains the
// block before it.  Level 1: coarse block cb is bounded by far warp cb / 32, lane cb % 32 (a lane per rectangle costs a
// warp the same for 1 or 32 rectangles, so they are packed); the survivors go to a shared list and, after a barrier among
// the far warps, are dealt round-robin and split into 4-row x 8-column rectangles (level 2, one lane each); what
// survives again goes to a second list.  Level 3 (after another barrier): the listed rectangles are dealt round-robin and evaluated exactly, 4 in flight per
// warp, lane = (row of the group, column of the sub-block).  Every far warp keeps a running (max, first arg-max) for
// all 32 rows (lane = row) and publishes it in its slice of sFarV / sFarA; far warp 0 also covers column 0, which
// is in no block.  Returns the number of cells skipped (per lane; the caller sums).
template <bool AI>
__device__ __forceinline__ u64 far_pass(int jb, int N, int nfar, const ColRec *sCol, const CoarseRec *sCoarse,
                                        const float4 *sRow, double lbabs, unsigned short *sList, unsigned short *sDense,
                                        unsigned short *sSurv, int *sListCount /* [0] fine list, [1] dense list, [2] level-1 survivors */,
                                        double *sFarVW, int *sFarAW, double delta,
                                        const double *__restrict__ gtab, const double *__restrict__ ltab,
                                        int alpha_int, double alpha PROF_ARGS)
{
    const int lane = threadIdx.x & 31, w7 = (threadIdx.x >> 5) - 1;
    const int nrows = min(DP_JB, N - jb);
    const int2 rowF = col_lc(sCol, jb), rowL = col_lc(sCol, jb + nrows - 1);           // (L, C)
    const int2 me = col_lc(sCol, min(jb + lane, N - 1));
    const RowConst<AI> rme = make_row<AI>(me.y, me.x, alpha_int, alpha);

    // running far result of row `lane`
    double best = -INFINITY;
    int arg = 0x7fffffff;
    if (w7 == 0 && lane < nrows) {
        const ColRec a0 = sCol[0];
        best = __dadd_rn(self_score<AI>(a0.C, a0.L, rme, gtab, ltab), a0.P);
        arg = 0;
    }
    u64 skipped = 0;

    const int rg = lane >> 2, q = lane & 3;                 // level 2: row group, sub-block
    const int r0 = 4 * rg, r1 = min(r0 + 3, nrows - 1);
    const bool act2 = r0 < nrows;
    const int2 gF = col_lc(sCol, jb + min(r0, nrows - 1)), gL = col_lc(sCol, jb + r1);

    // level 2: a block as 8 row groups x 4 sub-blocks of 8 columns, one lane per rectangle (a whole warp per block)
    auto level2 = [&](int cb1) {
        const CoarseRec *rec = sCoarse + cb1;
        const double a = rec->a, b = rec->b;
        bool surv2 = false;
        if (act2) {
            const int i0 = 1 + PR_CB * cb1 + PR_FB * q;
            const int2 cF = col_lc(sCol, i0), cL = col_lc(sCol, i0 + PR_FB - 1);
            const double m2 = tilted_box_max<AI>(gF.y - cL.y, gL.y - cF.y, gF.x - cL.x, gL.x - cF.x, a, b,
                                                 gtab, ltab, alpha_int, alpha);
            const double m3 = tilted_row_min(sRow, r0, r1, a, b, lbabs, gL.y, gL.x);
            surv2 = !(rec->mpt8[q] + m2 - m3 + delta < 0.0);
            if (!surv2) skipped += (u64)(PR_FB * (r1 - r0 + 1));
        }
        const unsigned mask2 = __ballot_sync(0xffffffffu, surv2);
        const int n2 = __popc(mask2);
        if (n2 >= PR_DENSE) {
            // most of the block is needed: the whole 32 x 32 block goes to the sweep list (its rectangles are not skipped)
            if (act2 && !surv2) skipped -= (u64)(PR_FB * (r1 - r0 + 1));
            if (lane == 0) sDense[atomicAdd(sListCount + 1, 1)] = (unsigned short)cb1;
        } else if (n2) {
            int slot = 0;
            if (lane == 0) slot = atomicAdd(sListCount, n2);
            slot = __shfl_sync(0xffffffffu, slot, 0);
            if (surv2) sList[slot + __popc(mask2 & ((1u << lane) - 1u))] = (unsigned short)((cb1 << 5) | lane);
        }
    };
    // The nearest blocks nearly always survive level 1, and level 1 (packed) leaves warps idle: those warps take the nearest
    // blocks straight to level 2 while the others bound the rest, which takes a level-2 pass off the critical path.
    const int l1_warps = min(WD_FARW, (nfar + 31) / 32);
    const int n_direct = max(0, min(nfar, WD_FARW - l1_warps));
    const int nfar1 = nfar - n_direct;                     // level 1 covers blocks [0, nfar1)
    if (w7 >= l1_warps && w7 - l1_warps < n_direct) level2(nfar - 1 - (w7 - l1_warps));

    // ---- level 1: 32 rows x 32 columns, one lane per rectangle, the rectangles packed into as few warps as they fill
    // (77 blocks of a 2500-candidate window: 3 warps) ----
    for (int base = 0; base + 32 * w7 < nfar1 && w7 < l1_warps; base += 32 * l1_warps) {
        const int cb = base + 32 * w7 + lane;
        bool surv1 = false;
        if (cb < nfar1) {
            const CoarseRec *rec = sCoarse + cb;
            const int4 ends = *reinterpret_cast<const int4 *>(rec);
            const double a1 = rec->a, b1 = rec->b;
            const double ub1 = rec->mpt + tilted_box_max<AI>(rowF.y - ends.y, rowL.y - ends.x, rowF.x - ends.w, rowL.x - ends.z,
                                                             a1, b1, gtab, ltab, alpha_int, alpha);
            // min_r (lb_r + a*C_r + b*L_r): every lane walks the 32 rows (broadcast reads of sRow)
            const double m3 = tilted_row_min(sRow, 0, nrows - 1, a1, b1, lbabs, rowL.y, rowL.x);
            surv1 = !(ub1 - m3 + delta < 0.0);                           // NaN keeps the block
            if (!surv1) skipped += (u64)(PR_CB * nrows);
        }
        const unsigned mask1 = __ballot_sync(0xffffffffu, surv1);
        if (mask1) {
            int slot = 0;
            if (lane == 0) slot = atomicAdd(sListCount + 2, __popc(mask1));
            slot = __shfl_sync(0xffffffffu, slot, 0);
            if (surv1) sSurv[slot + __popc(mask1 & ((1u << lane) - 1u))] = (unsigned short)cb;
        }
    }
    PROF_T(4);
    asm volatile("bar.sync 1, %0;" ::"n"(WD_FARW * 32) : "memory");
    const int nsurv = *reinterpret_cast<volatile int *>(sListCount + 2);

    // ---- level 2 of the blocks that survived level 1, dealt round-robin to the far warps ----
    for (int e = w7; e < nsurv; e += WD_FARW) level2(sSurv[e]);
    PROF_T(5);
    // ---- all far warps: the list is complete ----
    asm volatile("bar.sync 1, %0;" ::"n"(WD_FARW * 32) : "memory");
    const int total = *reinterpret_cast<volatile int *>(sListCount);
    const int ndense = *reinterpret_cast<volatile int *>(sListCount + 1);
    PROF_T(3);

    // ---- dense blocks: plain sweeps, one warp per 32 x 32 block (a lane: 2 rows, 4 apart, x 4 columns, 8 apart) ----
    for (int e = w7; e < ndense; e += WD_FARW) {
        const int i0 = 1 + PR_CB * (int)sDense[e];
        const int rr = lane & 3, cph = lane >> 2;
#pragma unroll 1
        for (int g = 0; g < 4; ++g) {
            RowConst<AI> r[2];
            double bst[2];
            int ag[2];
#pragma unroll
            for (int k = 0; k < 2; ++k) {
                const int2 rl = col_lc(sCol, min(jb + g * 8 + k * 4 + rr, N - 1));
                r[k] = make_row<AI>(rl.y, rl.x, alpha_int, alpha);
                bst[k] = -INFINITY;
                ag[k] = i0 + cph;
            }
            sweep_columns<AI, 4, 2>(i0, i0 + PR_CB, cph, 8, sCol, r, gtab, ltab, bst, ag);
#pragma unroll
            for (int k = 0; k < 2; ++k) {
                merge_column_phases<4>(bst[k], ag[k]);
                // lanes 0..3 (column phase 0) hold rows g*8 + k*4 + rr: hand them to the lanes that own those rows
                const double v = __shfl_sync(0xffffffffu, bst[k], lane & 3);
                const int va = __shfl_sync(0xffffffffu, ag[k], lane & 3);
                if ((lane >> 2) == g * 2 + k && lane < nrows && (v > best || (v == best && va < arg))) { best = v; arg = va; }
            }
        }
    }

    // ---- level 3: the survivors exactly; lane = (row er of the group, column ec of the sub-block) ----
    constexpr int UX = 4;
    const int er = lane >> 3, ec = lane & 7;
    for (int e0 = w7 * UX; e0 < total; e0 += WD_FARW * UX) {
        double t[UX];
        int ta[UX], g4[UX];
#pragma unroll
        for (int u = 0; u < UX; ++u) {
            t[u] = -INFINITY;
            ta[u] = 0x7fffffff;
            g4[u] = 0;
            if (e0 + u < total) {
                const int ent = sList[e0 + u];
                const int l2 = ent & 31;
                g4[u] = 4 * (l2 >> 2);
                const int row = g4[u] + er;                            // row of the block step
                const int col = 1 + PR_CB * (ent >> 5) + PR_FB * (l2 & 3) + ec;
                ta[u] = col;
                if (row < nrows) {
                    const int2 rl = col_lc(sCol, jb + row);
                    const RowConst<AI> rc = make_row<AI>(rl.y, rl.x, alpha_int, alpha);
                    const ColRec cc = sCol[col];
                    t[u] = __dadd_rn(self_score<AI>(cc.C, cc.L, rc, gtab, ltab), cc.P);
                }
            }
        }
#pragma unroll
        for (int u = 0; u < UX; ++u) {
#pragma unroll
            for (int off = 1; off < 8; off <<= 1) {
                const double ob = __shfl_xor_sync(0xffffffffu, t[u], off);
                const int oa = __shfl_xor_sync(0xffffffffu, ta[u], off);
                if (ob > t[u] || (ob == t[u] && oa < ta[u])) { t[u] = ob; ta[u] = oa; }
            }
            // hand the 4 row results (lanes 0, 8, 16, 24) to the lanes that own those rows
            const int rel = lane - g4[u];
            const double v = __shfl_sync(0xffffffffu, t[u], (rel & 3) * 8);
            const int va = __shfl_sync(0xffffffffu, ta[u], (rel & 3) * 8);
            if (rel >= 0 && rel < 4 && (v > best || (v == best && va < arg))) { best = v; arg = va; }
        }
    }
    sFarVW[lane] = best;
    sFarAW[lane] = arg;
    return skipped;
}

// The nearest 32 columns [jb-32, jb) (all final) and the triangle self scores of the block starting at row jb,
// by NW warps.  The rectangle is 16 tasks of 8 rows x 8 columns (a lane: 2 rows, 4 apart, one column; so the 32
// addresses of one gather span 4+8 candidates); task t covers row group t & 3, column chunk t >> 2.  Per-chunk
// (max, first arg-max) go to sPartV / sPartA [chunk*32 + row].
template <bool AI, int NW>
__device__ __forceinline__ void near_tri_farwarps(int w7 /* 0 .. NW-1 */, int jb, int N, const ColRec *sCol, double *sPartV,
                                                  int *sPartA, double *sTri,
                                                  const double *__restrict__ gtab, const double *__restrict__ ltab,
                                                  int alpha_int, double alpha)
{
    const int lane = threadIdx.x & 31;
    const int rr = lane & 3, cc = lane >> 2;
    constexpr int NT = (16 + NW - 1) / NW;               // tasks per warp
    double tv[NT][2];
    int tcol[NT];
#pragma unroll
    for (int u = 0; u < NT; ++u) {
        const int t = w7 + u * NW;
        const int grp = t & 3, qc = (t >> 2) & 3;
        tcol[u] = jb - PR_CB + qc * 8 + cc;
        const ColRec a = sCol[tcol[u]];
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const int j = min(jb + grp * 8 + k * 4 + rr, N - 1);
            const int2 me = col_lc(sCol, j);
            const RowConst<AI> r = make_row<AI>(me.y, me.x, alpha_int, alpha);
            tv[u][k] = (t < 16) ? __dadd_rn(self_score<AI>(a.C, a.L, r, gtab, ltab), a.P) : -INFINITY;
        }
    }
    // triangle: lane = row, this warp's columns k = w7, w7+7, ...
    const int2 mt = col_lc(sCol, min(jb + lane, N - 1));
    const RowConst<AI> rt = make_row<AI>(mt.y, mt.x, alpha_int, alpha);
    constexpr int NK = (DP_JB + NW - 1) / NW;
    double w[NK];
#pragma unroll
    for (int kk = 0; kk < NK; ++kk) {
        const int k = w7 + kk * NW;
        w[kk] = 0.0;
        if (k < lane && jb + lane < N) {
            const int2 a = col_lc(sCol, jb + k);
            w[kk] = self_score<AI>(a.y, a.x, rt, gtab, ltab);
        }
    }
#pragma unroll
    for (int u = 0; u < NT; ++u) {
        const int t = w7 + u * NW;
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            double best = tv[u][k];
            int arg = tcol[u];
            merge_column_phases<4>(best, arg);
            if (cc == 0 && t < 16) {
                const int row = (t & 3) * 8 + k * 4 + rr;
                sPartV[(t >> 2) * 32 + row] = best;
                sPartA[(t >> 2) * 32 + row] = arg;
            }
        }
    }
#pragma unroll
    for (int kk = 0; kk < NK; ++kk) {
        const int k = w7 + kk * NW;
        if (k < lane && jb + lane < N) sTri[k * DP_JB + lane] = w[kk];
    }
}

// After the chain finished rows [jb, jb+32) (a full block of 32 columns from now on): least-squares tilt, tilted
// maxima, end points (fit_column_record in bound.cuh).  One warp, lane = column.
__device__ __forceinline__ void build_coarse_record(int jb, const ColRec *sCol, CoarseRec *rec, double tilt_scale_c,
                                                    double tilt_scale_l)
{
    const ColRec me = sCol[jb + (threadIdx.x & 31)];
    fit_column_record(me.C, me.L, me.P, rec, tilt_scale_c, tilt_scale_l);
}

// ---- the whole window under one hypothesis ---------------------------------------------------
// In the later rounds most windows keep every candidate: the first maximum of every row j is column j-1.  Fixing that
// hypothesis for the whole window up front makes every P known before any cell is looked at,
//     P_j = (self(j-1, j) + P_{j-1}) + pen        (block_chain_speculative's operation order),
// so the checks of all rows are independent: row j holds iff every cell i < j-1 is strictly below T_j = t_{j-1,j}
// (a tie at a smaller column would be the first maximum).  If every row holds, by induction over the rows P and
// prev = j-1 are what the block pipeline computes, bit for bit.  If row j* fails, the same induction proves every row
// before j*: the pipeline resumes at the block holding j*.
// The rows go in groups of CT_RB blocks (sT and sRowG hold one group).  Per group: (a) self(j-1, j) in parallel,
// (b) the sequential sum by one thread, (c) the column-block records of the group and, exactly, the near columns of
// every row (the previous block, the triangle, column 0), (d) far columns bounded per 32 x 32 rectangle (far_pass's
// level 1, with T_j as the row value: it is exact, so no delta_path), (e) the survivors again per 4 x 8 rectangle
// (level 2) and what survives that cell by cell.  The far levels skip rows at and past a failure already found, and a
// group with a failure ends the check.  Returns the first failing row, N if none.
constexpr int CT_RB = 16;

template <bool AI>
__device__ __forceinline__ int certify_window(const WinDpParams &p, int N, ColRec *sCol, CoarseRec *sCoarse, const double *sScal0,
                                              double *sScal1, double *sT, float4 *sRowG, double *sLbAbs, int *sSkip,
                                              unsigned short *sL1, int *sFail, int *sL1Count, double tilt_c, double tilt_l,
                                              u64 &skipped)
{
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nrb = (N - 1 + DP_JB - 1) / DP_JB;            // row blocks: rows [1 + 32k, 33 + 32k)
    if (tid == 0) { *sFail = N; *sL1Count = 0; }
    if (tid < CT_RB) sSkip[tid] = 0;
    for (int kg = 0; kg < nrb; kg += CT_RB) {
        const int r0 = 1 + DP_JB * kg, r1 = min(N, r0 + DP_JB * CT_RB), kge = min(nrb, kg + CT_RB);
        // (a)
        for (int j = r0 + tid; j < r1; j += WD_THREADS) {
            const int2 me = col_lc(sCol, j), bf = col_lc(sCol, j - 1);
            sT[j - r0] = self_score<AI>(bf.y, bf.x, make_row<AI>(me.y, me.x, p.alpha_int, p.alpha), p.gtab, p.ltab);
        }
        __syncthreads();
        // (b) sT becomes T_j; running max |P| (the scale of delta)
        if (tid == 0) {
            double P = sCol[r0 - 1].P, mx = *sScal1;
            for (int j = r0; j < r1; ++j) {
                const double t = __dadd_rn(sT[j - r0], P);
                P = __dadd_rn(t, p.pen);
                sT[j - r0] = t;
                sCol[j].P = P;
                mx = fmax(mx, fabs(P));
            }
            *sScal1 = mx;
        }
        __syncthreads();
        // (c) lane = row; the near columns j-2 .. c0 by distance (rows of a warp then gather nearby table entries)
        for (int k = kg + warp; k < kge; k += WD_WARPS) {
            const int jb = 1 + DP_JB * k;
            if (jb + DP_JB <= N) build_coarse_record(jb, sCol, sCoarse + k, tilt_c, tilt_l);
            const bool valid = jb + lane < N;
            const int j = min(jb + lane, N - 1);
            const double T = sT[j - r0];
            const int2 me = col_lc(sCol, j);
            const RowConst<AI> rme = make_row<AI>(me.y, me.x, p.alpha_int, p.alpha);
            const int c0 = k == 0 ? 0 : jb - DP_JB;
            const int dmax = j - c0, dmax_w = __reduce_max_sync(0xffffffffu, dmax);
            bool ok = fabs(T) < 1e30;                           // beyond float range the far bound has no row value
            constexpr int UN = 4;
            for (int d = 2; d <= dmax_w; d += UN) {
                double t[UN];
#pragma unroll
                for (int u = 0; u < UN; ++u) {
                    const ColRec c = sCol[max(j - d - u, 0)];
                    t[u] = d + u <= dmax ? __dadd_rn(self_score<AI>(c.C, c.L, rme, p.gtab, p.ltab), c.P) : -INFINITY;
                }
#pragma unroll
                for (int u = 0; u < UN; ++u) ok &= t[u] < T;
            }
            if (c0 > 0) {                                       // column 0 is in no column block
                const ColRec c = sCol[0];
                ok &= __dadd_rn(self_score<AI>(c.C, c.L, rme, p.gtab, p.ltab), c.P) < T;
            }
            if (valid && !ok) atomicMin(sFail, j);
            sRowG[(k - kg) * 32 + lane] = make_float4((float)T, (float)me.y, (float)me.x, 0.f);
            double ab = valid && ok ? fabs(T) : 0.0;
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) ab = fmax(ab, __shfl_xor_sync(0xffffffffu, ab, off));
            if (lane == 0) sLbAbs[k - kg] = ab;
        }
        __syncthreads();
        const double delta = (*sScal0 + *sScal1 + fabs(p.pen) * DP_JB) * 5.684341886080802e-14;   // 2^-44, as far_delta
        // (d) rectangles (row block k, column block cb < k-1) of the blocks before the first failure, flat over the threads
        {
            const int f = *sFail;
            const int kend = min(kge, f >= N ? nrb : (f - 1) / DP_JB), k1 = max(kg, 2);
            int ntot = 0;
            for (int k = k1; k < kend; ++k) ntot += k - 1;
            for (int base = 0; base < ntot; base += WD_THREADS) {
                const int e = base + tid;
                bool surv = false;
                int k = k1, cb = e;
                if (e < ntot) {
                    while (cb >= k - 1) { cb -= k - 1; ++k; }
                    const int jb = 1 + DP_JB * k, nrows = min(DP_JB, N - jb);
                    const int2 rowF = col_lc(sCol, jb), rowL = col_lc(sCol, jb + nrows - 1);
                    const CoarseRec *rec = sCoarse + cb;
                    const int4 ends = *reinterpret_cast<const int4 *>(rec);
                    const double a1 = rec->a, b1 = rec->b;
                    const double ub1 = rec->mpt + tilted_box_max<AI>(rowF.y - ends.y, rowL.y - ends.x, rowF.x - ends.w, rowL.x - ends.z,
                                                                     a1, b1, p.gtab, p.ltab, p.alpha_int, p.alpha);
                    const double m3 = tilted_row_min(sRowG + (k - kg) * 32, 0, nrows - 1, a1, b1, sLbAbs[k - kg], rowL.y, rowL.x);
                    surv = !(ub1 - m3 + delta < 0.0);                     // NaN keeps the rectangle
                    if (!surv) atomicAdd(sSkip + (k - kg), PR_CB * nrows);
                }
                const unsigned mask = __ballot_sync(0xffffffffu, surv);
                if (mask) {
                    int slot = 0;
                    if (lane == 0) slot = atomicAdd(sL1Count, __popc(mask));
                    slot = __shfl_sync(0xffffffffu, slot, 0);
                    if (surv) sL1[slot + __popc(mask & ((1u << lane) - 1u))] = (unsigned short)(((k - kg) << 8) | cb);
                }
            }
        }
        __syncthreads();
        // (e) a warp per surviving rectangle: level 2 (lane = 4 rows x 8 columns), then the cells of the surviving
        // sub-rectangles, 4 at a time (lane = row er, column ec)
        {
            const int nl1 = *sL1Count;
            const int rg = lane >> 2, q = lane & 3, er = lane >> 3, ec = lane & 7;
            for (int e = warp; e < nl1; e += WD_WARPS) {
                const int ent = sL1[e], kl = ent >> 8, cb = ent & 255;
                const int jb = 1 + DP_JB * (kg + kl), nrows = min(DP_JB, N - jb);
                const int f = __shfl_sync(0xffffffffu, *reinterpret_cast<volatile int *>(sFail), 0);
                if (f < min(jb + DP_JB, N)) continue;           // a failure in this block or before it: not needed
                const CoarseRec *rec = sCoarse + cb;
                const double a = rec->a, b = rec->b;
                const int rr0 = 4 * rg, rr1 = min(rr0 + 3, nrows - 1);
                bool surv2 = false;
                int sk = 0;
                if (rr0 < nrows) {
                    const int i0 = 1 + PR_CB * cb + PR_FB * q;
                    const int2 cF = col_lc(sCol, i0), cL = col_lc(sCol, i0 + PR_FB - 1);
                    const int2 gF = col_lc(sCol, jb + rr0), gL = col_lc(sCol, jb + rr1);
                    const double m2 = tilted_box_max<AI>(gF.y - cL.y, gL.y - cF.y, gF.x - cL.x, gL.x - cF.x, a, b,
                                                         p.gtab, p.ltab, p.alpha_int, p.alpha);
                    const double m3 = tilted_row_min(sRowG + kl * 32, rr0, rr1, a, b, sLbAbs[kl], gL.y, gL.x);
                    surv2 = !(rec->mpt8[q] + m2 - m3 + delta < 0.0);
                    if (!surv2) sk = PR_FB * (rr1 - rr0 + 1);
                }
                unsigned m = __ballot_sync(0xffffffffu, surv2);
                int bad = N;
                while (m) {
                    constexpr int UX = 4;
                    double t[UX], T[UX];
                    int row[UX];
#pragma unroll
                    for (int u = 0; u < UX; ++u) {
                        t[u] = -INFINITY;
                        T[u] = 0.0;
                        row[u] = N;
                        if (m) {
                            const int l2 = __ffs(m) - 1;
                            m &= m - 1;
                            const int r = 4 * (l2 >> 2) + er;
                            if (r < nrows) {
                                row[u] = jb + r;
                                const int2 rl = col_lc(sCol, jb + r);
                                const RowConst<AI> rc = make_row<AI>(rl.y, rl.x, p.alpha_int, p.alpha);
                                const ColRec cc = sCol[1 + PR_CB * cb + PR_FB * (l2 & 3) + ec];
                                t[u] = __dadd_rn(self_score<AI>(cc.C, cc.L, rc, p.gtab, p.ltab), cc.P);
                                T[u] = sT[jb + r - r0];
                            }
                        }
                    }
#pragma unroll
                    for (int u = 0; u < UX; ++u)
                        if (row[u] < N && !(t[u] < T[u])) bad = min(bad, row[u]);
                }
                if (bad < N) atomicMin(sFail, bad);
#pragma unroll
                for (int off = 16; off > 0; off >>= 1) sk += __shfl_xor_sync(0xffffffffu, sk, off);
                if (lane == 0 && sk) atomicAdd(sSkip + kl, sk);
            }
        }
        __syncthreads();
        const int f = *sFail;
        if (tid == 0) {                                         // skips count for the rows that stay proven only
            const int kf = f >= N ? nrb : (f - 1) / DP_JB;
            for (int k = kg; k < kge; ++k) {
                if (k < kf) skipped += (u64)sSkip[k - kg];
                sSkip[k - kg] = 0;
            }
            *sL1Count = 0;
        }
        if (f < N) return f;
    }
    return N;
}

template <bool AI, int U, int RPL, bool PRUNE>
__global__ void __launch_bounds__(WD_THREADS, 3)
window_dp_kernel(WinDpParams p)
{
    extern __shared__ __align__(16) unsigned char smem[];
    const int capr = (p.cap + 31) & ~31;
    ColRec *sCol = reinterpret_cast<ColRec *>(smem);
    double *sPartV = reinterpret_cast<double *>(sCol + capr);
    double *sTri = sPartV + NEAR_Q * 32;
    int *sPartA = reinterpret_cast<int *>(sTri + DP_JB * DP_JB);
    int *sMisc = sPartA + NEAR_Q * 32;
    unsigned short *sPrev = reinterpret_cast<unsigned short *>(sMisc + 24);
    CoarseRec *sCoarse = reinterpret_cast<CoarseRec *>(sPrev + capr);   // capr*2 bytes is a multiple of 16
    float4 *sRow = reinterpret_cast<float4 *>(sCoarse + capr / PR_CB);
    double *sFarV = reinterpret_cast<double *>(sRow + 2 * 32);          // [2][WD_FARW][32]   (sRow: [2][32], by parity of the block)
    int *sFarA = reinterpret_cast<int *>(sFarV + 2 * WD_FARW * 32);     // [2][WD_FARW][32]
    double *sScal = reinterpret_cast<double *>(sFarA + 2 * WD_FARW * 32);   // [0] magnitude of the window's largest self score, [1] max |P|, [2], [3] tilt scales, [4], [5] max |lb| of the two sRow buffers
    unsigned short *sList = reinterpret_cast<unsigned short *>(sScal + 8);
    int *sListCount = sMisc + 16;                                        // [2][4], by parity of the block
    // the back-trace runs after the DP, when these are dead
    unsigned short *sJump = reinterpret_cast<unsigned short *>(sCoarse); // capr*2 bytes <= (capr/32)*80
    unsigned char *sMark = reinterpret_cast<unsigned char *>(sTri);     // capr <= 8192 bytes

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    PROF_DECL;

    while (true) {
        PROF_T(7);
        PROF_FLUSH;
        if (tid == 0) sMisc[0] = (int)atomicAdd(p.work_counter, 1u);
        __syncthreads();
        const i64 widx = (unsigned)sMisc[0];
        if (widx >= p.nwin) break;
        const bool second = widx >= p.n_p1;          // stored from the back of the list
        const bool phase2 = second && p.skip_covered;
        const i64 w = !p.list ? p.w_begin + widx
                              : (second ? (i64)__ldg(p.list + (p.list_len - 1 - (widx - p.n_p1))) : (i64)__ldg(p.list + widx));
        if (phase2) {
            // wait for the phase-1 windows on both sides (they overlap this one).  Every phase-1 window was handed out
            // before this one, so each is finished or being worked on: no deadlock.
            if (tid == 0) {
                const i64 rel = w - p.w_begin, lo = rel - rel % p.p1_stride, hi = lo + p.p1_stride;
                const volatile unsigned char *f = p.done_flags;
                while (!f[lo] || (hi < p.list_len && !f[hi])) __nanosleep(200);
                __threadfence();
                // fast path: both neighbours kept every one of their candidates (flag bit 1) and together they cover this
                // window, so every candidate of this window is a survivor already -- no need to read them
                i64 skip_cells = -1;
                if (hi < p.list_len && (f[lo] & 2) && (f[hi] & 2)) {
                    i64 s0, e0, s1, e1, s2, e2;
                    window_range(p.geom, w, s0, e0);
                    window_range(p.geom, p.w_begin + lo, s1, e1);
                    window_range(p.geom, p.w_begin + hi, s2, e2);
                    if (s1 <= s0 && e1 >= s2 && e2 >= e0) skip_cells = (e0 - s0) * (e0 - s0 - 1) / 2;
                }
                if (skip_cells >= 0) {
                    atomicAdd(p.cells, (u64)skip_cells);
                    atomicAdd(p.cells_skipped, (u64)skip_cells);
                }
                sMisc[1] = skip_cells >= 0;
            }
            __syncthreads();
            if (sMisc[1]) continue;
        }
        int kept_all = 1;                           // phase 2: are all candidates of this window survivors already?

        // ---- (A) candidates of the window, filtered, re-based ---------------------------------
        i64 st, en;
        window_range(p.geom, w, st, en);
        const int nq = (int)(en - st);
        const i64 first = p.cand ? (i64)__ldg(p.cand + st) : st;
        const i64 last = p.cand ? (i64)__ldg(p.cand + en - 1) : en - 1;
        const i64 cg_first = p.cand ? __ldg(p.cgc + st) : __ldg(p.cg + first);
        const bool all_zero = (p.constraint == PASIO_CONSTRAINT_ZEROS) && ((p.cand ? __ldg(p.cgc + en - 1) : __ldg(p.cg + last)) == cg_first);
        int count = 0;
        const bool by_words = !p.cand && p.constraint == PASIO_CONSTRAINT_CONSTANTS;
        if (by_words) {
            // all positions are candidates (round 1): the survivors of the NotConstant filter are the set
            // bits of the change-point bitmap inside [first, last], plus both ends -- one thread per word
            const i64 w0 = first >> 5, w1 = last >> 5;
            const int nwords = (int)(w1 - w0 + 1);
            for (int base = 0; base < nwords; base += WD_THREADS) {
                const int t = base + tid;
                unsigned word = 0;
                if (t < nwords) {
                    word = __ldg(p.cpbits + w0 + t);
                    if (t == 0) word = (word & (0xffffffffu << (first & 31))) | (1u << (first & 31));
                    if (t == nwords - 1) word = (word & (0xffffffffu >> (31 - (last & 31)))) | (1u << (last & 31));
                }
                int incl = __popc(word);
                const int mine = incl;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const int o = __shfl_up_sync(0xffffffffu, incl, d);
                    if (lane >= d) incl += o;
                }
                if (lane == 31) sMisc[4 + warp] = incl;
                __syncthreads();
                int woff = 0, tot = 0;
#pragma unroll
                for (int w2 = 0; w2 < WD_WARPS; ++w2) {
                    const int c = sMisc[4 + w2];
                    if (w2 < warp) woff += c;
                    tot += c;
                }
                int k = count + woff + incl - mine;
                const i64 pos0 = (w0 + t) << 5;
                while (word) {
                    const i64 pos = pos0 + (__ffs(word) - 1);
                    word &= word - 1;
                    sCol[k].L = (int)(pos - first);
                    sCol[k].C = (int)(__ldg(p.cg + pos) - cg_first);
                    ++k;
                }
                count += tot;
                __syncthreads();
            }
        }
        for (int base = 0; !by_words && base < nq; base += WD_THREADS) {
            const int q = base + tid;
            i64 pos = 0;
            bool take = false;
            if (q < nq) {
                pos = p.cand ? (i64)__ldg(p.cand + st + q) : st + q;
                if (q == 0 || q == nq - 1 || p.constraint == PASIO_CONSTRAINT_NONE) take = true;
                else if (p.constraint == PASIO_CONSTRAINT_CONSTANTS) take = bit_test(p.cpbits, pos);
                else take = !all_zero;
                if (phase2 && !((__ldcg(p.keepbits + (pos >> 5)) >> (pos & 31)) & 1u)) kept_all = 0;
            }
            const unsigned bal = __ballot_sync(0xffffffffu, take);
            if (lane == 0) sMisc[4 + warp] = __popc(bal);
            __syncthreads();
            int woff = 0, tot = 0;
#pragma unroll
            for (int w2 = 0; w2 < WD_WARPS; ++w2) {
                const int c = sMisc[4 + w2];
                if (w2 < warp) woff += c;
                tot += c;
            }
            if (take) {
                const int k = count + woff + __popc(bal & ((1u << lane) - 1u));
                sCol[k].L = (int)(pos - first);
                sCol[k].C = (int)((p.cand ? __ldg(p.cgc + st + q) : __ldg(p.cg + pos)) - cg_first);
            }
            count += tot;
            __syncthreads();
        }
        const int N = count;
        PROF_T(0);
        if (phase2 && __syncthreads_and(kept_all)) {
            // the window's survivors are a subset of its candidates, and those are all marked: nothing to add
            // (sliding_window_reducer.py:22-29 takes the UNION over the windows).  Its cells count as skipped.
            if (tid == 0) {
                const u64 c = (u64)N * (u64)(N - 1) / 2;
                atomicAdd(p.cells, c);
                atomicAdd(p.cells_skipped, c);
            }
            continue;
        }

        // ---- (B) DP ---------------------------------------------------------------------------
        if (tid == 0) { sCol[0].P = 0.0; sPrev[0] = 0; }
        __syncthreads();
        u64 skipped = 0;
        if (PRUNE && tid == 0) {
            // largest |G| + s*Lg any cell of this window can reach (both monotone): the scale of delta
            const ColRec z = sCol[N - 1];
            const int x = z.C + (AI ? p.alpha_int : 0);
            sScal[0] = fabs(__ldg(p.gtab + x)) + ((double)z.C + p.alpha) * fabs(__ldg(p.ltab + z.L)) + 1.0;
            sScal[1] = 0.0;
            sScal[2] = (double)z.C + p.alpha;       // |a*C| and |b*L| of a tilt stay below |a|*this and |b|*that
            sScal[3] = (double)z.L;
        }
        // finished rows [jb, jb+32) become a block of 32 columns; running max |P| (scale of delta).  Warp 0 only.
        auto finish_block = [&](int jb) {
            if (jb + DP_JB <= N) build_coarse_record(jb, sCol, sCoarse + (jb - 1) / PR_CB, sScal[2], sScal[3]);
            double ab = jb + lane < N ? fabs(sCol[jb + lane].P) : 0.0;
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) ab = fmax(ab, __shfl_xor_sync(0xffffffffu, ab, off));
            if (lane == 0) sScal[1] = fmax(sScal[1], ab);
        };
        auto far_delta = [&]() { return (sScal[0] + sScal[1] + fabs(p.pen) * DP_JB) * 5.684341886080802e-14; };   // 2^-44
        // warp 0: lower bounds of the rows of block [jbn, jbn+32) for the far pass that runs next
        // warp 0: lower bounds of the rows of block [jbn, jbn+32) for the far pass that runs one phase later, from the P of the
        // rows before jbp (jbp = jbn - 32: the block between is still to be chained).  Buffers by parity of the block.
        auto prepare_rows = [&](int jbn) {
            const int par = ((jbn - 1) / DP_JB) & 1;
            const double delta_path = (sScal[0] + sScal[1] + fabs(p.pen) * DP_JB) * 1.8189894035458565e-12;   // 2^-39
            compute_row_lb<AI>(jbn - DP_JB, jbn, N, sCol, sRow + 32 * par, sScal + 4 + par, delta_path, p.pen, p.gtab, p.ltab,
                               p.alpha_int, p.alpha);
            if (lane == 0) { sListCount[4 * par] = 0; sListCount[4 * par + 1] = 0; sListCount[4 * par + 2] = 0; }
        };
        auto run_far = [&](int jbf) {               // warps 1..7: far pass of the block starting at row jbf
            const int kf = (jbf - 1) / DP_JB, par = kf & 1;
            skipped += far_pass<AI>(jbf, N, kf - 1, sCol, sCoarse, sRow + 32 * par, sScal[4 + par], sList, sList + capr,
                                    sList + capr + capr / PR_CB + 8, sListCount + 4 * par, sFarV + (par * WD_FARW + warp - 1) * 32,
                                    sFarA + (par * WD_FARW + warp - 1) * 32,
                                    far_delta(), p.gtab, p.ltab, p.alpha_int, p.alpha PROF_PASS);
        };
        int jb = 1;
        // the first two blocks (and everything without pruning, and small windows, where bounding costs more than
        // it saves): plain block steps over all columns
        // (with all positions as candidates -- round 1 -- most candidates are noise, the arg-max is far away and the
        // bounds cut little: plain sweeps are faster there)
        const bool pipelined = PRUNE && N > PR_MIN_N && p.cand != nullptr;
        bool passed = false;
        if (pipelined && p.certify) {
            __syncthreads();                                // sScal
            const int f = certify_window<AI>(p, N, sCol, sCoarse, sScal, sScal + 1, sFarV, reinterpret_cast<float4 *>(sTri), sPartV,
                                             sPartA, sList, sMisc + 2, sMisc + 3, sScal[2], sScal[3], skipped);
            passed = f >= N;
            // resume at the block holding the failure; rows before it are final (in the first two blocks: from the start)
            const int kf = (f - 1) / DP_JB, res = passed || kf < 2 ? 1 : 1 + DP_JB * kf;
            for (int j = 1 + tid; j < res; j += WD_THREADS) sPrev[j] = (unsigned short)(j - 1);
            if (warp == 0 && !passed) {                     // max |P| of the finished rows, as finish_block leaves it
                double ab = 0.0;
                for (int j = 1 + lane; j < res; j += 32) ab = fmax(ab, fabs(sCol[j].P));
#pragma unroll
                for (int off = 16; off > 0; off >>= 1) ab = fmax(ab, __shfl_xor_sync(0xffffffffu, ab, off));
                if (lane == 0) sScal[1] = ab;
            }
            if (tid == 0) {
                atomicAdd(p.certify_stats + (passed ? 0 : 1), 1ull);
                if (res > 1) atomicAdd(p.certify_stats + 2, (u64)(res - 1));
            }
            jb = passed ? N : res;
            __syncthreads();
        }
        for (; jb < N && (!pipelined || jb < 1 + 2 * DP_JB); jb += DP_JB) {
            dp_block_step<AI, WD_WARPS, U, RPL>(jb, N, 0, sCol, sPrev, nullptr, sPartV, sPartA, sTri,
                                                p.gtab, p.ltab, p.alpha_int, p.alpha, p.pen, -INFINITY, 0, 0);
            if (pipelined && warp == 0) finish_block(jb);
        }
        PROF_T(6);
        if (pipelined && jb < N) {
            // Software pipeline over the remaining blocks k = 2, 3, ...:
            //   phase X(k): all warps sweep the nearest 32 columns (block k-1) and the triangle of block k
            //   phase Y(k): warp 0 resolves the chain of block k, turns the block into a column block and prepares the row
            //               bounds of block k+2; warps 1..7 run the far pass of block k+1 (columns up to block k-1, row
            //               bounds prepared one phase earlier)
            int spec_wait = 0, spec_back = 1;       // warp 0: blocks to sit out before speculating again, and the next back-off
            if (warp == 0) prepare_rows(jb);
            __syncthreads();
            if (warp > 0) run_far(jb);
            else if (jb + DP_JB < N) prepare_rows(jb + DP_JB);
            __syncthreads();
            for (; jb < N; jb += DP_JB) {
                const int k = (jb - 1) / DP_JB, buf = k & 1;
                near_tri_farwarps<AI, WD_WARPS>(warp, jb, N, sCol, sPartV, sPartA, sTri, p.gtab, p.ltab, p.alpha_int, p.alpha);
                PROF_T(1);
                __syncthreads();
                PROF_T(6);
                if (warp == 0) {
                    // far results first (smaller columns; the warps' column sets interleave, hence the index-aware
                    // merge), then the near chunks in ascending order, then the triangle
                    double fbest = -INFINITY;
                    int farg = 0;
#pragma unroll
                    for (int w2 = 0; w2 < WD_FARW; ++w2) {
                        const double v = sFarV[(buf * WD_FARW + w2) * 32 + lane];
                        const int a = sFarA[(buf * WD_FARW + w2) * 32 + lane];
                        if (v > fbest || (v == fbest && a < farg)) { fbest = v; farg = a; }
                    }
                    const double ib = jb + lane < N ? fbest : -INFINITY;
                    const int ia = jb + lane < N ? farg : 0;
                    // speculate unless it just failed: a failure costs a fifth of a chain, so back off (1, 2, 4, ... 16
                    // blocks) where candidates are still being dropped and return to it where they are not
                    bool resolved = false;
                    if (p.speculate && spec_wait == 0) {
                        resolved = block_chain_speculative<NEAR_Q>(jb, N, sCol, sPrev, sPartV, sPartA, sTri, p.pen, ib, ia);
                        if (resolved) spec_back = 1;
                        else { spec_wait = spec_back; spec_back = min(spec_back * 2, 16); }
                    } else if (spec_wait > 0) {
                        --spec_wait;
                    }
                    if (!resolved) block_chain<NEAR_Q>(jb, N, sCol, sPrev, nullptr, sPartV, sPartA, sTri, p.pen, ib, ia, 0, nullptr);
                    __syncwarp();
                    finish_block(jb);
                    if (jb + 2 * DP_JB < N) prepare_rows(jb + 2 * DP_JB);
                } else if (jb + DP_JB < N) {
                    run_far(jb + DP_JB);
                }
                PROF_T(2);
                __syncthreads();
                PROF_T(7);
            }
        }

        // ---- (C) back-trace by pointer doubling, scatter survivors ----------------------------
        for (int k = tid; k < N; k += WD_THREADS) sMark[k] = passed || k == N - 1;
        __syncthreads();
        unsigned short *ja = sPrev, *jb2 = sJump;
        for (int reach = passed ? N : 1; reach < N; reach <<= 1) {
            // nodes within `reach` hops of the end are marked; ja[k] is the node 'reach' hops before k
            for (int k = tid; k < N; k += WD_THREADS)
                if (sMark[k]) sMark[ja[k]] = 1;
            for (int k = tid; k < N; k += WD_THREADS) jb2[k] = ja[ja[k]];
            __syncthreads();
            unsigned short *t = ja; ja = jb2; jb2 = t;
        }
        int every = N == nq;                         // did every candidate of the window (none filtered) survive?
        for (int k = tid; k < N; k += WD_THREADS) {
            if (sMark[k]) {
                const i64 pos = first + sCol[k].L;
                atomicOr(p.keepbits + (pos >> 5), 1u << (pos & 31));
            } else {
                every = 0;
            }
        }
        if (!second && p.skip_covered && p.n_p1 < p.nwin) {             // phase-2 windows wait for this
            __threadfence();
            every = __syncthreads_and(every);
            if (tid == 0) {
                __threadfence();
                *reinterpret_cast<volatile unsigned char *>(p.done_flags + (w - p.w_begin)) = every ? 3 : 1;
            }
        }
        if (tid == 0) atomicAdd(p.cells, (u64)N * (u64)(N - 1) / 2);
        if (PRUNE) {
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) skipped += __shfl_xor_sync(0xffffffffu, skipped, off);
            if (lane == 0 && skipped) atomicAdd(p.cells_skipped, skipped);
        }
        __syncthreads();
    }
}

// ---- small windows: one WARP per window ----------------------------------------------------------
// Round 1 of the default pipeline is ~200 000 windows of ~100 candidates: a few thousand cells each, but every
// window is a chain of ~100 dependent row steps.  With a CTA per window only three such chains run per SM; here
// every warp owns a window (40 per SM), so the SM is busy with other windows while one waits on its chain.
// Same arithmetic, same order and the same first-maximum rule as the CTA kernel: 16-row block steps, a lane
// sweeps every second finished column for its row, the 16 x 16 triangle is resolved in order by shuffles.
// Two size classes: up to 160 candidates (8 windows per CTA, 5 CTAs per SM) and up to 512 (4 per CTA, 4 CTAs per SM).
constexpr int SW_JB = 16;
constexpr int SW_SMALL_N = WD_SMALL_MAX_CANDIDATES, SW_SMALL_WARPS = 8, SW_SMALL_CTAS = 5;
constexpr int SW_MEDIUM_N = WD_MEDIUM_MAX_CANDIDATES, SW_MEDIUM_WARPS = 4, SW_MEDIUM_CTAS = 4;

template <int MAXN>
struct __align__(16) SmallWin {
    ColRec col[MAXN];
    double tri[SW_JB * SW_JB];
    unsigned short prev[MAXN];
    unsigned char mark[MAXN];
};

template <bool AI, int MAXN, int NWARPS, int CTAS, int U, bool LGS>
__global__ void __launch_bounds__(NWARPS * 32, CTAS)
small_window_dp_kernel(WinDpParams p)
{
    extern __shared__ __align__(16) unsigned char smem[];
    const int lane = threadIdx.x & 31;
    SmallWin<MAXN> &W = reinterpret_cast<SmallWin<MAXN> *>(smem)[threadIdx.x >> 5];
    u64 my_cells = 0;
    // LGS (all positions are candidates, i.e. round 1: no length exceeds the window size): the log table's first
    // p.n_lg entries are copied to shared memory once per CTA and every Lg look-up of the DP reads that copy
    const double *lgt = p.ltab;
    if (LGS) {
        double *sLg = reinterpret_cast<double *>(smem + sizeof(SmallWin<MAXN>) * NWARPS);
        for (int k = threadIdx.x; k < p.n_lg; k += NWARPS * 32) sLg[k] = __ldg(p.ltab + k);
        __syncthreads();
        lgt = sLg;
    }

    while (true) {
        unsigned widx = 0;
        if (lane == 0) widx = atomicAdd(p.work_counter, 1u);
        widx = __shfl_sync(0xffffffffu, widx, 0);
        if ((i64)widx >= p.nwin) break;
        const i64 w = __ldg(p.list + widx);

        // ---- (A) candidates of the window, filtered, re-based ----
        i64 st, en;
        window_range(p.geom, w, st, en);
        const int nq = (int)(en - st);
        const i64 first = p.cand ? (i64)__ldg(p.cand + st) : st;
        const i64 last = p.cand ? (i64)__ldg(p.cand + en - 1) : en - 1;
        const i64 cg_first = p.cand ? __ldg(p.cgc + st) : __ldg(p.cg + first);
        const bool all_zero = (p.constraint == PASIO_CONSTRAINT_ZEROS) && ((p.cand ? __ldg(p.cgc + en - 1) : __ldg(p.cg + last)) == cg_first);
        int count = 0;
        if (!p.cand && p.constraint == PASIO_CONSTRAINT_CONSTANTS) {
            const i64 w0 = first >> 5, w1 = last >> 5;
            const int nwords = (int)(w1 - w0 + 1);
            for (int base = 0; base < nwords; base += 32) {
                const int t = base + lane;
                unsigned word = 0;
                if (t < nwords) {
                    word = __ldg(p.cpbits + w0 + t);
                    if (t == 0) word = (word & (0xffffffffu << (first & 31))) | (1u << (first & 31));
                    if (t == nwords - 1) word = (word & (0xffffffffu >> (31 - (last & 31)))) | (1u << (last & 31));
                }
                int incl = __popc(word);
                const int mine = incl;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const int o = __shfl_up_sync(0xffffffffu, incl, d);
                    if (lane >= d) incl += o;
                }
                int k = count + incl - mine;
                const i64 pos0 = (w0 + t) << 5;
                while (word) {
                    const i64 pos = pos0 + (__ffs(word) - 1);
                    word &= word - 1;
                    W.col[k].L = (int)(pos - first);
                    W.col[k].C = (int)(__ldg(p.cg + pos) - cg_first);
                    ++k;
                }
                count += __shfl_sync(0xffffffffu, incl, 31);
            }
        } else {
            for (int base = 0; base < nq; base += 32) {
                const int q = base + lane;
                i64 pos = 0;
                bool take = false;
                if (q < nq) {
                    pos = p.cand ? (i64)__ldg(p.cand + st + q) : st + q;
                    if (q == 0 || q == nq - 1 || p.constraint == PASIO_CONSTRAINT_NONE) take = true;
                    else if (p.constraint == PASIO_CONSTRAINT_CONSTANTS) take = bit_test(p.cpbits, pos);
                    else take = !all_zero;
                }
                const unsigned bal = __ballot_sync(0xffffffffu, take);
                if (take) {
                    const int k = count + __popc(bal & ((1u << lane) - 1u));
                    W.col[k].L = (int)(pos - first);
                    W.col[k].C = (int)((p.cand ? __ldg(p.cgc + st + q) : __ldg(p.cg + pos)) - cg_first);
                }
                count += __popc(bal);
            }
        }
        const int N = count;
        if (lane == 0) { W.col[0].P = 0.0; W.prev[0] = 0; }
        __syncwarp();

        // ---- (B) DP, 16 rows per step: lane = (row r, column phase ph) ----
        const int r = lane & 15, ph = lane >> 4;
        for (int jb = 1; jb < N; jb += SW_JB) {
            const ColRec me = W.col[min(jb + r, N - 1)];
            RowConst<AI> rc[1] = {make_row<AI>(me.C, me.L, p.alpha_int, p.alpha)};
            double best[1] = {-INFINITY};
            int arg[1] = {ph};
            sweep_columns<AI, U, 1, LGS>(0, jb, ph, 2, W.col, rc, p.gtab, lgt, best, arg);
            {   // the two column phases of a row: larger value, equal values keep the smaller column
                const double ob = __shfl_xor_sync(0xffffffffu, best[0], 16);
                const int oa = __shfl_xor_sync(0xffffffffu, arg[0], 16);
                if (ob > best[0] || (ob == best[0] && oa < arg[0])) { best[0] = ob; arg[0] = oa; }
            }
            // triangle self scores (independent of P)
            for (int k = ph; k < r; k += 2)
                if (jb + r < N) {
                    const ColRec a = W.col[jb + k];
                    W.tri[k * SW_JB + r] = self_score<AI, LGS>(a.C, a.L, rc[0], p.gtab, lgt);
                }
            __syncwarp();
            double bst = best[0], mine = 0.0;
            int ag = arg[0];
            const int rows = min(SW_JB, N - jb);
#pragma unroll 4
            for (int k = 0; k < rows; ++k) {
                const double pf = __dadd_rn(bst, p.pen);          // prefix_scores[j] = max + segment_creation_cost
                const double pk = __shfl_sync(0xffffffffu, pf, k);
                if (r == k) mine = pf;
                if (r > k) {
                    const double t = __dadd_rn(W.tri[k * SW_JB + r], pk);
                    if (t > bst) { bst = t; ag = jb + k; }
                }
            }
            if (lane < SW_JB && jb + r < N) {
                W.col[jb + r].P = mine;
                W.prev[jb + r] = (unsigned short)ag;
            }
            __syncwarp();
        }

        // ---- (C) back-trace, scatter survivors ----
        for (int k = lane; k < N; k += 32) W.mark[k] = 0;
        __syncwarp();
        if (lane == 0) {
            int k = N - 1;
            while (true) {
                W.mark[k] = 1;
                if (k == 0) break;
                k = W.prev[k];
            }
        }
        __syncwarp();
        for (int k = lane; k < N; k += 32)
            if (W.mark[k]) {
                const i64 pos = first + W.col[k].L;
                atomicOr(p.keepbits + (pos >> 5), 1u << (pos & 31));
            }
        my_cells += (u64)N * (u64)(N - 1) / 2;
        __syncwarp();
    }
    if (lane == 0 && my_cells) atomicAdd(p.cells, my_cells);
}

}  // namespace

int small_window_max_candidates() { return SW_SMALL_N; }
int medium_window_max_candidates() { return SW_MEDIUM_N; }

int window_dp_max_candidates(pasio_ctx *ctx)
{
    int cap = 32;
    while (cap + 32 <= 8192 && window_smem_bytes(cap + 32) <= (size_t)ctx->smem_optin) cap += 32;
    return cap;
}

int launch_window_dp(pasio_ctx *ctx, i64 nwin, int wsize, int wshift, int constraint, i64 w_begin, bool keep_cell_counters)
{
    WinDpParams p;
    p.geom = make_geom(ctx, wsize, wshift);
    p.nwin = nwin;
    p.cand = cur_cand(ctx);
    p.cg = ctx->cg.as<i64>();
    p.cgc = cur_cand_cg(ctx);
    p.cpbits = ctx->cpbits.as<uint32_t>();
    p.keepbits = ctx->keepbits.as<uint32_t>();
    p.gtab = ctx->tab[ctx->alpha_is_int ? PASIO_TAB_LGAMMA : PASIO_TAB_LGAMMA_ALPHA].as<double>();
    p.ltab = ctx->tab[PASIO_TAB_LOG].as<double>();
    p.constraint = constraint;
    p.alpha_int = (int)ctx->alpha_int;
    p.alpha = ctx->alpha;
    p.pen = ctx->pen;
    i64 cap = (i64)wsize + 1;
    if (cap > ctx->m) cap = ctx->m;
    if (cap > 8192 || window_smem_bytes((int)cap) > (size_t)ctx->smem_optin)
        return pasio_fail(ctx, PASIO_E_TOO_LARGE, "window of %lld candidates does not fit one CTA's shared memory (max %d)",
                          (long long)cap, window_dp_max_candidates(ctx));
    p.cap = (int)cap;
    p.cells = ctx->scalars.as<u64>() + 10;
    p.cells_skipped = ctx->scalars.as<u64>() + 12;
    p.work_counter = ctx->scalars.as<unsigned>() + 2 * 11;   // scalars[11]
    p.w_begin = w_begin;
    p.certify_stats = ctx->scalars.as<u64>() + 16;
    if (keep_cell_counters) CUDA_TRY(ctx, cudaMemsetAsync(ctx->scalars.as<u64>() + 11, 0, 8, ctx->stream));   // work counter only
    else {
        CUDA_TRY(ctx, cudaMemsetAsync(ctx->scalars.as<u64>() + 10, 0, 24, ctx->stream));
        CUDA_TRY(ctx, cudaMemsetAsync(p.certify_stats, 0, 24, ctx->stream));
    }
    CUDA_TRY(ctx, cudaMemsetAsync(ctx->scalars.as<u64>() + 15, 0, 8, ctx->stream));    // work counters of the warp-per-window kernels

    // The work lists of the prepass (launch_window_prepass with classification).  The CTA-per-window kernel is
    // submitted first, on the main (high-priority) stream; the warp-per-window kernels follow on the low-priority side
    // stream and fill the SMs as the persistent CTAs of the big kernel run out of windows.  All of them only OR bits
    // into the survivor bitmap.
    static const int small_env = getenv("PASIO_WD_SMALL") ? atoi(getenv("PASIO_WD_SMALL")) : 1;
    const int phase_env = ctx->tune[PASIO_TUNE_WINDOW_PHASES];
    const bool use_lists = small_env && ctx->n_small + ctx->n_medium + ctx->n_large == nwin;
    const i64 n_small = use_lists ? ctx->n_small : 0, n_medium = use_lists ? ctx->n_medium : 0;
    const i64 n_large = use_lists ? ctx->n_large : nwin;
    p.list = use_lists ? ctx->win_large.as<int32_t>() : nullptr;     // PASIO_WD_SMALL=0 (experiments): every window through the CTA kernel
    p.nwin = n_large;
    p.list_len = nwin;
    p.n_p1 = use_lists ? ctx->n_large_p1 : n_large;
    p.skip_covered = phase_env;                                       // PASIO_WD_PHASES=0 (experiments): no window is skipped
    p.speculate = ctx->tune[PASIO_TUNE_WINDOW_SPECULATE];
    // The check pays where most windows keep every candidate.  The previous round on the same candidates predicts that:
    // on chr1, round 2 removes 10 % and round 3 only 0.3 %, after which most windows pass (DESIGN K4).
    const int certify_env = ctx->tune[PASIO_TUNE_WINDOW_CERTIFY];
    p.certify = certify_env >= 2 ||
                (certify_env == 1 && ctx->prev_round_in > 0 && (ctx->prev_round_in - ctx->prev_round_out) * 100 < ctx->prev_round_in);
    p.done_flags = ctx->win_flags.as<unsigned char>();
    p.p1_stride = wshift > 0 && wsize / wshift > 1 ? wsize / wshift : 1;
    if (!use_lists) p.skip_covered = 0;
    ctx->n_small = ctx->n_medium = ctx->n_large = ctx->n_large_p1 = -1;           // the lists are consumed
    TimingScope ts_all(ctx, TF_WINDOW_DP, 0);      // one span over all window kernels of the round (they overlap)
    // a handful of small windows (the tail windows of the later rounds) run beside the big kernel on the side stream;
    // when there are many (round 1) the kernels are faster one after the other, the longest chains first
    const bool fork = n_small + n_medium > 0 && n_small + n_medium <= 64;
    const bool serial_small = n_small + n_medium > 64;
    if (fork) CUDA_TRY(ctx, cudaEventRecord(ctx->ev_fork, ctx->stream));        // the side stream waits for the resets only

    auto launch_small = [&](auto kern, const int32_t *list, i64 n, int nwarps, int ctas, size_t smem_bytes, unsigned *counter,
                            cudaStream_t stream) -> int {
        if (n <= 0) return PASIO_OK;
        WinDpParams ps = p;
        ps.list = list;
        ps.nwin = n;
        ps.n_p1 = n;
        ps.work_counter = counter;
        CUDA_TRY(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes));
        int resident = ctas;                          // persistent CTAs: one resident wave (fewer fit with the log table on board)
        CUDA_TRY(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&resident, kern, nwarps * 32, smem_bytes));
        if (resident < 1) resident = 1;
        if (resident > ctas) resident = ctas;
        i64 g = (n + nwarps - 1) / nwarps;
        if (g > (i64)ctx->sm_count * resident) g = (i64)ctx->sm_count * resident;
        ctx->fam_launches[TF_WINDOW_DP] += 1;
        kern<<<(unsigned)g, nwarps * 32, smem_bytes, stream>>>(ps);
        CUDA_TRY(ctx, cudaGetLastError());
        return PASIO_OK;
    };
    // round 1 (all positions are candidates): lengths stay below the window size, so the log table fits shared memory
    static const int lgs_env = getenv("PASIO_WD_LGS") ? atoi(getenv("PASIO_WD_LGS")) : 0;   // measured slower (5.50 vs 5.19 ms for round 1 of chr1, profiles/r02_rounds_lgs*.txt): off
    const bool lgs = lgs_env && p.cand == nullptr && (i64)wsize + 2 <= 4096 && ctx->ntab[PASIO_TAB_LOG] >= (i64)wsize + 2;
    p.n_lg = lgs ? wsize + 2 : 0;
    const size_t lg_bytes = (size_t)((p.n_lg + 1) & ~1) * 8;
    auto launch_small_kernels = [&](cudaStream_t stream) -> int {
        unsigned *c_small = ctx->scalars.as<unsigned>() + 2 * 15, *c_medium = c_small + 1;     // scalars[15]
        const size_t sm_small = sizeof(SmallWin<SW_SMALL_N>) * SW_SMALL_WARPS + lg_bytes,
                     sm_medium = sizeof(SmallWin<SW_MEDIUM_N>) * SW_MEDIUM_WARPS + lg_bytes;
#define PASIO_SMALL_LAUNCH(AIV, LGV)                                                                                                          \
        PASIO_TRY(launch_small(small_window_dp_kernel<AIV, SW_SMALL_N, SW_SMALL_WARPS, SW_SMALL_CTAS, 4, LGV>, ctx->win_small.as<int32_t>(),   \
                               n_small, SW_SMALL_WARPS, SW_SMALL_CTAS, sm_small, c_small, stream));                                            \
        PASIO_TRY(launch_small(small_window_dp_kernel<AIV, SW_MEDIUM_N, SW_MEDIUM_WARPS, SW_MEDIUM_CTAS, 8, LGV>, ctx->win_medium.as<int32_t>(), \
                               n_medium, SW_MEDIUM_WARPS, SW_MEDIUM_CTAS, sm_medium, c_medium, stream));
        if (ctx->alpha_is_int) {
            if (lgs) { PASIO_SMALL_LAUNCH(true, true) } else { PASIO_SMALL_LAUNCH(true, false) }
        } else {
            if (lgs) { PASIO_SMALL_LAUNCH(false, true) } else { PASIO_SMALL_LAUNCH(false, false) }
        }
#undef PASIO_SMALL_LAUNCH
        return PASIO_OK;
    };
    if (serial_small) PASIO_TRY(launch_small_kernels(ctx->stream));

    i64 grid = 0;
    if (n_large > 0) {
        const size_t smem = window_smem_bytes(p.cap);
        // PASIO_WD_PRUNE=0 disables the exact far-column pruning (experiments / cross-checks)
        const int prune_env = ctx->tune[PASIO_TUNE_WINDOW_PRUNE];
        const bool prune = prune_env != 0 && ctx->alpha >= 0.0009765625;   // tiny alpha: lgamma(alpha) dwarfs the delta scale; alpha = 0: G[0] = inf
        void (*kern)(WinDpParams);
        if (ctx->alpha_is_int) kern = prune ? window_dp_kernel<true, 4, 2, true> : window_dp_kernel<true, 4, 2, false>;
        else kern = prune ? window_dp_kernel<false, 4, 2, true> : window_dp_kernel<false, 4, 2, false>;
        CUDA_TRY(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        int per_sm = 0;
        CUDA_TRY(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, WD_THREADS, smem));
        if (per_sm < 1) per_sm = 1;
#ifdef PASIO_WD_PROF
        if (getenv("PASIO_WD_CTAS") && atoi(getenv("PASIO_WD_CTAS")) < per_sm) per_sm = atoi(getenv("PASIO_WD_CTAS"));
#endif
        grid = (i64)ctx->sm_count * per_sm;     // persistent CTAs: one resident wave
        if (grid > n_large) grid = n_large;
        if (grid < 1) grid = 1;
        ctx->fam_launches[TF_WINDOW_DP] += 1;
        kern<<<(unsigned)grid, WD_THREADS, smem, ctx->stream>>>(p);
        CUDA_TRY(ctx, cudaGetLastError());
    }
    if (fork) {
        CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->stream2, ctx->ev_fork, 0));
        PASIO_TRY(launch_small_kernels(ctx->stream2));
        CUDA_TRY(ctx, cudaEventRecord(ctx->ev_join, ctx->stream2));
        CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_join, 0));
    }
#ifdef PASIO_WD_PROF
    {
        cudaStreamSynchronize(ctx->stream);
        unsigned long long h[16], z[16] = {0};
        cudaMemcpyFromSymbol(h, g_wd_prof, sizeof h);
        cudaMemcpyToSymbol(g_wd_prof, z, sizeof z);
        static const char *names[8] = {"compact", "X:work", "Y:work(chain|far L3)", "far:listwait", "far:L1", "far:L2", "wait@X+plain", "wait@Y+rest"};
        for (int side = 0; side < 2; ++side) {
            double tot = 0;
            for (int i = 0; i < 8; ++i) tot += (double)h[8 * side + i];
            fprintf(stderr, "[wd_prof %s] nwin=%lld grid=%lld:", side ? "warp1" : "warp0", (long long)nwin, (long long)grid);
            for (int i = 0; i < 8; ++i) if (h[8 * side + i]) fprintf(stderr, " %s=%.1f%%", names[i], 100.0 * (double)h[8 * side + i] / tot);
            fprintf(stderr, " | cycles/CTA=%.3g\n", tot / (double)grid);
        }
    }
#endif
    return PASIO_OK;
}
