// The DP cell and the in-CTA block step shared by the batched window kernel (K4) and the
// diagonal step of the exact kernel (K3).
//
// One cell restates, in the reference's operation order (SURVEY 3.3),
//   LogMarginalLikelyhood{Int,Real}AlphaComputer.all_suffixes_self_score
//     /root/reference/src/pasio/log_marginal_likelyhood.py:105-115 (int alpha), :121-132 (real alpha)
//   + the row update of SquareSplitter.split_without_normalizations
//     /root/reference/src/pasio/splitters/square_splitter.py:84-94
//       s    = (alpha + C_j) - C_i
//       self = G[s] - s * Lg[L_j - L_i]          (un-fused DMUL then DADD, like numpy's two ufunc loops)
//       t    = self + P_i
//       P_j  = max_i t  + segment_creation_cost,  prev_j = first index of the maximum (np.argmax)
// G and Lg are host-built tables (numpy/scipy values), so the device does no transcendental math.
#pragma once
#include "common.cuh"

// Flags between the CTAs of a cooperatively launched pipeline (K3 exact_dp.cu, K9 regularized_exact.cu): a CTA waits
// until *flag >= target, then reads what was published before it; publish() makes the CTA's earlier writes visible first.
__device__ __forceinline__ int ld_flag(const int *p) { return *reinterpret_cast<const volatile int *>(p); }
__device__ __forceinline__ void st_flag(int *p, int v) { *reinterpret_cast<volatile int *>(p) = v; }

__device__ __forceinline__ void wait_at_least(const int *flag, int target)
{
    if (threadIdx.x == 0) {
        while (ld_flag(flag) < target) __nanosleep(40);
        __threadfence();
    }
    __syncthreads();
}
__device__ __forceinline__ void publish(int *flag, int value)
{
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        st_flag(flag, value);
    }
}

// Per-row constants.  AI = integer alpha (table index includes alpha, s is that integer);
// real alpha: table index is the raw count, s = (alpha + C_j) - C_i in float64 with the
// reference's two roundings.
template <bool AI>
struct RowConst {
    int cjx;      // AI: C_j + alpha ; else C_j
    int lj;       // L_j
    double aj;    // !AI: fl(alpha + C_j)
};

template <bool AI>
__device__ __forceinline__ RowConst<AI> make_row(int cj, int lj, int alpha_int, double alpha)
{
    RowConst<AI> r;
    r.lj = lj;
    if (AI) {
        r.cjx = cj + alpha_int;
        r.aj = 0.0;
    } else {
        r.cjx = cj;
        r.aj = __dadd_rn(alpha, u32_to_double(cj));
    }
    return r;
}

// self score of segment [i, j): G[s] - s * Lg[len]
// LGS: ltab points to a copy of the first entries of the log table in SHARED memory (round 1 of the sliding-window
// pipeline: every length is below the window size, and the lengths of one warp's gather spread over tens of cache
// lines -- from shared memory the same gather costs a few bank conflicts instead)
template <bool AI, bool LGS = false>
__device__ __forceinline__ double self_score(int ci, int li, const RowConst<AI> &r,
                                             const double *__restrict__ gtab, const double *__restrict__ ltab)
{
    const int idx = r.cjx - ci;
    const int len = r.lj - li;
    const double g = __ldg(gtab + idx);
    const double lg = LGS ? ltab[len] : __ldg(ltab + len);
    const double s = AI ? u32_to_double(idx) : __dsub_rn(r.aj, u32_to_double(ci));
    return __dsub_rn(g, __dmul_rn(s, lg));
}

// One candidate as a column of the DP: position, cumulative count, finished prefix score.
// 16 bytes so a column is one LDS.128 (the 8 column phases of a warp read 8 x 16 B = one wavefront).
struct __align__(16) ColRec {
    int L;
    int C;
    double P;
};

// Combine the (max, arg) of the lanes that swept interleaved column phases of one row:
// larger value wins, equal values keep the smaller column index (np.argmax's first maximum).
template <int RPW>
__device__ __forceinline__ void merge_column_phases(double &best, int &arg)
{
#pragma unroll
    for (int off = RPW; off < 32; off <<= 1) {
        const double ob = __shfl_xor_sync(0xffffffffu, best, off);
        const int oa = __shfl_xor_sync(0xffffffffu, arg, off);
        if (ob > best || (ob == best && oa < arg)) { best = ob; arg = oa; }
    }
}

// Sweep columns i0+phase, i0+phase+stride, ... < i1 for the RPL rows of this lane; strict '>' keeps
// the first maximum among the lane's own (ascending) columns.  Every column record read from shared
// memory feeds RPL cells.  The table gathers are the long-latency part: a batch of U columns first
// issues all 2*U*RPL gathers, then does the arithmetic.
template <bool AI, int U, int RPL, bool LGS = false>
__device__ __forceinline__ void sweep_columns(int i0, int i1, int phase, int stride, const ColRec *sCol,
                                              const RowConst<AI> (&r)[RPL],
                                              const double *__restrict__ gtab, const double *__restrict__ ltab,
                                              double (&best)[RPL], int (&arg)[RPL])
{
    int i = i0 + phase;
    for (; i + (U - 1) * stride < i1; i += U * stride) {
        double g[U][RPL], lg[U][RPL], pc[U];
        int sx[U][RPL];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const ColRec a = sCol[i + u * stride];
            pc[u] = a.P;
#pragma unroll
            for (int k = 0; k < RPL; ++k) {
                const int idx = r[k].cjx - a.C;
                g[u][k] = __ldg(gtab + idx);
                lg[u][k] = LGS ? ltab[r[k].lj - a.L] : __ldg(ltab + (r[k].lj - a.L));
                sx[u][k] = AI ? idx : a.C;
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u)
#pragma unroll
            for (int k = 0; k < RPL; ++k) {
                const double s = AI ? u32_to_double(sx[u][k]) : __dsub_rn(r[k].aj, u32_to_double(sx[u][k]));
                const double t = __dadd_rn(__dsub_rn(g[u][k], __dmul_rn(s, lg[u][k])), pc[u]);
                if (t > best[k]) { best[k] = t; arg[k] = i + u * stride; }
            }
    }
    for (; i < i1; i += stride) {
        const ColRec a = sCol[i];
#pragma unroll
        for (int k = 0; k < RPL; ++k) {
            const double t = __dadd_rn(self_score<AI, LGS>(a.C, a.L, r[k], gtab, ltab), a.P);
            if (t > best[k]) { best[k] = t; arg[k] = i; }
        }
    }
}

constexpr int DP_JB = 32;   // rows resolved per block step
constexpr int DP_RPW = 4;   // a warp's gather spans DP_RPW rows x (32/DP_RPW) column phases

// ---- pieces of one block step over rows [jb, jb+32) of a candidate list in shared memory ------
//   rectangle: columns [col0, jb).  A warp covers RPL*4 rows (a lane: RPL rows, 4 apart) x 8
//              interleaved column phases, so the 32 addresses of one gather span 4 candidates of rows
//              plus 8 of columns instead of 32 -- that is what sets the number of L1 lines a gather
//              touches (profiles/r01_window_dp_*).  Warps beyond the row groups split the columns
//              into chunks; per-chunk (max, first arg-max) go to sPartV / sPartA.
//   triangle : columns [jb, j) -- the 32x32 self scores (independent of P) go to sTri.
template <bool AI, int NW, int U, int RPL>
__device__ __forceinline__ void block_rect_tri(int jb, int N, int col0, const ColRec *sCol,
                                               double *sPartV, int *sPartA, double *sTri,
                                               const double *__restrict__ gtab, const double *__restrict__ ltab,
                                               int alpha_int, double alpha)
{
    constexpr int RPW = DP_RPW;
    constexpr int CPW = 32 / RPW;               // column phases per warp
    constexpr int NG = DP_JB / (RPW * RPL);     // row groups per 32-row block
    constexpr int NQ = NW / NG;                 // column chunks (warps per row group)
    static_assert(NW % NG == 0 && NQ >= 1, "warps must tile the row groups");
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int grp = warp % NG, q = warp / NG;
    const int rr = lane % RPW, cc = lane / RPW;
    {
        RowConst<AI> r[RPL];
        double best[RPL];
        int arg[RPL];
        const int ncol = jb - col0;
        const int chunk = (ncol + NQ - 1) / NQ;
        const int i0 = col0 + q * chunk;
        const int i1 = min(i0 + chunk, jb);
#pragma unroll
        for (int k = 0; k < RPL; ++k) {
            const int j = min(jb + grp * RPW * RPL + k * RPW + rr, N - 1);
            const ColRec me = sCol[j];
            r[k] = make_row<AI>(me.C, me.L, alpha_int, alpha);
            best[k] = -INFINITY;
            arg[k] = i0 + cc;
        }
        sweep_columns<AI, U, RPL>(i0, i1, cc, CPW, sCol, r, gtab, ltab, best, arg);
#pragma unroll
        for (int k = 0; k < RPL; ++k) {
            merge_column_phases<RPW>(best[k], arg[k]);
            if (cc == 0) {
                const int row = grp * RPW * RPL + k * RPW + rr;
                sPartV[q * 32 + row] = best[k];
                sPartA[q * 32 + row] = arg[k];
            }
        }
    }
    {   // lane = row here
        const ColRec me = sCol[min(jb + lane, N - 1)];
        const RowConst<AI> r = make_row<AI>(me.C, me.L, alpha_int, alpha);
        static_assert(DP_JB % NW == 0, "warps must tile the triangle rows");
        double w[DP_JB / NW];
#pragma unroll
        for (int kk = 0; kk < DP_JB / NW; ++kk) {                 // all gathers of the warp's columns in flight together
            const int k = warp + kk * NW;
            w[kk] = 0.0;
            if (k < lane && jb + lane < N) {
                const ColRec a = sCol[jb + k];
                w[kk] = self_score<AI>(a.C, a.L, r, gtab, ltab);
            }
        }
#pragma unroll
        for (int kk = 0; kk < DP_JB / NW; ++kk) {
            const int k = warp + kk * NW;
            if (k < lane && jb + lane < N) sTri[k * DP_JB + lane] = w[kk];
        }
    }
    __syncthreads();
}

// The dependent part, one warp: merge the NQ column-chunk partials (ascending columns, strict '>'),
// then resolve the 32 rows in order, broadcasting each finished P by shuffle.
// init_best/init_arg (per lane) seed the maximum with what columns BEFORE the chunks contributed.
// sLB (optional) receives, per row, the maximum itself (before the creation cost is added).
template <int NQ>
__device__ __forceinline__ void block_chain(int jb, int N, ColRec *sCol, unsigned short *sPrev16, int *sPrev32,
                                            const double *sPartV, const int *sPartA, const double *sTri, double pen,
                                            double init_best, int init_arg, int arg_offset, double *sLB)
{
    const int lane = threadIdx.x & 31;
    double best = init_best;
    int arg = init_arg;
#pragma unroll
    for (int w = 0; w < NQ; ++w) {
        const double v = sPartV[w * 32 + lane];
        if (v > best) { best = v; arg = sPartA[w * 32 + lane] + arg_offset; }
    }
    double mine = 0.0, lb = 0.0;
    const int rows = min(DP_JB, N - jb);
#pragma unroll 8
    for (int k = 0; k < rows; ++k) {
        const double pf = __dadd_rn(best, pen);          // prefix_scores[j] = max + segment_creation_cost
        const double pk = __shfl_sync(0xffffffffu, pf, k);
        if (lane == k) { mine = pf; lb = best; }
        if (lane > k) {
            const double t = __dadd_rn(sTri[k * DP_JB + lane], pk);
            if (t > best) { best = t; arg = jb + k + arg_offset; }
        }
    }
    if (jb + lane < N) {
        sCol[jb + lane].P = mine;
        if (sPrev16) sPrev16[jb + lane] = (unsigned short)arg;
        else sPrev32[jb + lane] = arg;
        if (sLB) sLB[lane] = lb;
    }
}

// The same block under the hypothesis "the first maximum of row j is column j-1" for the rows after the block's
// first -- what the later sliding-window rounds find for nearly every row, since nearly every candidate survives.
// Then P_j = (self(j-1, j) + P_{j-1}) + pen is a sequential sum whose dependent path is two DADDs per row instead
// of block_chain's DADD, shuffle, DADD, compare, select; every lane still folds all columns of its row with those P
// (off the critical path) and the warp votes whether each first maximum is where assumed.  If so, by induction over
// the rows every P used was the true one: P and prev are what block_chain writes, bit for bit (same operations in the
// same order).  If not, nothing is written and the caller runs block_chain.
template <int NQ>
__device__ __forceinline__ bool block_chain_speculative(int jb, int N, ColRec *sCol, unsigned short *sPrev16,
                                                        const double *sPartV, const int *sPartA, const double *sTri,
                                                        double pen, double init_best, int init_arg)
{
    const int lane = threadIdx.x & 31;
    double best = init_best;
    int arg = init_arg;
#pragma unroll
    for (int w = 0; w < NQ; ++w) {
        const double v = sPartV[w * 32 + lane];
        if (v > best) { best = v; arg = sPartA[w * 32 + lane]; }
    }
    const int rows = min(DP_JB, N - jb);
    const double below = (lane >= 1 && lane < rows) ? sTri[(lane - 1) * DP_JB + lane] : 0.0;   // self(j-1, j) of my row
    double pk = __shfl_sync(0xffffffffu, __dadd_rn(best, pen), 0);        // the block's first row depends on no other
    double mine = pk;
#pragma unroll 8
    for (int k = 0; k < rows; ++k) {
        if (lane == k) mine = pk;
        if (lane > k) {
            const double t = __dadd_rn(sTri[k * DP_JB + lane], pk);
            if (t > best) { best = t; arg = jb + k; }
        }
        const double dn = __shfl_sync(0xffffffffu, below, (k + 1) & 31);
        pk = __dadd_rn(__dadd_rn(dn, pk), pen);
    }
    const bool as_assumed = lane == 0 || lane >= rows || arg == jb + lane - 1;
    if (!__all_sync(0xffffffffu, as_assumed)) return false;
    if (lane < rows) {
        sCol[jb + lane].P = mine;
        sPrev16[jb + lane] = (unsigned short)arg;
    }
    return true;
}

// The dependent part of a 32-row step of the whole-list regularised DP (K6 regularized_dp.cu, K9 regularized_exact.cu),
// one warp, lane = row jb + lane.  best / arg come in as the row's (max, first arg-max) over the columns before jb, with
// arg a column index of the list; triS / triR hold self score and length penalty of (column jb + k, row jb + lane).
// Resolves the rows in order: the split number of row jb + k follows its arg-max a, from this warp's registers when
// a >= jb, else from ns[] (rows already written back).  Returns the row's P (mine), split number and NR[split number].
__device__ __forceinline__ void reg_block_chain(int jb, int rows, const int *ns, const double *nrtab, int use_num, int use_len,
                                                double pen, const double (*triS)[33], const double (*triR)[33],
                                                double &best_io, int &arg_io, double &mine_out, int &ns_out, double &nrv_out)
{
    const int lane = threadIdx.x & 31;
    double best = best_io;          // (local copies: the compiler keeps the arg-max update branch-free)
    int arg = arg_io;
    double mine = 0.0, my_nrv = 0.0;
    int my_ns = 0;
    for (int k = 0; k < rows; ++k) {
        const int a = __shfl_sync(0xffffffffu, arg, k);                       // previous_splits of row jb + k
        const int from_block = __shfl_sync(0xffffffffu, my_ns, max(a - jb, 0));
        const int nsrc = a >= jb ? from_block : ns[a];
        const int ns_k = a != 0 ? nsrc + 1 : 0;                               // square_splitter.py:59-60
        const double pk = __shfl_sync(0xffffffffu, __dadd_rn(best, pen), k);  // :62
        const double nrvk = use_num ? __ldg(nrtab + ns_k) : 0.0;
        if (lane == k) { mine = pk; my_ns = ns_k; my_nrv = nrvk; }
        if (lane > k) {
            double t = __dadd_rn(triS[k][lane], pk);
            if (use_num) t = __dsub_rn(t, nrvk);
            if (use_len) t = __dsub_rn(t, triR[k][lane]);
            if (t > best) { best = t; arg = jb + k; }
        }
    }
    best_io = best;
    arg_io = arg;
    mine_out = mine;
    ns_out = my_ns;
    nrv_out = my_nrv;
}

// One full block step: rectangle over [col0, jb), triangle, chain.  Requires col0 <= jb and
// blockDim.x == NW*32.  Ends with a __syncthreads().
template <bool AI, int NW, int U, int RPL>
__device__ __forceinline__ void dp_block_step(int jb, int N, int col0, ColRec *sCol,
                                              unsigned short *sPrev16, int *sPrev32,
                                              double *sPartV, int *sPartA, double *sTri,
                                              const double *__restrict__ gtab, const double *__restrict__ ltab,
                                              int alpha_int, double alpha, double pen,
                                              double init_best, int init_arg, int arg_offset)
{
    constexpr int NQ = NW / (DP_JB / (DP_RPW * RPL));
    block_rect_tri<AI, NW, U, RPL>(jb, N, col0, sCol, sPartV, sPartA, sTri, gtab, ltab, alpha_int, alpha);
    if ((threadIdx.x >> 5) == 0)
        block_chain<NQ>(jb, N, sCol, sPrev16, sPrev32, sPartV, sPartA, sTri, pen, init_best, init_arg, arg_offset, nullptr);
    __syncthreads();
}
