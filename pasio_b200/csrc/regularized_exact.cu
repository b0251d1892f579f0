// K9: the regularised whole-list SquareSplitter DP (the DP of K6, regularized_dp.cu) over the whole chip, for long
// candidate lists: --algorithm exact over a contig, or the final DP of --algorithm slidingwindow over the survivors of its
// window step, with --split-number-regularization / --length-regularization.
//
// The structure of K3's every-cell pipeline (exact_dp.cu: exact_pipeline_kernel) with K6's cell in K6's operation order
// (square_splitter.py:29-65):
//     t = self_score(i, j) + P_i
//     t = t - NR[ns_i]               if the split-number term is on;  column 0: t = t + refund
//     t = t - LR[L_j - L_i]          if the length term is on
//     prev_j = first arg-max, ns_j = prev_j ? ns[prev_j] + 1 : 0, P_j = t[prev_j] + creation cost
// Row blocks of 128 rows, block b = rows [1 + 128 b, 1 + 128 (b + 1)); column block c = the same rows once final (block 0
// also carries column 0).
//   CTA 0 (diagonal): for b = 0, 1, ...: waits for the owner's partial of block b, folds in tile (column block b - 1) x
//       (row block b) -- the partial holds older columns, so it wins ties --, then resolves the block in 32-row steps:
//       the block's finished rows as columns, the 32 x 32 triangle, and K6's chain (reg_block_chain, dp_core.cuh), which
//       also keeps the split numbers.  P, prev, ns and NR[ns] of the block are written before `done_block` is raised.
//   CTAs 1..W (workers): worker w owns row blocks b == w (mod W).  It stages each column block as it becomes final
//       (L, C, P and NR[ns] of every column) and folds tile (c, b) into a running (max, first arg-max) for every owned
//       block b >= c + 2: column blocks in ascending order, a later one replaces the running value only when strictly
//       greater (np.argmax's first maximum).  After column block b - 2 the partial of block b is complete: `ready[b]`.
// Every cell is evaluated (no bound: the length term breaks the convexity K3's pruned variant relies on), each cell is the
// same double whichever CTA computes it, and every merge keeps the smaller column on ties, so P, prev and the split
// numbers are bit-identical to K6's.  All CTAs are co-resident (cooperative launch): workers wait only for `done_block`,
// and the diagonal waits only for partials whose inputs it has already published, so the waits cannot deadlock.
#include "dp_core.cuh"

namespace {

constexpr int RX_ROWS = 128;            // rows per block (4 steps of 32)
constexpr int RX_THREADS = 256;
constexpr int RX_WARPS = RX_THREADS / 32;
constexpr int RX_RPL = 4;               // tile rows per lane
constexpr int RX_U = 2;                 // tile columns per lane whose gathers are issued together

struct RxParams {
    int N, nB, W;
    const int32_t *L;
    const int32_t *C;
    double *P;
    int *prev;
    int *ns;                // number of splits of the best segmentation of each prefix
    double *nrv;            // NR[ns_i]: the split-number penalty column i carries
    double *run_val;        // per row: running max over the worker-owned columns
    int *run_arg;
    int *ready;             // per row block: worker partial complete
    int *done_block;        // number of row blocks the diagonal has finished
    const double *gtab;
    const double *ltab;
    const double *lrtab;    // LR[len]
    const double *nrtab;    // NR[k]
    int use_num, use_len;
    double add0, pen, alpha;
    int alpha_int;
};

// the penalty terms of one cell, after self + P (K6: reg_cell)
__device__ __forceinline__ double rx_cell(double self, double pc, double nrvc, double lr, bool col0, const RxParams &p)
{
    double t = __dadd_rn(self, pc);
    if (p.use_num) {
        t = __dsub_rn(t, nrvc);
        if (col0) t = __dadd_rn(t, p.add0);             // the reference subtracts the penalty from column 0 too, then adds it back
    }
    if (p.use_len) t = __dsub_rn(t, lr);
    return t;
}

// One 128-row x ncol-column tile (K3's xd_tile): warp w owns rows [16w, 16w+16), a lane holds 4 of them (rows 4k + lane%4)
// and sweeps the columns of phase lane/4 (stride 8).  col0: local index of column 0 of the list, or -1.  Lanes 0..3 end
// with (max, first arg-max local to the tile) of their 4 rows.
template <bool AI>
__device__ __forceinline__ void rx_tile(int row0, int ncol, const ColRec *sCol, const double *sNrv, int col0, const RxParams &p,
                                        double (&best)[RX_RPL], int (&arg)[RX_RPL])
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int rr = lane & 3, cc = lane >> 2;
    RowConst<AI> r[RX_RPL];
#pragma unroll
    for (int k = 0; k < RX_RPL; ++k) {
        const int j = min(row0 + 16 * warp + 4 * k + rr, p.N - 1);
        r[k] = make_row<AI>(__ldg(p.C + j), __ldg(p.L + j), p.alpha_int, p.alpha);
        best[k] = -INFINITY;
        arg[k] = cc;
    }
    int i = cc;
    for (; i + (RX_U - 1) * 8 < ncol; i += RX_U * 8) {       // all gathers of RX_U columns in flight, then the arithmetic
        double g[RX_U][RX_RPL], lg[RX_U][RX_RPL], lr[RX_U][RX_RPL], pc[RX_U], nv[RX_U];
        int sx[RX_U][RX_RPL];
#pragma unroll
        for (int u = 0; u < RX_U; ++u) {
            const ColRec a = sCol[i + 8 * u];
            pc[u] = a.P;
            nv[u] = sNrv[i + 8 * u];
#pragma unroll
            for (int k = 0; k < RX_RPL; ++k) {
                const int idx = r[k].cjx - a.C;
                const int len = r[k].lj - a.L;
                g[u][k] = __ldg(p.gtab + idx);
                lg[u][k] = __ldg(p.ltab + len);
                lr[u][k] = p.use_len ? __ldg(p.lrtab + len) : 0.0;
                sx[u][k] = AI ? idx : a.C;
            }
        }
#pragma unroll
        for (int u = 0; u < RX_U; ++u)
#pragma unroll
            for (int k = 0; k < RX_RPL; ++k) {
                const double s = AI ? u32_to_double(sx[u][k]) : __dsub_rn(r[k].aj, u32_to_double(sx[u][k]));
                const double t = rx_cell(__dsub_rn(g[u][k], __dmul_rn(s, lg[u][k])), pc[u], nv[u], lr[u][k], i + 8 * u == col0, p);
                if (t > best[k]) { best[k] = t; arg[k] = i + 8 * u; }
            }
    }
    for (; i < ncol; i += 8) {
        const ColRec a = sCol[i];
#pragma unroll
        for (int k = 0; k < RX_RPL; ++k) {
            const double lr = p.use_len ? __ldg(p.lrtab + (r[k].lj - a.L)) : 0.0;
            const double t = rx_cell(self_score<AI>(a.C, a.L, r[k], p.gtab, p.ltab), a.P, sNrv[i], lr, i == col0, p);
            if (t > best[k]) { best[k] = t; arg[k] = i; }
        }
    }
#pragma unroll
    for (int k = 0; k < RX_RPL; ++k) merge_column_phases<4>(best[k], arg[k]);
}

template <bool AI>
__global__ void __launch_bounds__(RX_THREADS)
regularized_exact_kernel(RxParams p)
{
    constexpr int XR = RX_ROWS;
    __shared__ ColRec sColP[XR + 1];        // previous / column block
    __shared__ double sNrvP[XR + 1];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    if (blockIdx.x != 0) {
        // ------------------------------- worker -------------------------------------------------
        const int w = blockIdx.x - 1;
        for (int c = 0; c + 2 < p.nB; ++c) {
            int bfirst = c + 2;
            bfirst += ((w - bfirst) % p.W + p.W) % p.W;           // first owned block >= c+2
            if (bfirst >= p.nB) break;                              // owned set only shrinks with c
            wait_at_least(p.done_block, c + 1);
            const int c0 = c == 0 ? 0 : 1 + XR * c;
            const int c1 = min(1 + XR * (c + 1), p.N);
            const int ncol = c1 - c0;
            for (int i = tid; i < ncol; i += RX_THREADS) {
                sColP[i].L = __ldg(p.L + c0 + i);
                sColP[i].C = __ldg(p.C + c0 + i);
                sColP[i].P = __ldcg(p.P + c0 + i);
                sNrvP[i] = __ldcg(p.nrv + c0 + i);
            }
            __syncthreads();
            for (int b = bfirst; b < p.nB; b += p.W) {
                const int row0 = 1 + XR * b;
                double best[RX_RPL];
                int arg[RX_RPL];
                rx_tile<AI>(row0, ncol, sColP, sNrvP, c == 0 ? 0 : -1, p, best, arg);
                if (lane < 4) {
#pragma unroll
                    for (int k = 0; k < RX_RPL; ++k) {
                        const int row = row0 + 16 * warp + 4 * k + lane;
                        if (row < p.N) {
                            bool take = true;
                            if (c > 0) take = best[k] > __ldcg(p.run_val + row);   // later columns must be strictly better
                            if (take) {
                                __stcg(p.run_val + row, best[k]);
                                __stcg(p.run_arg + row, arg[k] + c0);
                            }
                        }
                    }
                }
                if (b == c + 2) publish(p.ready + b, 1);
            }
            __syncthreads();                                       // column block buffer is reloaded next
        }
        return;
    }

    // ----------------------------------- diagonal ---------------------------------------------
    __shared__ ColRec sColC[XR];
    __shared__ double sNrvC[XR];
    __shared__ double sInitV[XR];
    __shared__ int sInitA[XR];
    __shared__ double sPartV[RX_WARPS][32];
    __shared__ int sPartA[RX_WARPS][32];
    __shared__ double sTriS[32][33], sTriR[32][33];      // self score / length penalty of (column k of the step, row)

    if (tid == 0) {
        const double nrv0 = p.use_num ? __ldg(p.nrtab) : 0.0;
        sColP[0].L = __ldg(p.L);
        sColP[0].C = __ldg(p.C);
        sColP[0].P = 0.0;                   // prefix_scores[0] = 0 (square_splitter.py:34)
        sNrvP[0] = nrv0;
        __stcg(p.P, 0.0);
        __stcg(p.prev, 0);
        __stcg(p.ns, 0);
        __stcg(p.nrv, nrv0);
    }
    int ncol = 1, col_base = 0;
    __syncthreads();
    for (int b = 0; b < p.nB; ++b) {
        const int r0 = 1 + XR * b;
        const int nrows = min(XR, p.N - r0);
        if (tid < nrows) { sColC[tid].L = __ldg(p.L + r0 + tid); sColC[tid].C = __ldg(p.C + r0 + tid); }
        if (b >= 2) wait_at_least(p.ready + b, 1);
        // tile (previous block) x (this block), merged with the worker partial
        {
            double best[RX_RPL];
            int arg[RX_RPL];
            rx_tile<AI>(r0, ncol, sColP, sNrvP, col_base == 0 ? 0 : -1, p, best, arg);
            if (lane < 4) {
#pragma unroll
                for (int k = 0; k < RX_RPL; ++k) {
                    const int t = 16 * warp + 4 * k + lane;
                    double bv = best[k];
                    int ba = arg[k] + col_base;
                    if (b >= 2 && t < nrows) {
                        const double rv = __ldcg(p.run_val + r0 + t);
                        if (!(bv > rv)) { bv = rv; ba = __ldcg(p.run_arg + r0 + t); }   // older columns win ties
                    }
                    sInitV[t] = bv;
                    sInitA[t] = ba;
                }
            }
        }
        __syncthreads();
        for (int sb = 0; sb < nrows; sb += 32) {
            const int jb = r0 + sb;
            const ColRec me = sColC[min(sb + lane, nrows - 1)];
            const RowConst<AI> row = make_row<AI>(me.C, me.L, p.alpha_int, p.alpha);
            {   // this block's finished rows [r0, jb) as columns: this warp's contiguous chunk, every lane its own row
                const int chunk = (sb + RX_WARPS - 1) / RX_WARPS;
                const int i0 = warp * chunk, i1 = min(i0 + chunk, sb);
                double best = -INFINITY;
                int arg = i0;
                for (int i = i0; i < i1; ++i) {
                    const ColRec a = sColC[i];
                    const double lr = p.use_len ? __ldg(p.lrtab + (row.lj - a.L)) : 0.0;
                    const double t = rx_cell(self_score<AI>(a.C, a.L, row, p.gtab, p.ltab), a.P, sNrvC[i], lr, false, p);
                    if (t > best) { best = t; arg = i; }
                }
                sPartV[warp][lane] = best;
                sPartA[warp][lane] = arg;
            }
#pragma unroll
            for (int k = warp; k < 32; k += RX_WARPS) {     // the step's own triangle (P-independent parts)
                if (k < lane && sb + lane < nrows) {
                    const ColRec a = sColC[sb + k];
                    sTriS[k][lane] = self_score<AI>(a.C, a.L, row, p.gtab, p.ltab);
                    sTriR[k][lane] = p.use_len ? __ldg(p.lrtab + (row.lj - a.L)) : 0.0;
                }
            }
            __syncthreads();
            if (warp == 0) {
                const int rows = min(32, nrows - sb);
                double best = lane < rows ? sInitV[sb + lane] : -INFINITY;
                int arg = lane < rows ? sInitA[sb + lane] : 0;
#pragma unroll
                for (int w2 = 0; w2 < RX_WARPS; ++w2) {     // ascending column chunks after the older columns: strictly greater wins
                    const double v = sPartV[w2][lane];
                    if (v > best) { best = v; arg = r0 + sPartA[w2][lane]; }
                }
                double mine, my_nrv;
                int my_ns;
                reg_block_chain(jb, rows, p.ns, p.nrtab, p.use_num, p.use_len, p.pen, sTriS, sTriR, best, arg, mine, my_ns, my_nrv);
                if (lane < rows) {
                    sColC[sb + lane].P = mine;
                    sNrvC[sb + lane] = my_nrv;
                    __stcg(p.P + jb + lane, mine);
                    __stcg(p.prev + jb + lane, arg);
                    p.ns[jb + lane] = my_ns;                 // read back by this warp's later chains only
                    __stcg(p.nrv + jb + lane, my_nrv);
                }
            }
            __syncthreads();
        }
        // this block becomes the column block of the next one; block 0 keeps column 0 in front of it
        const int keep0 = (b == 0) ? 1 : 0;
        if (tid < nrows) {
            sColP[tid + keep0] = sColC[tid];
            sNrvP[tid + keep0] = sNrvC[tid];
        }
        ncol = nrows + keep0;
        col_base = r0 - keep0;
        publish(p.done_block, b + 1);
        __syncthreads();
    }
}

template <bool AI>
int run_regularized_exact(pasio_ctx *ctx, RxParams &p)
{
    int per_sm = 0;
    CUDA_TRY(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, regularized_exact_kernel<AI>, RX_THREADS, 0));
    if (per_sm < 1) return pasio_fail(ctx, PASIO_E_CUDA, "regularised exact DP kernel cannot be resident");
    if (per_sm > 3) per_sm = 3;
    int workers = ctx->sm_count * per_sm - 1;
    if (workers > p.nB - 2) workers = p.nB - 2;
    if (workers < 0) workers = 0;
    p.W = workers > 0 ? workers : 1;
    CUDA_TRY(ctx, cudaMemsetAsync(p.ready, 0, (size_t)(p.nB + 1) * sizeof(int), ctx->stream));
    void *args[] = {&p};
    TimingScope ts(ctx, TF_EXACT_DP);
    // cooperative launch = all CTAs co-resident, which the flag waits rely on
    CUDA_TRY(ctx, cudaLaunchCooperativeKernel((void *)regularized_exact_kernel<AI>, dim3(1 + workers), dim3(RX_THREADS),
                                              args, 0, ctx->stream));
    return PASIO_OK;
}

}  // namespace

// the same contract as launch_regularized_dp: over ctx->dpL / dpC -> dpP / dpPrev (split numbers in dpPartArg, NR of them
// in dpPart); d_lr / d_nr: device copies of the penalty tables or NULL
int launch_regularized_exact(pasio_ctx *ctx, i64 N, const double *d_lr, const double *d_nr, double add0)
{
    const i64 nB = (N - 1 + RX_ROWS - 1) / RX_ROWS;
    PASIO_TRY(pasio_reserve(ctx, ctx->dpP, (size_t)N * 8));
    PASIO_TRY(pasio_reserve(ctx, ctx->dpPrev, (size_t)N * 4));
    PASIO_TRY(pasio_reserve(ctx, ctx->dpPart, (size_t)N * 8));
    PASIO_TRY(pasio_reserve(ctx, ctx->dpPartArg, (size_t)N * 4));
    PASIO_TRY(pasio_reserve(ctx, ctx->dpJump, (size_t)N * 8));                  // running max (the back-trace reuses it)
    PASIO_TRY(pasio_reserve(ctx, ctx->dpMark, (size_t)(N + nB + 1) * 4));       // running arg-max, then the flags
    RxParams p;
    p.N = (int)N;
    p.nB = (int)nB;
    p.L = ctx->dpL.as<int32_t>();
    p.C = ctx->dpC.as<int32_t>();
    p.P = ctx->dpP.as<double>();
    p.prev = ctx->dpPrev.as<int>();
    p.ns = ctx->dpPartArg.as<int>();
    p.nrv = ctx->dpPart.as<double>();
    p.run_val = ctx->dpJump.as<double>();
    p.run_arg = ctx->dpMark.as<int>();
    p.ready = p.run_arg + N;
    p.done_block = p.ready + nB;
    p.gtab = ctx->tab[ctx->alpha_is_int ? PASIO_TAB_LGAMMA : PASIO_TAB_LGAMMA_ALPHA].as<double>();
    p.ltab = ctx->tab[PASIO_TAB_LOG].as<double>();
    p.lrtab = d_lr;
    p.nrtab = d_nr;
    p.use_len = d_lr != nullptr;
    p.use_num = d_nr != nullptr;
    p.add0 = add0;
    p.pen = ctx->pen;
    p.alpha = ctx->alpha;
    p.alpha_int = (int)ctx->alpha_int;
    PASIO_TRY(ctx->alpha_is_int ? run_regularized_exact<true>(ctx, p) : run_regularized_exact<false>(ctx, p));
    ctx->last_cells = N * (N - 1) / 2;
    ctx->last_cells_skipped = 0;
    return PASIO_OK;
}
