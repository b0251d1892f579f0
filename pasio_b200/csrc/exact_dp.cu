// K3: the exact O(N^2) SquareSplitter DP for one long candidate list (N up to a few 1e5),
// spread over the whole chip.
//
// Replaces SquareSplitter.split_without_normalizations + collect_split_points
// (/root/reference/src/pasio/splitters/square_splitter.py:67-109) driven by
// all_suffixes_self_score (/root/reference/src/pasio/log_marginal_likelyhood.py:105-132).
//
// One persistent, cooperatively launched kernel: a diagonal CTA resolves the dependent chain of rows
// while worker CTAs fold the finished columns into the rows ahead of it (blocked wave-front with
// look-ahead; details above exact_pipeline_kernel).  Back-trace is pointer doubling.
#include "dp_core.cuh"

namespace {

constexpr int XD_ROWS = 128;           // rows per block step (4 sub-blocks of 32)
constexpr int XD_THREADS = 256;
constexpr int XD_WARPS = XD_THREADS / 32;

__global__ void gather_candidates_kernel(const int32_t *__restrict__ cand, i64 m, const i64 *__restrict__ cg,
                                         int32_t *__restrict__ L, int32_t *__restrict__ C)
{
    const i64 first = cand ? (i64)__ldg(cand) : 0;
    const i64 cg_first = __ldg(cg + first);
    for (i64 k = (i64)blockIdx.x * blockDim.x + threadIdx.x; k < m; k += (i64)gridDim.x * blockDim.x) {
        const i64 pos = cand ? (i64)__ldg(cand + k) : k;
        L[k] = (int32_t)(pos - first);
        C[k] = (int32_t)(__ldg(cg + pos) - cg_first);
    }
}

// ---- persistent pipeline ---------------------------------------------------------------------
// Row-blocks of XR rows; block b = rows [1 + XR*b, 1 + XR*(b+1)).  Row 0 is the base (P[0] = 0).
// Column block c = the same rows used as columns once final (block 0 also carries column 0).
//   CTA 0 (diagonal): for b = 0, 1, ...: waits for the owner's partial of block b, adds the tile
//       (column block b-1) x (row block b) from shared memory, resolves the XR x XR triangle with
//       the 32-row block step, publishes P / prev and bumps `done_block`.
//   CTAs 1..W (workers): worker w owns row blocks b == w (mod W).  It walks the column blocks in
//       order as they become final and folds tile (c, b) into a running (max, first arg-max) for
//       every owned block b >= c + 2; after column b-2 the partial of block b is complete and its
//       `ready` flag is raised.  Columns are folded in ascending order with strict '>', so the first
//       maximum wins exactly as in np.argmax.
// All CTAs are co-resident (cooperative launch), so the flag waits cannot deadlock: the diagonal
// waits only for work that depends on blocks it has already published.
struct XdParams {
    int N, nB, W;
    const int32_t *L;
    const int32_t *C;
    double *P;
    int *prev;
    double *run_val;      // per row: running max over the worker-owned columns
    int *run_arg;
    int *ready;           // per row block: worker partial complete
    int *done_block;      // number of row blocks the diagonal has finished
    const double *gtab;
    const double *ltab;
    int alpha_int;
    double alpha, pen;
};

// One XR-row x ncol-column tile.  Warp w owns rows [16w, 16w+16) of the tile; a lane holds 4 of
// them (rows 4k + lane%4, k = 0..3) and sweeps the columns of phase lane/4 (stride 8), so one gather
// instruction spans 4 rows + 8 columns of candidates (few L1 lines) and every column record read
// from shared memory feeds 4 cells.  After the sweep the 8 column phases of a row are merged with
// the first-maximum rule; lanes 0..3 then hold (max, arg local to the tile) for their 4 rows each.
constexpr int XT_RPL = 4;      // rows per lane
template <bool AI>
__device__ __forceinline__ void xd_tile(int row0, int N, int ncol, const ColRec *sCol,
                                        const int32_t *__restrict__ L, const int32_t *__restrict__ C,
                                        const double *__restrict__ gtab, const double *__restrict__ ltab,
                                        int alpha_int, double alpha, double (&best)[XT_RPL], int (&arg)[XT_RPL])
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int rr = lane & 3, cc = lane >> 2;
    RowConst<AI> r[XT_RPL];
#pragma unroll
    for (int k = 0; k < XT_RPL; ++k) {
        const int j = min(row0 + 16 * warp + 4 * k + rr, N - 1);
        r[k] = make_row<AI>(__ldg(C + j), __ldg(L + j), alpha_int, alpha);
        best[k] = -INFINITY;
        arg[k] = cc;
    }
    sweep_columns<AI, 4, XT_RPL>(0, ncol, cc, 8, sCol, r, gtab, ltab, best, arg);
#pragma unroll
    for (int k = 0; k < XT_RPL; ++k) merge_column_phases<4>(best[k], arg[k]);
}

template <bool AI>
__global__ void __launch_bounds__(XD_THREADS)
exact_pipeline_kernel(XdParams p)
{
    constexpr int XR = XD_ROWS;
    __shared__ ColRec sColP[XR + 1];        // previous / column block
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
            for (int i = tid; i < ncol; i += XD_THREADS) {
                sColP[i].L = __ldg(p.L + c0 + i);
                sColP[i].C = __ldg(p.C + c0 + i);
                sColP[i].P = __ldcg(p.P + c0 + i);
            }
            __syncthreads();
            for (int b = bfirst; b < p.nB; b += p.W) {
                const int row0 = 1 + XR * b;
                double best[XT_RPL];
                int arg[XT_RPL];
                xd_tile<AI>(row0, p.N, ncol, sColP, p.L, p.C, p.gtab, p.ltab, p.alpha_int, p.alpha, best, arg);
                if (lane < 4) {
#pragma unroll
                    for (int k = 0; k < XT_RPL; ++k) {
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
    __shared__ int sPrevc[XR];
    __shared__ double sInitV[XR];
    __shared__ int sInitA[XR];
    __shared__ double sPartV[XD_WARPS * 32];
    __shared__ int sPartA[XD_WARPS * 32];
    __shared__ double sTri[DP_JB * DP_JB];

    if (tid == 0) {
        sColP[0].L = __ldg(p.L);
        sColP[0].C = __ldg(p.C);
        sColP[0].P = 0.0;                   // prefix_scores[0] = 0 (square_splitter.py:72)
        __stcg(p.P, 0.0);
        __stcg(p.prev, 0);
    }
    int ncol = 1, col_base = 0;
    __syncthreads();
    for (int b = 0; b < p.nB; ++b) {
        const int r0 = 1 + XR * b;
        const int nrows = min(XR, p.N - r0);
        if (tid < nrows) { sColC[tid].L = __ldg(p.L + r0 + tid); sColC[tid].C = __ldg(p.C + r0 + tid); }
        if (b >= 2) wait_at_least(p.ready + b, 1);
        // tile (previous block) x (this block), seeded with the worker partial
        {
            double best[XT_RPL];
            int arg[XT_RPL];
            xd_tile<AI>(r0, p.N, ncol, sColP, p.L, p.C, p.gtab, p.ltab, p.alpha_int, p.alpha, best, arg);
            if (lane < 4) {
#pragma unroll
                for (int k = 0; k < XT_RPL; ++k) {
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
        for (int sb = 0; sb < nrows; sb += DP_JB) {
            double ib = -INFINITY;
            int ia = 0;
            if (tid < 32 && sb + lane < nrows) { ib = sInitV[sb + lane]; ia = sInitA[sb + lane]; }
            dp_block_step<AI, XD_WARPS, 8, 1>(sb, nrows, 0, sColC, nullptr, sPrevc, sPartV, sPartA, sTri,
                                           p.gtab, p.ltab, p.alpha_int, p.alpha, p.pen, ib, ia, r0);
        }
        // this block becomes the column block of the next one; block 0 keeps column 0 in front of it
        const int keep0 = (b == 0) ? 1 : 0;
        if (tid < nrows) {
            __stcg(p.P + r0 + tid, sColC[tid].P);
            __stcg(p.prev + r0 + tid, sPrevc[tid]);
            sColP[tid + keep0] = sColC[tid];
        }
        ncol = nrows + keep0;
        col_base = r0 - keep0;
        publish(p.done_block, b + 1);
        __syncthreads();
    }
}

// ---- back-trace by pointer doubling over global arrays --------------------------------------
__global__ void bt_init_kernel(const int *__restrict__ prev, i64 N, int *jump, uint8_t *mark)
{
    for (i64 k = (i64)blockIdx.x * blockDim.x + threadIdx.x; k < N; k += (i64)gridDim.x * blockDim.x) {
        jump[k] = prev[k];
        mark[k] = (k == N - 1);
    }
}
__global__ void bt_step_kernel(const int *__restrict__ jump_in, int *__restrict__ jump_out, uint8_t *mark, i64 N)
{
    for (i64 k = (i64)blockIdx.x * blockDim.x + threadIdx.x; k < N; k += (i64)gridDim.x * blockDim.x) {
        const int jk = jump_in[k];
        if (mark[k]) mark[jk] = 1;
        jump_out[k] = jump_in[jk];
    }
}
__global__ void bt_scatter_kernel(const uint8_t *__restrict__ mark, i64 N, const int32_t *__restrict__ cand,
                                  uint32_t *keepbits)
{
    for (i64 k = (i64)blockIdx.x * blockDim.x + threadIdx.x; k < N; k += (i64)gridDim.x * blockDim.x) {
        if (mark[k]) {
            const i64 pos = cand ? (i64)__ldg(cand + k) : k;
            atomicOr(keepbits + (pos >> 5), 1u << (pos & 31));
        }
    }
}

template <bool AI>
__global__ void suffix_row_kernel(i64 stop, const int32_t *__restrict__ cand, const i64 *__restrict__ cg,
                                  const double *__restrict__ gtab, const double *__restrict__ ltab,
                                  int alpha_int, double alpha, double *__restrict__ out)
{
    const i64 first = cand ? (i64)__ldg(cand) : 0;
    const i64 cg_first = __ldg(cg + first);
    const i64 pj = cand ? (i64)__ldg(cand + stop) : stop;
    const RowConst<AI> r = make_row<AI>((int)(__ldg(cg + pj) - cg_first), (int)(pj - first), alpha_int, alpha);
    for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < stop; i += (i64)gridDim.x * blockDim.x) {
        const i64 pi = cand ? (i64)__ldg(cand + i) : i;
        out[i] = self_score<AI>((int)(__ldg(cg + pi) - cg_first), (int)(pi - first), r, gtab, ltab);
    }
}

inline unsigned grid_for(pasio_ctx *ctx, i64 n, int threads)
{
    i64 g = (n + threads - 1) / threads;
    i64 cap = (i64)ctx->sm_count * 16;
    if (g > cap) g = cap;
    if (g < 1) g = 1;
    return (unsigned)g;
}

}  // namespace

int launch_gather_candidates(pasio_ctx *ctx)
{
    const i64 m = ctx->m;
    PASIO_TRY(pasio_reserve(ctx, ctx->dpL, (size_t)m * 4));
    PASIO_TRY(pasio_reserve(ctx, ctx->dpC, (size_t)m * 4));
    gather_candidates_kernel<<<grid_for(ctx, m, 256), 256, 0, ctx->stream>>>(
        cur_cand(ctx), m, ctx->cg.as<i64>(), ctx->dpL.as<int32_t>(), ctx->dpC.as<int32_t>());
    CUDA_TRY(ctx, cudaGetLastError());
    return PASIO_OK;
}

template <bool AI>
static int run_exact_dp(pasio_ctx *ctx, i64 N)
{
    XdParams p;
    p.N = (int)N;
    p.nB = (int)((N - 1 + XD_ROWS - 1) / XD_ROWS);
    p.L = ctx->dpL.as<int32_t>();
    p.C = ctx->dpC.as<int32_t>();
    p.P = ctx->dpP.as<double>();
    p.prev = ctx->dpPrev.as<int>();
    p.run_val = ctx->dpPart.as<double>();
    p.run_arg = ctx->dpPartArg.as<int>();
    p.ready = ctx->dpMark.as<int>();
    p.done_block = p.ready + p.nB;
    p.gtab = ctx->tab[AI ? PASIO_TAB_LGAMMA : PASIO_TAB_LGAMMA_ALPHA].as<double>();
    p.ltab = ctx->tab[PASIO_TAB_LOG].as<double>();
    p.alpha_int = (int)ctx->alpha_int;
    p.alpha = ctx->alpha;
    p.pen = ctx->pen;
    int per_sm = 0;
    CUDA_TRY(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, exact_pipeline_kernel<AI>, XD_THREADS, 0));
    if (per_sm < 1) return pasio_fail(ctx, PASIO_E_CUDA, "exact DP kernel cannot be resident");
    if (per_sm > 3) per_sm = 3;
    int workers = ctx->sm_count * per_sm - 1;
    if (workers > p.nB - 2) workers = p.nB - 2;
    if (workers < 0) workers = 0;
    p.W = workers > 0 ? workers : 1;
    CUDA_TRY(ctx, cudaMemsetAsync(p.ready, 0, (size_t)(p.nB + 1) * sizeof(int), ctx->stream));
    void *args[] = {&p};
    TimingScope ts(ctx, TF_EXACT_DP);
    // cooperative launch = all CTAs co-resident, which the flag waits rely on
    CUDA_TRY(ctx, cudaLaunchCooperativeKernel((void *)exact_pipeline_kernel<AI>, dim3(1 + workers), dim3(XD_THREADS),
                                              args, 0, ctx->stream));
    return PASIO_OK;
}

int launch_exact_dp(pasio_ctx *ctx, i64 N)
{
    // tiny alpha: lgamma(alpha) dwarfs the delta scale of the bound; alpha = 0: G[0] = inf (as in window_dp.cu)
    if (ctx->tune[PASIO_TUNE_EXACT_PRUNE] && ctx->alpha >= 0.0009765625) {
        ctx->fam_launches[TF_EXACT_DP] += 0;
        return launch_exact_dp_pruned(ctx, N, ctx->tune[PASIO_TUNE_EXACT_LAG]);
    }
    ctx->last_cells = N * (N - 1) / 2;
    ctx->last_cells_skipped = 0;
    const i64 nB = (N - 1 + XD_ROWS - 1) / XD_ROWS;
    PASIO_TRY(pasio_reserve(ctx, ctx->dpP, (size_t)N * 8));
    PASIO_TRY(pasio_reserve(ctx, ctx->dpPrev, (size_t)N * 4));
    PASIO_TRY(pasio_reserve(ctx, ctx->dpPart, (size_t)N * 8));
    PASIO_TRY(pasio_reserve(ctx, ctx->dpPartArg, (size_t)N * 4));
    PASIO_TRY(pasio_reserve(ctx, ctx->dpMark, (size_t)(nB + 2) * sizeof(int) > (size_t)N ? (size_t)(nB + 2) * sizeof(int) : (size_t)N));
    return ctx->alpha_is_int ? run_exact_dp<true>(ctx, N) : run_exact_dp<false>(ctx, N);
}

int launch_backtrace_mark(pasio_ctx *ctx, i64 N)
{
    PASIO_TRY(pasio_reserve(ctx, ctx->dpJump, (size_t)N * 8));
    PASIO_TRY(pasio_reserve(ctx, ctx->dpMark, (size_t)N));
    int *ja = ctx->dpJump.as<int>();
    int *jb = ja + N;
    uint8_t *mark = ctx->dpMark.as<uint8_t>();
    const unsigned g = grid_for(ctx, N, 256);
    bt_init_kernel<<<g, 256, 0, ctx->stream>>>(ctx->dpPrev.as<int>(), N, ja, mark);
    for (i64 reach = 1; reach < N; reach <<= 1) {
        bt_step_kernel<<<g, 256, 0, ctx->stream>>>(ja, jb, mark, N);
        int *t = ja; ja = jb; jb = t;
    }
    const size_t bit_bytes = (size_t)((ctx->n + 1 + 31) / 32 + 2) * 4;
    CUDA_TRY(ctx, cudaMemsetAsync(ctx->keepbits.p, 0, bit_bytes, ctx->stream));
    bt_scatter_kernel<<<g, 256, 0, ctx->stream>>>(mark, N, cur_cand(ctx), ctx->keepbits.as<uint32_t>());
    CUDA_TRY(ctx, cudaGetLastError());
    return PASIO_OK;
}

int launch_suffix_row(pasio_ctx *ctx, i64 stop, double *d_out)
{
    const double *gtab = ctx->tab[ctx->alpha_is_int ? PASIO_TAB_LGAMMA : PASIO_TAB_LGAMMA_ALPHA].as<double>();
    const double *ltab = ctx->tab[PASIO_TAB_LOG].as<double>();
    const unsigned g = grid_for(ctx, stop, 256);
    TimingScope ts(ctx, TF_SCORE);
    if (ctx->alpha_is_int)
        suffix_row_kernel<true><<<g, 256, 0, ctx->stream>>>(stop, cur_cand(ctx), ctx->cg.as<i64>(), gtab, ltab,
                                                           (int)ctx->alpha_int, ctx->alpha, d_out);
    else
        suffix_row_kernel<false><<<g, 256, 0, ctx->stream>>>(stop, cur_cand(ctx), ctx->cg.as<i64>(), gtab, ltab,
                                                            (int)ctx->alpha_int, ctx->alpha, d_out);
    CUDA_TRY(ctx, cudaGetLastError());
    return PASIO_OK;
}
