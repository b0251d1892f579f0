// The regularised SquareSplitter DP on the device (SURVEY 8 f-3).
//
// Replaces SquareSplitter.split_with_normalizations (/root/reference/src/pasio/splitters/square_splitter.py:29-65) for the
// penalty functions the reference's CLI can select (default_splitters.py:36-39, cli.py:41-53): per cell, in the
// reference's operation order,
//     t = self_score(i, j) + P_i                                  log_marginal_likelyhood.py:105-132, square_splitter.py:44
//     t = t - lambda_n * f(num_splits_i + 1)   (+ lambda_n * f(1) again for i = 0)          square_splitter.py:46-49
//     t = t - lambda_L * g(L_j - L_i)                                                       square_splitter.py:51-54
//     prev_j = first arg-max, P_j = t[prev_j] + creation cost, num_splits_j = prev_j ? num_splits[prev_j] + 1 : 0    :56-62
// The two penalty terms come from host-built tables NR[k] = lambda_n * f(k + 1) and LR[len] = lambda_L * g(len)
// (numpy values, like the log / lgamma tables), so the device adds exactly the doubles the reference adds.
// One CTA of 1024 threads per candidate list: 32-row block steps, the finished columns swept by 32 warps in contiguous
// chunks (ascending columns, strict '>': np.argmax's first maximum), the 32 x 32 triangle resolved in order by warp 0.
// Not a throughput kernel like K3/K4 (the CLI flags it serves are rarely used); what it removes is the host loop that
// launched one kernel and copied one row back per candidate.
#include "dp_core.cuh"

namespace {

constexpr int RG_THREADS = 1024;
constexpr int RG_WARPS = RG_THREADS / 32;

struct RegParams {
    int N;
    const int32_t *L;
    const int32_t *C;
    double *P;
    int *prev;
    int *ns;                // number of splits of the best segmentation of each prefix
    double *nrv;            // NR[ns_i]: the split-number penalty column i carries
    const double *gtab;
    const double *ltab;
    const double *lrtab;    // LR[len]
    const double *nrtab;    // NR[k]
    int use_num, use_len;
    double add0, pen, alpha;
    int alpha_int;
};

template <bool AI>
__device__ __forceinline__ double reg_cell(int i, int ci, int li, double pi, double nrvi, const RowConst<AI> &r, const RegParams &p)
{
    double t = __dadd_rn(self_score<AI>(ci, li, r, p.gtab, p.ltab), pi);
    if (p.use_num) {
        t = __dsub_rn(t, nrvi);
        if (i == 0) t = __dadd_rn(t, p.add0);           // the reference subtracts the penalty from column 0 too, then adds it back
    }
    if (p.use_len) t = __dsub_rn(t, __ldg(p.lrtab + (r.lj - li)));
    return t;
}

template <bool AI>
__global__ void __launch_bounds__(RG_THREADS, 1)
regularized_dp_kernel(RegParams p)
{
    __shared__ double sPartV[RG_WARPS][32];
    __shared__ int sPartA[RG_WARPS][32];
    __shared__ double sTriS[32][33], sTriR[32][33];      // self score / length penalty of (column k of the block, row)
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int N = p.N;
    if (tid == 0) {
        p.P[0] = 0.0;                                     // prefix_scores[0] = 0 (square_splitter.py:34)
        p.prev[0] = 0;
        p.ns[0] = 0;
        p.nrv[0] = p.use_num ? __ldg(p.nrtab) : 0.0;
    }
    __syncthreads();
    for (int jb = 1; jb < N; jb += 32) {
        const int j = min(jb + lane, N - 1);
        const RowConst<AI> row = make_row<AI>(__ldg(p.C + j), __ldg(p.L + j), p.alpha_int, p.alpha);
        {   // finished columns [0, jb): this warp's contiguous chunk, every lane its own row
            const int chunk = (jb + RG_WARPS - 1) / RG_WARPS;
            const int i0 = warp * chunk, i1 = min(i0 + chunk, jb);
            double best = -INFINITY;
            int arg = i0;
            int i = i0;
            for (; i + 3 < i1; i += 4) {
                double t[4];
#pragma unroll
                for (int u = 0; u < 4; ++u)
                    t[u] = reg_cell<AI>(i + u, __ldg(p.C + i + u), __ldg(p.L + i + u), p.P[i + u], p.nrv[i + u], row, p);
#pragma unroll
                for (int u = 0; u < 4; ++u)
                    if (t[u] > best) { best = t[u]; arg = i + u; }
            }
            for (; i < i1; ++i) {
                const double t = reg_cell<AI>(i, __ldg(p.C + i), __ldg(p.L + i), p.P[i], p.nrv[i], row, p);
                if (t > best) { best = t; arg = i; }
            }
            sPartV[warp][lane] = best;
            sPartA[warp][lane] = arg;
        }
        {   // the block's own triangle: column k = warp, row = lane (the P-independent parts)
            const int k = warp;
            if (k < lane && jb + lane < N) {
                const int ck = __ldg(p.C + jb + k), lk = __ldg(p.L + jb + k);
                sTriS[k][lane] = self_score<AI>(ck, lk, row, p.gtab, p.ltab);
                sTriR[k][lane] = p.use_len ? __ldg(p.lrtab + (row.lj - lk)) : 0.0;
            }
        }
        __syncthreads();
        if (warp == 0) {
            double best = -INFINITY;
            int arg = 0;
            for (int w = 0; w < RG_WARPS; ++w) {         // ascending column chunks: a later one wins only when strictly greater
                const double v = sPartV[w][lane];
                if (v > best) { best = v; arg = sPartA[w][lane]; }
            }
            const int rows = min(32, N - jb);
            double mine, my_nrv;
            int my_ns;
            reg_block_chain(jb, rows, p.ns, p.nrtab, p.use_num, p.use_len, p.pen, sTriS, sTriR, best, arg, mine, my_ns, my_nrv);
            if (lane < rows) {
                p.P[jb + lane] = mine;
                p.prev[jb + lane] = arg;
                p.ns[jb + lane] = my_ns;
                p.nrv[jb + lane] = my_nrv;
            }
        }
        __syncthreads();
    }
}

}  // namespace

// over ctx->dpL / dpC (launch_gather_candidates) -> dpP / dpPrev; d_lr / d_nr: device copies of the penalty tables or NULL
int launch_regularized_dp(pasio_ctx *ctx, i64 N, const double *d_lr, const double *d_nr, double add0)
{
    PASIO_TRY(pasio_reserve(ctx, ctx->dpP, (size_t)N * 8));
    PASIO_TRY(pasio_reserve(ctx, ctx->dpPrev, (size_t)N * 4));
    PASIO_TRY(pasio_reserve(ctx, ctx->dpPart, (size_t)N * 8));
    PASIO_TRY(pasio_reserve(ctx, ctx->dpPartArg, (size_t)N * 4));
    RegParams p;
    p.N = (int)N;
    p.L = ctx->dpL.as<int32_t>();
    p.C = ctx->dpC.as<int32_t>();
    p.P = ctx->dpP.as<double>();
    p.prev = ctx->dpPrev.as<int>();
    p.ns = ctx->dpPartArg.as<int>();
    p.nrv = ctx->dpPart.as<double>();
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
    TimingScope ts(ctx, TF_EXACT_DP);
    if (ctx->alpha_is_int) regularized_dp_kernel<true><<<1, RG_THREADS, 0, ctx->stream>>>(p);
    else regularized_dp_kernel<false><<<1, RG_THREADS, 0, ctx->stream>>>(p);
    CUDA_TRY(ctx, cudaGetLastError());
    ctx->last_cells = N * (N - 1) / 2;
    ctx->last_cells_skipped = 0;
    return PASIO_OK;
}
