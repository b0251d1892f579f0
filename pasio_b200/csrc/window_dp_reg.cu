// K8: all windows of one sliding-window round with a regularised SquareSplitter as the window's base splitter
// (--split-number-regularization / --length-regularization with the `rounds` and `slidingwindow` algorithms).
//
// Replaces, per window, the chain of K4 (window_dp.cu) with split_with_normalizations in place of
// split_without_normalizations (/root/reference/src/pasio/splitters/square_splitter.py:29-65).  Per cell, in the
// reference's operation order (the cell of K6, regularized_dp.cu: reg_cell):
//     t = self_score(i, j) + P_i
//     t = t - NR[ns_i]               if the split-number term is on;  column 0: t = t + refund      :46-49
//     t = t - LR[L_j - L_i]          if the length term is on                                         :51-54
//     prev_j = first arg-max, ns_j = prev_j ? ns[prev_j] + 1 : 0, P_j = t[prev_j] + creation cost     :56-62
// NR[k] = lambda_n * f(k + 1) and LR[len] = lambda_L * g(len) are host-built tables (pasio_set_penalties), so the device
// adds exactly the doubles the reference adds.  Windows are local contigs exactly as in K4: positions and cumulative
// counts re-based to the window's first candidate, split numbers counted from 0 in every window.
//
// Every cell is evaluated: the far-column bound of K4 relies on F + P_i being convex in (u, len), which the
// -lambda_L / log(1 + len) term breaks.  Size classes as in K4 (the prepass in compact.cu sorts the windows): a warp
// per window up to 160 and up to 512 candidates, a persistent CTA per window above that.  A phase-2 window (explicit
// candidate lists) whose candidates all survived already is skipped: its survivors are a subset of its candidates.
#include "dp_core.cuh"

namespace {

constexpr int RW_THREADS = 256;
constexpr int RW_WARPS = RW_THREADS / 32;
constexpr int RW_MAX_CANDIDATES = 7168;         // largest fused window; its CTA fits 227 KB of shared memory
constexpr int RS_JB = 16;                        // rows per block step of the warp-per-window kernels
// the prepass sorts the windows into the small / medium lists by K4's limits: the per-warp structs are sized by the same
constexpr int RS_SMALL_N = WD_SMALL_MAX_CANDIDATES, RS_SMALL_WARPS = 8, RS_SMALL_CTAS = 5;
constexpr int RS_MEDIUM_N = WD_MEDIUM_MAX_CANDIDATES, RS_MEDIUM_WARPS = 4, RS_MEDIUM_CTAS = 4;

struct RegWinParams {
    WinGeom geom;
    i64 nwin;
    const int32_t *cand;        // nullptr: all positions
    const i64 *cg;
    const i64 *cgc;             // cg at the candidates; nullptr with all positions
    const uint32_t *cpbits;
    uint32_t *keepbits;
    const double *gtab;
    const double *ltab;
    const double *lrtab;        // LR[len] (use_len)
    const double *nrtab;        // NR[k]   (use_num)
    int use_num, use_len;
    double add0;                // first-column refund
    int constraint;
    int alpha_int;
    double alpha;
    double pen;
    int cap;
    u64 *cells;                 // algorithmic cells N(N-1)/2
    u64 *cells_skipped;         // cells of skipped (covered) windows
    unsigned *work_counter;
    const int32_t *list;        // window numbers: [0, n_p1) from the front, the rest from the back of the list_len-long list
    i64 n_p1, list_len;
};

template <bool AI>
__device__ __forceinline__ double rw_cell(int i, const ColRec &a, double nrvi, const RowConst<AI> &r, const RegWinParams &p)
{
    double t = __dadd_rn(self_score<AI>(a.C, a.L, r, p.gtab, p.ltab), a.P);
    if (p.use_num) {
        t = __dsub_rn(t, nrvi);
        if (i == 0) t = __dadd_rn(t, p.add0);
    }
    if (p.use_len) t = __dsub_rn(t, __ldg(p.lrtab + (r.lj - a.L)));
    return t;
}

// (A) of K4, by one warp: the window's candidates after the constraint filter, re-based, into col[]; returns their
// count.  covered (asked for): is every candidate of the window a survivor already?
__device__ int rw_load_window(const RegWinParams &p, i64 w, bool *covered, ColRec *col, i64 &first)
{
    const int lane = threadIdx.x & 31;
    i64 st, en;
    window_range(p.geom, w, st, en);
    const int nq = (int)(en - st);
    first = p.cand ? (i64)__ldg(p.cand + st) : st;
    const i64 last = p.cand ? (i64)__ldg(p.cand + en - 1) : en - 1;
    const i64 cg_first = p.cand ? __ldg(p.cgc + st) : __ldg(p.cg + first);
    const bool all_zero = (p.constraint == PASIO_CONSTRAINT_ZEROS) && ((p.cand ? __ldg(p.cgc + en - 1) : __ldg(p.cg + last)) == cg_first);
    int count = 0;
    if (!p.cand && p.constraint == PASIO_CONSTRAINT_CONSTANTS) {
        // all positions are candidates (round 1): the survivors of the NotConstant filter are the set bits of the
        // change-point bitmap inside [first, last], plus both ends
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
                col[k].L = (int)(pos - first);
                col[k].C = (int)(__ldg(p.cg + pos) - cg_first);
                ++k;
            }
            count += __shfl_sync(0xffffffffu, incl, 31);
        }
        return count;
    }
    int kept_all = 1;
    for (int base = 0; base < nq; base += 32) {
        const int q = base + lane;
        i64 pos = 0;
        bool take = false;
        if (q < nq) {
            pos = p.cand ? (i64)__ldg(p.cand + st + q) : st + q;
            if (q == 0 || q == nq - 1 || p.constraint == PASIO_CONSTRAINT_NONE) take = true;
            else if (p.constraint == PASIO_CONSTRAINT_CONSTANTS) take = bit_test(p.cpbits, pos);
            else take = !all_zero;
            if (covered && !((__ldcg(p.keepbits + (pos >> 5)) >> (pos & 31)) & 1u)) kept_all = 0;
        }
        const unsigned bal = __ballot_sync(0xffffffffu, take);
        if (take) {
            const int k = count + __popc(bal & ((1u << lane) - 1u));
            col[k].L = (int)(pos - first);
            col[k].C = (int)((p.cand ? __ldg(p.cgc + st + q) : __ldg(p.cg + pos)) - cg_first);
        }
        count += __popc(bal);
    }
    if (covered) *covered = __all_sync(0xffffffffu, kept_all);
    return count;
}

// (C): follow prev from the last candidate to 0 and mark the path in the position bitmap (one thread)
__device__ __forceinline__ void rw_backtrace(const RegWinParams &p, const ColRec *col, const unsigned short *prev, int N, i64 first)
{
    int k = N - 1;
    while (true) {
        const i64 pos = first + col[k].L;
        atomicOr(p.keepbits + (pos >> 5), 1u << (pos & 31));
        if (k == 0) break;
        k = prev[k];
    }
}

// ---- small and medium windows: one WARP per window ---------------------------------------------------------------
// 16-row block steps: lane = (row r, column phase ph); the finished columns are swept in two interleaved phases, the
// 16 x 16 triangle is resolved in order by shuffles.
template <int MAXN>
struct __align__(16) RegSmallWin {
    ColRec col[MAXN];
    double nrv[MAXN];           // NR[ns_i] of column i
    double triS[RS_JB * RS_JB]; // self score of (column k of the block, row r)
    double triR[RS_JB * RS_JB]; // LR of the same cell
    unsigned short ns[MAXN];
    unsigned short prev[MAXN];
};

template <bool AI, int MAXN, int NWARPS, int CTAS>
__global__ void __launch_bounds__(NWARPS * 32, CTAS)
small_window_dp_reg_kernel(RegWinParams p)
{
    extern __shared__ __align__(16) unsigned char smem[];
    const int lane = threadIdx.x & 31;
    RegSmallWin<MAXN> &W = reinterpret_cast<RegSmallWin<MAXN> *>(smem)[threadIdx.x >> 5];
    u64 my_cells = 0;
    while (true) {
        unsigned widx = 0;
        if (lane == 0) widx = atomicAdd(p.work_counter, 1u);
        widx = __shfl_sync(0xffffffffu, widx, 0);
        if ((i64)widx >= p.nwin) break;
        const i64 w = __ldg(p.list + widx);
        i64 first;
        const int N = rw_load_window(p, w, nullptr, W.col, first);
        if (lane == 0) {
            W.col[0].P = 0.0;
            W.prev[0] = 0;
            W.ns[0] = 0;
            W.nrv[0] = p.use_num ? __ldg(p.nrtab) : 0.0;
        }
        __syncwarp();

        const int r = lane & 15, ph = lane >> 4;
        for (int jb = 1; jb < N; jb += RS_JB) {
            const ColRec me = W.col[min(jb + r, N - 1)];
            const RowConst<AI> rc = make_row<AI>(me.C, me.L, p.alpha_int, p.alpha);
            double best = -INFINITY;
            int arg = ph;
#pragma unroll 4
            for (int i = ph; i < jb; i += 2) {
                const double t = rw_cell<AI>(i, W.col[i], W.nrv[i], rc, p);
                if (t > best) { best = t; arg = i; }
            }
            {   // the two column phases of a row: larger value, equal values keep the smaller column
                const double ob = __shfl_xor_sync(0xffffffffu, best, 16);
                const int oa = __shfl_xor_sync(0xffffffffu, arg, 16);
                if (ob > best || (ob == best && oa < arg)) { best = ob; arg = oa; }
            }
            for (int k = ph; k < r; k += 2)
                if (jb + r < N) {
                    const ColRec a = W.col[jb + k];
                    W.triS[k * RS_JB + r] = self_score<AI>(a.C, a.L, rc, p.gtab, p.ltab);
                    W.triR[k * RS_JB + r] = p.use_len ? __ldg(p.lrtab + (rc.lj - a.L)) : 0.0;
                }
            __syncwarp();
            double mine = 0.0, my_nrv = 0.0;
            int my_ns = 0;
            const int rows = min(RS_JB, N - jb);
            for (int k = 0; k < rows; ++k) {
                const int a = __shfl_sync(0xffffffffu, arg, k);                        // previous split of row jb + k
                const int from_block = __shfl_sync(0xffffffffu, my_ns, max(a - jb, 0));
                const int ns_k = a != 0 ? (a >= jb ? from_block : (int)W.ns[a]) + 1 : 0;
                const double pk = __shfl_sync(0xffffffffu, __dadd_rn(best, p.pen), k);
                const double nrvk = p.use_num ? __ldg(p.nrtab + ns_k) : 0.0;
                if (r == k) { mine = pk; my_ns = ns_k; my_nrv = nrvk; }
                if (r > k) {
                    double t = __dadd_rn(W.triS[k * RS_JB + r], pk);
                    if (p.use_num) t = __dsub_rn(t, nrvk);
                    if (p.use_len) t = __dsub_rn(t, W.triR[k * RS_JB + r]);
                    if (t > best) { best = t; arg = jb + k; }
                }
            }
            if (lane < RS_JB && jb + r < N) {
                W.col[jb + r].P = mine;
                W.prev[jb + r] = (unsigned short)arg;
                W.ns[jb + r] = (unsigned short)my_ns;
                W.nrv[jb + r] = my_nrv;
            }
            __syncwarp();
        }
        if (lane == 0) rw_backtrace(p, W.col, W.prev, N, first);
        my_cells += (u64)N * (u64)(N - 1) / 2;
        __syncwarp();
    }
    if (lane == 0 && my_cells) atomicAdd(p.cells, my_cells);
}

// ---- large windows: a persistent CTA per window ------------------------------------------------------------------
// 32-row block steps: every warp sweeps a contiguous chunk of the finished columns for the 32 rows (lane = row), the
// chunks are merged in ascending order (strict '>': np.argmax's first maximum) and warp 0 resolves the triangle.
__host__ __device__ inline size_t reg_window_smem_bytes(int cap)
{
    const size_t capr = (size_t)((cap + 31) & ~31);
    return capr * (16 + 8 + 2 + 2);     // col (L, C, P), nrv, ns, prev
}

template <bool AI>
__global__ void __launch_bounds__(RW_THREADS, 2)
window_dp_reg_kernel(RegWinParams p)
{
    extern __shared__ __align__(16) unsigned char smem[];
    __shared__ double sPartV[RW_WARPS][32];
    __shared__ int sPartA[RW_WARPS][32];
    __shared__ double sTriS[32][33], sTriR[32][33];
    __shared__ i64 sFirst;
    __shared__ int sN;          // candidates of the window, -1: covered (skipped)
    __shared__ unsigned sWork;  // the window's work index: a slot of its own, because after a covered window thread 0 takes
                                // the next index while other warps may still be reading sN
    const int capr = (p.cap + 31) & ~31;
    ColRec *col = reinterpret_cast<ColRec *>(smem);
    double *nrv = reinterpret_cast<double *>(col + capr);
    unsigned short *ns = reinterpret_cast<unsigned short *>(nrv + capr);
    unsigned short *prev = ns + capr;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    while (true) {
        if (tid == 0) sWork = atomicAdd(p.work_counter, 1u);
        __syncthreads();
        const i64 widx = sWork;
        __syncthreads();
        if (widx >= p.nwin) break;
        const bool second = widx >= p.n_p1;
        const i64 w = second ? (i64)__ldg(p.list + (p.list_len - 1 - (widx - p.n_p1))) : (i64)__ldg(p.list + widx);
        if (warp == 0) {
            i64 first;
            bool covered = false;
            const int n = rw_load_window(p, w, second ? &covered : nullptr, col, first);
            if (lane == 0) {
                sN = covered ? -1 : n;
                sFirst = first;
                col[0].P = 0.0;
                prev[0] = 0;
                ns[0] = 0;
                nrv[0] = p.use_num ? __ldg(p.nrtab) : 0.0;
                if (covered) {              // every candidate survived already: the window cannot add a survivor
                    const u64 c = (u64)n * (u64)(n - 1) / 2;
                    atomicAdd(p.cells, c);
                    atomicAdd(p.cells_skipped, c);
                }
            }
        }
        __syncthreads();
        const int N = sN;
        if (N < 0) continue;

        for (int jb = 1; jb < N; jb += 32) {
            const int j = min(jb + lane, N - 1);
            const ColRec me = col[j];
            const RowConst<AI> row = make_row<AI>(me.C, me.L, p.alpha_int, p.alpha);
            {   // finished columns [0, jb): this warp's contiguous chunk, every lane its own row
                const int chunk = (jb + RW_WARPS - 1) / RW_WARPS;
                const int i0 = warp * chunk, i1 = min(i0 + chunk, jb);
                double best = -INFINITY;
                int arg = i0;
#pragma unroll 4
                for (int i = i0; i < i1; ++i) {
                    const double t = rw_cell<AI>(i, col[i], nrv[i], row, p);
                    if (t > best) { best = t; arg = i; }
                }
                sPartV[warp][lane] = best;
                sPartA[warp][lane] = arg;
            }
#pragma unroll
            for (int k = warp; k < 32; k += RW_WARPS) {     // the block's own triangle (P-independent parts)
                if (k < lane && jb + lane < N) {
                    const ColRec a = col[jb + k];
                    sTriS[k][lane] = self_score<AI>(a.C, a.L, row, p.gtab, p.ltab);
                    sTriR[k][lane] = p.use_len ? __ldg(p.lrtab + (row.lj - a.L)) : 0.0;
                }
            }
            __syncthreads();
            if (warp == 0) {
                double best = -INFINITY;
                int arg = 0;
#pragma unroll
                for (int w2 = 0; w2 < RW_WARPS; ++w2) {     // ascending column chunks: a later one wins only when strictly greater
                    const double v = sPartV[w2][lane];
                    if (v > best) { best = v; arg = sPartA[w2][lane]; }
                }
                const int rows = min(32, N - jb);
                double mine = 0.0, my_nrv = 0.0;
                int my_ns = 0;
                for (int k = 0; k < rows; ++k) {
                    const int a = __shfl_sync(0xffffffffu, arg, k);
                    const int from_block = __shfl_sync(0xffffffffu, my_ns, max(a - jb, 0));
                    const int ns_k = a != 0 ? (a >= jb ? from_block : (int)ns[a]) + 1 : 0;
                    const double pk = __shfl_sync(0xffffffffu, __dadd_rn(best, p.pen), k);
                    const double nrvk = p.use_num ? __ldg(p.nrtab + ns_k) : 0.0;
                    if (lane == k) { mine = pk; my_ns = ns_k; my_nrv = nrvk; }
                    if (lane > k) {
                        double t = __dadd_rn(sTriS[k][lane], pk);
                        if (p.use_num) t = __dsub_rn(t, nrvk);
                        if (p.use_len) t = __dsub_rn(t, sTriR[k][lane]);
                        if (t > best) { best = t; arg = jb + k; }
                    }
                }
                if (lane < rows) {
                    col[jb + lane].P = mine;
                    prev[jb + lane] = (unsigned short)arg;
                    ns[jb + lane] = (unsigned short)my_ns;
                    nrv[jb + lane] = my_nrv;
                }
            }
            __syncthreads();
        }
        if (tid == 0) {
            rw_backtrace(p, col, prev, N, sFirst);
            atomicAdd(p.cells, (u64)N * (u64)(N - 1) / 2);
        }
        __syncthreads();
    }
}

}  // namespace

int window_dp_reg_max_candidates(pasio_ctx *ctx)
{
    int cap = RW_MAX_CANDIDATES;
    while (cap > 32 && reg_window_smem_bytes(cap) + 20480 > (size_t)ctx->smem_optin) cap -= 32;
    return cap;
}

int launch_window_dp_reg(pasio_ctx *ctx, i64 nwin, int wsize, int wshift, int constraint, bool keep_cell_counters)
{
    RegWinParams p;
    p.geom = make_geom(ctx, wsize, wshift);
    p.cand = cur_cand(ctx);
    p.cg = ctx->cg.as<i64>();
    p.cgc = cur_cand_cg(ctx);
    p.cpbits = ctx->cpbits.as<uint32_t>();
    p.keepbits = ctx->keepbits.as<uint32_t>();
    p.gtab = ctx->tab[ctx->alpha_is_int ? PASIO_TAB_LGAMMA : PASIO_TAB_LGAMMA_ALPHA].as<double>();
    p.ltab = ctx->tab[PASIO_TAB_LOG].as<double>();
    p.use_num = ctx->pen_num;
    p.use_len = ctx->pen_len;
    p.nrtab = ctx->pen_num ? ctx->penNR.as<double>() : nullptr;
    p.lrtab = ctx->pen_len ? ctx->penLR.as<double>() : nullptr;
    p.add0 = ctx->pen_refund;
    p.constraint = constraint;
    p.alpha_int = (int)ctx->alpha_int;
    p.alpha = ctx->alpha;
    p.pen = ctx->pen;
    i64 cap = (i64)wsize + 1;
    if (cap > ctx->m) cap = ctx->m;
    if (cap > window_dp_reg_max_candidates(ctx))
        return pasio_fail(ctx, PASIO_E_TOO_LARGE, "regularised window of %lld candidates does not fit one CTA's shared memory (max %d)",
                          (long long)cap, window_dp_reg_max_candidates(ctx));
    if (ctx->pen_num && ctx->n_pen_nr < cap)
        return pasio_fail(ctx, PASIO_E_ARG, "split-number penalty table has %lld entries, a window may have %lld candidates",
                          (long long)ctx->n_pen_nr, (long long)cap);
    p.cap = (int)cap;
    p.cells = ctx->scalars.as<u64>() + 10;
    p.cells_skipped = ctx->scalars.as<u64>() + 12;
    if (keep_cell_counters) CUDA_TRY(ctx, cudaMemsetAsync(ctx->scalars.as<u64>() + 11, 0, 8, ctx->stream));
    else CUDA_TRY(ctx, cudaMemsetAsync(ctx->scalars.as<u64>() + 10, 0, 24, ctx->stream));
    CUDA_TRY(ctx, cudaMemsetAsync(ctx->scalars.as<u64>() + 15, 0, 8, ctx->stream));

    // the work lists of the prepass (launch_window_prepass with classification)
    if (ctx->n_small + ctx->n_medium + ctx->n_large != nwin)
        return pasio_fail(ctx, PASIO_E_STATE, "regularised window DP without the prepass work lists");
    const i64 n_small = ctx->n_small, n_medium = ctx->n_medium, n_large = ctx->n_large, n_p1 = ctx->n_large_p1;
    ctx->n_small = ctx->n_medium = ctx->n_large = ctx->n_large_p1 = -1;           // the lists are consumed
    TimingScope ts_all(ctx, TF_WINDOW_DP, 0);

    auto launch = [&](auto kern, const int32_t *list, i64 n, i64 np1, int threads, int per_cta, int ctas, size_t smem_bytes,
                      unsigned *counter) -> int {
        if (n <= 0) return PASIO_OK;
        RegWinParams ps = p;
        ps.list = list;
        ps.nwin = n;
        ps.n_p1 = np1;
        ps.list_len = nwin;
        ps.work_counter = counter;
        CUDA_TRY(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes));
        int resident = ctas;
        CUDA_TRY(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&resident, kern, threads, smem_bytes));
        if (resident < 1) resident = 1;
        if (resident > ctas) resident = ctas;
        i64 g = (n + per_cta - 1) / per_cta;
        if (g > (i64)ctx->sm_count * resident) g = (i64)ctx->sm_count * resident;   // persistent: one resident wave
        ctx->fam_launches[TF_WINDOW_DP] += 1;
        kern<<<(unsigned)g, threads, smem_bytes, ctx->stream>>>(ps);
        CUDA_TRY(ctx, cudaGetLastError());
        return PASIO_OK;
    };
    unsigned *c_large = ctx->scalars.as<unsigned>() + 2 * 11, *c_small = ctx->scalars.as<unsigned>() + 2 * 15, *c_medium = c_small + 1;
    const size_t sm_small = sizeof(RegSmallWin<RS_SMALL_N>) * RS_SMALL_WARPS,
                 sm_medium = sizeof(RegSmallWin<RS_MEDIUM_N>) * RS_MEDIUM_WARPS, sm_large = reg_window_smem_bytes(p.cap);
    if (ctx->alpha_is_int) {
        PASIO_TRY(launch(window_dp_reg_kernel<true>, ctx->win_large.as<int32_t>(), n_large, n_p1, RW_THREADS, 1, 2, sm_large, c_large));
        PASIO_TRY(launch(small_window_dp_reg_kernel<true, RS_MEDIUM_N, RS_MEDIUM_WARPS, RS_MEDIUM_CTAS>, ctx->win_medium.as<int32_t>(),
                         n_medium, n_medium, RS_MEDIUM_WARPS * 32, RS_MEDIUM_WARPS, RS_MEDIUM_CTAS, sm_medium, c_medium));
        PASIO_TRY(launch(small_window_dp_reg_kernel<true, RS_SMALL_N, RS_SMALL_WARPS, RS_SMALL_CTAS>, ctx->win_small.as<int32_t>(),
                         n_small, n_small, RS_SMALL_WARPS * 32, RS_SMALL_WARPS, RS_SMALL_CTAS, sm_small, c_small));
    } else {
        PASIO_TRY(launch(window_dp_reg_kernel<false>, ctx->win_large.as<int32_t>(), n_large, n_p1, RW_THREADS, 1, 2, sm_large, c_large));
        PASIO_TRY(launch(small_window_dp_reg_kernel<false, RS_MEDIUM_N, RS_MEDIUM_WARPS, RS_MEDIUM_CTAS>, ctx->win_medium.as<int32_t>(),
                         n_medium, n_medium, RS_MEDIUM_WARPS * 32, RS_MEDIUM_WARPS, RS_MEDIUM_CTAS, sm_medium, c_medium));
        PASIO_TRY(launch(small_window_dp_reg_kernel<false, RS_SMALL_N, RS_SMALL_WARPS, RS_SMALL_CTAS>, ctx->win_small.as<int32_t>(),
                         n_small, n_small, RS_SMALL_WARPS * 32, RS_SMALL_WARPS, RS_SMALL_CTAS, sm_small, c_small));
    }
    return PASIO_OK;
}
