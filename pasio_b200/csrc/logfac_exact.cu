// logfac_cumsum with the reference's rounding (SURVEY 8 f-4).
//
// The reference forms logfac_cumsum = hstack([0, np.cumsum(gammaln(counts + 1))])[candidates]
// (/root/reference/src/pasio/log_marginal_likelyhood.py:59-60): a strictly sequential float64 sum over every position of
// the contig.  A parallel scan adds the same terms in another order and differs in the last bits, which shows in the
// `bedgraph+length+LMM` column (scores - np.diff(logfac_cumsum), :76-78).  Here the sum is reproduced bit for bit:
//   1. the terms that are exactly 0.0 (counts 0 and 1: gammaln(1) = gammaln(2) = 0) cannot change a float64 running sum,
//      so only the positions with a non-zero term are kept: ballot stream compaction into (position, term) arrays;
//   2. every contig of the batch is summed left to right by ONE thread (s = fl(s + x), the reference's order and
//      rounding), contigs in parallel; the running sum after every kept term is stored;
//   3. a candidate's value is the running sum after the last kept term before it (binary search), 0 at the start of its
//      contig -- exactly what indexing the reference's cumulative array gives.
// Sparse coverage (DNase-like: ~1 % of the positions carry a non-zero term) makes step 2 short (2.5 M dependent adds for
// a chr1-sized contig); on dense coverage it is one add per position and PASIO_TUNE_LOGFAC_EXACT = 0 selects the
// three-pass parallel scan of scan.cu instead (1e-9 relative).
#include "common.cuh"

namespace {

constexpr int LX_THREADS = 256;
constexpr int LX_ITEMS = 8;
constexpr int LX_TILE = LX_THREADS * LX_ITEMS;

// gammaln(counts + 1) from the host-built table.  CHECK: the chunked variant runs before anybody has looked at the
// counts: a count outside the table (or negative) raises *flag and contributes nothing; the host then discards the sums and takes the ordinary path, which
// reports negative counts and grows the table
template <bool CHECK>
__device__ __forceinline__ double term_at(const i64 *__restrict__ counts, i64 p, const double *__restrict__ gtab, i64 ntab, int *flag)
{
    const i64 c = __ldg(counts + p);
    if (CHECK && (c < 0 || c + 1 >= ntab)) { *flag = 1; return 0.0; }
    return __ldg(gtab + c + 1);
}

// tile0: first tile of the launch (chunked variant: the tiles of the chunk that has just arrived)
template <bool CHECK>
__global__ void __launch_bounds__(LX_THREADS)
nonzero_count_kernel(const i64 *__restrict__ counts, i64 n, const double *__restrict__ gtab, unsigned *__restrict__ tile_count,
                     i64 tile0, i64 ntab, int *flag)
{
    const i64 tile = tile0 + blockIdx.x;
    const i64 base = tile * LX_TILE;
    int c = 0;
#pragma unroll
    for (int k = 0; k < LX_ITEMS; ++k) {
        const i64 p = base + (i64)k * LX_THREADS + threadIdx.x;
        if (p < n && term_at<CHECK>(counts, p, gtab, ntab, flag) != 0.0) ++c;
    }
    c = __reduce_add_sync(0xffffffffu, c);
    __shared__ int s[LX_THREADS / 32];
    if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        int t = 0;
        for (int w = 0; w < LX_THREADS / 32; ++w) t += s[w];
        tile_count[tile] = (unsigned)t;
    }
}

// exclusive scan of the tile counts in place (one CTA); total -> *total
// running != nullptr (chunked variant): the scan starts at running[0] (terms of the chunks before), which moves to
// running[1], and running[0] becomes the new total
__global__ void __launch_bounds__(1024)
tile_offsets_kernel(unsigned *tile_count, i64 n_tiles, i64 *total, i64 *running)
{
    __shared__ i64 s_warp[32];
    __shared__ i64 s_carry;
    if (threadIdx.x == 0) s_carry = running ? running[0] : 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (i64 base = 0; base < n_tiles; base += 1024) {
        const i64 i = base + threadIdx.x;
        const i64 x = i < n_tiles ? (i64)tile_count[i] : 0;
        i64 incl = x;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const i64 o = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += o;
        }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        i64 off = 0, tot = 0;
        for (int w = 0; w < 32; ++w) {
            const i64 t = s_warp[w];
            if (w < warp) off += t;
            tot += t;
        }
        const i64 carry = s_carry;
        __syncthreads();
        if (i < n_tiles) {
            const i64 ex = carry + off + incl - x;
            tile_count[i] = (unsigned)ex;                 // fewer than 2^31 positions per batch
        }
        if (threadIdx.x == 0) s_carry = carry + tot;
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        if (running) { running[1] = running[0]; running[0] = s_carry; }
        else *total = s_carry;
    }
}

template <bool CHECK>
__global__ void __launch_bounds__(LX_THREADS)
nonzero_scatter_kernel(const i64 *__restrict__ counts, i64 n, const double *__restrict__ gtab,
                       const unsigned *__restrict__ tile_offset, int32_t *__restrict__ pos_out, double *__restrict__ term_out,
                       i64 tile0, i64 ntab, int *flag)
{
    __shared__ int s_warp[LX_THREADS / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const i64 tile = tile0 + blockIdx.x;
    const i64 base = tile * LX_TILE;
    i64 at = tile_offset[tile];
#pragma unroll 1
    for (int k = 0; k < LX_ITEMS; ++k) {                  // positions ascend with k, then with the thread index
        const i64 p = base + (i64)k * LX_THREADS + threadIdx.x;
        double x = 0.0;
        if (p < n) x = term_at<CHECK>(counts, p, gtab, ntab, flag);
        const bool keep = x != 0.0;
        const unsigned bal = __ballot_sync(0xffffffffu, keep);
        if (lane == 0) s_warp[warp] = __popc(bal);
        __syncthreads();
        int woff = 0, tot = 0;
#pragma unroll
        for (int w = 0; w < LX_THREADS / 32; ++w) {
            const int c = s_warp[w];
            if (w < warp) woff += c;
            tot += c;
        }
        if (keep) {
            const i64 slot = at + woff + __popc(bal & ((1u << lane) - 1u));
            pos_out[slot] = (int32_t)p;
            term_out[slot] = x;
        }
        at += tot;
        __syncthreads();
    }
}

__device__ __forceinline__ i64 lower_bound_pos(const int32_t *__restrict__ pos, i64 n, i64 p)
{
    i64 lo = 0, hi = n;                                    // first kept term at a position >= p
    while (lo < hi) {
        const i64 mid = (lo + hi) >> 1;
        if ((i64)__ldg(pos + mid) < p) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// One thread per contig: the reference's left-to-right float64 sum over the contig's kept terms.
__global__ void sequential_sum_kernel(const int32_t *__restrict__ pos, double *__restrict__ terms_to_sums, i64 n_terms,
                                      const int32_t *__restrict__ bounds, i64 n_contigs, i64 *__restrict__ contig_first)
{
    for (i64 c = (i64)blockIdx.x * blockDim.x + threadIdx.x; c < n_contigs; c += (i64)gridDim.x * blockDim.x) {
        const i64 k0 = lower_bound_pos(pos, n_terms, __ldg(bounds + c)), k1 = lower_bound_pos(pos, n_terms, __ldg(bounds + c + 1));
        contig_first[c] = k0;
        double s = 0.0;
        i64 k = k0;
        for (; k + 7 < k1; k += 8) {                       // the loads of a group are independent of the running sum
            double x[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) x[u] = terms_to_sums[k + u];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                s = __dadd_rn(s, x[u]);
                terms_to_sums[k + u] = s;
            }
        }
        for (; k < k1; ++k) {
            s = __dadd_rn(s, terms_to_sums[k]);
            terms_to_sums[k] = s;
        }
    }
}

// Chunked variant, one contig: continue the running sum over the terms the chunk added, [running[1], running[0]).
__global__ void sequential_append_kernel(double *__restrict__ terms_to_sums, const i64 *__restrict__ running, double *carry)
{
    if (blockIdx.x || threadIdx.x) return;
    const i64 k0 = running[1], k1 = running[0];
    double s = *carry;
    i64 k = k0;
    for (; k + 7 < k1; k += 8) {
        double x[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) x[u] = terms_to_sums[k + u];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            s = __dadd_rn(s, x[u]);
            terms_to_sums[k + u] = s;
        }
    }
    for (; k < k1; ++k) {
        s = __dadd_rn(s, terms_to_sums[k]);
        terms_to_sums[k] = s;
    }
    *carry = s;
}

__device__ __forceinline__ double cumsum_at(const int32_t *__restrict__ pos, const double *__restrict__ sums, i64 n_terms,
                                            i64 first_of_contig, i64 p)
{
    const i64 k = lower_bound_pos(pos, n_terms, p);       // kept terms before position p: [first_of_contig, k)
    return k > first_of_contig ? sums[k - 1] : 0.0;
}

__device__ __forceinline__ i64 contig_of(const int32_t *__restrict__ bounds, i64 n_contigs, i64 p)
{
    i64 lo = 0, hi = n_contigs;                            // last c with bounds[c] <= p, p < bounds[n_contigs]
    while (hi - lo > 1) {
        const i64 mid = (lo + hi) >> 1;
        if ((i64)__ldg(bounds + mid) <= p) lo = mid; else hi = mid;
    }
    return lo;
}

// lmm[k] = scores[k] - (logfac_cumsum[k+1] - logfac_cumsum[k]) per segment (log_marginal_likelyhood.py:76-78); a segment
// never crosses a contig boundary, and its contig's cumulative array starts at 0
__global__ void lmm_exact_kernel(const double *__restrict__ scores, const int32_t *__restrict__ cand, i64 m,
                                 const int32_t *__restrict__ pos, const double *__restrict__ sums, i64 n_terms,
                                 const int32_t *__restrict__ bounds, i64 n_contigs, const i64 *__restrict__ contig_first,
                                 double *__restrict__ lmm)
{
    for (i64 k = (i64)blockIdx.x * blockDim.x + threadIdx.x; k < m - 1; k += (i64)gridDim.x * blockDim.x) {
        const i64 a = cand ? (i64)__ldg(cand + k) : k;
        const i64 b = cand ? (i64)__ldg(cand + k + 1) : k + 1;
        const i64 first = contig_first[contig_of(bounds, n_contigs, a)];
        const double la = cumsum_at(pos, sums, n_terms, first, a), lb = cumsum_at(pos, sums, n_terms, first, b);
        lmm[k] = __dsub_rn(scores[k], __dsub_rn(lb, la));
    }
}

// logfac_cumsum at the candidates of a single contig (the scorer attribute)
__global__ void logfac_at_candidates_kernel(const int32_t *__restrict__ cand, i64 m, const int32_t *__restrict__ pos,
                                            const double *__restrict__ sums, i64 n_terms, double *__restrict__ out)
{
    for (i64 k = (i64)blockIdx.x * blockDim.x + threadIdx.x; k < m; k += (i64)gridDim.x * blockDim.x) {
        const i64 p = cand ? (i64)__ldg(cand + k) : k;
        out[k] = cumsum_at(pos, sums, n_terms, 0, p);
    }
}

inline unsigned grid_for(pasio_ctx *ctx, i64 n)
{
    i64 g = (n + 255) / 256;
    const i64 cap = (i64)ctx->sm_count * 16;
    if (g > cap) g = cap;
    if (g < 1) g = 1;
    return (unsigned)g;
}

}  // namespace

// steps 1 and 2 for the loaded batch; cached in the context until the next load.  stream: the context's main stream, or
// its side stream when the sums are prefetched beside the rounds (pasio_logfac_prefetch)
int launch_logfac_exact(pasio_ctx *ctx, cudaStream_t stream)
{
    if (!stream) stream = ctx->stream;
    const i64 n = ctx->n;
    if (ctx->max_count + 2 > ctx->ntab[PASIO_TAB_LGAMMA]) {
        ctx->need[PASIO_TAB_LGAMMA] = ctx->max_count + 2;
        return pasio_fail(ctx, PASIO_E_TABLE_TOO_SHORT, "lgamma table has %lld entries, logfac needs %lld",
                          (long long)ctx->ntab[PASIO_TAB_LGAMMA], (long long)(ctx->max_count + 2));
    }
    const double *gtab = ctx->tab[PASIO_TAB_LGAMMA].as<double>();
    const i64 tiles = (n + LX_TILE - 1) / LX_TILE;
    PASIO_TRY(pasio_reserve(ctx, ctx->fscan, (size_t)tiles * 4 + 16));
    PASIO_TRY(pasio_reserve(ctx, ctx->lxFirst, (size_t)ctx->n_contigs * 8));
    unsigned *d_tiles = ctx->fscan.as<unsigned>();
    i64 *d_total = ctx->scalars.as<i64>() + 9;
    TimingScope ts(ctx, TF_SCORE, 4, stream);
    nonzero_count_kernel<false><<<(unsigned)tiles, LX_THREADS, 0, stream>>>(ctx->counts.as<i64>(), n, gtab, d_tiles, 0, 0, nullptr);
    tile_offsets_kernel<<<1, 1024, 0, stream>>>(d_tiles, tiles, d_total, nullptr);
    CUDA_TRY(ctx, cudaGetLastError());
    CUDA_TRY(ctx, cudaMemcpyAsync(ctx->h_scalars + 9, d_total, 8, cudaMemcpyDeviceToHost, stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(stream));
    const i64 n_terms = ctx->h_scalars[9];
    PASIO_TRY(pasio_reserve(ctx, ctx->lxPos, (size_t)(n_terms + 1) * 4));
    PASIO_TRY(pasio_reserve(ctx, ctx->lxSum, (size_t)(n_terms + 1) * 8));
    nonzero_scatter_kernel<false><<<(unsigned)tiles, LX_THREADS, 0, stream>>>(ctx->counts.as<i64>(), n, gtab, d_tiles,
                                                                                  ctx->lxPos.as<int32_t>(), ctx->lxSum.as<double>(), 0, 0, nullptr);
    const unsigned g = (unsigned)((ctx->n_contigs + 63) / 64);
    sequential_sum_kernel<<<g < 1 ? 1 : g, 64, 0, stream>>>(ctx->lxPos.as<int32_t>(), ctx->lxSum.as<double>(), n_terms,
                                                                 ctx->bounds.as<int32_t>(), ctx->n_contigs, ctx->lxFirst.as<i64>());
    CUDA_TRY(ctx, cudaGetLastError());
    ctx->lx_terms = n_terms;
    return PASIO_OK;
}

// ---- the same sums chunk by chunk behind an upload (pasio_contig_load_round with PASIO_TUNE_LOGFAC_EAGER) ----------
// One contig.  The chunks' terms are appended in order on `stream` (each launch waits for its chunk's event there), so the
// sequential sum -- 30 ms of one thread for a chr1-sized contig -- is nearly finished when the upload is, instead of
// starting then.  Device state (ctx->lxState): [0] terms so far, [1] terms before the current chunk, [2] running sum,
// [3] flag: a count outside the lgamma table or negative was seen (the sums are then discarded by the host).
int launch_logfac_exact_begin(pasio_ctx *ctx, cudaStream_t stream)
{
    const i64 n = ctx->n;
    const i64 tiles = (n + LX_TILE - 1) / LX_TILE;
    PASIO_TRY(pasio_reserve(ctx, ctx->fscan, (size_t)tiles * 4 + 16));
    PASIO_TRY(pasio_reserve(ctx, ctx->lxFirst, 8));
    PASIO_TRY(pasio_reserve(ctx, ctx->lxState, 64));
    PASIO_TRY(pasio_reserve(ctx, ctx->lxPos, (size_t)(n + 1) * 4));         // worst case: every position carries a term
    PASIO_TRY(pasio_reserve(ctx, ctx->lxSum, (size_t)(n + 1) * 8));
    CUDA_TRY(ctx, cudaMemsetAsync(ctx->lxState.p, 0, 64, stream));
    CUDA_TRY(ctx, cudaMemsetAsync(ctx->lxFirst.p, 0, 8, stream));
    return PASIO_OK;
}

int launch_logfac_exact_chunk(pasio_ctx *ctx, i64 p0, i64 p1, cudaStream_t stream)     // positions [p0, p1), p0 a multiple of the tile
{
    if (p1 <= p0) return PASIO_OK;
    const double *gtab = ctx->tab[PASIO_TAB_LGAMMA].as<double>();
    const i64 ntab = ctx->ntab[PASIO_TAB_LGAMMA];
    const i64 tile0 = p0 / LX_TILE, tiles = (p1 - p0 + LX_TILE - 1) / LX_TILE;
    unsigned *d_tiles = ctx->fscan.as<unsigned>();
    i64 *st = ctx->lxState.as<i64>();
    int *flag = reinterpret_cast<int *>(st + 3);
    TimingScope ts(ctx, TF_SCORE, 4, stream);
    nonzero_count_kernel<true><<<(unsigned)tiles, LX_THREADS, 0, stream>>>(ctx->counts.as<i64>(), p1, gtab, d_tiles, tile0, ntab, flag);
    tile_offsets_kernel<<<1, 1024, 0, stream>>>(d_tiles + tile0, tiles, nullptr, st);
    nonzero_scatter_kernel<true><<<(unsigned)tiles, LX_THREADS, 0, stream>>>(ctx->counts.as<i64>(), p1, gtab, d_tiles,
                                                                                 ctx->lxPos.as<int32_t>(), ctx->lxSum.as<double>(), tile0, ntab, flag);
    sequential_append_kernel<<<1, 32, 0, stream>>>(ctx->lxSum.as<double>(), st, reinterpret_cast<double *>(st + 2));
    CUDA_TRY(ctx, cudaGetLastError());
    return PASIO_OK;
}

// after the stream has finished: number of terms; *usable = false if the sums must be discarded
int logfac_exact_chunks_result(pasio_ctx *ctx, bool *usable)
{
    i64 h[4];
    CUDA_TRY(ctx, cudaMemcpy(h, ctx->lxState.p, sizeof h, cudaMemcpyDeviceToHost));
    ctx->lx_terms = h[0];
    *usable = (int)(h[3] & 0xffffffff) == 0;
    return PASIO_OK;
}

int launch_lmm_exact(pasio_ctx *ctx, const double *d_scores, double *d_lmm)
{
    TimingScope ts(ctx, TF_SCORE);
    lmm_exact_kernel<<<grid_for(ctx, ctx->m), 256, 0, ctx->stream>>>(d_scores, cur_cand(ctx), ctx->m, ctx->lxPos.as<int32_t>(),
                                                                    ctx->lxSum.as<double>(), ctx->lx_terms, ctx->bounds.as<int32_t>(),
                                                                    ctx->n_contigs, ctx->lxFirst.as<i64>(), d_lmm);
    CUDA_TRY(ctx, cudaGetLastError());
    return PASIO_OK;
}

int launch_logfac_at_candidates_exact(pasio_ctx *ctx, double *d_out)
{
    logfac_at_candidates_kernel<<<grid_for(ctx, ctx->m), 256, 0, ctx->stream>>>(cur_cand(ctx), ctx->m, ctx->lxPos.as<int32_t>(),
                                                                               ctx->lxSum.as<double>(), ctx->lx_terms, d_out);
    CUDA_TRY(ctx, cudaGetLastError());
    return PASIO_OK;
}

// the contig total (logfac_cumsum[-1]) of a single-contig context; of a batch, the last contig's total, which is 0 when
// that contig has no non-zero term (the last kept term then belongs to an earlier contig)
int logfac_exact_total(pasio_ctx *ctx, double *h_out)
{
    *h_out = 0.0;
    if (ctx->lx_terms == 0) return PASIO_OK;
    if (ctx->n_contigs > 1) {
        i64 first = 0;
        CUDA_TRY(ctx, cudaMemcpyAsync(&first, ctx->lxFirst.as<i64>() + (ctx->n_contigs - 1), 8, cudaMemcpyDeviceToHost, ctx->stream));
        CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
        if (first == ctx->lx_terms) return PASIO_OK;
    }
    CUDA_TRY(ctx, cudaMemcpyAsync(h_out, ctx->lxSum.as<double>() + (ctx->lx_terms - 1), 8, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return PASIO_OK;
}
