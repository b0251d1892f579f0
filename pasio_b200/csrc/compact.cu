// K2: survivor bitmap -> sorted candidate list (stream compaction), plus the small per-round
// helpers around it: boundary ranks, window requirements, candidate validation.
//
// Replaces the set-union + sort of SlidingWindowReducer.reduce_candidate_list
// (/root/reference/src/pasio/splitters/sliding_window_reducer.py:22-29): windows scatter
// survivor bits into a position bitmap, and one ordered compaction of the bitmap yields the
// next round's ascending candidate array.  HBM-trivial: (n+1)/8 bytes read, 4 B per survivor.
#include "common.cuh"

namespace {

constexpr int CP_THREADS = 256;
constexpr int CP_WORDS = 4;                       // words per thread
constexpr int CP_TILE = CP_THREADS * CP_WORDS;    // words per block

__global__ void __launch_bounds__(CP_THREADS)
popc_block_sums(const uint32_t *__restrict__ bits, i64 nwords, int *__restrict__ blocksum)
{
    __shared__ int s_warp[CP_THREADS / 32];
    const i64 base = (i64)blockIdx.x * CP_TILE + (i64)threadIdx.x * CP_WORDS;
    int c = 0;
#pragma unroll
    for (int k = 0; k < CP_WORDS; ++k)
        if (base + k < nwords) c += __popc(__ldg(bits + base + k));
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) c += __shfl_xor_sync(0xffffffffu, c, d);
    if ((threadIdx.x & 31) == 0) s_warp[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        int t = 0;
        for (int w = 0; w < CP_THREADS / 32; ++w) t += s_warp[w];
        blocksum[blockIdx.x] = t;
    }
}

__device__ __forceinline__ int block_excl_scan_int(int x, int *s_warp, int *total)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int incl = x;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        int o = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += o;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    int off = 0, tot = 0;
    for (int w = 0; w < CP_THREADS / 32; ++w) {
        int t = s_warp[w];
        if (w < warp) off += t;
        tot += t;
    }
    __syncthreads();
    *total = tot;
    return off + incl - x;
}

__global__ void __launch_bounds__(CP_THREADS)
scan_block_sums(int *blocksum, i64 nblocks, i64 *total_out)
{
    __shared__ int s_warp[CP_THREADS / 32];
    int carry = 0;
    for (i64 base = 0; base < nblocks; base += CP_THREADS) {
        i64 i = base + threadIdx.x;
        int x = (i < nblocks) ? blocksum[i] : 0;
        int tot;
        int ex = block_excl_scan_int(x, s_warp, &tot);
        if (i < nblocks) blocksum[i] = carry + ex;
        carry += tot;
    }
    if (threadIdx.x == 0) *total_out = carry;
}

__global__ void __launch_bounds__(CP_THREADS)
scatter_bits(const uint32_t *__restrict__ bits, i64 nwords, const int *__restrict__ blockprefix,
             int32_t *__restrict__ out, const i64 *__restrict__ cg, i64 *__restrict__ cg_out)
{
    __shared__ int s_warp[CP_THREADS / 32];
    const i64 base = (i64)blockIdx.x * CP_TILE + (i64)threadIdx.x * CP_WORDS;
    uint32_t w[CP_WORDS];
    int c = 0;
#pragma unroll
    for (int k = 0; k < CP_WORDS; ++k) {
        w[k] = (base + k < nwords) ? __ldg(bits + base + k) : 0u;
        c += __popc(w[k]);
    }
    int tot;
    int off = blockprefix[blockIdx.x] + block_excl_scan_int(c, s_warp, &tot);
#pragma unroll
    for (int k = 0; k < CP_WORDS; ++k) {
        uint32_t x = w[k];
        const int32_t pos0 = (int32_t)((base + k) << 5);
        while (x) {
            int b = __ffs(x) - 1;
            out[off] = pos0 + b;
            cg_out[off] = __ldg(cg + pos0 + b);       // the candidate's prefix sum travels with it: the window kernels read
            ++off;                                    // both arrays coalesced instead of gathering 8 bytes per 32-byte sector
            x &= x - 1;
        }
    }
}

// every contig boundary survives (sliding_window_reducer.py:22 starts the union from {0, len(counts)}): a window shift
// larger than the window size leaves candidates, the last one among them, in no window
__global__ void mark_boundaries_kernel(const int32_t *__restrict__ bounds, i64 nb, uint32_t *keepbits)
{
    i64 c = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= nb) return;
    const int32_t b = bounds[c];
    atomicOr(keepbits + (b >> 5), 1u << (b & 31));
}

// index of every contig boundary in the (sorted) candidate list
__global__ void boundary_ranks_kernel(const int32_t *__restrict__ cand, i64 m,
                                      const int32_t *__restrict__ bounds, i64 nb, int32_t *__restrict__ brank)
{
    i64 c = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= nb) return;
    int32_t b = bounds[c];
    if (!cand) { brank[c] = b; return; }
    i64 lo = 0, hi = m;               // lower_bound
    while (lo < hi) {
        i64 mid = (lo + hi) >> 1;
        if (__ldg(cand + mid) < b) lo = mid + 1; else hi = mid;
    }
    brank[c] = (int32_t)lo;
}

// largest window span (nt) and window count: the table lengths a round needs.  Optionally sorts the windows into
// two work lists by an upper bound of their candidate count after the constraint filter: small windows go to the
// warp-per-window kernel, the others to the CTA-per-window kernel (window_dp.cu).
__global__ void window_prepass_kernel(WinGeom g, i64 w_begin, i64 nwin, const int32_t *__restrict__ cand,
                                      const i64 *__restrict__ cg, u64 *out /* [0]=span, [1]=count */,
                                      const uint32_t *__restrict__ cpbits, int constraint, int small_max, int medium_max,
                                      int32_t *__restrict__ small_list, int32_t *__restrict__ medium_list,
                                      int32_t *__restrict__ large_list, int p1_stride, unsigned char *__restrict__ done_flags,
                                      unsigned *list_counts /* [0]=small, [1]=medium, [2]=large phase 1, [3]=large phase 2 */)
{
    i64 span = 0, cnt = 0;
    for (i64 wi = (i64)blockIdx.x * blockDim.x + threadIdx.x; wi < nwin; wi += (i64)gridDim.x * blockDim.x) {
        const i64 w = w_begin + wi;
        i64 st, en;
        window_range(g, w, st, en);
        i64 a = cand ? __ldg(cand + st) : st;
        i64 b = cand ? __ldg(cand + en - 1) : en - 1;
        span = max(span, b - a);
        cnt = max(cnt, __ldg(cg + b) - __ldg(cg + a));
        if (small_list) {
            i64 est = en - st;
            if (est > small_max && !cand && constraint == PASIO_CONSTRAINT_CONSTANTS) {   // (est = all positions of the window here)
                // all positions are candidates: change points strictly inside (a, b), plus both ends
                est = 2;
                for (i64 word = (a + 1) >> 5; word <= (b - 1) >> 5 && est <= medium_max; ++word) {
                    uint32_t x = __ldg(cpbits + word);
                    if (word == (a + 1) >> 5) x &= 0xffffffffu << ((a + 1) & 31);
                    if (word == (b - 1) >> 5) x &= 0xffffffffu >> (31 - ((b - 1) & 31));
                    est += __popc(x);
                }
            }
            const bool large_p1 = est > medium_max && (p1_stride <= 1 || w % p1_stride == 0);
            done_flags[wi] = large_p1 ? 0 : 1;          // a phase-2 window waits for the phase-1 windows next to it; others never block it
            if (est <= small_max) small_list[atomicAdd(list_counts, 1u)] = (int32_t)w;
            else if (est <= medium_max) medium_list[atomicAdd(list_counts + 1, 1u)] = (int32_t)w;
            else if (p1_stride <= 1 || w % p1_stride == 0) large_list[atomicAdd(list_counts + 2, 1u)] = (int32_t)w;   // from the front
            else large_list[nwin - 1 - atomicAdd(list_counts + 3, 1u)] = (int32_t)w;                               // from the back
        }
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        span = max(span, __shfl_xor_sync(0xffffffffu, span, d));
        cnt = max(cnt, __shfl_xor_sync(0xffffffffu, cnt, d));
    }
    if ((threadIdx.x & 31) == 0) {
        atomicMax(out + 0, (u64)span);
        atomicMax(out + 1, (u64)cnt);
    }
}

// assert_correct_split_candidates (log_marginal_likelyhood.py:36-40) + boundaries present
__global__ void validate_candidates_kernel(const int32_t *__restrict__ cand, i64 m, i64 n,
                                           const int32_t *__restrict__ bounds, const int32_t *__restrict__ brank,
                                           i64 nb, i64 *bad)
{
    i64 stride = (i64)gridDim.x * blockDim.x;
    i64 t = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    bool b = false;
    for (i64 i = t; i < m; i += stride) {
        int32_t v = __ldg(cand + i);
        if (i == 0 && v != 0) b = true;
        if (i == m - 1 && v != n) b = true;
        if (i > 0 && __ldg(cand + i - 1) >= v) b = true;
    }
    for (i64 c = t; c < nb; c += stride) {
        int32_t r = brank[c];
        if (r < 0 || r >= m || __ldg(cand + r) != bounds[c]) b = true;
    }
    if (b) *bad = 1;
}

// constants_reducer.py:5-21 over the whole contig: mark the surviving candidates in the position bitmap
__global__ void filter_candidates_kernel(const int32_t *__restrict__ cand, i64 m, int constraint, int all_zero,
                                         const uint32_t *__restrict__ cpbits, uint32_t *keepbits)
{
    for (i64 k = (i64)blockIdx.x * blockDim.x + threadIdx.x; k < m; k += (i64)gridDim.x * blockDim.x) {
        const i64 pos = cand ? (i64)__ldg(cand + k) : k;
        bool keep = (k == 0) || (k == m - 1);
        if (!keep) {
            if (constraint == PASIO_CONSTRAINT_CONSTANTS) keep = bit_test(cpbits, pos);
            else if (constraint == PASIO_CONSTRAINT_ZEROS) keep = !all_zero;
            else keep = true;
        }
        if (keep) atomicOr(keepbits + (pos >> 5), 1u << (pos & 31));
    }
}

}  // namespace

int launch_filter_candidates(pasio_ctx *ctx, int constraint)
{
    const size_t bit_bytes = (size_t)((ctx->n + 1 + 31) / 32 + 2) * 4;
    CUDA_TRY(ctx, cudaMemsetAsync(ctx->keepbits.p, 0, bit_bytes, ctx->stream));
    i64 g = (ctx->m + 255) / 256;
    if (g > (i64)ctx->sm_count * 16) g = (i64)ctx->sm_count * 16;
    TimingScope ts(ctx, TF_COMPACT);
    filter_candidates_kernel<<<(unsigned)g, 256, 0, ctx->stream>>>(cur_cand(ctx), ctx->m, constraint, ctx->total == 0,
                                                                  ctx->cpbits.as<uint32_t>(), ctx->keepbits.as<uint32_t>());
    CUDA_TRY(ctx, cudaGetLastError());
    return PASIO_OK;
}

WinGeom make_geom(const pasio_ctx *ctx, int wsize, int wshift)
{
    WinGeom g;
    if (ctx->n_contigs > 1) {
        g.st_tab = ctx->win_st.as<int32_t>();
        g.en_tab = ctx->win_en.as<int32_t>();
    } else {
        g.st_tab = nullptr;
        g.en_tab = nullptr;
    }
    g.m = ctx->m;
    g.wsize = wsize;
    g.wshift = wshift;
    return g;
}

int launch_compact_keepbits(pasio_ctx *ctx, int slot, i64 *h_count)
{
    int32_t *d_out = ctx->cand[slot].as<int32_t>();
    PASIO_TRY(pasio_reserve(ctx, ctx->candC[slot], ctx->cand[slot].bytes * 2));
    const i64 nwords = (ctx->n + 1 + 31) / 32;
    const i64 nblocks = (nwords + CP_TILE - 1) / CP_TILE;
    PASIO_TRY(pasio_reserve(ctx, ctx->blocksum, (size_t)nblocks * sizeof(int)));
    const uint32_t *bits = ctx->keepbits.as<uint32_t>();
    int *bs = ctx->blocksum.as<int>();
    i64 *d_total = ctx->scalars.as<i64>() + 4;
    {
        TimingScope ts(ctx, TF_COMPACT, 4);
        const i64 nb = ctx->n_contigs + 1;
        mark_boundaries_kernel<<<(unsigned)((nb + 255) / 256), 256, 0, ctx->stream>>>(ctx->bounds.as<int32_t>(), nb, ctx->keepbits.as<uint32_t>());
        popc_block_sums<<<(unsigned)nblocks, CP_THREADS, 0, ctx->stream>>>(bits, nwords, bs);
        scan_block_sums<<<1, CP_THREADS, 0, ctx->stream>>>(bs, nblocks, d_total);
        scatter_bits<<<(unsigned)nblocks, CP_THREADS, 0, ctx->stream>>>(bits, nwords, bs, d_out, ctx->cg.as<i64>(), ctx->candC[slot].as<i64>());
    }
    CUDA_TRY(ctx, cudaGetLastError());
    CUDA_TRY(ctx, cudaMemcpyAsync(ctx->h_scalars + 4, d_total, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    *h_count = ctx->h_scalars[4];
    return PASIO_OK;
}

int launch_boundary_ranks(pasio_ctx *ctx)
{
    const i64 nb = ctx->n_contigs + 1;
    boundary_ranks_kernel<<<(unsigned)((nb + 255) / 256), 256, 0, ctx->stream>>>(
        cur_cand(ctx), ctx->m, ctx->bounds.as<int32_t>(), nb, ctx->brank.as<int32_t>());
    CUDA_TRY(ctx, cudaGetLastError());
    return PASIO_OK;
}

int launch_window_prepass(pasio_ctx *ctx, i64 nwin, int wsize, int wshift, i64 *h_max_span, i64 *h_max_cnt,
                          int classify_constraint, i64 w_begin)
{
    u64 *d_out = ctx->scalars.as<u64>() + 6;
    CUDA_TRY(ctx, cudaMemsetAsync(d_out, 0, 16, ctx->stream));
    unsigned *d_counts = ctx->scalars.as<unsigned>() + 2 * 13;      // scalars[13], [14]: small / medium / large list lengths
    const bool classify = classify_constraint >= 0;
    if (classify) {
        if (w_begin + nwin > 2147483647LL) return pasio_fail(ctx, PASIO_E_TOO_LARGE, "too many windows");
        PASIO_TRY(pasio_reserve(ctx, ctx->win_small, (size_t)nwin * 4));
        PASIO_TRY(pasio_reserve(ctx, ctx->win_medium, (size_t)nwin * 4));
        PASIO_TRY(pasio_reserve(ctx, ctx->win_large, (size_t)nwin * 4));
        PASIO_TRY(pasio_reserve(ctx, ctx->win_flags, (size_t)nwin + 16));
        CUDA_TRY(ctx, cudaMemsetAsync(d_counts, 0, 16, ctx->stream));
    }
    unsigned blocks = (unsigned)((nwin + 255) / 256);
    if (blocks > (unsigned)ctx->sm_count * 8) blocks = ctx->sm_count * 8;
    if (blocks == 0) blocks = 1;
    {
        TimingScope ts(ctx, TF_COMPACT);
        window_prepass_kernel<<<blocks, 256, 0, ctx->stream>>>(
            make_geom(ctx, wsize, wshift), w_begin, nwin, cur_cand(ctx), ctx->cg.as<i64>(), d_out, ctx->cpbits.as<uint32_t>(),
            classify_constraint, small_window_max_candidates(), medium_window_max_candidates(),
            classify ? ctx->win_small.as<int32_t>() : nullptr, classify ? ctx->win_medium.as<int32_t>() : nullptr,
            classify ? ctx->win_large.as<int32_t>() : nullptr,
            // phase 1 = every (size / shift)-th window: together they cover every candidate; a phase-2 window whose
            // candidates all survived phase 1 cannot add a survivor (window_dp.cu).  Explicit candidate lists only.
            (cur_cand(ctx) && wshift > 0) ? wsize / wshift : 0, classify ? ctx->win_flags.as<unsigned char>() : nullptr, d_counts);
    }
    CUDA_TRY(ctx, cudaGetLastError());
    CUDA_TRY(ctx, cudaMemcpyAsync(ctx->h_scalars + 6, d_out, 16, cudaMemcpyDeviceToHost, ctx->stream));
    if (classify) CUDA_TRY(ctx, cudaMemcpyAsync(ctx->h_scalars + 13, d_counts, 16, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    *h_max_span = ctx->h_scalars[6];
    *h_max_cnt = ctx->h_scalars[7];
    if (classify) {
        const unsigned *c = reinterpret_cast<const unsigned *>(ctx->h_scalars + 13);
        ctx->n_small = c[0];
        ctx->n_medium = c[1];
        ctx->n_large = (i64)c[2] + (i64)c[3];
        ctx->n_large_p1 = c[2];
    }
    return PASIO_OK;
}

int launch_validate_candidates(pasio_ctx *ctx, i64 *h_bad)
{
    i64 *d_bad = ctx->scalars.as<i64>() + 5;
    CUDA_TRY(ctx, cudaMemsetAsync(d_bad, 0, 8, ctx->stream));
    validate_candidates_kernel<<<ctx->sm_count * 4, 256, 0, ctx->stream>>>(
        ctx->cand[ctx->cur].as<int32_t>(), ctx->m, ctx->n, ctx->bounds.as<int32_t>(),
        ctx->brank.as<int32_t>(), ctx->n_contigs + 1, d_bad);
    CUDA_TRY(ctx, cudaGetLastError());
    CUDA_TRY(ctx, cudaMemcpyAsync(ctx->h_scalars + 5, d_bad, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    *h_bad = ctx->h_scalars[5];
    return PASIO_OK;
}
