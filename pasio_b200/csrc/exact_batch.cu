// The per-contig pieces of pasio_square_split_batch (api.cu): SquareSplitter.split (square_splitter.py:67-109) of every
// contig's slice of the candidate list of a loaded batch.  Lists that fit one K4 window run as whole-list windows of the
// window DP; the longer ones run through K3 one after another, and these kernels carry them in and out of K3's
// contig-local arrays:
//   - batch_contig_stats_kernel: per contig span and total count -> the table lengths and the 32-bit limit, checked
//     before any DP runs;
//   - gather_slice_kernel: one contig's candidates -> dpL / dpC, re-based to its first candidate (what
//     launch_gather_candidates does for the whole list);
//   - back-trace by pointer doubling over dpPrev, whose marks are OR-ed into the survivor bitmap at the contig's own
//     positions.  Unlike launch_backtrace_mark it does not clear the bitmap: the short lists' windows and every earlier
//     long list have already written their splits there.
#include "common.cuh"

namespace {

// out[0] = largest span (nt), out[1] = largest total count, out[2] = first contig whose total + alpha_int does not fit
// the 32-bit DP index (all ones: none)
__global__ void batch_contig_stats_kernel(const int32_t *__restrict__ bounds, i64 n_contigs, const i64 *__restrict__ cg,
                                          i64 alpha_int, u64 *out)
{
    i64 span = 0, cnt = 0;
    for (i64 c = (i64)blockIdx.x * blockDim.x + threadIdx.x; c < n_contigs; c += (i64)gridDim.x * blockDim.x) {
        const i64 a = __ldg(bounds + c), b = __ldg(bounds + c + 1);
        const i64 t = __ldg(cg + b) - __ldg(cg + a);
        span = max(span, b - a);
        cnt = max(cnt, t);
        if (t + alpha_int >= 2147483647LL) atomicMin(out + 2, (u64)c);
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

// candidates [b0, b0 + m) of the list (implicit list: positions b0 ..) -> L / C relative to the first of them
__global__ void gather_slice_kernel(const int32_t *__restrict__ cand, i64 b0, i64 m, const i64 *__restrict__ cg,
                                    int32_t *__restrict__ L, int32_t *__restrict__ C)
{
    const i64 first = cand ? (i64)__ldg(cand + b0) : b0;
    const i64 cg_first = __ldg(cg + first);
    for (i64 k = (i64)blockIdx.x * blockDim.x + threadIdx.x; k < m; k += (i64)gridDim.x * blockDim.x) {
        const i64 pos = cand ? (i64)__ldg(cand + b0 + k) : b0 + k;
        L[k] = (int32_t)(pos - first);
        C[k] = (int32_t)(__ldg(cg + pos) - cg_first);
    }
}

__global__ void slice_bt_init_kernel(const int *__restrict__ prev, i64 N, int *jump, uint8_t *mark)
{
    for (i64 k = (i64)blockIdx.x * blockDim.x + threadIdx.x; k < N; k += (i64)gridDim.x * blockDim.x) {
        jump[k] = prev[k];
        mark[k] = (k == N - 1);
    }
}

__global__ void slice_bt_step_kernel(const int *__restrict__ jump_in, int *__restrict__ jump_out, uint8_t *mark, i64 N)
{
    for (i64 k = (i64)blockIdx.x * blockDim.x + threadIdx.x; k < N; k += (i64)gridDim.x * blockDim.x) {
        const int jk = jump_in[k];
        if (mark[k]) mark[jk] = 1;
        jump_out[k] = jump_in[jk];
    }
}

// marked entry k of the slice = candidate b0 + k of the list
__global__ void slice_bt_scatter_kernel(const uint8_t *__restrict__ mark, i64 N, const int32_t *__restrict__ cand, i64 b0,
                                        uint32_t *keepbits)
{
    for (i64 k = (i64)blockIdx.x * blockDim.x + threadIdx.x; k < N; k += (i64)gridDim.x * blockDim.x) {
        if (mark[k]) {
            const i64 pos = cand ? (i64)__ldg(cand + b0 + k) : b0 + k;
            atomicOr(keepbits + (pos >> 5), 1u << (pos & 31));
        }
    }
}

inline unsigned grid_for(const pasio_ctx *ctx, i64 n, int threads)
{
    i64 g = (n + threads - 1) / threads;
    const i64 cap = (i64)ctx->sm_count * 16;
    if (g > cap) g = cap;
    if (g < 1) g = 1;
    return (unsigned)g;
}

}  // namespace

int launch_batch_contig_stats(pasio_ctx *ctx, u64 *d_out)
{
    CUDA_TRY(ctx, cudaMemsetAsync(d_out, 0, 16, ctx->stream));
    CUDA_TRY(ctx, cudaMemsetAsync(d_out + 2, 0xff, 8, ctx->stream));
    TimingScope ts(ctx, TF_COMPACT);
    batch_contig_stats_kernel<<<grid_for(ctx, ctx->n_contigs, 256), 256, 0, ctx->stream>>>(
        ctx->bounds.as<int32_t>(), ctx->n_contigs, ctx->cg.as<i64>(), ctx->alpha_int, d_out);
    CUDA_TRY(ctx, cudaGetLastError());
    return PASIO_OK;
}

int launch_gather_slice(pasio_ctx *ctx, i64 b0, i64 m)
{
    PASIO_TRY(pasio_reserve(ctx, ctx->dpL, (size_t)m * 4));
    PASIO_TRY(pasio_reserve(ctx, ctx->dpC, (size_t)m * 4));
    gather_slice_kernel<<<grid_for(ctx, m, 256), 256, 0, ctx->stream>>>(cur_cand(ctx), b0, m, ctx->cg.as<i64>(),
                                                                         ctx->dpL.as<int32_t>(), ctx->dpC.as<int32_t>());
    CUDA_TRY(ctx, cudaGetLastError());
    return PASIO_OK;
}

int launch_backtrace_mark_slice(pasio_ctx *ctx, i64 b0, i64 N)
{
    PASIO_TRY(pasio_reserve(ctx, ctx->dpJump, (size_t)N * 8));
    PASIO_TRY(pasio_reserve(ctx, ctx->dpMark, (size_t)N));
    int *ja = ctx->dpJump.as<int>();
    int *jb = ja + N;
    uint8_t *mark = ctx->dpMark.as<uint8_t>();
    const unsigned g = grid_for(ctx, N, 256);
    slice_bt_init_kernel<<<g, 256, 0, ctx->stream>>>(ctx->dpPrev.as<int>(), N, ja, mark);
    for (i64 reach = 1; reach < N; reach <<= 1) {
        slice_bt_step_kernel<<<g, 256, 0, ctx->stream>>>(ja, jb, mark, N);
        int *t = ja; ja = jb; jb = t;
    }
    slice_bt_scatter_kernel<<<g, 256, 0, ctx->stream>>>(mark, N, cur_cand(ctx), b0, ctx->keepbits.as<uint32_t>());
    CUDA_TRY(ctx, cudaGetLastError());
    return PASIO_OK;
}
