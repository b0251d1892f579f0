// C-ABI entry points of libpasio_b200.so (declared in include/pasio_b200.h).
// Host-side orchestration only: buffer management, table bookkeeping, the per-round loop.
// All arithmetic of the hot path happens in the kernels; nothing here computes on the CPU.
#include "common.cuh"

#include <algorithm>
#include <thread>
#include <atomic>
#include <chrono>
#include <memory>
#include <cstdarg>
#include <cstdlib>
#include <cstdio>
#include <cstring>

// ---- small infrastructure ---------------------------------------------------------------------
static thread_local std::string g_create_error;

int pasio_fail(pasio_ctx *ctx, int code, const char *fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (ctx) ctx->err = buf; else g_create_error = buf;
    return code;
}

int pasio_reserve(pasio_ctx *ctx, DevBuf &b, size_t bytes)
{
    if (bytes <= b.bytes && b.p) return PASIO_OK;
    if (b.p) { cudaFree(b.p); b.p = nullptr; b.bytes = 0; }
    size_t want = bytes < 256 ? 256 : bytes;
    cudaError_t e = cudaMalloc(&b.p, want);
    if (e != cudaSuccess) {
        b.p = nullptr;
        return pasio_fail(ctx, PASIO_E_NOMEM, "cudaMalloc(%zu bytes) failed: %s", want, cudaGetErrorString(e));
    }
    b.bytes = want;
    return PASIO_OK;
}

static cudaEvent_t take_event(pasio_ctx *ctx)
{
    if (!ctx->event_pool.empty()) {
        cudaEvent_t e = ctx->event_pool.back();
        ctx->event_pool.pop_back();
        return e;
    }
    cudaEvent_t e;
    cudaEventCreate(&e);
    return e;
}

TimingScope::TimingScope(pasio_ctx *c, int family, i64 launches, cudaStream_t stream) : ctx(c), idx(-1), on(stream ? stream : c->stream)
{
    ctx->fam_launches[family] += launches;
    if (!ctx->timing) return;
    TimedSpan s;
    s.family = family;
    s.a = take_event(ctx);
    s.b = take_event(ctx);
    cudaEventRecord(s.a, on);
    ctx->spans.push_back(s);
    idx = (int)ctx->spans.size() - 1;
}
TimingScope::~TimingScope()
{
    if (idx >= 0) cudaEventRecord(ctx->spans[idx].b, on);
}

static int resolve_spans(pasio_ctx *ctx)
{
    if (ctx->spans.empty()) return PASIO_OK;
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    if (ctx->stream_lx) CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream_lx));
    if (ctx->stream_copy) CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream_copy));
    if (ctx->stream2) CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream2));
    for (auto &s : ctx->spans) {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, s.a, s.b);
        ctx->fam_ms[s.family] += ms;
        ctx->event_pool.push_back(s.a);
        ctx->event_pool.push_back(s.b);
    }
    ctx->spans.clear();
    return PASIO_OK;
}

static int h2d(pasio_ctx *ctx, void *dst, const void *src, size_t bytes)
{
    TimingScope ts(ctx, TF_H2D);
    CUDA_TRY(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
    return PASIO_OK;
}
static int d2h(pasio_ctx *ctx, void *dst, const void *src, size_t bytes)
{
    {
        TimingScope ts(ctx, TF_D2H);
        CUDA_TRY(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    }
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return PASIO_OK;
}


// Host -> device copy of a large buffer that may be PAGEABLE (numpy arrays are): a plain cudaMemcpyAsync from
// pageable memory is staged by the driver on one thread (~10 GB/s).  Here a few host threads copy slices into
// page-locked staging buffers (3 x 32 MB, ring) and each slice is DMA'd as soon as it is staged.  A page-locked
// source (cudaHostAlloc / cudaHostRegister / pasio_host_alloc) goes straight to cudaMemcpyAsync.
static bool host_is_pinned(const void *p)
{
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost || a.type == cudaMemoryTypeManaged;
}

static void parallel_memcpy(char *dst, const char *src, size_t bytes, int threads)
{
    if (threads <= 1 || bytes < ((size_t)4 << 20)) { memcpy(dst, src, bytes); return; }
    std::vector<std::thread> pool;
    const size_t per = ((bytes / threads) + 4095) & ~(size_t)4095;
    for (int t = 1; t < threads; ++t) {
        const size_t lo = (size_t)t * per;
        if (lo >= bytes) break;
        const size_t len = std::min(per, bytes - lo);
        pool.emplace_back([=] { memcpy(dst + lo, src + lo, len); });
    }
    memcpy(dst, src, std::min(per, bytes));
    for (auto &th : pool) th.join();
}

static int upload(pasio_ctx *ctx, void *dst, const void *src, size_t bytes, cudaStream_t stream)
{
    static const int staged_env = getenv("PASIO_B200_STAGED_UPLOAD") ? atoi(getenv("PASIO_B200_STAGED_UPLOAD")) : 1;
    if (bytes < ((size_t)16 << 20) || !staged_env || host_is_pinned(src)) {
        CUDA_TRY(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, stream));
        return PASIO_OK;
    }
    constexpr size_t SLICE = (size_t)32 << 20;
    constexpr int NBUF = 3;
    if (!ctx->stage[0]) {
        for (int k = 0; k < NBUF; ++k) {
            if (cudaHostAlloc(&ctx->stage[k], SLICE, cudaHostAllocDefault) != cudaSuccess ||
                cudaEventCreateWithFlags(&ctx->stage_free[k], cudaEventDisableTiming) != cudaSuccess) {
                cudaGetLastError();
                for (int j = 0; j <= k; ++j) if (ctx->stage[j]) { cudaFreeHost(ctx->stage[j]); ctx->stage[j] = nullptr; }
                CUDA_TRY(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, stream));    // no staging memory: plain copy
                return PASIO_OK;
            }
        }
    }
    unsigned hc = std::thread::hardware_concurrency();
    const int threads = (int)std::max(1u, std::min(8u, hc ? hc / 2 : 4u));
    size_t done = 0;
    while (done < bytes) {
        const int k = ctx->stage_next;
        ctx->stage_next = (k + 1) % NBUF;
        if (ctx->stage_used[k]) CUDA_TRY(ctx, cudaEventSynchronize(ctx->stage_free[k]));     // its last DMA has finished
        const size_t len = std::min(SLICE, bytes - done);
        parallel_memcpy((char *)ctx->stage[k], (const char *)src + done, len, threads);
        CUDA_TRY(ctx, cudaMemcpyAsync((char *)dst + done, ctx->stage[k], len, cudaMemcpyHostToDevice, stream));
        CUDA_TRY(ctx, cudaEventRecord(ctx->stage_free[k], stream));
        ctx->stage_used[k] = true;
        done += len;
    }
    return PASIO_OK;
}

// ---- narrowed upload ------------------------------------------------------------------------------
// Coverage counts are small numbers in 8-byte slots, and a chr1-sized upload is bound by the PCIe link (2 GB at 55 GB/s =
// 36 ms of an 80 ms end-to-end step).  Host threads therefore pack the counts to uint8 (uint16 / int32 for a slice that
// holds a count of 2^8 / 2^16 or more) into page-locked slices (reading the
// caller's buffer -- pinned or pageable -- at memory bandwidth: 87 GB/s with 16 threads on the bench box,
// profiles/r02_host_narrow_probe.txt), each slice is DMA'd as soon as it is packed and widened to the int64 layout the
// kernels use by a small kernel behind the copy on the same stream.  A slice that holds a count outside [0, 2^31) goes up
// as it is (the scan then reports negative counts as before).  Slices are handed out in order; the thread that completes
// a chunk records the chunk's event, and the loading thread waits (host side) for that record before it makes its
// stream wait for the event.
__global__ void __launch_bounds__(256) widen_counts_kernel(const int4 *__restrict__ src, longlong2 *__restrict__ dst, i64 n4)
{
    for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (i64)gridDim.x * blockDim.x) {
        const int4 v = __ldg(src + i);
        dst[2 * i] = make_longlong2(v.x, v.y);
        dst[2 * i + 1] = make_longlong2(v.z, v.w);
    }
}

// dst[i] = (int32) src[i]; returns the OR of all values (bits 31..63 set <=> some count is negative or >= 2^31); textio.cpp
uint64_t pasio_narrow_slice(int32_t *dst, const int64_t *src, size_t n);
uint64_t pasio_narrow_slice16(uint16_t *dst, const int64_t *src, size_t n);     // the same to uint16 (saturating)
uint64_t pasio_narrow_slice8(uint8_t *dst, const int64_t *src, size_t n);       // and to uint8

__global__ void __launch_bounds__(256) widen_counts8_kernel(const uint4 *__restrict__ src, longlong2 *__restrict__ dst, i64 n16)
{
    for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += (i64)gridDim.x * blockDim.x) {
        const uint4 v = __ldg(src + i);                    // 16 counts
        const unsigned w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            dst[8 * i + 2 * k] = make_longlong2(w[k] & 0xffu, (w[k] >> 8) & 0xffu);
            dst[8 * i + 2 * k + 1] = make_longlong2((w[k] >> 16) & 0xffu, w[k] >> 24);
        }
    }
}
#define narrow_slice pasio_narrow_slice

__global__ void __launch_bounds__(256) widen_counts16_kernel(const uint4 *__restrict__ src, longlong2 *__restrict__ dst, i64 n8)
{
    for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (i64)gridDim.x * blockDim.x) {
        const uint4 v = __ldg(src + i);                    // 8 counts
        dst[4 * i] = make_longlong2(v.x & 0xffffu, v.x >> 16);
        dst[4 * i + 1] = make_longlong2(v.y & 0xffffu, v.y >> 16);
        dst[4 * i + 2] = make_longlong2(v.z & 0xffffu, v.z >> 16);
        dst[4 * i + 3] = make_longlong2(v.w & 0xffffu, v.w >> 16);
    }
}

namespace {
struct NarrowUpload {
    static constexpr size_t SLICE = (size_t)1 << 19;       // elements per slice: 4 MB of int64 -> 2 MB of int32
    pasio_ctx *ctx = nullptr;
    const int64_t *src = nullptr;
    i64 n = 0, chunk_elems = 0, n_chunks = 0, n_slices = 0;
    std::vector<std::thread> threads;
    std::atomic<i64> next_slice{0};
    std::atomic<int> cancel{0}, failed{0};
    std::unique_ptr<std::atomic<int>[]> left_in_chunk, recorded;
    std::atomic<i64> wire_bytes{0};
    // A page-locked source can also be DMA'd as it is, at the PCIe rate and without any host thread.  Packing only pays while
    // the host threads read faster than that -- not when eight ranks pack on one host and share its memory bandwidth (8-GPU
    // weak-scaling run: 156 ms per rank packed, 94-127 ms plain).  So the rate of the first 512 MB decides for the rest.
    bool src_pinned = false;
    std::chrono::steady_clock::time_point t_start;
    std::atomic<i64> packed_elems{0};
    std::atomic<int> decided{0}, plain_mode{0};
    static constexpr double PLAIN_RATE = 60e9;             // source bytes per second a plain copy from pinned memory reaches (55 GB/s) + margin
    int limit_bits = 31;                                // test switch (< 25): slices fitting this many bits go as uint8, 3 more as uint16, 6 more as int32

    // every slice lies inside one chunk (chunk_elems is a multiple of SLICE)
    int start(pasio_ctx *c, const int64_t *counts, i64 n_, i64 chunk_elems_, i64 n_chunks_)
    {
        ctx = c; src = counts; n = n_; chunk_elems = chunk_elems_; n_chunks = n_chunks_;
        n_slices = (n + (i64)SLICE - 1) / (i64)SLICE;
        unsigned hc = std::thread::hardware_concurrency();
        const int T = (int)std::max(1u, std::min(16u, hc ? hc : 4u));
        if (ctx->nstage_threads < T) {
            if (ctx->nstage_host) { cudaFreeHost(ctx->nstage_host); ctx->nstage_host = nullptr; }
            if (ctx->nstage_dev) { cudaFree(ctx->nstage_dev); ctx->nstage_dev = nullptr; }
            for (cudaEvent_t e : ctx->nstage_free) cudaEventDestroy(e);
            ctx->nstage_free.clear();
            ctx->nstage_threads = 0;
            if (cudaHostAlloc(&ctx->nstage_host, (size_t)T * 2 * SLICE * 4, cudaHostAllocDefault) != cudaSuccess ||
                cudaMalloc(&ctx->nstage_dev, (size_t)T * 2 * SLICE * 4) != cudaSuccess) {
                cudaGetLastError();
                if (ctx->nstage_host) { cudaFreeHost(ctx->nstage_host); ctx->nstage_host = nullptr; }
                return 1;                                   // no staging memory: the caller copies plainly
            }
            for (int k = 0; k < 2 * T; ++k) {
                cudaEvent_t e;
                if (cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) { cudaGetLastError(); return 1; }
                ctx->nstage_free.push_back(e);
            }
            ctx->nstage_threads = T;
        }
        left_in_chunk.reset(new std::atomic<int>[(size_t)n_chunks]);
        recorded.reset(new std::atomic<int>[(size_t)n_chunks]);
        for (i64 q = 0; q < n_chunks; ++q) {
            const i64 e0 = q * chunk_elems, e1 = std::min<i64>(n, (q + 1) * chunk_elems);
            const i64 cnt = e1 > e0 ? (e1 - e0 + (i64)SLICE - 1) / (i64)SLICE : 0;
            left_in_chunk[(size_t)q].store((int)cnt);
            recorded[(size_t)q].store(0);
            if (cnt == 0) {                                 // (a chunk past the end of the counts: only position n)
                cudaEventRecord(ctx->chunk_events[(size_t)q], ctx->stream_copy);
                recorded[(size_t)q].store(1, std::memory_order_release);
            }
        }
        src_pinned = host_is_pinned(counts);
        t_start = std::chrono::steady_clock::now();
        for (int t = 0; t < T; ++t) threads.emplace_back([this, t] { work(t); });
        return 0;
    }

    void work(int t)
    {
        cudaSetDevice(ctx->device);
        bool used[2] = {false, false};
        int which = 0;
        while (!cancel.load(std::memory_order_relaxed)) {
            const i64 sidx = next_slice.fetch_add(1);
            if (sidx >= n_slices) break;
            const i64 e0 = sidx * (i64)SLICE, e1 = std::min<i64>(n, e0 + (i64)SLICE), len = e1 - e0;
            const int buf = 2 * t + which;
            which ^= 1;
            int32_t *hst = (int32_t *)ctx->nstage_host + (size_t)buf * SLICE;
            int32_t *dev = (int32_t *)ctx->nstage_dev + (size_t)buf * SLICE;
            i64 *dst = ctx->counts.as<i64>() + e0;
            bool ok = true;
            if (plain_mode.load(std::memory_order_relaxed)) {
                ok = cudaMemcpyAsync(dst, src + e0, (size_t)len * 8, cudaMemcpyHostToDevice, ctx->stream_copy) == cudaSuccess;
                wire_bytes.fetch_add(len * 8);
                which ^= 1;                                   // (this slice used no staging buffer)
                if (!ok) { cudaGetLastError(); failed.store(1); cancel.store(1); }
                const i64 qp = e0 / chunk_elems;
                if (left_in_chunk[(size_t)qp].fetch_sub(1) == 1) {
                    if (cudaEventRecord(ctx->chunk_events[(size_t)qp], ctx->stream_copy) != cudaSuccess) { cudaGetLastError(); failed.store(1); }
                    recorded[(size_t)qp].store(1, std::memory_order_release);
                }
                continue;
            }
            if (used[buf & 1]) ok = cudaEventSynchronize(ctx->nstage_free[(size_t)buf]) == cudaSuccess;   // its last copy has left
            // most coverage fits 8 bits: try that first (an eighth of the bytes); the OR of the slice says whether to redo it wider
            const uint64_t bits = ok ? pasio_narrow_slice8(reinterpret_cast<uint8_t *>(hst), src + e0, (size_t)len) : 0;
            const bool sw = limit_bits < 25;                                           // (test switch: a mix of all four kinds)
            const int lim8 = sw ? limit_bits : 8, lim16 = sw ? limit_bits + 3 : 16, lim32 = sw ? limit_bits + 6 : 31;
            if (ok && (bits >> lim8) == 0 && (len & 15) == 0) {
                ok = cudaMemcpyAsync(dev, hst, (size_t)len, cudaMemcpyHostToDevice, ctx->stream_copy) == cudaSuccess;
                if (ok) {
                    ok = cudaEventRecord(ctx->nstage_free[(size_t)buf], ctx->stream_copy) == cudaSuccess;
                    used[buf & 1] = true;
                    const i64 n16 = len / 16;
                    widen_counts8_kernel<<<(unsigned)std::min<i64>((n16 + 255) / 256, 296), 256, 0, ctx->stream_copy>>>(
                        reinterpret_cast<const uint4 *>(dev), reinterpret_cast<longlong2 *>(dst), n16);
                    ok = ok && cudaGetLastError() == cudaSuccess;
                    wire_bytes.fetch_add(len);
                }
            } else if (ok && (bits >> lim16) == 0 && (len & 7) == 0) {
                pasio_narrow_slice16(reinterpret_cast<uint16_t *>(hst), src + e0, (size_t)len);
                ok = cudaMemcpyAsync(dev, hst, (size_t)len * 2, cudaMemcpyHostToDevice, ctx->stream_copy) == cudaSuccess;
                if (ok) {
                    ok = cudaEventRecord(ctx->nstage_free[(size_t)buf], ctx->stream_copy) == cudaSuccess;
                    used[buf & 1] = true;
                    const i64 n8 = len / 8;
                    widen_counts16_kernel<<<(unsigned)std::min<i64>((n8 + 255) / 256, 296), 256, 0, ctx->stream_copy>>>(
                        reinterpret_cast<const uint4 *>(dev), reinterpret_cast<longlong2 *>(dst), n8);
                    ok = ok && cudaGetLastError() == cudaSuccess;
                    wire_bytes.fetch_add(len * 2);
                }
            } else if (ok && (bits >> lim32) == 0 && (len & 3) == 0) {
                narrow_slice(hst, src + e0, (size_t)len);
                ok = cudaMemcpyAsync(dev, hst, (size_t)len * 4, cudaMemcpyHostToDevice, ctx->stream_copy) == cudaSuccess;
                if (ok) {
                    ok = cudaEventRecord(ctx->nstage_free[(size_t)buf], ctx->stream_copy) == cudaSuccess;
                    used[buf & 1] = true;
                    const i64 n4 = len / 4;
                    widen_counts_kernel<<<(unsigned)std::min<i64>((n4 + 255) / 256, 296), 256, 0, ctx->stream_copy>>>(
                        reinterpret_cast<const int4 *>(dev), reinterpret_cast<longlong2 *>(dst), n4);
                    // (the next copy into `dev` is ordered behind this kernel by the stream)
                    ok = ok && cudaGetLastError() == cudaSuccess;
                    wire_bytes.fetch_add(len * 4);
                }
            } else if (ok) {
                // a count outside [0, 2^31), or the ragged last slice: as it is
                ok = cudaMemcpyAsync(dst, src + e0, (size_t)len * 8, cudaMemcpyHostToDevice, ctx->stream_copy) == cudaSuccess;
                wire_bytes.fetch_add(len * 8);
            }
            if (!ok) { cudaGetLastError(); failed.store(1); cancel.store(1); }
            if (src_pinned && packed_elems.fetch_add(len) + len >= ((i64)64 << 20) && !decided.exchange(1)) {
                const double secs = std::chrono::duration<double>(std::chrono::steady_clock::now() - t_start).count();
                if ((double)packed_elems.load() * 8.0 < PLAIN_RATE * secs) plain_mode.store(1);
            }
            const i64 q = e0 / chunk_elems;
            if (left_in_chunk[(size_t)q].fetch_sub(1) == 1) {
                // every slice of chunk q has been queued (by this or another thread, before its decrement)
                if (cudaEventRecord(ctx->chunk_events[(size_t)q], ctx->stream_copy) != cudaSuccess) { cudaGetLastError(); failed.store(1); }
                recorded[(size_t)q].store(1, std::memory_order_release);
            }
        }
    }

    // host-side wait until chunk q's event has been recorded; false if the upload failed or was cancelled
    bool wait_recorded(i64 q)
    {
        while (!recorded[(size_t)q].load(std::memory_order_acquire)) {
            if (failed.load() || cancel.load()) return false;
            std::this_thread::sleep_for(std::chrono::microseconds(20));      // (not a spin: the packing threads want every core)
        }
        return !failed.load();
    }

    void finish()
    {
        for (auto &th : threads) th.join();
        threads.clear();
    }
    ~NarrowUpload()
    {
        if (!threads.empty()) { cancel.store(1); finish(); }
    }
};
}  // namespace

static void drop_borrowed_counts(pasio_ctx *ctx)
{
    if (ctx->counts_borrowed) { ctx->counts.p = nullptr; ctx->counts.bytes = 0; ctx->counts_borrowed = false; }
}

#define NEED_CTX(ctx) do { if (!(ctx)) return PASIO_E_ARG; cudaSetDevice((ctx)->device); } while (0)

// ---- context ------------------------------------------------------------------------------------
extern "C" int pasio_abi_version(void) { return PASIO_ABI_VERSION; }

extern "C" const char *pasio_last_error(const pasio_ctx *ctx)
{
    return ctx ? ctx->err.c_str() : g_create_error.c_str();
}

extern "C" int pasio_ctx_create(int device, pasio_ctx **out)
{
    if (!out) return pasio_fail(nullptr, PASIO_E_ARG, "out is NULL");
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return pasio_fail(nullptr, PASIO_E_CUDA, "no CUDA device: %s (pasio_b200 has no CPU fallback)",
                          e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
    if (device < 0 || device >= count)
        return pasio_fail(nullptr, PASIO_E_ARG, "device %d out of range (have %d)", device, count);
    cudaDeviceProp prop;
    e = cudaGetDeviceProperties(&prop, device);
    if (e != cudaSuccess) return pasio_fail(nullptr, PASIO_E_CUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(e));
    if (prop.major != 10)
        return pasio_fail(nullptr, PASIO_E_CUDA, "device %d is sm_%d%d; this library is built for sm_100a only",
                          device, prop.major, prop.minor);
    e = cudaSetDevice(device);
    if (e != cudaSuccess) return pasio_fail(nullptr, PASIO_E_CUDA, "cudaSetDevice: %s", cudaGetErrorString(e));
    pasio_ctx *ctx = new pasio_ctx();
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;
    ctx->smem_optin = (int)prop.sharedMemPerBlockOptin;
    int prio_lo = 0, prio_hi = 0;
    cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);      // main stream: highest priority, side stream: lowest
    if (cudaStreamCreateWithPriority(&ctx->stream, cudaStreamNonBlocking, prio_hi) != cudaSuccess ||
        cudaStreamCreateWithPriority(&ctx->stream2, cudaStreamNonBlocking, 0) != cudaSuccess ||      // (lowest priority)
        cudaStreamCreateWithFlags(&ctx->stream_copy, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithPriority(&ctx->stream_lx, cudaStreamNonBlocking, 0) != cudaSuccess ||
        cudaEventCreateWithFlags(&ctx->ev_lx0, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&ctx->ev_lx1, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming) != cudaSuccess ||
        cudaMallocHost((void **)&ctx->h_scalars, 20 * sizeof(i64)) != cudaSuccess ||
        pasio_reserve(ctx, ctx->scalars, 20 * sizeof(i64)) != PASIO_OK) {
        g_create_error = "context allocation failed: " + ctx->err;
        delete ctx;
        return PASIO_E_CUDA;
    }
    memset(ctx->h_scalars, 0, 20 * sizeof(i64));
    auto env_int = [](const char *name, int dflt) { const char *v = getenv(name); return v ? atoi(v) : dflt; };
    ctx->tune[PASIO_TUNE_WINDOW_PRUNE] = env_int("PASIO_WD_PRUNE", 1);
    ctx->tune[PASIO_TUNE_WINDOW_PHASES] = env_int("PASIO_WD_PHASES", 1);
    ctx->tune[PASIO_TUNE_EXACT_PRUNE] = env_int("PASIO_XD_PRUNE", 1);
    ctx->tune[PASIO_TUNE_EXACT_LAG] = env_int("PASIO_XD_LAG", 5);
    ctx->tune[PASIO_TUNE_EXACT_RING] = env_int("PASIO_XD_RING", 1);
    ctx->tune[PASIO_TUNE_LOGFAC_EXACT] = env_int("PASIO_B200_EXACT_LMM", 1);
    ctx->tune[PASIO_TUNE_WINDOW_SPECULATE] = env_int("PASIO_WD_SPECULATE", 1);
    ctx->tune[PASIO_TUNE_UPLOAD_NARROW] = env_int("PASIO_B200_UPLOAD_NARROW", 1);
    ctx->tune[PASIO_TUNE_LOGFAC_EAGER] = env_int("PASIO_B200_LOGFAC_EAGER", 0);
    ctx->tune[PASIO_TUNE_EXACT_NBLOCK] = env_int("PASIO_XD_NBLOCK", 3);
    ctx->tune[PASIO_TUNE_WINDOW_CERTIFY] = env_int("PASIO_WD_CERTIFY", 1);
    if (ctx->tune[PASIO_TUNE_EXACT_LAG] < 3 || ctx->tune[PASIO_TUNE_EXACT_LAG] > 5) ctx->tune[PASIO_TUNE_EXACT_LAG] = 5;
    *out = ctx;
    return PASIO_OK;
}

extern "C" int pasio_ctx_destroy(pasio_ctx *ctx)
{
    if (!ctx) return PASIO_OK;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    drop_borrowed_counts(ctx);
    DevBuf *bufs[] = {&ctx->tab[0], &ctx->tab[1], &ctx->tab[2], &ctx->counts, &ctx->cg, &ctx->cpbits, &ctx->keepbits,
                      &ctx->bounds, &ctx->brank, &ctx->cand[0], &ctx->cand[1], &ctx->candC[0], &ctx->candC[1], &ctx->win_st, &ctx->win_en, &ctx->win_small, &ctx->win_medium, &ctx->win_large, &ctx->win_flags,
                      &ctx->blocksum, &ctx->tilestate, &ctx->scalars, &ctx->dpL, &ctx->dpC, &ctx->dpP, &ctx->dpPrev,
                      &ctx->dpPart, &ctx->dpPartArg, &ctx->dpMark, &ctx->dpJump, &ctx->fscan, &ctx->logfac_full,
                      &ctx->xpRing, &ctx->xpRec, &ctx->xpTasks, &ctx->regLR, &ctx->regNR, &ctx->lxPos, &ctx->lxSum, &ctx->lxFirst, &ctx->lxState};
    for (DevBuf *b : bufs) if (b->p) cudaFree(b->p);
    for (auto &s : ctx->spans) { cudaEventDestroy(s.a); cudaEventDestroy(s.b); }
    for (auto e : ctx->event_pool) cudaEventDestroy(e);
    if (ctx->h_scalars) cudaFreeHost(ctx->h_scalars);
    for (int k = 0; k < 3; ++k) {
        if (ctx->stage[k]) cudaFreeHost(ctx->stage[k]);
        if (k == 0) {
            if (ctx->nstage_host) cudaFreeHost(ctx->nstage_host);
            if (ctx->nstage_dev) cudaFree(ctx->nstage_dev);
            for (cudaEvent_t e : ctx->nstage_free) cudaEventDestroy(e);
        }
        if (ctx->stage_free[k]) cudaEventDestroy(ctx->stage_free[k]);
    }
    if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
    if (ctx->ev_join) cudaEventDestroy(ctx->ev_join);
    if (ctx->stream2) cudaStreamDestroy(ctx->stream2);
    if (ctx->stream_copy) cudaStreamDestroy(ctx->stream_copy);
    if (ctx->stream_lx) { cudaStreamSynchronize(ctx->stream_lx); cudaStreamDestroy(ctx->stream_lx); }
    if (ctx->ev_lx0) cudaEventDestroy(ctx->ev_lx0);
    if (ctx->ev_lx1) cudaEventDestroy(ctx->ev_lx1);
    for (auto e : ctx->chunk_events) cudaEventDestroy(e);
    cudaStreamDestroy(ctx->stream);
    delete ctx;
    return PASIO_OK;
}

// ---- parameters and tables ----------------------------------------------------------------------
extern "C" int pasio_set_params(pasio_ctx *ctx, int alpha_is_int, double alpha, double beta, double pen)
{
    NEED_CTX(ctx);
    if (!(alpha >= 0) || !(beta >= 0)) return pasio_fail(ctx, PASIO_E_ARG, "alpha and beta must be >= 0");
    if (alpha_is_int && (alpha != (double)(i64)alpha || alpha > 1e9))
        return pasio_fail(ctx, PASIO_E_ARG, "alpha_is_int set but alpha=%g is not a small integer", alpha);
    ctx->alpha_is_int = alpha_is_int ? 1 : 0;
    ctx->alpha = alpha;
    ctx->alpha_int = alpha_is_int ? (i64)alpha : 0;
    ctx->beta = beta;
    ctx->pen = pen;
    ctx->have_params = true;
    return PASIO_OK;
}

extern "C" int pasio_table_upload(pasio_ctx *ctx, int id, const double *values, int64_t n)
{
    NEED_CTX(ctx);
    if (id < 0 || id > 2 || !values || n < 1) return pasio_fail(ctx, PASIO_E_ARG, "bad table upload (id=%d n=%lld)", id, (long long)n);
    PASIO_TRY(pasio_reserve(ctx, ctx->tab[id], (size_t)n * 8));
    PASIO_TRY(h2d(ctx, ctx->tab[id].p, values, (size_t)n * 8));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->ntab[id] = n;
    return PASIO_OK;
}

extern "C" int pasio_table_need(const pasio_ctx *ctx, int64_t *n_log, int64_t *n_lgamma, int64_t *n_lgamma_alpha)
{
    if (!ctx) return PASIO_E_ARG;
    if (n_log) *n_log = ctx->need[PASIO_TAB_LOG];
    if (n_lgamma) *n_lgamma = ctx->need[PASIO_TAB_LGAMMA];
    if (n_lgamma_alpha) *n_lgamma_alpha = ctx->need[PASIO_TAB_LGAMMA_ALPHA];
    return PASIO_OK;
}

static bool penalties_on(const pasio_ctx *ctx) { return ctx->pen_num || ctx->pen_len; }

// DP tables must cover span (log) and count (+alpha for integer alpha); with_penalties (the rounds): the length penalty
// table is indexed by span exactly like the log table
static int check_dp_tables(pasio_ctx *ctx, i64 max_span, i64 max_cnt, bool with_penalties = false)
{
    if (!ctx->have_params) return pasio_fail(ctx, PASIO_E_STATE, "pasio_set_params has not been called");
    if (max_cnt + ctx->alpha_int >= 2147483647LL)
        return pasio_fail(ctx, PASIO_E_TOO_LARGE, "count %lld does not fit the 32-bit DP index", (long long)max_cnt);
    const i64 need_log = max_span + 1;
    const int gid = ctx->alpha_is_int ? PASIO_TAB_LGAMMA : PASIO_TAB_LGAMMA_ALPHA;
    const i64 need_g = max_cnt + ctx->alpha_int + 1;
    bool bad = false;
    if (ctx->ntab[PASIO_TAB_LOG] < need_log) { ctx->need[PASIO_TAB_LOG] = need_log; bad = true; }
    if (ctx->ntab[gid] < need_g) { ctx->need[gid] = need_g; bad = true; }
    if (with_penalties && ctx->pen_len && ctx->n_pen_lr < need_log) { ctx->need[PASIO_TAB_LOG] = need_log; bad = true; }
    if (bad)
        return pasio_fail(ctx, PASIO_E_TABLE_TOO_SHORT, "tables too short: need log>=%lld, lgamma[%d]>=%lld (have %lld, %lld%s)",
                          (long long)need_log, gid, (long long)need_g, (long long)ctx->ntab[PASIO_TAB_LOG],
                          (long long)ctx->ntab[gid], with_penalties && ctx->pen_len ? ", length penalty as long as log" : "");
    return PASIO_OK;
}

extern "C" int pasio_set_penalties(pasio_ctx *ctx, const double *split_number_penalty, int64_t n_split_number_penalty,
                                   double first_column_refund, const double *length_penalty, int64_t n_length_penalty)
{
    NEED_CTX(ctx);
    if ((split_number_penalty && n_split_number_penalty < 1) || (length_penalty && n_length_penalty < 1))
        return pasio_fail(ctx, PASIO_E_ARG, "a penalty table needs at least one entry");
    ctx->pen_num = ctx->pen_len = false;
    if (split_number_penalty) {
        PASIO_TRY(pasio_reserve(ctx, ctx->penNR, (size_t)n_split_number_penalty * 8));
        PASIO_TRY(h2d(ctx, ctx->penNR.p, split_number_penalty, (size_t)n_split_number_penalty * 8));
    }
    if (length_penalty) {
        PASIO_TRY(pasio_reserve(ctx, ctx->penLR, (size_t)n_length_penalty * 8));
        PASIO_TRY(h2d(ctx, ctx->penLR.p, length_penalty, (size_t)n_length_penalty * 8));
    }
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));      // the caller's tables were read by the copies above
    ctx->pen_num = split_number_penalty != nullptr;
    ctx->n_pen_nr = ctx->pen_num ? n_split_number_penalty : 0;
    ctx->pen_refund = ctx->pen_num ? first_column_refund : 0.0;
    ctx->pen_len = length_penalty != nullptr;
    ctx->n_pen_lr = ctx->pen_len ? n_length_penalty : 0;
    return PASIO_OK;
}

// ---- contig -------------------------------------------------------------------------------------
static int finish_load(pasio_ctx *ctx, const int64_t *offsets, int64_t n_contigs)
{
    const i64 n = ctx->n;
    ctx->h_bounds.resize((size_t)n_contigs + 1);
    if (offsets) {
        for (i64 c = 0; c <= n_contigs; ++c) {
            if (offsets[c] < 0 || offsets[c] > n || (c > 0 && offsets[c] <= offsets[c - 1]))
                return pasio_fail(ctx, PASIO_E_ARG, "contig offsets must be strictly ascending within [0, n] (empty contigs are not allowed)");
            ctx->h_bounds[(size_t)c] = (int32_t)offsets[c];
        }
        if (offsets[0] != 0 || offsets[n_contigs] != n)
            return pasio_fail(ctx, PASIO_E_ARG, "offsets[0] must be 0 and offsets[n_contigs] must be n");
    } else {
        ctx->h_bounds[0] = 0;
        ctx->h_bounds[1] = (int32_t)n;
    }
    ctx->n_contigs = n_contigs;
    // bitmaps over positions 0..n, padded to whole scan tiles (4096 positions) so the scan writes 64-bit words freely
    const size_t bit_bytes = (size_t)((n + 1 + 4095) / 4096) * 512 + 16;
    PASIO_TRY(pasio_reserve(ctx, ctx->cg, (size_t)(n + 2) * 8));
    PASIO_TRY(pasio_reserve(ctx, ctx->cpbits, bit_bytes));
    PASIO_TRY(pasio_reserve(ctx, ctx->keepbits, bit_bytes));
    PASIO_TRY(pasio_reserve(ctx, ctx->bounds, (size_t)(n_contigs + 1) * 4));
    PASIO_TRY(pasio_reserve(ctx, ctx->brank, (size_t)(n_contigs + 1) * 4));
    PASIO_TRY(h2d(ctx, ctx->bounds.p, ctx->h_bounds.data(), (size_t)(n_contigs + 1) * 4));
    PASIO_TRY(launch_scan_counts(ctx));
    PASIO_TRY(d2h(ctx, ctx->h_scalars, ctx->scalars.p, 3 * sizeof(i64)));
    if (ctx->h_scalars[1]) return pasio_fail(ctx, PASIO_E_COUNTS, "counts must be >= 0");
    ctx->total = ctx->h_scalars[0];
    ctx->max_count = ctx->h_scalars[2];
    ctx->have_contig = true;
    ctx->implicit_all = true;
    ctx->prev_round_in = 0;
    ctx->m = n + 1;
    ctx->cur = 0;
    PASIO_TRY(launch_boundary_ranks(ctx));
    ctx->h_brank = ctx->h_bounds;
    return PASIO_OK;
}

static int check_load_args(pasio_ctx *ctx, int64_t n, const int64_t *offsets, int64_t n_contigs)
{
    if (ctx->logfac_pending) {                 // a prefetch nobody consumed still reads the buffers that are about to change
        cudaStreamSynchronize(ctx->stream_lx);
        ctx->logfac_pending = false;
    }
    ctx->logfac_ready = false;
    ctx->logfac_eager = false;
    ctx->have_contig = false;
    if (n < 1) return pasio_fail(ctx, PASIO_E_COUNTS, "contig is empty");            // len(counts) > 0
    if (n > 2147483645LL) return pasio_fail(ctx, PASIO_E_TOO_LARGE, "contig of %lld nt exceeds 2^31-3", (long long)n);
    if (n_contigs < 1 || (n_contigs > 1 && !offsets)) return pasio_fail(ctx, PASIO_E_ARG, "bad n_contigs/offsets");
    return PASIO_OK;
}

extern "C" int pasio_contig_load(pasio_ctx *ctx, const int64_t *counts, int64_t n, const int64_t *offsets,
                                 int64_t n_contigs)
{
    NEED_CTX(ctx);
    if (!counts) return pasio_fail(ctx, PASIO_E_ARG, "counts is NULL");
    PASIO_TRY(check_load_args(ctx, n, offsets, n_contigs));
    ctx->n = n;
    drop_borrowed_counts(ctx);
    PASIO_TRY(pasio_reserve(ctx, ctx->counts, (size_t)n * 8 + 16));
    bool sent = false;
    if (ctx->tune[PASIO_TUNE_UPLOAD_NARROW] && n >= ((i64)1 << 24)) {
        // a large batch: packed to int32 by the host threads on the way (NarrowUpload), as one chunk
        if (ctx->chunk_events.empty()) {
            cudaEvent_t e;
            CUDA_TRY(ctx, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
            ctx->chunk_events.push_back(e);
        }
        CUDA_TRY(ctx, cudaEventRecord(ctx->ev_fork, ctx->stream));      // the buffers may still be in use by earlier work
        CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->stream_copy, ctx->ev_fork, 0));
        NarrowUpload narrow;
        std::unique_ptr<TimingScope> span(new TimingScope(ctx, TF_H2D, 1, ctx->stream_copy));
        if (ctx->tune[PASIO_TUNE_UPLOAD_NARROW] >= 2 && ctx->tune[PASIO_TUNE_UPLOAD_NARROW] < 31) narrow.limit_bits = ctx->tune[PASIO_TUNE_UPLOAD_NARROW];
        const i64 one_chunk = (n + (i64)NarrowUpload::SLICE - 1) / (i64)NarrowUpload::SLICE * (i64)NarrowUpload::SLICE;
        if (narrow.start(ctx, counts, n, one_chunk, 1) == 0) {
            const bool ok = narrow.wait_recorded(0);
            narrow.finish();
            span.reset();
            ctx->last_wire_bytes = narrow.wire_bytes.load();
            if (!ok || narrow.failed.load()) {
                cudaStreamSynchronize(ctx->stream_copy);
                return pasio_fail(ctx, PASIO_E_CUDA, "narrowed upload failed: %s", cudaGetErrorString(cudaGetLastError()));
            }
            CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->stream, ctx->chunk_events[0], 0));
            sent = true;
        } else {
            span.reset();
        }
    }
    if (!sent) {
        TimingScope ts(ctx, TF_H2D);
        PASIO_TRY(upload(ctx, ctx->counts.p, counts, (size_t)n * 8, ctx->stream));
        ctx->last_wire_bytes = n * 8;
    }
    return finish_load(ctx, offsets, n_contigs);
}

extern "C" int pasio_contig_load_device(pasio_ctx *ctx, const int64_t *d_counts, int64_t n, const int64_t *offsets,
                                        int64_t n_contigs)
{
    NEED_CTX(ctx);
    if (!d_counts) return pasio_fail(ctx, PASIO_E_ARG, "d_counts is NULL");
    if (reinterpret_cast<uintptr_t>(d_counts) & 15) return pasio_fail(ctx, PASIO_E_ARG, "d_counts must be 16-byte aligned");
    PASIO_TRY(check_load_args(ctx, n, offsets, n_contigs));
    ctx->n = n;
    if (ctx->counts.p && !ctx->counts_borrowed) cudaFree(ctx->counts.p);
    ctx->counts.p = const_cast<int64_t *>(d_counts);
    ctx->counts.bytes = (size_t)n * 8;
    ctx->counts_borrowed = true;
    return finish_load(ctx, offsets, n_contigs);
}

extern "C" int pasio_contig_load_rle(pasio_ctx *ctx, const int64_t *starts, const int64_t *values, int64_t n_runs,
                                     const int64_t *offsets, int64_t n_contigs)
{
    NEED_CTX(ctx);
    if (!starts || !values || n_runs < 1) return pasio_fail(ctx, PASIO_E_ARG, "bad run-length input");
    if (starts[0] != 0) return pasio_fail(ctx, PASIO_E_ARG, "starts[0] must be 0");
    const i64 n = starts[n_runs];
    PASIO_TRY(check_load_args(ctx, n, offsets, n_contigs));
    ctx->n = n;
    drop_borrowed_counts(ctx);
    PASIO_TRY(pasio_reserve(ctx, ctx->counts, (size_t)n * 8 + 16));
    // stage the runs in scratch buffers (dpP / dpJump are free while a contig is being loaded)
    PASIO_TRY(pasio_reserve(ctx, ctx->dpP, (size_t)(n_runs + 1) * 8));
    PASIO_TRY(pasio_reserve(ctx, ctx->dpJump, (size_t)n_runs * 8));
    PASIO_TRY(h2d(ctx, ctx->dpP.p, starts, (size_t)(n_runs + 1) * 8));
    PASIO_TRY(h2d(ctx, ctx->dpJump.p, values, (size_t)n_runs * 8));
    PASIO_TRY(launch_expand_rle(ctx, ctx->dpP.as<i64>(), ctx->dpJump.as<i64>(), n_runs));
    return finish_load(ctx, offsets, n_contigs);
}


static int refresh_boundary_ranks(pasio_ctx *ctx);

// Load one contig from host memory AND run the first sliding-window round (all positions are candidates) while the
// upload is still in flight: the counts go up in chunks on a copy stream; as soon as a chunk has arrived its tiles
// are scanned and the windows that lie completely inside the scanned prefix are processed.
extern "C" int pasio_contig_load_round(pasio_ctx *ctx, const int64_t *counts, int64_t n, int64_t window_size,
                                       int64_t window_shift, int constraint, int64_t *n_in, int64_t *n_out, int64_t *cells)
{
    NEED_CTX(ctx);
    if (!counts) return pasio_fail(ctx, PASIO_E_ARG, "counts is NULL");
    if (window_size < 1 || window_shift < 1 || window_size > 2147483000LL || window_shift > 2147483000LL)
        return pasio_fail(ctx, PASIO_E_ARG, "window_size and window_shift must be positive");
    if (constraint < 0 || constraint > 2) return pasio_fail(ctx, PASIO_E_ARG, "unknown constraint %d", constraint);
    PASIO_TRY(check_load_args(ctx, n, nullptr, 1));
    ctx->n = n;
    drop_borrowed_counts(ctx);
    PASIO_TRY(pasio_reserve(ctx, ctx->counts, (size_t)n * 8 + 16));
    ctx->h_bounds.assign({0, (int32_t)n});
    ctx->n_contigs = 1;
    const size_t bit_alloc = (size_t)((n + 1 + 4095) / 4096) * 512 + 16;
    PASIO_TRY(pasio_reserve(ctx, ctx->cg, (size_t)(n + 2) * 8));
    PASIO_TRY(pasio_reserve(ctx, ctx->cpbits, bit_alloc));
    PASIO_TRY(pasio_reserve(ctx, ctx->keepbits, bit_alloc));
    PASIO_TRY(pasio_reserve(ctx, ctx->bounds, 2 * 4));
    PASIO_TRY(pasio_reserve(ctx, ctx->brank, 2 * 4));
    PASIO_TRY(h2d(ctx, ctx->bounds.p, ctx->h_bounds.data(), 2 * 4));
    const size_t bit_bytes = (size_t)((n + 1 + 31) / 32 + 2) * 4;
    CUDA_TRY(ctx, cudaMemsetAsync(ctx->keepbits.p, 0, bit_bytes, ctx->stream));
    i64 n_tiles = 0, tile_elems = 0;
    PASIO_TRY(launch_scan_prepare(ctx, &n_tiles, &tile_elems));
    ctx->implicit_all = true;
    ctx->prev_round_in = 0;
    ctx->m = n + 1;
    ctx->cur = 0;
    ctx->n_small = ctx->n_medium = ctx->n_large = -1;

    // chunk copies are queued two ahead of the chunk being processed: a pinned source keeps the link busy back to
    // back, a pageable source (whose staging blocks the host) is staged while the GPU works on the chunks before it
    const i64 chunk_tiles = (i64)(32 << 20) / tile_elems;              // 32 Mi positions = 256 MB per chunk
    const i64 n_chunks = (n_tiles + chunk_tiles - 1) / chunk_tiles;
    while ((i64)ctx->chunk_events.size() < n_chunks) {
        cudaEvent_t e;
        CUDA_TRY(ctx, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        ctx->chunk_events.push_back(e);
    }
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev_fork, ctx->stream));          // buffers may still be in use by earlier work
    CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->stream_copy, ctx->ev_fork, 0));
    i64 queued = 0;
    auto queue_copies = [&](i64 upto) -> int {
        for (; queued < upto && queued < n_chunks; ++queued) {
            const i64 e0 = queued * chunk_tiles * tile_elems, e1 = std::min<i64>(n, (queued + 1) * chunk_tiles * tile_elems);
            if (e1 > e0) {
                TimingScope ts(ctx, TF_H2D, 1, ctx->stream_copy);
                PASIO_TRY(upload(ctx, ctx->counts.as<i64>() + e0, counts + e0, (size_t)(e1 - e0) * 8, ctx->stream_copy));
            }
            CUDA_TRY(ctx, cudaEventRecord(ctx->chunk_events[(size_t)queued], ctx->stream_copy));
        }
        return PASIO_OK;
    };

    // the sequential log-factorial sums follow the chunks on the side stream when the caller announced that it wants them
    // (PASIO_TUNE_LOGFAC_EAGER; the lgamma table in place decides whether the terms can be looked up at all)
    const bool eager = ctx->tune[PASIO_TUNE_LOGFAC_EXACT] && ctx->tune[PASIO_TUNE_LOGFAC_EAGER] && ctx->ntab[PASIO_TAB_LGAMMA] > 2;
    if (eager) {
        CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->stream_lx, ctx->ev_fork, 0));
        PASIO_TRY(launch_logfac_exact_begin(ctx, ctx->stream_lx));
    }
    // large loads go up narrowed to int32 by a team of host threads (NarrowUpload above) while this thread drives the GPU
    NarrowUpload narrow;
    std::unique_ptr<TimingScope> narrow_span;
    bool narrow_on = false;
    if (ctx->tune[PASIO_TUNE_UPLOAD_NARROW] && n >= ((i64)1 << 24) && (chunk_tiles * tile_elems) % (i64)NarrowUpload::SLICE == 0) {
        narrow_span.reset(new TimingScope(ctx, TF_H2D, 1, ctx->stream_copy));
        if (ctx->tune[PASIO_TUNE_UPLOAD_NARROW] >= 2 && ctx->tune[PASIO_TUNE_UPLOAD_NARROW] < 31) narrow.limit_bits = ctx->tune[PASIO_TUNE_UPLOAD_NARROW];   // (tests: mixes narrowed and plain slices)
        narrow_on = narrow.start(ctx, counts, n, chunk_tiles * tile_elems, n_chunks) == 0;
        if (!narrow_on) narrow_span.reset();
    }
    auto stop_upload = [&]() {                      // before any return: nothing may read the caller's buffer afterwards
        if (narrow_on) { narrow.cancel.store(1); narrow.finish(); narrow_span.reset(); }
        if (eager) cudaStreamSynchronize(ctx->stream_lx);
    };

    const i64 nwin_total = (ctx->m - 1 + window_shift - 1) / window_shift;
    i64 w_done = 0;
    int table_rc = ctx->have_params ? PASIO_OK : pasio_fail(ctx, PASIO_E_STATE, "pasio_set_params has not been called");
    bool first_dp = true;
    for (i64 c = 0; c < n_chunks; ++c) {
        if (narrow_on) {
            if (!narrow.wait_recorded(c)) {
                stop_upload();
                cudaStreamSynchronize(ctx->stream_copy);
                return pasio_fail(ctx, PASIO_E_CUDA, "narrowed upload failed: %s", cudaGetErrorString(cudaGetLastError()));
            }
        } else {
            PASIO_TRY(queue_copies(c + 3));
        }
        CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->stream, ctx->chunk_events[(size_t)c], 0));
        if (eager) {
            CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->stream_lx, ctx->chunk_events[(size_t)c], 0));
            PASIO_TRY(launch_logfac_exact_chunk(ctx, c * chunk_tiles * tile_elems, std::min<i64>(n, (c + 1) * chunk_tiles * tile_elems),
                                                ctx->stream_lx));
        }
        const i64 t1 = std::min<i64>(n_tiles, (c + 1) * chunk_tiles);
        PASIO_TRY(launch_scan_tiles(ctx, t1 - c * chunk_tiles));
        // positions < scanned are final (prefix sums and change-point bits); the last chunk covers position n as well
        const i64 scanned = t1 * tile_elems;
        i64 w_ready = nwin_total;
        if (c + 1 < n_chunks) {
            w_ready = scanned > window_size ? (scanned - window_size - 1) / window_shift + 1 : 0;
            if (w_ready > nwin_total) w_ready = nwin_total;
        }
        if (table_rc == PASIO_OK && w_ready > w_done) {
            i64 max_span = 0, max_cnt = 0;
            // the scan's "negative count seen" flag comes back with the prepass results: a negative count makes the
            // prefix sums non-monotone and the DP's table indices meaningless, so no window is processed after it
            // (the reference asserts counts >= 0 before anything else, log_marginal_likelyhood.py:33)
            CUDA_TRY(ctx, cudaMemcpyAsync(ctx->h_scalars + 1, ctx->scalars.as<i64>() + 1, 8, cudaMemcpyDeviceToHost, ctx->stream));
            PASIO_TRY(launch_window_prepass(ctx, w_ready - w_done, (int)window_size, (int)window_shift, &max_span, &max_cnt,
                                            constraint, w_done));
            if (ctx->h_scalars[1]) {
                stop_upload();
                cudaStreamSynchronize(ctx->stream_copy);      // the caller's buffer must not be read after we return
                return pasio_fail(ctx, PASIO_E_COUNTS, "counts must be >= 0");
            }
            table_rc = check_dp_tables(ctx, max_span, max_cnt, true);
            if (table_rc == PASIO_OK) {
                if (penalties_on(ctx))
                    PASIO_TRY(launch_window_dp_reg(ctx, w_ready - w_done, (int)window_size, (int)window_shift, constraint, !first_dp));
                else
                    PASIO_TRY(launch_window_dp(ctx, w_ready - w_done, (int)window_size, (int)window_shift, constraint, w_done,
                                               !first_dp));
                first_dp = false;
            } else if (table_rc != PASIO_E_TABLE_TOO_SHORT) {
                return table_rc;
            }
            w_done = w_ready;
        }
    }
    if (narrow_on) {
        narrow.finish();
        narrow_span.reset();
        ctx->last_wire_bytes = narrow.wire_bytes.load();
        if (narrow.failed.load()) {
            cudaStreamSynchronize(ctx->stream_copy);
            return pasio_fail(ctx, PASIO_E_CUDA, "narrowed upload failed: %s", cudaGetErrorString(cudaGetLastError()));
        }
    } else {
        ctx->last_wire_bytes = n * 8;
    }
    PASIO_TRY(d2h(ctx, ctx->h_scalars, ctx->scalars.p, 3 * sizeof(i64)));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream_copy));
    if (ctx->h_scalars[1]) return pasio_fail(ctx, PASIO_E_COUNTS, "counts must be >= 0");
    ctx->total = ctx->h_scalars[0];
    ctx->max_count = ctx->h_scalars[2];
    ctx->have_contig = true;
    if (eager) {                                       // the sums are (nearly) done on the side stream; verdict at first use
        CUDA_TRY(ctx, cudaEventRecord(ctx->ev_lx1, ctx->stream_lx));
        ctx->logfac_ready = true;
        ctx->logfac_is_exact = true;
        ctx->logfac_pending = true;
        ctx->logfac_eager = true;
    }
    PASIO_TRY(launch_boundary_ranks(ctx));
    ctx->h_brank = ctx->h_bounds;
    if (n_in) *n_in = ctx->m;
    if (n_out) *n_out = ctx->m;
    if (cells) *cells = 0;
    if (table_rc != PASIO_OK) return table_rc;        // the contig is loaded: grow the tables, then pasio_round

    const int nxt = 1 - ctx->cur;
    PASIO_TRY(pasio_reserve(ctx, ctx->cand[nxt], (size_t)ctx->m * 4));
    i64 m_new = 0;
    PASIO_TRY(launch_compact_keepbits(ctx, nxt, &m_new));
    PASIO_TRY(d2h(ctx, ctx->h_scalars + 10, ctx->scalars.as<i64>() + 10, 24));
    PASIO_TRY(d2h(ctx, ctx->h_scalars + 16, ctx->scalars.as<i64>() + 16, 24));
    if (cells) *cells = ctx->h_scalars[10];
    ctx->last_cells = ctx->h_scalars[10];
    ctx->last_cells_skipped = ctx->h_scalars[12];
    for (int k = 0; k < 3; ++k) ctx->last_certify[k] = ctx->h_scalars[16 + k];
    ctx->prev_round_in = ctx->m;
    ctx->prev_round_out = m_new;
    ctx->cur = nxt;
    ctx->implicit_all = false;
    ctx->m = m_new;
    if (n_out) *n_out = m_new;
    return refresh_boundary_ranks(ctx);
}

extern "C" int pasio_contig_info(const pasio_ctx *ctx, int64_t *n, int64_t *total_count, int64_t *n_contigs)
{
    if (!ctx || !ctx->have_contig) return PASIO_E_STATE;
    if (n) *n = ctx->n;
    if (total_count) *total_count = ctx->total;
    if (n_contigs) *n_contigs = ctx->n_contigs;
    return PASIO_OK;
}

extern "C" int pasio_cumsum_at(pasio_ctx *ctx, const int64_t *positions, int64_t m, int64_t *out)
{
    NEED_CTX(ctx);
    if (!ctx->have_contig) return pasio_fail(ctx, PASIO_E_STATE, "no contig loaded");
    if (m < 0 || !out) return pasio_fail(ctx, PASIO_E_ARG, "bad arguments");
    if (m == 0) return PASIO_OK;
    PASIO_TRY(pasio_reserve(ctx, ctx->dpP, (size_t)m * 8));
    if (positions) {
        for (i64 k = 0; k < m; ++k)
            if (positions[k] < 0 || positions[k] > ctx->n) return pasio_fail(ctx, PASIO_E_ARG, "position out of range");
        PASIO_TRY(pasio_reserve(ctx, ctx->dpJump, (size_t)m * 8));
        PASIO_TRY(h2d(ctx, ctx->dpJump.p, positions, (size_t)m * 8));
        PASIO_TRY(launch_gather_i64(ctx, ctx->cg.as<i64>(), nullptr, ctx->dpJump.as<i64>(), m, ctx->dpP.as<i64>()));
    } else {   // at the current candidates
        if (m != ctx->m) return pasio_fail(ctx, PASIO_E_ARG, "m must equal the candidate count");
        PASIO_TRY(launch_gather_i64(ctx, ctx->cg.as<i64>(), cur_cand(ctx), nullptr, m, ctx->dpP.as<i64>()));
    }
    return d2h(ctx, out, ctx->dpP.p, (size_t)m * 8);
}

// ---- candidates ---------------------------------------------------------------------------------
__global__ void narrow_candidates_kernel(const i64 *__restrict__ in, i64 m, i64 n, int32_t *__restrict__ out, i64 *bad)
{
    for (i64 k = (i64)blockIdx.x * blockDim.x + threadIdx.x; k < m; k += (i64)gridDim.x * blockDim.x) {
        i64 v = in[k];
        if (v < 0 || v > n) { *bad = 1; v = 0; }
        out[k] = (int32_t)v;
    }
}

static int refresh_boundary_ranks(pasio_ctx *ctx)
{
    PASIO_TRY(launch_boundary_ranks(ctx));
    if (ctx->n_contigs > 1) {
        ctx->h_brank.resize((size_t)ctx->n_contigs + 1);
        PASIO_TRY(d2h(ctx, ctx->h_brank.data(), ctx->brank.p, (size_t)(ctx->n_contigs + 1) * 4));
    }
    return PASIO_OK;
}

extern "C" int pasio_candidates_set(pasio_ctx *ctx, const int64_t *cands, int64_t m)
{
    NEED_CTX(ctx);
    if (!ctx->have_contig) return pasio_fail(ctx, PASIO_E_STATE, "no contig loaded");
    ctx->prev_round_in = 0;
    if (!cands) {
        ctx->implicit_all = true;
    ctx->prev_round_in = 0;
        ctx->m = ctx->n + 1;
        return refresh_boundary_ranks(ctx);
    }
    if (m < 2 || m > ctx->n + 1) return pasio_fail(ctx, PASIO_E_CANDIDATES, "need 2 <= len(candidates) <= n+1");
    PASIO_TRY(pasio_reserve(ctx, ctx->dpJump, (size_t)m * 8));
    PASIO_TRY(pasio_reserve(ctx, ctx->cand[ctx->cur], (size_t)m * 4));
    PASIO_TRY(h2d(ctx, ctx->dpJump.p, cands, (size_t)m * 8));
    i64 *d_bad = ctx->scalars.as<i64>() + 5;
    CUDA_TRY(ctx, cudaMemsetAsync(d_bad, 0, 8, ctx->stream));
    narrow_candidates_kernel<<<ctx->sm_count * 4, 256, 0, ctx->stream>>>(ctx->dpJump.as<i64>(), m, ctx->n,
                                                                        ctx->cand[ctx->cur].as<int32_t>(), d_bad);
    CUDA_TRY(ctx, cudaGetLastError());
    PASIO_TRY(d2h(ctx, ctx->h_scalars + 5, d_bad, 8));
    if (ctx->h_scalars[5]) { ctx->implicit_all = true; ctx->m = ctx->n + 1; return pasio_fail(ctx, PASIO_E_CANDIDATES, "candidate out of range"); }
    ctx->implicit_all = false;
    ctx->m = m;
    PASIO_TRY(pasio_reserve(ctx, ctx->candC[ctx->cur], (size_t)m * 8));
    PASIO_TRY(launch_gather_i64(ctx, ctx->cg.as<i64>(), ctx->cand[ctx->cur].as<int32_t>(), nullptr, m, ctx->candC[ctx->cur].as<i64>()));
    PASIO_TRY(refresh_boundary_ranks(ctx));
    i64 bad = 0;
    PASIO_TRY(launch_validate_candidates(ctx, &bad));
    if (bad) {
        ctx->implicit_all = true;
    ctx->prev_round_in = 0;
        ctx->m = ctx->n + 1;
        refresh_boundary_ranks(ctx);
        return pasio_fail(ctx, PASIO_E_CANDIDATES,
                          "candidates must start at 0, end at len(counts), ascend strictly and contain every contig boundary");
    }
    return PASIO_OK;
}

extern "C" int pasio_candidates_count(const pasio_ctx *ctx, int64_t *m)
{
    if (!ctx || !ctx->have_contig || !m) return PASIO_E_STATE;
    *m = ctx->m;
    return PASIO_OK;
}

__global__ void widen_candidates_kernel(const int32_t *__restrict__ in, i64 m, i64 *__restrict__ out)
{
    for (i64 k = (i64)blockIdx.x * blockDim.x + threadIdx.x; k < m; k += (i64)gridDim.x * blockDim.x)
        out[k] = in ? (i64)in[k] : k;
}

extern "C" int pasio_candidates_download(pasio_ctx *ctx, int64_t *out, int64_t capacity, int64_t *m)
{
    NEED_CTX(ctx);
    if (!ctx->have_contig) return pasio_fail(ctx, PASIO_E_STATE, "no contig loaded");
    if (m) *m = ctx->m;
    if (!out) return PASIO_OK;
    if (capacity < ctx->m) return pasio_fail(ctx, PASIO_E_ARG, "capacity %lld < %lld candidates", (long long)capacity, (long long)ctx->m);
    PASIO_TRY(pasio_reserve(ctx, ctx->dpJump, (size_t)ctx->m * 8));
    widen_candidates_kernel<<<ctx->sm_count * 4, 256, 0, ctx->stream>>>(cur_cand(ctx), ctx->m, ctx->dpJump.as<i64>());
    CUDA_TRY(ctx, cudaGetLastError());
    return d2h(ctx, out, ctx->dpJump.p, (size_t)ctx->m * 8);
}

extern "C" int pasio_filter_candidates(pasio_ctx *ctx, int constraint, int64_t *n_in, int64_t *n_out)
{
    NEED_CTX(ctx);
    if (!ctx->have_contig) return pasio_fail(ctx, PASIO_E_STATE, "no contig loaded");
    if (ctx->n_contigs != 1) return pasio_fail(ctx, PASIO_E_STATE, "pasio_filter_candidates works on a single-contig context");
    if (constraint < 0 || constraint > 2) return pasio_fail(ctx, PASIO_E_ARG, "unknown constraint %d", constraint);
    if (n_in) *n_in = ctx->m;
    PASIO_TRY(launch_filter_candidates(ctx, constraint));
    ctx->prev_round_in = 0;
    const int nxt = 1 - ctx->cur;
    PASIO_TRY(pasio_reserve(ctx, ctx->cand[nxt], (size_t)ctx->m * 4));
    i64 m_new = 0;
    PASIO_TRY(launch_compact_keepbits(ctx, nxt, &m_new));
    ctx->cur = nxt;
    ctx->implicit_all = false;
    ctx->m = m_new;
    if (n_out) *n_out = m_new;
    return refresh_boundary_ranks(ctx);
}

// ---- rounds -------------------------------------------------------------------------------------
// Window table of a batch: windows are generated per contig over that contig's slice of the
// candidate list (dto/sliding_window.py:9-15 applied per contig).
static int build_window_table(pasio_ctx *ctx, i64 wsize, i64 wshift, i64 *nwin_out)
{
    if (ctx->n_contigs == 1) {
        *nwin_out = (ctx->m - 1 + wshift - 1) / wshift;        // len(range(0, m-1, shift))
        return PASIO_OK;
    }
    ctx->h_win_st.clear();
    ctx->h_win_en.clear();
    for (i64 c = 0; c < ctx->n_contigs; ++c) {
        const i64 b0 = ctx->h_brank[(size_t)c], b1 = ctx->h_brank[(size_t)c + 1];
        const i64 mc = b1 - b0 + 1;
        for (i64 st = 0; st < mc - 1; st += wshift) {
            i64 en = st + wsize + 1;
            if (en > mc) en = mc;
            ctx->h_win_st.push_back((int32_t)(b0 + st));
            ctx->h_win_en.push_back((int32_t)(b0 + en));
        }
    }
    const size_t nw = ctx->h_win_st.size();
    PASIO_TRY(pasio_reserve(ctx, ctx->win_st, nw * 4));
    PASIO_TRY(pasio_reserve(ctx, ctx->win_en, nw * 4));
    PASIO_TRY(h2d(ctx, ctx->win_st.p, ctx->h_win_st.data(), nw * 4));
    PASIO_TRY(h2d(ctx, ctx->win_en.p, ctx->h_win_en.data(), nw * 4));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));   // host vectors are reused next round
    *nwin_out = (i64)nw;
    return PASIO_OK;
}

extern "C" int pasio_round(pasio_ctx *ctx, int64_t window_size, int64_t window_shift, int constraint,
                           int64_t *n_in, int64_t *n_out, int64_t *cells)
{
    NEED_CTX(ctx);
    if (!ctx->have_contig) return pasio_fail(ctx, PASIO_E_STATE, "no contig loaded");
    if (window_size < 1 || window_shift < 1 || window_size > 2147483000LL || window_shift > 2147483000LL)
        return pasio_fail(ctx, PASIO_E_ARG, "window_size and window_shift must be positive");
    if (constraint < 0 || constraint > 2) return pasio_fail(ctx, PASIO_E_ARG, "unknown constraint %d", constraint);
    if (n_in) *n_in = ctx->m;
    if (n_out) *n_out = ctx->m;
    if (cells) *cells = 0;
    i64 nwin = 0;
    PASIO_TRY(build_window_table(ctx, window_size, window_shift, &nwin));
    i64 max_span = 0, max_cnt = 0;
    PASIO_TRY(launch_window_prepass(ctx, nwin, (int)window_size, (int)window_shift, &max_span, &max_cnt, constraint));
    static const bool debug = getenv("PASIO_DEBUG") != nullptr;
    if (debug)
        fprintf(stderr, "[pasio_round] n=%lld contigs=%lld m=%lld implicit=%d nwin=%lld size=%lld shift=%lld max_span=%lld max_cnt=%lld ntab=%lld,%lld,%lld\n",
                (long long)ctx->n, (long long)ctx->n_contigs, (long long)ctx->m, (int)ctx->implicit_all, (long long)nwin,
                (long long)window_size, (long long)window_shift, (long long)max_span, (long long)max_cnt,
                (long long)ctx->ntab[0], (long long)ctx->ntab[1], (long long)ctx->ntab[2]);
    if (max_cnt > ctx->total || max_span > ctx->n)      // cannot happen with a consistent prefix-sum / candidate state
        return pasio_fail(ctx, PASIO_E_CUDA, "internal inconsistency before the window DP: window count %lld / span %lld exceed "
                          "contig total %lld / length %lld (m=%lld, implicit=%d, windows=%lld)", (long long)max_cnt,
                          (long long)max_span, (long long)ctx->total, (long long)ctx->n, (long long)ctx->m,
                          (int)ctx->implicit_all, (long long)nwin);
    PASIO_TRY(check_dp_tables(ctx, max_span, max_cnt, true));

    const size_t bit_bytes = (size_t)((ctx->n + 1 + 31) / 32 + 2) * 4;
    CUDA_TRY(ctx, cudaMemsetAsync(ctx->keepbits.p, 0, bit_bytes, ctx->stream));
    if (penalties_on(ctx)) PASIO_TRY(launch_window_dp_reg(ctx, nwin, (int)window_size, (int)window_shift, constraint));
    else PASIO_TRY(launch_window_dp(ctx, nwin, (int)window_size, (int)window_shift, constraint));

    // survivors: at most the current count (the new list is a subset, round_reducer.py:25)
    const int nxt = 1 - ctx->cur;
    PASIO_TRY(pasio_reserve(ctx, ctx->cand[nxt], (size_t)ctx->m * 4));
    i64 m_new = 0;
    PASIO_TRY(launch_compact_keepbits(ctx, nxt, &m_new));
    PASIO_TRY(d2h(ctx, ctx->h_scalars + 10, ctx->scalars.as<i64>() + 10, 24));
    PASIO_TRY(d2h(ctx, ctx->h_scalars + 16, ctx->scalars.as<i64>() + 16, 24));
    if (cells) *cells = ctx->h_scalars[10];
    ctx->last_cells = ctx->h_scalars[10];
    ctx->last_cells_skipped = ctx->h_scalars[12];
    for (int k = 0; k < 3; ++k) ctx->last_certify[k] = ctx->h_scalars[16 + k];
    ctx->prev_round_in = ctx->m;
    ctx->prev_round_out = m_new;
    ctx->cur = nxt;
    ctx->implicit_all = false;
    ctx->m = m_new;
    if (n_out) *n_out = m_new;
    return refresh_boundary_ranks(ctx);
}

extern "C" int pasio_rounds(pasio_ctx *ctx, int64_t window_size, int64_t window_shift, int constraint,
                            int64_t max_rounds, int64_t *rounds_done, int64_t *n_out, int64_t *cells,
                            int64_t *sizes, int64_t sizes_cap)
{
    NEED_CTX(ctx);
    if (!ctx->have_contig) return pasio_fail(ctx, PASIO_E_STATE, "no contig loaded");
    // round_reducer.py:11-15: None -> len(counts); at least one round
    i64 limit = max_rounds <= 0 ? ctx->n : max_rounds;
    if (limit < 1) limit = 1;
    i64 done = 0, total_cells = 0;
    int rc = PASIO_OK;
    while (done < limit) {
        int64_t a = 0, b = 0, c = 0;
        rc = pasio_round(ctx, window_size, window_shift, constraint, &a, &b, &c);
        if (rc != PASIO_OK) break;
        if (sizes && done < sizes_cap) sizes[done] = a;
        ++done;
        total_cells += c;
        if (a == b) break;               // np.array_equal(new, old): fixed point (round_reducer.py:21)
    }
    if (rounds_done) *rounds_done = done;
    if (n_out) *n_out = ctx->m;
    if (cells) *cells = total_cells;
    return rc;
}

extern "C" int pasio_upload_stats(const pasio_ctx *ctx, int64_t *wire_bytes)
{
    if (!ctx || !wire_bytes) return PASIO_E_ARG;
    *wire_bytes = ctx->last_wire_bytes;
    return PASIO_OK;
}

extern "C" int pasio_round_stats(const pasio_ctx *ctx, int64_t *cells, int64_t *cells_skipped)
{
    if (!ctx) return PASIO_E_ARG;
    if (cells) *cells = ctx->last_cells;
    if (cells_skipped) *cells_skipped = ctx->last_cells_skipped;
    return PASIO_OK;
}

extern "C" int pasio_round_certify_stats(const pasio_ctx *ctx, int64_t *passed, int64_t *fell_back, int64_t *resume_rows_sum)
{
    if (!ctx) return PASIO_E_ARG;
    if (passed) *passed = ctx->last_certify[0];
    if (fell_back) *fell_back = ctx->last_certify[1];
    if (resume_rows_sum) *resume_rows_sum = ctx->last_certify[2];
    return PASIO_OK;
}

extern "C" int pasio_set_tuning(pasio_ctx *ctx, int key, int value)
{
    if (!ctx) return PASIO_E_ARG;
    if (key < 0 || key >= PASIO_TUNE_COUNT) return pasio_fail(ctx, PASIO_E_ARG, "unknown tuning key %d", key);
    if (key == PASIO_TUNE_EXACT_LAG && (value < 3 || value > 5)) return pasio_fail(ctx, PASIO_E_ARG, "exact lag must be 3, 4 or 5");
    ctx->tune[key] = value;
    if (key == PASIO_TUNE_LOGFAC_EXACT) {
        if (ctx->logfac_pending) { cudaStreamSynchronize(ctx->stream_lx); ctx->logfac_pending = false; }
        ctx->logfac_ready = false;
        ctx->logfac_eager = false;
    }
    return PASIO_OK;
}

// ---- exact DP -----------------------------------------------------------------------------------
// shared tail of the two exact-DP entry points: results of the DP over the current candidates -> caller, back-trace, the
// splits become the current candidates
static int finish_square_split(pasio_ctx *ctx, i64 N, int64_t *out_splits, int64_t cap, int64_t *n_splits, double *score,
                               double *prefix_scores, int64_t *previous_splits)
{
    if (score) PASIO_TRY(d2h(ctx, score, ctx->dpP.as<double>() + (N - 1), 8));
    if (prefix_scores) PASIO_TRY(d2h(ctx, prefix_scores, ctx->dpP.p, (size_t)N * 8));
    if (previous_splits) {
        std::vector<int> tmp((size_t)N);
        PASIO_TRY(d2h(ctx, tmp.data(), ctx->dpPrev.p, (size_t)N * 4));
        for (i64 k = 0; k < N; ++k) previous_splits[k] = tmp[(size_t)k];
    }
    PASIO_TRY(launch_backtrace_mark(ctx, N));
    ctx->prev_round_in = 0;
    const int nxt = 1 - ctx->cur;
    PASIO_TRY(pasio_reserve(ctx, ctx->cand[nxt], (size_t)N * 4));
    i64 m_new = 0;
    PASIO_TRY(launch_compact_keepbits(ctx, nxt, &m_new));
    ctx->cur = nxt;
    ctx->implicit_all = false;
    ctx->m = m_new;
    PASIO_TRY(refresh_boundary_ranks(ctx));
    if (n_splits) *n_splits = m_new;
    if (out_splits) {
        if (cap < m_new) return pasio_fail(ctx, PASIO_E_ARG, "capacity %lld < %lld splits", (long long)cap, (long long)m_new);
        return pasio_candidates_download(ctx, out_splits, cap, nullptr);
    }
    return PASIO_OK;
}

extern "C" int pasio_square_split(pasio_ctx *ctx, int64_t *out_splits, int64_t cap, int64_t *n_splits,
                                  double *score, double *prefix_scores, int64_t *previous_splits)
{
    NEED_CTX(ctx);
    if (!ctx->have_contig) return pasio_fail(ctx, PASIO_E_STATE, "no contig loaded");
    if (ctx->n_contigs != 1) return pasio_fail(ctx, PASIO_E_STATE, "pasio_square_split works on a single-contig context");
    const i64 N = ctx->m;
    // candidates span the whole contig: first = 0, last = n
    PASIO_TRY(check_dp_tables(ctx, ctx->n, ctx->total));
    PASIO_TRY(launch_gather_candidates(ctx));
    PASIO_TRY(launch_exact_dp(ctx, N));
    return finish_square_split(ctx, N, out_splits, cap, n_splits, score, prefix_scores, previous_splits);
}

extern "C" int pasio_square_split_regularized(pasio_ctx *ctx, const double *length_penalty, int64_t n_length_penalty,
                                              const double *split_number_penalty, int64_t n_split_number_penalty,
                                              double first_column_refund, int64_t *out_splits, int64_t cap, int64_t *n_splits,
                                              double *score, double *prefix_scores, int64_t *previous_splits)
{
    NEED_CTX(ctx);
    if (!ctx->have_contig) return pasio_fail(ctx, PASIO_E_STATE, "no contig loaded");
    if (ctx->n_contigs != 1) return pasio_fail(ctx, PASIO_E_STATE, "pasio_square_split_regularized works on a single-contig context");
    const i64 N = ctx->m;
    if (length_penalty && n_length_penalty < ctx->n + 1)
        return pasio_fail(ctx, PASIO_E_ARG, "length penalty table needs %lld entries (0 .. contig length)", (long long)(ctx->n + 1));
    if (split_number_penalty && n_split_number_penalty < N)
        return pasio_fail(ctx, PASIO_E_ARG, "split-number penalty table needs %lld entries (one per candidate)", (long long)N);
    PASIO_TRY(check_dp_tables(ctx, ctx->n, ctx->total));
    PASIO_TRY(launch_gather_candidates(ctx));
    const double *d_lr = nullptr, *d_nr = nullptr;
    if (length_penalty) {
        PASIO_TRY(pasio_reserve(ctx, ctx->regLR, (size_t)(ctx->n + 1) * 8));
        PASIO_TRY(h2d(ctx, ctx->regLR.p, length_penalty, (size_t)(ctx->n + 1) * 8));
        d_lr = ctx->regLR.as<double>();
    }
    if (split_number_penalty) {
        PASIO_TRY(pasio_reserve(ctx, ctx->regNR, (size_t)N * 8));
        PASIO_TRY(h2d(ctx, ctx->regNR.p, split_number_penalty, (size_t)N * 8));
        d_nr = ctx->regNR.as<double>();
    }
    PASIO_TRY(launch_regularized_dp(ctx, N, d_lr, d_nr, first_column_refund));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));      // the caller's tables were read by the copies above
    return finish_square_split(ctx, N, out_splits, cap, n_splits, score, prefix_scores, previous_splits);
}

extern "C" int pasio_suffix_scores(pasio_ctx *ctx, int64_t stop, double *out)
{
    NEED_CTX(ctx);
    if (!ctx->have_contig) return pasio_fail(ctx, PASIO_E_STATE, "no contig loaded");
    if (stop < 0 || stop >= ctx->m || !out) return pasio_fail(ctx, PASIO_E_ARG, "stop out of range");
    if (stop == 0) return PASIO_OK;
    // arguments are bounded by the span / count between candidate 0 and candidate `stop`
    i64 ends[2] = {0, stop};
    i64 pos[2] = {0, stop};
    if (!ctx->implicit_all) {
        int32_t p32[2];
        PASIO_TRY(d2h(ctx, &p32[0], ctx->cand[ctx->cur].as<int32_t>() + ends[0], 4));
        PASIO_TRY(d2h(ctx, &p32[1], ctx->cand[ctx->cur].as<int32_t>() + ends[1], 4));
        pos[0] = p32[0];
        pos[1] = p32[1];
    }
    i64 c[2];
    PASIO_TRY(d2h(ctx, &c[0], ctx->cg.as<i64>() + pos[0], 8));
    PASIO_TRY(d2h(ctx, &c[1], ctx->cg.as<i64>() + pos[1], 8));
    PASIO_TRY(check_dp_tables(ctx, pos[1] - pos[0], c[1] - c[0]));
    PASIO_TRY(pasio_reserve(ctx, ctx->dpP, (size_t)stop * 8));
    PASIO_TRY(launch_suffix_row(ctx, stop, ctx->dpP.as<double>()));
    return d2h(ctx, out, ctx->dpP.p, (size_t)stop * 8);
}

// ---- per-segment outputs ------------------------------------------------------------------------
// float64 prefix sums of lgamma(counts + 1) over the loaded contig (logfac_cumsum, log_marginal_likelyhood.py:59-60)
// in ctx->logfac_full, computed once per loaded contig.  (Running it on a side stream beside the rounds was tried:
// the bandwidth-bound scan and the latency-bound window kernels slow each other down by as much as is hidden.)
static int ensure_logfac(pasio_ctx *ctx)
{
    if (ctx->logfac_pending) {                 // prefetched on the side stream: order the consumers behind it
        CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_lx1, 0));
        ctx->logfac_pending = false;
    }
    if (ctx->logfac_eager) {                   // formed chunk by chunk behind the upload: how many terms, and were they all in the table?
        ctx->logfac_eager = false;
        CUDA_TRY(ctx, cudaEventSynchronize(ctx->ev_lx1));
        bool usable = false;
        PASIO_TRY(logfac_exact_chunks_result(ctx, &usable));
        if (!usable) ctx->logfac_ready = false;           // the ordinary path below checks the table and reports what is wrong
    }
    if (ctx->logfac_ready) return PASIO_OK;
    if (ctx->tune[PASIO_TUNE_LOGFAC_EXACT]) {
        PASIO_TRY(launch_logfac_exact(ctx));              // the reference's sequential sum, bit for bit (logfac_exact.cu)
    } else {
        PASIO_TRY(pasio_reserve(ctx, ctx->logfac_full, (size_t)(ctx->n + 1) * 8));
        PASIO_TRY(launch_logfac_scan(ctx, ctx->logfac_full.as<double>()));
    }
    ctx->logfac_ready = true;
    ctx->logfac_is_exact = ctx->tune[PASIO_TUNE_LOGFAC_EXACT] != 0;
    return PASIO_OK;
}

// Start the sequential log-factorial sums of the loaded batch on a side stream, so that they run (one thread per contig:
// no SM is taken away) beside the rounds that follow; pasio_segment_lmm / pasio_segment_scores then find them done.
extern "C" int pasio_logfac_prefetch(pasio_ctx *ctx)
{
    NEED_CTX(ctx);
    if (!ctx->have_contig) return pasio_fail(ctx, PASIO_E_STATE, "no contig loaded");
    if (ctx->logfac_ready || ctx->logfac_pending || !ctx->tune[PASIO_TUNE_LOGFAC_EXACT]) return PASIO_OK;
    if (ctx->max_count + 2 > ctx->ntab[PASIO_TAB_LGAMMA]) return PASIO_OK;     // the table must grow first: left to the consumer
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev_lx0, ctx->stream));
    CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->stream_lx, ctx->ev_lx0, 0));
    PASIO_TRY(launch_logfac_exact(ctx, ctx->stream_lx));
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev_lx1, ctx->stream_lx));
    ctx->logfac_ready = true;
    ctx->logfac_is_exact = true;
    ctx->logfac_pending = true;
    return PASIO_OK;
}

extern "C" int pasio_segment_scores(pasio_ctx *ctx, double *scores, int64_t *segment_counts, double *mean_counts,
                                    double *logfac_cumsum, int64_t capacity, int64_t *n_segments)
{
    NEED_CTX(ctx);
    if (!ctx->have_contig) return pasio_fail(ctx, PASIO_E_STATE, "no contig loaded");
    if (!ctx->have_params) return pasio_fail(ctx, PASIO_E_STATE, "pasio_set_params has not been called");
    const i64 nseg = ctx->m - 1;
    if (n_segments) *n_segments = nseg;
    if (capacity < nseg && (scores || segment_counts || mean_counts))
        return pasio_fail(ctx, PASIO_E_ARG, "capacity %lld < %lld segments", (long long)capacity, (long long)nseg);
    if (scores || segment_counts || mean_counts) {
        // largest segment length / count decide the table lengths (windows of 2 candidates, shift 1)
        const i64 saved_contigs = ctx->n_contigs;
        ctx->n_contigs = 1;   // closed-form geometry over the whole list; segments never cross boundaries
        i64 max_len = 0, max_cnt = 0;
        int rc = launch_window_prepass(ctx, nseg, 1, 1, &max_len, &max_cnt);
        ctx->n_contigs = saved_contigs;
        PASIO_TRY(rc);
        bool bad = false;
        if (ctx->ntab[PASIO_TAB_LOG] < max_len + 1) { ctx->need[PASIO_TAB_LOG] = max_len + 1; bad = true; }
        if (ctx->ntab[PASIO_TAB_LGAMMA_ALPHA] < max_cnt + 1) { ctx->need[PASIO_TAB_LGAMMA_ALPHA] = max_cnt + 1; bad = true; }
        if (bad) return pasio_fail(ctx, PASIO_E_TABLE_TOO_SHORT, "tables too short for segment scores: need log>=%lld, lgamma_alpha>=%lld",
                                   (long long)(max_len + 1), (long long)(max_cnt + 1));
        PASIO_TRY(pasio_reserve(ctx, ctx->dpP, (size_t)nseg * 8));
        PASIO_TRY(pasio_reserve(ctx, ctx->dpJump, (size_t)nseg * 8));
        PASIO_TRY(pasio_reserve(ctx, ctx->dpPart, (size_t)nseg * 8));
        PASIO_TRY(launch_segment_scores(ctx, ctx->dpP.as<double>(), ctx->dpJump.as<i64>(), ctx->dpPart.as<double>()));
        if (scores) PASIO_TRY(d2h(ctx, scores, ctx->dpP.p, (size_t)nseg * 8));
        if (segment_counts) PASIO_TRY(d2h(ctx, segment_counts, ctx->dpJump.p, (size_t)nseg * 8));
        if (mean_counts) PASIO_TRY(d2h(ctx, mean_counts, ctx->dpPart.p, (size_t)nseg * 8));
    }
    if (logfac_cumsum) {
        if (capacity < nseg) return pasio_fail(ctx, PASIO_E_ARG, "capacity too small");
        // n+1 doubles of scratch, kept for the next call (a 2 GB cudaMalloc/cudaFree per contig is not free)
        PASIO_TRY(ensure_logfac(ctx));
        PASIO_TRY(pasio_reserve(ctx, ctx->dpP, (size_t)ctx->m * 8));
        if (ctx->logfac_is_exact) PASIO_TRY(launch_logfac_at_candidates_exact(ctx, ctx->dpP.as<double>()));
        else PASIO_TRY(launch_gather_f64_at_cands(ctx, ctx->logfac_full.as<double>(), ctx->dpP.as<double>()));
        PASIO_TRY(d2h(ctx, logfac_cumsum, ctx->dpP.p, (size_t)ctx->m * 8));
    }
    return PASIO_OK;
}


// ---- np.sum of the segment scores, in numpy's pairwise order ------------------------------------
static void pw_leaves(i64 lo, i64 n, std::vector<i64> &starts)
{
    if (n <= 128) { starts.push_back(lo); return; }
    i64 n2 = n / 2;
    n2 -= n2 % 8;
    pw_leaves(lo, n2, starts);
    pw_leaves(lo + n2, n - n2, starts);
}
static double pw_combine(const double *leaf, i64 &next, i64 n)
{
    if (n <= 128) return leaf[next++];
    i64 n2 = n / 2;
    n2 -= n2 % 8;
    const double a = pw_combine(leaf, next, n2);
    const double b = pw_combine(leaf, next, n - n2);
    return a + b;
}

extern "C" int pasio_segment_scores_sum(pasio_ctx *ctx, double *total)
{
    NEED_CTX(ctx);
    if (!total) return pasio_fail(ctx, PASIO_E_ARG, "NULL output");
    int64_t nseg = 0;
    // scores of the current candidates into dpP (same checks and kernel as pasio_segment_scores)
    PASIO_TRY(pasio_segment_scores(ctx, nullptr, nullptr, nullptr, nullptr, 0, &nseg));
    {
        const i64 saved_contigs = ctx->n_contigs;
        ctx->n_contigs = 1;
        i64 max_len = 0, max_cnt = 0;
        int rc = launch_window_prepass(ctx, nseg, 1, 1, &max_len, &max_cnt);
        ctx->n_contigs = saved_contigs;
        PASIO_TRY(rc);
        bool bad = false;
        if (ctx->ntab[PASIO_TAB_LOG] < max_len + 1) { ctx->need[PASIO_TAB_LOG] = max_len + 1; bad = true; }
        if (ctx->ntab[PASIO_TAB_LGAMMA_ALPHA] < max_cnt + 1) { ctx->need[PASIO_TAB_LGAMMA_ALPHA] = max_cnt + 1; bad = true; }
        if (bad) return pasio_fail(ctx, PASIO_E_TABLE_TOO_SHORT, "tables too short for segment scores");
    }
    PASIO_TRY(pasio_reserve(ctx, ctx->dpP, (size_t)nseg * 8));
    PASIO_TRY(launch_segment_scores(ctx, ctx->dpP.as<double>(), nullptr, nullptr));
    if (ctx->pw_n != nseg) {
        ctx->pw_leaf_start.clear();
        pw_leaves(0, nseg, ctx->pw_leaf_start);
        ctx->pw_leaf_start.push_back(nseg);
        ctx->pw_n = nseg;
    }
    const i64 n_leaves = (i64)ctx->pw_leaf_start.size() - 1;
    PASIO_TRY(pasio_reserve(ctx, ctx->dpJump, (size_t)(n_leaves + 1) * 8));
    PASIO_TRY(pasio_reserve(ctx, ctx->dpPart, (size_t)n_leaves * 8));
    PASIO_TRY(h2d(ctx, ctx->dpJump.p, ctx->pw_leaf_start.data(), (size_t)(n_leaves + 1) * 8));
    PASIO_TRY(launch_pairwise_leaves(ctx, ctx->dpP.as<double>(), ctx->dpJump.as<i64>(), n_leaves, ctx->dpPart.as<double>()));
    ctx->pw_leaf_sum.resize((size_t)n_leaves);
    PASIO_TRY(d2h(ctx, ctx->pw_leaf_sum.data(), ctx->dpPart.p, (size_t)n_leaves * 8));
    i64 next = 0;
    *total = pw_combine(ctx->pw_leaf_sum.data(), next, nseg);
    return PASIO_OK;
}

extern "C" int pasio_segment_lmm(pasio_ctx *ctx, double *lmm, int64_t capacity, double *sum_logfac)
{
    NEED_CTX(ctx);
    if (!ctx->have_contig) return pasio_fail(ctx, PASIO_E_STATE, "no contig loaded");
    const i64 nseg = ctx->m - 1;
    if (lmm && capacity < nseg) return pasio_fail(ctx, PASIO_E_ARG, "capacity %lld < %lld segments", (long long)capacity, (long long)nseg);
    if (!ctx->have_params) return pasio_fail(ctx, PASIO_E_STATE, "pasio_set_params has not been called");
    i64 max_len = 0, max_cnt = 0;
    {
        const i64 saved = ctx->n_contigs;
        ctx->n_contigs = 1;
        int rc = launch_window_prepass(ctx, nseg, 1, 1, &max_len, &max_cnt);
        ctx->n_contigs = saved;
        PASIO_TRY(rc);
    }
    bool bad = false;
    if (ctx->ntab[PASIO_TAB_LOG] < max_len + 1) { ctx->need[PASIO_TAB_LOG] = max_len + 1; bad = true; }
    if (ctx->ntab[PASIO_TAB_LGAMMA_ALPHA] < max_cnt + 1) { ctx->need[PASIO_TAB_LGAMMA_ALPHA] = max_cnt + 1; bad = true; }
    if (bad) return pasio_fail(ctx, PASIO_E_TABLE_TOO_SHORT, "tables too short for segment scores");
    PASIO_TRY(pasio_reserve(ctx, ctx->dpP, (size_t)nseg * 8));
    PASIO_TRY(launch_segment_scores(ctx, ctx->dpP.as<double>(), nullptr, nullptr));
    PASIO_TRY(ensure_logfac(ctx));
    PASIO_TRY(pasio_reserve(ctx, ctx->dpPart, (size_t)nseg * 8));
    if (ctx->logfac_is_exact) PASIO_TRY(launch_lmm_exact(ctx, ctx->dpP.as<double>(), ctx->dpPart.as<double>()));
    else PASIO_TRY(launch_lmm(ctx, ctx->dpP.as<double>(), ctx->logfac_full.as<double>(), ctx->dpPart.as<double>()));
    if (lmm) PASIO_TRY(d2h(ctx, lmm, ctx->dpPart.p, (size_t)nseg * 8));
    if (sum_logfac) {
        if (ctx->logfac_is_exact) PASIO_TRY(logfac_exact_total(ctx, sum_logfac));     // (a batch: the last contig's total)
        else PASIO_TRY(d2h(ctx, sum_logfac, ctx->logfac_full.as<double>() + ctx->n, 8));
    }
    return PASIO_OK;
}

// ---- pinned host buffers ------------------------------------------------------------------------
extern "C" int pasio_host_alloc(int64_t bytes, void **out)
{
    if (!out || bytes < 0) return PASIO_E_ARG;
    *out = nullptr;
    cudaError_t e = cudaHostAlloc(out, (size_t)(bytes > 0 ? bytes : 1), cudaHostAllocDefault);
    if (e != cudaSuccess) return pasio_fail(nullptr, PASIO_E_NOMEM, "cudaHostAlloc(%lld) failed: %s", (long long)bytes, cudaGetErrorString(e));
    return PASIO_OK;
}

extern "C" int pasio_host_free(void *ptr)
{
    if (ptr) cudaFreeHost(ptr);
    return PASIO_OK;
}

// ---- measurement hooks --------------------------------------------------------------------------
extern "C" void *pasio_stream(pasio_ctx *ctx) { return ctx ? (void *)ctx->stream : nullptr; }

__global__ void __launch_bounds__(256) fp64_peak_kernel(double *out, int iters, double a, double b)
{
    double x0 = threadIdx.x, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
    for (int i = 0; i < iters; ++i) {
        x0 = __fma_rn(x0, a, b); x1 = __fma_rn(x1, a, b); x2 = __fma_rn(x2, a, b); x3 = __fma_rn(x3, a, b);
        x4 = __fma_rn(x4, a, b); x5 = __fma_rn(x5, a, b); x6 = __fma_rn(x6, a, b); x7 = __fma_rn(x7, a, b);
    }
    out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = ((x0 + x1) + (x2 + x3)) + ((x4 + x5) + (x6 + x7));
}

extern "C" int pasio_fp64_peak(pasio_ctx *ctx, double *instr_per_sec)
{
    NEED_CTX(ctx);
    if (!instr_per_sec) return pasio_fail(ctx, PASIO_E_ARG, "NULL output");
    const int blocks = ctx->sm_count * 8, iters = 1 << 15;
    PASIO_TRY(pasio_reserve(ctx, ctx->dpPart, (size_t)blocks * 256 * 8));
    cudaEvent_t a, b;
    cudaEventCreate(&a);
    cudaEventCreate(&b);
    double best = 0;
    for (int rep = 0; rep < 4; ++rep) {
        cudaEventRecord(a, ctx->stream);
        fp64_peak_kernel<<<blocks, 256, 0, ctx->stream>>>(ctx->dpPart.as<double>(), iters, 0.999999, 1e-9);
        cudaEventRecord(b, ctx->stream);
        cudaError_t e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) return pasio_fail(ctx, PASIO_E_CUDA, "fp64 peak kernel: %s", cudaGetErrorString(e));
        float ms = 0;
        cudaEventElapsedTime(&ms, a, b);
        double rate = (double)blocks * 256 * 8.0 * iters / (ms * 1e-3);
        if (rep > 0 && rate > best) best = rate;
    }
    cudaEventDestroy(a);
    cudaEventDestroy(b);
    *instr_per_sec = best;
    return PASIO_OK;
}

extern "C" int pasio_timing_reset(pasio_ctx *ctx, int enable)
{
    NEED_CTX(ctx);
    PASIO_TRY(resolve_spans(ctx));
    for (int f = 0; f < TF_COUNT; ++f) { ctx->fam_ms[f] = 0; ctx->fam_launches[f] = 0; }
    ctx->timing = enable != 0;
    return PASIO_OK;
}

extern "C" int pasio_timing_get(pasio_ctx *ctx, int family, double *ms, int64_t *launches)
{
    NEED_CTX(ctx);
    if (family < 0 || family >= TF_COUNT) return pasio_fail(ctx, PASIO_E_ARG, "unknown timing family");
    PASIO_TRY(resolve_spans(ctx));
    if (ms) *ms = ctx->fam_ms[family];
    if (launches) *launches = ctx->fam_launches[family];
    return PASIO_OK;
}
