// context.cu — runtime layer of libvgl_b200: device selection, stream, HBM allocations, error reporting.
// Replaces VGL_RUNTIME::init_library / select_device (vgl_runtime/vgl_runtime.hpp:5-16,
// helpers/gpu_API/select_device.cuh:5-8) and MemoryAPI (helpers/memory_API/memory_API.hpp:3-101): explicit
// cudaMalloc'ed HBM instead of cudaMallocManaged + prefetch hints, one stream per context instead of the
// reference's six streams + cudaDeviceSynchronize after every operator.
#include <stdarg.h>
#include <stdlib.h>

#include "common.cuh"

static thread_local char g_error[512] = "";

void vglb_set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_error, sizeof(g_error), fmt, ap);
    va_end(ap);
}

extern "C" const char *vglb_last_error(void) { return g_error; }

// ---- device memory: a size-keyed cache in front of cudaMalloc / cudaFree ----------------------------------------------
// cudaMalloc and cudaFree cost milliseconds each and cudaFree synchronises the device; a host program that moves a graph
// to the device, runs an algorithm and drops it (the end-to-end path: VGL_Graph::move_to_device + vgl_page_rank) spent
// more time in them than in its 20 sweeps. Freed blocks are kept and handed out again for requests of exactly the same
// size (re-created graphs repeat their sizes); the cache is bounded and emptied when an allocation fails. Buffers exported
// to other processes (CUDA IPC) are never recycled. (MemoryAPI::allocate_array / free_array, memory_API.hpp:3-15,95-101.)
#include <map>
#include <mutex>
#include <unordered_map>
#include <unordered_set>

namespace
{
struct DeviceCache
{
    std::mutex mu;
    std::unordered_map<void *, size_t> live;     // blocks handed out by vglb_dev_alloc
    std::unordered_set<void *> exported;         // never recycled
    struct Idle { void *ptr; uint64_t epoch; };
    std::multimap<size_t, Idle> idle;            // freed blocks by size, with the sync epoch they were freed in
    size_t idle_bytes = 0;
    uint64_t epoch = 1;                          // bumped by every device-wide synchronisation the cache performs
};
DeviceCache &cache_of_current_device()
{
    static DeviceCache caches[64];
    int dev = 0;
    cudaGetDevice(&dev);
    return caches[dev & 63];
}
size_t cache_limit()
{
    static size_t limit = 0;
    if (!limit)
    {
        size_t free_b = 0, total_b = 0;
        if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) total_b = (size_t)16 << 30;
        limit = total_b / 4;
        if (const char *e = getenv("VGLB_DEVICE_CACHE_MB")) limit = (size_t)atoll(e) << 20;
    }
    return limit;
}
void cache_release_all(DeviceCache &C)
{
    for (auto &kv : C.idle) cudaFree(kv.second.ptr);
    C.idle.clear();
    C.idle_bytes = 0;
}
} // namespace

cudaError_t vglb_dev_alloc_bytes(void **ptr, size_t bytes)
{
    if (bytes == 0) bytes = 16;
    DeviceCache &C = cache_of_current_device();
    std::lock_guard<std::mutex> lock(C.mu);
    auto it = C.idle.find(bytes);
    if (it != C.idle.end())
    {
        // Work enqueued before the block was freed may still be using it, and the next user is ordered behind that work
        // only on the same stream. Freeing does not wait (a graph frees twenty blocks in a row); the first re-use of a
        // block freed since the last device-wide synchronisation pays for ONE synchronisation that covers them all.
        if (it->second.epoch == C.epoch)
        {
            cudaDeviceSynchronize();
            C.epoch++;
        }
        *ptr = it->second.ptr;
        C.idle.erase(it);
        C.idle_bytes -= bytes;
        C.live[*ptr] = bytes;
        return cudaSuccess;
    }
    cudaError_t e = cudaMalloc(ptr, bytes);
    if (e != cudaSuccess && !C.idle.empty())
    {
        cudaGetLastError();
        cache_release_all(C); // give the cached blocks back and try once more
        e = cudaMalloc(ptr, bytes);
    }
    if (e == cudaSuccess) C.live[*ptr] = bytes;
    return e;
}

void vglb_dev_free(void *ptr)
{
    if (!ptr) return;
    DeviceCache &C = cache_of_current_device();
    std::lock_guard<std::mutex> lock(C.mu);
    auto it = C.live.find(ptr);
    if (it == C.live.end())
    {
        cudaFree(ptr); // not ours (or another device's): plain free
        return;
    }
    const size_t bytes = it->second;
    C.live.erase(it);
    if (C.exported.erase(ptr) || bytes > cache_limit())
    {
        cudaFree(ptr);
        return;
    }
    C.idle.emplace(bytes, DeviceCache::Idle{ptr, C.epoch});
    C.idle_bytes += bytes;
    while (C.idle_bytes > cache_limit() && !C.idle.empty())
    {
        auto big = std::prev(C.idle.end()); // largest first (cudaFree synchronises by itself)
        cudaFree(big->second.ptr);
        C.idle_bytes -= big->first;
        C.idle.erase(big);
    }
}

void vglb_dev_mark_exported(void *ptr)
{
    DeviceCache &C = cache_of_current_device();
    std::lock_guard<std::mutex> lock(C.mu);
    if (C.live.count(ptr)) C.exported.insert(ptr);
}

void vglb_dev_cache_release(void)
{
    DeviceCache &C = cache_of_current_device();
    std::lock_guard<std::mutex> lock(C.mu);
    cache_release_all(C);
}


extern "C" int vglb_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess)
    {
        cudaGetLastError();
        return 0;
    }
    return n;
}

extern "C" int vglb_init(int device, vglb_ctx **out_ctx)
{
    VGLB_REQUIRE(out_ctx != NULL, "vglb_init: out_ctx is NULL");
    int n = vglb_device_count();
    if (n <= 0 || device < 0 || device >= n)
    {
        vglb_set_error("vglb_init: no usable CUDA device %d (found %d); libvgl_b200 has no CPU fallback", device, n);
        return VGLB_ENODEVICE;
    }
    CUDA_TRY(cudaSetDevice(device));
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    vglb_ctx *ctx = (vglb_ctx *)calloc(1, sizeof(vglb_ctx));
    if (!ctx) return VGLB_ENOMEM;
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;
    ctx->l2_bytes = (size_t)prop.l2CacheSize;
    CUDA_TRY(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    CUDA_TRY(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
    for (int i = 0; i < 8; i++) CUDA_TRY(cudaEventCreateWithFlags(&ctx->ev_chunk[i], cudaEventDisableTiming));
    CUDA_TRY(cudaEventCreate(&ctx->ev_start));
    CUDA_TRY(cudaEventCreate(&ctx->ev_stop));
    CUDA_TRY(cudaMallocHost((void **)&ctx->h_counters, 64 * sizeof(int64_t)));
    CUDA_TRY(cudaHostAlloc((void **)&ctx->h_mailbox, 64 * sizeof(unsigned long long), cudaHostAllocMapped));
    memset(ctx->h_mailbox, 0, 64 * sizeof(unsigned long long));
    ctx->mailbox_seq = 0;
    CUDA_TRY(vglb_dev_alloc((void **)&ctx->d_counters, 64 * sizeof(int64_t)));
    CUDA_TRY(cudaMemset(ctx->d_counters, 0, 64 * sizeof(int64_t)));
    ctx->flush_bytes = ctx->l2_bytes * 2 > (size_t)(256u << 20) ? ctx->l2_bytes * 2 : (size_t)(256u << 20);
    ctx->d_flush = NULL;
    *out_ctx = ctx;
    return VGLB_OK;
}

extern "C" int vglb_finalize(vglb_ctx *ctx)
{
    if (!ctx) return VGLB_OK;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    if (ctx->d_flush) vglb_dev_free(ctx->d_flush);
    vglb_dev_free(ctx->d_counters);
    cudaFreeHost(ctx->h_counters);
    cudaFreeHost(ctx->h_mailbox);
    cudaEventDestroy(ctx->ev_start);
    cudaEventDestroy(ctx->ev_stop);
    cudaStreamDestroy(ctx->stream);
    cudaStreamDestroy(ctx->copy_stream);
    for (int i = 0; i < 8; i++) cudaEventDestroy(ctx->ev_chunk[i]);
    free(ctx);
    vglb_dev_cache_release(); // cached blocks of this device go back to the driver
    return VGLB_OK;
}

extern "C" int vglb_synchronize(vglb_ctx *ctx)
{
    VGLB_REQUIRE(ctx != NULL, "vglb_synchronize: ctx is NULL");
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return VGLB_OK;
}

// ---- counter mailbox --------------------------------------------------------------------------------------------------
__global__ void counters_publish_kernel(const unsigned long long *__restrict__ src, int words, volatile unsigned long long *mailbox,
                                        unsigned long long seq)
{
    if ((int)threadIdx.x < words) mailbox[threadIdx.x] = src[threadIdx.x];
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) mailbox[63] = seq;
}

int vglb_counters_fetch(vglb_ctx *ctx, const void *d_src, int words)
{
    VGLB_REQUIRE(words > 0 && words <= 56, "vglb_counters_fetch: at most 56 counters");
    const unsigned long long seq = ++ctx->mailbox_seq;
    counters_publish_kernel<<<1, 64, 0, ctx->stream>>>((const unsigned long long *)d_src, words, ctx->h_mailbox, seq);
    KERNEL_TRY();
    volatile unsigned long long *flag = ctx->h_mailbox + 63;
    for (unsigned spins = 1;; spins++)
    {
        if (*flag == seq) break;
        if ((spins & 0x3ff) == 0) // every ~1000 probes: has the stream died (or finished without the flag being visible yet)?
        {
            cudaError_t q = cudaStreamQuery(ctx->stream);
            if (q != cudaSuccess && q != cudaErrorNotReady)
            {
                vglb_set_error("CUDA error %s while waiting for the round's counters", cudaGetErrorString(q));
                return VGLB_ECUDA;
            }
        }
    }
    for (int i = 0; i < words; i++) ((unsigned long long *)ctx->h_counters)[i] = ctx->h_mailbox[i];
    return VGLB_OK;
}

int vglb_finish_run(vglb_ctx *ctx, int64_t launches0, vglb_stats *stats)
{
    CUDA_TRY(cudaEventRecord(ctx->ev_stop, ctx->stream));
    CUDA_TRY(cudaEventSynchronize(ctx->ev_stop));
    if (!stats) return VGLB_OK;
    float ms = 0.f;
    CUDA_TRY(cudaEventElapsedTime(&ms, ctx->ev_start, ctx->ev_stop));
    memset(stats, 0, sizeof(*stats));
    stats->seconds = ms * 1e-3;
    stats->kernel_launches = ctx->launches - launches0;
    return VGLB_OK;
}

extern "C" void *vglb_stream(vglb_ctx *ctx) { return ctx ? (void *)ctx->stream : NULL; }

extern "C" int vglb_malloc(vglb_ctx *ctx, size_t bytes, void **d_ptr)
{
    VGLB_REQUIRE(ctx != NULL && d_ptr != NULL, "vglb_malloc: NULL argument");
    CUDA_TRY(cudaSetDevice(ctx->device));
    cudaError_t e = vglb_dev_alloc(d_ptr, bytes ? bytes : 16);
    if (e != cudaSuccess)
    {
        cudaGetLastError();
        vglb_set_error("vglb_malloc: cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e));
        return VGLB_ENOMEM;
    }
    return VGLB_OK;
}

extern "C" int vglb_free(vglb_ctx *ctx, void *d_ptr)
{
    VGLB_REQUIRE(ctx != NULL, "vglb_free: ctx is NULL");
    vglb_dev_free(d_ptr);
    return VGLB_OK;
}

extern "C" int vglb_memcpy_h2d(vglb_ctx *ctx, void *d_dst, const void *h_src, size_t bytes)
{
    VGLB_REQUIRE(ctx != NULL, "vglb_memcpy_h2d: ctx is NULL");
    CUDA_TRY(cudaMemcpyAsync(d_dst, h_src, bytes, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return VGLB_OK;
}

extern "C" int vglb_memcpy_d2h(vglb_ctx *ctx, void *h_dst, const void *d_src, size_t bytes)
{
    VGLB_REQUIRE(ctx != NULL, "vglb_memcpy_d2h: ctx is NULL");
    CUDA_TRY(cudaMemcpyAsync(h_dst, d_src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return VGLB_OK;
}

extern "C" int vglb_memcpy_d2d(vglb_ctx *ctx, void *d_dst, const void *d_src, size_t bytes)
{
    VGLB_REQUIRE(ctx != NULL, "vglb_memcpy_d2d: ctx is NULL");
    CUDA_TRY(cudaMemcpyAsync(d_dst, d_src, bytes, cudaMemcpyDeviceToDevice, ctx->stream));
    return VGLB_OK;
}

extern "C" int vglb_memset(vglb_ctx *ctx, void *d_dst, int byte_value, size_t bytes)
{
    VGLB_REQUIRE(ctx != NULL, "vglb_memset: ctx is NULL");
    CUDA_TRY(cudaMemsetAsync(d_dst, byte_value, bytes, ctx->stream));
    return VGLB_OK;
}

extern "C" int vglb_host_alloc_pinned(size_t bytes, void **h_ptr)
{
    VGLB_REQUIRE(h_ptr != NULL, "vglb_host_alloc_pinned: NULL argument");
    cudaError_t e = cudaMallocHost(h_ptr, bytes ? bytes : 16);
    if (e != cudaSuccess)
    {
        cudaGetLastError();
        vglb_set_error("vglb_host_alloc_pinned(%zu): %s", bytes, cudaGetErrorString(e));
        return VGLB_ENOMEM;
    }
    return VGLB_OK;
}

extern "C" int vglb_host_free_pinned(void *h_ptr)
{
    if (h_ptr) CUDA_TRY(cudaFreeHost(h_ptr));
    return VGLB_OK;
}

__global__ void flush_l2_kernel(uint4 *buf, size_t n16, uint32_t tag)
{
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    size_t stride = (size_t)gridDim.x * blockDim.x;
    for (; i < n16; i += stride) buf[i] = make_uint4(tag, tag + 1, tag + 2, tag + 3);
}

extern "C" int vglb_flush_l2(vglb_ctx *ctx)
{
    VGLB_REQUIRE(ctx != NULL, "vglb_flush_l2: ctx is NULL");
    if (!ctx->d_flush) CUDA_TRY(vglb_dev_alloc(&ctx->d_flush, ctx->flush_bytes));
    static uint32_t tag = 1;
    flush_l2_kernel<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>((uint4 *)ctx->d_flush, ctx->flush_bytes / 16, tag++);
    KERNEL_TRY();
    return VGLB_OK;
}

// ---- synthetic inputs --------------------------------------------------------------------------------------------

__global__ void generate_edges_kernel(int kind, int scale, int64_t edges, uint64_t seed, int a, int b, int c,
                                      int32_t *__restrict__ src, int32_t *__restrict__ dst)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; i < edges; i += stride)
    {
        int32_t s, d;
        vglb_gen_edge(kind, scale, seed, (uint64_t)i, a, b, c, &s, &d);
        src[i] = s;
        dst[i] = d;
    }
}

extern "C" int vglb_generate_edges_device(vglb_ctx *ctx, int kind, int scale, int64_t edges, uint64_t seed, int a,
                                          int b, int c, int32_t *d_src, int32_t *d_dst)
{
    VGLB_REQUIRE(ctx != NULL && d_src != NULL && d_dst != NULL, "vglb_generate_edges_device: NULL argument");
    VGLB_REQUIRE(scale >= 1 && scale <= 30 && edges >= 0, "vglb_generate_edges_device: bad scale/edges");
    VGLB_REQUIRE(kind >= 0 && kind <= 2 && a > 0 && b >= 0 && c >= 0 && a + b + c < 100,
                 "vglb_generate_edges_device: bad kind or probabilities");
    if (edges == 0) return VGLB_OK;
    generate_edges_kernel<<<ctx->sm_count * 16, 256, 0, ctx->stream>>>(kind, scale, edges, seed, a, b, c, d_src, d_dst);
    KERNEL_TRY();
    ctx->launches++;
    return VGLB_OK;
}

extern "C" int vglb_generate_edges_host(int kind, int scale, int64_t edges, uint64_t seed, int a, int b, int c,
                                        int32_t *h_src, int32_t *h_dst)
{
    VGLB_REQUIRE(h_src != NULL && h_dst != NULL, "vglb_generate_edges_host: NULL argument");
    VGLB_REQUIRE(scale >= 1 && scale <= 30 && edges >= 0, "vglb_generate_edges_host: bad scale/edges");
    VGLB_REQUIRE(kind >= 0 && kind <= 2 && a > 0 && b >= 0 && c >= 0 && a + b + c < 100,
                 "vglb_generate_edges_host: bad kind or probabilities");
    for (int64_t i = 0; i < edges; i++) vglb_gen_edge(kind, scale, seed, (uint64_t)i, a, b, c, &h_src[i], &h_dst[i]);
    return VGLB_OK;
}
