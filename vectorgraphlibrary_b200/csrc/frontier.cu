// frontier.cu — the GPU frontier object and the lambda-free operators on it (sm_100a):
//   VGL_Frontier / FrontierVectorCSR (vgl_datastructures/frontier/containers/vect_csr/frontier_vect_csr.h:5-53,
//   modification.hpp:5-145), generate_new_frontier (vgl_compute_api/common/generate_new_frontier.hpp:4-43 ->
//   multicore/generate_new_frontier.hpp:35-108, ParallelPrimitives::copy_if_indexes copy_if.hpp:127-191,276-301)
//   and reduce (common/reduce.hpp:4-67 -> multicore/reduce.hpp:5-151).
//
// Reference GNF: three `estimate_sorted_frontier_part_size` passes write int flags[V] and count, then a second pass
// (copy_if_indexes: per-thread buckets + offset scan) compacts the ids — two V-passes, 8 bytes of frontier state per
// vertex; the reference GPU path uses set_frontier_flags + thrust::copy_if + split_frontier + a reduce
// (gpu/generate_new_frontier.hpp:86-157), four launches and three host syncs.
//
// B200 design: ONE kernel. A CTA owns a tile of 2048 consecutive vertices; every warp evaluates the predicate on 32
// consecutive vertices at a time (coalesced), `__ballot_sync` turns the 32 answers into one word of the dense bitmap
// (V/8 bytes), `__popc` counts them; warp totals are scanned through shared memory, the CTA's exclusive offset comes
// from a decoupled look-back over per-tile status words (tiles are claimed through an atomic ticket so predecessors are
// always resident), and active ids are written in ascending order — order-preserving like copy_if_indexes, which is what
// keeps degree tiers contiguous prefixes of the id list (ids are degree-sorted). The same pass accumulates the frontier
// size, the sum of degrees (neighbours) and the three tier populations, so no further kernel or reduce is needed.
// Density switch as the multicore reference: size == V -> ALL_ACTIVE, size/V > 0.7 -> DENSE (bitmap is the
// authoritative form), else SPARSE (multicore/generate_new_frontier.hpp:67-91).
#include <stdlib.h>

#include "common.cuh"
#include "frontier.cuh"

#define GNF_THREADS 256
#define GNF_WORDS_PER_WARP 8
#define GNF_TILE (GNF_THREADS * GNF_WORDS_PER_WARP) // vertices per CTA

#define TILE_FLAG_AGGREGATE (1ULL << 62)
#define TILE_FLAG_PREFIX (2ULL << 62)
#define TILE_VALUE_MASK ((1ULL << 62) - 1ULL)

// counter slots used by the GNF kernel (unsigned long long, in the frontier's own counter block)
enum
{
    G_TICKET = 0,
    G_SIZE = 1,
    G_NEIGHBOURS = 2,
    G_TIER0 = 3,
    G_TIER1 = 4,
    G_TIER2 = 5,
    G_COUNT = 8
};

struct PredFlags
{
    const int32_t *flags;
    __device__ __forceinline__ bool operator()(int32_t v) const { return flags[v] > 0; }
};
struct PredEqI32
{
    const int32_t *values;
    int32_t key;
    __device__ __forceinline__ bool operator()(int32_t v) const { return values[v] == key; }
};
struct PredNeU32
{
    const uint32_t *a, *b;
    __device__ __forceinline__ bool operator()(int32_t v) const { return a[v] != b[v]; }
};

struct PredBitmap
{
    const uint32_t *bits;
    __device__ __forceinline__ bool operator()(int32_t v) const { return (bits[v >> 5] >> (v & 31)) & 1u; }
};

template <class Pred>
__global__ void __launch_bounds__(GNF_THREADS)
gnf_compact_kernel(Pred pred, const int64_t *__restrict__ ptr, int32_t V, int32_t b0, int32_t b1,
                   uint32_t *__restrict__ bitmap, int32_t *__restrict__ ids, unsigned long long *tile_status,
                   unsigned long long *counters)
{
    __shared__ int s_tile;
    __shared__ int s_warp_count[GNF_THREADS / 32];
    __shared__ unsigned long long s_prefix;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) s_tile = (int)atomicAdd(&counters[G_TICKET], 1ULL);
    __syncthreads();
    const int tile = s_tile;
    const int64_t warp_base = (int64_t)tile * GNF_TILE + (int64_t)warp * (32 * GNF_WORDS_PER_WARP);

    uint32_t words[GNF_WORDS_PER_WARP];
    int count = 0;
    long long deg_sum = 0;
    int t0 = 0, t1 = 0;
#pragma unroll
    for (int j = 0; j < GNF_WORDS_PER_WARP; j++)
    {
        const int64_t v = warp_base + j * 32 + lane;
        const bool in = v < V && pred((int32_t)v);
        const uint32_t w = __ballot_sync(0xffffffffu, in);
        words[j] = w;
        if (in) deg_sum += ptr[v + 1] - ptr[v];
        if (warp_base + j * 32 < V)
        {
            if (lane == 0) bitmap[(warp_base >> 5) + j] = w;
            count += __popc(w);
            const int32_t base = (int32_t)(warp_base + j * 32);
            const uint32_t m0 = below_border_mask(base, b0), m1 = below_border_mask(base, b1);
            t0 += __popc(w & m0);
            t1 += __popc(w & m1 & ~m0);
        }
    }
    if (lane == 0) s_warp_count[warp] = count;
    deg_sum = warp_sum_i64(deg_sum);
    __syncthreads();
    int warp_offset = 0, cta_count = 0;
#pragma unroll
    for (int w = 0; w < GNF_THREADS / 32; w++)
    {
        if (w < warp) warp_offset += s_warp_count[w];
        cta_count += s_warp_count[w];
    }
    if (threadIdx.x == 0)
    {
        // decoupled look-back: publish this tile's aggregate, then walk predecessors until an inclusive prefix
        unsigned long long excl = 0;
        volatile unsigned long long *status = tile_status;
        if (tile == 0)
            status[0] = TILE_FLAG_PREFIX | (unsigned long long)cta_count;
        else
        {
            status[tile] = TILE_FLAG_AGGREGATE | (unsigned long long)cta_count;
            __threadfence();
            int t = tile - 1;
            for (;;)
            {
                const unsigned long long s = status[t];
                if ((s >> 62) == 0) continue; // predecessor has not published yet (it is resident: ticket order)
                excl += s & TILE_VALUE_MASK;
                if (s & TILE_FLAG_PREFIX) break;
                t--;
            }
            status[tile] = TILE_FLAG_PREFIX | (excl + (unsigned long long)cta_count);
        }
        s_prefix = excl;
    }
    if (lane == 0)
    {
        if (count) atomicAdd(&counters[G_SIZE], (unsigned long long)count);
        if (deg_sum) atomicAdd(&counters[G_NEIGHBOURS], (unsigned long long)deg_sum);
        if (t0) atomicAdd(&counters[G_TIER0], (unsigned long long)t0);
        if (t1) atomicAdd(&counters[G_TIER1], (unsigned long long)t1);
        if (count - t0 - t1) atomicAdd(&counters[G_TIER2], (unsigned long long)(count - t0 - t1));
    }
    __syncthreads();
    if (cta_count == 0) return;
    int64_t pos = (int64_t)s_prefix + warp_offset;
#pragma unroll
    for (int j = 0; j < GNF_WORDS_PER_WARP; j++)
    {
        const uint32_t w = words[j];
        if ((w >> lane) & 1u) ids[pos + __popc(w & ((1u << lane) - 1u))] = (int32_t)(warp_base + j * 32 + lane);
        pos += __popc(w);
    }
}

__global__ void frontier_single_kernel(uint32_t *bitmap, int32_t *ids, int32_t v)
{
    bitmap[v >> 5] = 1u << (v & 31);
    ids[0] = v;
}

__global__ void frontier_fill_bitmap_kernel(uint32_t *bitmap, int32_t V)
{
    const int64_t nwords = ((int64_t)V + 31) >> 5;
    for (int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; w < nwords; w += (int64_t)gridDim.x * blockDim.x)
        bitmap[w] = (w == nwords - 1 && (V & 31)) ? ((1u << (V & 31)) - 1u) : 0xffffffffu;
}

extern "C" int vglb_frontier_create(vglb_ctx *ctx, vglb_graph *g, vglb_frontier **out)
{
    return vglb_frontier_create_borrowed(ctx, g, NULL, out);
}

// `d_ids` != NULL: the id list lives in the caller's array of at least `vertices` ints (the reference frontier's own ids[],
// base_frontier.h:18 — the compaction then writes straight into the object the algorithm holds)
extern "C" int vglb_frontier_create_borrowed(vglb_ctx *ctx, vglb_graph *g, int32_t *d_ids, vglb_frontier **out)
{
    VGLB_REQUIRE(ctx != NULL && g != NULL && out != NULL, "vglb_frontier_create: NULL argument");
    CUDA_TRY(cudaSetDevice(ctx->device));
    vglb_frontier *f = (vglb_frontier *)calloc(1, sizeof(vglb_frontier));
    if (!f) return VGLB_ENOMEM;
    f->g = g;
    const size_t words = ((size_t)g->V + 31) / 32 + 32;
    const size_t tiles = ((size_t)g->V + GNF_TILE - 1) / GNF_TILE + 1;
    cudaError_t e = vglb_dev_alloc(&f->d_bitmap, words * 4);
    if (d_ids)
    {
        f->d_ids = d_ids;
        f->borrowed_ids = 1;
    }
    else if (e == cudaSuccess) e = vglb_dev_alloc(&f->d_ids, ((size_t)g->V + 32) * 4);
    if (e == cudaSuccess) e = vglb_dev_alloc(&f->d_tile_status, (tiles + G_COUNT) * 8);
    if (e != cudaSuccess)
    {
        cudaGetLastError();
        vglb_dev_free(f->d_bitmap); if (!f->borrowed_ids) vglb_dev_free(f->d_ids); vglb_dev_free(f->d_tile_status);
        free(f);
        vglb_set_error("vglb_frontier_create: cudaMalloc failed: %s", cudaGetErrorString(e));
        return VGLB_ENOMEM;
    }
    f->tiles = (int64_t)tiles;
    CUDA_TRY(cudaMemsetAsync(f->d_bitmap, 0, words * 4, ctx->stream));
    f->sparsity_type = VGLB_FRONTIER_SPARSE; // an empty frontier (FrontierVectorCSR ctor + clear())
    *out = f;
    return VGLB_OK;
}

extern "C" int vglb_frontier_destroy(vglb_ctx *ctx, vglb_frontier *f)
{
    VGLB_REQUIRE(ctx != NULL, "vglb_frontier_destroy: ctx is NULL");
    if (!f) return VGLB_OK;
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    vglb_dev_free(f->d_bitmap); if (!f->borrowed_ids) vglb_dev_free(f->d_ids); vglb_dev_free(f->d_tile_status);
    free(f);
    return VGLB_OK;
}

static void frontier_set_tiers_all(vglb_frontier *f)
{
    const vglb_graph *g = f->g;
    f->tier_size[0] = g->tier_border[0];
    f->tier_size[1] = g->tier_border[1] - g->tier_border[0];
    f->tier_size[2] = g->V - g->tier_border[1];
}

// FrontierVectorCSR::set_all_active (modification.hpp:5-29)
extern "C" int vglb_frontier_set_all_active(vglb_ctx *ctx, vglb_frontier *f)
{
    VGLB_REQUIRE(ctx != NULL && f != NULL, "vglb_frontier_set_all_active: NULL argument");
    f->sparsity_type = VGLB_FRONTIER_ALL_ACTIVE;
    f->size = f->g->V;
    f->neighbours = f->g->E;
    frontier_set_tiers_all(f);
    frontier_fill_bitmap_kernel<<<ctx->sm_count * 4, 256, 0, ctx->stream>>>(f->d_bitmap, f->g->V);
    KERNEL_TRY();
    ctx->launches++;
    return VGLB_OK;
}

// FrontierVectorCSR::clear
extern "C" int vglb_frontier_clear(vglb_ctx *ctx, vglb_frontier *f)
{
    VGLB_REQUIRE(ctx != NULL && f != NULL, "vglb_frontier_clear: NULL argument");
    f->sparsity_type = VGLB_FRONTIER_SPARSE;
    f->size = 0;
    f->neighbours = 0;
    f->tier_size[0] = f->tier_size[1] = f->tier_size[2] = 0;
    CUDA_TRY(cudaMemsetAsync(f->d_bitmap, 0, (((size_t)f->g->V + 31) / 32) * 4, ctx->stream));
    return VGLB_OK;
}

// FrontierVectorCSR::add_vertex (modification.hpp:31-84): only on an empty frontier, like the reference
extern "C" int vglb_frontier_add_vertex(vglb_ctx *ctx, vglb_frontier *f, int32_t v)
{
    VGLB_REQUIRE(ctx != NULL && f != NULL, "vglb_frontier_add_vertex: NULL argument");
    VGLB_REQUIRE(v >= 0 && v < f->g->V, "vglb_frontier_add_vertex: vertex out of range");
    if (f->size > 0)
    {
        vglb_set_error("VGL error! can not add vertex to non-empty frontier"); // modification.hpp:33-36
        return VGLB_EINVAL;
    }
    const vglb_graph *g = f->g;
    frontier_single_kernel<<<1, 1, 0, ctx->stream>>>(f->d_bitmap, f->d_ids, v);
    KERNEL_TRY();
    ctx->launches++;
    int64_t pp[2];
    CUDA_TRY(cudaMemcpyAsync(pp, g->d_out_ptr + v, 16, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    f->sparsity_type = VGLB_FRONTIER_SPARSE;
    f->size = 1;
    f->neighbours = pp[1] - pp[0];
    const int tier = v < g->tier_border[0] ? 0 : (v < g->tier_border[1] ? 1 : 2);
    f->tier_size[0] = f->tier_size[1] = f->tier_size[2] = 0;
    f->tier_size[tier] = 1;
    return VGLB_OK;
}

// FrontierVectorCSR::add_group_of_vertices (modification.hpp:88-145): an explicit id list becomes the frontier. The reference
// sorts the list ascending first (Sorter::sort) — which is what makes the degree tiers contiguous prefixes; here the list must
// arrive ascending and duplicate-free (checked on the device). Only on an empty frontier, like the reference.
__global__ void frontier_set_ids_kernel(const int32_t *__restrict__ ids, int32_t n, int32_t V, const int64_t *__restrict__ ptr, int32_t b0,
                                        int32_t b1, uint32_t *__restrict__ bitmap, unsigned long long *__restrict__ counters)
{
    long long deg = 0;
    int t0 = 0, t1 = 0, bad = 0;
    for (int32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    {
        const int32_t v = ids[i];
        if (v < 0 || v >= V || (i > 0 && ids[i - 1] >= v))
        {
            bad = 1;
            continue;
        }
        atomicOr(&bitmap[v >> 5], 1u << (v & 31));
        deg += ptr[v + 1] - ptr[v];
        t0 += v < b0;
        t1 += v >= b0 && v < b1;
    }
    deg = warp_sum_i64(deg);
    t0 = (int)warp_sum_i64(t0);
    t1 = (int)warp_sum_i64(t1);
    bad = __any_sync(0xffffffffu, bad);
    if ((threadIdx.x & 31) == 0)
    {
        if (deg) atomicAdd(&counters[G_NEIGHBOURS], (unsigned long long)deg);
        if (t0) atomicAdd(&counters[G_TIER0], (unsigned long long)t0);
        if (t1) atomicAdd(&counters[G_TIER1], (unsigned long long)t1);
        if (bad) atomicAdd(&counters[G_TICKET], 1ULL);
    }
}

extern "C" int vglb_frontier_set_ids(vglb_ctx *ctx, vglb_frontier *f, const int32_t *ids, int32_t n, int ids_on_device)
{
    VGLB_REQUIRE(ctx != NULL && f != NULL && (n == 0 || ids != NULL), "vglb_frontier_set_ids: NULL argument");
    VGLB_REQUIRE(n >= 0 && n <= f->g->V, "vglb_frontier_set_ids: more ids than vertices");
    if (f->size > 0)
    {
        vglb_set_error("VGL ERROR: can not add vertices to non-empty frontier"); // modification.hpp:90-93
        return VGLB_EINVAL;
    }
    const vglb_graph *g = f->g;
    CUDA_TRY(cudaSetDevice(ctx->device));
    if (n > 0 && ids != f->d_ids)
        CUDA_TRY(cudaMemcpyAsync(f->d_ids, ids, (size_t)n * 4, ids_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, ctx->stream));
    unsigned long long *counters = (unsigned long long *)f->d_tile_status;
    CUDA_TRY(cudaMemsetAsync(counters, 0, G_COUNT * 8, ctx->stream));
    CUDA_TRY(cudaMemsetAsync(f->d_bitmap, 0, (((size_t)g->V + 31) / 32) * 4, ctx->stream));
    if (n > 0)
    {
        const int blocks = (int)(ceil_div64(n, 256) < ctx->sm_count * 8 ? ceil_div64(n, 256) : ctx->sm_count * 8);
        frontier_set_ids_kernel<<<blocks, 256, 0, ctx->stream>>>(f->d_ids, n, g->V, g->d_out_ptr, g->tier_border[0], g->tier_border[1],
                                                                f->d_bitmap, counters);
        KERNEL_TRY();
        ctx->launches++;
    }
    unsigned long long *h = (unsigned long long *)ctx->h_counters;
    CUDA_TRY(cudaMemcpyAsync(h, counters, G_COUNT * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    if (h[G_TICKET])
    {
        CUDA_TRY(cudaMemsetAsync(f->d_bitmap, 0, (((size_t)g->V + 31) / 32) * 4, ctx->stream));
        vglb_set_error("vglb_frontier_set_ids: ids must be ascending, distinct and in [0, V)");
        return VGLB_EINVAL;
    }
    f->size = n;
    f->neighbours = (int64_t)h[G_NEIGHBOURS];
    f->tier_size[0] = (int32_t)h[G_TIER0];
    f->tier_size[1] = (int32_t)h[G_TIER1];
    f->tier_size[2] = n - f->tier_size[0] - f->tier_size[1];
    f->sparsity_type = n == g->V ? VGLB_FRONTIER_ALL_ACTIVE : VGLB_FRONTIER_SPARSE;
    return VGLB_OK;
}

extern "C" int vglb_frontier_get_info(vglb_ctx *ctx, vglb_frontier *f, vglb_frontier_info *info)
{
    VGLB_REQUIRE(ctx != NULL && f != NULL && info != NULL, "vglb_frontier_get_info: NULL argument");
    memset(info, 0, sizeof(*info));
    info->sparsity_type = f->sparsity_type;
    info->size = f->size;
    info->neighbours = f->neighbours;
    for (int t = 0; t < 3; t++) info->tier_size[t] = f->tier_size[t];
    info->d_ids = f->d_ids;
    info->d_bitmap = f->d_bitmap;
    return VGLB_OK;
}

template <class Pred>
static int gnf_run(vglb_ctx *ctx, vglb_frontier *f, Pred pred)
{
    const vglb_graph *g = f->g;
    CUDA_TRY(cudaSetDevice(ctx->device));
    unsigned long long *counters = (unsigned long long *)f->d_tile_status;
    unsigned long long *status = counters + G_COUNT;
    const int64_t tiles = ceil_div64(g->V, GNF_TILE);
    CUDA_TRY(cudaMemsetAsync(f->d_tile_status, 0, (size_t)(tiles + G_COUNT) * 8, ctx->stream));
    gnf_compact_kernel<Pred><<<(unsigned)tiles, GNF_THREADS, 0, ctx->stream>>>(
        pred, g->d_out_ptr, g->V, g->tier_border[0], g->tier_border[1], f->d_bitmap, f->d_ids, status, counters);
    KERNEL_TRY();
    ctx->launches++;
    unsigned long long *h = (unsigned long long *)ctx->h_counters;
    int rc_fetch = vglb_counters_fetch(ctx, counters, G_COUNT);
    if (rc_fetch != VGLB_OK) return rc_fetch;
    f->size = (int32_t)h[G_SIZE];
    f->neighbours = (int64_t)h[G_NEIGHBOURS];
    f->tier_size[0] = (int32_t)h[G_TIER0];
    f->tier_size[1] = (int32_t)h[G_TIER1];
    f->tier_size[2] = (int32_t)h[G_TIER2];
    // multicore/generate_new_frontier.hpp:67-91
    if (f->size == g->V) f->sparsity_type = VGLB_FRONTIER_ALL_ACTIVE;
    else if ((double)f->size / (double)g->V > 0.7) f->sparsity_type = VGLB_FRONTIER_DENSE;
    else f->sparsity_type = VGLB_FRONTIER_SPARSE;
    return VGLB_OK;
}

extern "C" int vglb_gnf_from_flags(vglb_ctx *ctx, vglb_frontier *f, const int32_t *d_flags)
{
    VGLB_REQUIRE(ctx != NULL && f != NULL && d_flags != NULL, "vglb_gnf_from_flags: NULL argument");
    PredFlags p{d_flags};
    return gnf_run(ctx, f, p);
}

extern "C" int vglb_gnf_from_bitmap(vglb_ctx *ctx, vglb_frontier *f, const uint32_t *d_bits)
{
    VGLB_REQUIRE(ctx != NULL && f != NULL && d_bits != NULL, "vglb_gnf_from_bitmap: NULL argument");
    VGLB_REQUIRE(d_bits != (const uint32_t *)f->d_bitmap, "vglb_gnf_from_bitmap: the input must not be the frontier's own bitmap");
    PredBitmap p{d_bits};
    return gnf_run(ctx, f, p);
}

extern "C" int vglb_gnf_eq_i32(vglb_ctx *ctx, vglb_frontier *f, const int32_t *d_values, int32_t key)
{
    VGLB_REQUIRE(ctx != NULL && f != NULL && d_values != NULL, "vglb_gnf_eq_i32: NULL argument");
    PredEqI32 p{d_values, key};
    return gnf_run(ctx, f, p);
}

extern "C" int vglb_gnf_ne_u32(vglb_ctx *ctx, vglb_frontier *f, const uint32_t *d_a, const uint32_t *d_b)
{
    VGLB_REQUIRE(ctx != NULL && f != NULL && d_a != NULL && d_b != NULL, "vglb_gnf_ne_u32: NULL argument");
    PredNeU32 p{d_a, d_b};
    return gnf_run(ctx, f, p);
}

// ---- reduce over the frontier: one pass, block reduction, one atomic per CTA (common/reduce.hpp:4-67) -----------------
// ALL_ACTIVE / DENSE walk the vertex range coalesced (DENSE tests the bitmap word), SPARSE walks the id list.

enum { RED_SUM_I32 = 0, RED_SUM_F32 = 1, RED_MAX_I32 = 2 };

template <int OP>
__global__ void __launch_bounds__(256)
frontier_reduce_kernel(const void *__restrict__ values, int32_t n, const int32_t *__restrict__ ids,
                       const uint32_t *__restrict__ bitmap, unsigned long long *out)
{
    __shared__ double s_f[8];
    __shared__ long long s_i[8];
    long long acc_i = OP == RED_MAX_I32 ? (long long)INT32_MIN : 0;
    double acc_f = 0.0;
    for (int32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    {
        const int32_t v = ids ? ids[i] : i;
        if (bitmap && !bm_test(bitmap, v)) continue;
        if (OP == RED_SUM_I32) acc_i += ((const int32_t *)values)[v];
        else if (OP == RED_MAX_I32) acc_i = max(acc_i, (long long)((const int32_t *)values)[v]);
        else acc_f += (double)((const float *)values)[v];
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (OP == RED_SUM_F32)
    {
        acc_f = warp_sum_f64(acc_f);
        if (lane == 0) s_f[warp] = acc_f;
    }
    else
    {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1)
        {
            const long long other = __shfl_xor_sync(0xffffffffu, acc_i, o);
            acc_i = OP == RED_MAX_I32 ? max(acc_i, other) : acc_i + other;
        }
        if (lane == 0) s_i[warp] = acc_i;
    }
    __syncthreads();
    if (threadIdx.x == 0)
    {
        if (OP == RED_SUM_F32)
        {
            double t = 0.0;
            for (int w = 0; w < 8; w++) t += s_f[w];
            atomicAdd((double *)out, t);
        }
        else if (OP == RED_SUM_I32)
        {
            long long t = 0;
            for (int w = 0; w < 8; w++) t += s_i[w];
            atomicAdd(out, (unsigned long long)t);
        }
        else
        {
            long long t = (long long)INT32_MIN;
            for (int w = 0; w < 8; w++) t = max(t, s_i[w]);
            atomicMax((long long *)out, t);
        }
    }
}

template <int OP>
static int reduce_run(vglb_ctx *ctx, vglb_frontier *f, const void *d_values, void *h_out8)
{
    CUDA_TRY(cudaSetDevice(ctx->device));
    unsigned long long *d_out = (unsigned long long *)ctx->d_counters + 32;
    long long init = OP == RED_MAX_I32 ? (long long)INT32_MIN : 0;
    double initf = 0.0;
    CUDA_TRY(cudaMemcpyAsync(d_out, OP == RED_SUM_F32 ? (void *)&initf : (void *)&init, 8, cudaMemcpyHostToDevice, ctx->stream));
    const bool sparse = f->sparsity_type == VGLB_FRONTIER_SPARSE;
    const int32_t n = sparse ? f->size : f->g->V;
    if (n > 0)
    {
        const int grid = (int)min((int64_t)ctx->sm_count * 8, ceil_div64(n, 256));
        frontier_reduce_kernel<OP><<<grid, 256, 0, ctx->stream>>>(
            d_values, n, sparse ? f->d_ids : NULL, f->sparsity_type == VGLB_FRONTIER_DENSE ? f->d_bitmap : NULL, d_out);
        KERNEL_TRY();
        ctx->launches++;
    }
    CUDA_TRY(cudaMemcpyAsync(h_out8, d_out, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return VGLB_OK;
}

extern "C" int vglb_reduce_sum_i32(vglb_ctx *ctx, vglb_frontier *f, const int32_t *d_values, int64_t *out)
{
    VGLB_REQUIRE(ctx != NULL && f != NULL && d_values != NULL && out != NULL, "vglb_reduce_sum_i32: NULL argument");
    return reduce_run<RED_SUM_I32>(ctx, f, d_values, out);
}

extern "C" int vglb_reduce_sum_f32(vglb_ctx *ctx, vglb_frontier *f, const float *d_values, double *out)
{
    VGLB_REQUIRE(ctx != NULL && f != NULL && d_values != NULL && out != NULL, "vglb_reduce_sum_f32: NULL argument");
    return reduce_run<RED_SUM_F32>(ctx, f, d_values, out);
}

extern "C" int vglb_reduce_max_i32(vglb_ctx *ctx, vglb_frontier *f, const int32_t *d_values, int32_t *out)
{
    VGLB_REQUIRE(ctx != NULL && f != NULL && d_values != NULL && out != NULL, "vglb_reduce_max_i32: NULL argument");
    long long r = 0;
    int rc = reduce_run<RED_MAX_I32>(ctx, f, d_values, &r);
    if (rc == VGLB_OK) *out = (int32_t)r;
    return rc;
}

// ---- the per-level counters of the partitioned BFS / SSSP drivers, staged for their allreduce -------------------------
__global__ void stage_counters_kernel(unsigned long long *c)
{
    if (threadIdx.x < C_COUNT) c[C_COUNT + threadIdx.x] = c[threadIdx.x];
    if (threadIdx.x == 0) c[2 * C_COUNT] = c[C_MF];
}

int vglb_stage_counters(vglb_ctx *ctx)
{
    stage_counters_kernel<<<1, 32, 0, ctx->stream>>>((unsigned long long *)ctx->d_counters);
    KERNEL_TRY();
    ctx->launches++;
    return VGLB_OK;
}
