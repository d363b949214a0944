// graph_build.cu — device VectCSR layout: VGL_Graph::import -> VectorCSRGraph::import rebuilt on the GPU.
//
// Reference behaviour reproduced bit-for-bit (vgl_datastructures/graphs/undirected_containers/vect_csr/import.hpp:257-337):
//   extract_connection_count (:5-57)       -> out-degree histogram with atomics
//   sort_vertices_by_degree (:61-99)       -> STABLE sort of ids by degree descending (sorter.h:55-92 std::stable_sort)
//                                             == stable LSD radix sort of (~degree) with ascending ids as payload
//   renumber_vertices (edges_container.h:163-213) + preprocess_into_csr_based (:101-161)
//                                          -> STABLE sort of edges by new src id, payload = input edge index
//   construct_CSR (import.hpp:103-153)     -> row pointers = exclusive scan of sorted degrees
//   estimate_thresholds (nec_api.hpp:5-50) -> tier borders (contiguous id ranges because ids are degree-sorted)
// The sort/scan primitives are CUB's (toolkit library) — graph construction is setup, outside every timed region
// (reference: bfs.hpp:76-79 starts its timer after import); the hot path kernels are hand-written (pagerank.cu, ...).
// B200 layout choices that differ from the reference: the incoming CSR is built on the SAME (SCATTER) numbering as
// the outgoing one so top-down and bottom-up BFS share one levels array / visited bitmap (SURVEY §7.1), and no
// VectorExtension (ELL copy of the tail) is kept — sub-warp row groups read the CSR tail coalesced instead.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <stdlib.h>

#include "common.cuh"

namespace
{

__global__ void degree_histogram_kernel(const int32_t *__restrict__ ids, int64_t n, int32_t V, int32_t *__restrict__ deg,
                                        int *__restrict__ bad)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride)
    {
        int32_t v = ids[i];
        if (v < 0 || v >= V) { *bad = 1; continue; }
        atomicAdd(&deg[v], 1);
    }
}

__global__ void id_range_check_kernel(const int32_t *__restrict__ ids, int64_t n, int64_t limit, int *__restrict__ bad)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride)
        if (ids[i] < 0 || ids[i] >= limit) *bad = 1;
}

__global__ void degree_sort_keys_kernel(const int32_t *__restrict__ deg, int32_t V, uint32_t *__restrict__ keys,
                                        uint32_t *__restrict__ ids)
{
    int32_t v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v < V)
    {
        keys[v] = ~(uint32_t)deg[v]; // ascending ~deg == descending deg; stable => ascending original id in ties
        ids[v] = (uint32_t)v;
    }
}

__global__ void conversions_kernel(const uint32_t *__restrict__ sorted_ids, const int32_t *__restrict__ deg, int32_t V,
                                   int32_t *__restrict__ fwd, int32_t *__restrict__ bwd, int64_t *__restrict__ deg_sorted)
{
    int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < V)
    {
        int32_t orig = (int32_t)sorted_ids[i];
        bwd[i] = orig;
        fwd[orig] = i;
        deg_sorted[i] = deg[orig];
    }
    if (i == V) deg_sorted[V] = 0;
}

__global__ void edge_keys_kernel(const int32_t *__restrict__ key_ids, const int32_t *__restrict__ fwd, int64_t E,
                                 uint32_t *__restrict__ keys, uint32_t *__restrict__ vals)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; i < E; i += stride)
    {
        keys[i] = (uint32_t)fwd[key_ids[i]];
        vals[i] = (uint32_t)i;
    }
}

__global__ void gather_adj_kernel(const uint32_t *__restrict__ order, const int32_t *__restrict__ other_ids,
                                  const int32_t *__restrict__ fwd, int64_t E, int32_t *__restrict__ adj,
                                  int64_t *__restrict__ edge_order)
{
    int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; p < E; p += stride)
    {
        uint32_t e = order[p];
        adj[p] = fwd[other_ids[e]];
        if (edge_order) edge_order[p] = (int64_t)e;
    }
}

// in-degree without self loops of the rows [row0, row1) of an out-CSR (one upload chunk of vglb_graph_from_csr).
// The CSR comes from the caller (or from a file): row ranges are clamped to [e_lo, e_hi) — the part of the adjacency
// this chunk has uploaded — and ids outside [0, V) raise *bad instead of being used as an index.
__global__ void indegree_noloops_rows_kernel(const int64_t *__restrict__ ptr, const int32_t *__restrict__ adj, int32_t row0, int32_t row1,
                                             int64_t e_lo, int64_t e_hi, int32_t V, int32_t *__restrict__ indeg, int *__restrict__ bad)
{
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t v = row0 + warp; v < row1; v += nwarps)
    {
        int64_t s = ptr[v], e = ptr[v + 1];
        if (s < e_lo || e > e_hi || s > e)
        {
            if (lane == 0) *bad = 1;
            continue;
        }
        for (int64_t p = s + lane; p < e; p += 32)
        {
            const int32_t d = adj[p];
            if ((uint32_t)d >= (uint32_t)V) *bad = 1;
            else if (d != (int32_t)v) atomicAdd(&indeg[d], 1);
        }
    }
}

// The same for a chunk of rows with fewer than 32 edges each (the tail of the degree-sorted CSR, half of it without edges):
// one lane per row — with a warp per row the chunk is a chain of dependent loads per row, 1.6 ms for the 15.7 M tail rows of
// the BASELINE PageRank graph, all of it after the upload has finished.
__global__ void indegree_noloops_short_rows_kernel(const int64_t *__restrict__ ptr, const int32_t *__restrict__ adj, int32_t row0, int32_t row1,
                                                   int64_t e_lo, int64_t e_hi, int32_t V, int32_t *__restrict__ indeg, int *__restrict__ bad)
{
    for (int64_t v = row0 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < row1; v += (int64_t)gridDim.x * blockDim.x)
    {
        const int64_t s = ptr[v], e = ptr[v + 1];
        if (s < e_lo || e > e_hi || s > e)
        {
            *bad = 1;
            continue;
        }
        for (int64_t p = s; p < e; p++)
        {
            const int32_t d = adj[p];
            if ((uint32_t)d >= (uint32_t)V) *bad = 1;
            else if (d != (int32_t)v) atomicAdd(&indeg[d], 1);
        }
    }
}

// row pointers of a caller-supplied CSR: ptr[0] == 0, non-decreasing, ptr[rows] == E
__global__ void csr_ptr_check_kernel(const int64_t *__restrict__ ptr, int32_t rows, int64_t E, int *__restrict__ bad)
{
    const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (v == 0 && (ptr[0] != 0 || ptr[rows] != E)) *bad = 1;
    if (v < rows && ptr[v] > ptr[v + 1]) *bad = 1;
}

// map supplied by the caller (ORIGINAL -> sorted, or ORIGINAL -> column of a partitioned graph): bwd was filled with -1; every
// vertex must go to a distinct slot in [0, limit)
__global__ void invert_map_checked_kernel(const int32_t *__restrict__ fwd, int32_t n, int64_t limit, int32_t *__restrict__ bwd,
                                          int *__restrict__ bad)
{
    int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int32_t f = fwd[i];
    if (f < 0 || f >= limit) { *bad = 1; return; }
    if (atomicExch(&bwd[f], i) != -1) *bad = 1;
}

// in-degree (on the SCATTER numbering) as int64 for the scan
__global__ void indegree_sorted_kernel(const int32_t *__restrict__ dst, const int32_t *__restrict__ fwd, int64_t E,
                                       unsigned long long *__restrict__ indeg)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; i < E; i += stride) atomicAdd(&indeg[fwd[dst[i]]], 1ULL);
}

__global__ void iota_kernel(int32_t *a, int32_t n)
{
    int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) a[i] = i;
}

// tier borders: border[t] = first id whose degree < tier_degree[t]; also checks the rows are degree-sorted.
__global__ void tier_border_kernel(const int64_t *__restrict__ ptr, int32_t V, int32_t *__restrict__ out /*[NUM_TIERS+2]*/)
{
    int32_t v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= V) return;
    const int64_t p0 = ptr[v], p1 = ptr[v + 1];
    const int64_t d = p1 - p0;
    const int64_t dn = (v == V - 1) ? -1 : ptr[v + 2] - p1;
    if (v == 0) out[VGLB_NUM_TIERS] = (int32_t)(d > 0x7fffffff ? 0x7fffffff : d); // max degree
    if (dn > d) out[VGLB_NUM_TIERS + 1] = 1;                                       // not sorted
#pragma unroll
    for (int t = 0; t < VGLB_NUM_TIERS; t++)
    {
        const int64_t T = vglb_tier_degree(t);
        if (d >= T && dn < T) out[t] = v + 1;
    }
}

} // namespace


void vglb_graph_set_unpartitioned(vglb_graph *g)
{
    g->comm = NULL;
    g->part_rank = 0;
    g->part_world = 1;
    g->vp = g->V;
    g->V_orig = g->V;
    g->cols = g->V;
    g->E_global = g->E;
    g->col_of_row0 = 0;
}

int vglb_graph_compute_tiers(vglb_ctx *ctx, vglb_graph *g)
{
    int32_t *d_out = (int32_t *)(ctx->d_counters + CTR_SCRATCH_I32);
    CUDA_TRY(cudaMemsetAsync(d_out, 0, (VGLB_NUM_TIERS + 2) * sizeof(int32_t), ctx->stream));
    if (g->V > 0)
    {
        tier_border_kernel<<<(unsigned)ceil_div64(g->V, 256), 256, 0, ctx->stream>>>(g->d_out_ptr, g->V, d_out);
        KERNEL_TRY();
    }
    int32_t h[VGLB_NUM_TIERS + 2];
    CUDA_TRY(cudaMemcpyAsync(h, d_out, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    CUDA_TRY(cudaMemsetAsync(d_out, 0, (VGLB_NUM_TIERS + 2) * sizeof(int32_t), ctx->stream));
    if (h[VGLB_NUM_TIERS + 1])
    {
        vglb_set_error("graph rows are not sorted by degree descending: not a VectCSR layout");
        return VGLB_EUNSORTED;
    }
    for (int t = 0; t < VGLB_NUM_TIERS; t++)
    {
        g->tier_degree[t] = vglb_tier_degree(t);
        g->tier_border[t] = h[t];
    }
    // borders must be monotone even when a tier is empty
    for (int t = 1; t < VGLB_NUM_TIERS; t++)
        if (g->tier_border[t] < g->tier_border[t - 1]) g->tier_border[t] = g->tier_border[t - 1];
    g->tier_border[VGLB_NUM_TIERS - 1] = g->V;
    g->max_degree = h[VGLB_NUM_TIERS];
    return VGLB_OK;
}

// close this process's mappings of the peers' buffers (CUDA IPC)
static void graph_close_peer_mappings(vglb_graph *g)
{
    for (int b = 0; b < 2; b++)
        for (int p = 0; p < 8; p++)
            if (g->d_pr_peer[b][p])
            {
                cudaIpcCloseMemHandle(g->d_pr_peer[b][p]);
                g->d_pr_peer[b][p] = NULL;
            }
    for (int p = 0; p < 8; p++)
        if (g->d_vec_peer[p] && p != g->part_rank)
        {
            cudaIpcCloseMemHandle(g->d_vec_peer[p]);
            g->d_vec_peer[p] = NULL;
        }
}

void vglb_graph_free_fields(vglb_graph *g)
{
    graph_close_peer_mappings(g); // importers close before any exporter frees (vglb_graph_free orders the ranks)
    vglb_dev_free(g->d_part_bm[0]); vglb_dev_free(g->d_part_bm[1]); vglb_dev_free(g->d_part_bm[2]); vglb_dev_free(g->d_part_stage);
    vglb_dev_free(g->d_part_vec); vglb_dev_free(g->d_part_prev); vglb_dev_free(g->d_part_lists);
    if (!g->borrowed_csr)
    {
        vglb_dev_free(g->d_out_ptr);
        vglb_dev_free(g->d_out_adj);
    }
    vglb_dev_free(g->d_in_ptr); vglb_dev_free(g->d_in_adj);
    vglb_dev_free(g->d_fwd); vglb_dev_free(g->d_bwd); vglb_dev_free(g->d_edge_order); vglb_dev_free(g->d_in_to_out_pos);
    vglb_dev_free(g->d_indeg_noloops); vglb_dev_free(g->d_pr_inv); vglb_dev_free(g->d_pr_contrib[0]); vglb_dev_free(g->d_pr_contrib[1]); vglb_dev_free(g->d_pr_dangling); vglb_dev_free(g->d_pr_tasks); vglb_dev_free(g->d_pr_piece_partial); vglb_dev_free(g->d_pr_piece_count); vglb_dev_free(g->d_pr_ve_adj); vglb_dev_free(g->d_pr_ve_ptr);
    vglb_pr_bins_free(g);
    vglb_dev_free(g->d_visited); vglb_dev_free(g->d_front_bm[0]); vglb_dev_free(g->d_front_bm[1]);
    vglb_dev_free(g->d_queue[0]); vglb_dev_free(g->d_queue[1]); vglb_dev_free(g->d_scratch_i32);
}

extern "C" int vglb_graph_free(vglb_ctx *ctx, vglb_graph *g)
{
    VGLB_REQUIRE(ctx != NULL, "vglb_graph_free: ctx is NULL");
    if (!g) return VGLB_OK;
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    if (g->ipc_exported && g->comm && g->comm->nccl && g->part_world > 1)
    {
        // CUDA leaves cudaFree of an exported buffer undefined while an importer still maps it: every rank first closes
        // its own mappings, then all ranks meet (one allreduce on the graph's communicator), and only then does anybody
        // free what it exported. vglb_graph_free is therefore a collective on such a graph, and the graph must be freed
        // before its communicator is destroyed.
        graph_close_peer_mappings(g);
        int rc = vglb_comm_barrier(g->comm);
        if (rc != VGLB_OK) return rc;
    }
    vglb_graph_free_fields(g);
    cudaGetLastError();
    free(g);
    return VGLB_OK;
}

// outgoing direction: stable sort of the edges by fwd[src]; adjacency = fwd[dst] in that order. When d_row_of_pos is
// non-NULL it receives the (ascending) row id of every CSR position, which the incoming build reuses.
static int build_outgoing(vglb_ctx *ctx, int32_t V, int64_t E, const int32_t *d_src, const int32_t *d_dst,
                          const int32_t *d_fwd, int32_t *d_adj, int64_t *d_edge_order, uint32_t *d_row_of_pos)
{
    if (E == 0) return VGLB_OK;
    const size_t eb = (size_t)E * sizeof(uint32_t);
    dev_ptr<uint32_t> k0, k1, v0, v1;
    dev_ptr<void> tmp;
    CUDA_TRY(vglb_dev_alloc(k0, eb)); CUDA_TRY(vglb_dev_alloc(k1, eb));
    CUDA_TRY(vglb_dev_alloc(v0, eb)); CUDA_TRY(vglb_dev_alloc(v1, eb));
    const int grid = ctx->sm_count * 16;
    edge_keys_kernel<<<grid, 256, 0, ctx->stream>>>(d_src, d_fwd, E, k0.get(), v0.get());
    KERNEL_TRY();
    cub::DoubleBuffer<uint32_t> keys(k0.get(), k1.get()), vals(v0.get(), v1.get());
    CUDA_TRY(vglb_cub(tmp, [&](void *t, size_t &bytes) {
        return cub::DeviceRadixSort::SortPairs(t, bytes, keys, vals, E, 0, vglb_key_bits(V), ctx->stream);
    }));
    gather_adj_kernel<<<grid, 256, 0, ctx->stream>>>(vals.Current(), d_dst, d_fwd, E, d_adj, d_edge_order);
    KERNEL_TRY();
    if (d_row_of_pos)
        CUDA_TRY(cudaMemcpyAsync(d_row_of_pos, keys.Current(), eb, cudaMemcpyDeviceToDevice, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return VGLB_OK;
}

// incoming direction on the SAME numbering: stable sort of the out-CSR positions by destination. Because the
// positions are already ordered by source id, every in-row lists its sources in ascending id = descending out-degree
// (hubs first), which is what makes the bottom-up early exit short. d_row_of_pos is consumed (becomes in_adj).
static int build_incoming(vglb_ctx *ctx, int32_t V, int64_t E, const int32_t *d_out_adj, uint32_t *d_row_of_pos,
                          int32_t *d_in_adj)
{
    if (E == 0) return VGLB_OK;
    const size_t eb = (size_t)E * sizeof(uint32_t);
    dev_ptr<uint32_t> k0, k1, v1;
    dev_ptr<void> tmp;
    CUDA_TRY(vglb_dev_alloc(k0, eb)); CUDA_TRY(vglb_dev_alloc(k1, eb)); CUDA_TRY(vglb_dev_alloc(v1, eb));
    CUDA_TRY(cudaMemcpyAsync(k0.get(), d_out_adj, eb, cudaMemcpyDeviceToDevice, ctx->stream));
    cub::DoubleBuffer<uint32_t> keys(k0.get(), k1.get()), vals(d_row_of_pos, v1.get());
    CUDA_TRY(vglb_cub(tmp, [&](void *t, size_t &bytes) {
        return cub::DeviceRadixSort::SortPairs(t, bytes, keys, vals, E, 0, vglb_key_bits(V), ctx->stream);
    }));
    CUDA_TRY(cudaMemcpyAsync(d_in_adj, vals.Current(), eb, cudaMemcpyDeviceToDevice, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return VGLB_OK;
}

int vglb_degree_order(vglb_ctx *ctx, const int32_t *d_deg, int32_t V, DegreeOrder &order)
{
    for (auto *p : {&order.keys[0], &order.keys[1], &order.ids[0], &order.ids[1]}) CUDA_TRY(vglb_dev_alloc(*p, (size_t)V * 4));
    degree_sort_keys_kernel<<<(unsigned)ceil_div64(V, 256), 256, 0, ctx->stream>>>(d_deg, V, order.keys[0].get(), order.ids[0].get());
    KERNEL_TRY();
    cub::DoubleBuffer<uint32_t> keys(order.keys[0].get(), order.keys[1].get()), vals(order.ids[0].get(), order.ids[1].get());
    CUDA_TRY(vglb_cub(order.tmp, [&](void *t, size_t &bytes) {
        return cub::DeviceRadixSort::SortPairs(t, bytes, keys, vals, V, 0, 32, ctx->stream);
    }));
    order.sorted = vals.Current();
    return VGLB_OK;
}

int vglb_csr_validate_device(vglb_ctx *ctx, const int64_t *d_ptr, int32_t rows, int64_t E, const int32_t *d_adj, int64_t id_limit)
{
    int *d_bad = (int *)(ctx->d_counters + CTR_BAD);
    csr_ptr_check_kernel<<<(unsigned)ceil_div64((int64_t)rows + 1, 256), 256, 0, ctx->stream>>>(d_ptr, rows, E, d_bad);
    KERNEL_TRY();
    if (E > 0)
    {
        id_range_check_kernel<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(d_adj, E, id_limit, d_bad);
        KERNEL_TRY();
    }
    return VGLB_OK;
}

int vglb_invert_map_checked(vglb_ctx *ctx, const int32_t *d_fwd, int32_t n, int64_t limit, int32_t *d_bwd)
{
    invert_map_checked_kernel<<<(unsigned)ceil_div64(n, 256), 256, 0, ctx->stream>>>(d_fwd, n, limit, d_bwd,
                                                                                     (int *)(ctx->d_counters + CTR_BAD));
    KERNEL_TRY();
    return VGLB_OK;
}

extern "C" int vglb_graph_from_edges(vglb_ctx *ctx, int32_t V, int64_t E, const int32_t *src, const int32_t *dst,
                                     int src_on_device, int flags, vglb_graph **out_graph)
{
    VGLB_REQUIRE(ctx != NULL && out_graph != NULL, "vglb_graph_from_edges: NULL argument");
    VGLB_REQUIRE(V > 0 && E >= 0 && E < 0xFFFFFFFFLL, "vglb_graph_from_edges: need V > 0 and 0 <= E < 2^32-1 per device");
    VGLB_REQUIRE(E == 0 || (src != NULL && dst != NULL), "vglb_graph_from_edges: NULL edge arrays");
    CUDA_TRY(cudaSetDevice(ctx->device));
    graph_ptr owner = vglb_graph_new();
    if (!owner) return VGLB_ENOMEM;
    vglb_graph *g = owner.get();
    g->V = V;
    g->E = E;
    dev_ptr<int32_t> d_src_own, d_dst_own, d_deg;
    dev_ptr<int64_t> d_deg_sorted;
    dev_ptr<uint32_t> d_row_of_pos;
    dev_ptr<int> d_bad;
    const int32_t *d_src = src, *d_dst = dst;
    const size_t eb = (size_t)(E ? E : 1) * sizeof(int32_t);
    if (!src_on_device)
    {
        CUDA_TRY(vglb_dev_alloc(d_src_own, eb));
        CUDA_TRY(vglb_dev_alloc(d_dst_own, eb));
        CUDA_TRY(cudaMemcpyAsync(d_src_own.get(), src, (size_t)E * 4, cudaMemcpyHostToDevice, ctx->stream));
        CUDA_TRY(cudaMemcpyAsync(d_dst_own.get(), dst, (size_t)E * 4, cudaMemcpyHostToDevice, ctx->stream));
        d_src = d_src_own.get();
        d_dst = d_dst_own.get();
    }
    const int grid = ctx->sm_count * 16;
    const unsigned vgrid = (unsigned)ceil_div64((int64_t)V + 1, 256);

    // 1. out-degree histogram (extract_connection_count)
    CUDA_TRY(vglb_dev_alloc(d_deg, (size_t)V * 4));
    CUDA_TRY(vglb_dev_alloc(d_bad, 4));
    CUDA_TRY(cudaMemsetAsync(d_deg.get(), 0, (size_t)V * 4, ctx->stream));
    CUDA_TRY(cudaMemsetAsync(d_bad.get(), 0, 4, ctx->stream));
    if (E)
    {
        degree_histogram_kernel<<<grid, 256, 0, ctx->stream>>>(d_src, E, V, d_deg.get(), d_bad.get());
        KERNEL_TRY();
        id_range_check_kernel<<<grid, 256, 0, ctx->stream>>>(d_dst, E, V, d_bad.get());
        KERNEL_TRY();
    }
    int bad = 0;
    CUDA_TRY(cudaMemcpyAsync(&bad, d_bad.get(), 4, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    if (bad)
    {
        vglb_set_error("vglb_graph_from_edges: vertex id out of range [0, V)");
        return VGLB_EINVAL;
    }
    // 2. stable sort of vertex ids by degree descending (sort_vertices_by_degree)
    {
        DegreeOrder order;
        VGLB_TRY(vglb_degree_order(ctx, d_deg.get(), V, order));
        CUDA_TRY(vglb_dev_alloc(&g->d_fwd, (size_t)V * 4));
        CUDA_TRY(vglb_dev_alloc(&g->d_bwd, (size_t)V * 4));
        CUDA_TRY(vglb_dev_alloc(d_deg_sorted, ((size_t)V + 1) * 8));
        conversions_kernel<<<vgrid, 256, 0, ctx->stream>>>(order.sorted, d_deg.get(), V, g->d_fwd, g->d_bwd, d_deg_sorted.get());
        KERNEL_TRY();
        CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    }
    // 3. row pointers (construct_CSR)
    CUDA_TRY(vglb_dev_alloc(&g->d_out_ptr, ((size_t)V + 2) * 8));
    {
        dev_ptr<void> tmp;
        CUDA_TRY(vglb_cub(tmp, [&](void *t, size_t &bytes) {
            return cub::DeviceScan::ExclusiveSum(t, bytes, d_deg_sorted.get(), g->d_out_ptr, V + 1, ctx->stream);
        }));
        CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    }
    // 4. edges: stable sort by new src id, adjacency in new ids (renumber + preprocess_into_csr_based)
    CUDA_TRY(vglb_dev_alloc(&g->d_out_adj, eb + 16));
    if (flags & VGLB_GRAPH_WITH_EDGE_ORDER) CUDA_TRY(vglb_dev_alloc(&g->d_edge_order, (size_t)(E ? E : 1) * 8));
    if ((flags & VGLB_GRAPH_WITH_INCOMING) && E) CUDA_TRY(vglb_dev_alloc(d_row_of_pos, eb));
    VGLB_TRY(build_outgoing(ctx, V, E, d_src, d_dst, g->d_fwd, g->d_out_adj, g->d_edge_order, d_row_of_pos.get()));
    // 5. incoming CSR on the same numbering
    if (flags & VGLB_GRAPH_WITH_INCOMING)
    {
        CUDA_TRY(cudaMemsetAsync(d_deg_sorted.get(), 0, ((size_t)V + 1) * 8, ctx->stream));
        if (E)
        {
            indegree_sorted_kernel<<<grid, 256, 0, ctx->stream>>>(d_dst, g->d_fwd, E, (unsigned long long *)d_deg_sorted.get());
            KERNEL_TRY();
        }
        CUDA_TRY(vglb_dev_alloc(&g->d_in_ptr, ((size_t)V + 2) * 8));
        {
            dev_ptr<void> tmp;
            CUDA_TRY(vglb_cub(tmp, [&](void *t, size_t &bytes) {
                return cub::DeviceScan::ExclusiveSum(t, bytes, d_deg_sorted.get(), g->d_in_ptr, V + 1, ctx->stream);
            }));
            CUDA_TRY(cudaStreamSynchronize(ctx->stream));
        }
        CUDA_TRY(vglb_dev_alloc(&g->d_in_adj, eb + 16));
        VGLB_TRY(build_incoming(ctx, V, E, g->d_out_adj, d_row_of_pos.get(), g->d_in_adj));
    }
    VGLB_TRY(vglb_graph_compute_tiers(ctx, g));
    vglb_graph_set_unpartitioned(g);
    *out_graph = owner.release();
    return VGLB_OK;
}

extern "C" int vglb_set_upload_hint(vglb_ctx *ctx, int hints)
{
    VGLB_REQUIRE(ctx != NULL && (hints & ~VGLB_HINT_PAGERANK) == 0, "vglb_set_upload_hint: bad argument");
    ctx->upload_hint = hints;
    return VGLB_OK;
}

extern "C" int vglb_graph_from_csr(vglb_ctx *ctx, int32_t V, int64_t E, const int64_t *h_out_ptr,
                                   const int32_t *h_out_adj, const int32_t *h_orig_to_sorted, const int64_t *h_in_ptr,
                                   const int32_t *h_in_adj, vglb_graph **out_graph)
{
    VGLB_REQUIRE(ctx != NULL && out_graph != NULL && h_out_ptr != NULL, "vglb_graph_from_csr: NULL argument");
    VGLB_REQUIRE(V > 0 && E >= 0 && (E == 0 || h_out_adj != NULL), "vglb_graph_from_csr: bad sizes");
    VGLB_REQUIRE((h_in_ptr == NULL) == (h_in_adj == NULL) || E == 0, "vglb_graph_from_csr: incoming arrays must come together");
    CUDA_TRY(cudaSetDevice(ctx->device));
    graph_ptr owner = vglb_graph_new();
    if (!owner) return VGLB_ENOMEM;
    vglb_graph *g = owner.get();
    g->V = V;
    g->E = E;
    // The arrays come from the caller or straight from a .vgl file (vglb_graph_load_vgl): nothing below may index with
    // a value that has not been checked. Host side: the end points and every chunk border used for a copy; device side
    // (csr_ptr_check_kernel, the guarded in-degree pass, vglb_csr_validate_device, vglb_invert_map_checked): the rest.
    if (h_out_ptr[0] != 0 || h_out_ptr[V] != E || (h_in_ptr && (h_in_ptr[0] != 0 || h_in_ptr[V] != E)))
    {
        vglb_set_error("vglb_graph_from_csr: row pointers must start at 0 and end at the edge count");
        return VGLB_EINVAL;
    }
    const bool csr_trace = getenv("VGLB_CSR_TRACE") != NULL; // developer aid: host timeline of the upload on stderr
    struct timespec ts0;
    clock_gettime(CLOCK_MONOTONIC, &ts0);
    auto stamp = [&](const char *what) {
        if (!csr_trace) return;
        struct timespec ts;
        clock_gettime(CLOCK_MONOTONIC, &ts);
        fprintf(stderr, "from_csr: %-44s %8.2f ms\n", what, 1e3 * (double)(ts.tv_sec - ts0.tv_sec) + 1e-6 * (double)(ts.tv_nsec - ts0.tv_nsec));
    };
    int *d_bad = (int *)(ctx->d_counters + CTR_BAD);
    CUDA_TRY(cudaMemsetAsync(d_bad, 0, sizeof(int), ctx->stream));
    const size_t eb = (size_t)(E ? E : 1) * 4;
    CUDA_TRY(vglb_dev_alloc(&g->d_out_ptr, ((size_t)V + 2) * 8));
    stamp("first allocation");
    CUDA_TRY(vglb_dev_alloc(&g->d_out_adj, eb + 16));
    // The upload is PCIe-bound (1.3 GB at ~55 GB/s for the BASELINE PageRank graph), so the device works while it runs: the
    // adjacency goes up in 8 row-aligned chunks on a second stream and the in-degrees without self loops — what PageRank's
    // preparation needs first (pr.hpp:28-73), a 7 ms pass of atomics — are counted chunk by chunk behind it.
    CUDA_TRY(cudaMemcpyAsync(g->d_out_ptr, h_out_ptr, ((size_t)V + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(vglb_dev_alloc(&g->d_indeg_noloops, (size_t)V * 4));
    CUDA_TRY(cudaMemsetAsync(g->d_indeg_noloops, 0, (size_t)V * 4, ctx->stream));
    csr_ptr_check_kernel<<<(unsigned)ceil_div64((int64_t)V + 1, 256), 256, 0, ctx->stream>>>(g->d_out_ptr, V, E, d_bad);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaEventRecord(ctx->ev_chunk[0], ctx->stream));
    CUDA_TRY(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_chunk[0], 0)); // (orders the copy stream after earlier work on the buffers)
    const int chunks = E >= (1 << 22) ? 8 : 1;
    // rows are degree-sorted: binary search the first row with fewer than d edges
    auto rows_with_degree_at_least = [&](int64_t d) {
        int32_t lo = 0, hi = V;
        while (lo < hi)
        {
            const int32_t mid = lo + (hi - lo) / 2;
            if (h_out_ptr[mid + 1] - h_out_ptr[mid] >= d) lo = mid + 1;
            else hi = mid;
        }
        return lo;
    };
    // chunk k = rows [border[k], border[k+1]): border[k] = first row whose edges start at or after the k-th eighth of the edge array
    int32_t border[9];
    border[0] = 0;
    for (int k = 1; k < chunks; k++)
    {
        const int64_t target = E / chunks * k;
        int32_t lo = border[k - 1], hi = V;
        while (lo < hi)
        {
            const int32_t mid = lo + (hi - lo) / 2;
            if (h_out_ptr[mid] < target) lo = mid + 1;
            else hi = mid;
        }
        border[k] = lo;
    }
    border[chunks] = V;
    // PageRank's column-binned copy of the rows with >= 32 edges (pagerank_bins.cu) only needs those rows: when the caller's
    // buffer is pinned (every copy can be queued at once) it is built as soon as their last chunk has landed, behind the rest of
    // the upload. The border nearest to the end of those rows is moved there.
    int heavy_chunk = -1; // chunk that ends the heavy rows
    int32_t heavy_rows = 0;
    const int32_t short_rows_from = chunks > 1 ? rows_with_degree_at_least(32) : V; // (a small graph goes up as one chunk)
    if (chunks > 1 && (ctx->upload_hint & VGLB_HINT_PAGERANK) && vglb_pr_bins_wanted(g))
    {
        cudaPointerAttributes attr;
        const bool pinned = cudaPointerGetAttributes(&attr, h_out_adj) == cudaSuccess && attr.type == cudaMemoryTypeHost;
        cudaGetLastError();
        heavy_rows = rows_with_degree_at_least(vglb_tier_degree(1));
        if (pinned && heavy_rows > 0 && heavy_rows < V && h_out_ptr[heavy_rows] >= 0 && h_out_ptr[heavy_rows] <= E)
        {
            int best = 1;
            for (int k = 2; k < chunks; k++)
                if (llabs(h_out_ptr[border[k]] - h_out_ptr[heavy_rows]) < llabs(h_out_ptr[border[best]] - h_out_ptr[heavy_rows])) best = k;
            border[best] = heavy_rows;
            for (int k = best - 1; k > 0; k--) border[k] = std::min(border[k], heavy_rows);
            for (int k = best + 1; k < chunks; k++) border[k] = std::max(border[k], heavy_rows);
            heavy_chunk = best - 1;
        }
    }
    for (int k = 0; k < chunks; k++)
    {
        const int64_t e0 = h_out_ptr[border[k]], e1 = h_out_ptr[border[k + 1]];
        if (e0 < 0 || e1 < e0 || e1 > E)
        {
            cudaStreamSynchronize(ctx->copy_stream);
            cudaStreamSynchronize(ctx->stream);
            vglb_set_error("vglb_graph_from_csr: row pointers are not non-decreasing within [0, E]");
            return VGLB_EINVAL;
        }
    }
    // the other arrays of the caller: queued on the copy stream behind the adjacency (before the host waits for anything)
    CUDA_TRY(vglb_dev_alloc(&g->d_fwd, (size_t)V * 4));
    CUDA_TRY(vglb_dev_alloc(&g->d_bwd, (size_t)V * 4));
    if (h_in_ptr)
    {
        CUDA_TRY(vglb_dev_alloc(&g->d_in_ptr, ((size_t)V + 2) * 8));
        CUDA_TRY(vglb_dev_alloc(&g->d_in_adj, eb + 16));
    }
    bool others_queued = false;
    auto queue_others = [&]() -> cudaError_t {
        if (others_queued) return cudaSuccess;
        others_queued = true;
        cudaError_t e = cudaSuccess;
        if (h_orig_to_sorted) e = cudaMemcpyAsync(g->d_fwd, h_orig_to_sorted, (size_t)V * 4, cudaMemcpyHostToDevice, ctx->copy_stream);
        if (e == cudaSuccess && h_in_ptr) e = cudaMemcpyAsync(g->d_in_ptr, h_in_ptr, ((size_t)V + 1) * 8, cudaMemcpyHostToDevice, ctx->copy_stream);
        if (e == cudaSuccess && h_in_ptr) e = cudaMemcpyAsync(g->d_in_adj, h_in_adj, (size_t)E * 4, cudaMemcpyHostToDevice, ctx->copy_stream);
        return e;
    };
    if (heavy_chunk >= 0) // pinned source: queue every copy first
        for (int k = 0; k < chunks; k++)
        {
            const int64_t e0 = h_out_ptr[border[k]], e1 = h_out_ptr[border[k + 1]];
            if (e1 > e0)
                CUDA_TRY(cudaMemcpyAsync(g->d_out_adj + e0, h_out_adj + e0, (size_t)(e1 - e0) * 4, cudaMemcpyHostToDevice, ctx->copy_stream));
            CUDA_TRY(cudaEventRecord(ctx->ev_chunk[k], ctx->copy_stream));
        }
    if (heavy_chunk >= 0) CUDA_TRY(queue_others());
    for (int k = 0; k < chunks; k++)
    {
        const int32_t row0 = border[k], row1 = border[k + 1];
        const int64_t e0 = h_out_ptr[row0], e1 = h_out_ptr[row1];
        if (e1 > e0)
        {
            if (heavy_chunk < 0)
            {
                CUDA_TRY(cudaMemcpyAsync(g->d_out_adj + e0, h_out_adj + e0, (size_t)(e1 - e0) * 4, cudaMemcpyHostToDevice, ctx->copy_stream));
                CUDA_TRY(cudaEventRecord(ctx->ev_chunk[k], ctx->copy_stream));
            }
            CUDA_TRY(cudaStreamWaitEvent(ctx->stream, ctx->ev_chunk[k], 0));
            // (rows are degree-sorted: a chunk that starts at or after the first row with fewer than 32 edges has only such rows)
            if (row0 >= short_rows_from)
                indegree_noloops_short_rows_kernel<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(g->d_out_ptr, g->d_out_adj, row0, row1, e0, e1, V,
                                                                                               g->d_indeg_noloops, d_bad);
            else
                indegree_noloops_rows_kernel<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(g->d_out_ptr, g->d_out_adj, row0, row1, e0, e1, V,
                                                                                         g->d_indeg_noloops, d_bad);
            CUDA_TRY(cudaGetLastError());
            ctx->launches++;
        }
        if (k == heavy_chunk)
        {
            // (the row pointers were checked by csr_ptr_check_kernel: a bad array fails the call below, not the build)
            int bad = 0;
            stamp("copies queued");
            CUDA_TRY(cudaMemcpyAsync(&bad, d_bad, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
            CUDA_TRY(cudaStreamSynchronize(ctx->stream));
            stamp("heavy rows have landed");
            if (!bad)
            {
                g->pr_bins_tried = 1;
                const int rcb = vglb_pr_bins_build_rows(ctx, g, heavy_rows);
                if (rcb != VGLB_ENOMEM) VGLB_TRY(rcb); // (no memory for the binned copy: PageRank falls back to warp tasks)
                stamp("column bins built");
            }
        }
    }
    CUDA_TRY(queue_others());
    const unsigned vgrid = (unsigned)ceil_div64(V, 256);
    if (chunks > 1 && !vglb_pr_bins_wanted(g))
    {
        // the host is idle while the DMA runs: PageRank's warp-task table of the rows with >= 32 edges (pagerank.cu) is built
        // from the caller's row pointers now instead of costing 3-4 ms later
        VGLB_TRY(vglb_pr_build_tasks_host(ctx, g, h_out_ptr, rows_with_degree_at_least(vglb_tier_degree(1)),
                                           rows_with_degree_at_least(vglb_tier_degree(0))));
    }
    CUDA_TRY(cudaEventRecord(ctx->ev_chunk[0], ctx->copy_stream));
    CUDA_TRY(cudaStreamWaitEvent(ctx->stream, ctx->ev_chunk[0], 0)); // every upload is ordered before later work on `stream`
    if (!h_orig_to_sorted)
    {
        iota_kernel<<<vgrid, 256, 0, ctx->stream>>>(g->d_fwd, V);
        CUDA_TRY(cudaGetLastError());
    }
    CUDA_TRY(cudaMemsetAsync(g->d_bwd, 0xFF, (size_t)V * 4, ctx->stream));
    VGLB_TRY(vglb_invert_map_checked(ctx, g->d_fwd, V, V, g->d_bwd));
    if (h_in_ptr) VGLB_TRY(vglb_csr_validate_device(ctx, g->d_in_ptr, V, E, g->d_in_adj, V));
    int bad = 0;
    stamp("checks queued");
    CUDA_TRY(cudaMemcpyAsync(&bad, d_bad, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    stamp("uploads and checks done");
    if (bad)
    {
        vglb_set_error("vglb_graph_from_csr: not a CSR (row pointers must be non-decreasing from 0 to E, vertex ids in [0, V), "
                       "the ORIGINAL -> sorted map a permutation)");
        return VGLB_EINVAL;
    }
    VGLB_TRY(vglb_graph_compute_tiers(ctx, g));
    stamp("tiers");
    vglb_graph_set_unpartitioned(g);
    *out_graph = owner.release();
    return VGLB_OK;
}

// One direction of a VectorCSRGraph that already lives in device-accessible memory (cudaMalloc'ed or managed: the reference's
// GPU build keeps vertex_pointers / adjacent_ids in cudaMallocManaged memory, memory_API.hpp:3-15): nothing is copied, the
// arrays stay the caller's. What the borrowed graph adds is what the operators need on top of the arrays: the degree-tier
// borders (estimate_thresholds, vect_csr/nec_api.hpp:5-50) and a home for frontier objects.
extern "C" int vglb_graph_borrow_csr(vglb_ctx *ctx, int32_t V, int64_t E, const int64_t *d_ptr, const int32_t *d_adj, vglb_graph **out_graph)
{
    VGLB_REQUIRE(ctx != NULL && out_graph != NULL && d_ptr != NULL, "vglb_graph_borrow_csr: NULL argument");
    VGLB_REQUIRE(V > 0 && E >= 0 && (E == 0 || d_adj != NULL), "vglb_graph_borrow_csr: bad sizes");
    CUDA_TRY(cudaSetDevice(ctx->device));
    graph_ptr owner = vglb_graph_new();
    if (!owner) return VGLB_ENOMEM;
    vglb_graph *g = owner.get();
    g->V = V;
    g->E = E;
    g->borrowed_csr = 1;
    g->d_out_ptr = const_cast<int64_t *>(d_ptr);
    g->d_out_adj = const_cast<int32_t *>(d_adj);
    VGLB_TRY(vglb_graph_compute_tiers(ctx, g)); // also rejects rows that are not degree-sorted (VGLB_EUNSORTED)
    vglb_graph_set_unpartitioned(g);
    *out_graph = owner.release();
    return VGLB_OK;
}

// incoming CSR of an uploaded graph, derived on the device from the outgoing one (same numbering)
__global__ void row_of_position_kernel(const int64_t *__restrict__ ptr, int32_t V, uint32_t *__restrict__ row_of_pos)
{
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t v = warp; v < V; v += nwarps)
        for (int64_t p = ptr[v] + lane; p < ptr[v + 1]; p += 32) row_of_pos[p] = (uint32_t)v;
}

__global__ void indegree_from_adj_kernel(const int32_t *__restrict__ adj, int64_t E, unsigned long long *__restrict__ indeg)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; i < E; i += stride) atomicAdd(&indeg[adj[i]], 1ULL);
}

int vglb_graph_derive_incoming(vglb_ctx *ctx, vglb_graph *g)
{
    VGLB_REQUIRE(ctx != NULL && g != NULL && g->comm == NULL, "vglb_graph_derive_incoming: needs an unpartitioned graph");
    if (g->d_in_ptr) return VGLB_OK;
    const int32_t V = g->V;
    const int64_t E = g->E;
    const size_t eb = (size_t)(E ? E : 1) * 4;
    dev_ptr<int64_t> d_deg, in_ptr;
    dev_ptr<int32_t> in_adj;
    dev_ptr<uint32_t> d_row_of_pos;
    dev_ptr<void> tmp;
    CUDA_TRY(vglb_dev_alloc(d_deg, ((size_t)V + 2) * 8));
    CUDA_TRY(cudaMemsetAsync(d_deg.get(), 0, ((size_t)V + 2) * 8, ctx->stream));
    CUDA_TRY(vglb_dev_alloc(in_ptr, ((size_t)V + 2) * 8));
    CUDA_TRY(vglb_dev_alloc(in_adj, eb + 16));
    if (E)
    {
        CUDA_TRY(vglb_dev_alloc(d_row_of_pos, eb));
        row_of_position_kernel<<<ctx->sm_count * 16, 256, 0, ctx->stream>>>(g->d_out_ptr, V, d_row_of_pos.get());
        KERNEL_TRY();
        indegree_from_adj_kernel<<<ctx->sm_count * 16, 256, 0, ctx->stream>>>(g->d_out_adj, E, (unsigned long long *)d_deg.get());
        KERNEL_TRY();
    }
    CUDA_TRY(vglb_cub(tmp, [&](void *t, size_t &bytes) {
        return cub::DeviceScan::ExclusiveSum(t, bytes, d_deg.get(), in_ptr.get(), V + 1, ctx->stream);
    }));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    VGLB_TRY(build_incoming(ctx, V, E, g->d_out_adj, d_row_of_pos.get(), in_adj.get()));
    g->d_in_ptr = in_ptr.release(); // (the graph gets its incoming CSR only when it is complete)
    g->d_in_adj = in_adj.release();
    return VGLB_OK;
}

extern "C" int vglb_graph_get_info(vglb_graph *g, vglb_graph_info *info)
{
    VGLB_REQUIRE(g != NULL && info != NULL, "vglb_graph_get_info: NULL argument");
    memset(info, 0, sizeof(*info));
    info->vertices = g->V;
    info->edges = g->E;
    info->has_incoming = g->d_in_ptr != NULL;
    info->max_degree = g->max_degree;
    for (int t = 0; t < VGLB_NUM_TIERS; t++)
    {
        info->tier_degree[t] = g->tier_degree[t];
        info->tier_border[t] = g->tier_border[t];
    }
    info->d_out_ptr = g->d_out_ptr;
    info->d_out_adj = g->d_out_adj;
    info->d_in_ptr = g->d_in_ptr;
    info->d_in_adj = g->d_in_adj;
    info->d_orig_to_sorted = g->d_fwd;
    info->d_sorted_to_orig = g->d_bwd;
    info->d_edge_order = g->d_edge_order;
    info->part_rank = g->part_rank;
    info->part_world = g->part_world;
    info->rows_per_rank = g->vp;
    info->col_of_row0 = g->col_of_row0;
    info->vertices_global = g->V_orig;
    info->columns = g->cols;
    info->edges_global = g->E_global;
    return VGLB_OK;
}

// ---- estimate_thresholds twin for an arbitrary threshold -------------------------------------------------------------

__global__ void threshold_vertex_kernel(const int64_t *__restrict__ ptr, int32_t V, int32_t T, int32_t *out)
{
    int32_t v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= V) return;
    const int64_t d = ptr[v + 1] - ptr[v];
    const int64_t dn = (v == V - 1) ? -1 : ptr[v + 2] - ptr[v + 1];
    if (d >= T && dn < T) *out = v + 1;
}

extern "C" int vglb_graph_threshold_vertex(vglb_ctx *ctx, vglb_graph *g, int32_t degree_threshold, int32_t *out_vertex)
{
    VGLB_REQUIRE(ctx != NULL && g != NULL && out_vertex != NULL, "vglb_graph_threshold_vertex: NULL argument");
    int32_t *d_out = (int32_t *)(ctx->d_counters + CTR_SCRATCH_I32);
    CUDA_TRY(cudaMemsetAsync(d_out, 0, 4, ctx->stream));
    threshold_vertex_kernel<<<(unsigned)ceil_div64(g->V, 256), 256, 0, ctx->stream>>>(g->d_out_ptr, g->V, degree_threshold, d_out);
    KERNEL_TRY();
    CUDA_TRY(cudaMemcpyAsync(out_vertex, d_out, 4, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    CUDA_TRY(cudaMemsetAsync(d_out, 0, 4, ctx->stream));
    return VGLB_OK;
}

// ---- VerticesArray::reorder (vgl_graph/reorder.hpp:3-170, cuda_reorder.cu:5-37): one out-of-place gather ------------

__global__ void reorder_gather_kernel(const uint32_t *__restrict__ in, uint32_t *__restrict__ out,
                                      const int32_t *__restrict__ index, int32_t V)
{
    int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < V) out[i] = in[index[i]];
}

extern "C" int vglb_varray_reorder_u32(vglb_ctx *ctx, vglb_graph *g, const uint32_t *d_in, uint32_t *d_out, int from_dir,
                                       int to_dir)
{
    VGLB_REQUIRE(ctx != NULL && g != NULL && d_in != NULL && d_out != NULL, "vglb_varray_reorder_u32: NULL argument");
    VGLB_REQUIRE(d_in != (const uint32_t *)d_out, "vglb_varray_reorder_u32: reorder is out-of-place");
    const bool to_orig = from_dir == VGLB_SCATTER && to_dir == VGLB_ORIGINAL;
    const bool to_sorted = from_dir == VGLB_ORIGINAL && to_dir == VGLB_SCATTER;
    if (!to_orig && !to_sorted)
    {
        vglb_set_error("vglb_varray_reorder_u32: only ORIGINAL <-> SCATTER is supported on the device layout "
                       "(the incoming CSR shares the SCATTER numbering)");
        return VGLB_EINVAL;
    }
    if (g->comm)
    {
        // partitioned graph: SCATTER arrays hold this rank's rows, ORIGINAL arrays the whole graph (collective call)
        if (to_sorted)
        {
            if (g->V > 0)
            {
                reorder_gather_kernel<<<(unsigned)ceil_div64(g->V, 256), 256, 0, ctx->stream>>>(d_in, d_out, g->d_bwd + g->col_of_row0, g->V);
                KERNEL_TRY();
            }
            ctx->launches++;
            return VGLB_OK;
        }
        dev_ptr<uint32_t> full;
        CUDA_TRY(vglb_dev_alloc(full, (size_t)g->cols * 4));
        CUDA_TRY(cudaMemsetAsync(full.get() + g->col_of_row0, 0, (size_t)g->vp * 4, ctx->stream));
        CUDA_TRY(cudaMemcpyAsync(full.get() + g->col_of_row0, d_in, (size_t)g->V * 4, cudaMemcpyDeviceToDevice, ctx->stream));
        VGLB_TRY(vglb_comm_allgather_async(g->comm, full.get(), (size_t)g->vp * 4));
        reorder_gather_kernel<<<(unsigned)ceil_div64(g->V_orig, 256), 256, 0, ctx->stream>>>(full.get(), d_out, g->d_fwd, g->V_orig);
        KERNEL_TRY();
        CUDA_TRY(cudaStreamSynchronize(ctx->stream));
        ctx->launches++;
        return VGLB_OK;
    }
    const int32_t *index = to_orig ? g->d_fwd : g->d_bwd; // out[orig] = in[fwd[orig]] / out[sorted] = in[bwd[sorted]]
    reorder_gather_kernel<<<(unsigned)ceil_div64(g->V, 256), 256, 0, ctx->stream>>>(d_in, d_out, index, g->V);
    KERNEL_TRY();
    ctx->launches++;
    return VGLB_OK;
}

// ---- EdgesArray synthetic weights (EdgesArray::set_all_random twin, deterministic) ---------------------------------

__global__ void fill_weights_kernel(const int64_t *__restrict__ ptr, const int32_t *__restrict__ adj,
                                    const int32_t *__restrict__ bwd, int32_t V, int32_t col0, uint64_t seed, float *__restrict__ w)
{
    // warp per row, lanes stride the row
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t v = warp; v < V; v += nwarps)
    {
        const int64_t s = ptr[v], e = ptr[v + 1];
        const int32_t ov = bwd[col0 + v];
        for (int64_t p = s + lane_id(); p < e; p += 32) w[p] = vglb_edge_weight(ov, bwd[adj[p]], seed);
    }
}

extern "C" int vglb_earray_fill_synthetic_weights(vglb_ctx *ctx, vglb_graph *g, uint64_t seed, float *d_weights)
{
    VGLB_REQUIRE(ctx != NULL && g != NULL && d_weights != NULL, "vglb_earray_fill_synthetic_weights: NULL argument");
    fill_weights_kernel<<<ctx->sm_count * 16, 256, 0, ctx->stream>>>(g->d_out_ptr, g->d_out_adj, g->d_bwd, g->V, g->col_of_row0, seed, d_weights);
    KERNEL_TRY();
    ctx->launches++;
    return VGLB_OK;
}

// ---- in-degree without self loops on the SCATTER numbering (pr.hpp:28-73) --------------------------------------------

__global__ void indegree_noloops_kernel(const int64_t *__restrict__ ptr, const int32_t *__restrict__ adj, int32_t V,
                                        int32_t *__restrict__ indeg)
{
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t v = warp; v < V; v += nwarps)
    {
        const int64_t s = ptr[v], e = ptr[v + 1];
        for (int64_t p = s + lane_id(); p < e; p += 32)
        {
            const int32_t d = adj[p];
            if (d != (int32_t)v) atomicAdd(&indeg[d], 1);
        }
    }
}

extern "C" int vglb_graph_indegree_noloops(vglb_ctx *ctx, vglb_graph *g, int32_t *d_indeg)
{
    VGLB_REQUIRE(ctx != NULL && g != NULL && d_indeg != NULL, "vglb_graph_indegree_noloops: NULL argument");
    VGLB_REQUIRE(g->comm == NULL, "vglb_graph_indegree_noloops: not available on a partitioned graph (in-degrees are counted by the partitioned build)");
    if (g->d_indeg_noloops) // counted while the graph was uploaded
    {
        CUDA_TRY(cudaMemcpyAsync(d_indeg, g->d_indeg_noloops, (size_t)g->V * 4, cudaMemcpyDeviceToDevice, ctx->stream));
        return VGLB_OK;
    }
    CUDA_TRY(cudaMemsetAsync(d_indeg, 0, (size_t)g->V * 4, ctx->stream));
    indegree_noloops_kernel<<<ctx->sm_count * 16, 256, 0, ctx->stream>>>(g->d_out_ptr, g->d_out_adj, g->V, d_indeg);
    KERNEL_TRY();
    ctx->launches++;
    return VGLB_OK;
}
