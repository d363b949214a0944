// graph_io.cu — the reference's on-disk formats, read and written by libvgl_b200 (SURVEY §8f row 3).
//
//   .el_container : EdgesContainer::save_to_binary_file / load_from_binary_file
//                   (vgl_runtime/graph_generation/edges_container.h:58-99) — int32 V, int64 E, int32 EDGES_CONTAINER (= 4),
//                   int32 src[E], int32 dst[E]; what the apps read with `-import <file>` (cmd_parser.hpp:64-68).
//   .vgl / .vcsr  : VGL_Graph::save_to_binary_file / load_from_binary_file (vgl_graph.hpp:109-161) — int32 V, int64 E,
//                   int32 container type (VECTOR_CSR_GRAPH = 1), then the OUTGOING and the INCOMING VectorCSRGraph
//                   (vect_csr_graph.hpp:141-180): int32 V, int64 E, int32 format, int64 vertex_pointers[V+1], int32
//                   adjacent_ids[E], int32 forward_conversion[V], int32 backward_conversion[V], int64 edges_reorder_indexes[E].
//                   The incoming container is the import of the TRANSPOSED edge list (its own, in-degree-sorted numbering).
// Files written here are byte-identical to the reference's (tests/test_gpu_io.py compares them); files written by the
// reference load straight into the device layout: the outgoing container is uploaded as is, the incoming direction is
// re-derived on the device on the SAME numbering as the outgoing one (the layout bottom-up BFS wants, DESIGN.md §3).
#include <stdio.h>
#include <stdlib.h>

#include "common.cuh"

#define VGL_FORMAT_VECTOR_CSR_GRAPH 1 /* framework_types.h:49-57 */
#define VGL_FORMAT_EDGES_CONTAINER 4

namespace
{
struct File
{
    FILE *f;
    explicit File(const char *path, const char *mode) : f(fopen(path, mode)) {}
    ~File() { if (f) fclose(f); }
    bool write(const void *p, size_t bytes) { return bytes == 0 || fwrite(p, 1, bytes, f) == bytes; }
    bool read(void *p, size_t bytes) { return bytes == 0 || fread(p, 1, bytes, f) == bytes; }
};
} // namespace

extern "C" int vglb_el_container_save(const char *path, int32_t vertices, int64_t edges, const int32_t *h_src,
                                      const int32_t *h_dst)
{
    VGLB_REQUIRE(path != NULL && vertices > 0 && edges >= 0 && (edges == 0 || (h_src && h_dst)), "vglb_el_container_save: bad argument");
    File F(path, "wb");
    if (!F.f)
    {
        vglb_set_error("vglb_el_container_save: cannot open %s", path);
        return VGLB_EINVAL;
    }
    const int32_t type = VGL_FORMAT_EDGES_CONTAINER;
    long long e = edges;
    if (!F.write(&vertices, 4) || !F.write(&e, 8) || !F.write(&type, 4) || !F.write(h_src, (size_t)edges * 4) || !F.write(h_dst, (size_t)edges * 4))
    {
        vglb_set_error("vglb_el_container_save: write to %s failed", path);
        return VGLB_EINVAL;
    }
    return VGLB_OK;
}

// VGL_Graph::import of a file (apps: `-import <file>`): the edge list goes through pinned memory into the GPU builder
extern "C" int vglb_graph_import_el_container(vglb_ctx *ctx, const char *path, int flags, vglb_graph **out_graph)
{
    VGLB_REQUIRE(ctx != NULL && path != NULL && out_graph != NULL, "vglb_graph_import_el_container: NULL argument");
    File F(path, "rb");
    if (!F.f)
    {
        vglb_set_error("vglb_graph_import_el_container: cannot open %s", path);
        return VGLB_EINVAL;
    }
    int32_t V = 0, type = 0;
    long long E = 0;
    if (!F.read(&V, 4) || !F.read(&E, 8) || !F.read(&type, 4) || V <= 0 || E < 0)
    {
        vglb_set_error("vglb_graph_import_el_container: %s is not an edges container", path);
        return VGLB_EINVAL;
    }
    if (type != VGL_FORMAT_EDGES_CONTAINER)
    {
        // EdgesContainer::load_from_binary_file throws the same complaint (edges_container.h:88-89)
        vglb_set_error("Error in EdgesContainer::load_from_binary_file : incorrect type of graph in file");
        return VGLB_EINVAL;
    }
    int32_t *h_src = NULL, *h_dst = NULL;
    const size_t bytes = (size_t)(E > 0 ? E : 1) * 4;
    if (cudaMallocHost((void **)&h_src, bytes) != cudaSuccess || cudaMallocHost((void **)&h_dst, bytes) != cudaSuccess)
    {
        cudaGetLastError();
        cudaFreeHost(h_src);
        vglb_set_error("vglb_graph_import_el_container: cannot allocate %zu bytes of pinned memory", 2 * bytes);
        return VGLB_ENOMEM;
    }
    int rc = VGLB_OK;
    if (!F.read(h_src, (size_t)E * 4) || !F.read(h_dst, (size_t)E * 4))
    {
        vglb_set_error("vglb_graph_import_el_container: %s is truncated", path);
        rc = VGLB_EINVAL;
    }
    if (rc == VGLB_OK) rc = vglb_graph_from_edges(ctx, V, E, h_src, h_dst, 0, flags, out_graph);
    cudaFreeHost(h_src);
    cudaFreeHost(h_dst);
    return rc;
}

// the edge list in outgoing-CSR order, ORIGINAL ids: position p of row r holds (bwd[r], bwd[adj[p]])
__global__ void csr_order_edges_kernel(const int64_t *__restrict__ ptr, const int32_t *__restrict__ adj, const int32_t *__restrict__ bwd,
                                       int32_t V, int32_t *__restrict__ src, int32_t *__restrict__ dst)
{
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t v = warp; v < V; v += nwarps)
    {
        const int32_t ov = bwd[v];
        for (int64_t p = ptr[v] + lane; p < ptr[v + 1]; p += 32)
        {
            src[p] = ov;
            dst[p] = bwd[adj[p]];
        }
    }
}

// one VectorCSRGraph::save_main_content_to_binary_file (vect_csr_graph.hpp:141-155) from a device graph built WITH_EDGE_ORDER
static int save_container(vglb_ctx *ctx, File &F, vglb_graph *g)
{
    const int32_t V = g->V, fmt = VGL_FORMAT_VECTOR_CSR_GRAPH;
    long long E = g->E;
    const size_t biggest = (size_t)(E > V + 1 ? E : V + 1) * 8;
    void *h = malloc(biggest ? biggest : 8);
    if (!h) return VGLB_ENOMEM;
    bool ok = F.write(&V, 4) && F.write(&E, 8) && F.write(&fmt, 4);
    struct Piece { const void *d; size_t bytes; } pieces[5] = {{g->d_out_ptr, ((size_t)V + 1) * 8}, {g->d_out_adj, (size_t)E * 4},
                                                                {g->d_fwd, (size_t)V * 4}, {g->d_bwd, (size_t)V * 4},
                                                                {g->d_edge_order, (size_t)E * 8}};
    for (int i = 0; i < 5 && ok; i++)
    {
        if (pieces[i].bytes == 0) continue;
        if (cudaMemcpyAsync(h, pieces[i].d, pieces[i].bytes, cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess ||
            cudaStreamSynchronize(ctx->stream) != cudaSuccess)
        {
            cudaGetLastError();
            ok = false;
            break;
        }
        ok = F.write(h, pieces[i].bytes);
    }
    free(h);
    if (!ok)
    {
        vglb_set_error("vglb_graph_save_vgl: writing a container failed");
        return VGLB_EINVAL;
    }
    return VGLB_OK;
}

// VGL_Graph::import + save_to_binary_file (vgl_graph.hpp:57-68,109-131): both containers are built on the GPU — the
// incoming one as the import of the transposed edge list, exactly what the reference does — and written in its format.
extern "C" int vglb_graph_save_vgl(vglb_ctx *ctx, const char *path, int32_t vertices, int64_t edges, const int32_t *src,
                                   const int32_t *dst, int src_on_device)
{
    VGLB_REQUIRE(ctx != NULL && path != NULL, "vglb_graph_save_vgl: NULL argument");
    File F(path, "wb");
    if (!F.f)
    {
        vglb_set_error("vglb_graph_save_vgl: cannot open %s", path);
        return VGLB_EINVAL;
    }
    const int32_t type = VGL_FORMAT_VECTOR_CSR_GRAPH;
    long long e = edges;
    if (!F.write(&vertices, 4) || !F.write(&e, 8) || !F.write(&type, 4))
    {
        vglb_set_error("vglb_graph_save_vgl: write to %s failed", path);
        return VGLB_EINVAL;
    }
    // outgoing container
    vglb_graph *g_out = NULL;
    VGLB_TRY(vglb_graph_from_edges(ctx, vertices, edges, src, dst, src_on_device, VGLB_GRAPH_WITH_EDGE_ORDER, &g_out));
    graph_ptr out_owner(g_out);
    VGLB_TRY(save_container(ctx, F, g_out));
    // incoming container = import of the transposed edge list — in the order the OUTGOING import left the container in:
    // VectorCSRGraph::import sorts the EdgesContainer by the new source id and only renumbers the ids back afterwards
    // (vect_csr/import.hpp:299-326), so VGL_Graph::import (vgl_graph.hpp:57-68) hands the incoming import the edges in
    // outgoing-CSR order, and its edges_reorder_indexes refer to that order.
    dev_ptr<int32_t> d_s, d_d;
    if (edges > 0)
    {
        CUDA_TRY(vglb_dev_alloc(d_s, (size_t)edges * 4));
        CUDA_TRY(vglb_dev_alloc(d_d, (size_t)edges * 4));
        csr_order_edges_kernel<<<ctx->sm_count * 16, 256, 0, ctx->stream>>>(g_out->d_out_ptr, g_out->d_out_adj, g_out->d_bwd, vertices,
                                                                            d_s.get(), d_d.get());
        KERNEL_TRY();
    }
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    out_owner.reset();
    vglb_graph *g_in = NULL;
    VGLB_TRY(vglb_graph_from_edges(ctx, vertices, edges, d_d.get(), d_s.get(), 1, VGLB_GRAPH_WITH_EDGE_ORDER, &g_in)); // transposed
    graph_ptr in_owner(g_in);
    VGLB_TRY(save_container(ctx, F, g_in));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return VGLB_OK;
}

// VGL_Graph::load_from_binary_file + move_to_device (vgl_graph.hpp:133-161, vect_csr_graph.hpp:158-196)
extern "C" int vglb_graph_load_vgl(vglb_ctx *ctx, const char *path, int flags, vglb_graph **out_graph)
{
    VGLB_REQUIRE(ctx != NULL && path != NULL && out_graph != NULL, "vglb_graph_load_vgl: NULL argument");
    VGLB_REQUIRE(!(flags & VGLB_GRAPH_WITH_EDGE_ORDER), "vglb_graph_load_vgl: VGLB_GRAPH_WITH_EDGE_ORDER is not supported");
    File F(path, "rb");
    if (!F.f)
    {
        vglb_set_error("vglb_graph_load_vgl: cannot open %s", path);
        return VGLB_EINVAL;
    }
    int32_t V = 0, type = 0, cV = 0, cfmt = 0;
    long long E = 0, cE = 0;
    if (!F.read(&V, 4) || !F.read(&E, 8) || !F.read(&type, 4) || !F.read(&cV, 4) || !F.read(&cE, 8) || !F.read(&cfmt, 4) || V <= 0 ||
        E < 0 || cV != V || cE != E)
    {
        vglb_set_error("vglb_graph_load_vgl: %s is not a VGL graph file", path);
        return VGLB_EINVAL;
    }
    if (type != VGL_FORMAT_VECTOR_CSR_GRAPH || cfmt != VGL_FORMAT_VECTOR_CSR_GRAPH)
    {
        vglb_set_error("vglb_graph_load_vgl: %s holds container type %d, only VECTOR_CSR_GRAPH is supported", path, type);
        return VGLB_EINVAL;
    }
    int64_t *h_ptr = NULL;
    int32_t *h_adj = NULL, *h_fwd = NULL;
    const size_t eb = (size_t)(E > 0 ? E : 1) * 4;
    cudaError_t ce = cudaMallocHost((void **)&h_ptr, ((size_t)V + 1) * 8);
    if (ce == cudaSuccess) ce = cudaMallocHost((void **)&h_adj, eb);
    if (ce == cudaSuccess) ce = cudaMallocHost((void **)&h_fwd, (size_t)V * 4);
    int rc = VGLB_OK;
    if (ce != cudaSuccess)
    {
        cudaGetLastError();
        vglb_set_error("vglb_graph_load_vgl: cannot allocate pinned memory");
        rc = VGLB_ENOMEM;
    }
    else if (!F.read(h_ptr, ((size_t)V + 1) * 8) || !F.read(h_adj, (size_t)E * 4) || !F.read(h_fwd, (size_t)V * 4))
    {
        vglb_set_error("vglb_graph_load_vgl: %s is truncated", path);
        rc = VGLB_EINVAL;
    }
    // (backward_conversion, edges_reorder_indexes and the incoming container are not needed: the inverse map and the
    //  incoming direction are derived on the device)
    if (rc == VGLB_OK) rc = vglb_graph_from_csr(ctx, V, E, h_ptr, h_adj, h_fwd, NULL, NULL, out_graph);
    if (rc == VGLB_OK && (flags & VGLB_GRAPH_WITH_INCOMING))
    {
        rc = vglb_graph_derive_incoming(ctx, *out_graph);
        if (rc != VGLB_OK)
        {
            vglb_graph_free(ctx, *out_graph);
            *out_graph = NULL;
        }
    }
    cudaFreeHost(h_ptr);
    cudaFreeHost(h_adj);
    cudaFreeHost(h_fwd);
    return rc;
}
