/*
 * vgl_b200.h — C ABI of libvgl_b200.so: the B200-native (sm_100a) backend for VectorGraphLibrary's
 * frontier-processing hot path (GraphAbstractions scatter/gather/compute/reduce/generate_new_frontier over
 * VectCSRGraph / VerticesArray / EdgesArray / frontier, and BFS / PageRank / SSSP / CC built on them).
 *
 * The reference has no FFI for this path: the backend is a compile-time plugin slot
 * (architecture_independent_api.h:33-43, `#define VGL_GRAPH_ABSTRACTIONS <BackendClass>`), so "what the reference's
 * FFI would bind" is the set of calls its GPU backend class makes (vgl_compute_api/gpu/graph_abstractions_gpu.h:16-190)
 * plus the data-structure moves around it. Each entry point below cites the reference interface it replaces.
 * Device lambdas cannot cross a C ABI; the arbitrary-lambda path is the header-only template shim
 * include/vgl_b200/graph_abstractions_b200.cuh, which sits on top of these entry points (INTEGRATION.md).
 *
 * Conventions: every function returns 0 on success or a VGLB_E* code; the message is in vglb_last_error()
 * (reference: `throw "literal"` / SAFE_CALL, vgl_runtime/helpers/gpu_API/cuda_error_handling.h:7-27).
 * There is NO CPU fallback: every compute entry point fails with VGLB_ENODEVICE when no CUDA device is usable.
 * Pointers named d_* are device pointers owned by the caller (vglb_malloc) unless stated; h_* are host pointers
 * borrowed for the duration of the call. Vertex ids are int32, row pointers / edge positions int64, levels / labels
 * int32, ranks / distances / weights fp32 (SURVEY §8).
 */
#ifndef VGL_B200_H
#define VGL_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VGLB_OK 0
#define VGLB_EINVAL 1      /* bad argument (reference: throw "Error in ... wrong ...", common/advance.hpp:19-26) */
#define VGLB_ENODEVICE 2   /* no usable CUDA device: there is no CPU fallback */
#define VGLB_ECUDA 3       /* CUDA runtime / kernel failure (SAFE_CALL / SAFE_KERNEL_CALL) */
#define VGLB_ENOMEM 4
#define VGLB_ENCCL 5
#define VGLB_EUNSORTED 6   /* CSR rows are not degree-sorted descending (not a VectCSR layout) */

/* TraversalDirection, framework_types.h:115-119 */
#define VGLB_SCATTER 0
#define VGLB_GATHER 1
#define VGLB_ORIGINAL 2

/* BFS constants, algorithms/bfs/change_state/change_state.h:21-23 */
#define VGLB_UNVISITED_VERTEX (-1)
#define VGLB_FIRST_LEVEL_VERTEX 1

typedef struct vglb_ctx vglb_ctx;
typedef struct vglb_graph vglb_graph;

/* ---- runtime: VGL_RUNTIME::init_library -> select_device (vgl_runtime.hpp:5-16, gpu_API/select_device.cuh:5-8) ---- */
int vglb_init(int device, vglb_ctx **out_ctx);
int vglb_finalize(vglb_ctx *ctx);
const char *vglb_last_error(void);
int vglb_device_count(void);
int vglb_synchronize(vglb_ctx *ctx);
/* the CUDA stream every kernel of this context is launched on (a cudaStream_t), for event timing by the caller */
void *vglb_stream(vglb_ctx *ctx);

/* ---- memory: MemoryAPI::allocate_array / free_array / move_array_to_device (memory_API.hpp:3-15,95-101); explicit
 *      HBM allocations instead of cudaMallocManaged ---- */
int vglb_malloc(vglb_ctx *ctx, size_t bytes, void **d_ptr);
int vglb_free(vglb_ctx *ctx, void *d_ptr);
int vglb_memcpy_h2d(vglb_ctx *ctx, void *d_dst, const void *h_src, size_t bytes);
int vglb_memcpy_d2h(vglb_ctx *ctx, void *h_dst, const void *d_src, size_t bytes);
int vglb_memcpy_d2d(vglb_ctx *ctx, void *d_dst, const void *d_src, size_t bytes);
int vglb_memset(vglb_ctx *ctx, void *d_dst, int byte_value, size_t bytes);
int vglb_host_alloc_pinned(size_t bytes, void **h_ptr);
int vglb_host_free_pinned(void *h_ptr);
/* write `bytes` of a private scratch buffer (> L2) so the next timed step starts with a cold L2 */
int vglb_flush_l2(vglb_ctx *ctx);

/* ---- synthetic inputs (include/vglb_synth.h), device and host twins producing identical edges ---- */
int vglb_generate_edges_device(vglb_ctx *ctx, int kind, int scale, int64_t edges, uint64_t seed, int a, int b, int c,
                               int32_t *d_src, int32_t *d_dst);
int vglb_generate_edges_host(int kind, int scale, int64_t edges, uint64_t seed, int a, int b, int c,
                             int32_t *h_src, int32_t *h_dst);

/* ---- graph: VGL_Graph::import -> VectorCSRGraph::import (vgl_graph.hpp:57-68, vect_csr/import.hpp:257-337) ----
 * Builds, ON THE GPU, the reference's degree-sorted CSR: vertices stable-sorted by out-degree descending
 * (sorter.h:55-92), edges stable-sorted by new src (edges_container.h:101-161) => row order and adjacency order are
 * bit-identical to VectorCSRGraph's. `d_src/d_dst` are device pointers when src_on_device != 0, else host pointers.
 * flags: VGLB_GRAPH_WITH_INCOMING also builds the incoming CSR on the SAME (SCATTER) numbering (bottom-up BFS);
 *        VGLB_GRAPH_WITH_EDGE_ORDER keeps edges_reorder_indexes (CSR position -> input edge index). */
#define VGLB_GRAPH_WITH_INCOMING 1
#define VGLB_GRAPH_WITH_EDGE_ORDER 2
int vglb_graph_from_edges(vglb_ctx *ctx, int32_t vertices, int64_t edges, const int32_t *src, const int32_t *dst,
                          int src_on_device, int flags, vglb_graph **out_graph);
/* VGL_Graph::move_to_device (vect_csr_graph.hpp:185-196): borrow an already-built VectorCSRGraph (host arrays in
 * sorted numbering: get_vertex_pointers()/get_adjacent_ids(), vect_csr_graph.h:99-100) and copy it to HBM.
 * h_orig_to_sorted (forward_conversion) may be NULL (identity). Incoming arrays may be NULL. The upload is pipelined
 * (pinned host memory recommended): the adjacency goes up in chunks on a second stream while the in-degrees without self
 * loops are counted behind it. All copies have completed on return.
 * vglb_set_upload_hint(ctx, VGLB_HINT_PAGERANK): the caller will run PageRank on the graphs it uploads next, so everything the
 * sweep needs beyond the CSR (pr.hpp:28-73 and the column-binned copy of the rows with >= 32 edges, csrc/pagerank_bins.cu) is
 * built behind the upload as well instead of inside the first vglb_pagerank call. 0 clears the hint. */
#define VGLB_HINT_PAGERANK 1
int vglb_set_upload_hint(vglb_ctx *ctx, int hints);
int vglb_graph_from_csr(vglb_ctx *ctx, int32_t vertices, int64_t edges, const int64_t *h_out_ptr,
                        const int32_t *h_out_adj, const int32_t *h_orig_to_sorted, const int64_t *h_in_ptr,
                        const int32_t *h_in_adj, vglb_graph **out_graph);
/* On a partitioned graph whose buffers were mapped by the peers (vglb_graph_set_exchange(P2P), or any BFS / SSSP run over the
 * per-owner lists) this is a COLLECTIVE: every rank closes its own CUDA IPC mappings, all ranks meet, and only then are the
 * exported buffers released. Free partitioned graphs on every rank, before vglb_comm_destroy. */
int vglb_graph_free(vglb_ctx *ctx, vglb_graph *g);
/* One direction of a VectorCSRGraph that already lives in device-accessible memory (the reference's GPU build keeps
 * vertex_pointers / adjacent_ids in managed memory, memory_API.hpp:3-15; vect_csr_graph.h:99-100): nothing is copied and the
 * arrays stay the caller's. Adds the degree-tier borders and a home for frontier objects; VGLB_EUNSORTED if the rows are not
 * degree-sorted. This is what the drop-in backend (include/vgl_b200/overlay) attaches to each direction of a VGL_Graph. */
int vglb_graph_borrow_csr(vglb_ctx *ctx, int32_t vertices, int64_t edges, const int64_t *d_ptr, const int32_t *d_adj,
                          vglb_graph **out_graph);

/* ---- the reference's on-disk formats (csrc/graph_io.cu) ----
 * .el_container: EdgesContainer::save_to_binary_file / load_from_binary_file (graph_generation/edges_container.h:58-99),
 *                the apps' `-import <file>` input (cmd_parser.hpp:64-68).
 * .vgl / .vcsr : VGL_Graph::save_to_binary_file / load_from_binary_file (vgl_graph.hpp:109-161) with VECTOR_CSR_GRAPH
 *                containers (vect_csr_graph.hpp:141-180). Written files are byte-identical to the reference's. */
int vglb_el_container_save(const char *path, int32_t vertices, int64_t edges, const int32_t *h_src, const int32_t *h_dst);
int vglb_graph_import_el_container(vglb_ctx *ctx, const char *path, int flags, vglb_graph **out_graph);
int vglb_graph_save_vgl(vglb_ctx *ctx, const char *path, int32_t vertices, int64_t edges, const int32_t *src,
                        const int32_t *dst, int src_on_device);
int vglb_graph_load_vgl(vglb_ctx *ctx, const char *path, int flags, vglb_graph **out_graph);

#define VGLB_NUM_TIERS 8
typedef struct vglb_graph_info
{
    int32_t vertices;
    int64_t edges;
    int32_t has_incoming;
    int32_t max_degree;
    /* tier_border[t] = first sorted id whose out-degree is < tier_degree[t]; tiers are contiguous id ranges because
     * ids are degree-sorted (reference: vector_engine/vector_core_threshold_vertex, vect_csr/nec_api.hpp:5-50) */
    int32_t tier_degree[VGLB_NUM_TIERS];
    int32_t tier_border[VGLB_NUM_TIERS];
    /* device pointers (read-only for callers) */
    const int64_t *d_out_ptr;
    const int32_t *d_out_adj;
    const int64_t *d_in_ptr;
    const int32_t *d_in_adj;
    const int32_t *d_orig_to_sorted; /* forward_conversion */
    const int32_t *d_sorted_to_orig; /* backward_conversion */
    const int64_t *d_edge_order;     /* edges_reorder_indexes or NULL */
    /* 1D partition (see "multi-GPU" below); on one GPU: rank 0 of 1, columns = vertices_global = vertices */
    int32_t part_rank, part_world;
    int32_t rows_per_rank;           /* slice stride: column id = owner * rows_per_rank + local row */
    int32_t col_of_row0;             /* part_rank * rows_per_rank */
    int32_t vertices_global;         /* vertices of the whole graph (`vertices` = this rank's rows) */
    int32_t reserved;
    int64_t columns;                 /* length of a replicated vertex array = part_world * rows_per_rank */
    int64_t edges_global;            /* edges of the whole graph (`edges` = this rank's) */
} vglb_graph_info;
int vglb_graph_get_info(vglb_graph *g, vglb_graph_info *info);
/* threshold vertex for an arbitrary degree threshold (estimate_thresholds twin) */
int vglb_graph_threshold_vertex(vglb_ctx *ctx, vglb_graph *g, int32_t degree_threshold, int32_t *out_vertex);

/* ---- vertices / edges arrays ----
 * VerticesArray::reorder / VGL_Graph::reorder (vgl_graph/reorder.hpp:3-170, cuda_reorder.cu:5-71): permute a
 * 4-byte-element vertex array between ORIGINAL and SCATTER numbering (out-of-place gather). */
int vglb_varray_reorder_u32(vglb_ctx *ctx, vglb_graph *g, const uint32_t *d_in, uint32_t *d_out, int from_dir, int to_dir);
/* EdgesArray weights for every out-CSR position from vglb_edge_weight(orig_src, orig_dst, seed)
 * (reference: EdgesArray::set_all_random, vect_csr_edges_array.hpp:49-65) */
int vglb_earray_fill_synthetic_weights(vglb_ctx *ctx, vglb_graph *g, uint64_t seed, float *d_weights);
/* VGL_Graph::copy_outgoing_to_incoming_edges (vgl_graph/reorder.hpp:229-233 -> VectorCSRGraph::reorder_edges_gather,
 * vect_csr/reorder.hpp:61-75): per-edge 4-byte values at outgoing-CSR positions -> the positions of the same edges in the
 * incoming CSR, the second segment of an EdgesArray ([outgoing | incoming], vect_csr_edges_array.hpp:49-65), so that gather-
 * direction operators (pull SSSP, shortest_paths.hpp:168-291) can index weights with global_edge_pos. Derives the incoming
 * CSR if the graph was built without it; the permutation is computed on first use and kept with the graph. */
int vglb_earray_mirror_out_to_in_u32(vglb_ctx *ctx, vglb_graph *g, const uint32_t *d_out_values, uint32_t *d_in_values);
/* per-vertex in-degree without self loops in SCATTER numbering (pr.hpp:28-73) */
int vglb_graph_indegree_noloops(vglb_ctx *ctx, vglb_graph *g, int32_t *d_indeg);

/* ---- per-run counters: PerformanceStats (performance_stats.h:104, multicore/advance_worker.hpp:305-318) ---- */
typedef struct vglb_stats
{
    double seconds;              /* device time of the algorithm loop (CUDA events on the context stream) */
    int64_t iterations;          /* BFS levels / PR sweeps / SSSP rounds / CC hook rounds */
    int64_t edges_inspected;     /* e: edges actually read */
    int64_t vertices_processed;  /* f: frontier vertices whose row range was read */
    int64_t frontier_bytes;      /* g: frontier bytes written + read */
    int64_t algorithmic_bytes;   /* SURVEY §8(d) formula evaluated with the counters above */
    int64_t kernel_launches;     /* kernels launched by this call */
    int32_t bottom_up_levels;    /* BFS only */
    int32_t reserved;
} vglb_stats;

/* ---- fused algorithms (the four call sites of SURVEY §8 a11-a14) ---- */

/* PageRank, multicore semantics (algorithms/pr/pr.hpp:7-148): r'[u] = k + d*(sum_{u->v, v!=u} r[v]/indeg_noloops(v) + D).
 * Runs exactly `iters` sweeps; d_ranks (fp32[V]) is returned in SCATTER numbering. The first call on a graph builds what the
 * sweep needs beyond the CSR (inverse in-degrees, padded copy of the short rows, column-binned copy of the rows with >= 32 edges:
 * +0.9 GB at scale 24; or earlier, behind the upload: vglb_set_upload_hint). Sums are taken in a fixed order: two runs give the
 * same bits. */
int vglb_pagerank(vglb_ctx *ctx, vglb_graph *g, int iters, float damping, float *d_ranks, vglb_stats *stats);
/* How the dangling mass D is summed. The reference's reduce (pr.hpp:94-103 -> multicore/reduce.hpp:18-31) is an OpenMP static-
 * chunk fp32 reduction whose rounding error depends on the thread count and exceeds the 1e-6 parity tolerance by orders of
 * magnitude on large graphs (SURVEY §0 item 4b). FP64 (default, what vglb_pagerank does) sums D in double inside the sweep:
 * within 1e-7 of the exact recurrence. REFERENCE_ORDER replays the reference's summation — `reference_threads` static chunks
 * of the sorted id range, sequential fp32 inside a chunk, partials added in thread order — so the result is within 1e-6 of
 * the reference run with OMP_NUM_THREADS = reference_threads (one GPU only; a few ms slower per sweep). */
#define VGLB_PR_DANGLING_FP64 0
#define VGLB_PR_DANGLING_REFERENCE_ORDER 1
typedef struct vglb_pr_opts
{
    int32_t dangling_mode;
    int32_t reference_threads;
} vglb_pr_opts;
int vglb_pagerank_ex(vglb_ctx *ctx, vglb_graph *g, int iters, float damping, const vglb_pr_opts *opts, float *d_ranks,
                     vglb_stats *stats);

/* BFS levels (algorithms/bfs/bfs.hpp:5-86; DO heuristic change_state.hpp:100-141): source = 1, unreachable = -1,
 * SCATTER numbering. direction_optimising uses the incoming CSR: a one-GPU graph without one (vglb_graph_from_csr with NULL incoming
 * arrays, vglb_graph_from_edges without WITH_INCOMING) gets it derived on the device by the first such call; a partitioned graph
 * must be built WITH_INCOMING. alpha/beta <= 0 select 15 / 18. */
typedef struct vglb_bfs_opts
{
    int32_t direction_optimising;
    int32_t alpha;
    int32_t beta;
    int32_t reserved;
} vglb_bfs_opts;
int vglb_bfs(vglb_ctx *ctx, vglb_graph *g, int32_t source_sorted, int32_t *d_levels, const vglb_bfs_opts *opts,
             vglb_stats *stats);

/* Multi-source BFS: the levels of num_sources (1..VGLB_BFS_MULTI_MAX_SOURCES) BFS runs over one graph in one traversal
 * (bit-parallel frontiers: bit i of a vertex's word = source i). Row i of d_levels (d_levels + i*V, SCATTER numbering)
 * equals what vglb_bfs(g, h_sources_sorted[i], ...) writes: source = 1, unreachable = -1. Sources may repeat.
 * h_sources_sorted is a host array. opts as for vglb_bfs (direction_optimising, alpha, beta); the direction choice never
 * changes the levels. One-GPU graphs only: a partitioned graph returns VGLB_EINVAL.
 * The per-vertex words are w = 4 bytes for num_sources <= 32 and 8 bytes above; the call takes 3*V*w bytes of scratch for its
 * duration. stats: edges_inspected (e) and vertices_processed (f) count each edge / row once per level, not once per source;
 * iterations = levels. With e_l, f_l the edges and rows of level l, R the (vertex, source) pairs reached (sources included)
 * and k = num_sources:
 *   algorithmic_bytes = sum_l [ (4 + w) e_l + (12 + w) f_l + g_l ] + 4 k V + 4 R
 * (an edge reads its 4-byte id and one gathered word; a row its two row pointers, its queue entry and its own word; 4kV
 * initialises the output, 4R are the level stores), where the frontier traffic g_l (= frontier_bytes) is (8 + w) n_l for a
 * top-down level that queues n_l vertices, plus (4 + w) per queued vertex whose word is cleared for the next top-down level,
 * 2 w V + V/8 for a bottom-up level (seen and next words, no-in-edge mask), and 2 w V + 4 n for turning n dense words back
 * into queues. */
#define VGLB_BFS_MULTI_MAX_SOURCES 64
int vglb_bfs_multi(vglb_ctx *ctx, vglb_graph *g, int32_t num_sources, const int32_t *h_sources_sorted,
                   int32_t *d_levels, const vglb_bfs_opts *opts, vglb_stats *stats);

/* SSSP, frontier Bellman-Ford (algorithms/sssp/shortest_paths.hpp:7-78, gpu_shortest_paths.hpp:133-196): min-plus
 * fixed point in fp32 (bit-identical to the reference's seq_dijkstra), unreachable = FLT_MAX; d_weights indexed by
 * out-CSR position. Weights must be non-negative (+0.0 and -0.0 included; a distance is never -0.0). +inf and NaN weights
 * (either sign) are edges that never relax, as in seq_dijkstra; a sum that overflows to +inf leaves the distance as it was.
 * Negative weights are outside the contract: candidates are ordered on their uint32 view, where a negative candidate sorts
 * above every distance and is dropped. The frontier is scheduled near/far around a moving distance threshold (fewer
 * re-relaxations than the reference's "everything that changed" schedule, same fixed point); stats->edges_inspected =
 * edges actually relaxed. */
int vglb_sssp(vglb_ctx *ctx, vglb_graph *g, const float *d_weights, int32_t source_sorted, float *d_dist,
              vglb_stats *stats);

/* CC, min-label hook + pointer jumping (algorithms/cc/shiloach_vishkin.hpp:7-88): labels[v] = min SCATTER id over
 * {v} U ancestors(v) (= component minimum on symmetric graphs). */
int vglb_cc(vglb_ctx *ctx, vglb_graph *g, int32_t *d_labels, vglb_stats *stats);

/* ---- operators with fixed predicates (generate_new_frontier / reduce / compute without lambdas) ----
 * FrontierVectorCSR (frontier_vect_csr.h:5-53): sparse id queue + dense bitmap, chosen by density. */
typedef struct vglb_frontier vglb_frontier;
#define VGLB_FRONTIER_ALL_ACTIVE 0
#define VGLB_FRONTIER_DENSE 1
#define VGLB_FRONTIER_SPARSE 2
int vglb_frontier_create(vglb_ctx *ctx, vglb_graph *g, vglb_frontier **out);
/* the same, with the id list kept in the caller's array of >= vertices ints (the reference frontier's own ids[],
 * frontier/containers/base_frontier.h:18): compaction writes straight into the object the algorithm holds */
int vglb_frontier_create_borrowed(vglb_ctx *ctx, vglb_graph *g, int32_t *d_ids, vglb_frontier **out);
/* FrontierVectorCSR::add_group_of_vertices (modification.hpp:88-145): an ascending, duplicate-free id list becomes the
 * frontier (only on an empty frontier, like the reference). `ids` may be the frontier's own (borrowed) array. */
int vglb_frontier_set_ids(vglb_ctx *ctx, vglb_frontier *f, const int32_t *ids, int32_t n, int ids_on_device);
int vglb_frontier_destroy(vglb_ctx *ctx, vglb_frontier *f);
int vglb_frontier_set_all_active(vglb_ctx *ctx, vglb_frontier *f);
int vglb_frontier_clear(vglb_ctx *ctx, vglb_frontier *f);
int vglb_frontier_add_vertex(vglb_ctx *ctx, vglb_frontier *f, int32_t v);
typedef struct vglb_frontier_info
{
    int32_t sparsity_type;
    int32_t size;                /* number of active vertices */
    int64_t neighbours;          /* sum of their degrees */
    int32_t tier_size[3];        /* active vertices per tier (large / medium / small) */
    int32_t reserved;
    const int32_t *d_ids;        /* ascending ids when SPARSE */
    const uint32_t *d_bitmap;    /* V/32 words, always valid */
} vglb_frontier_info;
int vglb_frontier_get_info(vglb_ctx *ctx, vglb_frontier *f, vglb_frontier_info *info);
/* generate_new_frontier (common/generate_new_frontier.hpp:4-43) with the predicates the four algorithms use:
 * flags given explicitly, `values[v] == key` (BFS on_next_level), `a[v] != b[v]` (SSSP changes_occurred). */
int vglb_gnf_from_flags(vglb_ctx *ctx, vglb_frontier *f, const int32_t *d_flags);
/* flags as a bitmap (bit v of word v/32): what the lambda shim's filter kernel produces (gnf_bitmap_kernel) */
int vglb_gnf_from_bitmap(vglb_ctx *ctx, vglb_frontier *f, const uint32_t *d_bits);
int vglb_gnf_eq_i32(vglb_ctx *ctx, vglb_frontier *f, const int32_t *d_values, int32_t key);
int vglb_gnf_ne_u32(vglb_ctx *ctx, vglb_frontier *f, const uint32_t *d_a, const uint32_t *d_b);
/* reduce (common/reduce.hpp:4-67): sum / max of a vertex array over the frontier */
int vglb_reduce_sum_i32(vglb_ctx *ctx, vglb_frontier *f, const int32_t *d_values, int64_t *out);
int vglb_reduce_sum_f32(vglb_ctx *ctx, vglb_frontier *f, const float *d_values, double *out);
int vglb_reduce_max_i32(vglb_ctx *ctx, vglb_frontier *f, const int32_t *d_values, int32_t *out);

/* ---- result verification on the device (vgl_runtime/helpers/verify_results/verify_results.h) ----
 * The reference's checkers reorder both arrays to ORIGINAL and compare on the host; here both arrays are device arrays in the
 * same numbering (vglb_varray_reorder_u32) and only the verdict comes back.
 *   vglb_verify_i32 / _f32       verify_results (:33-93): the `error count` of elements that are not are_same (:9-28: exact for
 *                                int, |a - b| <= 100 * FLT_EPSILON for float)
 *   vglb_verify_ranking_f32      verify_ranking_results (:97-148): mean |a - ref| (error_count = n unless it is < 1e-4), plus the
 *                                relative L1 distance sum|a - ref| / sum|ref| that the parity bar of this backend is stated in
 *   vglb_verify_components_i32   equal_components (:198-254): the two label arrays describe the same partition (labels in [0, n + 1]) */
int vglb_verify_i32(vglb_ctx *ctx, const int32_t *d_a, const int32_t *d_b, int64_t n, int64_t *error_count);
int vglb_verify_f32(vglb_ctx *ctx, const float *d_a, const float *d_b, int64_t n, int64_t *error_count);
int vglb_verify_ranking_f32(vglb_ctx *ctx, const float *d_a, const float *d_ref, int64_t n, double *mean_abs_difference,
                            double *relative_l1, int64_t *error_count);
int vglb_verify_components_i32(vglb_ctx *ctx, const int32_t *d_a, const int32_t *d_b, int32_t n, int64_t *error_count);

/* ---- multi-GPU: one process per GPU, 1D vertex partition, NCCL over NVLink ----------------------------------------
 * Reference: the MPI layer of the NEC backend — vgl_mpi_init (vgl_runtime/helpers/library_data/init.hpp:5-38), the
 * per-rank vertex ranges (vect_csr/mpi_api.hpp:6-26, get_api.hpp:66-94) and exchange_vertices_array
 * (vgl_compute_api/common/mpi_exchange.hpp:155-271). Here the GRAPH is partitioned too (the reference replicates it):
 * the degree-sorted ids s = 0..V-1 are dealt round-robin, owner(s) = s mod P, local row = s div P, so every rank owns
 * a degree-sorted slice with ~V/P rows and ~E/P edges (hubs are spread over all ranks). Vertex state is replicated
 * and indexed by COLUMN id = owner * rows_per_rank + local row; each rank computes the slice it owns and exchanges once
 * per iteration: PageRank contributions are stored into the peers' vectors by the sweep itself (CUDA IPC peer memory) or
 * allgathered; top-down BFS discoveries and SSSP distance updates travel as per-owner lists that the owners read out of
 * the peers' memory; bottom-up BFS allgathers frontier-bitmap slices; CC allreduces (min) the label vector; a small
 * allreduce of counters closes every iteration. Without CUDA IPC everything falls back to NCCL collectives. vglb_pagerank / vglb_bfs / vglb_sssp / vglb_cc accept a partitioned graph: vertex
 * outputs then hold THIS RANK's rows (info.vertices entries), `source_sorted` is a column id, and every rank must
 * make the same call (they are collectives). */
typedef struct vglb_comm vglb_comm;
#define VGLB_UNIQUE_ID_BYTES 128
int vglb_comm_unique_id(void *out_id /* VGLB_UNIQUE_ID_BYTES */);
int vglb_comm_init(vglb_ctx *ctx, int rank, int world, const void *unique_id, vglb_comm **out);
/* carries (rank, world) only — builds / inspects any rank's part in one process; collectives on it fail (VGLB_ENCCL) */
int vglb_comm_init_detached(vglb_ctx *ctx, int rank, int world, vglb_comm **out);
int vglb_comm_destroy(vglb_comm *comm);
int vglb_comm_barrier(vglb_comm *comm);
/* exchange_vertices_array: in-place allgather of equal slices of a device array (slice r at offset r*bytes_per_rank) */
int vglb_comm_allgather(vglb_comm *comm, void *d_buf, size_t bytes_per_rank);
int vglb_comm_allreduce_sum_i64(vglb_comm *comm, int64_t *d_buf, int count);
int vglb_comm_allreduce_max_f64(vglb_comm *comm, double *h_value); /* host scalar, e.g. max-over-ranks timings */

/* Build THIS RANK's part of the graph. Every rank passes the same edge list (host or device pointers) or the same
 * generator arguments; edges are streamed in chunks twice (degree pass, then a pass that keeps the owned rows), so
 * device memory is O(E/P + V) and E may exceed 2^31. symmetrize != 0 appends the reversed copy of every edge (CC).
 * flags: VGLB_GRAPH_WITH_INCOMING. Rows list their neighbours hubs-first. */
int vglb_graph_from_edges_partitioned(vglb_ctx *ctx, vglb_comm *comm, int32_t vertices, int64_t edges,
                                      const int32_t *src, const int32_t *dst, int src_on_device, int symmetrize,
                                      int flags, vglb_graph **out_graph);
int vglb_graph_from_generator_partitioned(vglb_ctx *ctx, vglb_comm *comm, int kind, int scale, int64_t edges,
                                          uint64_t seed, int a, int b, int c, int symmetrize, int flags,
                                          vglb_graph **out_graph);
/* VGL_Graph::move_to_device for one rank's part: host arrays of an already-built part (row pointers of this rank's
 * `rows` rows, adjacency in column ids, ORIGINAL -> column map of the whole graph) copied to HBM. A collective when
 * the communicator is live (edge totals are allreduced). */
int vglb_graph_from_csr_partitioned(vglb_ctx *ctx, vglb_comm *comm, int32_t vertices_global, int32_t rows,
                                    const int64_t *h_out_ptr, const int32_t *h_out_adj, const int32_t *h_orig_to_col,
                                    const int64_t *h_in_ptr, const int32_t *h_in_adj, vglb_graph **out_graph);
/* PageRank exchange on a partitioned graph: 0 = ncclAllGather after every sweep; 1 = the sweep's epilogue stores each
 * contribution straight into every peer's copy of the vector over NVLink (CUDA IPC peer memory), and the dangling-mass
 * allreduce doubles as the inter-sweep barrier. */
#define VGLB_EXCHANGE_NCCL 0
#define VGLB_EXCHANGE_P2P 1
int vglb_graph_set_exchange(vglb_ctx *ctx, vglb_graph *g, int mode);

#ifdef __cplusplus
}
#endif
#endif /* VGL_B200_H */
