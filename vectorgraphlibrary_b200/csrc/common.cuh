// common.cuh — internal declarations shared by the libvgl_b200 translation units (not part of the C ABI).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "vgl_b200.h"
#include "vglb_synth.h"

#define VGLB_SM_COUNT_B200 148

void vglb_set_error(const char *fmt, ...);

// cached device allocations (context.cu); drop-in for cudaMalloc / cudaFree inside the library
cudaError_t vglb_dev_alloc_bytes(void **ptr, size_t bytes);
void vglb_dev_free(void *ptr);
void vglb_dev_mark_exported(void *ptr); // the block is visible to other processes (CUDA IPC): free it for real
void vglb_dev_cache_release(void);
template <class T>
static inline cudaError_t vglb_dev_alloc(T **ptr, size_t bytes)
{
    return vglb_dev_alloc_bytes((void **)ptr, bytes);
}

// SAFE_CALL twin (cuda_error_handling.h:7-13): record the message and return an error code instead of throwing.
#define CUDA_TRY(call)                                                                               \
    do                                                                                               \
    {                                                                                                \
        cudaError_t err__ = (call);                                                                  \
        if (err__ != cudaSuccess)                                                                    \
        {                                                                                            \
            vglb_set_error("CUDA error %s at %s:%d (%s)", cudaGetErrorString(err__), __FILE__,       \
                           __LINE__, #call);                                                         \
            return VGLB_ECUDA;                                                                       \
        }                                                                                            \
    } while (0)

#define KERNEL_TRY() CUDA_TRY(cudaGetLastError())

#define VGLB_REQUIRE(cond, msg)                                       \
    do                                                                \
    {                                                                 \
        if (!(cond))                                                  \
        {                                                             \
            vglb_set_error("%s (%s:%d)", msg, __FILE__, __LINE__);    \
            return VGLB_EINVAL;                                       \
        }                                                             \
    } while (0)

struct vglb_ctx
{
    int device;
    int sm_count;
    size_t l2_bytes;
    cudaStream_t stream;
    cudaStream_t copy_stream;   // host -> device uploads that overlap kernels on `stream` (vglb_graph_from_csr)
    cudaEvent_t ev_chunk[8];
    cudaEvent_t ev_start, ev_stop;
    // host-visible scratch for counters read back once per level / round
    int64_t *h_counters;   // pinned, 64 x int64
    int64_t *d_counters;   // device, 64 x int64
    void *d_flush;         // L2 flush buffer
    size_t flush_bytes;
    int64_t launches;      // kernels launched since the last reset (gpu_launches evidence)
    // counter mailbox: pinned host memory mapped into the device; a 1-warp kernel at the end of a round copies the round's
    // counters there and raises a sequence number the host spins on (vglb_counters_fetch) — a level / round boundary costs a
    // PCIe write instead of cudaMemcpyAsync + cudaStreamSynchronize
    unsigned long long *h_mailbox; // 64 words, word 63 = sequence number
    unsigned long long mailbox_seq;
    int pr_carveout_set;   // the PageRank sweep kernels' shared-memory carve-out preferences have been set on this device
    int upload_hint;       // VGLB_HINT_* (vglb_set_upload_hint)
    int prb_smem_set;      // pr_bin_kernel's dynamic shared-memory limit has been raised on this device
};

struct vglb_graph
{
    int32_t V;
    int64_t E;
    int32_t max_degree;
    int64_t *d_out_ptr;
    int32_t *d_out_adj;
    int64_t *d_in_ptr;
    int32_t *d_in_adj;
    int32_t *d_fwd; // orig -> sorted
    int32_t *d_bwd; // sorted -> orig
    int64_t *d_edge_order;
    uint32_t *d_in_to_out_pos; // incoming-CSR position -> outgoing-CSR position of the same edge (verify.cu, built on first use)
    int32_t tier_degree[VGLB_NUM_TIERS];
    int32_t tier_border[VGLB_NUM_TIERS];
    // lazily created per-algorithm state (owned by the graph, freed with it)
    int32_t *d_indeg_noloops; // in-degree without self loops, counted while the adjacency is uploaded (vglb_graph_from_csr)
    float *d_pr_inv;       // 1/indeg_noloops (0 when none), SCATTER numbering
    float *d_pr_contrib[2];
    double *d_pr_dangling; // one slot per sweep
    int pr_dangling_slots;
    void *d_pr_tasks;           // warp-task table of the PageRank sweep (pagerank.cu)
    float *d_pr_piece_partial;  // partial sums of the pieces of long rows
    int32_t *d_pr_piece_count;  // arrival counters of the long rows
    int32_t pr_ntasks;
    int32_t *d_pr_ve_adj;       // padded column-major copy of the rows with 1..31 edges (VectorExtension twin)
    int64_t *d_pr_ve_ptr;
    int32_t pr_ve_segments;
    void *pr_bins;              // column-binned copy of the heavy rows (PrBins, pagerank_bins.cu); NULL = warp tasks
    int pr_bins_tried;
    int pr_zero_ready;          // pr_zero_kept / pr_zero_dangling are counted (one GPU; PrParams::zero_kept)
    int32_t pr_zero_kept;
    int32_t pr_zero_dangling;
    int32_t col_of_row0;        // column id of local row 0 (0 unless the graph is one rank's part of a partitioned graph)
    // 1D partition (partition.cu). On one GPU: cols = V_orig = vp = V, E_global = E, comm = NULL.
    // On a partitioned graph V / E are this rank's rows / edges; vertex state is indexed by COLUMN id in [0, cols):
    // column = owner * vp + local row; d_fwd maps ORIGINAL id -> column, d_bwd column -> ORIGINAL id (-1 = padding).
    struct vglb_comm *comm;
    int32_t part_rank, part_world;
    int32_t vp;                 // rows per rank (slice stride, a multiple of 32)
    int32_t V_orig;             // vertices of the whole graph
    int64_t cols;               // part_world * vp
    int64_t E_global;
    // partitioned-algorithm scratch (owned by the graph)
    uint32_t *d_part_bm[3];     // full-length bitmaps: visited, candidates / current frontier, next frontier
    uint32_t *d_part_stage;     // part_world received bitmap slices
    uint32_t *d_part_vec;       // full-length 4-byte vertex state (dist / labels)
    uint32_t *d_part_prev;      // this rank's slice of the previous round's state
    // PageRank peer-store exchange: the peers' copies of the two contribution vectors (CUDA IPC mappings)
    int pr_exchange;            // VGLB_EXCHANGE_NCCL | VGLB_EXCHANGE_P2P
    float *d_pr_peer[2][8];     // [buffer][peer rank]; NULL for this rank
    void *d_part_lists;         // SSSP: per-owner lists of (column, distance) updates this rank produced in a round
    uint32_t *d_vec_peer[8];    // the peers' d_part_lists, CUDA IPC mappings (own entry = own buffer)
    int vec_peers_mapped;       // 0 = not tried, 1 = mapped, -1 = mapping failed (dense allreduce exchange is used)
    int borrowed_csr;           // d_out_ptr / d_out_adj belong to the caller (vglb_graph_borrow_csr): never freed here
    int ipc_exported;           // buffers of this graph were offered to the peers over CUDA IPC: vglb_graph_free is a collective
    // BFS / SSSP / CC scratch
    uint32_t *d_visited, *d_front_bm[2];
    int32_t *d_queue[2];
    int32_t *d_scratch_i32;
    int32_t sssp_mid_rows_per_warp; // queue entries of the mid tier per warp (~2048 edges), set with the border
    int64_t cc_hub_edges_plus1;    // 0 = not read yet; else 1 + row pointer at tier_border[0] (cc.cu)
    int32_t bfs_big_border_plus1;  // 0 = not computed yet; else 1 + first id with fewer than BFS_BIG_DEGREE edges (bfs.cu)
    int32_t sssp_big_border_plus1; // 0 = not computed yet; else 1 + first id with fewer than 512 edges (sssp.cu)
};

// NCCL communicator of one rank (partition.cu); the library dlopen()s libnccl.so.2 on first use
struct vglb_comm
{
    void *nccl;        // ncclComm_t
    int rank, world;
    vglb_ctx *ctx;
};

struct vglb_frontier
{
    vglb_graph *g;
    int32_t sparsity_type;
    int32_t size;
    int64_t neighbours;
    int32_t tier_size[3];
    int32_t *d_ids;
    int borrowed_ids;      // d_ids belongs to the caller (vglb_frontier_create_borrowed)
    uint32_t *d_bitmap;
    void *d_tile_status;   // [8 counters][one look-back status word per GNF tile]
    int64_t tiles;
};

// degree thresholds of the tiers: tier t holds rows with degree in [tier_degree[t], tier_degree[t-1]).
// CTA per row | warp per row | 16 | 8 | 4 | 2 lanes per row | 1 lane per row (degree 1) | degree 0
#ifdef __CUDACC__
__host__ __device__
#endif
constexpr int32_t vglb_tier_degree(int t)
{
    return t == 0 ? 4096 : t == 1 ? 32 : t == 2 ? 16 : t == 3 ? 8 : t == 4 ? 4 : t == 5 ? 2 : t == 6 ? 1 : 0;
}

// copy `words` (<= 56) 8-byte counters from device memory to ctx->h_counters, ordered after everything enqueued on ctx->stream
int vglb_counters_fetch(vglb_ctx *ctx, const void *d_src, int words);
// end of a run timed from ctx->ev_start: records ev_stop on ctx->stream and waits for it; with stats, zeroes *stats and fills in
// seconds and kernel_launches (launches since launches0). The algorithm fills in its own fields.
int vglb_finish_run(vglb_ctx *ctx, int64_t launches0, vglb_stats *stats);
int vglb_graph_compute_tiers(vglb_ctx *ctx, vglb_graph *g);
void vglb_graph_set_unpartitioned(vglb_graph *g);
int vglb_graph_derive_incoming(vglb_ctx *ctx, vglb_graph *g);
int vglb_pr_build_tasks_host(vglb_ctx *ctx, vglb_graph *g, const int64_t *h_ptr, int32_t heavy_rows, int32_t long_rows);
void vglb_graph_free_fields(vglb_graph *g);
void vglb_pr_bins_free(vglb_graph *g);   // pagerank_bins.cu
int vglb_pr_bins_build_rows(vglb_ctx *ctx, vglb_graph *g, int32_t rows); // rows = ids with >= 32 edges (tier_border[1])
int vglb_pr_bins_wanted(const vglb_graph *g); // 1: the PageRank sweep of this graph uses the column-binned heavy rows

// collectives on the context stream (partition.cu); asynchronous, every rank must make the same call
enum { VGLB_DT_I32 = 0, VGLB_DT_U32 = 1, VGLB_DT_I64 = 2, VGLB_DT_F64 = 3 };
enum { VGLB_OP_SUM = 0, VGLB_OP_MIN = 1, VGLB_OP_MAX = 2 };
int vglb_comm_allgather_async(vglb_comm *comm, void *d_buf, size_t bytes_per_rank);
int vglb_comm_allreduce_async(vglb_comm *comm, void *d_buf, size_t count, int dtype, int op);
int vglb_comm_alltoall_async(vglb_comm *comm, const void *d_send, void *d_recv, size_t bytes_per_rank);
int vglb_comm_ipc_map(vglb_comm *comm, void *d_local, void **peers /* [world] */);
int vglb_part_map_lists(vglb_ctx *ctx, vglb_graph *g);

static inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }

#ifdef __CUDACC__
// ---- device helpers -------------------------------------------------------------------------------------------

// L2 eviction policies (sm_100a accepts the bare .L2::evict_* qualifier only on 256-bit loads, so 32/128-bit loads
// carry a createpolicy descriptor through .L2::cache_hint).
__device__ __forceinline__ uint64_t l2_policy_evict_first()
{
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_last()
{
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    return p;
}
// streaming loads of CSR column indices / weights: read once, keep out of L1 and first to leave L2
__device__ __forceinline__ int4 ld_stream_v4(const int4 *p, uint64_t pol)
{
    int4 r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.s32 {%0,%1,%2,%3}, [%4], %5;"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p), "l"(pol));
    return r;
}
__device__ __forceinline__ int ld_stream_s32(const int *p, uint64_t pol)
{
    int r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.s32 %0, [%1], %2;" : "=r"(r) : "l"(p), "l"(pol));
    return r;
}
__device__ __forceinline__ float ld_stream_f32(const float *p, uint64_t pol)
{
    float r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.f32 %0, [%1], %2;" : "=f"(r) : "l"(p), "l"(pol));
    return r;
}
// gathered vertex value: random 4-byte reads of a V-sized vector that should stay L2-resident (L1 allocating)
__device__ __forceinline__ float ld_gather_f32(const float *p, uint64_t pol)
{
    float r;
    asm volatile("ld.global.nc.L2::cache_hint.f32 %0, [%1], %2;" : "=f"(r) : "l"(p), "l"(pol));
    return r;
}
__device__ __forceinline__ int ld_gather_s32(const int *p, uint64_t pol)
{
    int r;
    asm volatile("ld.global.nc.L2::cache_hint.s32 %0, [%1], %2;" : "=r"(r) : "l"(p), "l"(pol));
    return r;
}

// gathered value that is unlikely to be re-used by this SM: do not let it push hot lines out of L1
__device__ __forceinline__ float ld_gather_cold_f32(const float *p, uint64_t pol)
{
    float r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.f32 %0, [%1], %2;" : "=f"(r) : "l"(p), "l"(pol));
    return r;
}
// streaming stores of per-vertex results (written once per sweep, read by the next kernel)
__device__ __forceinline__ void st_stream_f32(float *p, float v)
{
    asm volatile("st.global.L1::no_allocate.f32 [%0], %1;" ::"l"(p), "f"(v) : "memory");
}

__device__ __forceinline__ float warp_sum_f32(float v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum_f64(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ long long warp_sum_i64(long long v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ int lane_id() { return threadIdx.x & 31; }
#endif
