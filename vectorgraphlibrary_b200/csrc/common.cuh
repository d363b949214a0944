// common.cuh — internal declarations shared by the libvgl_b200 translation units (not part of the C ABI).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <memory>

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

// Owning handle of a block from the cache: the block goes back on every exit of the scope that holds it. release() hands it
// over to a graph or PrBins field; reset() frees it early.
struct vglb_dev_deleter
{
    void operator()(void *p) const { vglb_dev_free(p); }
};
template <class T>
using dev_ptr = std::unique_ptr<T, vglb_dev_deleter>;
// (a block the handle already holds goes back first, as a vglb_dev_free before the allocation would)
template <class T>
static inline cudaError_t vglb_dev_alloc(dev_ptr<T> &p, size_t bytes)
{
    p.reset();
    T *raw = NULL;
    const cudaError_t e = vglb_dev_alloc(&raw, bytes);
    if (e == cudaSuccess) p.reset(raw);
    return e;
}

// SAFE_CALL twin (cuda_error_handling.h:7-13): record the message and return an error code instead of throwing. The
// runtime's last error is cleared, so a failed allocation is reported once, as VGLB_ENOMEM.
#define CUDA_TRY(call)                                                                               \
    do                                                                                               \
    {                                                                                                \
        cudaError_t err__ = (call);                                                                  \
        if (err__ != cudaSuccess)                                                                    \
        {                                                                                            \
            cudaGetLastError();                                                                      \
            vglb_set_error("CUDA error %s at %s:%d (%s)", cudaGetErrorString(err__), __FILE__,       \
                           __LINE__, #call);                                                         \
            return err__ == cudaErrorMemoryAllocation ? VGLB_ENOMEM : VGLB_ECUDA;                    \
        }                                                                                            \
    } while (0)

#define KERNEL_TRY() CUDA_TRY(cudaGetLastError())

// a library call that returns a VGLB_* code
#define VGLB_TRY(call)                \
    do                                \
    {                                 \
        const int rc__ = (call);      \
        if (rc__ != VGLB_OK)          \
            return rc__;              \
    } while (0)

// A two-phase CUB call run(d_temp, bytes): asks for the size of its temporary, takes that from the cache into `tmp` and runs
// it. Nothing is synchronised; the caller decides when `tmp` goes back (the cache orders its re-use after the call).
template <class Run>
static inline cudaError_t vglb_cub(dev_ptr<void> &tmp, Run &&run)
{
    size_t bytes = 0;
    cudaError_t e = run(nullptr, bytes);
    if (e == cudaSuccess) e = vglb_dev_alloc(tmp, bytes);
    return e == cudaSuccess ? run(tmp.get(), bytes) : e;
}

// bits of a radix-sort key that holds the values [0, n): at least 1, at most 32
static inline int vglb_key_bits(int64_t n)
{
    int b = 1;
    while (b < 32 && ((int64_t)1 << b) < n) b++;
    return b;
}

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
    // host-visible scratch for counters read back once per level / round (layout: CTR_* below)
    int64_t *h_counters;   // pinned, CTR_WORDS x int64
    int64_t *d_counters;   // device, CTR_WORDS x int64
    void *d_flush;         // L2 flush buffer
    size_t flush_bytes;
    int64_t launches;      // kernels launched since the last reset (gpu_launches evidence)
    // counter mailbox: pinned host memory mapped into the device; a 1-warp kernel at the end of a round copies the round's
    // counters there and raises a sequence number the host spins on (vglb_counters_fetch) — a level / round boundary costs a
    // PCIe write instead of cudaMemcpyAsync + cudaStreamSynchronize
    unsigned long long *h_mailbox; // CTR_WORDS words, word MAILBOX_SEQ = sequence number
    unsigned long long mailbox_seq;
    int pr_carveout_set;   // the PageRank sweep kernels' shared-memory carve-out preferences have been set on this device
    int upload_hint;       // VGLB_HINT_* (vglb_set_upload_hint)
    int prb_smem_set;      // pr_bin_kernel's dynamic shared-memory limit has been raised on this device
};

// The words (8 bytes each) of the counter block ctx->d_counters and its pinned host copy ctx->h_counters. Every user of the
// block names its words here; a word without a name is free. Two names on one word are users that never run together.
enum
{
    // level / round counters of BFS, multi-source BFS and SSSP (u64): the level's kernels add to them, the driver clears
    // them before the first level and again after each read-back
    C_NEXT_BIG = 0,   // rows queued for the next level, per tier
    C_NEXT_MID = 1,
    C_NEXT_SMALL = 2,
    C_EDGES = 3,      // edges inspected this level
    C_FOUND = 4,      // vertices discovered this level
    C_MF = 5,         // sum of out-degrees of the next frontier
    C_ROWS = 6,       // rows whose pointer pair was read this level
    C_COUNT = 8,
    // int32 scratch of graph set-up (the tier borders of vglb_graph_compute_tiers, the vertex of
    // vglb_graph_threshold_vertex): used outside any run only, so it shares the level counters; both zero it again
    // afterwards, because a run expects its counters at 0
    CTR_SCRATCH_I32 = 0,
    // a partitioned level's counters, copied by the staging kernel and summed over the ranks (vglb_part_round_counters)
    C_STAGED = C_COUNT,
    // multi-source BFS level counters (u64). vglb_bfs_multi rejects partitioned graphs, so they share the staged copy
    M_PAIRS = C_STAGED,     // (vertex, source) pairs reached this level = level stores
    M_FULL = M_PAIRS + 1,   // vertices whose seen word became full this level
    M_COUNT = M_FULL + 1,
    // SSSP: complement of this rank's smallest pending distance (u64), C_MF copied by the staging kernel every round
    CTR_PENDING_MIN = C_STAGED + C_COUNT,
    CTR_SSSP_ROUND = CTR_PENDING_MIN + 1, // words an SSSP round reads back
    // partitioned BFS / SSSP: one-word allreduce that is the barrier of the discovery / update list exchange (value unused)
    CTR_LIST_BARRIER = CTR_PENDING_MIN + 2,
    // SSSP drain results (u64, written by sssp_drain_kernel). The drain never runs on a partitioned graph, so DR_REASON
    // shares the list barrier
    DR_REASON = CTR_LIST_BARRIER,
    DR_ROUNDS,
    DR_ROWS,
    DR_END,
    // partitioned BFS / SSSP: the peers' update lists (g->d_vec_peer, 8 device pointers), copied in before the run
    CTR_PEER_TABLE = 24,
    CTR_REDUCE = 32,         // vglb_reduce_*: the frontier reduce result (i64 or f64)
    CTR_CC_CHANGED = 40,     // CC: a hook changed a label this round (int32, device and host)
    // triangle counting (u64, tc.cu): cleared at the start of vglb_tc, read back once at its end
    CTR_TC_TOTAL = 41,       // triangles (row sums of tc_count_kernel)
    CTR_TC_UNIQUE = 42,      // distinct keys of the oriented-CSR build (the self-loop key included)
    CTR_TC_EDGES = 43,       // E+: edges of the oriented CSR
    CTR_TC_ROWS = 44,        // rows of the oriented CSR with at least one entry
    CTR_TC_ELEMENTS = 45,    // list elements the intersections read
    CTR_TC_END = 46,
    CTR_HOST_ALLREDUCE = 52, // vglb_comm_allreduce_host: up to two 8-byte host values on their way through the allreduce
    CTR_BAD = 56,            // CSR / label validation: a check failed (int32)
    CTR_VERIFY_COUNT = 57,   // vglb_verify_*: mismatches (u64)
    CTR_VERIFY_SUMS = 58,    // vglb_verify_ranking_f32: two f64 sums
    CTR_SSSP_WMAX = 60,      // SSSP: the largest sampled weight (u32 bits of a float)
    CTR_WORDS = 64,          // size of the block, and of the mailbox
    MAILBOX_WORDS = 56,      // vglb_counters_fetch copies at most this many words
    MAILBOX_SEQ = 63         // mailbox word that carries the sequence number
};
static_assert(DR_END <= CTR_PEER_TABLE && CTR_REDUCE < CTR_CC_CHANGED && CTR_CC_CHANGED < CTR_TC_TOTAL &&
                  CTR_TC_END <= CTR_HOST_ALLREDUCE &&
                  CTR_HOST_ALLREDUCE + 2 <= CTR_BAD && CTR_VERIFY_SUMS + 2 <= CTR_SSSP_WMAX && CTR_SSSP_WMAX < CTR_WORDS &&
                  MAILBOX_WORDS < MAILBOX_SEQ && MAILBOX_SEQ < CTR_WORDS,
              "counter slots in order, each inside the block");
static_assert(C_COUNT <= MAILBOX_WORDS && CTR_SSSP_ROUND <= MAILBOX_WORDS && DR_END <= MAILBOX_WORDS && M_COUNT <= MAILBOX_WORDS &&
                  CTR_TC_END <= MAILBOX_WORDS,
              "every run read through the mailbox fits it");

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
static_assert(sizeof(vglb_graph::d_vec_peer) <= (CTR_REDUCE - CTR_PEER_TABLE) * 8, "the peer table holds d_vec_peer");

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

// copy `words` (<= MAILBOX_WORDS) 8-byte counters from device memory to ctx->h_counters, ordered after everything enqueued on ctx->stream
int vglb_counters_fetch(vglb_ctx *ctx, const void *d_src, int words);
// end of a run timed from ctx->ev_start: records ev_stop on ctx->stream and waits for it; with stats, zeroes *stats and fills in
// seconds and kernel_launches (launches since launches0). The algorithm fills in its own fields.
int vglb_finish_run(vglb_ctx *ctx, int64_t launches0, vglb_stats *stats);
int vglb_graph_compute_tiers(vglb_ctx *ctx, vglb_graph *g);
void vglb_graph_set_unpartitioned(vglb_graph *g);
int vglb_graph_derive_incoming(vglb_ctx *ctx, vglb_graph *g);
int vglb_pr_build_tasks_host(vglb_ctx *ctx, vglb_graph *g, const int64_t *h_ptr, int32_t heavy_rows, int32_t long_rows);
void vglb_graph_free_fields(vglb_graph *g);
// owner of a graph that is still being built: its fields and the struct go back unless it is released into *out_graph
struct vglb_graph_deleter
{
    void operator()(vglb_graph *g) const
    {
        vglb_graph_free_fields(g);
        free(g);
    }
};
using graph_ptr = std::unique_ptr<vglb_graph, vglb_graph_deleter>;
static inline graph_ptr vglb_graph_new() { return graph_ptr((vglb_graph *)calloc(1, sizeof(vglb_graph))); }

// checks of caller-supplied construction input (graph_build.cu); a failed check sets the CTR_BAD word, which the caller
// clears before and reads back after
// row pointers d_ptr[0..rows] from 0 to E, non-decreasing, and the E ids of d_adj in [0, id_limit)
int vglb_csr_validate_device(vglb_ctx *ctx, const int64_t *d_ptr, int32_t rows, int64_t E, const int32_t *d_adj, int64_t id_limit);
// bwd[fwd[i]] = i for i in [0, n); bwd must be filled with -1, and every fwd[i] must be a distinct value in [0, limit)
int vglb_invert_map_checked(vglb_ctx *ctx, const int32_t *d_fwd, int32_t n, int64_t limit, int32_t *d_bwd);
// the ids [0, V) stably sorted by degree descending (ties by ascending id, the reference's std::stable_sort): `sorted`
// points into ids[]. The buffers go back when the struct does.
struct DegreeOrder
{
    dev_ptr<uint32_t> keys[2], ids[2];
    dev_ptr<void> tmp;
    const uint32_t *sorted = nullptr;
};
int vglb_degree_order(vglb_ctx *ctx, const int32_t *d_deg, int32_t V, DegreeOrder &order);
void vglb_pr_bins_free(vglb_graph *g);   // pagerank_bins.cu
int vglb_pr_bins_build_rows(vglb_ctx *ctx, vglb_graph *g, int32_t rows); // rows = ids with >= 32 edges (tier_border[1])
int vglb_pr_bins_wanted(const vglb_graph *g); // 1: the PageRank sweep of this graph uses the column-binned heavy rows

// collectives on the context stream (partition.cu); asynchronous, every rank must make the same call
enum { VGLB_DT_I32 = 0, VGLB_DT_U32 = 1, VGLB_DT_I64 = 2, VGLB_DT_F64 = 3 };
enum { VGLB_OP_SUM = 0, VGLB_OP_MIN = 1, VGLB_OP_MAX = 2 };
int vglb_comm_allgather_async(vglb_comm *comm, void *d_buf, size_t bytes_per_rank);
int vglb_comm_allreduce_async(vglb_comm *comm, void *d_buf, size_t count, int dtype, int op);
// allreduce of `count` host values (at most 16 bytes) through CTR_HOST_ALLREDUCE; waits, and leaves the result in h_inout
int vglb_comm_allreduce_host(vglb_comm *comm, void *h_inout, int count, int dtype, int op);
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
