// partition.cu — multi-GPU plumbing of libvgl_b200: the NCCL communicator of one rank (one process per GPU) and the
// builder of ONE RANK's part of a 1D-partitioned device VectCSR.
//
// Reference: the MPI layer of the NEC backend. vgl_mpi_init (vgl_runtime/helpers/library_data/init.hpp:5-38) gives every
// rank the WHOLE graph plus a vertex range per degree tier (vect_csr/mpi_api.hpp:6-26, get_api.hpp:66-94), and
// exchange_vertices_array (vgl_compute_api/common/mpi_exchange.hpp:155-271) circulates whole vertex arrays after
// every operator. B200 design: the graph itself is partitioned (HBM per GPU is O(E/P + V)), vertex state is
// replicated, and one NCCL collective per iteration moves only the owned slices over NVLink 5 / NVSwitch.
//
// Partition: the reference's degree-sorted ids s = 0..V-1 (sort_vertices_by_degree, vect_csr/import.hpp:61-99) are
// dealt round-robin: owner(s) = s mod P, local row = s div P. Every rank therefore owns a degree-sorted slice (tiers
// stay contiguous local row ranges) with ~V/P rows and ~E/P edges, hubs spread over all ranks — the contiguous ranges
// of the reference would put every hub on rank 0. Replicated vertex arrays are indexed by COLUMN id
//     column(s) = (s mod P) * vp + s div P,      vp = rows per rank rounded up to a multiple of 32,
// so the slice a rank owns is contiguous (equal-size slices => plain ncclAllGather) and bitmap slices are whole words.
//
// Build (setup, outside every timed region): the edge list — generator arguments, device arrays or host arrays, the
// same on every rank — is streamed in chunks twice: pass 1 counts degrees of ALL vertices (every rank computes the same
// global numbering, no communication), pass 2 keeps the edges whose row this rank owns as 64-bit keys
// (local row << 32 | sorted id of the neighbour), one radix sort per direction turns them into CSR rows that list their
// neighbours hubs-first. The order of a row's neighbours does not change any result (BFS levels, min-plus distances
// and min labels are order-free; PageRank row sums are within the 1e-6 tolerance either way).
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <dlfcn.h>
#include <nccl.h>
#include <stdlib.h>

#include "common.cuh"

// ---- NCCL through dlopen: the single-GPU library has no link-time dependency on NCCL, and inside a process that
//      already loaded a libnccl.so.2 (torch's bundled copy) the same instance is reused --------------------------------
namespace
{
struct NcclApi
{
    void *handle;
    ncclResult_t (*GetUniqueId)(ncclUniqueId *);
    ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int);
    ncclResult_t (*CommDestroy)(ncclComm_t);
    ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t);
    ncclResult_t (*AllReduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t);
    ncclResult_t (*Send)(const void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t);
    ncclResult_t (*Recv)(void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t);
    ncclResult_t (*GroupStart)();
    ncclResult_t (*GroupEnd)();
    const char *(*GetErrorString)(ncclResult_t);
};

NcclApi *nccl_api()
{
    static NcclApi api;
    static int state = 0; // 0 = not tried, 1 = ok, -1 = failed
    if (state == 0)
    {
        const char *names[] = {"libnccl.so.2", "libnccl.so", NULL};
        for (int i = 0; names[i] && !api.handle; i++) api.handle = dlopen(names[i], RTLD_NOW | RTLD_GLOBAL);
        if (!api.handle)
        {
            vglb_set_error("NCCL is not loadable (dlopen libnccl.so.2: %s)", dlerror());
            state = -1;
            return NULL;
        }
#define LOAD(field, sym)                                                            \
    *(void **)(&api.field) = dlsym(api.handle, sym);                               \
    if (!api.field)                                                                 \
    {                                                                               \
        vglb_set_error("NCCL symbol %s not found", sym);                            \
        state = -1;                                                                 \
        return NULL;                                                                \
    }
        LOAD(GetUniqueId, "ncclGetUniqueId")
        LOAD(CommInitRank, "ncclCommInitRank")
        LOAD(CommDestroy, "ncclCommDestroy")
        LOAD(AllGather, "ncclAllGather")
        LOAD(AllReduce, "ncclAllReduce")
        LOAD(Send, "ncclSend")
        LOAD(Recv, "ncclRecv")
        LOAD(GroupStart, "ncclGroupStart")
        LOAD(GroupEnd, "ncclGroupEnd")
        LOAD(GetErrorString, "ncclGetErrorString")
#undef LOAD
        state = 1;
    }
    return state == 1 ? &api : NULL;
}
} // namespace

#define NCCL_TRY(call)                                                                                       \
    do                                                                                                       \
    {                                                                                                        \
        ncclResult_t r__ = (call);                                                                           \
        if (r__ != ncclSuccess)                                                                              \
        {                                                                                                    \
            vglb_set_error("NCCL error %s at %s:%d (%s)", nccl_api()->GetErrorString(r__), __FILE__, __LINE__, \
                           #call);                                                                           \
            return VGLB_ENCCL;                                                                               \
        }                                                                                                    \
    } while (0)

#define DETACHED_CHECK(comm)                                                                    \
    do                                                                                          \
    {                                                                                           \
        if (!(comm)->nccl)                                                                      \
        {                                                                                       \
            vglb_set_error("collective on a detached communicator (vglb_comm_init_detached)");  \
            return VGLB_ENCCL;                                                                  \
        }                                                                                       \
    } while (0)

extern "C" int vglb_comm_unique_id(void *out_id)
{
    VGLB_REQUIRE(out_id != NULL, "vglb_comm_unique_id: NULL argument");
    static_assert(sizeof(ncclUniqueId) <= VGLB_UNIQUE_ID_BYTES, "unique id size");
    NcclApi *N = nccl_api();
    if (!N) return VGLB_ENCCL;
    ncclUniqueId id;
    NCCL_TRY(N->GetUniqueId(&id));
    memset(out_id, 0, VGLB_UNIQUE_ID_BYTES);
    memcpy(out_id, &id, sizeof(id));
    return VGLB_OK;
}

extern "C" int vglb_comm_init(vglb_ctx *ctx, int rank, int world, const void *unique_id, vglb_comm **out)
{
    VGLB_REQUIRE(ctx != NULL && unique_id != NULL && out != NULL, "vglb_comm_init: NULL argument");
    VGLB_REQUIRE(world >= 1 && world <= 64 && rank >= 0 && rank < world, "vglb_comm_init: bad rank / world");
    NcclApi *N = nccl_api();
    if (!N) return VGLB_ENCCL;
    CUDA_TRY(cudaSetDevice(ctx->device));
    ncclUniqueId id;
    memcpy(&id, unique_id, sizeof(id));
    ncclComm_t c;
    NCCL_TRY(N->CommInitRank(&c, world, id, rank));
    vglb_comm *comm = (vglb_comm *)calloc(1, sizeof(vglb_comm));
    if (!comm) return VGLB_ENOMEM;
    comm->nccl = (void *)c;
    comm->rank = rank;
    comm->world = world;
    comm->ctx = ctx;
    *out = comm;
    return VGLB_OK;
}

// a communicator that only carries (rank, world): lets one process build / inspect any rank's part of a graph
// (tests, offline partitioning). Collectives on it fail.
extern "C" int vglb_comm_init_detached(vglb_ctx *ctx, int rank, int world, vglb_comm **out)
{
    VGLB_REQUIRE(ctx != NULL && out != NULL, "vglb_comm_init_detached: NULL argument");
    VGLB_REQUIRE(world >= 1 && world <= 64 && rank >= 0 && rank < world, "vglb_comm_init_detached: bad rank / world");
    vglb_comm *comm = (vglb_comm *)calloc(1, sizeof(vglb_comm));
    if (!comm) return VGLB_ENOMEM;
    comm->rank = rank;
    comm->world = world;
    comm->ctx = ctx;
    *out = comm;
    return VGLB_OK;
}

extern "C" int vglb_comm_destroy(vglb_comm *comm)
{
    if (!comm) return VGLB_OK;
    NcclApi *N = nccl_api();
    if (N && comm->nccl)
    {
        cudaStreamSynchronize(comm->ctx->stream);
        N->CommDestroy((ncclComm_t)comm->nccl);
    }
    free(comm);
    return VGLB_OK;
}

// ---- collectives on the context stream (asynchronous; used by the partitioned algorithm drivers) -------------------

int vglb_comm_allgather_async(vglb_comm *comm, void *d_buf, size_t bytes_per_rank)
{
    NcclApi *N = nccl_api();
    if (!N) return VGLB_ENCCL;
    DETACHED_CHECK(comm);
    NCCL_TRY(N->AllGather((const char *)d_buf + (size_t)comm->rank * bytes_per_rank, d_buf, bytes_per_rank, ncclUint8,
                          (ncclComm_t)comm->nccl, comm->ctx->stream));
    return VGLB_OK;
}

static inline size_t dtype_bytes(int dtype) { return dtype == VGLB_DT_I64 || dtype == VGLB_DT_F64 ? 8 : 4; }

int vglb_comm_allreduce_async(vglb_comm *comm, void *d_buf, size_t count, int dtype, int op)
{
    NcclApi *N = nccl_api();
    if (!N) return VGLB_ENCCL;
    DETACHED_CHECK(comm);
    const ncclDataType_t t = dtype == VGLB_DT_I64 ? ncclInt64 : dtype == VGLB_DT_F64 ? ncclFloat64 : dtype == VGLB_DT_U32 ? ncclUint32 : ncclInt32;
    const ncclRedOp_t o = op == VGLB_OP_MIN ? ncclMin : op == VGLB_OP_MAX ? ncclMax : ncclSum;
    NCCL_TRY(N->AllReduce(d_buf, d_buf, count, t, o, (ncclComm_t)comm->nccl, comm->ctx->stream));
    return VGLB_OK;
}

// the host side of the slot is pinned (ctx->h_counters), so both copies are plain asynchronous DMA on the context stream
int vglb_comm_allreduce_host(vglb_comm *comm, void *h_inout, int count, int dtype, int op)
{
    const size_t bytes = (size_t)count * dtype_bytes(dtype);
    VGLB_REQUIRE(count > 0 && bytes <= 16, "vglb_comm_allreduce_host: at most 16 bytes");
    vglb_ctx *ctx = comm->ctx;
    void *h = ctx->h_counters + CTR_HOST_ALLREDUCE, *d = ctx->d_counters + CTR_HOST_ALLREDUCE;
    memcpy(h, h_inout, bytes);
    CUDA_TRY(cudaMemcpyAsync(d, h, bytes, cudaMemcpyHostToDevice, ctx->stream));
    int rc = vglb_comm_allreduce_async(comm, d, (size_t)count, dtype, op);
    if (rc != VGLB_OK) return rc;
    CUDA_TRY(cudaMemcpyAsync(h, d, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    memcpy(h_inout, h, bytes);
    return VGLB_OK;
}

// all-to-all of equal slices: slice q of d_send goes to rank q, which stores it as slice `rank` of its d_recv
int vglb_comm_alltoall_async(vglb_comm *comm, const void *d_send, void *d_recv, size_t bytes_per_rank)
{
    NcclApi *N = nccl_api();
    if (!N) return VGLB_ENCCL;
    DETACHED_CHECK(comm);
    NCCL_TRY(N->GroupStart());
    for (int q = 0; q < comm->world; q++)
    {
        NCCL_TRY(N->Send((const char *)d_send + (size_t)q * bytes_per_rank, bytes_per_rank, ncclUint8, q, (ncclComm_t)comm->nccl, comm->ctx->stream));
        NCCL_TRY(N->Recv((char *)d_recv + (size_t)q * bytes_per_rank, bytes_per_rank, ncclUint8, q, (ncclComm_t)comm->nccl, comm->ctx->stream));
    }
    NCCL_TRY(N->GroupEnd());
    return VGLB_OK;
}

// Map a cudaMalloc'ed buffer of every rank into this process (CUDA IPC; NVLink peer access): peers[q] = rank q's buffer,
// peers[rank] = d_local. The handles travel through the communicator (an allgather of 72 bytes per rank).
// A collective that every rank completes whatever happens locally: a rank that cannot export its buffer still takes
// part in the allgather (with its slot marked invalid), success is decided only after it, and mappings opened before
// a later failure are closed again. On failure peers[] is left all-NULL except peers[rank]. The ranks may disagree
// about the outcome (an open can fail on one rank only); callers agree on it with an allreduce (vglb_part_map_lists).
struct IpcSlot
{
    cudaIpcMemHandle_t handle;
    int64_t valid;
};

int vglb_comm_ipc_map(vglb_comm *comm, void *d_local, void **peers)
{
    DETACHED_CHECK(comm);
    vglb_ctx *ctx = comm->ctx;
    const int P = comm->world, rank = comm->rank;
    const size_t hb = sizeof(IpcSlot);
    for (int q = 0; q < P; q++) peers[q] = NULL;
    peers[rank] = d_local;
    IpcSlot mine;
    memset(&mine, 0, sizeof(mine));
    int local_ok = 1;
    char local_msg[256] = "";
    vglb_dev_mark_exported(d_local);
    cudaError_t e = cudaIpcGetMemHandle(&mine.handle, d_local);
    if (e != cudaSuccess)
    {
        cudaGetLastError();
        snprintf(local_msg, sizeof(local_msg), "vglb_comm_ipc_map: cudaIpcGetMemHandle failed: %s", cudaGetErrorString(e));
        memset(&mine, 0, sizeof(mine));
        local_ok = 0;
    }
    mine.valid = local_ok;
    char *d_all = NULL;
    IpcSlot all[64];
    memset(all, 0, sizeof(all));
    // the staging block lives in the context's counter area when it fits (no allocation that could fail before the
    // collective); 64 ranks x 72 bytes do not, so larger worlds allocate — and still join the allgather on failure
    static_assert(sizeof(IpcSlot) == 72, "IpcSlot layout");
    if (vglb_dev_alloc(&d_all, (size_t)P * hb) != cudaSuccess)
    {
        cudaGetLastError();
        d_all = NULL;
    }
    int rc = VGLB_OK;
    if (d_all)
    {
        if (cudaMemcpyAsync(d_all + (size_t)rank * hb, &mine, hb, cudaMemcpyHostToDevice, ctx->stream) != cudaSuccess) local_ok = 0;
        rc = vglb_comm_allgather_async(comm, d_all, hb);
        if (rc == VGLB_OK && cudaMemcpyAsync(all, d_all, (size_t)P * hb, cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess) rc = VGLB_ECUDA;
        if (cudaStreamSynchronize(ctx->stream) != cudaSuccess) rc = VGLB_ECUDA;
        vglb_dev_free(d_all);
    }
    else
    {
        // cannot stage: this rank cannot join the allgather. 72 x P bytes failing to allocate means the device is out of
        // memory; the peers' next collective will report the mismatch through NCCL's own error path.
        vglb_set_error("vglb_comm_ipc_map: out of device memory for the handle exchange");
        return VGLB_ENOMEM;
    }
    if (rc != VGLB_OK) return rc;
    int all_valid = local_ok;
    for (int q = 0; q < P; q++)
        if (!all[q].valid) all_valid = 0;
    if (!all_valid)
    {
        vglb_set_error("%s", local_msg[0] ? local_msg : "vglb_comm_ipc_map: a peer could not export its buffer");
        return VGLB_ECUDA;
    }
    for (int q = 0; q < P; q++)
    {
        if (q == rank) continue;
        void *ptr = NULL;
        e = cudaIpcOpenMemHandle(&ptr, all[q].handle, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess)
        {
            cudaGetLastError();
            for (int r = 0; r < q; r++)
                if (r != rank && peers[r])
                {
                    cudaIpcCloseMemHandle(peers[r]);
                    peers[r] = NULL;
                }
            vglb_set_error("vglb_comm_ipc_map: cudaIpcOpenMemHandle of rank %d failed: %s", q, cudaGetErrorString(e));
            return VGLB_ECUDA;
        }
        peers[q] = ptr;
    }
    return VGLB_OK;
}

// The per-owner update lists of a partitioned graph (SSSP distance updates, BFS discoveries): P 8-byte counters followed by
// room for vp entries per owner, mapped into every peer once per graph. A collective: every rank ends up in the same
// mode — g->vec_peers_mapped = 1 (mapped) or -1 (some rank could not map: the dense / bitmap exchanges are used).
int vglb_part_map_lists(vglb_ctx *ctx, vglb_graph *g)
{
    if (g->vec_peers_mapped != 0) return VGLB_OK;
    if (!g->d_part_lists) CUDA_TRY(vglb_dev_alloc(&g->d_part_lists, ((size_t)g->cols + g->part_world + 8) * 8));
    int ok = 1;
    if (g->part_world > 8 || getenv("VGLB_DENSE_EXCHANGE")) ok = 0; // (the same decision on every rank)
    else
    {
        g->ipc_exported = 1;
        if (vglb_comm_ipc_map(g->comm, g->d_part_lists, (void **)g->d_vec_peer) != VGLB_OK) ok = 0;
    }
    int rc = vglb_comm_allreduce_host(g->comm, &ok, 1, VGLB_DT_I32, VGLB_OP_MIN);
    if (rc != VGLB_OK) return rc;
    g->vec_peers_mapped = ok ? 1 : -1;
    return VGLB_OK;
}

extern "C" int vglb_comm_allgather(vglb_comm *comm, void *d_buf, size_t bytes_per_rank)
{
    VGLB_REQUIRE(comm != NULL && d_buf != NULL, "vglb_comm_allgather: NULL argument");
    return vglb_comm_allgather_async(comm, d_buf, bytes_per_rank);
}

extern "C" int vglb_comm_allreduce_sum_i64(vglb_comm *comm, int64_t *d_buf, int count)
{
    VGLB_REQUIRE(comm != NULL && d_buf != NULL && count > 0, "vglb_comm_allreduce_sum_i64: bad argument");
    return vglb_comm_allreduce_async(comm, d_buf, (size_t)count, VGLB_DT_I64, VGLB_OP_SUM);
}

extern "C" int vglb_comm_allreduce_max_f64(vglb_comm *comm, double *h_value)
{
    VGLB_REQUIRE(comm != NULL && h_value != NULL, "vglb_comm_allreduce_max_f64: NULL argument");
    return vglb_comm_allreduce_host(comm, h_value, 1, VGLB_DT_F64, VGLB_OP_MAX);
}

extern "C" int vglb_comm_barrier(vglb_comm *comm)
{
    double x = 0.0;
    return vglb_comm_allreduce_max_f64(comm, &x);
}

// ---- partitioned build ------------------------------------------------------------------------------------------------

namespace
{

struct EdgeSource
{
    int mode; // 0 = generator, 1 = device arrays, 2 = host arrays
    int kind, scale, a, b, c;
    uint64_t seed;
    const int32_t *src, *dst;
    int64_t edges; // before symmetrisation
};

__global__ void part_generate_kernel(int kind, int scale, uint64_t seed, int a, int b, int c, int64_t first, int64_t n,
                                     int32_t *__restrict__ src, int32_t *__restrict__ dst)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride)
    {
        int32_t s, d;
        vglb_gen_edge(kind, scale, seed, (uint64_t)(first + i), a, b, c, &s, &d);
        src[i] = s;
        dst[i] = d;
    }
}

// pass 1: out-degree, in-degree and in-degree without self loops of every ORIGINAL vertex
__global__ void part_degree_kernel(const int32_t *__restrict__ src, const int32_t *__restrict__ dst, int64_t n, int32_t V,
                                   int32_t *__restrict__ deg_out, int32_t *__restrict__ deg_in,
                                   int32_t *__restrict__ deg_in_noloops, int *__restrict__ bad)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride)
    {
        const int32_t s = src[i], d = dst[i];
        if (s < 0 || s >= V || d < 0 || d >= V) { *bad = 1; continue; }
        atomicAdd(&deg_out[s], 1);
        atomicAdd(&deg_in[d], 1);
        if (s != d) atomicAdd(&deg_in_noloops[d], 1);
    }
}

// sorted id s -> column (s mod P) * vp + s div P; also this rank's edge totals for both directions
__global__ void part_numbering_kernel(const uint32_t *__restrict__ sorted_ids, int32_t V, int32_t P, int32_t vp, int32_t rank,
                                      const int32_t *__restrict__ deg_out, const int32_t *__restrict__ deg_in,
                                      int32_t *__restrict__ fwd, int32_t *__restrict__ bwd,
                                      unsigned long long *__restrict__ totals /* [2] */)
{
    long long e_out = 0, e_in = 0;
    for (int32_t s = blockIdx.x * blockDim.x + threadIdx.x; s < V; s += gridDim.x * blockDim.x)
    {
        const int32_t orig = (int32_t)sorted_ids[s];
        const int32_t col = (s % P) * vp + s / P;
        fwd[orig] = col;
        bwd[col] = orig;
        if (s % P == rank)
        {
            e_out += deg_out[orig];
            e_in += deg_in[orig];
        }
    }
    e_out = warp_sum_i64(e_out);
    e_in = warp_sum_i64(e_in);
    if ((threadIdx.x & 31) == 0)
    {
        if (e_out) atomicAdd(&totals[0], (unsigned long long)e_out);
        if (e_in) atomicAdd(&totals[1], (unsigned long long)e_in);
    }
}

// pass 2: keep the edges whose row (dir 0: source, dir 1: destination) this rank owns
__global__ void part_collect_kernel(const int32_t *__restrict__ src, const int32_t *__restrict__ dst, int64_t n,
                                    const int32_t *__restrict__ fwd, int32_t P, int32_t vp, int32_t rank, int dir,
                                    uint64_t *__restrict__ keys, unsigned long long *__restrict__ kept,
                                    unsigned long long *__restrict__ row_count)
{
    const int lane = threadIdx.x & 31;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t n_padded = (n + 31) & ~(int64_t)31;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_padded; i += stride)
    {
        bool keep = false;
        uint64_t key = 0;
        if (i < n)
        {
            const int32_t cs = fwd[src[i]], cd = fwd[dst[i]];
            const int32_t own = dir == 0 ? cs : cd, other = dir == 0 ? cd : cs;
            if (own / vp == rank)
            {
                keep = true;
                const uint32_t row = (uint32_t)(own - rank * vp);
                const uint32_t s_other = (uint32_t)(other % vp) * (uint32_t)P + (uint32_t)(other / vp);
                key = ((uint64_t)row << 32) | s_other;
                atomicAdd(&row_count[row], 1ULL);
            }
        }
        const unsigned mask = __ballot_sync(0xffffffffu, keep);
        if (mask)
        {
            unsigned long long base = 0;
            const int leader = __ffs(mask) - 1;
            if (lane == leader) base = atomicAdd(kept, (unsigned long long)__popc(mask));
            base = __shfl_sync(0xffffffffu, base, leader);
            if (keep) keys[base + __popc(mask & ((1u << lane) - 1u))] = key;
        }
    }
}

__global__ void part_adjacency_kernel(const uint64_t *__restrict__ keys, int64_t n, int32_t P, int32_t vp,
                                      int32_t *__restrict__ adj)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride)
    {
        const uint32_t s = (uint32_t)keys[i];
        adj[i] = (int32_t)((s % (uint32_t)P) * (uint32_t)vp + s / (uint32_t)P);
    }
}

// inv[r] = 1 / indeg_noloops of local row r (pr.hpp:66-73: double division, then narrowing)
__global__ void part_pr_inverse_kernel(const int32_t *__restrict__ deg_in_noloops, const int32_t *__restrict__ bwd,
                                       int32_t col0, int32_t rows, float *__restrict__ inv)
{
    int32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r < rows)
    {
        const int32_t d = deg_in_noloops[bwd[col0 + r]];
        inv[r] = d == 0 ? 0.0f : (float)(1.0 / (double)d);
    }
}

} // namespace

static const int64_t kChunkEdges = (int64_t)1 << 26;

// device pointers to the edges [first, first + n) of one half (half 1 = the reversed copy when symmetrising)
static int provide_chunk(vglb_ctx *ctx, const EdgeSource &S, int half, int64_t first, int64_t n, int32_t *buf_a,
                         int32_t *buf_b, const int32_t **out_src, const int32_t **out_dst)
{
    const int32_t *ps = NULL, *pd = NULL;
    if (S.mode == 0)
    {
        part_generate_kernel<<<ctx->sm_count * 16, 256, 0, ctx->stream>>>(S.kind, S.scale, S.seed, S.a, S.b, S.c, first, n, buf_a, buf_b);
        KERNEL_TRY();
        ctx->launches++;
        ps = buf_a;
        pd = buf_b;
    }
    else if (S.mode == 1)
    {
        ps = S.src + first;
        pd = S.dst + first;
    }
    else
    {
        CUDA_TRY(cudaMemcpyAsync(buf_a, S.src + first, (size_t)n * 4, cudaMemcpyHostToDevice, ctx->stream));
        CUDA_TRY(cudaMemcpyAsync(buf_b, S.dst + first, (size_t)n * 4, cudaMemcpyHostToDevice, ctx->stream));
        ps = buf_a;
        pd = buf_b;
    }
    *out_src = half == 0 ? ps : pd;
    *out_dst = half == 0 ? pd : ps;
    return VGLB_OK;
}

static int build_partitioned(vglb_ctx *ctx, vglb_comm *comm, int32_t V, const EdgeSource &S, int symmetrize, int flags,
                             vglb_graph **out_graph)
{
    VGLB_REQUIRE(ctx != NULL && comm != NULL && out_graph != NULL, "partitioned build: NULL argument");
    VGLB_REQUIRE(V > 0 && S.edges >= 0, "partitioned build: need V > 0 and E >= 0");
    VGLB_REQUIRE(!(flags & VGLB_GRAPH_WITH_EDGE_ORDER), "partitioned build: VGLB_GRAPH_WITH_EDGE_ORDER is not supported");
    CUDA_TRY(cudaSetDevice(ctx->device));
    const int32_t P = comm->world, rank = comm->rank;
    const int64_t vp64 = ((ceil_div64(V, P) + 31) / 32) * 32;
    VGLB_REQUIRE(vp64 * P < 0x7fffffffLL, "partitioned build: too many vertices for int32 column ids");
    const int32_t vp = (int32_t)vp64;
    const int32_t rows = V > rank ? (V - rank + P - 1) / P : 0; // sorted ids rank, rank + P, ...
    const int halves = symmetrize ? 2 : 1;

    graph_ptr owner = vglb_graph_new();
    if (!owner) return VGLB_ENOMEM;
    vglb_graph *g = owner.get();
    dev_ptr<int32_t> buf_a, buf_b, d_deg_out, d_deg_in, d_deg_nl;
    dev_ptr<unsigned long long> d_rowcnt, d_misc;
    dev_ptr<int> d_bad;
    const int grid = ctx->sm_count * 16;
    cudaStream_t st = ctx->stream;
    const int64_t chunk = S.edges < kChunkEdges ? (S.edges > 0 ? S.edges : 1) : kChunkEdges;
    if (S.mode != 1)
    {
        CUDA_TRY(vglb_dev_alloc(buf_a, (size_t)chunk * 4));
        CUDA_TRY(vglb_dev_alloc(buf_b, (size_t)chunk * 4));
    }
    // pass 1: degrees of every vertex (identical on every rank)
    CUDA_TRY(vglb_dev_alloc(d_deg_out, (size_t)V * 4));
    CUDA_TRY(vglb_dev_alloc(d_deg_in, (size_t)V * 4));
    CUDA_TRY(vglb_dev_alloc(d_deg_nl, (size_t)V * 4));
    CUDA_TRY(vglb_dev_alloc(d_bad, 4));
    CUDA_TRY(vglb_dev_alloc(d_misc, 8 * 8));
    CUDA_TRY(cudaMemsetAsync(d_deg_out.get(), 0, (size_t)V * 4, st));
    CUDA_TRY(cudaMemsetAsync(d_deg_in.get(), 0, (size_t)V * 4, st));
    CUDA_TRY(cudaMemsetAsync(d_deg_nl.get(), 0, (size_t)V * 4, st));
    CUDA_TRY(cudaMemsetAsync(d_bad.get(), 0, 4, st));
    CUDA_TRY(cudaMemsetAsync(d_misc.get(), 0, 8 * 8, st));
    for (int half = 0; half < halves; half++)
        for (int64_t first = 0; first < S.edges; first += chunk)
        {
            const int64_t n = S.edges - first < chunk ? S.edges - first : chunk;
            const int32_t *ps, *pd;
            VGLB_TRY(provide_chunk(ctx, S, half, first, n, buf_a.get(), buf_b.get(), &ps, &pd));
            part_degree_kernel<<<grid, 256, 0, st>>>(ps, pd, n, V, d_deg_out.get(), d_deg_in.get(), d_deg_nl.get(), d_bad.get());
            KERNEL_TRY();
            CUDA_TRY(cudaStreamSynchronize(st)); // the chunk buffers are reused
        }
    int bad = 0;
    CUDA_TRY(cudaMemcpy(&bad, d_bad.get(), 4, cudaMemcpyDeviceToHost));
    if (bad)
    {
        vglb_set_error("partitioned build: vertex id out of range [0, V)");
        return VGLB_EINVAL;
    }
    // the reference's numbering: stable sort by out-degree descending, then the round-robin deal
    const int64_t cols = (int64_t)vp * P;
    {
        DegreeOrder order;
        VGLB_TRY(vglb_degree_order(ctx, d_deg_out.get(), V, order));
        CUDA_TRY(vglb_dev_alloc(&g->d_fwd, (size_t)V * 4));
        CUDA_TRY(vglb_dev_alloc(&g->d_bwd, (size_t)cols * 4));
        CUDA_TRY(cudaMemsetAsync(g->d_bwd, 0xFF, (size_t)cols * 4, st));
        part_numbering_kernel<<<ctx->sm_count * 8, 256, 0, st>>>(order.sorted, V, P, vp, rank, d_deg_out.get(), d_deg_in.get(), g->d_fwd,
                                                                g->d_bwd, d_misc.get());
        KERNEL_TRY();
        CUDA_TRY(cudaStreamSynchronize(st));
    }
    unsigned long long totals[2] = {0, 0};
    CUDA_TRY(cudaMemcpy(totals, d_misc.get(), 16, cudaMemcpyDeviceToHost));
    g->V = rows;
    g->vp = vp;
    g->cols = cols;
    g->V_orig = V;
    g->E_global = S.edges * halves;
    g->part_rank = rank;
    g->part_world = P;
    g->col_of_row0 = rank * vp;
    g->comm = comm;

    // PageRank's inverse in-degrees of the owned rows come from pass 1 (the single-GPU path counts them from the CSR)
    CUDA_TRY(vglb_dev_alloc(&g->d_pr_inv, (size_t)(vp > 0 ? vp : 1) * 4));
    CUDA_TRY(cudaMemsetAsync(g->d_pr_inv, 0, (size_t)vp * 4, st));
    if (rows > 0)
    {
        part_pr_inverse_kernel<<<(unsigned)ceil_div64(rows, 256), 256, 0, st>>>(d_deg_nl.get(), g->d_bwd, g->col_of_row0, rows, g->d_pr_inv);
        KERNEL_TRY();
    }

    // pass 2, once per direction
    CUDA_TRY(vglb_dev_alloc(d_rowcnt, ((size_t)vp + 2) * 8));
    for (int dir = 0; dir < ((flags & VGLB_GRAPH_WITH_INCOMING) ? 2 : 1); dir++)
    {
        const int64_t e_local = (int64_t)totals[dir];
        if (e_local >= 0xFFFFFFFFLL)
        {
            vglb_set_error("partitioned build: more than 2^32-1 edges on one rank");
            return VGLB_EINVAL;
        }
        const size_t kb = (size_t)(e_local > 0 ? e_local : 1) * 8;
        dev_ptr<uint64_t> keys0, keys1;
        CUDA_TRY(vglb_dev_alloc(keys0, kb));
        CUDA_TRY(vglb_dev_alloc(keys1, kb));
        CUDA_TRY(cudaMemsetAsync(d_rowcnt.get(), 0, ((size_t)vp + 2) * 8, st));
        CUDA_TRY(cudaMemsetAsync(d_misc.get() + 2, 0, 8, st));
        for (int half = 0; half < halves; half++)
            for (int64_t first = 0; first < S.edges; first += chunk)
            {
                const int64_t n = S.edges - first < chunk ? S.edges - first : chunk;
                const int32_t *ps, *pd;
                VGLB_TRY(provide_chunk(ctx, S, half, first, n, buf_a.get(), buf_b.get(), &ps, &pd));
                part_collect_kernel<<<grid, 256, 0, st>>>(ps, pd, n, g->d_fwd, P, vp, rank, dir, keys0.get(), d_misc.get() + 2,
                                                          d_rowcnt.get());
                KERNEL_TRY();
                CUDA_TRY(cudaStreamSynchronize(st));
            }
        unsigned long long kept = 0;
        CUDA_TRY(cudaMemcpy(&kept, d_misc.get() + 2, 8, cudaMemcpyDeviceToHost));
        if ((int64_t)kept != e_local)
        {
            vglb_set_error("partitioned build: kept %lld edges, expected %lld", (long long)kept, (long long)e_local);
            return VGLB_ECUDA;
        }
        int64_t **ptr_field = dir == 0 ? &g->d_out_ptr : &g->d_in_ptr;
        int32_t **adj_field = dir == 0 ? &g->d_out_adj : &g->d_in_adj;
        CUDA_TRY(vglb_dev_alloc(ptr_field, ((size_t)vp + 2) * 8));
        CUDA_TRY(vglb_dev_alloc(adj_field, (size_t)(e_local > 0 ? e_local : 1) * 4 + 16));
        {
            dev_ptr<void> tmp;
            CUDA_TRY(vglb_cub(tmp, [&](void *t, size_t &bytes) {
                return cub::DeviceScan::ExclusiveSum(t, bytes, (const int64_t *)d_rowcnt.get(), *ptr_field, vp + 1, st);
            }));
            CUDA_TRY(cudaStreamSynchronize(st));
        }
        if (e_local > 0)
        {
            cub::DoubleBuffer<uint64_t> keys(keys0.get(), keys1.get());
            const int end_bit = 32 + vglb_key_bits(vp);
            dev_ptr<void> tmp;
            CUDA_TRY(vglb_cub(tmp, [&](void *t, size_t &bytes) {
                return cub::DeviceRadixSort::SortKeys(t, bytes, keys, e_local, 0, end_bit, st);
            }));
            part_adjacency_kernel<<<grid, 256, 0, st>>>(keys.Current(), e_local, P, vp, *adj_field);
            KERNEL_TRY();
            CUDA_TRY(cudaStreamSynchronize(st));
        }
        if (dir == 0) g->E = e_local;
    }
    VGLB_TRY(vglb_graph_compute_tiers(ctx, g));
    *out_graph = owner.release();
    return VGLB_OK;
}

extern "C" int vglb_graph_from_edges_partitioned(vglb_ctx *ctx, vglb_comm *comm, int32_t vertices, int64_t edges,
                                                 const int32_t *src, const int32_t *dst, int src_on_device,
                                                 int symmetrize, int flags, vglb_graph **out_graph)
{
    VGLB_REQUIRE(edges == 0 || (src != NULL && dst != NULL), "vglb_graph_from_edges_partitioned: NULL edge arrays");
    EdgeSource S;
    memset(&S, 0, sizeof(S));
    S.mode = src_on_device ? 1 : 2;
    S.src = src;
    S.dst = dst;
    S.edges = edges;
    return build_partitioned(ctx, comm, vertices, S, symmetrize, flags, out_graph);
}

extern "C" int vglb_graph_from_generator_partitioned(vglb_ctx *ctx, vglb_comm *comm, int kind, int scale, int64_t edges,
                                                     uint64_t seed, int a, int b, int c, int symmetrize, int flags,
                                                     vglb_graph **out_graph)
{
    VGLB_REQUIRE(scale >= 1 && scale <= 30 && edges >= 0, "vglb_graph_from_generator_partitioned: bad scale/edges");
    VGLB_REQUIRE(kind >= 0 && kind <= 2 && a > 0 && b >= 0 && c >= 0 && a + b + c < 100,
                 "vglb_graph_from_generator_partitioned: bad kind or probabilities");
    EdgeSource S;
    memset(&S, 0, sizeof(S));
    S.mode = 0;
    S.kind = kind;
    S.scale = scale;
    S.a = a;
    S.b = b;
    S.c = c;
    S.seed = seed;
    S.edges = edges;
    return build_partitioned(ctx, comm, (int32_t)1 << scale, S, symmetrize, flags, out_graph);
}

// ---- VGL_Graph::move_to_device for one rank's part (vect_csr_graph.hpp:185-196): host arrays of an already-built part
//      (this rank's row pointers and adjacency in column ids, the ORIGINAL -> column map) copied to HBM ----------------

extern "C" int vglb_graph_from_csr_partitioned(vglb_ctx *ctx, vglb_comm *comm, int32_t vertices_global, int32_t rows,
                                               const int64_t *h_out_ptr, const int32_t *h_out_adj,
                                               const int32_t *h_orig_to_col, const int64_t *h_in_ptr,
                                               const int32_t *h_in_adj, vglb_graph **out_graph)
{
    VGLB_REQUIRE(ctx != NULL && comm != NULL && out_graph != NULL && h_out_ptr != NULL && h_orig_to_col != NULL,
                 "vglb_graph_from_csr_partitioned: NULL argument");
    const int32_t P = comm->world, rank = comm->rank, V = vertices_global;
    VGLB_REQUIRE(V > 0 && rows == (V > rank ? (V - rank + P - 1) / P : 0), "vglb_graph_from_csr_partitioned: rows does not match the round-robin deal");
    VGLB_REQUIRE((h_in_ptr == NULL) == (h_in_adj == NULL), "vglb_graph_from_csr_partitioned: incoming arrays must come together");
    CUDA_TRY(cudaSetDevice(ctx->device));
    const int32_t vp = (int32_t)(((ceil_div64(V, P) + 31) / 32) * 32);
    const int64_t E = h_out_ptr[rows], E_in = h_in_ptr ? h_in_ptr[rows] : 0;
    VGLB_REQUIRE(E >= 0 && E_in >= 0 && (E == 0 || h_out_adj != NULL), "vglb_graph_from_csr_partitioned: bad sizes");
    graph_ptr owner = vglb_graph_new();
    if (!owner) return VGLB_ENOMEM;
    vglb_graph *g = owner.get();
    cudaStream_t st = ctx->stream;
    g->V = rows;
    g->E = E;
    g->vp = vp;
    g->cols = (int64_t)vp * P;
    g->V_orig = V;
    g->part_rank = rank;
    g->part_world = P;
    g->col_of_row0 = rank * vp;
    g->comm = comm;
    CUDA_TRY(vglb_dev_alloc(&g->d_out_ptr, ((size_t)vp + 2) * 8));
    CUDA_TRY(vglb_dev_alloc(&g->d_out_adj, (size_t)(E > 0 ? E : 1) * 4 + 16));
    CUDA_TRY(cudaMemcpyAsync(g->d_out_ptr, h_out_ptr, ((size_t)rows + 1) * 8, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(g->d_out_adj, h_out_adj, (size_t)E * 4, cudaMemcpyHostToDevice, st));
    if (h_in_ptr)
    {
        CUDA_TRY(vglb_dev_alloc(&g->d_in_ptr, ((size_t)vp + 2) * 8));
        CUDA_TRY(vglb_dev_alloc(&g->d_in_adj, (size_t)(E_in > 0 ? E_in : 1) * 4 + 16));
        CUDA_TRY(cudaMemcpyAsync(g->d_in_ptr, h_in_ptr, ((size_t)rows + 1) * 8, cudaMemcpyHostToDevice, st));
        CUDA_TRY(cudaMemcpyAsync(g->d_in_adj, h_in_adj, (size_t)E_in * 4, cudaMemcpyHostToDevice, st));
    }
    CUDA_TRY(vglb_dev_alloc(&g->d_fwd, (size_t)V * 4));
    CUDA_TRY(vglb_dev_alloc(&g->d_bwd, (size_t)g->cols * 4));
    CUDA_TRY(cudaMemcpyAsync(g->d_fwd, h_orig_to_col, (size_t)V * 4, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemsetAsync(g->d_bwd, 0xFF, (size_t)g->cols * 4, st));
    // caller-supplied arrays are checked on the device before anything indexes with them (row pointers non-decreasing
    // from 0 to E, column ids in [0, cols), the map injective); the verdict travels with the edge count so that a
    // rank with a bad part takes every rank out of the call together instead of leaving the others in a collective
    int *d_bad = (int *)(ctx->d_counters + CTR_BAD);
    CUDA_TRY(cudaMemsetAsync(d_bad, 0, sizeof(int), st));
    VGLB_TRY(vglb_invert_map_checked(ctx, g->d_fwd, V, g->cols, g->d_bwd));
    VGLB_TRY(vglb_csr_validate_device(ctx, g->d_out_ptr, rows, E, g->d_out_adj, g->cols));
    if (h_in_ptr) VGLB_TRY(vglb_csr_validate_device(ctx, g->d_in_ptr, rows, E_in, g->d_in_adj, g->cols));
    int bad = 0;
    CUDA_TRY(cudaMemcpyAsync(&bad, d_bad, sizeof(int), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    // whole-graph edge count and the number of ranks with a bad part (a collective when the communicator is live)
    g->E_global = E;
    int64_t bad_ranks = bad ? 1 : 0;
    if (comm->nccl && P > 1)
    {
        int64_t r2[2] = {E, bad_ranks};
        VGLB_TRY(vglb_comm_allreduce_host(comm, r2, 2, VGLB_DT_I64, VGLB_OP_SUM));
        g->E_global = r2[0];
        bad_ranks = r2[1];
    }
    if (bad_ranks)
    {
        vglb_set_error("vglb_graph_from_csr_partitioned: %s part is not a CSR (row pointers non-decreasing from 0 to E, column "
                       "ids in [0, columns), ORIGINAL -> column map injective)", bad ? "this rank's" : "another rank's");
        return VGLB_EINVAL;
    }
    VGLB_TRY(vglb_graph_compute_tiers(ctx, g));
    *out_graph = owner.release();
    return VGLB_OK;
}
