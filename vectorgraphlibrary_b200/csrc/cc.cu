// cc.cu — connected components by min-label hooking + pointer jumping over the device VectCSR (sm_100a).
//
// Reference: ConnectedComponents::vgl_shiloach_vishkin (algorithms/cc/shiloach_vishkin.hpp:7-88):
//   compute(comp[v] = v)                                           (:19-24, v = SCATTER-sorted id)
//   while (hook_changes):
//       scatter(all-active, if comp[src] < comp[dst] then comp[dst] = comp[src])   (:30-53, racy but monotone)
//       while (jump_changes): compute(comp[v] = comp[comp[v]])     (:55-76)
// The unique fixed point is comp[v] = min sorted id over {v} U ancestors(v) (SURVEY §8c), the component minimum on
// symmetric graphs, so any schedule of monotone hooks and jumps reaches bit-identical labels.
//
// B200 design: the hook is an all-active advance with an atomicMin edge op, one launch covering all degree tiers —
// cc_hook_kernel below (load-balanced, several independent gathers per lane); hooks are applied in place, so a label
// travels many hops within one round (Gauss-Seidel), and the whole jump loop of the reference collapses into ONE kernel
// that chases every vertex to its current root (comp[x] <= x always holds, so the chase terminates and concurrent writes
// only shorten it). The convergence flag is a device word read back once per round (the reference returns a reduce<int> to
// the host per round, :47-52).
// HBM roofline: algorithmic bytes = sum_hook [ 8E + 12V ] + sum_jump 8V (SURVEY §8d).
#include <limits.h>

#include "common.cuh"


// ---- the hook as a load-balanced all-active advance specialised for min-label propagation ---------------------------
// The edge op of shiloach_vishkin.hpp:38-46, scheduled for memory-level parallelism: the lambda-generic per-row advance
// that the GraphAbstractionsB200 shim instantiates for user lambdas (include/vgl_b200/advance.cuh) issues one dependent
// chain (index -> label -> atomic) per lane and step and reaches a third of the PageRank sweep's edge rate. Here rows with
// >= 4096 edges get one CTA per CC_BIG_CHUNK edges, and a warp takes 32 consecutive smaller rows and walks the
// concatenation of their edge ranges (shuffle search over the degree prefix sums, as in sssp.cu), CC_UNROLL edges per lane:
// the index loads, then the label gathers, are independent.
#define CC_THREADS 256
#define CC_UNROLL 4
#define CC_BIG_CHUNK 8192

// The label gathered a moment ago decides: if it is larger, the hook is issued as a fire-and-forget reduction (no return
// value to wait for — four value-returning atomics per step were four serialised round trips) and the round counts as
// "changed". That is conservative only when somebody else lowered the label in between; a round in which no gathered label
// is larger issues no atomic at all, so the final, change-free round is still recognised.
__device__ __forceinline__ void cc_hook_one(int32_t *__restrict__ comp, int32_t cs, int32_t dst, int32_t cd, bool &changed)
{
    if (cs < cd)
    {
        atomicMin(&comp[dst], cs);
        changed = true;
    }
}

__global__ void __launch_bounds__(CC_THREADS)
cc_hook_kernel(const int64_t *__restrict__ ptr, const int32_t *__restrict__ adj, int32_t n_big, int32_t big_chunks, int32_t rows_with_edges,
               int32_t *__restrict__ comp, int32_t col0, int *changed_flag)
{
    // the convergence flag is written once per CTA: in the first round ~10^7 hooks succeed, and as many stores to one
    // word serialise in L2
    bool changed = false;
    const unsigned FULL = 0xffffffffu;
    const uint64_t pol = l2_policy_evict_first();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // rows with >= 4096 edges: their edges are the prefix [0, ptr[n_big]) of the adjacency array (ids are degree-sorted), cut
    // into CC_BIG_CHUNK-edge chunks, one CTA each; a chunk spans at most three such rows, found by a binary search over the
    // row pointers. (One CTA per (row, chunk slot of the LONGEST row) launched ~10^6 CTAs with nothing to do at scale 24.)
    const int big_blocks = big_chunks;
    if ((int)blockIdx.x < big_blocks)
    {
        const int64_t hub_edges = ptr[n_big];
        const int64_t e0 = (int64_t)blockIdx.x * CC_BIG_CHUNK, e1 = min(hub_edges, e0 + CC_BIG_CHUNK);
        int32_t lo = 0, hi = n_big; // largest row with ptr[row] <= e0
        while (hi - lo > 1)
        {
            const int32_t mid = lo + (hi - lo) / 2;
            if (ptr[mid] <= e0) lo = mid;
            else hi = mid;
        }
        int32_t row = lo;
        int64_t row_end = ptr[row + 1];
        int32_t cs = comp[col0 + row];
        for (int64_t p0 = e0 + threadIdx.x; p0 < e1; p0 += CC_THREADS * CC_UNROLL)
        {
            int32_t d[CC_UNROLL], cd[CC_UNROLL], csk[CC_UNROLL];
#pragma unroll
            for (int k = 0; k < CC_UNROLL; k++)
            {
                const int64_t p = p0 + (int64_t)k * CC_THREADS;
                d[k] = -1;
                if (p < e1)
                {
                    while (p >= row_end) // (positions only grow: at most two steps per chunk)
                    {
                        row++;
                        row_end = ptr[row + 1];
                        cs = comp[col0 + row];
                    }
                    d[k] = ld_stream_s32(adj + p, pol);
                }
                csk[k] = cs;
            }
#pragma unroll
            for (int k = 0; k < CC_UNROLL; k++) cd[k] = d[k] >= 0 ? comp[d[k]] : INT_MIN;
#pragma unroll
            for (int k = 0; k < CC_UNROLL; k++) cc_hook_one(comp, csk[k], d[k], cd[k], changed);
        }
        if (__syncthreads_or(changed) && threadIdx.x == 0) *changed_flag = 1;
        return;
    }
    const int32_t row = n_big + (((int)blockIdx.x - big_blocks) * (CC_THREADS / 32) + warp) * 32 + lane;
    int64_t s = 0;
    int deg = 0;
    int32_t cs = 0;
    if (row < rows_with_edges)
    {
        s = ptr[row];
        deg = (int)(ptr[row + 1] - s);
        cs = comp[col0 + row];
    }
    int incl = deg;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1)
    {
        const int t = __shfl_up_sync(FULL, incl, o);
        if (lane >= o) incl += t;
    }
    const int excl = incl - deg;
    const int total = __shfl_sync(FULL, incl, 31);
    for (int base = 0; base < total; base += 32 * CC_UNROLL)
    {
        int32_t d[CC_UNROLL], csj[CC_UNROLL], cd[CC_UNROLL];
#pragma unroll
        for (int k = 0; k < CC_UNROLL; k++)
        {
            const int idx = base + k * 32 + lane;
            int j = 0; // largest lane whose range starts at or before idx
#pragma unroll
            for (int step = 16; step > 0; step >>= 1)
            {
                const int ex = __shfl_sync(FULL, excl, j + step);
                if (ex <= idx) j += step;
            }
            const int64_t sj = __shfl_sync(FULL, s, j);
            const int exj = __shfl_sync(FULL, excl, j);
            csj[k] = __shfl_sync(FULL, cs, j);
            d[k] = idx < total ? ld_stream_s32(adj + sj + (idx - exj), pol) : -1;
        }
#pragma unroll
        for (int k = 0; k < CC_UNROLL; k++) cd[k] = d[k] >= 0 ? comp[d[k]] : INT_MIN;
#pragma unroll
        for (int k = 0; k < CC_UNROLL; k++) cc_hook_one(comp, csj[k], d[k], cd[k], changed);
    }
    if (__syncthreads_or(changed) && threadIdx.x == 0) *changed_flag = 1;
}

static int cc_launch_hook(vglb_ctx *ctx, const vglb_graph *g, int32_t *comp, int32_t col0, int *d_changed)
{
    const int32_t n_big = g->tier_border[0], rows_with_edges = g->tier_border[VGLB_NUM_TIERS - 2];
    if (g->cc_hub_edges_plus1 == 0) // edges of the rows with >= 4096 edges = row pointer at the first tier border, once per graph
    {
        int64_t e = 0;
        if (n_big > 0)
        {
            CUDA_TRY(cudaMemcpyAsync(&e, g->d_out_ptr + n_big, 8, cudaMemcpyDeviceToHost, ctx->stream));
            CUDA_TRY(cudaStreamSynchronize(ctx->stream));
        }
        ((vglb_graph *)g)->cc_hub_edges_plus1 = e + 1;
    }
    const int big_chunks = (int)ceil_div64(g->cc_hub_edges_plus1 - 1, CC_BIG_CHUNK);
    const int64_t warps = ceil_div64(rows_with_edges - n_big, 32);
    const int64_t grid = (int64_t)big_chunks + ceil_div64(warps, CC_THREADS / 32);
    VGLB_REQUIRE(grid < 0x7fffffffLL, "vglb_cc: grid too large");
    if (grid > 0)
    {
        cc_hook_kernel<<<(unsigned)grid, CC_THREADS, 0, ctx->stream>>>(g->d_out_ptr, g->d_out_adj, n_big, big_chunks, rows_with_edges, comp,
                                                                      col0, d_changed);
        KERNEL_TRY();
        ctx->launches++;
    }
    return VGLB_OK;
}

__global__ void cc_init_kernel(int32_t *__restrict__ comp, int32_t V)
{
    for (int32_t v = blockIdx.x * blockDim.x + threadIdx.x; v < V; v += gridDim.x * blockDim.x) comp[v] = v;
}

// all jump rounds of shiloach_vishkin.hpp:55-76 at once: comp[v] = root of v's current label chain
__global__ void cc_jump_kernel(int32_t *__restrict__ comp, int32_t V)
{
    for (int32_t v = blockIdx.x * blockDim.x + threadIdx.x; v < V; v += gridDim.x * blockDim.x)
    {
        const int32_t c = comp[v];
        int32_t r = c;
        for (;;)
        {
            const int32_t n = comp[r];
            if (n == r) break;
            r = n;
        }
        if (r != c) comp[v] = r;
    }
}


// ---- 1D-partitioned CC -----------------------------------------------------------------------------------------------
// Labels stay the reference's SCATTER-sorted ids (so the result is bit-identical to one GPU): the replicated label
// vector is indexed by column id and initialised with the sorted id of every column. Each rank hooks over the rows it
// owns into its replica, one allreduce(min) per round combines the replicas (the reference exchanges the whole array
// after its advance too, mpi_exchange.hpp:155-271), and every rank then runs the same pointer-jump over the whole
// vector (deterministic: a chain's root never changes during the jump), so the replicas stay identical.
__device__ __forceinline__ int32_t cc_col_of_sorted(int32_t s, int32_t P, int32_t vp) { return (s % P) * vp + s / P; }

__global__ void cc_part_init_kernel(int32_t *__restrict__ comp, int64_t cols, int32_t P, int32_t vp)
{
    for (int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; c < cols; c += (int64_t)gridDim.x * blockDim.x)
        comp[c] = (int32_t)(c % vp) * P + (int32_t)(c / vp);
}

__global__ void cc_part_jump_kernel(int32_t *__restrict__ comp, int64_t cols, int32_t P, int32_t vp)
{
    for (int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; c < cols; c += (int64_t)gridDim.x * blockDim.x)
    {
        const int32_t l = comp[c];
        int32_t r = l;
        for (;;)
        {
            const int32_t n = comp[cc_col_of_sorted(r, P, vp)];
            if (n == r) break;
            r = n;
        }
        if (r != l) comp[c] = r;
    }
}

static int cc_partitioned(vglb_ctx *ctx, vglb_graph *g, int32_t *d_labels, vglb_stats *stats)
{
    CUDA_TRY(cudaSetDevice(ctx->device));
    vglb_comm *comm = g->comm;
    const int64_t launches0 = ctx->launches;
    const int32_t rows = g->V, P = g->part_world, vp = g->vp;
    cudaStream_t st = ctx->stream;
    int *d_changed = (int *)(ctx->d_counters + 40);
    int *h_changed = (int *)(ctx->h_counters + 40);
    if (!g->d_part_vec) CUDA_TRY(vglb_dev_alloc(&g->d_part_vec, (size_t)g->cols * 4));
    int32_t *comp = (int32_t *)g->d_part_vec;

    CUDA_TRY(cudaEventRecord(ctx->ev_start, st));
    cc_part_init_kernel<<<ctx->sm_count * 8, 256, 0, st>>>(comp, g->cols, P, vp);
    KERNEL_TRY();
    ctx->launches++;
    int64_t hook_rounds = 0;
    int rc;
    for (;;)
    {
        CUDA_TRY(cudaMemsetAsync(d_changed, 0, sizeof(int), st));
        rc = cc_launch_hook(ctx, g, comp, g->col_of_row0, d_changed);
        if (rc != VGLB_OK) return rc;
        hook_rounds++;
        rc = vglb_comm_allreduce_async(comm, comp, (size_t)g->cols, VGLB_DT_I32, VGLB_OP_MIN);
        if (rc != VGLB_OK) return rc;
        rc = vglb_comm_allreduce_async(comm, d_changed, 1, VGLB_DT_I32, VGLB_OP_MAX);
        if (rc != VGLB_OK) return rc;
        CUDA_TRY(cudaMemcpyAsync(h_changed, d_changed, sizeof(int), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        if (!*h_changed) break;
        cc_part_jump_kernel<<<ctx->sm_count * 8, 256, 0, st>>>(comp, g->cols, P, vp);
        KERNEL_TRY();
        ctx->launches++;
    }
    if (rows > 0) CUDA_TRY(cudaMemcpyAsync(d_labels, comp + g->col_of_row0, (size_t)rows * 4, cudaMemcpyDeviceToDevice, st));
    rc = vglb_finish_run(ctx, launches0, stats);
    if (rc != VGLB_OK || !stats) return rc;
    stats->iterations = hook_rounds;
    stats->edges_inspected = hook_rounds * g->E;
    stats->vertices_processed = hook_rounds * (int64_t)rows;
    stats->frontier_bytes = hook_rounds * g->cols * 4 * 2; // the allreduced label vector
    stats->algorithmic_bytes = hook_rounds * (8 * g->E + 12 * (int64_t)rows) + (hook_rounds - 1) * 8 * g->cols + stats->frontier_bytes;
    return VGLB_OK;
}

extern "C" int vglb_cc(vglb_ctx *ctx, vglb_graph *g, int32_t *d_labels, vglb_stats *stats)
{
    VGLB_REQUIRE(ctx != NULL && g != NULL && d_labels != NULL, "vglb_cc: NULL argument");
    if (g->comm) return cc_partitioned(ctx, g, d_labels, stats);
    CUDA_TRY(cudaSetDevice(ctx->device));
    const int64_t launches0 = ctx->launches;
    const int32_t V = g->V;
    cudaStream_t st = ctx->stream;
    int *d_changed = (int *)(ctx->d_counters + 40);
    int *h_changed = (int *)(ctx->h_counters + 40);


    CUDA_TRY(cudaEventRecord(ctx->ev_start, st));
    cc_init_kernel<<<ctx->sm_count * 8, 256, 0, st>>>(d_labels, V);
    KERNEL_TRY();
    ctx->launches++;
    int64_t hook_rounds = 0;
    for (;;)
    {
        CUDA_TRY(cudaMemsetAsync(d_changed, 0, sizeof(int), st));
        int rc = cc_launch_hook(ctx, g, d_labels, 0, d_changed);
        if (rc != VGLB_OK) return rc;
        hook_rounds++;
        CUDA_TRY(cudaMemcpyAsync(h_changed, d_changed, sizeof(int), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        if (!*h_changed) break;
        cc_jump_kernel<<<ctx->sm_count * 8, 256, 0, st>>>(d_labels, V);
        KERNEL_TRY();
        ctx->launches++;
    }
    int rc = vglb_finish_run(ctx, launches0, stats);
    if (rc != VGLB_OK || !stats) return rc;
    stats->iterations = hook_rounds;
    stats->edges_inspected = hook_rounds * g->E;
    stats->vertices_processed = hook_rounds * (int64_t)V;
    stats->algorithmic_bytes = hook_rounds * (8 * g->E + 12 * (int64_t)V) + (hook_rounds - 1) * 8 * (int64_t)V;
    return VGLB_OK;
}
