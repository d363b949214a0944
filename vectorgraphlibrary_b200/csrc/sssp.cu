// sssp.cu — SSSP as frontier Bellman-Ford over the device VectCSR (sm_100a).
//
// Reference: ShortestPaths::vgl_dijkstra_partial_active (algorithms/sssp/shortest_paths.hpp:7-78): per round
//   compute(prev = dist) over all V, scatter(work_frontier, if dist[dst] > dist[src]+w then dist[dst] = dist[src]+w),
//   generate_new_frontier(dist != prev) over all V. The multicore relax is a racy non-atomic read-modify-write
//   (SURVEY §0 hazard 1); the GPU reference is racy too (sssp/gpu_shortest_paths.hpp:156-167). The parity target is
//   the unique min-plus fixed point in fp32 = ShortestPaths::seq_dijkstra (seq_shortest_paths.hpp:8-68), bit-exact:
//   every candidate is one fp32 add `dist[src] + w`, fp32 add is monotone, so the minimum over paths does not depend
//   on the relaxation order. Unreachable = FLT_MAX - 100 = FLT_MAX in fp32 (shortest_paths.hpp:22).
//
// B200 design
//   * distances of non-negative floats order like their bit patterns: relax = atomicMin on the uint32 view, after a
//     plain (L2-resident) read that filters the candidates that cannot win;
//   * the winner of an atomicMin marks the vertex in a "due" bitmap, so the next frontier comes from a 2 MB bitmap scan —
//     the reference's `prev = dist` copy and its V-pass generate_new_frontier (shortest_paths.hpp:40-44,58-66) disappear;
//   * near/far schedule (see vglb_sssp): only due vertices below a moving distance threshold are relaxed, which cuts
//     the edges relaxed on the BASELINE graph from 5.8 E (the reference's schedule) to ~1.2 E with bit-identical results;
//   * load balance: a warp takes up to 32 queued rows and walks the concatenation of their edge ranges (shuffle search
//     over the prefix sums), rows with >= 4096 edges get a CTA; column indices and weights are streamed
//     (ld.global.nc.L1::no_allocate + L2 evict-first), the distance vector is the L2-resident gather target.
// HBM roofline: algorithmic bytes = sum_rounds [ 12 e_i (index + weight + dist[dst]) + 24 f_i + 8 n(F_{i+1}) ] + scans.
#include <float.h>
#include <math.h>
#include <time.h>
#include <stdlib.h>

#include "common.cuh"
#include "frontier.cuh"

#define SSSP_THREADS 256
#define SSSP_SMALL_LANES 8

// Row-per-group relax used by the partitioned driver: NT threads (a CTA, a warp or an 8-lane group) stride the out-row
// [s,e) of one frontier vertex and lower the distances in this rank's replica of the vector (column ids); owners find
// their changed vertices after the allreduce(min).
template <int NT>
__device__ __forceinline__ void sssp_expand(const int32_t *__restrict__ adj, const float *__restrict__ wgt, int64_t s,
                                            int64_t e, int tid, float du, uint32_t *__restrict__ dist, uint64_t pol_stream)
{
    for (int64_t p = s + tid; p < e; p += NT)
    {
        const int32_t v = ld_stream_s32(adj + p, pol_stream);
        const float w = ld_stream_f32(wgt + p, pol_stream);
        const uint32_t cand = __float_as_uint(__fadd_rn(du, w)); // shortest_paths.hpp:50-53
        if (cand < dist[v]) atomicMin(&dist[v], cand);
    }
}

__global__ void __launch_bounds__(SSSP_THREADS)
sssp_relax_rows_kernel(const int64_t *__restrict__ ptr, const int32_t *__restrict__ adj, const float *__restrict__ wgt,
                       TierQueues cq, int32_t n_big, int32_t n_mid, int32_t n_small, int32_t blocks_mid, int32_t blocks_small,
                       uint32_t *__restrict__ dist, unsigned long long *counters, int32_t col0)
{
    const uint64_t pol = l2_policy_evict_first();
    const int b = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    long long edges = 0;
    if (b < n_big)
    {
        const int32_t u = cq.q[0][b];
        const int64_t s = ptr[u], e = ptr[u + 1];
        const float du = __uint_as_float(dist[col0 + u]);
        if (threadIdx.x == 0) edges = e - s;
        sssp_expand<SSSP_THREADS>(adj, wgt, s, e, threadIdx.x, du, dist, pol);
    }
    else if (b < n_big + blocks_mid)
    {
        const int nwarps = blocks_mid * (SSSP_THREADS / 32);
        for (int i = (b - n_big) * (SSSP_THREADS / 32) + warp; i < n_mid; i += nwarps)
        {
            const int32_t u = cq.q[1][i];
            const int64_t s = ptr[u], e = ptr[u + 1];
            const float du = __uint_as_float(dist[col0 + u]);
            if (lane == 0) edges += e - s;
            sssp_expand<32>(adj, wgt, s, e, lane, du, dist, pol);
        }
    }
    else
    {
        constexpr int G = SSSP_SMALL_LANES;
        constexpr int GROUPS = SSSP_THREADS / G;
        const int ngroups = blocks_small * GROUPS;
        const int gid = threadIdx.x / G, gl = threadIdx.x % G;
        for (int i = (b - n_big - blocks_mid) * GROUPS + gid; i < n_small; i += ngroups)
        {
            const int32_t u = cq.q[2][i];
            const int64_t s = ptr[u], e = ptr[u + 1];
            const float du = __uint_as_float(dist[col0 + u]);
            if (gl == 0) edges += e - s;
            sssp_expand<G>(adj, wgt, s, e, gl, du, dist, pol);
        }
    }
    edges = warp_sum_i64(edges);
    if (lane == 0 && edges) atomicAdd(&counters[C_EDGES], (unsigned long long)edges);
}

// ---- 1D-partitioned SSSP, dense exchange (fallback when the peers' replicas cannot be mapped) ---------------------------------------------------------------------------------------------
// Each rank relaxes the out-edges of the frontier vertices it owns into its replica of the distance vector (atomicMin),
// the replicas are combined with one allreduce(min) on the uint32 view per round — the reference MPI_Allreduce(MIN)es
// the same array after its advance (mpi_exchange.hpp:155-271, gpu_shortest_paths.hpp:133-196) — and every owner queues
// the vertices of its slice whose distance dropped (generate_new_frontier dist != prev, shortest_paths.hpp:58-66).

__global__ void sssp_part_init_kernel(uint32_t *__restrict__ dist, int64_t cols, int32_t source_col,
                                      uint32_t *__restrict__ prev, int32_t vp, int32_t src_row, int32_t *queue_slot)
{
    const uint32_t inf_bits = __float_as_uint(FLT_MAX - 100.0f);
    for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < cols; v += (int64_t)gridDim.x * blockDim.x)
    {
        dist[v] = v == source_col ? 0u : inf_bits;
        if (v < vp) prev[v] = (int32_t)v == src_row ? 0u : inf_bits;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0 && src_row >= 0) *queue_slot = src_row;
}

__global__ void __launch_bounds__(256)
sssp_part_frontier_kernel(const uint32_t *__restrict__ dist_slice, uint32_t *__restrict__ prev, int32_t rows, int32_t b0,
                          int32_t b1, TierQueues nq, unsigned long long *counters)
{
    const int32_t rpad = (rows + 31) & ~31;
    for (int32_t r = blockIdx.x * blockDim.x + threadIdx.x; r < rpad; r += gridDim.x * blockDim.x)
    {
        bool changed = false;
        if (r < rows)
        {
            const uint32_t d = dist_slice[r];
            if (d < prev[r])
            {
                prev[r] = d;
                changed = true;
            }
        }
        enqueue_binned(changed, r, b0, b1, nq, counters);
    }
}

__global__ void sssp_copy_counters_kernel(unsigned long long *c)
{
    if (threadIdx.x < C_COUNT) c[C_COUNT + threadIdx.x] = c[threadIdx.x];
}

static int sssp_partitioned_dense(vglb_ctx *ctx, vglb_graph *g, const float *d_weights, int32_t source, float *d_dist,
                            vglb_stats *stats)
{
    VGLB_REQUIRE(source >= 0 && source < g->cols, "vglb_sssp: source column out of range");
    CUDA_TRY(cudaSetDevice(ctx->device));
    vglb_comm *comm = g->comm;
    const int32_t rank = g->part_rank, vp = g->vp, rows = g->V, col0 = g->col_of_row0;
    if (!g->d_part_vec) CUDA_TRY(vglb_dev_alloc(&g->d_part_vec, (size_t)g->cols * 4));
    if (!g->d_part_prev) CUDA_TRY(vglb_dev_alloc(&g->d_part_prev, (size_t)vp * 4));
    if (!g->d_queue[0]) CUDA_TRY(vglb_dev_alloc(&g->d_queue[0], ((size_t)vp + 3) * 4));
    if (!g->d_queue[1]) CUDA_TRY(vglb_dev_alloc(&g->d_queue[1], ((size_t)vp + 3) * 4));
    const int64_t launches0 = ctx->launches;
    const int32_t b0 = g->tier_border[0], b1 = g->tier_border[1];
    unsigned long long *d_cnt = (unsigned long long *)ctx->d_counters;
    unsigned long long *h_cnt = (unsigned long long *)ctx->h_counters;
    cudaStream_t st = ctx->stream;
    uint32_t *dist = g->d_part_vec;
    auto regions = [&](int32_t *base) {
        TierQueues q;
        q.q[0] = base;
        q.q[1] = base + b0;
        q.q[2] = base + b1;
        return q;
    };
    TierQueues cq = regions(g->d_queue[0]), nq = regions(g->d_queue[1]);

    CUDA_TRY(cudaEventRecord(ctx->ev_start, st));
    const bool own_source = source / vp == rank;
    const int32_t src_row = own_source ? source - col0 : -1;
    VGLB_REQUIRE(!own_source || src_row < rows, "vglb_sssp: source is a padding column");
    const int src_tier = src_row < 0 ? 0 : (src_row < b0 ? 0 : (src_row < b1 ? 1 : 2));
    sssp_part_init_kernel<<<ctx->sm_count * 8, 256, 0, st>>>(dist, g->cols, source, g->d_part_prev, vp, src_row, cq.q[src_tier]);
    KERNEL_TRY();
    ctx->launches++;
    CUDA_TRY(cudaMemsetAsync(d_cnt, 0, 2 * C_COUNT * 8, st));
    int32_t n[3] = {0, 0, 0};
    if (own_source) n[src_tier] = 1;
    long long n_cur = 1;
    int64_t tot_edges = 0, tot_rows = 0, tot_next = 0, rounds = 0;
    const int max_blocks = ctx->sm_count * 16;
    int rc;
    while (n_cur > 0)
    {
        const int blocks_mid = (int)min((int64_t)max_blocks, ceil_div64(n[1], SSSP_THREADS / 32));
        const int blocks_small = (int)min((int64_t)max_blocks, ceil_div64(n[2], SSSP_THREADS / SSSP_SMALL_LANES));
        const int64_t grid = (int64_t)n[0] + blocks_mid + blocks_small;
        if (grid > 0)
        {
            sssp_relax_rows_kernel<<<(unsigned)grid, SSSP_THREADS, 0, st>>>(g->d_out_ptr, g->d_out_adj, d_weights, cq, n[0], n[1], n[2],
                                                                           blocks_mid, blocks_small, dist, d_cnt, col0);
            KERNEL_TRY();
            ctx->launches++;
        }
        rc = vglb_comm_allreduce_async(comm, dist, (size_t)g->cols, VGLB_DT_U32, VGLB_OP_MIN);
        if (rc != VGLB_OK) return rc;
        if (rows > 0)
        {
            sssp_part_frontier_kernel<<<(unsigned)min((int64_t)max_blocks, ceil_div64(rows, 256)), 256, 0, st>>>(
                dist + col0, g->d_part_prev, rows, b0, b1, nq, d_cnt);
            KERNEL_TRY();
        }
        sssp_copy_counters_kernel<<<1, 32, 0, st>>>(d_cnt);
        KERNEL_TRY();
        ctx->launches += 2;
        rc = vglb_comm_allreduce_async(comm, d_cnt + C_COUNT, C_COUNT, VGLB_DT_I64, VGLB_OP_SUM);
        if (rc != VGLB_OK) return rc;
        CUDA_TRY(cudaMemcpyAsync(h_cnt, d_cnt, 2 * C_COUNT * 8, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        CUDA_TRY(cudaMemsetAsync(d_cnt, 0, 2 * C_COUNT * 8, st));
        rounds++;
        tot_rows += (int64_t)n[0] + n[1] + n[2];
        tot_edges += (int64_t)h_cnt[C_EDGES];
        n[0] = (int32_t)h_cnt[C_NEXT_BIG];
        n[1] = (int32_t)h_cnt[C_NEXT_MID];
        n[2] = (int32_t)h_cnt[C_NEXT_SMALL];
        const unsigned long long *gl = h_cnt + C_COUNT;
        n_cur = (long long)(gl[C_NEXT_BIG] + gl[C_NEXT_MID] + gl[C_NEXT_SMALL]);
        tot_next += (int64_t)n[0] + n[1] + n[2];
        TierQueues t = cq; cq = nq; nq = t;
    }
    if (rows > 0) CUDA_TRY(cudaMemcpyAsync(d_dist, dist + col0, (size_t)rows * 4, cudaMemcpyDeviceToDevice, st));
    CUDA_TRY(cudaEventRecord(ctx->ev_stop, st));
    CUDA_TRY(cudaEventSynchronize(ctx->ev_stop));
    if (stats)
    {
        float ms = 0.f;
        CUDA_TRY(cudaEventElapsedTime(&ms, ctx->ev_start, ctx->ev_stop));
        memset(stats, 0, sizeof(*stats));
        stats->seconds = ms * 1e-3;
        stats->iterations = rounds;
        stats->edges_inspected = tot_edges; // this rank's
        stats->vertices_processed = tot_rows;
        stats->frontier_bytes = 8 * tot_next + rounds * g->cols * 4 * 2; // queues + the allreduced vector (read + written)
        stats->algorithmic_bytes = 12 * tot_edges + 24 * tot_rows + stats->frontier_bytes;
        stats->kernel_launches = ctx->launches - launches0;
    }
    return VGLB_OK;
}


// ---- load-balanced relax of the queued rows with < 4096 edges ("warp-level merge path") -------------------------------
// A warp takes 32 queue entries; lane j holds row j's edge range and source distance. The 32 ranges are concatenated
// (warp prefix sum of the degrees) and the warp walks the concatenation 32 * SSSP_FLAT_UNROLL edges at a time: every lane
// finds the row of its edge with a 5-step shuffle search over the prefix, so all lanes carry an edge whatever the degree
// mix, loads of one row are consecutive (the queue is ascending, so neighbouring rows are neighbours in memory too),
// and SSSP_FLAT_UNROLL independent index/weight loads are in flight per lane before the dependent distance gathers.
#ifndef SSSP_FLAT_UNROLL
#define SSSP_FLAT_UNROLL 4
#endif
// the gathered distance: kept in L2 ahead of the streamed adjacency / weights (evict-last hint), or a plain load
#ifndef SSSP_GATHER_KEEP
#define SSSP_GATHER_KEEP 1
#endif
#if SSSP_GATHER_KEEP
#define SSSP_GATHER(p) sssp_ld_keep((p), pol_keep)
#else
#define SSSP_GATHER(p) (*(p))
#endif
__device__ __forceinline__ uint32_t sssp_ld_keep(const uint32_t *p, uint64_t pol)
{
    uint32_t r;
    asm volatile("ld.global.L2::cache_hint.u32 %0, [%1], %2;" : "=r"(r) : "l"(p), "l"(pol));
    return r;
}
#ifndef SSSP_FIRE_AND_FORGET
#define SSSP_FIRE_AND_FORGET 1
#endif
#define SSSP_BIG_CHUNK 8192
#define SSSP_BIG_DEGREE 512  // rows with at least this many edges are relaxed by CTAs (the graph-wide tier border is 4096)
#ifndef SSSP_WARP_EDGES
#define SSSP_WARP_EDGES 1280
#endif

// relax one edge: atomicMin on the uint32 view after a plain read that filters the losers; the winner marks the vertex
// as due in the near (new distance below the threshold) or the far bitmap
__device__ __forceinline__ void sssp_relax_one(uint32_t *__restrict__ dist, uint32_t *__restrict__ near_bm,
                                               uint32_t *__restrict__ far_bm, uint32_t *__restrict__ changed_bm, int32_t col0,
                                               int32_t vp, uint32_t threshold_bits, int32_t v, uint32_t c)
{
    if (c < dist[v])
    {
        const uint32_t old = atomicMin(&dist[v], c);
        if (c < old)
        {
            // a vertex of this rank's slice (every vertex on one GPU) becomes due here; a vertex owned by a peer is
            // flagged in the changed bitmap, whose slices go to the owners after the round
            const uint32_t r = (uint32_t)(v - col0);
            const bool local = r < (uint32_t)vp;
            uint32_t *bm = local ? (c < threshold_bits ? near_bm : far_bm) : changed_bm;
            const uint32_t i = local ? r : (uint32_t)v;
            const uint32_t bit = 1u << (i & 31);
            if (!(bm[i >> 5] & bit)) atomicOr(&bm[i >> 5], bit);
        }
    }
}

// relax SSSP_FLAT_UNROLL edges whose destination distances have been gathered, in PHASES: all atomicMin of the step (they
// return the old value, so each is a full round trip), then the due-bitmap words of the winners, then the atomicOr marks.
// Edge by edge the winners of a step paid up to 2 x SSSP_FLAT_UNROLL dependent round trips; in phases two. (The gathers are
// issued together before any atomic for the same reason: an atomic orders the loads behind it.)
template <int N>
__device__ __forceinline__ void sssp_relax_batch(uint32_t *__restrict__ dist, uint32_t *__restrict__ near_bm, uint32_t *__restrict__ far_bm,
                                                 uint32_t *__restrict__ changed_bm, int32_t col0, int32_t vp, uint32_t threshold_bits,
                                                 const int32_t (&v)[N], const uint32_t (&c)[N], const uint32_t (&seen)[N])
{
#if SSSP_FIRE_AND_FORGET
    // Every candidate that beats the distance it saw lowers the distance AND marks the vertex due, both as reductions that
    // return nothing: no round trip left in the step after the gathers. A vertex may be marked by a candidate that lost to a
    // smaller one — it is due anyway (its distance dropped) — or, rarely, marked far by the loser and near by the winner: the far
    // select then queues it once more, which relaxes nothing new. Same fixed point.
#pragma unroll
    for (int k = 0; k < N; k++)
        if (v[k] >= 0 && c[k] < seen[k])
        {
            atomicMin(&dist[v[k]], c[k]);
            const uint32_t r = (uint32_t)(v[k] - col0);
            const bool local = r < (uint32_t)vp;
            uint32_t *bm = local ? (c[k] < threshold_bits ? near_bm : far_bm) : changed_bm;
            const uint32_t i = local ? r : (uint32_t)v[k];
            atomicOr(bm + (i >> 5), 1u << (i & 31));
        }
#else
    uint32_t old[N];
#pragma unroll
    for (int k = 0; k < N; k++) old[k] = (v[k] >= 0 && c[k] < seen[k]) ? atomicMin(&dist[v[k]], c[k]) : 0u;
    uint32_t *word_ptr[N];
    uint32_t word[N], bit[N];
#pragma unroll
    for (int k = 0; k < N; k++)
    {
        word_ptr[k] = NULL;
        word[k] = 0xffffffffu;
        bit[k] = 0;
        if (c[k] < old[k]) // (old is 0 for the edges that did not try)
        {
            // a vertex of this rank's slice (every vertex on one GPU) becomes due here; a vertex owned by a peer is flagged in
            // the changed bitmap, whose slices go to the owners after the round
            const uint32_t r = (uint32_t)(v[k] - col0);
            const bool local = r < (uint32_t)vp;
            uint32_t *bm = local ? (c[k] < threshold_bits ? near_bm : far_bm) : changed_bm;
            const uint32_t i = local ? r : (uint32_t)v[k];
            word_ptr[k] = bm + (i >> 5);
            bit[k] = 1u << (i & 31);
            word[k] = *word_ptr[k];
        }
    }
#pragma unroll
    for (int k = 0; k < N; k++)
        if (bit[k] && !(word[k] & bit[k])) atomicOr(word_ptr[k], bit[k]);
#endif
}

__global__ void __launch_bounds__(SSSP_THREADS)
sssp_relax_flat_kernel(const int64_t *__restrict__ ptr, const int32_t *__restrict__ adj, const float *__restrict__ wgt,
                       TierQueues cq, int32_t n_big, int32_t big_chunks, int32_t n_mid, int32_t n_small, int32_t per_warp_mid, int32_t per_warp,
                       uint32_t *__restrict__ dist, uint32_t *__restrict__ near_bm, uint32_t *__restrict__ far_bm,
                       uint32_t *__restrict__ changed_bm, int32_t col0, int32_t vp, uint32_t threshold_bits,
                       unsigned long long *counters)
{
    const unsigned FULL = 0xffffffffu;
    const uint64_t pol = l2_policy_evict_first();
    const uint64_t pol_keep = l2_policy_evict_last();
    (void)pol_keep;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    long long edges = 0;
    const int big_blocks = n_big * big_chunks;
    if ((int)blockIdx.x < big_blocks)
    {
        // a row with >= 4096 edges: one CTA per SSSP_BIG_CHUNK edges (hubs of power-law graphs have 10^5..10^6 edges and are
        // relaxed again whenever their distance drops), SSSP_FLAT_UNROLL independent edges per thread and step
        const int32_t u = cq.q[0][blockIdx.x / big_chunks];
        const int64_t s = ptr[u] + (int64_t)(blockIdx.x % big_chunks) * SSSP_BIG_CHUNK, e = min(ptr[u + 1], s + SSSP_BIG_CHUNK);
        if (s >= e) return;
        const float du = __uint_as_float(dist[col0 + u]);
        if (threadIdx.x == 0) edges = e - s;
        for (int64_t p0 = s + threadIdx.x; p0 < e; p0 += SSSP_THREADS * SSSP_FLAT_UNROLL)
        {
            int32_t v[SSSP_FLAT_UNROLL];
            uint32_t c[SSSP_FLAT_UNROLL];
#pragma unroll
            for (int k = 0; k < SSSP_FLAT_UNROLL; k++)
            {
                const int64_t p = p0 + (int64_t)k * SSSP_THREADS;
                v[k] = -1;
                c[k] = 0;
                if (p < e)
                {
                    v[k] = ld_stream_s32(adj + p, pol);
                    c[k] = __float_as_uint(__fadd_rn(du, ld_stream_f32(wgt + p, pol)));
                }
            }
            uint32_t seen[SSSP_FLAT_UNROLL];
#pragma unroll
            for (int k = 0; k < SSSP_FLAT_UNROLL; k++) seen[k] = v[k] >= 0 ? SSSP_GATHER(dist + v[k]) : 0u;
            sssp_relax_batch<SSSP_FLAT_UNROLL>(dist, near_bm, far_bm, changed_bm, col0, vp, threshold_bits, v, c, seen);
        }
    }
    else
    {
        // queue entries per warp (powers of two <= 32): few for the mid queue, whose rows have up to SSSP_BIG_DEGREE - 1 edges
        // each (a warp should not get much more than a few thousand edges), fewer than 32 for the small queue when the
        // frontier would otherwise leave SMs idle
        const int batches_mid = (n_mid + per_warp_mid - 1) / per_warp_mid, batches_small = (n_small + per_warp - 1) / per_warp;
        const int batch = ((int)blockIdx.x - big_blocks) * (SSSP_THREADS / 32) + warp;
        if (batch < batches_mid + batches_small)
        {
            const bool mid = batch < batches_mid;
            const int32_t *q = mid ? cq.q[1] : cq.q[2];
            const int n = mid ? n_mid : n_small;
            const int pw = mid ? per_warp_mid : per_warp;
            const int i = (mid ? batch : batch - batches_mid) * pw + lane;
            int64_t s = 0;
            int deg = 0;
            float du = 0.f;
            if (lane < pw && i < n)
            {
                const int32_t u = q[i];
                s = ptr[u];
                deg = (int)(ptr[u + 1] - s);
                du = __uint_as_float(dist[col0 + u]);
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
            if (lane == 0) edges = total;
            // per step: index / weight loads, then the step's distance gathers together, then its atomics (an atomic orders the
            // loads behind it). A/B on the BASELINE graph: prefetching step i + 1 before step i's gathers (40 registers, 75 %
            // occupancy) was 3 % SLOWER than this (32 registers, full occupancy): the kernel lives on resident warps.
            for (int base = 0; base < total; base += 32 * SSSP_FLAT_UNROLL)
            {
                int32_t v[SSSP_FLAT_UNROLL];
                uint32_t c[SSSP_FLAT_UNROLL], seen[SSSP_FLAT_UNROLL];
#pragma unroll
                for (int k = 0; k < SSSP_FLAT_UNROLL; k++)
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
                    const float duj = __shfl_sync(FULL, du, j);
                    v[k] = -1;
                    c[k] = 0;
                    if (idx < total)
                    {
                        const int64_t p = sj + (idx - exj);
                        v[k] = ld_stream_s32(adj + p, pol);
                        c[k] = __float_as_uint(__fadd_rn(duj, ld_stream_f32(wgt + p, pol))); // shortest_paths.hpp:50-53
                    }
                }
#pragma unroll
                for (int k = 0; k < SSSP_FLAT_UNROLL; k++) seen[k] = v[k] >= 0 ? SSSP_GATHER(dist + v[k]) : 0u;
                sssp_relax_batch<SSSP_FLAT_UNROLL>(dist, near_bm, far_bm, changed_bm, col0, vp, threshold_bits, v, c, seen);
            }
        }
    }
    edges = warp_sum_i64(edges);
    if (lane == 0 && edges) atomicAdd(&counters[C_EDGES], (unsigned long long)edges);
}

// ---- device-resident rounds for small frontiers (one GPU) ---------------------------------------------------------------
// Most rounds of a run are tiny: on the BASELINE graph 55 of 80 rounds relax fewer than 10^4 edges and cost ~30 us each —
// a select launch, a relax launch and a host read-back that decides what to launch next. One CTA drains such a stretch on
// the device instead: it keeps the frontier as an id list in shared memory, relaxes it (block-wide prefix sum of the
// degrees, every thread walks the flat edge range), and builds the next list on the fly — the thread whose atomicMin wins
// AND that is first to set the vertex's bit in the near bitmap appends it (the bitmap, empty when the drain starts, is the
// membership test). It returns to the host when the list runs empty (the near bucket is done: the host moves the
// threshold), or outgrows one CTA (the bits already set in the near bitmap ARE the pending list: the regular select /
// relax kernels take over). Same relaxations, same fixed point.
#define SSSP_DRAIN_THREADS 1024
#define SSSP_DRAIN_MAX_ROWS 1024   // one row per thread for the prefix sum
#define SSSP_DRAIN_MAX_EDGES 65536 // edges one CTA relaxes per round
#define SSSP_DRAIN_LIST 2048
enum { DRAIN_NOT_STARTED = 0, DRAIN_EMPTY = 1, DRAIN_PENDING = 2 };
// result slots in the counter block (after the 2 * C_COUNT + 1 words the host loop reads)
enum { DR_REASON = 2 * C_COUNT + 2, DR_ROUNDS, DR_ROWS, DR_END };

__global__ void __launch_bounds__(SSSP_DRAIN_THREADS)
sssp_drain_kernel(const int64_t *__restrict__ ptr, const int32_t *__restrict__ adj, const float *__restrict__ wgt, TierQueues cq,
                  int32_t n_big, int32_t n_mid, int32_t n_small, uint32_t *__restrict__ dist, uint32_t *__restrict__ near_bm,
                  uint32_t *__restrict__ far_bm, uint32_t threshold_bits, unsigned long long *counters)
{
    __shared__ int32_t s_list[2][SSSP_DRAIN_LIST];
    __shared__ int32_t s_prefix[SSSP_DRAIN_MAX_ROWS + 1];
    __shared__ int64_t s_start[SSSP_DRAIN_MAX_ROWS];
    __shared__ float s_du[SSSP_DRAIN_MAX_ROWS];
    __shared__ int32_t s_warp_tot[32];
    __shared__ int s_next_n, s_overflow;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int n_cur = n_big + n_mid + n_small, cur = 0;
    if (tid < n_cur) s_list[0][tid] = tid < n_big ? cq.q[0][tid] : (tid < n_big + n_mid ? cq.q[1][tid - n_big] : cq.q[2][tid - n_big - n_mid]);
    long long edges = 0, rows = 0;
    int rounds = 0, reason = DRAIN_NOT_STARTED;
    __syncthreads();
    for (;;)
    {
        // degrees of the current list and their block-wide exclusive prefix sum
        int32_t u = -1;
        int64_t start = 0;
        int deg = 0;
        if (tid < n_cur)
        {
            u = s_list[cur][tid];
            start = ptr[u];
            deg = (int)(ptr[u + 1] - start);
        }
        int incl = deg;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1)
        {
            const int t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) s_warp_tot[warp] = incl;
        if (tid == 0)
        {
            s_next_n = 0;
            s_overflow = 0;
        }
        __syncthreads();
        int warp_base = 0, total = 0;
#pragma unroll
        for (int w = 0; w < 32; w++)
        {
            const int t = s_warp_tot[w];
            if (w < warp) warp_base += t;
            total += t;
        }
        if (total > SSSP_DRAIN_MAX_EDGES)
        {
            // too much for one CTA. Round 0: nothing has been touched, the queue the host selected is still valid (the host
            // launches the regular relax). Later rounds: the list's bits are still set in the near bitmap.
            if (rounds > 0) reason = DRAIN_PENDING;
            break;
        }
        if (tid < n_cur)
        {
            // pop: the vertex leaves the due sets before its distance is read (a later drop re-queues it)
            const uint32_t bit = 1u << (u & 31);
            if (rounds > 0) atomicAnd(&near_bm[u >> 5], ~bit);
            if (far_bm[u >> 5] & bit) atomicAnd(&far_bm[u >> 5], ~bit);
            s_prefix[tid] = warp_base + incl - deg;
            s_start[tid] = start;
        }
        if (tid == 0) s_prefix[n_cur] = total;
        __threadfence_block();
        __syncthreads();
        if (tid < n_cur) s_du[tid] = __uint_as_float(dist[u]);
        __syncthreads();
        const int nxt = cur ^ 1;
        // 4 independent edges per thread and step (index / weight loads, then the distance gathers, then the atomics): one CTA
        // has little parallelism to hide latency with, so the loads of a step must not wait for each other
        for (int idx0 = tid; idx0 < total; idx0 += SSSP_DRAIN_THREADS * 4)
        {
            int32_t v[4];
            uint32_t c[4], dv[4];
#pragma unroll
            for (int k = 0; k < 4; k++)
            {
                const int idx = idx0 + k * SSSP_DRAIN_THREADS;
                v[k] = -1;
                c[k] = 0;
                if (idx < total)
                {
                    int lo = 0, hi = n_cur; // largest j with prefix[j] <= idx
                    while (hi - lo > 1)
                    {
                        const int mid = (lo + hi) >> 1;
                        if (s_prefix[mid] <= idx) lo = mid;
                        else hi = mid;
                    }
                    const int64_t p = s_start[lo] + (idx - s_prefix[lo]);
                    v[k] = adj[p];
                    c[k] = __float_as_uint(__fadd_rn(s_du[lo], wgt[p])); // shortest_paths.hpp:50-53
                }
            }
#pragma unroll
            for (int k = 0; k < 4; k++) dv[k] = v[k] >= 0 ? dist[v[k]] : 0u;
#pragma unroll
            for (int k = 0; k < 4; k++)
            {
                if (v[k] < 0 || c[k] >= dv[k]) continue;
                const uint32_t old = atomicMin(&dist[v[k]], c[k]);
                if (c[k] < old)
                {
                    const uint32_t bit = 1u << (v[k] & 31);
                    if (c[k] < threshold_bits)
                    {
                        if (!(atomicOr(&near_bm[v[k] >> 5], bit) & bit))
                        {
                            const int slot = atomicAdd(&s_next_n, 1);
                            if (slot < SSSP_DRAIN_LIST) s_list[nxt][slot] = v[k];
                            else s_overflow = 1;
                        }
                    }
                    else if (!(far_bm[v[k] >> 5] & bit)) atomicOr(&far_bm[v[k] >> 5], bit);
                }
            }
        }
        edges += total;
        rows += n_cur;
        rounds++;
        __syncthreads();
        const int n_next = s_next_n;
        if (n_next == 0)
        {
            reason = DRAIN_EMPTY;
            break;
        }
        if (s_overflow || n_next > SSSP_DRAIN_MAX_ROWS)
        {
            reason = DRAIN_PENDING;
            break;
        }
        n_cur = n_next;
        cur = nxt;
        __syncthreads();
    }
    if (tid == 0)
    {
        counters[C_EDGES] += (unsigned long long)edges;
        counters[DR_REASON] = (unsigned long long)reason;
        counters[DR_ROUNDS] = (unsigned long long)rounds;
        counters[DR_ROWS] = (unsigned long long)rows;
    }
}

// frontier selection of one round (generate_new_frontier, shortest_paths.hpp:58-66) from the due bitmaps: one thread
// per 32-vertex word. FAR = false: every bit of the near bitmap is due and below the threshold — the word is taken and
// cleared (and the same bits are cleared in the far bitmap: the vertex is being relaxed with a smaller distance).
// FAR = true (the near bitmap ran dry, the threshold moved): bits of the far bitmap whose distance is now below the
// threshold are taken, the rest are counted as pending and their minimum distance recorded. Queue slots are claimed
// once per CTA and degree tier.
template <bool FAR>
__global__ void __launch_bounds__(256)
sssp_select_kernel(uint32_t *__restrict__ near_bm, uint32_t *__restrict__ far_bm, const uint32_t *__restrict__ dist, int32_t rows,
                   uint32_t threshold_bits, int32_t b0, int32_t b1, TierQueues nq, unsigned long long *counters)
{
    __shared__ int s_count[8][3];
    __shared__ unsigned long long s_base[3];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int32_t nwords = (rows + 31) >> 5;
    const int32_t w = blockIdx.x * 256 + threadIdx.x;
    uint32_t take = 0;
    int pending = 0;
    uint32_t min_pending = 0xffffffffu;
    if (w < nwords)
    {
        if (!FAR)
        {
            take = near_bm[w];
            if (take)
            {
                near_bm[w] = 0;
                const uint32_t f = far_bm[w];
                if (f & take) far_bm[w] = f & ~take;
            }
        }
        else
        {
            uint32_t bits = far_bm[w];
            const uint32_t all = bits;
            while (bits)
            {
                const int b = __ffs(bits) - 1;
                bits &= bits - 1;
                const uint32_t d = dist[(w << 5) + b];
                if (d < threshold_bits) take |= 1u << b;
                else
                {
                    pending++;
                    min_pending = min(min_pending, d);
                }
            }
            if (take) far_bm[w] = all & ~take;
        }
    }
    const int32_t base = w << 5;
    const uint32_t m0 = below_border_mask(base, b0), m1 = below_border_mask(base, b1);
    uint32_t part[3] = {take & m0, take & m1 & ~m0, take & ~m1};
    int incl[3];
#pragma unroll
    for (int t = 0; t < 3; t++)
    {
        int x = __popc(part[t]);
#pragma unroll
        for (int o = 1; o < 32; o <<= 1)
        {
            const int y = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= o) x += y;
        }
        incl[t] = x;
        if (lane == 31) s_count[warp][t] = x;
    }
    __syncthreads();
    if (threadIdx.x < 3)
    {
        int total = 0;
#pragma unroll
        for (int i = 0; i < 8; i++) total += s_count[i][threadIdx.x];
        s_base[threadIdx.x] = total ? atomicAdd(&counters[C_NEXT_BIG + threadIdx.x], (unsigned long long)total) : 0ULL;
    }
    __syncthreads();
#pragma unroll
    for (int t = 0; t < 3; t++)
    {
        if (!part[t]) continue;
        unsigned long long pos = s_base[t] + incl[t] - __popc(part[t]);
        for (int i = 0; i < warp; i++) pos += s_count[i][t];
        uint32_t bits = part[t];
        while (bits)
        {
            const int b = __ffs(bits) - 1;
            bits &= bits - 1;
            nq.q[t][pos++] = base + b;
        }
    }
    if (FAR)
    {
        pending = (int)warp_sum_i64(pending);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) min_pending = min(min_pending, __shfl_xor_sync(0xffffffffu, min_pending, o));
        if (lane == 0 && pending)
        {
            atomicAdd(&counters[C_FOUND], (unsigned long long)pending);
            atomicMax(&counters[C_MF], (unsigned long long)(0xffffffffu - min_pending)); // min as max of the complement
        }
    }
}

// largest weight among a sample of the edge array (threshold step of the near/far split)
__global__ void sssp_weight_sample_kernel(const float *__restrict__ w, int64_t E, int64_t stride, unsigned int *out)
{
    float m = 0.f;
    for (int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * stride; i < E; i += (int64_t)gridDim.x * blockDim.x * stride)
        m = fmaxf(m, w[i]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) atomicMax(out, __float_as_uint(m));
}

// ---- sparse exchange of a partitioned round ---------------------------------------------------------------------------
// Sender side: the changed bitmap (one bit per column a relaxation of this round lowered in THIS rank's replica) is
// compacted, per owning rank q, into a contiguous list of (column << 32 | distance bits) entries; lists[q] counts them,
// the entries of owner q start at lists[P + q * vp]. The bits are cleared on the way. One thread per 32-column word;
// queue slots are claimed once per warp and owner (__match_any_sync groups the lanes by owner).
__global__ void __launch_bounds__(256)
sssp_compact_updates_kernel(uint32_t *__restrict__ changed_bm, const uint32_t *__restrict__ dist, int32_t words_full, int32_t wslice,
                            int32_t rank, int32_t P, int32_t vp, unsigned long long *__restrict__ lists)
{
    const int lane = threadIdx.x & 31;
    const int32_t w = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t bits = 0;
    int32_t q = -1;
    if (w < words_full)
    {
        q = w / wslice;
        if (q != rank) bits = changed_bm[w];
        if (bits) changed_bm[w] = 0;
    }
    const unsigned active = __ballot_sync(0xffffffffu, bits != 0);
    if (!bits) return;
    const unsigned peers = __match_any_sync(active, q); // lanes of this warp with updates for the same owner
    const int cnt = __popc(bits);
    // exclusive prefix of cnt over the lanes of `peers` below this lane, and the group total
    int before = 0, total = 0;
    for (unsigned m = peers; m;)
    {
        const int l = __ffs(m) - 1;
        m &= m - 1;
        const int c = __shfl_sync(peers, cnt, l);
        if (l < lane) before += c;
        total += c;
    }
    const int leader = __ffs(peers) - 1;
    unsigned long long base = 0;
    if (lane == leader) base = atomicAdd(&lists[q], (unsigned long long)total);
    base = __shfl_sync(peers, base, leader);
    unsigned long long *out = lists + P + (int64_t)q * vp + base + before;
    while (bits)
    {
        const int b = __ffs(bits) - 1;
        bits &= bits - 1;
        const uint32_t col = (uint32_t)(w << 5) + b;
        *out++ = ((unsigned long long)col << 32) | dist[col];
    }
}

// Owner side: read every peer's list for this rank out of the peer's memory (CUDA IPC peer loads over NVLink —
// contiguous 8-byte entries in full-width transactions; reading the flagged values one by one out of the peers'
// replicas ran at 6-8 G values/s, NVLink small-read bound), lower the owned distances and mark the improved vertices due.
__global__ void __launch_bounds__(256)
sssp_apply_updates_kernel(const unsigned long long *const *__restrict__ peer_lists, int32_t P, int32_t rank, int32_t vp, int32_t col0,
                          uint32_t *__restrict__ dist, uint32_t *__restrict__ near_bm, uint32_t *__restrict__ far_bm,
                          uint32_t threshold_bits, unsigned long long *counters)
{
    long long applied = 0;
    for (int p = 0; p < P; p++)
    {
        if (p == rank) continue;
        const unsigned long long *lists = peer_lists[p];
        const long long n = (long long)lists[rank];
        const unsigned long long *entries = lists + P + (int64_t)rank * vp;
        for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        {
            const unsigned long long e = entries[i];
            const uint32_t col = (uint32_t)(e >> 32), val = (uint32_t)e;
            applied++;
            if (val < dist[col])
            {
                const uint32_t old = atomicMin(&dist[col], val);
                if (val < old)
                {
                    const uint32_t r = col - (uint32_t)col0;
                    uint32_t *bm = val < threshold_bits ? near_bm : far_bm;
                    atomicOr(&bm[r >> 5], 1u << (r & 31));
                }
            }
        }
    }
    applied = warp_sum_i64(applied);
    if ((threadIdx.x & 31) == 0 && applied) atomicAdd(&counters[C_ROWS], (unsigned long long)applied);
}

__global__ void sssp_part_seed_kernel(uint32_t *__restrict__ dist, int64_t cols, int32_t source_col, uint32_t *near_bm, int32_t src_row)
{
    const uint32_t inf_bits = __float_as_uint(FLT_MAX - 100.0f);
    for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < cols; v += (int64_t)gridDim.x * blockDim.x)
        dist[v] = v == source_col ? 0u : inf_bits;
    if (blockIdx.x == 0 && threadIdx.x == 0 && src_row >= 0) near_bm[src_row >> 5] = 1u << (src_row & 31);
}

// counters [0, C_COUNT) -> [C_COUNT, 2 C_COUNT) (summed over ranks) and the pending minimum -> slot 2 C_COUNT (max over ranks)
__global__ void sssp_stage_counters_kernel(unsigned long long *c)
{
    if (threadIdx.x < C_COUNT) c[C_COUNT + threadIdx.x] = c[threadIdx.x];
    if (threadIdx.x == 0) c[2 * C_COUNT] = c[C_MF];
}

// Schedule. The reference relaxes the out-edges of EVERY vertex whose distance changed in the previous round
// (shortest_paths.hpp:40-66); on the BASELINE graph that re-relaxes each edge ~5.8 times. The fixed point does not
// depend on the schedule, so the frontier is split near/far: only due vertices with dist < threshold are relaxed; when
// none is left the threshold moves up by delta (or jumps to the smallest pending distance + delta).
// delta = sampled max weight * VGLB_SSSP_DELTA_SCALE / average degree (default scale 4; 0 = the reference's plain schedule).
// Distances stay bit-exact (same min-plus fixed point); edges_inspected reports the edges actually relaxed.
//
// One driver serves one GPU and a 1D-partitioned graph (g->comm != NULL). Partitioned: every rank relaxes the due
// vertices it owns into its own replica of the distance vector; vertices of its own slice become due on the spot,
// vertices owned by peers are flagged in a changed bitmap. After the round the bitmap slices go to the owners
// (all-to-all, V/8/P bytes per pair), each owner pulls the flagged values out of the peers' replicas (sssp_pull_kernel)
// and the round's counters are allreduced so that every rank takes the same scheduling decision. The reference's MPI
// build allreduces the whole array after every advance instead (mpi_exchange.hpp:155-271). When the peers' replicas
// cannot be mapped (no CUDA IPC), sssp_partitioned_dense (allreduce(min) of the vector, plain schedule) is used.
static int sssp_run(vglb_ctx *ctx, vglb_graph *g, const float *d_weights, int32_t source, float *d_dist, vglb_stats *stats)
{
    CUDA_TRY(cudaSetDevice(ctx->device));
    vglb_comm *comm = g->comm;
    const bool part = comm != NULL;
    const int32_t rows = g->V, vp = part ? g->vp : g->V, col0 = g->col_of_row0, P = g->part_world, rank = g->part_rank;
    if (g->sssp_big_border_plus1 == 0) // first id with fewer than SSSP_BIG_DEGREE edges (ids are degree-sorted), once per graph
    {
        int32_t border = 0;
        int rc0 = vglb_graph_threshold_vertex(ctx, g, SSSP_BIG_DEGREE, &border);
        if (rc0 != VGLB_OK) return rc0;
        g->sssp_big_border_plus1 = border + 1;
        // rows of the mid queue (32 <= degree < SSSP_BIG_DEGREE) handed to one warp: about SSSP_WARP_EDGES edges on average
        const int32_t mid_last = g->tier_border[1] > border ? g->tier_border[1] : border;
        int64_t pp[2] = {0, 0};
        CUDA_TRY(cudaMemcpyAsync(&pp[0], g->d_out_ptr + border, 8, cudaMemcpyDeviceToHost, ctx->stream));
        CUDA_TRY(cudaMemcpyAsync(&pp[1], g->d_out_ptr + mid_last, 8, cudaMemcpyDeviceToHost, ctx->stream));
        CUDA_TRY(cudaStreamSynchronize(ctx->stream));
        const int64_t avg = mid_last > border ? (pp[1] - pp[0]) / (mid_last - border) : 32;
        int rows_per_warp = 32;
        while (rows_per_warp > 1 && rows_per_warp * (avg > 0 ? avg : 1) > SSSP_WARP_EDGES) rows_per_warp >>= 1;
        g->sssp_mid_rows_per_warp = rows_per_warp;
    }
    const int32_t b0 = g->sssp_big_border_plus1 - 1, b1 = g->tier_border[1] > b0 ? g->tier_border[1] : b0;
    const size_t words = ((size_t)vp + 31) / 32;          // bitmaps over this rank's rows
    const int32_t wslice = (int32_t)words;
    const size_t words_full = (size_t)(g->cols + 31) / 32;  // changed bitmap over all columns
    if (!g->d_queue[0])
    {
        CUDA_TRY(vglb_dev_alloc(&g->d_queue[0], ((size_t)vp + 3) * 4));
        CUDA_TRY(vglb_dev_alloc(&g->d_queue[1], ((size_t)vp + 3) * 4));
    }
    if (!g->d_visited) CUDA_TRY(vglb_dev_alloc(&g->d_visited, (words + 32) * 4));
    if (!g->d_front_bm[0]) CUDA_TRY(vglb_dev_alloc(&g->d_front_bm[0], (words + 32) * 4));
    uint32_t *dist = (uint32_t *)d_dist, *changed_bm = NULL;
    const unsigned long long **d_peer_table = NULL;
    unsigned long long *lists = (unsigned long long *)g->d_part_lists;
    if (part)
    {
        if (!g->d_part_bm[0]) CUDA_TRY(vglb_dev_alloc(&g->d_part_bm[0], (words_full + 32) * 4));
        dist = g->d_part_vec;
        changed_bm = g->d_part_bm[0];
        d_peer_table = (const unsigned long long **)(ctx->d_counters + 24); // 8 device pointers
        CUDA_TRY(cudaMemcpyAsync(d_peer_table, g->d_vec_peer, sizeof(g->d_vec_peer), cudaMemcpyHostToDevice, ctx->stream));
    }
    const int64_t launches0 = ctx->launches;
    unsigned long long *d_cnt = (unsigned long long *)ctx->d_counters;
    unsigned long long *h_cnt = (unsigned long long *)ctx->h_counters;
    cudaStream_t st = ctx->stream;
    uint32_t *near_bm = g->d_visited, *far_bm = g->d_front_bm[0];
    TierQueues cq;
    cq.q[0] = g->d_queue[0];
    cq.q[1] = g->d_queue[0] + b0;
    cq.q[2] = g->d_queue[0] + b1;
    int rc;

    CUDA_TRY(cudaEventRecord(ctx->ev_start, st));
    // threshold step
    double scale = 4.0;
    if (const char *e = getenv("VGLB_SSSP_DELTA_SCALE")) scale = atof(e);
    float delta = 0.f; // 0 = plain schedule
    if (scale > 0.0 && g->E_global > 0)
    {
        unsigned int *d_max = (unsigned int *)(d_cnt + 60);
        CUDA_TRY(cudaMemsetAsync(d_max, 0, 4, st));
        if (g->E > 0)
        {
            const int64_t stride = g->E > (1 << 22) ? g->E >> 22 : 1;
            sssp_weight_sample_kernel<<<64, 256, 0, st>>>(d_weights, g->E, stride, d_max);
            KERNEL_TRY();
            ctx->launches++;
        }
        if (part)
        {
            rc = vglb_comm_allreduce_async(comm, d_max, 1, VGLB_DT_U32, VGLB_OP_MAX); // same delta on every rank
            if (rc != VGLB_OK) return rc;
        }
        unsigned int bits = 0;
        CUDA_TRY(cudaMemcpyAsync(&bits, d_max, 4, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        float wmax;
        memcpy(&wmax, &bits, 4);
        const double avg_deg = (double)g->E_global / (double)g->V_orig;
        delta = (float)(scale * (double)wmax / (avg_deg > 1.0 ? avg_deg : 1.0));
    }
    const bool trace = getenv("VGLB_SSSP_TRACE") != NULL; // developer aid: one line per selection on stderr
    double trace_t = 0.0;
    const float inf = FLT_MAX - 100.0f;
    const bool split = delta > 0.f && delta < inf;
    float threshold = split ? delta : inf;
    CUDA_TRY(cudaMemsetAsync(near_bm, 0, words * 4, st));
    CUDA_TRY(cudaMemsetAsync(far_bm, 0, words * 4, st));
    if (part) CUDA_TRY(cudaMemsetAsync(changed_bm, 0, words_full * 4, st));
    const int32_t src_row = source - col0; // the owner seeds its near bitmap
    sssp_part_seed_kernel<<<ctx->sm_count * 8, 256, 0, st>>>(dist, part ? g->cols : (int64_t)rows, source, near_bm,
                                                            (src_row >= 0 && src_row < rows) ? src_row : -1);
    KERNEL_TRY();
    CUDA_TRY(cudaMemsetAsync(d_cnt, 0, (2 * C_COUNT + 1) * 8, st));
    ctx->launches++;
    int64_t tot_edges = 0, tot_rows = 0, tot_next = 0, rounds = 0, selects = 0, far_selects = 0, tot_pulled = 0;
    const unsigned select_grid = (unsigned)ceil_div64((int64_t)words, 256);
    const int big_chunks = (int)ceil_div64(g->max_degree > 0 ? g->max_degree : 1, SSSP_BIG_CHUNK);
    bool from_far = false, far_nonempty = false;
    long long tot_queued_global = 0;
    const bool use_drain = !part && getenv("VGLB_SSSP_NO_DRAIN") == NULL; // developer knob: every round through the host
    bool near_known_empty = false; // the drain ran the near bucket dry: the next near select would find nothing
    for (;;)
    {
        uint32_t tbits;
        if (threshold >= inf) tbits = 0xffffffffu; // everything that is due
        else memcpy(&tbits, &threshold, 4);
        if (near_known_empty && !from_far)
        {
            // same decision as after a near select that queued nothing, without launching it
            near_known_empty = false;
            if (!split || (threshold >= inf && !far_nonempty)) break;
            from_far = true;
            if (threshold < inf) threshold += delta;
            continue;
        }
        near_known_empty = false;
        if (from_far) sssp_select_kernel<true><<<select_grid, 256, 0, st>>>(near_bm, far_bm, dist + col0, rows, tbits, b0, b1, cq, d_cnt);
        else sssp_select_kernel<false><<<select_grid, 256, 0, st>>>(near_bm, far_bm, dist + col0, rows, tbits, b0, b1, cq, d_cnt);
        KERNEL_TRY();
        ctx->launches++;
        selects++;
        far_selects += from_far;
        if (part)
        {
            sssp_stage_counters_kernel<<<1, 32, 0, st>>>(d_cnt);
            KERNEL_TRY();
            ctx->launches++;
            rc = vglb_comm_allreduce_async(comm, d_cnt + C_COUNT, C_COUNT, VGLB_DT_I64, VGLB_OP_SUM);
            if (rc != VGLB_OK) return rc;
        }
        if (part)
        {
            CUDA_TRY(cudaMemcpyAsync(h_cnt, d_cnt, (2 * C_COUNT + 1) * 8, cudaMemcpyDeviceToHost, st));
            CUDA_TRY(cudaStreamSynchronize(st));
        }
        else
        {
            rc = vglb_counters_fetch(ctx, d_cnt, 2 * C_COUNT + 1);
            if (rc != VGLB_OK) return rc;
        }
        CUDA_TRY(cudaMemsetAsync(d_cnt, 0, (2 * C_COUNT + 1) * 8, st));
        const int32_t n[3] = {(int32_t)h_cnt[C_NEXT_BIG], (int32_t)h_cnt[C_NEXT_MID], (int32_t)h_cnt[C_NEXT_SMALL]};
        const unsigned long long *gl = part ? h_cnt + C_COUNT : h_cnt; // whole-job sums drive the schedule
        const long long n_local = (long long)n[0] + n[1] + n[2];
        const long long n_cur = (long long)(gl[C_NEXT_BIG] + gl[C_NEXT_MID] + gl[C_NEXT_SMALL]), pending = (long long)gl[C_FOUND];
        tot_edges += (int64_t)h_cnt[C_EDGES]; // relaxed by the previous round (this rank)
        tot_pulled += (int64_t)h_cnt[C_ROWS];
        if (trace)
        {
            struct timespec ts;
            clock_gettime(CLOCK_MONOTONIC, &ts);
            const double now = (double)ts.tv_sec + 1e-9 * (double)ts.tv_nsec;
            fprintf(stderr, "sssp select %lld (%s): threshold %.3f queued %lld (local %lld) pending %lld, previous round relaxed %lld edges, pulled %lld, %.1f us since the previous line\n",
                    (long long)selects, from_far ? "far" : "near", threshold, n_cur, n_local, pending, (long long)h_cnt[C_EDGES],
                    (long long)h_cnt[C_ROWS], trace_t > 0.0 ? (now - trace_t) * 1e6 : 0.0);
            trace_t = now;
        }
        if (from_far) far_nonempty = pending > 0;
        if (from_far && split)
        {
            // once most of the graph has been relaxed and little is left, ordering buys nothing and every bucket of the long
            // tail of distances (power-law graphs) would cost two selections: the rest is relaxed the reference's way
            const long long Vg = g->V_orig;
            if (tot_queued_global >= Vg / 2 && n_cur + pending < (Vg / 64 > 4096 ? Vg / 64 : 4096)) threshold = inf;
        }
        if (n_cur == 0)
        {
            if (!from_far)
            {
                if (!split || (threshold >= inf && !far_nonempty)) break; // nothing can be parked in the far bitmap any more
                from_far = true;        // near ran dry: move the threshold and look at the far bitmap
                if (threshold < inf) threshold += delta;
                continue;
            }
            if (pending == 0) break;
            if (threshold >= inf) continue; // the threshold was just opened: take everything that is pending
            if (part)
            {
                // the smallest pending distance of the whole job (every rank takes this branch: same allreduced counters)
                unsigned long long *d_min = d_cnt + 2 * C_COUNT;
                CUDA_TRY(cudaMemcpyAsync(d_min, h_cnt + 2 * C_COUNT, 8, cudaMemcpyHostToDevice, st));
                rc = vglb_comm_allreduce_async(comm, d_min, 1, VGLB_DT_I64, VGLB_OP_MAX);
                if (rc != VGLB_OK) return rc;
                CUDA_TRY(cudaMemcpyAsync(h_cnt + 2 * C_COUNT, d_min, 8, cudaMemcpyDeviceToHost, st));
                CUDA_TRY(cudaStreamSynchronize(st));
                CUDA_TRY(cudaMemsetAsync(d_min, 0, 8, st));
            }
            const uint32_t min_bits = 0xffffffffu - (uint32_t)(part ? h_cnt[2 * C_COUNT] : h_cnt[C_MF]);
            float min_pending;
            memcpy(&min_pending, &min_bits, 4);
            // nothing below the moved threshold: jump. The far select takes d < threshold, so the new threshold must lie
            // strictly above min_pending; a delta below half an ulp of min_pending rounds away in the sum (a sampled
            // w_max that missed the heavy edges, a tiny VGLB_SSSP_DELTA_SCALE), and the same empty select would repeat
            const float jumped = fmaxf(threshold, min_pending) + delta;
            threshold = jumped > min_pending ? jumped : nextafterf(min_pending, INFINITY);
            continue;
        }
        from_far = false;
        if (tbits != 0xffffffffu) far_nonempty = true; // this round relaxes against a finite threshold: it may park vertices
        if (use_drain && n_cur <= SSSP_DRAIN_MAX_ROWS)
        {
            // a small frontier: one CTA runs this round and the following ones on the device until the bucket is empty or the
            // frontier has outgrown it
            sssp_drain_kernel<<<1, SSSP_DRAIN_THREADS, 0, st>>>(g->d_out_ptr, g->d_out_adj, d_weights, cq, n[0], n[1], n[2], dist, near_bm,
                                                               far_bm, tbits, d_cnt);
            KERNEL_TRY();
            ctx->launches++;
            rc = vglb_counters_fetch(ctx, d_cnt, DR_END);
            if (rc != VGLB_OK) return rc;
            CUDA_TRY(cudaMemsetAsync(d_cnt, 0, DR_END * 8, st));
            const int reason = (int)h_cnt[DR_REASON];
            if (reason != DRAIN_NOT_STARTED)
            {
                tot_edges += (int64_t)h_cnt[C_EDGES];
                rounds += (int64_t)h_cnt[DR_ROUNDS];
                tot_rows += (int64_t)h_cnt[DR_ROWS];
                tot_next += (int64_t)h_cnt[DR_ROWS];
                tot_queued_global += (long long)h_cnt[DR_ROWS];
                near_known_empty = reason == DRAIN_EMPTY;
                if (trace) fprintf(stderr, "sssp drain: %lld rounds, %lld rows, %lld edges on the device, %s\n", (long long)h_cnt[DR_ROUNDS],
                                   (long long)h_cnt[DR_ROWS], (long long)h_cnt[C_EDGES], near_known_empty ? "bucket empty" : "frontier outgrew one CTA");
                continue;
            }
            // (the few rows are too long for one CTA: the regular relax below takes them)
        }
        tot_queued_global += n_cur;
        if (n_local > 0)
        {
            // queue entries per warp: 32 when the frontier is large, fewer when it would leave SMs idle
            int per_warp = 32;
            while (per_warp > 1 && ceil_div64(n[1] + n[2], per_warp) < (int64_t)ctx->sm_count * 32) per_warp >>= 1;
            const int per_warp_mid = per_warp < g->sssp_mid_rows_per_warp ? per_warp : g->sssp_mid_rows_per_warp;
            const int64_t batches = ceil_div64(n[1], per_warp_mid) + ceil_div64(n[2], per_warp);
            const int64_t grid = (int64_t)n[0] * big_chunks + ceil_div64(batches, SSSP_THREADS / 32);
            sssp_relax_flat_kernel<<<(unsigned)grid, SSSP_THREADS, 0, st>>>(g->d_out_ptr, g->d_out_adj, d_weights, cq, n[0], big_chunks, n[1], n[2], per_warp_mid, per_warp,
                                                                           dist, near_bm, far_bm, changed_bm, col0, vp, tbits, d_cnt);
            KERNEL_TRY();
            ctx->launches++;
        }
        if (part)
        {
            CUDA_TRY(cudaMemsetAsync(lists, 0, (size_t)P * 8, st)); // list lengths (the peers finished reading: see below)
            sssp_compact_updates_kernel<<<(unsigned)ceil_div64((int64_t)words_full, 256), 256, 0, st>>>(changed_bm, dist, (int32_t)words_full, wslice,
                                                                                                       rank, P, vp, lists);
            KERNEL_TRY();
            // barrier: every rank's lists are complete before anybody reads them; the NEXT round's lists are not touched
            // before every rank has passed the next counter allreduce, i.e. finished reading these
            rc = vglb_comm_allreduce_async(comm, d_cnt + 2 * C_COUNT + 2, 1, VGLB_DT_I64, VGLB_OP_SUM);
            if (rc != VGLB_OK) return rc;
            sssp_apply_updates_kernel<<<ctx->sm_count * 8, 256, 0, st>>>(d_peer_table, P, rank, vp, col0, dist, near_bm, far_bm, tbits, d_cnt);
            KERNEL_TRY();
            ctx->launches += 2;
        }
        rounds++;
        tot_rows += n_local;
        tot_next += n_local;
    }
    if (part && rows > 0) CUDA_TRY(cudaMemcpyAsync(d_dist, dist + col0, (size_t)rows * 4, cudaMemcpyDeviceToDevice, st));
    CUDA_TRY(cudaEventRecord(ctx->ev_stop, st));
    CUDA_TRY(cudaEventSynchronize(ctx->ev_stop));
    if (stats)
    {
        float ms = 0.f;
        CUDA_TRY(cudaEventElapsedTime(&ms, ctx->ev_start, ctx->ev_stop));
        memset(stats, 0, sizeof(*stats));
        stats->seconds = ms * 1e-3;
        stats->iterations = rounds;
        stats->edges_inspected = tot_edges;
        stats->vertices_processed = tot_rows;
        // queues, bitmap scans, far-pile distance reads; partitioned: + the changed-bitmap scan of every round and, per
        // update received, 8 bytes written by the sender + 8 read over NVLink + the owner's 12-byte read-modify-write
        stats->frontier_bytes = 8 * tot_next + selects * (int64_t)words * 4 + far_selects * 4 * (int64_t)rows
                                + (part ? rounds * (int64_t)words_full * 4 + 28 * tot_pulled : 0);
        stats->algorithmic_bytes = 12 * tot_edges + 24 * tot_rows + stats->frontier_bytes; // SURVEY §8(d)
        stats->kernel_launches = ctx->launches - launches0;
    }
    return VGLB_OK;
}

extern "C" int vglb_sssp(vglb_ctx *ctx, vglb_graph *g, const float *d_weights, int32_t source, float *d_dist,
                         vglb_stats *stats)
{
    VGLB_REQUIRE(ctx != NULL && g != NULL && d_dist != NULL, "vglb_sssp: NULL argument");
    VGLB_REQUIRE(d_weights != NULL || g->E == 0, "vglb_sssp: NULL weights");
    VGLB_REQUIRE(source >= 0 && source < g->cols, "vglb_sssp: source out of range");
    if (g->comm)
    {
        VGLB_REQUIRE(g->d_bwd != NULL, "vglb_sssp: partitioned graph without a column map");
        CUDA_TRY(cudaSetDevice(ctx->device));
        if (!g->d_part_vec) CUDA_TRY(vglb_dev_alloc(&g->d_part_vec, (size_t)g->cols * 4));
        int rc = vglb_part_map_lists(ctx, g); // per-owner update lists, mapped into the peers once per graph
        if (rc != VGLB_OK) return rc;
        if (g->vec_peers_mapped < 0) return sssp_partitioned_dense(ctx, g, d_weights, source, d_dist, stats);
    }
    return sssp_run(ctx, g, d_weights, source, d_dist, stats);
}
