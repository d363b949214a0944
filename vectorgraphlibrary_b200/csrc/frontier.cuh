// frontier.cuh — device-side pieces of the GPU frontier shared by bfs.cu / sssp.cu / frontier.cu:
// degree-binned sparse queues + dense bitmap (replaces FrontierVectorCSR's int flags[V] + int ids[V],
// vgl_datastructures/frontier/containers/vect_csr/frontier_vect_csr.h:5-53).
#pragma once
#include <type_traits>

#include "common.cuh"

struct TierQueues
{
    int32_t *q[3];       // big / mid / small regions
};

// queue regions over one V-entry buffer: capacity of a tier's queue = population of the tier (ids are degree-sorted)
static inline TierQueues tier_regions(int32_t *base, int32_t b0, int32_t b1)
{
    TierQueues q;
    q.q[0] = base;
    q.q[1] = base + b0;
    q.q[2] = base + b1;
    return q;
}

__device__ __forceinline__ bool bm_test(const uint32_t *bm, int32_t v) { return (bm[v >> 5] >> (v & 31)) & 1u; }

// warp-aggregated append of `v` (when `won`) to the queue of its degree tier
__device__ __forceinline__ void enqueue_binned(bool won, int32_t v, int32_t b0, int32_t b1, const TierQueues &nq,
                                               unsigned long long *counters)
{
    const int tier = v < b0 ? 0 : (v < b1 ? 1 : 2);
    const unsigned lane = threadIdx.x & 31;
#pragma unroll
    for (int t = 0; t < 3; t++)
    {
        const unsigned mask = __ballot_sync(0xffffffffu, won && tier == t);
        if (mask)
        {
            const int leader = __ffs(mask) - 1;
            unsigned long long base = 0;
            if ((int)lane == leader) base = atomicAdd(&counters[C_NEXT_BIG + t], (unsigned long long)__popc(mask));
            base = __shfl_sync(0xffffffffu, base, leader);
            if (won && tier == t) nq.q[t][base + __popc(mask & ((1u << lane) - 1u))] = v;
        }
    }
}

// bits of `word` (vertices base..base+31) whose id is < border
__device__ __forceinline__ uint32_t below_border_mask(int32_t base, int32_t border)
{
    if (base + 32 <= border) return 0xffffffffu;
    if (base >= border) return 0u;
    return (1u << (border - base)) - 1u;
}

#define BFS_BIG_DEGREE 512 // one GPU: rows with at least this many edges are big (a 2691-edge source row took one warp 150 us)

#define BFS_TD_UNROLL 4 // edges per thread and step: their loads, visited tests and atomics are independent

// one warp-aggregated queue claim per degree tier for BFS_TD_UNROLL candidates per lane
__device__ __forceinline__ void enqueue_binned_multi(const bool (&won)[BFS_TD_UNROLL], const int32_t (&v)[BFS_TD_UNROLL], int32_t b0,
                                                     int32_t b1, const TierQueues &nq, unsigned long long *counters)
{
    const unsigned lane = threadIdx.x & 31;
    const unsigned below = (1u << lane) - 1u;
#pragma unroll
    for (int t = 0; t < 3; t++)
    {
        unsigned mask[BFS_TD_UNROLL];
        int total = 0;
#pragma unroll
        for (int k = 0; k < BFS_TD_UNROLL; k++)
        {
            const int tier = v[k] < b0 ? 0 : (v[k] < b1 ? 1 : 2);
            mask[k] = __ballot_sync(0xffffffffu, won[k] && tier == t);
            total += __popc(mask[k]);
        }
        if (total == 0) continue;
        unsigned long long base = 0;
        if (lane == 0) base = atomicAdd(&counters[C_NEXT_BIG + t], (unsigned long long)total);
        base = __shfl_sync(0xffffffffu, base, 0);
#pragma unroll
        for (int k = 0; k < BFS_TD_UNROLL; k++)
        {
            if ((mask[k] >> lane) & 1u) nq.q[t][base + __popc(mask[k] & below)] = v[k];
            base += __popc(mask[k]);
        }
    }
}

#define BFS_THREADS 256
#define BFS_SMALL_LANES 8
#define BFS_BIG_CHUNK 8192 // a "big" row is expanded by CTAs, one per chunk of this many edges

// one top-down level: queued rows per tier and the CTAs of each part of the launch, in this order. The kernels take the
// fields as scalar parameters: as one struct parameter, bfs_td_kernel<0> took 48 registers instead of 40 and <3> spilled.
struct TdGrid
{
    int32_t n_big, hub_ctas, n_mid, n_small, blocks_mid, blocks_small;
    int64_t ctas() const { return (int64_t)hub_ctas + blocks_mid + blocks_small; }
};

// hub chunks go to at most 4 CTAs per SM, mid and small rows to at most 16 CTAs per SM each
static inline TdGrid td_grid(const vglb_ctx *ctx, const vglb_graph *g, const int32_t n[3])
{
    const int max_blocks = ctx->sm_count * 16;
    const int64_t big_chunks = ceil_div64(g->max_degree > 0 ? g->max_degree : 1, BFS_BIG_CHUNK);
    TdGrid L;
    L.n_big = n[0];
    L.n_mid = n[1];
    L.n_small = n[2];
    L.hub_ctas = (int)min((int64_t)n[0] * big_chunks, (int64_t)ctx->sm_count * 4);
    L.blocks_mid = (int)min((int64_t)max_blocks, ceil_div64(n[1], BFS_THREADS / 32));
    L.blocks_small = (int)min((int64_t)max_blocks, ceil_div64(n[2], BFS_THREADS / BFS_SMALL_LANES));
    return L;
}

// The top-down schedule of the BFS kernels (bfs.cu, bfs_multi.cu) over the queued rows cq of one level, launched with
// L.ctas() CTAs of BFS_THREADS threads. `expand(std::integral_constant<int, NT>(), u, s, e, tid)` is called for every
// (row or chunk, group of NT threads) the thread belongs to, with the edges [s, e) of row u and the thread's rank tid in
// the group; all lanes of a warp call it together (ballots inside), idle groups with u = -1 and s = e. `edges` counts the
// edges handed out, on one thread per group.
//   * hubs (the largest rows of a scale-26 Kronecker graph have > 10^6 edges): the queued hub rows are cut into
//     BFS_BIG_CHUNK-edge chunks and the chunks are dealt round-robin to L.hub_ctas CTAs (NT = BFS_THREADS). Every CTA stages
//     256 row ranges at a time in shared memory, scans their chunk counts (block prefix sum) and binary-searches the rows of
//     the chunks it owns — no CTA is launched for a chunk that does not exist (one CTA per (row, chunk slot of the LONGEST
//     row) launched hundreds of thousands of empty CTAs: 0.78 ms for an 18 M-edge level) and no CTA walks rows it has no
//     chunk of;
//   * one warp per mid row (NT = 32);
//   * BFS_SMALL_LANES lanes per small row (NT = BFS_SMALL_LANES), with a trip count padded to be uniform over the warp.
// ChunkCount is the type of the running chunk count (at most E / BFS_BIG_CHUNK + n_big, so int suffices). It sets the
// register allocation: with int, bfs_td_kernel<3> takes 32 registers instead of 40 and RMAT s20 top-down BFS ran 3 % slower on
// a B200; with long long, bfs_multi_td_kernel<uint32_t> spills.
template <class ChunkCount, class Expand>
__device__ __forceinline__ void td_schedule(const int64_t *__restrict__ ptr, const TierQueues &cq, const TdGrid &L, long long &edges,
                                            Expand &&expand)
{
    const int b = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int hub_ctas = L.hub_ctas, n_big = L.n_big;
    if (b < hub_ctas)
    {
        __shared__ int64_t s_row_start[BFS_THREADS], s_row_end[BFS_THREADS];
        __shared__ int s_chunk_prefix[BFS_THREADS + 1];
        __shared__ int s_warp_chunks[BFS_THREADS / 32];
        ChunkCount chunk_base = 0; // chunks of the batches before this one
        for (int base = 0; base < n_big; base += BFS_THREADS)
        {
            __syncthreads();
            int nch = 0;
            if (base + (int)threadIdx.x < n_big)
            {
                const int32_t u = cq.q[0][base + threadIdx.x];
                const int64_t rs = ptr[u], re = ptr[u + 1];
                s_row_start[threadIdx.x] = rs;
                s_row_end[threadIdx.x] = re;
                nch = (int)((re - rs + BFS_BIG_CHUNK - 1) / BFS_BIG_CHUNK);
            }
            int incl = nch;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1)
            {
                const int t = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += t;
            }
            if (lane == 31) s_warp_chunks[warp] = incl;
            __syncthreads();
            int wbase = 0;
#pragma unroll
            for (int w = 0; w < BFS_THREADS / 32; w++)
                if (w < warp) wbase += s_warp_chunks[w];
            s_chunk_prefix[threadIdx.x + 1] = wbase + incl;
            if (threadIdx.x == 0) s_chunk_prefix[0] = 0;
            __syncthreads();
            const int cnt = min(BFS_THREADS, n_big - base);
            const int total = s_chunk_prefix[cnt];
            int first = (int)((b - chunk_base % hub_ctas + hub_ctas) % hub_ctas);
            for (int c = first; c < total; c += hub_ctas)
            {
                int lo = 0, hi = cnt; // row k with prefix[k] <= c < prefix[k + 1]
                while (hi - lo > 1)
                {
                    const int mid = (lo + hi) >> 1;
                    if (s_chunk_prefix[mid] <= c) lo = mid;
                    else hi = mid;
                }
                const int64_t s = s_row_start[lo] + (int64_t)(c - s_chunk_prefix[lo]) * BFS_BIG_CHUNK, e = min(s_row_end[lo], s + BFS_BIG_CHUNK);
                if (threadIdx.x == 0) edges += e - s;
                expand(std::integral_constant<int, BFS_THREADS>(), cq.q[0][base + lo], s, e, (int)threadIdx.x);
            }
            chunk_base += total;
        }
    }
    else if (b < hub_ctas + L.blocks_mid)
    {
        const int nwarps = L.blocks_mid * (BFS_THREADS / 32);
        for (int i = (b - hub_ctas) * (BFS_THREADS / 32) + warp; i < L.n_mid; i += nwarps)
        {
            const int32_t u = cq.q[1][i];
            const int64_t s = ptr[u], e = ptr[u + 1];
            if (lane == 0) edges += e - s;
            expand(std::integral_constant<int, 32>(), u, s, e, lane);
        }
    }
    else
    {
        constexpr int G = BFS_SMALL_LANES;
        constexpr int GROUPS = BFS_THREADS / G;
        const int ngroups = L.blocks_small * GROUPS;
        const int gid = threadIdx.x / G, gl = threadIdx.x % G;
        const int first = (b - hub_ctas - L.blocks_mid) * GROUPS + gid;
        for (int base = first - gid; base < L.n_small; base += ngroups)
        {
            const int i = base + gid;
            int32_t u = -1;
            int64_t s = 0, e = 0;
            if (i < L.n_small)
            {
                u = cq.q[2][i];
                s = ptr[u];
                e = ptr[u + 1];
                if (gl == 0) edges += e - s;
            }
            expand(std::integral_constant<int, G>(), u, s, e, gl);
        }
    }
}

// direction heuristic of the reference (gpu_change_state, change_state.hpp:5-6,100-141): ALPHA 15, BETA 18
#define BFS_DEFAULT_ALPHA 15
#define BFS_DEFAULT_BETA 18

struct BfsDirection
{
    bool dopt; // direction-optimising
    long long alpha, beta, factor;
};

// E and V of the whole graph
static inline BfsDirection bfs_direction(const vglb_bfs_opts *opts, long long E, long long V)
{
    BfsDirection d;
    d.dopt = opts && opts->direction_optimising;
    d.alpha = (opts && opts->alpha > 0) ? opts->alpha : BFS_DEFAULT_ALPHA;
    d.beta = (opts && opts->beta > 0) ? opts->beta : BFS_DEFAULT_BETA;
    d.factor = (E / (V > 0 ? V : 1)) / 2 > 0 ? (E / V) / 2 : 1; // change_state.hpp:104
    return d;
}

// direction of the next level — gpu_change_state (change_state.hpp:100-141) on the frontier sizes of the level just done
// (n_cur -> n_next); the top-down test uses the out-edges of the next frontier (m_f), the edges the NEXT top-down level
// would inspect, instead of the level just done
static inline bool next_direction(const BfsDirection &d, bool bottom_up, long long n_cur, long long n_next, long long m_f,
                                  long long unvisited, long long V)
{
    if (!d.dopt) return bottom_up;
    if (!bottom_up) return n_cur < n_next && m_f >= (unvisited * d.factor + V) / d.alpha;
    return !(n_cur >= n_next && n_next < (unvisited * d.factor + V) / (d.factor * d.beta));
}

// bit v of g->d_scratch_i32 = vertex v has no in-edges; built once per graph that has an incoming CSR (bfs.cu)
int bfs_prepare_no_in_edges(vglb_ctx *ctx, vglb_graph *g);
// what vglb_bfs and vglb_bfs_multi share on one GPU, allocated or computed where missing: both tier queues, the no-in-edge
// mask and g->bfs_big_border_plus1 (bfs.cu)
int bfs_prepare_queues(vglb_ctx *ctx, vglb_graph *g);

// read-back of a partitioned level or round (frontier.cu): stages the counters [0, C_COUNT) at C_STAGED and C_MF at
// CTR_PENDING_MIN (one kernel), sums the staged copy over the ranks, copies `words` counters to ctx->h_counters and waits
// for them. [0, C_COUNT) stay this rank's own counts.
int vglb_part_round_counters(vglb_ctx *ctx, vglb_comm *comm, int words);
