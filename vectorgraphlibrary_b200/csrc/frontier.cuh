// frontier.cuh — device-side pieces of the GPU frontier shared by bfs.cu / sssp.cu / frontier.cu:
// degree-binned sparse queues + dense bitmap (replaces FrontierVectorCSR's int flags[V] + int ids[V],
// vgl_datastructures/frontier/containers/vect_csr/frontier_vect_csr.h:5-53).
#pragma once
#include "common.cuh"

// counter slots (unsigned long long) in ctx->d_counters
enum
{
    C_NEXT_BIG = 0,
    C_NEXT_MID = 1,
    C_NEXT_SMALL = 2,
    C_EDGES = 3,   // edges inspected this level
    C_FOUND = 4,   // vertices discovered this level
    C_MF = 5,      // sum of out-degrees of the next frontier
    C_ROWS = 6,    // rows whose pointer pair was read this level
    C_COUNT = 8
};

struct TierQueues
{
    int32_t *q[3];       // big / mid / small regions
};

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

// bit v of g->d_scratch_i32 = vertex v has no in-edges; built once per graph that has an incoming CSR (bfs.cu)
int bfs_prepare_no_in_edges(vglb_ctx *ctx, vglb_graph *g);
