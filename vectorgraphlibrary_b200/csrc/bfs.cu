// bfs.cu — direction-optimising BFS over the device VectCSR (sm_100a): top-down advance with degree-binned sparse
// queues, bottom-up advance over a dense bitmap, and the conversions between the two frontier forms.
//
// Reference: BFS::fast_vgl_top_down (algorithms/bfs/bfs.hpp:5-51) = per level one scatter (advance) + one
// generate_new_frontier; the DO heuristic gpu_change_state (algorithms/bfs/change_state/change_state.hpp:100-141,
// ALPHA 15 / BETA 18 :5-6); the dead hand-wired DO code (hardwired_do_bfs.hpp:859-1009) for the loop structure.
// Levels are unique whatever direction is taken: source = 1, unreachable = -1 (change_state.h:21-23).
//
// B200 design
//   * the next frontier is emitted INSIDE the advance (the thread that wins the atomicOr on the visited bitmap
//     enqueues), instead of the reference's separate 2-pass generate_new_frontier over all V
//     (multicore/generate_new_frontier.hpp:35-108 = 34 % of its BFS time);
//   * sparse frontier = three queues binned by degree tier; the tier of a vertex is a comparison of its id with two
//     borders because ids are degree-sorted: CTA per vertex (deg >= 4096), warp per vertex (deg >= 32), 8 lanes per
//     vertex (the tail) — replaces the ve / vc / collective kernels of multicore/advance_sparse.hpp:7-249;
//   * dense frontier = bitmap (V/8 bytes: 8 MiB at scale 26, L2-resident); bottom-up assigns one warp to one 32-vertex
//     word of the visited bitmap, so next-frontier and visited words are written without atomics; each lane probes the
//     first few in-neighbours of its vertex, longer rows are finished warp-cooperatively with ballot early exit;
//     in-rows list sources in ascending id = descending out-degree, so the likeliest parents come first;
//   * queue <-> bitmap conversion: ballot/popc + warp-aggregated atomics (north_star (c)).
// One host read-back of 8 counters per level drives termination and the direction switch.
#include <stdlib.h>

#include "common.cuh"
#include "frontier.cuh"

#include <time.h>
static double trace_now()
{
    struct timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return (double)ts.tv_sec + 1e-9 * (double)ts.tv_nsec;
}

// direction heuristic of the reference (gpu_change_state, change_state.hpp:5-6,100-141): ALPHA 15, BETA 18
#define BFS_DEFAULT_ALPHA 15
#define BFS_DEFAULT_BETA 18
#define BFS_THREADS 256
#define BFS_SMALL_LANES 8
#define BFS_BU_PROBE 4       // in-neighbours probed per batch by one lane
#define BFS_BU_PROBE_MAX 16  // lane-private probes before the warp takes the row over
#define BFS_BIG_CHUNK 8192 // a "big" row is expanded by CTAs, one per chunk of this many edges

// NT threads (a CTA, a warp or an 8-lane group) expand the out-row [s,e) of one frontier vertex.
// Every thread of the warp must call this together (ballots inside); `e <= s` for idle groups.
// PART = the graph is one rank's part: `visited` is the replicated bitmap (read only here) and discoveries are only
// marked in the candidate bitmap `levels` points to (reinterpreted) — owners resolve them after the exchange.
// how a partitioned top-down level hands a discovery to the vertex's owner
struct PartArgs
{
    int32_t col0, vp, P, rank;
    int32_t visited_via_l2; // developer A/B knob (VGLB_BFS_VISITED_L2): test the visited bitmap with L2 (.cg) loads instead of L1-cached ones
    unsigned long long *lists; // P counters, then vp 4-byte entries per owner starting at byte offset 8 * P
};

__device__ __forceinline__ uint32_t *part_list_entries(const PartArgs &A, int q)
{
    return reinterpret_cast<uint32_t *>(A.lists + A.P) + (int64_t)q * A.vp;
}

// append the columns this warp discovered for other ranks to the lists of their owners: one slot claim per owner and warp
__device__ __forceinline__ void append_remote(const PartArgs &A, bool remote, int32_t v)
{
    const unsigned active = __ballot_sync(0xffffffffu, remote);
    if (!remote) return;
    const int lane = threadIdx.x & 31;
    const int q = v / A.vp;
    const unsigned same = __match_any_sync(active, q);
    const int leader = __ffs(same) - 1;
    unsigned long long base = 0;
    if (lane == leader) base = atomicAdd(&A.lists[q], (unsigned long long)__popc(same));
    base = __shfl_sync(same, base, leader);
    part_list_entries(A, q)[base + __popc(same & ((1u << lane) - 1u))] = (uint32_t)v;
}

// NT threads (a CTA, a warp or an 8-lane group) expand the out-row [s,e) of one frontier vertex.
// Every thread of the warp must call this together (ballots inside); `e <= s` for idle groups.
// MODE 0: one GPU. MODE 1: one rank's part, discoveries marked in a candidate bitmap (`levels` reinterpreted) that the
// owners resolve after an all-to-all. MODE 2: one rank's part, `visited` is this rank's replica: the first thread to set
// a bit either owns the vertex (level written, queued by local row) or appends the column to its owner's list.
template <int NT, int MODE>
__device__ __forceinline__ void td_expand(const int64_t *__restrict__ ptr, const int32_t *__restrict__ adj, int64_t s, int64_t e, int tid,
                                          uint32_t *__restrict__ visited, int32_t *__restrict__ levels, int32_t next_level,
                                          int32_t b0, int32_t b1, const TierQueues &nq, unsigned long long *counters, long long &mf,
                                          const PartArgs &A, int &found)
{
    for (int64_t p0 = s + tid;; p0 += NT * BFS_TD_UNROLL)
    {
        if (!__any_sync(0xffffffffu, p0 < e)) break;
        bool won[BFS_TD_UNROLL];
        int32_t v[BFS_TD_UNROLL];
#pragma unroll
        for (int k = 0; k < BFS_TD_UNROLL; k++)
        {
            const int64_t p = p0 + (int64_t)k * NT;
            v[k] = p < e ? adj[p] : -1;
            won[k] = false;
        }
        uint32_t seen[BFS_TD_UNROLL];
#pragma unroll
        // (L1-cached: a stale "unvisited" only costs an atomic that cannot win, while the hubs' words — most of the edges of a big
        // level point at them — are answered by L1 instead of L2: top-down-only Kronecker s26 22.3 -> 8.6 ms, RMAT s20 0.75 -> 0.46 ms)
        for (int k = 0; k < BFS_TD_UNROLL; k++)
            seen[k] = v[k] >= 0 ? (A.visited_via_l2 ? __ldcg(&visited[v[k] >> 5]) : visited[v[k] >> 5]) : 0xffffffffu;
#pragma unroll
        for (int k = 0; k < BFS_TD_UNROLL; k++)
        {
            if (v[k] < 0) continue;
            const uint32_t bit = 1u << (v[k] & 31);
            if (seen[k] & bit) continue;
            if (MODE == 1)
            {
                uint32_t *cand = reinterpret_cast<uint32_t *>(levels);
                if (!(cand[v[k] >> 5] & bit)) atomicOr(&cand[v[k] >> 5], bit);
            }
            else
            {
                const uint32_t old = atomicOr(&visited[v[k] >> 5], bit);
                won[k] = !(old & bit);
            }
        }
        if (MODE == 0 || MODE == 3)
        {
#pragma unroll
            for (int k = 0; k < BFS_TD_UNROLL; k++)
                if (won[k])
                {
                    levels[v[k]] = next_level;
                    mf += ptr[v[k] + 1] - ptr[v[k]]; // out-degree of the new frontier (m_f of the direction heuristic)
                    if (MODE == 3)
                    {
                        // a level that discovers millions of vertices: the next frontier is emitted as a BITMAP (scattered
                        // atomicOr) instead of through the three queue counters, whose same-address atomics serialise
                        // (0.78 ms for an 18 M-edge / 4.8 M-discovery level); the next level is bottom-up more often than not
                        uint32_t *next_bm = reinterpret_cast<uint32_t *>(A.lists);
                        atomicOr(&next_bm[v[k] >> 5], 1u << (v[k] & 31));
                        found++;
                    }
                }
            if (MODE == 0) enqueue_binned_multi(won, v, b0, b1, nq, counters);
        }
        if (MODE == 2)
        {
            bool mine[BFS_TD_UNROLL];
            int32_t row[BFS_TD_UNROLL];
#pragma unroll
            for (int k = 0; k < BFS_TD_UNROLL; k++)
            {
                row[k] = v[k] - A.col0;
                mine[k] = won[k] && (uint32_t)row[k] < (uint32_t)A.vp;
                if (mine[k])
                {
                    levels[row[k]] = next_level;
                    mf += ptr[row[k] + 1] - ptr[row[k]];
                }
                if (__any_sync(0xffffffffu, won[k] && !mine[k])) append_remote(A, won[k] && !mine[k], v[k]);
            }
            enqueue_binned_multi(mine, row, b0, b1, nq, counters);
        }
    }
}

template <int MODE>
__global__ void __launch_bounds__(BFS_THREADS)
bfs_td_kernel(const int64_t *__restrict__ ptr, const int32_t *__restrict__ adj, TierQueues cq, int32_t n_big, int32_t hub_ctas,
              int32_t n_mid, int32_t n_small, int32_t blocks_mid, int32_t blocks_small, uint32_t *__restrict__ visited,
              int32_t *__restrict__ levels, int32_t next_level, int32_t b0, int32_t b1, TierQueues nq,
              unsigned long long *counters, PartArgs A)
{
    const int b = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    long long edges = 0, mf = 0;
    int found = 0;
    // hubs (>= 4096 edges; the largest rows of a scale-26 Kronecker graph have > 10^6): the queued hub rows are cut into
    // BFS_BIG_CHUNK-edge chunks and the chunks are dealt round-robin to `hub_ctas` CTAs. Every CTA stages 256 row ranges at a
    // time in shared memory, scans their chunk counts (block prefix sum) and binary-searches the rows of the chunks it owns —
    // no CTA is launched for a chunk that does not exist (one CTA per (row, chunk slot of the LONGEST row) launched
    // hundreds of thousands of empty CTAs: 0.78 ms for an 18 M-edge level) and no CTA walks rows it has no chunk of.
    const int big_blocks = hub_ctas;
    if (b < big_blocks)
    {
        __shared__ int64_t s_row_start[BFS_THREADS], s_row_end[BFS_THREADS];
        __shared__ int s_chunk_prefix[BFS_THREADS + 1];
        __shared__ int s_warp_chunks[BFS_THREADS / 32];
        long long chunk_base = 0; // chunks of the batches before this one
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
                td_expand<BFS_THREADS, MODE>(ptr, adj, s, e, threadIdx.x, visited, levels, next_level, b0, b1, nq, counters, mf, A, found);
            }
            chunk_base += total;
        }
    }
    else if (b < big_blocks + blocks_mid)
    {
        const int nwarps = blocks_mid * (BFS_THREADS / 32);
        for (int i = (b - big_blocks) * (BFS_THREADS / 32) + warp; i < n_mid; i += nwarps)
        {
            const int32_t u = cq.q[1][i];
            const int64_t s = ptr[u], e = ptr[u + 1];
            if (lane == 0) edges += e - s;
            td_expand<32, MODE>(ptr, adj, s, e, lane, visited, levels, next_level, b0, b1, nq, counters, mf, A, found);
        }
    }
    else
    {
        constexpr int G = BFS_SMALL_LANES;
        constexpr int GROUPS = BFS_THREADS / G;
        const int ngroups = blocks_small * GROUPS;
        const int gid = threadIdx.x / G, gl = threadIdx.x % G;
        // all groups of a warp iterate together (ballots in td_expand): pad the trip count to a multiple of the stride
        const int first = (b - big_blocks - blocks_mid) * GROUPS + gid;
        for (int base = first - gid; base < n_small; base += ngroups)
        {
            const int i = base + gid;
            int64_t s = 0, e = 0;
            if (i < n_small)
            {
                const int32_t u = cq.q[2][i];
                s = ptr[u];
                e = ptr[u + 1];
                if (gl == 0) edges += e - s;
            }
            td_expand<G, MODE>(ptr, adj, s, e, gl, visited, levels, next_level, b0, b1, nq, counters, mf, A, found);
        }
    }
    edges = warp_sum_i64(edges);
    mf = warp_sum_i64(mf);
    if (lane == 0 && edges) atomicAdd(&counters[C_EDGES], (unsigned long long)edges);
    if (lane == 0 && mf) atomicAdd(&counters[C_MF], (unsigned long long)mf);
    if (MODE == 3)
    {
        found = (int)warp_sum_i64(found);
        if (lane == 0 && found) atomicAdd(&counters[C_FOUND], (unsigned long long)found);
    }
}

// owner side of a partitioned top-down level: the peers' lists of columns they discovered in this rank's slice, read out
// of the peers' memory (CUDA IPC). The first claim of a vertex in the owner's visited slice makes the discovery real.
__global__ void __launch_bounds__(256)
bfs_apply_lists_kernel(const unsigned long long *const *__restrict__ peer_lists, PartArgs A, const int64_t *__restrict__ ptr,
                       uint32_t *__restrict__ visited, int32_t *__restrict__ levels_local, int32_t next_level, int32_t b0, int32_t b1,
                       TierQueues nq, unsigned long long *counters)
{
    long long mf = 0;
    for (int p = 0; p < A.P; p++)
    {
        if (p == A.rank) continue;
        const unsigned long long *lists = peer_lists[p];
        const long long n = (long long)lists[A.rank];
        const uint32_t *entries = reinterpret_cast<const uint32_t *>(lists + A.P) + (int64_t)A.rank * A.vp;
        const long long n_padded = (n + 31) & ~31LL;
        for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_padded; i += (long long)gridDim.x * blockDim.x)
        {
            bool won = false;
            int32_t row = 0;
            if (i < n)
            {
                const uint32_t v = entries[i];
                const uint32_t bit = 1u << (v & 31);
                if (!(visited[v >> 5] & bit)) won = !(atomicOr(&visited[v >> 5], bit) & bit);
                row = (int32_t)v - A.col0;
                if (won)
                {
                    levels_local[row] = next_level;
                    mf += ptr[row + 1] - ptr[row];
                }
            }
            enqueue_binned(won, row, b0, b1, nq, counters);
        }
    }
    mf = warp_sum_i64(mf);
    if ((threadIdx.x & 31) == 0 && mf) atomicAdd(&counters[C_MF], (unsigned long long)mf);
}

// bottom-up step. A warp takes 32 consecutive words of the visited bitmap per pass (1024 vertices): lane l loads word l (one
// coalesced 128-byte read) and works out which of its 32 vertices still need a parent (unvisited, with in-edges); groups
// without such vertices — most of them in the late levels — cost nothing more. The candidates are then COMPACTED through
// shared memory (lane l deposits the bit positions of its word behind a warp prefix sum of the popcounts), so that the probe
// phase runs with every lane on a real candidate whatever the density: in the first bottom-up level half of the vertices have
// no in-edges and later levels have a handful of candidates per word — one lane per bit position ran at 25-50 % SIMD
// efficiency and the kernel was issue-bound (63 % of the issue slots, 280 instructions per 32 vertices). Per candidate:
// lane-private probes of the first in-neighbours, BFS_BU_PROBE at a time (the ids and then the frontier bits are independent
// loads), BFS_BU_CAND candidates in flight per lane; rows longer than BFS_BU_PROBE_MAX are finished warp-cooperatively, 256
// neighbours per round trip, with ballot early exit. In-rows list sources hubs-first. Results go back through a per-warp
// shared-memory copy of the 32 words, so bitmap words are written without global atomics.
#define BFS_BU_CAND 4        // candidates in flight per lane
#define BFS_BU_LONG_UNROLL 8
#ifndef BFS_BU_MIN_CTAS
#define BFS_BU_MIN_CTAS 4 // 64 registers. A/B on Kronecker s26: 5 CTAs/SM (48 registers, one resident wave) 1.09-1.11 ms vs 1.06-1.07 ms
#endif

__global__ void __launch_bounds__(BFS_THREADS, BFS_BU_MIN_CTAS)
bfs_bu_kernel(const int64_t *__restrict__ in_ptr, const int32_t *__restrict__ in_adj, int32_t V, const uint32_t *__restrict__ no_in_edges,
              uint32_t *__restrict__ visited, const uint32_t *__restrict__ cur_bm, uint32_t *__restrict__ next_bm,
              int32_t *__restrict__ levels, int32_t next_level, unsigned long long *counters)
{
    const unsigned FULL = 0xffffffffu;
    __shared__ uint16_t s_cand[BFS_THREADS / 32][1024]; // offsets (0..1023) of the group's candidates, ascending
    __shared__ uint32_t s_found[BFS_THREADS / 32][32];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int64_t nwords = ((int64_t)V + 31) >> 5;
    uint16_t *cand = s_cand[wib];
    uint32_t *fnd_words = s_found[wib];
    int edges = 0, rows = 0, found_total = 0;
    for (int64_t wbase = warp * 32; wbase < nwords; wbase += nwarps * 32)
    {
        const int64_t wl = wbase + lane;
        uint32_t vis_l = 0, unv_l = 0;
        if (wl < nwords)
        {
            vis_l = visited[wl];
            const uint32_t valid = (wl == nwords - 1 && (V & 31)) ? ((1u << (V & 31)) - 1u) : 0xffffffffu;
            // vertices without in-edges can never be found from below (half of a Kronecker graph): not even their row
            // pointers are read
            unv_l = ~vis_l & valid & ~no_in_edges[wl];
        }
        int incl = __popc(unv_l);
        const int cnt_l = incl;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1)
        {
            const int t = __shfl_up_sync(FULL, incl, o);
            if (lane >= o) incl += t;
        }
        const int total = __shfl_sync(FULL, incl, 31);
        if (total == 0)
        {
            if (wl < nwords) next_bm[wl] = 0;
            continue;
        }
        // deposit: lane l writes the offsets of its word's candidates behind the candidates of the lower words
        {
            int pos = incl - cnt_l;
            uint32_t bits = unv_l;
            while (bits)
            {
                const int bpos = __ffs(bits) - 1;
                bits &= bits - 1;
                cand[pos++] = (uint16_t)((lane << 5) | bpos);
            }
        }
        fnd_words[lane] = 0;
        __syncwarp();
        rows += (lane == 0) ? total : 0;
        const int64_t vbase = wbase << 5;
        for (int i0 = 0; i0 < total; i0 += 32 * BFS_BU_CAND)
        {
            int off[BFS_BU_CAND];
            int64_t s[BFS_BU_CAND];
            int deg[BFS_BU_CAND];
#pragma unroll
            for (int c = 0; c < BFS_BU_CAND; c++)
            {
                const int idx = i0 + c * 32 + lane;
                off[c] = idx < total ? (int)cand[idx] : -1;
                s[c] = 0;
                deg[c] = 0;
                if (off[c] >= 0)
                {
                    const int64_t v = vbase + off[c];
                    s[c] = in_ptr[v];
                    deg[c] = (int)(in_ptr[v + 1] - s[c]);
                }
            }
            int32_t x[BFS_BU_CAND][BFS_BU_PROBE];
#pragma unroll
            for (int c = 0; c < BFS_BU_CAND; c++)
#pragma unroll
                for (int k = 0; k < BFS_BU_PROBE; k++) x[c][k] = k < deg[c] ? in_adj[s[c] + k] : -1;
            bool fnd[BFS_BU_CAND];
#pragma unroll
            for (int c = 0; c < BFS_BU_CAND; c++)
            {
                fnd[c] = false;
#pragma unroll
                for (int k = 0; k < BFS_BU_PROBE; k++)
                    if (x[c][k] >= 0)
                    {
                        edges++;
                        fnd[c] |= bm_test(cur_bm, x[c][k]);
                    }
            }
#pragma unroll
            for (int c = 0; c < BFS_BU_CAND; c++)
            {
                if (i0 + c * 32 >= total) break; // (uniform)
                bool f = fnd[c];
                // further lane-private probes, BFS_BU_PROBE at a time, up to BFS_BU_PROBE_MAX in-neighbours
                const int dmax = min(deg[c], BFS_BU_PROBE_MAX);
                for (int q = BFS_BU_PROBE; q < dmax && !f; q += BFS_BU_PROBE)
                {
                    int32_t y[BFS_BU_PROBE];
#pragma unroll
                    for (int k = 0; k < BFS_BU_PROBE; k++) y[k] = q + k < dmax ? in_adj[s[c] + q + k] : -1;
#pragma unroll
                    for (int k = 0; k < BFS_BU_PROBE; k++)
                        if (y[k] >= 0)
                        {
                            edges++;
                            f |= bm_test(cur_bm, y[k]);
                        }
                }
                // rows longer than the probe: finished by the whole warp
                unsigned pending = __ballot_sync(FULL, !f && deg[c] > BFS_BU_PROBE_MAX);
                while (pending)
                {
                    const int src_lane = __ffs(pending) - 1;
                    pending &= pending - 1;
                    const int64_t ps = __shfl_sync(FULL, s[c], src_lane) + BFS_BU_PROBE_MAX;
                    const int64_t pend = ps - BFS_BU_PROBE_MAX + __shfl_sync(FULL, deg[c], src_lane);
                    bool hit = false;
                    // BFS_BU_LONG_UNROLL x 32 neighbours per round trip: a vertex without a parent in the frontier (most of them in
                    // the first bottom-up level) scans its whole in-row, and 32 edges per dependent load pair is far too few
                    for (int64_t p0 = ps; p0 < pend; p0 += 32 * BFS_BU_LONG_UNROLL)
                    {
                        int32_t y[BFS_BU_LONG_UNROLL];
#pragma unroll
                        for (int k = 0; k < BFS_BU_LONG_UNROLL; k++)
                        {
                            const int64_t p = p0 + k * 32 + lane;
                            y[k] = p < pend ? in_adj[p] : -1;
                        }
                        bool h = false;
#pragma unroll
                        for (int k = 0; k < BFS_BU_LONG_UNROLL; k++)
                            if (y[k] >= 0)
                            {
                                edges++;
                                h |= bm_test(cur_bm, y[k]);
                            }
                        if (__any_sync(FULL, h))
                        {
                            hit = true;
                            break;
                        }
                    }
                    if (lane == src_lane && hit) f = true;
                }
                if (f)
                {
                    levels[vbase + off[c]] = next_level;
                    atomicOr(&fnd_words[off[c] >> 5], 1u << (off[c] & 31));
                }
            }
        }
        __syncwarp();
        if (wl < nwords)
        {
            const uint32_t fmask = fnd_words[lane];
            next_bm[wl] = fmask;
            if (fmask) visited[wl] = vis_l | fmask;
            found_total += __popc(fmask);
        }
        __syncwarp();
    }
    long long e64 = warp_sum_i64(edges), r64 = warp_sum_i64(rows);
    found_total = (int)warp_sum_i64(found_total);
    if (lane == 0)
    {
        if (e64) atomicAdd(&counters[C_EDGES], (unsigned long long)e64);
        if (r64) atomicAdd(&counters[C_ROWS], (unsigned long long)r64);
        if (found_total) atomicAdd(&counters[C_FOUND], (unsigned long long)found_total);
    }
}

// bit v = vertex v has no in-edges (built once per graph)
__global__ void bfs_no_in_edges_kernel(const int64_t *__restrict__ in_ptr, int32_t V, uint32_t *__restrict__ out)
{
    const int32_t padded = (V + 31) & ~31;
    for (int32_t v = blockIdx.x * blockDim.x + threadIdx.x; v < padded; v += gridDim.x * blockDim.x)
    {
        const bool none = v >= V || in_ptr[v + 1] == in_ptr[v];
        const uint32_t word = __ballot_sync(0xffffffffu, none);
        if ((threadIdx.x & 31) == 0) out[v >> 5] = word;
    }
}

int bfs_prepare_no_in_edges(vglb_ctx *ctx, vglb_graph *g)
{
    if (g->d_scratch_i32 || !g->d_in_ptr) return VGLB_OK;
    CUDA_TRY(vglb_dev_alloc(&g->d_scratch_i32, (((size_t)g->V + 31) / 32 + 32) * 4));
    bfs_no_in_edges_kernel<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(g->d_in_ptr, g->V, (uint32_t *)g->d_scratch_i32);
    KERNEL_TRY();
    ctx->launches++;
    return VGLB_OK;
}

// sparse queues -> dense bitmap (bitmap must be zeroed before)
__global__ void bfs_queue_to_bitmap_kernel(TierQueues q, int32_t n0, int32_t n1, int32_t n2, uint32_t *__restrict__ bm)
{
    const int n = n0 + n1 + n2;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    {
        const int32_t u = i < n0 ? q.q[0][i] : (i < n0 + n1 ? q.q[1][i - n0] : q.q[2][i - n0 - n1]);
        atomicOr(&bm[u >> 5], 1u << (u & 31));
    }
}

// dense bitmap -> degree-binned sparse queues: popc per word, warp scan, one atomic per warp and tier
__global__ void bfs_bitmap_to_queue_kernel(const uint32_t *__restrict__ bm, int32_t V, int32_t b0, int32_t b1, TierQueues q,
                                           unsigned long long *counters)
{
    const int lane = threadIdx.x & 31;
    const int64_t nwords = ((int64_t)V + 31) >> 5;
    const int64_t nwords_padded = (nwords + 31) & ~(int64_t)31;
    for (int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; w < nwords_padded; w += (int64_t)gridDim.x * blockDim.x)
    {
        const uint32_t word = w < nwords ? bm[w] : 0u;
        if (!__any_sync(0xffffffffu, word != 0)) continue;
        const int32_t base = (int32_t)(w << 5);
        const uint32_t m0 = below_border_mask(base, b0);
        const uint32_t m1 = below_border_mask(base, b1);
        const uint32_t part[3] = {word & m0, word & m1 & ~m0, word & ~m1};
#pragma unroll
        for (int t = 0; t < 3; t++)
        {
            const int cnt = __popc(part[t]);
            int incl = cnt;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1)
            {
                const int n = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += n;
            }
            const int total = __shfl_sync(0xffffffffu, incl, 31);
            if (total == 0) continue;
            unsigned long long wbase = 0;
            if (lane == 0) wbase = atomicAdd(&counters[C_NEXT_BIG + t], (unsigned long long)total);
            wbase = __shfl_sync(0xffffffffu, wbase, 0);
            int64_t pos = (int64_t)wbase + incl - cnt;
            uint32_t bits = part[t];
            while (bits)
            {
                const int bpos = __ffs(bits) - 1;
                bits &= bits - 1;
                q.q[t][pos++] = base + bpos;
            }
        }
    }
}

__global__ void bfs_init_kernel(int32_t *levels, uint32_t *visited, int32_t source, int32_t *queue_slot)
{
    levels[source] = VGLB_FIRST_LEVEL_VERTEX;
    visited[source >> 5] = 1u << (source & 31);
    *queue_slot = source;
}


// ---- 1D-partitioned BFS (one rank's part; every rank runs the same host loop on the same allreduced counters) -------
// Reference: the NEC backend replicates levels and MPI_Allreduce(MAX)es the whole int array after every advance
// (vgl_compute_api/common/mpi_exchange.hpp:155-271). Here only bitmaps travel:
//   top-down : each rank expands the frontier vertices it owns and marks every unvisited destination in a full-length
//              candidate bitmap; an all-to-all hands slice q of every rank's candidates to rank q, which ORs them, masks
//              its visited slice, writes the levels it owns and queues its new frontier vertices (bfs_combine_kernel);
//   bottom-up: each rank scans the in-rows of the unvisited vertices it owns against the replicated frontier bitmap
//              (same kernel as on one GPU, pointed at the owned slice);
//   both     : the owned slices of the new frontier are allgathered (V/8 bytes in total) and ORed into the replicated
//              visited bitmap; {found, m_f, edges, rows} are allreduced and drive termination and the alpha/beta switch.

__global__ void bfs_part_init_kernel(uint32_t *visited, uint32_t *cur_bm, int32_t source_col, int32_t *levels_local,
                                     int32_t local_row /* -1 unless owned */, int32_t *queue_slot)
{
    visited[source_col >> 5] = 1u << (source_col & 31);
    cur_bm[source_col >> 5] = 1u << (source_col & 31);
    if (local_row >= 0)
    {
        levels_local[local_row] = VGLB_FIRST_LEVEL_VERTEX;
        *queue_slot = local_row;
    }
}

// one thread per word of the owned slice: OR of the P received candidate slices, minus the visited ones
__global__ void __launch_bounds__(256)
bfs_combine_kernel(const uint32_t *__restrict__ stage, int32_t P, int32_t wslice, const uint32_t *__restrict__ visited_slice,
                   uint32_t *__restrict__ next_slice, const int64_t *__restrict__ ptr, int32_t *__restrict__ levels_local,
                   int32_t next_level, int32_t b0, int32_t b1, TierQueues nq, unsigned long long *counters)
{
    const int lane = threadIdx.x & 31;
    const int32_t wpad = (wslice + 31) & ~31;
    long long mf = 0;
    int found = 0;
    for (int32_t w = blockIdx.x * blockDim.x + threadIdx.x; w < wpad; w += gridDim.x * blockDim.x)
    {
        uint32_t bits = 0;
        if (w < wslice)
        {
            for (int p = 0; p < P; p++) bits |= stage[(int64_t)p * wslice + w];
            bits &= ~visited_slice[w];
            next_slice[w] = bits;
            found += __popc(bits);
        }
        while (__any_sync(0xffffffffu, bits != 0))
        {
            const bool has = bits != 0;
            int32_t row = 0;
            if (has)
            {
                const int b = __ffs(bits) - 1;
                bits &= bits - 1;
                row = (w << 5) + b;
                levels_local[row] = next_level;
                mf += ptr[row + 1] - ptr[row];
            }
            enqueue_binned(has, row, b0, b1, nq, counters);
        }
    }
    mf = warp_sum_i64(mf);
    found = (int)warp_sum_i64(found);
    if (lane == 0)
    {
        if (mf) atomicAdd(&counters[C_MF], (unsigned long long)mf);
        if (found) atomicAdd(&counters[C_FOUND], (unsigned long long)found);
    }
}

__global__ void bfs_or_kernel(uint32_t *__restrict__ visited, const uint32_t *__restrict__ next_bm, int64_t words)
{
    for (int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; w < words; w += (int64_t)gridDim.x * blockDim.x)
    {
        const uint32_t n = next_bm[w];
        if (n) visited[w] |= n;
    }
}

__global__ void bfs_copy_counters_kernel(unsigned long long *c)
{
    if (threadIdx.x < C_COUNT) c[C_COUNT + threadIdx.x] = c[threadIdx.x];
}

static int bfs_partitioned_bitmaps(vglb_ctx *ctx, vglb_graph *g, int32_t source, int32_t *d_levels, const vglb_bfs_opts *opts,
                                   vglb_stats *stats)
{
    VGLB_REQUIRE(source >= 0 && source < g->cols, "vglb_bfs: source column out of range");
    const bool dopt = opts && opts->direction_optimising;
    if (dopt && !g->d_in_ptr)
    {
        vglb_set_error("vglb_bfs: direction-optimising BFS needs a graph built with VGLB_GRAPH_WITH_INCOMING");
        return VGLB_EINVAL;
    }
    const long long alpha = (opts && opts->alpha > 0) ? opts->alpha : 15;
    const long long beta = (opts && opts->beta > 0) ? opts->beta : 18;
    CUDA_TRY(cudaSetDevice(ctx->device));
    int rc0;
    vglb_comm *comm = g->comm;
    const int32_t P = g->part_world, rank = g->part_rank, vp = g->vp, rows = g->V;
    const int32_t wslice = vp / 32;
    const int64_t words = g->cols / 32, my = (int64_t)rank * wslice;
    for (int i = 0; i < 3; i++)
        if (!g->d_part_bm[i]) CUDA_TRY(vglb_dev_alloc(&g->d_part_bm[i], (size_t)(words + 32) * 4));
    if (!g->d_part_stage) CUDA_TRY(vglb_dev_alloc(&g->d_part_stage, (size_t)(words + 32) * 4));
    if (!g->d_queue[0]) CUDA_TRY(vglb_dev_alloc(&g->d_queue[0], ((size_t)vp + 3) * 4));
    rc0 = bfs_prepare_no_in_edges(ctx, g);
    if (rc0 != VGLB_OK) return rc0;
    const int64_t launches0 = ctx->launches;
    const int32_t b0 = g->tier_border[0], b1 = g->tier_border[1];
    unsigned long long *d_cnt = (unsigned long long *)ctx->d_counters;
    unsigned long long *h_cnt = (unsigned long long *)ctx->h_counters;
    cudaStream_t st = ctx->stream;
    TierQueues cq;
    cq.q[0] = g->d_queue[0];
    cq.q[1] = g->d_queue[0] + b0;
    cq.q[2] = g->d_queue[0] + b1;
    uint32_t *visited = g->d_part_bm[0], *cur_bm = g->d_part_bm[1], *next_bm = g->d_part_bm[2];

    CUDA_TRY(cudaEventRecord(ctx->ev_start, st));
    if (rows > 0) CUDA_TRY(cudaMemsetAsync(d_levels, 0xFF, (size_t)rows * 4, st));
    CUDA_TRY(cudaMemsetAsync(visited, 0, (size_t)words * 4, st));
    CUDA_TRY(cudaMemsetAsync(cur_bm, 0, (size_t)words * 4, st));
    CUDA_TRY(cudaMemsetAsync(d_cnt, 0, 2 * C_COUNT * 8, st));
    const bool own_source = source / vp == rank;
    const int32_t src_row = own_source ? source - rank * vp : -1;
    VGLB_REQUIRE(!own_source || src_row < rows, "vglb_bfs: source is a padding column");
    const int src_tier = src_row < 0 ? 0 : (src_row < b0 ? 0 : (src_row < b1 ? 1 : 2));
    bfs_part_init_kernel<<<1, 1, 0, st>>>(visited, cur_bm, source, d_levels, src_row, cq.q[src_tier]);
    KERNEL_TRY();
    ctx->launches++;

    int32_t n[3] = {0, 0, 0};
    if (own_source) n[src_tier] = 1;
    long long n_cur = 1, visited_total = 1;
    bool bottom_up = false;
    int32_t level = VGLB_FIRST_LEVEL_VERTEX;
    int64_t tot_edges = 0, tot_rows = 0, tot_frontier_bytes = 0, levels_run = 0;
    int32_t bu_levels = 0;
    const long long Vg = g->V_orig;
    const long long factor = (g->E_global / (Vg > 0 ? Vg : 1)) / 2 > 0 ? (g->E_global / Vg) / 2 : 1;
    const int max_blocks = ctx->sm_count * 16;
    const int big_chunks = (int)ceil_div64(g->max_degree > 0 ? g->max_degree : 1, BFS_BIG_CHUNK);
    int rc;
    const bool trace = getenv("VGLB_BFS_TRACE") != NULL;
    double trace_t = 0.0;
    if (trace)
    {
        cudaStreamSynchronize(st);
        trace_t = trace_now();
    }

    while (n_cur > 0)
    {
        if (!bottom_up)
        {
            CUDA_TRY(cudaMemsetAsync(next_bm, 0, (size_t)words * 4, st)); // candidates
            const int blocks_mid = (int)min((int64_t)max_blocks, ceil_div64(n[1], BFS_THREADS / 32));
            const int blocks_small = (int)min((int64_t)max_blocks, ceil_div64(n[2], BFS_THREADS / BFS_SMALL_LANES));
            const int hub_ctas = (int)min((int64_t)n[0] * big_chunks, (int64_t)ctx->sm_count * 4); // CTAs that share the queued hub rows
            const int64_t grid = (int64_t)hub_ctas + blocks_mid + blocks_small;
            if (grid > 0)
            {
                bfs_td_kernel<1><<<(unsigned)grid, BFS_THREADS, 0, st>>>(g->d_out_ptr, g->d_out_adj, cq, n[0], hub_ctas, n[1], n[2], blocks_mid,
                                                                       blocks_small, visited, (int32_t *)next_bm, level + 1, b0, b1,
                                                                       cq, d_cnt, PartArgs());
                KERNEL_TRY();
                ctx->launches++;
            }
            rc = vglb_comm_alltoall_async(comm, next_bm, g->d_part_stage, (size_t)wslice * 4);
            if (rc != VGLB_OK) return rc;
            bfs_combine_kernel<<<(unsigned)min((int64_t)max_blocks, ceil_div64(wslice, 256)), 256, 0, st>>>(
                g->d_part_stage, P, wslice, visited + my, next_bm + my, g->d_out_ptr, d_levels, level + 1, b0, b1, cq, d_cnt);
            KERNEL_TRY();
            ctx->launches++;
            tot_frontier_bytes += (int64_t)wslice * 4 * (2 * P + 2);
        }
        else
        {
            CUDA_TRY(cudaMemsetAsync(next_bm + my, 0, (size_t)wslice * 4, st));
            bfs_bu_kernel<<<ctx->sm_count * 8, BFS_THREADS, 0, st>>>(g->d_in_ptr, g->d_in_adj, rows, (const uint32_t *)g->d_scratch_i32, visited + my, cur_bm,
                                                                    next_bm + my, d_levels, level + 1, d_cnt);
            KERNEL_TRY();
            ctx->launches++;
            bu_levels++;
            tot_frontier_bytes += (int64_t)wslice * 4 * 3;
        }
        rc = vglb_comm_allgather_async(comm, next_bm, (size_t)wslice * 4);
        if (rc != VGLB_OK) return rc;
        bfs_or_kernel<<<(unsigned)min((int64_t)max_blocks, ceil_div64(words, 256)), 256, 0, st>>>(visited, next_bm, words);
        KERNEL_TRY();
        bfs_copy_counters_kernel<<<1, 32, 0, st>>>(d_cnt);
        KERNEL_TRY();
        ctx->launches += 2;
        rc = vglb_comm_allreduce_async(comm, d_cnt + C_COUNT, C_COUNT, VGLB_DT_I64, VGLB_OP_SUM);
        if (rc != VGLB_OK) return rc;
        CUDA_TRY(cudaMemcpyAsync(h_cnt, d_cnt, 2 * C_COUNT * 8, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        CUDA_TRY(cudaMemsetAsync(d_cnt, 0, 2 * C_COUNT * 8, st));
        levels_run++;
        const unsigned long long *gl = h_cnt + C_COUNT; // global sums
        const long long n_next = (long long)gl[C_FOUND];
        if (trace)
        {
            const double now = trace_now();
            fprintf(stderr, "bfs level %d (%s, rank %d of %d): frontier %lld, this rank inspected %lld edges, found %lld, %.1f us since the previous line\n",
                    level, bottom_up ? "bottom-up" : "top-down", rank, P, n_cur, (long long)h_cnt[C_EDGES], n_next, (now - trace_t) * 1e6);
            trace_t = now;
        }
        tot_edges += (int64_t)h_cnt[C_EDGES];
        tot_rows += bottom_up ? (int64_t)h_cnt[C_ROWS] : (int64_t)n[0] + n[1] + n[2];
        tot_frontier_bytes += words * 4 * 3; // allgathered frontier written, ORed into visited
        visited_total += n_next;
        if (n_next == 0) break;

        bool next_bu = bottom_up;
        if (dopt)
        {
            const long long unvisited = Vg - visited_total;
            if (!bottom_up && n_cur < n_next)
            {
                if ((long long)gl[C_MF] >= (unvisited * factor + Vg) / alpha) next_bu = true;
            }
            else if (bottom_up && n_cur >= n_next)
            {
                if (n_next < (unvisited * factor + Vg) / (factor * beta)) next_bu = false;
            }
        }
        if (!next_bu)
        {
            if (!bottom_up)
            {
                n[0] = (int32_t)h_cnt[C_NEXT_BIG]; n[1] = (int32_t)h_cnt[C_NEXT_MID]; n[2] = (int32_t)h_cnt[C_NEXT_SMALL];
            }
            else
            {
                bfs_bitmap_to_queue_kernel<<<(unsigned)min((int64_t)max_blocks, ceil_div64(wslice, 256)), 256, 0, st>>>(
                    next_bm + my, rows, b0, b1, cq, d_cnt);
                KERNEL_TRY();
                ctx->launches++;
                CUDA_TRY(cudaMemcpyAsync(h_cnt, d_cnt, 3 * 8, cudaMemcpyDeviceToHost, st));
                CUDA_TRY(cudaStreamSynchronize(st));
                n[0] = (int32_t)h_cnt[0]; n[1] = (int32_t)h_cnt[1]; n[2] = (int32_t)h_cnt[2];
                CUDA_TRY(cudaMemsetAsync(d_cnt, 0, 2 * C_COUNT * 8, st));
            }
        }
        uint32_t *t = cur_bm; cur_bm = next_bm; next_bm = t;
        bottom_up = next_bu;
        n_cur = n_next;
        level++;
    }
    CUDA_TRY(cudaEventRecord(ctx->ev_stop, st));
    CUDA_TRY(cudaEventSynchronize(ctx->ev_stop));
    if (stats)
    {
        float ms = 0.f;
        CUDA_TRY(cudaEventElapsedTime(&ms, ctx->ev_start, ctx->ev_stop));
        memset(stats, 0, sizeof(*stats));
        stats->seconds = ms * 1e-3;
        stats->iterations = levels_run;
        stats->edges_inspected = tot_edges;      // this rank's
        stats->vertices_processed = tot_rows;
        stats->frontier_bytes = tot_frontier_bytes;
        stats->algorithmic_bytes = 8 * tot_edges + 12 * tot_rows + tot_frontier_bytes;
        stats->kernel_launches = ctx->launches - launches0;
        stats->bottom_up_levels = bu_levels;
    }
    return VGLB_OK;
}

// ---- 1D-partitioned BFS, discovery lists (the default; bfs_partitioned_bitmaps above is the fallback without CUDA IPC) ----
// A top-down level with a small frontier should not cost full-length bitmap traffic (memset + all-to-all + allgather + OR of
// V/8-byte bitmaps cost ~150 us per level at 2 GPUs and grow with V). Here every rank keeps its own replica of the visited
// bitmap: the first thread to set a bit either owns the vertex — level written, queued by local row — or appends the
// column to the list of its owner (at most once per rank and vertex in a whole run, so a list never outgrows the owner's
// slice). After a one-word allreduce as barrier every owner reads the lists addressed to it out of the peers' memory
// (bfs_apply_lists_kernel) and claims the vertices in its own slice, which is authoritative. Replicas may lag behind —
// a stale bit only costs a duplicate list entry. Bottom-up levels work as before on the owned slice and allgather the new
// frontier slices; at a top-down -> bottom-up switch the frontier bitmap is assembled once from the owners' queues.
static int bfs_partitioned(vglb_ctx *ctx, vglb_graph *g, int32_t source, int32_t *d_levels, const vglb_bfs_opts *opts,
                           vglb_stats *stats)
{
    VGLB_REQUIRE(source >= 0 && source < g->cols, "vglb_bfs: source column out of range");
    const bool dopt = opts && opts->direction_optimising;
    if (dopt && !g->d_in_ptr)
    {
        vglb_set_error("vglb_bfs: direction-optimising BFS needs a graph built with VGLB_GRAPH_WITH_INCOMING");
        return VGLB_EINVAL;
    }
    const long long alpha = (opts && opts->alpha > 0) ? opts->alpha : 15;
    const long long beta = (opts && opts->beta > 0) ? opts->beta : 18;
    CUDA_TRY(cudaSetDevice(ctx->device));
    vglb_comm *comm = g->comm;
    const int32_t P = g->part_world, rank = g->part_rank, vp = g->vp, rows = g->V;
    const int32_t wslice = vp / 32;
    const int64_t words = g->cols / 32, my = (int64_t)rank * wslice;
    for (int i = 0; i < 3; i++)
        if (!g->d_part_bm[i]) CUDA_TRY(vglb_dev_alloc(&g->d_part_bm[i], (size_t)(words + 32) * 4));
    for (int i = 0; i < 2; i++)
        if (!g->d_queue[i]) CUDA_TRY(vglb_dev_alloc(&g->d_queue[i], ((size_t)vp + 3) * 4));
    int rc = bfs_prepare_no_in_edges(ctx, g);
    if (rc != VGLB_OK) return rc;
    const int64_t launches0 = ctx->launches;
    const int32_t b0 = g->tier_border[0], b1 = g->tier_border[1];
    unsigned long long *d_cnt = (unsigned long long *)ctx->d_counters;
    unsigned long long *h_cnt = (unsigned long long *)ctx->h_counters;
    cudaStream_t st = ctx->stream;
    auto regions = [&](int32_t *base) {
        TierQueues q;
        q.q[0] = base;
        q.q[1] = base + b0;
        q.q[2] = base + b1;
        return q;
    };
    TierQueues cq = regions(g->d_queue[0]), nq = regions(g->d_queue[1]);
    uint32_t *visited = g->d_part_bm[0], *cur_bm = g->d_part_bm[1], *next_bm = g->d_part_bm[2];
    PartArgs A;
    A.col0 = g->col_of_row0;
    A.vp = vp;
    A.P = P;
    A.rank = rank;
    A.lists = (unsigned long long *)g->d_part_lists;
    const unsigned long long **d_peer_table = (const unsigned long long **)(ctx->d_counters + 24); // 8 device pointers
    CUDA_TRY(cudaMemcpyAsync(d_peer_table, g->d_vec_peer, sizeof(g->d_vec_peer), cudaMemcpyHostToDevice, st));

    CUDA_TRY(cudaEventRecord(ctx->ev_start, st));
    if (rows > 0) CUDA_TRY(cudaMemsetAsync(d_levels, 0xFF, (size_t)rows * 4, st));
    CUDA_TRY(cudaMemsetAsync(visited, 0, (size_t)words * 4, st));
    CUDA_TRY(cudaMemsetAsync(cur_bm, 0, (size_t)words * 4, st));
    CUDA_TRY(cudaMemsetAsync(d_cnt, 0, 2 * C_COUNT * 8, st));
    const bool own_source = source / vp == rank;
    const int32_t src_row = own_source ? source - rank * vp : -1;
    VGLB_REQUIRE(!own_source || src_row < rows, "vglb_bfs: source is a padding column");
    const int src_tier = src_row < 0 ? 0 : (src_row < b0 ? 0 : (src_row < b1 ? 1 : 2));
    bfs_part_init_kernel<<<1, 1, 0, st>>>(visited, cur_bm, source, d_levels, src_row, cq.q[src_tier]);
    KERNEL_TRY();
    ctx->launches++;

    int32_t n[3] = {0, 0, 0};
    if (own_source) n[src_tier] = 1;
    long long n_cur = 1, visited_total = 1;
    bool bottom_up = false;
    int32_t level = VGLB_FIRST_LEVEL_VERTEX;
    int64_t tot_edges = 0, tot_rows = 0, tot_frontier_bytes = 0, levels_run = 0;
    int32_t bu_levels = 0;
    const long long Vg = g->V_orig;
    const long long factor = (g->E_global / (Vg > 0 ? Vg : 1)) / 2 > 0 ? (g->E_global / Vg) / 2 : 1;
    const int max_blocks = ctx->sm_count * 16;
    const int big_chunks = (int)ceil_div64(g->max_degree > 0 ? g->max_degree : 1, BFS_BIG_CHUNK);
    const bool trace = getenv("VGLB_BFS_TRACE") != NULL;
    double trace_t = 0.0;
    if (trace)
    {
        cudaStreamSynchronize(st);
        trace_t = trace_now();
    }

    while (n_cur > 0)
    {
        if (!bottom_up)
        {
            CUDA_TRY(cudaMemsetAsync(A.lists, 0, (size_t)P * 8, st)); // list lengths (the peers finished reading them: see below)
            const int blocks_mid = (int)min((int64_t)max_blocks, ceil_div64(n[1], BFS_THREADS / 32));
            const int blocks_small = (int)min((int64_t)max_blocks, ceil_div64(n[2], BFS_THREADS / BFS_SMALL_LANES));
            const int hub_ctas = (int)min((int64_t)n[0] * big_chunks, (int64_t)ctx->sm_count * 4); // CTAs that share the queued hub rows
            const int64_t grid = (int64_t)hub_ctas + blocks_mid + blocks_small;
            if (grid > 0)
            {
                bfs_td_kernel<2><<<(unsigned)grid, BFS_THREADS, 0, st>>>(g->d_out_ptr, g->d_out_adj, cq, n[0], hub_ctas, n[1], n[2], blocks_mid,
                                                                       blocks_small, visited, d_levels, level + 1, b0, b1, nq, d_cnt, A);
                KERNEL_TRY();
                ctx->launches++;
            }
            // barrier: every rank's lists are complete before anybody reads them; they are not reset before every rank has
            // passed this level's counter allreduce, i.e. finished reading
            rc = vglb_comm_allreduce_async(comm, d_cnt + 2 * C_COUNT + 2, 1, VGLB_DT_I64, VGLB_OP_SUM);
            if (rc != VGLB_OK) return rc;
            bfs_apply_lists_kernel<<<ctx->sm_count * 4, 256, 0, st>>>(d_peer_table, A, g->d_out_ptr, visited, d_levels, level + 1, b0, b1, nq, d_cnt);
            KERNEL_TRY();
            ctx->launches++;
        }
        else
        {
            CUDA_TRY(cudaMemsetAsync(next_bm + my, 0, (size_t)wslice * 4, st));
            bfs_bu_kernel<<<ctx->sm_count * 8, BFS_THREADS, 0, st>>>(g->d_in_ptr, g->d_in_adj, rows, (const uint32_t *)g->d_scratch_i32, visited + my, cur_bm,
                                                                    next_bm + my, d_levels, level + 1, d_cnt);
            KERNEL_TRY();
            rc = vglb_comm_allgather_async(comm, next_bm, (size_t)wslice * 4);
            if (rc != VGLB_OK) return rc;
            bfs_or_kernel<<<(unsigned)min((int64_t)max_blocks, ceil_div64(words, 256)), 256, 0, st>>>(visited, next_bm, words);
            KERNEL_TRY();
            ctx->launches += 2;
            bu_levels++;
            tot_frontier_bytes += (int64_t)wslice * 4 * 3 + words * 4 * 3;
        }
        bfs_copy_counters_kernel<<<1, 32, 0, st>>>(d_cnt);
        KERNEL_TRY();
        ctx->launches++;
        rc = vglb_comm_allreduce_async(comm, d_cnt + C_COUNT, C_COUNT, VGLB_DT_I64, VGLB_OP_SUM);
        if (rc != VGLB_OK) return rc;
        CUDA_TRY(cudaMemcpyAsync(h_cnt, d_cnt, 2 * C_COUNT * 8, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        CUDA_TRY(cudaMemsetAsync(d_cnt, 0, 2 * C_COUNT * 8, st));
        levels_run++;
        const unsigned long long *gl = h_cnt + C_COUNT; // whole-job sums
        const int32_t nn[3] = {(int32_t)h_cnt[C_NEXT_BIG], (int32_t)h_cnt[C_NEXT_MID], (int32_t)h_cnt[C_NEXT_SMALL]};
        const long long n_next = bottom_up ? (long long)gl[C_FOUND] : (long long)(gl[C_NEXT_BIG] + gl[C_NEXT_MID] + gl[C_NEXT_SMALL]);
        if (trace)
        {
            const double now = trace_now();
            fprintf(stderr, "bfs level %d (%s, rank %d of %d): frontier %lld, this rank inspected %lld edges, found %lld, %.1f us since the previous line\n",
                    level, bottom_up ? "bottom-up" : "top-down", rank, P, n_cur, (long long)h_cnt[C_EDGES], n_next, (now - trace_t) * 1e6);
            trace_t = now;
        }
        tot_edges += (int64_t)h_cnt[C_EDGES];
        tot_rows += bottom_up ? (int64_t)h_cnt[C_ROWS] : (int64_t)n[0] + n[1] + n[2];
        if (!bottom_up) tot_frontier_bytes += 8 * ((int64_t)nn[0] + nn[1] + nn[2]); // queue written now, read next level (+ list entries)
        visited_total += n_next;
        if (n_next == 0) break;

        bool next_bu = bottom_up;
        if (dopt)
        {
            const long long unvisited = Vg - visited_total;
            if (!bottom_up && n_cur < n_next)
            {
                if ((long long)gl[C_MF] >= (unvisited * factor + Vg) / alpha) next_bu = true;
            }
            else if (bottom_up && n_cur >= n_next)
            {
                if (n_next < (unvisited * factor + Vg) / (factor * beta)) next_bu = false;
            }
        }
        if (!bottom_up && !next_bu)
        {
            TierQueues t = cq; cq = nq; nq = t;
            n[0] = nn[0]; n[1] = nn[1]; n[2] = nn[2];
        }
        else if (!bottom_up && next_bu)
        {
            // the frontier as a replicated bitmap, assembled once from the owners' queues; it is also ORed into every
            // replica of the visited bitmap (the replicas only knew their own discoveries)
            CUDA_TRY(cudaMemsetAsync(cur_bm + my, 0, (size_t)wslice * 4, st));
            const long long nl = (long long)nn[0] + nn[1] + nn[2];
            if (nl > 0)
            {
                bfs_queue_to_bitmap_kernel<<<(unsigned)min((int64_t)max_blocks, ceil_div64(nl, 256)), 256, 0, st>>>(nq, nn[0], nn[1], nn[2], cur_bm + my);
                KERNEL_TRY();
            }
            rc = vglb_comm_allgather_async(comm, cur_bm, (size_t)wslice * 4);
            if (rc != VGLB_OK) return rc;
            bfs_or_kernel<<<(unsigned)min((int64_t)max_blocks, ceil_div64(words, 256)), 256, 0, st>>>(visited, cur_bm, words);
            KERNEL_TRY();
            ctx->launches += 2;
            tot_frontier_bytes += words * 4 * 4;
        }
        else if (bottom_up && next_bu)
        {
            uint32_t *t = cur_bm; cur_bm = next_bm; next_bm = t;
        }
        else
        {
            bfs_bitmap_to_queue_kernel<<<(unsigned)min((int64_t)max_blocks, ceil_div64(wslice, 256)), 256, 0, st>>>(next_bm + my, rows, b0, b1, cq, d_cnt);
            KERNEL_TRY();
            ctx->launches++;
            CUDA_TRY(cudaMemcpyAsync(h_cnt, d_cnt, 3 * 8, cudaMemcpyDeviceToHost, st));
            CUDA_TRY(cudaStreamSynchronize(st));
            n[0] = (int32_t)h_cnt[0]; n[1] = (int32_t)h_cnt[1]; n[2] = (int32_t)h_cnt[2];
            CUDA_TRY(cudaMemsetAsync(d_cnt, 0, 2 * C_COUNT * 8, st));
        }
        bottom_up = next_bu;
        n_cur = n_next;
        level++;
    }
    CUDA_TRY(cudaEventRecord(ctx->ev_stop, st));
    CUDA_TRY(cudaEventSynchronize(ctx->ev_stop));
    if (stats)
    {
        float ms = 0.f;
        CUDA_TRY(cudaEventElapsedTime(&ms, ctx->ev_start, ctx->ev_stop));
        memset(stats, 0, sizeof(*stats));
        stats->seconds = ms * 1e-3;
        stats->iterations = levels_run;
        stats->edges_inspected = tot_edges;      // this rank's
        stats->vertices_processed = tot_rows;
        stats->frontier_bytes = tot_frontier_bytes;
        stats->algorithmic_bytes = 8 * tot_edges + 12 * tot_rows + tot_frontier_bytes;
        stats->kernel_launches = ctx->launches - launches0;
        stats->bottom_up_levels = bu_levels;
    }
    return VGLB_OK;
}

static int bfs_prepare(vglb_ctx *ctx, vglb_graph *g)
{
    if (g->bfs_ready) return VGLB_OK;
    // the scratch is shared with SSSP (sssp.cu allocates the same fields, same sizes, on first use): never overwrite
    // a pointer another algorithm has already filled in
    const size_t words = ((size_t)g->V + 31) / 32 + 32;
    if (!g->d_visited) CUDA_TRY(vglb_dev_alloc(&g->d_visited, words * 4));
    if (!g->d_front_bm[0]) CUDA_TRY(vglb_dev_alloc(&g->d_front_bm[0], words * 4));
    if (!g->d_front_bm[1]) CUDA_TRY(vglb_dev_alloc(&g->d_front_bm[1], words * 4));
    if (!g->d_queue[0]) CUDA_TRY(vglb_dev_alloc(&g->d_queue[0], ((size_t)g->V + 3) * 4));
    if (!g->d_queue[1]) CUDA_TRY(vglb_dev_alloc(&g->d_queue[1], ((size_t)g->V + 3) * 4));
    g->bfs_ready = 1;
    return bfs_prepare_no_in_edges(ctx, g);
}

extern "C" int vglb_bfs(vglb_ctx *ctx, vglb_graph *g, int32_t source, int32_t *d_levels, const vglb_bfs_opts *opts,
                        vglb_stats *stats)
{
    VGLB_REQUIRE(ctx != NULL && g != NULL && d_levels != NULL, "vglb_bfs: NULL argument");
    if (g->comm)
    {
        CUDA_TRY(cudaSetDevice(ctx->device));
        int rc = vglb_part_map_lists(ctx, g); // per-owner discovery lists, mapped into the peers once per graph
        if (rc != VGLB_OK) return rc;
        return g->vec_peers_mapped > 0 ? bfs_partitioned(ctx, g, source, d_levels, opts, stats)
                                       : bfs_partitioned_bitmaps(ctx, g, source, d_levels, opts, stats);
    }
    VGLB_REQUIRE(source >= 0 && source < g->V, "vglb_bfs: source out of range");
    const bool dopt = opts && opts->direction_optimising;
    if (dopt && !g->d_in_ptr)
    {
        // The bottom-up levels need the incoming CSR. A graph uploaded without it (vglb_graph_from_csr with NULL incoming arrays)
        // gets it here, once, from the outgoing one: a device sort of the edges is cheaper than a second 4.8 GB PCIe upload
        // (Kronecker s26: see DESIGN.md §6).
        int rc_in = vglb_graph_derive_incoming(ctx, g);
        if (rc_in != VGLB_OK) return rc_in;
    }
    long long alpha = (opts && opts->alpha > 0) ? opts->alpha : BFS_DEFAULT_ALPHA;
    long long beta = (opts && opts->beta > 0) ? opts->beta : BFS_DEFAULT_BETA;
    if (!(opts && opts->alpha > 0) && getenv("VGLB_BFS_ALPHA")) alpha = atoll(getenv("VGLB_BFS_ALPHA")); // developer knobs (A/B runs)
    if (!(opts && opts->beta > 0) && getenv("VGLB_BFS_BETA")) beta = atoll(getenv("VGLB_BFS_BETA"));
    if (alpha < 1) alpha = 1;
    if (beta < 1) beta = 1;
    CUDA_TRY(cudaSetDevice(ctx->device));
    int rc = bfs_prepare(ctx, g);
    if (rc != VGLB_OK) return rc;
    const int64_t launches0 = ctx->launches;
    const int32_t V = g->V;
    if (g->bfs_big_border_plus1 == 0) // first id with fewer than BFS_BIG_DEGREE edges (ids are degree-sorted), once per graph
    {
        int32_t border = 0;
        rc = vglb_graph_threshold_vertex(ctx, g, BFS_BIG_DEGREE, &border);
        if (rc != VGLB_OK) return rc;
        g->bfs_big_border_plus1 = border + 1;
    }
    const int32_t b0 = g->bfs_big_border_plus1 - 1, b1 = g->tier_border[1] > b0 ? g->tier_border[1] : b0;
    const size_t words = ((size_t)V + 31) / 32;
    unsigned long long *d_cnt = (unsigned long long *)ctx->d_counters;
    unsigned long long *h_cnt = (unsigned long long *)ctx->h_counters;
    cudaStream_t st = ctx->stream;

    // queue regions: capacity of a tier's queue = population of the tier
    auto regions = [&](int32_t *base) {
        TierQueues q;
        q.q[0] = base;
        q.q[1] = base + b0;
        q.q[2] = base + b1;
        return q;
    };
    TierQueues cq = regions(g->d_queue[0]), nq = regions(g->d_queue[1]);
    uint32_t *cur_bm = g->d_front_bm[0], *next_bm = g->d_front_bm[1];

    CUDA_TRY(cudaEventRecord(ctx->ev_start, st));
    CUDA_TRY(cudaMemsetAsync(d_levels, 0xFF, (size_t)V * 4, st)); // UNVISITED_VERTEX = -1
    CUDA_TRY(cudaMemsetAsync(g->d_visited, 0, words * 4, st));
    CUDA_TRY(cudaMemsetAsync(d_cnt, 0, C_COUNT * 8, st));
    const int src_tier = source < b0 ? 0 : (source < b1 ? 1 : 2);
    bfs_init_kernel<<<1, 1, 0, st>>>(d_levels, g->d_visited, source, cq.q[src_tier]);
    KERNEL_TRY();
    ctx->launches++;

    int32_t n[3] = {0, 0, 0};
    n[src_tier] = 1;
    long long n_cur = 1, visited_total = 1;
    bool bottom_up = false;
    int32_t level = VGLB_FIRST_LEVEL_VERTEX;
    int64_t tot_edges = 0, tot_rows = 0, tot_frontier_bytes = 0, levels_run = 0;
    int32_t bu_levels = 0;
    const long long factor = (g->E / (V > 0 ? V : 1)) / 2 > 0 ? (g->E / V) / 2 : 1; // change_state.hpp:104
    const int max_blocks = ctx->sm_count * 16;
    const int big_chunks = (int)ceil_div64(g->max_degree > 0 ? g->max_degree : 1, BFS_BIG_CHUNK);
    const bool trace = getenv("VGLB_BFS_TRACE") != NULL; // developer aid: one line per level on stderr
    double trace_t = 0.0;
    if (trace)
    {
        cudaStreamSynchronize(st);
        trace_t = trace_now();
    }

    const int visited_l2 = getenv("VGLB_BFS_VISITED_L2") != NULL; // developer knob
    long long m_f_cur = 0; // out-edges of the current frontier (accumulated by the level that produced it; unknown for the source)
    const long long bitmap_out_edges = getenv("VGLB_BFS_NO_BITMAP_OUT") ? (1LL << 62) : (1LL << 20); // developer knob
    while (n_cur > 0)
    {
        // a top-down level that is about to inspect more than a million edges emits its discoveries as a bitmap
        const bool bitmap_out = !bottom_up && m_f_cur > bitmap_out_edges;
        if (!bottom_up)
        {
            const int blocks_mid = (int)min((int64_t)max_blocks, ceil_div64(n[1], BFS_THREADS / 32));
            const int blocks_small = (int)min((int64_t)max_blocks, ceil_div64(n[2], BFS_THREADS / BFS_SMALL_LANES));
            const int hub_ctas = (int)min((int64_t)n[0] * big_chunks, (int64_t)ctx->sm_count * 4); // CTAs that share the queued hub rows
            const int64_t grid = (int64_t)hub_ctas + blocks_mid + blocks_small;
            if (bitmap_out)
            {
                PartArgs out;
                memset(&out, 0, sizeof(out));
                out.visited_via_l2 = visited_l2;
                out.lists = reinterpret_cast<unsigned long long *>(next_bm);
                CUDA_TRY(cudaMemsetAsync(next_bm, 0, words * 4, st));
                bfs_td_kernel<3><<<(unsigned)grid, BFS_THREADS, 0, st>>>(g->d_out_ptr, g->d_out_adj, cq, n[0], hub_ctas, n[1], n[2], blocks_mid,
                                                                       blocks_small, g->d_visited, d_levels, level + 1, b0, b1, nq, d_cnt, out);
                tot_frontier_bytes += (int64_t)words * 4;
            }
            else
            {
                PartArgs none;
                memset(&none, 0, sizeof(none));
                none.visited_via_l2 = visited_l2;
                bfs_td_kernel<0><<<(unsigned)grid, BFS_THREADS, 0, st>>>(g->d_out_ptr, g->d_out_adj, cq, n[0], hub_ctas, n[1], n[2], blocks_mid,
                                                                       blocks_small, g->d_visited, d_levels, level + 1, b0, b1, nq, d_cnt, none);
            }
            KERNEL_TRY();
            ctx->launches++;
            tot_rows += n_cur;
        }
        else
        {
            bfs_bu_kernel<<<ctx->sm_count * 8, BFS_THREADS, 0, st>>>(g->d_in_ptr, g->d_in_adj, V, (const uint32_t *)g->d_scratch_i32, g->d_visited, cur_bm,
                                                                    next_bm, d_levels, level + 1, d_cnt);
            KERNEL_TRY();
            ctx->launches++;
            bu_levels++;
            tot_frontier_bytes += (int64_t)words * 4 * 3; // visited read, frontier read, next written
        }
        rc = vglb_counters_fetch(ctx, d_cnt, C_COUNT);
        if (rc != VGLB_OK) return rc;
        levels_run++;
        int32_t nn[3] = {(int32_t)h_cnt[C_NEXT_BIG], (int32_t)h_cnt[C_NEXT_MID], (int32_t)h_cnt[C_NEXT_SMALL]};
        const bool out_is_bitmap = bottom_up || bitmap_out; // the next frontier sits in next_bm (else in the queues nq)
        const long long n_next = out_is_bitmap ? (long long)h_cnt[C_FOUND] : (long long)nn[0] + nn[1] + nn[2];
        const long long in_lvl = (long long)h_cnt[C_EDGES];
        const long long m_f_next = (long long)h_cnt[C_MF]; // accumulated by the top-down advance itself (0 after a bottom-up level)
        tot_edges += in_lvl;
        if (bottom_up) tot_rows += (long long)h_cnt[C_ROWS];
        else if (!bitmap_out) tot_frontier_bytes += 8 * n_next; // queue written now, read next level
        visited_total += n_next;
        if (trace)
        {
            const double now = trace_now();
            fprintf(stderr, "bfs level %d (%s%s): frontier %lld, inspected %lld edges, found %lld, %.1f us since the previous line\n", level,
                    bottom_up ? "bottom-up" : "top-down", bitmap_out ? ", bitmap out" : "", n_cur, in_lvl, n_next, (now - trace_t) * 1e6);
            trace_t = now;
        }
        if (n_next == 0) break;

        // direction switch — gpu_change_state (change_state.hpp:100-141) evaluated on the device counters; the
        // top-down test uses the edges the NEXT top-down level would inspect (m_f) instead of the level just done
        bool next_bu = bottom_up;
        if (dopt)
        {
            const long long unvisited = (long long)V - visited_total;
            if (!bottom_up && n_cur < n_next)
            {
                if (m_f_next >= (unvisited * factor + V) / alpha) next_bu = true;
            }
            else if (bottom_up && n_cur >= n_next)
            {
                if (n_next < (unvisited * factor + V) / (factor * beta)) next_bu = false;
            }
        }
        CUDA_TRY(cudaMemsetAsync(d_cnt, 0, C_COUNT * 8, st));
        if (!out_is_bitmap && !next_bu)
        {
            TierQueues t = cq; cq = nq; nq = t;
            n[0] = nn[0]; n[1] = nn[1]; n[2] = nn[2];
        }
        else if (!out_is_bitmap && next_bu)
        {
            CUDA_TRY(cudaMemsetAsync(cur_bm, 0, words * 4, st));
            bfs_queue_to_bitmap_kernel<<<(unsigned)min((int64_t)max_blocks, ceil_div64(n_next, 256)), 256, 0, st>>>(
                nq, nn[0], nn[1], nn[2], cur_bm);
            KERNEL_TRY();
            ctx->launches++;
            tot_frontier_bytes += (int64_t)words * 4 + 4 * n_next;
        }
        else if (out_is_bitmap && next_bu)
        {
            uint32_t *t = cur_bm; cur_bm = next_bm; next_bm = t;
        }
        else
        {
            bfs_bitmap_to_queue_kernel<<<(unsigned)min((int64_t)max_blocks, ceil_div64((int64_t)words, 256)), 256, 0, st>>>(
                next_bm, V, b0, b1, cq, d_cnt);
            KERNEL_TRY();
            ctx->launches++;
            rc = vglb_counters_fetch(ctx, d_cnt, 3);
            if (rc != VGLB_OK) return rc;
            n[0] = (int32_t)h_cnt[0]; n[1] = (int32_t)h_cnt[1]; n[2] = (int32_t)h_cnt[2];
            CUDA_TRY(cudaMemsetAsync(d_cnt, 0, C_COUNT * 8, st));
            tot_frontier_bytes += (int64_t)words * 4 + 4 * n_next;
        }
        // m_f of the frontier the next top-down level expands: known after a top-down level; after a bottom-up level the
        // frontier that goes back to top-down is small (that is why the heuristic switched)
        m_f_cur = bottom_up ? 0 : m_f_next;
        bottom_up = next_bu;
        n_cur = n_next;
        level++;
    }
    CUDA_TRY(cudaEventRecord(ctx->ev_stop, st));
    CUDA_TRY(cudaEventSynchronize(ctx->ev_stop));
    if (stats)
    {
        float ms = 0.f;
        CUDA_TRY(cudaEventElapsedTime(&ms, ctx->ev_start, ctx->ev_stop));
        memset(stats, 0, sizeof(*stats));
        stats->seconds = ms * 1e-3;
        stats->iterations = levels_run;
        stats->edges_inspected = tot_edges;
        stats->vertices_processed = tot_rows;
        stats->frontier_bytes = tot_frontier_bytes;
        // SURVEY §8(d): B = sum_levels [ 8 e_l + 12 f_l + g_l ]
        stats->algorithmic_bytes = 8 * tot_edges + 12 * tot_rows + tot_frontier_bytes;
        stats->kernel_launches = ctx->launches - launches0;
        stats->bottom_up_levels = bu_levels;
    }
    return VGLB_OK;
}
