// bfs_multi.cu — multi-source BFS (MS-BFS, Then et al., VLDB 2014; iBFS, Liu et al., SIGMOD 2016): up to 64 BFS runs over
// one graph in one level loop. Source i owns bit i of a per-vertex word of W = 32 or 64 bits (W from the batch size):
//   seen[v]  sources that have reached v;
//   front[v] sources whose frontier holds v at the current level (two arrays: current and next).
// One traversal reads each row once per level for all sources, and a level costs one host round trip whatever k is.
// Levels are those of k vglb_bfs calls, bit for bit: a (vertex, source) pair is claimed exactly once (atomicOr on seen in
// top-down, the vertex's owner thread in bottom-up) and is written level + 1.
//
//   * top-down: the vertices with a nonzero front word sit in the tier-binned queues of vglb_bfs (CTA chunks for rows
//     >= BFS_BIG_DEGREE edges, a warp per mid row, 8 lanes per small row). Per edge (u -> v): m = front[u] & ~seen[v]
//     (seen read through L1 as a filter: a stale word only costs an atomic that wins nothing), old = atomicOr(seen[v], m);
//     the bits won are ORed into next[v], v is queued by the thread that makes next[v] nonzero, and the level of every bit
//     won is stored. The next frontier's out-degree sum (m_f) is counted in the same kernel.
//   * bottom-up: a warp takes 32 consecutive vertices, one per lane. A vertex whose seen word is full or that has no in-edge
//     is skipped; the others OR front[u] & need over their in-neighbours (need = full & ~seen[v]) and stop once every missing
//     bit is found — lane-private for the first BFS_MS_PROBE_MAX in-neighbours, then warp-cooperatively. The owner writes
//     seen / next without atomics, and levels are stored one bit at a time for the whole warp (one 128-byte store per bit).
//   * direction: vglb_bfs's alpha/beta predicate (change_state.hpp:100-141) on union quantities — n_f = vertices with a
//     nonzero front word, m_f = their out-edges, unvisited = vertices whose seen word is not full.
// The three word arrays are taken from the context's size-keyed allocation cache for the duration of one call (not kept with
// the graph: at scale 26 and k = 64 they take 1.6 GB). The queues and the no-in-edge mask are the graph's BFS scratch, shared
// with vglb_bfs / vglb_sssp and allocated only where missing.
#include "common.cuh"
#include "frontier.cuh"

#define BFS_MS_THREADS 256
#define BFS_MS_SMALL_LANES 8
#define BFS_MS_BIG_CHUNK 8192 // a queued big row is expanded by CTAs, one per chunk of this many edges
#define BFS_MS_PROBE 4        // in-neighbours loaded per step by one lane (bottom-up)
#define BFS_MS_PROBE_MAX 16   // lane-private in-neighbours before the warp takes the row over
#define BFS_MS_LONG_UNROLL 8  // in-neighbours per lane and round trip when the warp scans one row

// counter slots: the vglb_bfs slots of frontier.cuh, then two of this file
enum
{
    M_PAIRS = C_COUNT,  // (vertex, source) pairs reached this level = level stores
    M_FULL = C_COUNT + 1, // vertices whose seen word became full this level
    M_COUNT = C_COUNT + 2
};

template <class W> __device__ __forceinline__ int word_popc(W x);
template <> __device__ __forceinline__ int word_popc<uint32_t>(uint32_t x) { return __popc(x); }
template <> __device__ __forceinline__ int word_popc<unsigned long long>(unsigned long long x) { return __popcll(x); }
template <class W> __device__ __forceinline__ int word_lowest(W x);
template <> __device__ __forceinline__ int word_lowest<uint32_t>(uint32_t x) { return __ffs(x) - 1; }
template <> __device__ __forceinline__ int word_lowest<unsigned long long>(unsigned long long x) { return __ffsll((long long)x) - 1; }
template <class W> __device__ __forceinline__ W warp_or(W x);
template <> __device__ __forceinline__ uint32_t warp_or<uint32_t>(uint32_t x) { return __reduce_or_sync(0xffffffffu, x); }
template <> __device__ __forceinline__ unsigned long long warp_or<unsigned long long>(unsigned long long x)
{
    const uint32_t lo = __reduce_or_sync(0xffffffffu, (uint32_t)x), hi = __reduce_or_sync(0xffffffffu, (uint32_t)(x >> 32));
    return ((unsigned long long)hi << 32) | lo;
}

// per-level counts a thread accumulates before the warp reduces them
struct MsCounts
{
    long long edges, mf, pairs, found, full, rows;
};

__device__ __forceinline__ void ms_count_add(long long v, unsigned long long *slot)
{
    v = warp_sum_i64(v);
    if ((threadIdx.x & 31) == 0 && v) atomicAdd(slot, (unsigned long long)v);
}

__device__ __forceinline__ void ms_counts_flush(const MsCounts &c, unsigned long long *counters)
{
    ms_count_add(c.edges, &counters[C_EDGES]);
    ms_count_add(c.mf, &counters[C_MF]);
    ms_count_add(c.pairs, &counters[M_PAIRS]);
    ms_count_add(c.found, &counters[C_FOUND]);
    ms_count_add(c.full, &counters[M_FULL]);
    ms_count_add(c.rows, &counters[C_ROWS]);
}

// NT threads (a CTA, a warp or an 8-lane group) expand the out-row [s,e) of one frontier vertex whose front word is `fu`.
// Every thread of the warp must call this together (ballots inside); `e <= s` for idle groups.
template <int NT, class W>
__device__ __forceinline__ void ms_td_expand(const int64_t *__restrict__ ptr, const int32_t *__restrict__ adj, int64_t s, int64_t e, int tid,
                                             W fu, W full, W *__restrict__ seen, W *__restrict__ next, int32_t *__restrict__ levels,
                                             int64_t V, int32_t next_level, int32_t b0, int32_t b1, const TierQueues &nq,
                                             unsigned long long *counters, MsCounts &c)
{
    for (int64_t p0 = s + tid;; p0 += NT * BFS_TD_UNROLL)
    {
        if (!__any_sync(0xffffffffu, p0 < e)) break;
        int32_t v[BFS_TD_UNROLL];
        W sv[BFS_TD_UNROLL], won[BFS_TD_UNROLL];
        bool enq[BFS_TD_UNROLL];
#pragma unroll
        for (int k = 0; k < BFS_TD_UNROLL; k++)
        {
            const int64_t p = p0 + (int64_t)k * NT;
            v[k] = p < e ? adj[p] : -1;
        }
#pragma unroll
        for (int k = 0; k < BFS_TD_UNROLL; k++) sv[k] = v[k] >= 0 ? seen[v[k]] : full;
#pragma unroll
        for (int k = 0; k < BFS_TD_UNROLL; k++)
        {
            won[k] = 0;
            const W m = fu & ~sv[k];
            if (m)
            {
                const W old = atomicOr(&seen[v[k]], m);
                won[k] = m & ~old;
                if (won[k] && (old | won[k]) == full) c.full++;
            }
        }
#pragma unroll
        for (int k = 0; k < BFS_TD_UNROLL; k++)
        {
            enq[k] = false;
            if (won[k])
            {
                enq[k] = atomicOr(&next[v[k]], won[k]) == 0;
                if (enq[k]) c.mf += ptr[v[k] + 1] - ptr[v[k]];
                c.pairs += word_popc(won[k]);
                for (W b = won[k]; b; b &= b - 1) levels[(int64_t)word_lowest(b) * V + v[k]] = next_level;
            }
        }
        enqueue_binned_multi(enq, v, b0, b1, nq, counters);
    }
}

template <class W>
__global__ void __launch_bounds__(BFS_MS_THREADS)
bfs_multi_td_kernel(const int64_t *__restrict__ ptr, const int32_t *__restrict__ adj, TierQueues cq, int32_t n_big, int32_t hub_ctas,
                    int32_t n_mid, int32_t n_small, int32_t blocks_mid, int32_t blocks_small, const W *__restrict__ front, W full,
                    W *__restrict__ seen, W *__restrict__ next, int32_t *__restrict__ levels, int32_t V, int32_t next_level,
                    int32_t b0, int32_t b1, TierQueues nq, unsigned long long *counters)
{
    const int b = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    MsCounts c = {0, 0, 0, 0, 0, 0};
    if (b < hub_ctas)
    {
        // queued big rows cut into BFS_MS_BIG_CHUNK-edge chunks dealt round-robin to `hub_ctas` CTAs (bfs_td_kernel's scheme)
        __shared__ int64_t s_row_start[BFS_MS_THREADS], s_row_end[BFS_MS_THREADS];
        __shared__ W s_word[BFS_MS_THREADS];
        __shared__ int s_chunk_prefix[BFS_MS_THREADS + 1];
        __shared__ int s_warp_chunks[BFS_MS_THREADS / 32];
        int chunk_base = 0; // chunks of the batches before this one
        for (int base = 0; base < n_big; base += BFS_MS_THREADS)
        {
            __syncthreads();
            int nch = 0;
            if (base + (int)threadIdx.x < n_big)
            {
                const int32_t u = cq.q[0][base + threadIdx.x];
                const int64_t rs = ptr[u], re = ptr[u + 1];
                s_row_start[threadIdx.x] = rs;
                s_row_end[threadIdx.x] = re;
                s_word[threadIdx.x] = front[u];
                nch = (int)((re - rs + BFS_MS_BIG_CHUNK - 1) / BFS_MS_BIG_CHUNK);
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
            for (int w = 0; w < BFS_MS_THREADS / 32; w++)
                if (w < warp) wbase += s_warp_chunks[w];
            s_chunk_prefix[threadIdx.x + 1] = wbase + incl;
            if (threadIdx.x == 0) s_chunk_prefix[0] = 0;
            __syncthreads();
            const int cnt = min(BFS_MS_THREADS, n_big - base);
            const int total = s_chunk_prefix[cnt];
            const int first = (int)((b - chunk_base % hub_ctas + hub_ctas) % hub_ctas);
            for (int ch = first; ch < total; ch += hub_ctas)
            {
                int lo = 0, hi = cnt;
                while (hi - lo > 1)
                {
                    const int mid = (lo + hi) >> 1;
                    if (s_chunk_prefix[mid] <= ch) lo = mid;
                    else hi = mid;
                }
                const int64_t s = s_row_start[lo] + (int64_t)(ch - s_chunk_prefix[lo]) * BFS_MS_BIG_CHUNK;
                const int64_t e = min(s_row_end[lo], s + BFS_MS_BIG_CHUNK);
                if (threadIdx.x == 0) c.edges += e - s;
                ms_td_expand<BFS_MS_THREADS, W>(ptr, adj, s, e, threadIdx.x, s_word[lo], full, seen, next, levels, V, next_level, b0, b1,
                                                nq, counters, c);
            }
            chunk_base += total;
        }
    }
    else if (b < hub_ctas + blocks_mid)
    {
        const int nwarps = blocks_mid * (BFS_MS_THREADS / 32);
        for (int i = (b - hub_ctas) * (BFS_MS_THREADS / 32) + warp; i < n_mid; i += nwarps)
        {
            const int32_t u = cq.q[1][i];
            const int64_t s = ptr[u], e = ptr[u + 1];
            if (lane == 0) c.edges += e - s;
            ms_td_expand<32, W>(ptr, adj, s, e, lane, front[u], full, seen, next, levels, V, next_level, b0, b1, nq, counters, c);
        }
    }
    else
    {
        constexpr int G = BFS_MS_SMALL_LANES;
        constexpr int GROUPS = BFS_MS_THREADS / G;
        const int ngroups = blocks_small * GROUPS;
        const int gid = threadIdx.x / G, gl = threadIdx.x % G;
        const int first = (b - hub_ctas - blocks_mid) * GROUPS + gid;
        for (int base = first - gid; base < n_small; base += ngroups) // trip count uniform over the warp (ballots inside)
        {
            const int i = base + gid;
            int64_t s = 0, e = 0;
            W fu = 0;
            if (i < n_small)
            {
                const int32_t u = cq.q[2][i];
                s = ptr[u];
                e = ptr[u + 1];
                fu = front[u];
                if (gl == 0) c.edges += e - s;
            }
            ms_td_expand<G, W>(ptr, adj, s, e, gl, fu, full, seen, next, levels, V, next_level, b0, b1, nq, counters, c);
        }
    }
    ms_counts_flush(c, counters);
}

template <class W>
__global__ void __launch_bounds__(BFS_MS_THREADS)
bfs_multi_bu_kernel(const int64_t *__restrict__ in_ptr, const int32_t *__restrict__ in_adj, int32_t V, const uint32_t *__restrict__ no_in_edges,
                    const W *__restrict__ front, W full, W *__restrict__ seen, W *__restrict__ next, int32_t *__restrict__ levels,
                    int32_t next_level, unsigned long long *counters)
{
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    MsCounts c = {0, 0, 0, 0, 0, 0};
    for (int64_t vbase = warp * 32; vbase < V; vbase += nwarps * 32)
    {
        const int64_t v = vbase + lane;
        const bool valid = v < V;
        const uint32_t noin = no_in_edges[vbase >> 5];
        const W sv = valid ? seen[v] : full;
        const W need = ((noin >> lane) & 1u) ? (W)0 : full & ~sv;
        W acc = 0;
        int64_t s = 0;
        int deg = 0;
        if (need)
        {
            s = in_ptr[v];
            deg = (int)(in_ptr[v + 1] - s);
            c.rows++;
        }
        // lane-private probes of the first in-neighbours (rows list their sources hubs-first: the likeliest parents)
        const int dmax = min(deg, BFS_MS_PROBE_MAX);
        for (int q = 0; q < dmax && acc != need; q += BFS_MS_PROBE)
        {
            int32_t y[BFS_MS_PROBE];
#pragma unroll
            for (int k = 0; k < BFS_MS_PROBE; k++) y[k] = q + k < dmax ? in_adj[s + q + k] : -1;
#pragma unroll
            for (int k = 0; k < BFS_MS_PROBE; k++)
                if (y[k] >= 0)
                {
                    c.edges++;
                    acc |= front[y[k]] & need;
                }
        }
        // rows longer than the probe and still missing bits: finished by the whole warp, one row at a time
        unsigned pending = __ballot_sync(FULL, acc != need && deg > BFS_MS_PROBE_MAX);
        while (pending)
        {
            const int src = __ffs(pending) - 1;
            pending &= pending - 1;
            const int64_t ps = __shfl_sync(FULL, s, src) + BFS_MS_PROBE_MAX;
            const int64_t pend = ps - BFS_MS_PROBE_MAX + __shfl_sync(FULL, deg, src);
            const W rneed = __shfl_sync(FULL, need, src);
            W racc = __shfl_sync(FULL, acc, src);
            for (int64_t p0 = ps; p0 < pend && racc != rneed; p0 += 32 * BFS_MS_LONG_UNROLL)
            {
                int32_t y[BFS_MS_LONG_UNROLL];
#pragma unroll
                for (int k = 0; k < BFS_MS_LONG_UNROLL; k++)
                {
                    const int64_t p = p0 + k * 32 + lane;
                    y[k] = p < pend ? in_adj[p] : -1;
                }
                W a = 0;
#pragma unroll
                for (int k = 0; k < BFS_MS_LONG_UNROLL; k++)
                    if (y[k] >= 0)
                    {
                        c.edges++;
                        a |= front[y[k]];
                    }
                racc |= warp_or<W>(a) & rneed;
            }
            if (lane == src) acc = racc;
        }
        if (valid)
        {
            next[v] = acc;
            if (acc)
            {
                seen[v] = sv | acc;
                c.found++;
                c.pairs += word_popc(acc);
                if ((sv | acc) == full) c.full++;
            }
        }
        // level stores: one store per source bit for the whole warp, each lane writing its own vertex
        for (W any = warp_or<W>(acc); any; any &= any - 1)
        {
            const int bit = word_lowest(any);
            if ((acc >> bit) & 1) levels[(int64_t)bit * V + v] = next_level;
        }
    }
    ms_counts_flush(c, counters);
}

// the vertices of a queued frontier get a zero front word (the array becomes the next top-down level's target)
template <class W>
__global__ void bfs_multi_clear_kernel(TierQueues q, int32_t n0, int32_t n1, int32_t n2, W *__restrict__ front)
{
    const int n = n0 + n1 + n2;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
        front[i < n0 ? q.q[0][i] : (i < n0 + n1 ? q.q[1][i - n0] : q.q[2][i - n0 - n1])] = 0;
}

// dense frontier words -> degree-binned queues of the vertices with a nonzero word
template <class W>
__global__ void bfs_multi_dense_to_queue_kernel(const W *__restrict__ front, int32_t V, int32_t b0, int32_t b1, TierQueues q,
                                                unsigned long long *counters)
{
    const int32_t padded = (int32_t)(((int64_t)V + 31) & ~31LL);
    for (int32_t v = blockIdx.x * blockDim.x + threadIdx.x; v < padded; v += gridDim.x * blockDim.x)
    {
        const bool active = v < V && front[v] != 0;
        if (__any_sync(0xffffffffu, active)) enqueue_binned(active, v, b0, b1, q, counters);
    }
}

struct MsSources
{
    int32_t src[VGLB_BFS_MULTI_MAX_SOURCES];  // source of row i
    int32_t uniq[VGLB_BFS_MULTI_MAX_SOURCES]; // distinct sources, ascending (so the tiers are contiguous runs)
    int32_t tier_start[4];                    // uniq[tier_start[t] .. tier_start[t + 1]) lie in tier t
    int32_t k, n_uniq;
};

template <class W>
__global__ void bfs_multi_init_kernel(MsSources S, int32_t V, int32_t *__restrict__ levels, W *__restrict__ seen, W *__restrict__ front,
                                      TierQueues q)
{
    const int i = threadIdx.x;
    if (i < S.k) levels[(int64_t)i * V + S.src[i]] = VGLB_FIRST_LEVEL_VERTEX;
    if (i < S.n_uniq)
    {
        const int32_t u = S.uniq[i];
        W m = 0;
        for (int j = 0; j < S.k; j++)
            if (S.src[j] == u) m |= (W)1 << j;
        seen[u] = m;
        front[u] = m;
        const int t = i < S.tier_start[1] ? 0 : (i < S.tier_start[2] ? 1 : 2);
        q.q[t][i - S.tier_start[t]] = u;
    }
}

template <class W>
static int bfs_multi_run(vglb_ctx *ctx, vglb_graph *g, const int32_t *h_sources, int32_t k, int32_t *d_levels, bool dopt,
                         long long alpha, long long beta, W *seen, W *front_a, W *front_b, vglb_stats *stats)
{
    const int32_t V = g->V;
    const int32_t b0 = g->bfs_big_border_plus1 - 1, b1 = g->tier_border[1] > b0 ? g->tier_border[1] : b0;
    const W full = k == (int)(8 * sizeof(W)) ? ~(W)0 : (((W)1 << k) - 1);
    const int64_t launches0 = ctx->launches;
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

    // the sources: distinct vertices ascending, binned by tier; a vertex that is every row's source starts out full
    MsSources S;
    memset(&S, 0, sizeof(S));
    S.k = k;
    for (int i = 0; i < k; i++) S.src[i] = h_sources[i];
    int32_t n[3] = {0, 0, 0};
    long long full_total = 0;
    for (int i = 0; i < k; i++)
    {
        int pos = 0;
        while (pos < S.n_uniq && S.uniq[pos] < h_sources[i]) pos++;
        if (pos < S.n_uniq && S.uniq[pos] == h_sources[i]) continue;
        memmove(&S.uniq[pos + 1], &S.uniq[pos], (size_t)(S.n_uniq - pos) * 4);
        S.uniq[pos] = h_sources[i];
        S.n_uniq++;
    }
    for (int i = 0; i < S.n_uniq; i++)
    {
        const int32_t u = S.uniq[i];
        n[u < b0 ? 0 : (u < b1 ? 1 : 2)]++;
        bool all = true;
        for (int j = 0; j < k; j++) all = all && S.src[j] == u;
        if (all) full_total++;
    }
    S.tier_start[0] = 0;
    S.tier_start[1] = n[0];
    S.tier_start[2] = n[0] + n[1];
    S.tier_start[3] = S.n_uniq;

    CUDA_TRY(cudaEventRecord(ctx->ev_start, st));
    CUDA_TRY(cudaMemsetAsync(d_levels, 0xFF, (size_t)k * V * 4, st)); // UNVISITED_VERTEX = -1
    CUDA_TRY(cudaMemsetAsync(seen, 0, (size_t)3 * V * sizeof(W), st)); // seen, front_a, front_b are one block
    CUDA_TRY(cudaMemsetAsync(d_cnt, 0, M_COUNT * 8, st));
    bfs_multi_init_kernel<W><<<1, VGLB_BFS_MULTI_MAX_SOURCES, 0, st>>>(S, V, d_levels, seen, front_a, cq);
    KERNEL_TRY();
    ctx->launches++;

    W *cur = front_a, *nxt = front_b;
    long long n_cur = S.n_uniq, m_f_next = 0;
    bool bottom_up = false;
    int32_t level = VGLB_FIRST_LEVEL_VERTEX;
    int64_t tot_edges = 0, tot_rows = 0, tot_frontier_bytes = 0, tot_pairs = k, levels_run = 0;
    int32_t bu_levels = 0;
    const int64_t w = sizeof(W);
    const long long factor = (g->E / (V > 0 ? V : 1)) / 2 > 0 ? (g->E / V) / 2 : 1; // change_state.hpp:104
    const int max_blocks = ctx->sm_count * 16;
    const int big_chunks = (int)ceil_div64(g->max_degree > 0 ? g->max_degree : 1, BFS_MS_BIG_CHUNK);
    int rc;
    while (n_cur > 0)
    {
        if (!bottom_up)
        {
            const int blocks_mid = (int)min((int64_t)max_blocks, ceil_div64(n[1], BFS_MS_THREADS / 32));
            const int blocks_small = (int)min((int64_t)max_blocks, ceil_div64(n[2], BFS_MS_THREADS / BFS_MS_SMALL_LANES));
            const int hub_ctas = (int)min((int64_t)n[0] * big_chunks, (int64_t)ctx->sm_count * 4);
            const int64_t grid = (int64_t)hub_ctas + blocks_mid + blocks_small;
            bfs_multi_td_kernel<W><<<(unsigned)grid, BFS_MS_THREADS, 0, st>>>(g->d_out_ptr, g->d_out_adj, cq, n[0], hub_ctas, n[1], n[2],
                                                                             blocks_mid, blocks_small, cur, full, seen, nxt, d_levels, V,
                                                                             level + 1, b0, b1, nq, d_cnt);
            KERNEL_TRY();
            ctx->launches++;
        }
        else
        {
            bfs_multi_bu_kernel<W><<<ctx->sm_count * 8, BFS_MS_THREADS, 0, st>>>(g->d_in_ptr, g->d_in_adj, V, (const uint32_t *)g->d_scratch_i32,
                                                                                cur, full, seen, nxt, d_levels, level + 1, d_cnt);
            KERNEL_TRY();
            ctx->launches++;
            bu_levels++;
        }
        rc = vglb_counters_fetch(ctx, d_cnt, M_COUNT);
        if (rc != VGLB_OK) return rc;
        levels_run++;
        const int32_t nn[3] = {(int32_t)h_cnt[C_NEXT_BIG], (int32_t)h_cnt[C_NEXT_MID], (int32_t)h_cnt[C_NEXT_SMALL]};
        const long long n_next = bottom_up ? (long long)h_cnt[C_FOUND] : (long long)nn[0] + nn[1] + nn[2];
        tot_edges += (int64_t)h_cnt[C_EDGES];
        tot_pairs += (int64_t)h_cnt[M_PAIRS];
        full_total += (long long)h_cnt[M_FULL];
        if (bottom_up)
        {
            tot_rows += (int64_t)h_cnt[C_ROWS];
            tot_frontier_bytes += (int64_t)V * 2 * w + ((int64_t)V + 7) / 8; // seen + next words, no-in-edge mask
        }
        else
        {
            tot_rows += n_cur;
            tot_frontier_bytes += n_next * (8 + w); // queue written + read, next word set
        }
        m_f_next = (long long)h_cnt[C_MF];
        if (n_next == 0) break;

        bool next_bu = bottom_up;
        if (dopt)
        {
            const long long unvisited = (long long)V - full_total;
            if (!bottom_up && n_cur < n_next)
            {
                if (m_f_next >= (unvisited * factor + V) / alpha) next_bu = true;
            }
            else if (bottom_up && n_cur >= n_next)
            {
                if (n_next < (unvisited * factor + V) / (factor * beta)) next_bu = false;
            }
        }
        CUDA_TRY(cudaMemsetAsync(d_cnt, 0, M_COUNT * 8, st));
        // Before a top-down level the target array must be all zero; a bottom-up level writes every word of its target.
        if (!bottom_up && !next_bu)
        {
            bfs_multi_clear_kernel<W><<<(unsigned)min((int64_t)max_blocks, ceil_div64(n_cur, 256)), 256, 0, st>>>(cq, n[0], n[1], n[2], cur);
            KERNEL_TRY();
            ctx->launches++;
            tot_frontier_bytes += n_cur * (4 + w);
            TierQueues t = cq; cq = nq; nq = t;
            n[0] = nn[0]; n[1] = nn[1]; n[2] = nn[2];
        }
        else if (bottom_up && !next_bu)
        {
            bfs_multi_dense_to_queue_kernel<W><<<(unsigned)min((int64_t)max_blocks, ceil_div64(V, 256)), 256, 0, st>>>(nxt, V, b0, b1, cq, d_cnt);
            KERNEL_TRY();
            ctx->launches++;
            rc = vglb_counters_fetch(ctx, d_cnt, 3);
            if (rc != VGLB_OK) return rc;
            n[0] = (int32_t)h_cnt[0]; n[1] = (int32_t)h_cnt[1]; n[2] = (int32_t)h_cnt[2];
            CUDA_TRY(cudaMemsetAsync(d_cnt, 0, M_COUNT * 8, st));
            CUDA_TRY(cudaMemsetAsync(cur, 0, (size_t)V * w, st));
            tot_frontier_bytes += (int64_t)V * 2 * w + 4 * n_next;
        }
        // top-down -> bottom-up: the top-down level left its discoveries as dense words in nxt, which is what the
        // bottom-up level reads
        W *t = cur; cur = nxt; nxt = t;
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
        // the formula of include/vgl_b200.h (vglb_bfs_multi)
        stats->algorithmic_bytes = (4 + w) * tot_edges + (12 + w) * tot_rows + tot_frontier_bytes + 4LL * k * V + 4 * tot_pairs;
        stats->kernel_launches = ctx->launches - launches0;
        stats->bottom_up_levels = bu_levels;
    }
    return VGLB_OK;
}

extern "C" int vglb_bfs_multi(vglb_ctx *ctx, vglb_graph *g, int32_t num_sources, const int32_t *h_sources_sorted, int32_t *d_levels,
                              const vglb_bfs_opts *opts, vglb_stats *stats)
{
    VGLB_REQUIRE(ctx != NULL && g != NULL && h_sources_sorted != NULL && d_levels != NULL, "vglb_bfs_multi: NULL argument");
    VGLB_REQUIRE(num_sources >= 1 && num_sources <= VGLB_BFS_MULTI_MAX_SOURCES, "vglb_bfs_multi: num_sources must be in 1..64");
    VGLB_REQUIRE(g->comm == NULL, "vglb_bfs_multi: partitioned graphs are not supported");
    for (int i = 0; i < num_sources; i++)
        VGLB_REQUIRE(h_sources_sorted[i] >= 0 && h_sources_sorted[i] < g->V, "vglb_bfs_multi: source out of range");
    const bool dopt = opts && opts->direction_optimising;
    CUDA_TRY(cudaSetDevice(ctx->device));
    if (dopt && !g->d_in_ptr)
    {
        int rc_in = vglb_graph_derive_incoming(ctx, g); // as vglb_bfs: the bottom-up levels need the incoming CSR
        if (rc_in != VGLB_OK) return rc_in;
    }
    const long long alpha = (opts && opts->alpha > 0) ? opts->alpha : 15;
    const long long beta = (opts && opts->beta > 0) ? opts->beta : 18;
    // the graph's BFS scratch, shared with vglb_bfs / vglb_sssp: only what is missing is allocated
    for (int i = 0; i < 2; i++)
        if (!g->d_queue[i]) CUDA_TRY(vglb_dev_alloc(&g->d_queue[i], ((size_t)g->V + 3) * 4));
    int rc = bfs_prepare_no_in_edges(ctx, g);
    if (rc != VGLB_OK) return rc;
    if (g->bfs_big_border_plus1 == 0) // first id with fewer than BFS_BIG_DEGREE edges, once per graph (shared with vglb_bfs)
    {
        int32_t border = 0;
        rc = vglb_graph_threshold_vertex(ctx, g, BFS_BIG_DEGREE, &border);
        if (rc != VGLB_OK) return rc;
        g->bfs_big_border_plus1 = border + 1;
    }
    // per-call word arrays from the context's allocation cache: seen | front_a | front_b, V words each
    const bool wide = num_sources > 32;
    const size_t wbytes = wide ? 8 : 4;
    void *words = NULL;
    CUDA_TRY(vglb_dev_alloc(&words, (size_t)3 * ((size_t)g->V > 0 ? g->V : 1) * wbytes));
    if (wide)
    {
        unsigned long long *p = (unsigned long long *)words;
        rc = bfs_multi_run<unsigned long long>(ctx, g, h_sources_sorted, num_sources, d_levels, dopt, alpha, beta, p, p + g->V, p + 2 * (size_t)g->V, stats);
    }
    else
    {
        uint32_t *p = (uint32_t *)words;
        rc = bfs_multi_run<uint32_t>(ctx, g, h_sources_sorted, num_sources, d_levels, dopt, alpha, beta, p, p + g->V, p + 2 * (size_t)g->V, stats);
    }
    if (rc != VGLB_OK) cudaStreamSynchronize(ctx->stream); // nothing may still use the block when it goes back to the cache
    vglb_dev_free(words);
    return rc;
}
