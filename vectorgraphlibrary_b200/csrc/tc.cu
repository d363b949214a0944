// tc.cu — triangle counting (algorithms/tc) over a degree-oriented CSR that every call builds on the device.
//
// What is counted: the triangles of the undirected simple graph under the OUTGOING CSR ({u, w} is an edge when u != w and
// u->w or w->u is in the CSR; duplicates count once, self loops are dropped). Only the outgoing CSR is read.
//
// Build (all on ctx->stream, scratch from the context's cache):
//   1. tc_key_kernel: CSR edge (u, w), u != w  ->  key (max(u, w) << b) | min(u, w), b = vglb_key_bits(V); a self loop gets
//      an all-ones key, which sorts last.
//   2. cub::DeviceRadixSort::SortKeys over bits [0, 2b) only.
//   3. cub::DeviceSelect::Unique drops the duplicates; tc_ids_kernel writes the int32 column ids, stops at the self-loop key
//      and adds each row's length at its two ends (no contention); cub::DeviceScan::ExclusiveSum gives the int64 row pointers.
// Row u of the oriented CSR holds N+(u) = {w < u : {u, w} an edge}, ascending. SCATTER ids are sorted by out-degree
// descending, so hubs get short rows. A triangle w < v < u is found exactly once: at row u, edge v (position j of N+(u)),
// element w, and the only candidates are N+(u)[0, j).
//
// Count (tc_count_kernel). For each oriented edge (u, v) at position j of its row, intersect N+(u)[0, j) with N+(v). One
// side is read whole and each of its elements is looked up in the other by binary search:
//   * 2 j < |N+(v)|: the prefix's elements are probed into N+(v) (global memory);
//   * otherwise N+(v) is streamed coalesced and each element is looked up in the prefix (shared memory when staged).
// A streamed element costs less than a probe, which is a chain of dependent global loads: on a B200, "probe the shorter side"
// (factor 1) took 1325 / 329 ms at RMAT / uniform scale 24, factor 2 1281 / 268 ms, 4 1563 / 265 ms, always streaming
// 2961 / 263 ms (DESIGN §4.8). So an edge reads m = j or |N+(v)| list elements (stats->edges_inspected = sum of m).
// Load balance: every edge has cost TC_EDGE_COST + m * (1 + bits(length of the searched list)), the last factor being the
// depth of the binary search. A merge path over the exclusive prefix sum of the costs cuts the edges into windows of
// TC_WINDOW cost units (a window holds the edges whose cost starts in it, so at most TC_WINDOW / TC_EDGE_COST of them);
// warps take groups of TC_GROUP consecutive windows, dealt round-robin. A warp copies its window's slice adj[ptr[first row], last edge] into its own
// TC_STAGE-entry shared-memory buffer, which holds every prefix the window needs. A window whose slice is longer (rows of
// more than TC_STAGE - TC_WINDOW / TC_EDGE_COST entries; a clique's last rows) reads the prefixes from global memory instead.
// Within a window, edges go 32 at a time (lane = edge) and their m elements are one flat range over the warp.
// Per-vertex counts: a match adds 1 to w, the edge's match count to v and the row's sum to u (one add per row per 32 edges).
// Adds for ids < TC_HUB (the highest-degree vertices, where the w adds pile up) go to a per-CTA shared-memory table of 64-bit
// counters flushed once per CTA; the other w adds are aggregated per warp over equal ids. The total goes to the counter word
// CTR_TC_TOTAL. All arithmetic is integer, so two calls give identical arrays.
#include <algorithm>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_select.cuh>

#include "common.cuh"

#define TC_THREADS 512
#define TC_WARPS (TC_THREADS / 32)
#define TC_EDGE_COST 32 // cost units of an edge before its elements: row search, the edge's id and its target's row pointers
#define TC_WINDOW 8192  // cost units per warp window; a window holds at most TC_WINDOW / TC_EDGE_COST = 256 edges
#define TC_GROUP 8      // consecutive windows a warp takes at a time; groups are dealt to the warps in turn
#define TC_STAGE 2048   // int32 entries of a warp's staging buffer: prefixes of rows up to 1792 entries are staged
#define TC_HUB 4096     // ids with a shared-memory counter in every CTA (32 KB)
#define TC_SMEM_BYTES ((size_t)TC_WARPS * TC_STAGE * 4 + (size_t)TC_WARPS * 32 * 4 + (size_t)TC_HUB * 8)

static_assert(TC_STAGE > TC_WINDOW / TC_EDGE_COST, "a window's edges fit its staging buffer");

typedef unsigned long long u64;
#define TC_SELF_LOOP (~0ULL)

// the row of edge e: the largest u in [0, V) with ptr[u] <= e
__device__ __forceinline__ int32_t tc_row_of(const int64_t *__restrict__ ptr, int32_t V, int64_t e)
{
    int32_t lo = 0, hi = V - 1;
    while (lo < hi)
    {
        const int32_t mid = lo + (hi - lo + 1) / 2;
        if (ptr[mid] <= e) lo = mid;
        else hi = mid - 1;
    }
    return lo;
}

__global__ void tc_key_kernel(const int64_t *__restrict__ ptr, const int32_t *__restrict__ adj, int32_t V, int64_t E, int b,
                              u64 *__restrict__ keys)
{
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < E; e += (int64_t)gridDim.x * blockDim.x)
    {
        const uint32_t u = (uint32_t)tc_row_of(ptr, V, e), w = (uint32_t)adj[e];
        keys[e] = u == w ? TC_SELF_LOOP : ((u64)max(u, w) << b) | (u64)min(u, w);
    }
}

// unique keys -> column ids, row lengths (added at both ends of each row's run), E+ and the rows with entries
__global__ void tc_ids_kernel(const u64 *__restrict__ uniq, int64_t E, int b, int32_t *__restrict__ oadj,
                              int64_t *__restrict__ len, u64 *__restrict__ ctr)
{
    const int64_t n = (int64_t)ctr[CTR_TC_UNIQUE];
    const u64 mask = (1ULL << b) - 1;
    // the block stays in the loop as a whole, so the row starts are counted with one add per warp
    for (int64_t i0 = (int64_t)blockIdx.x * blockDim.x; i0 < E; i0 += (int64_t)gridDim.x * blockDim.x)
    {
        const int64_t i = i0 + threadIdx.x;
        bool start = false;
        if (i < n)
        {
            const u64 k = uniq[i];
            if (i == n - 1) ctr[CTR_TC_EDGES] = k == TC_SELF_LOOP ? i : i + 1;
            if (k != TC_SELF_LOOP)
            {
                const u64 r = k >> b;
                oadj[i] = (int32_t)(k & mask);
                start = i == 0 || (uniq[i - 1] >> b) != r;
                // the self-loop key's row bits (>= 2^(64-b) - 1) never equal a row id
                const bool end = i == n - 1 || (uniq[i + 1] >> b) != r;
                if (start) atomicAdd((u64 *)(len + r), (u64)(-i));
                if (end) atomicAdd((u64 *)(len + r), (u64)(i + 1));
            }
        }
        const unsigned starts = __ballot_sync(0xffffffffu, start);
        if (starts && (threadIdx.x & 31) == 0) atomicAdd(ctr + CTR_TC_ROWS, (u64)__popc(starts));
    }
}

__device__ __forceinline__ int tc_bits(int64_t x) { return 64 - __clzll(x); }

// cost[i] = TC_EDGE_COST + m * (1 + bits(the searched list's length)) for the oriented edges, 0 for the slots [E+, E]
__global__ void tc_cost_kernel(const u64 *__restrict__ uniq, int64_t E, int b, const int64_t *__restrict__ optr,
                               const u64 *__restrict__ ctr, int64_t *__restrict__ cost)
{
    const int64_t Ep = (int64_t)ctr[CTR_TC_EDGES];
    const u64 mask = (1ULL << b) - 1;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i <= E; i += (int64_t)gridDim.x * blockDim.x)
    {
        int64_t c = 0;
        if (i < Ep)
        {
            const u64 k = uniq[i];
            const int64_t u = (int64_t)(k >> b), v = (int64_t)(k & mask);
            const int64_t j = i - optr[u], nv = optr[v + 1] - optr[v];
            const bool probe = 2 * j < nv;
            const int64_t m = probe ? j : nv;
            c = TC_EDGE_COST + m * (1 + tc_bits(probe ? nv : j));
        }
        cost[i] = c;
    }
}

// smallest r in [lo, hi] with a[r] >= target (hi when none in [lo, hi)), 32 probes at a time
__device__ __forceinline__ int64_t tc_lower_bound(const int64_t *__restrict__ a, int64_t lo, int64_t hi, int64_t target, int lane)
{
    while (lo < hi)
    {
        const int64_t step = (hi - lo + 31) / 32;
        const int64_t pos = lo + (int64_t)lane * step;
        const bool ge = pos < hi ? a[pos] >= target : true;
        const unsigned m = __ballot_sync(0xffffffffu, ge);
        if (m == 0u)
        {
            lo = lo + 31 * step + 1;
            continue;
        }
        const int k = __ffs(m) - 1;
        const int64_t found = lo + (int64_t)k * step;
        if (k > 0) lo = found - step + 1;
        hi = found < hi ? found : hi;
        if (k == 0) break;
    }
    return lo;
}

struct TcCount
{
    const int64_t *optr;  // oriented CSR
    const int32_t *oadj;
    const int64_t *pre;   // exclusive prefix sum of the edge costs, [E+ + 1] used
    int32_t V;
    const u64 *ctr;       // ctx->d_counters: CTR_TC_EDGES in, CTR_TC_TOTAL / CTR_TC_ELEMENTS out
    u64 *counts;          // int64[V], zeroed
};

// one add to vertex id's count: the CTA's table for the hub ids, global memory for the others
__device__ __forceinline__ void tc_add(const TcCount &P, u64 *s_hub, int64_t id, u64 val)
{
    if (id < TC_HUB) atomicAdd(s_hub + id, val);
    else atomicAdd(P.counts + id, val);
}

// binary search of x in the ascending list (staged ? buf[i - s] : adj[i]), i in [lo, lo + n)
__device__ __forceinline__ bool tc_find(const int32_t *__restrict__ adj, const int32_t *buf, int64_t s, bool staged, int64_t lo,
                                        int64_t n, int32_t x)
{
    while (n > 0)
    {
        const int64_t h = n >> 1;
        const int32_t y = staged ? buf[lo + h - s] : adj[lo + h];
        if (y == x) return true;
        if (y < x)
        {
            lo += h + 1;
            n -= h + 1;
        }
        else n = h;
    }
    return false;
}

__global__ void __launch_bounds__(TC_THREADS, 1) tc_count_kernel(const __grid_constant__ TcCount P)
{
    const unsigned FULL = 0xffffffffu;
    extern __shared__ __align__(16) unsigned char tc_smem[];
    u64 *s_hub = (u64 *)tc_smem;
    int32_t *s_hit_all = (int32_t *)(tc_smem + (size_t)TC_HUB * 8);
    int32_t *s_stage_all = s_hit_all + TC_WARPS * 32;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int32_t *s_hit = s_hit_all + warp * 32, *buf = s_stage_all + warp * TC_STAGE;
    for (int i = threadIdx.x; i < TC_HUB; i += TC_THREADS) s_hub[i] = 0;
    s_hit[lane] = 0;
    __syncthreads();

    const int64_t Ep = (int64_t)P.ctr[CTR_TC_EDGES];
    const int64_t nwin = (P.pre[Ep] + TC_WINDOW - 1) / TC_WINDOW;
    const int64_t nw = (int64_t)gridDim.x * TC_WARPS, gw = (int64_t)blockIdx.x * TC_WARPS + warp;
    u64 tri = 0, elems = 0;
    for (int64_t w0 = gw * TC_GROUP; w0 < nwin; w0 += nw * TC_GROUP)
    {
        const int64_t w1 = w0 + TC_GROUP < nwin ? w0 + TC_GROUP : nwin;
        int64_t e0 = tc_lower_bound(P.pre, 0, Ep, w0 * TC_WINDOW, lane);
        for (int64_t w = w0; w < w1; w++)
        {
            const int64_t near = e0 + TC_WINDOW / TC_EDGE_COST < Ep ? e0 + TC_WINDOW / TC_EDGE_COST : Ep;
            const int64_t e1 = tc_lower_bound(P.pre, e0, near, (w + 1) * TC_WINDOW, lane);
            if (e0 == e1) continue;
            // rows of the window: ub = row of e0; the slice adj[ptr[ub], e1) holds every prefix the window needs
            int32_t ub = (int32_t)tc_lower_bound(P.optr, 0, P.V, e0 + 1, lane) - 1;
            const int64_t s = P.optr[ub];
            const bool staged = e1 - s <= TC_STAGE;
            if (staged)
            {
                for (int64_t i = lane; i < e1 - s; i += 32) buf[i] = P.oadj[s + i];
                __syncwarp();
            }
            for (int64_t base = e0; base < e1; base += 32)
            {
                const int64_t p = base + lane;
                const bool have = p < e1;
                const int64_t plast = base + 31 < e1 - 1 ? base + 31 : e1 - 1;
                const int32_t uh = (int32_t)tc_lower_bound(P.optr, ub, P.V, plast + 1, lane) - 1;
                int32_t u = ub;
                int64_t pu = 0, vs = 0;
                int32_t v = 0, m = 0, j = 0, nv = 0;
                bool probe = false;
                if (have)
                {
                    int32_t lo = ub, hi = uh; // the largest u with optr[u] <= p
                    while (lo < hi)
                    {
                        const int32_t mid = lo + (hi - lo + 1) / 2;
                        if (P.optr[mid] <= p) lo = mid;
                        else hi = mid - 1;
                    }
                    u = lo;
                    pu = P.optr[u];
                    j = (int32_t)(p - pu);
                    v = staged ? buf[p - s] : P.oadj[p];
                    vs = P.optr[v];
                    nv = (int32_t)(P.optr[v + 1] - vs);
                    probe = 2 * (int64_t)j < nv;
                    m = probe ? j : nv;
                }
                elems += (u64)m;
                // a row holds fewer than sqrt(2 E) entries, so 32 edges' elements fit an int
                int incl = m;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1)
                {
                    const int up = __shfl_up_sync(FULL, incl, o);
                    if (lane >= o) incl += up;
                }
                const int excl = incl - m;
                const int total = __shfl_sync(FULL, incl, 31);
                for (int fb = 0; fb < total; fb += 32)
                {
                    const int f = fb + lane;
                    const int probe_f = f < total ? f : total - 1;
                    int k = 0; // largest k with excl[k] <= f (edges without elements are stepped over)
#pragma unroll
                    for (int st = 16; st > 0; st >>= 1)
                    {
                        const int cand = k + st;
                        const int o = __shfl_sync(FULL, excl, cand & 31);
                        if (cand < 32 && o <= probe_f) k = cand;
                    }
                    const int i = probe_f - __shfl_sync(FULL, excl, k);
                    const bool kprobe = __shfl_sync(FULL, probe, k);
                    const int64_t kpu = __shfl_sync(FULL, pu, k), kvs = __shfl_sync(FULL, vs, k);
                    const int32_t kj = __shfl_sync(FULL, j, k), kn = __shfl_sync(FULL, nv, k);
                    bool found = false;
                    int32_t x = 0;
                    if (f < total)
                    {
                        if (kprobe)
                        {
                            // prefix element i, looked up in N+(v) = adj[kvs, kvs + kn)
                            x = staged ? buf[kpu + i - s] : P.oadj[kpu + i];
                            found = tc_find(P.oadj, buf, s, false, kvs, kn, x);
                        }
                        else
                        {
                            // element i of N+(v), looked up in the prefix adj[kpu, kpu + kj)
                            x = P.oadj[kvs + i];
                            found = tc_find(P.oadj, buf, s, staged, kpu, kj, x);
                        }
                    }
                    if (found)
                    {
                        atomicAdd(s_hit + k, 1);
                        if (x < TC_HUB) atomicAdd(s_hub + x, 1ULL);
                    }
                    const bool far = found && x >= TC_HUB;
                    const unsigned fm = __ballot_sync(FULL, far);
                    if (far)
                    {
                        const unsigned peers = __match_any_sync(fm, x);
                        if (lane == __ffs(peers) - 1) atomicAdd(P.counts + x, (u64)__popc(peers));
                    }
                }
                __syncwarp();
                const int t = s_hit[lane];
                s_hit[lane] = 0;
                __syncwarp();
                if (t > 0) tc_add(P, s_hub, v, (u64)t);
                tri += (u64)t;
                // u: the sum over this batch's edges of each row, added by the last lane of the row's run
                int rs = t;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1)
                {
                    const int up = __shfl_up_sync(FULL, rs, o);
                    const int uu = __shfl_up_sync(FULL, u, o);
                    if (lane >= o && uu == u) rs += up;
                }
                const int32_t unext = __shfl_down_sync(FULL, u, 1);
                const bool hnext = __shfl_down_sync(FULL, have, 1);
                if (have && rs > 0 && (lane == 31 || !hnext || unext != u)) tc_add(P, s_hub, u, (u64)rs);
                ub = __shfl_sync(FULL, u, (int)(plast - base));
            }
            e0 = e1;
            __syncwarp(); // the next window overwrites the staging buffer
        }
    }
    // totals: per warp, then one add per CTA
    __shared__ u64 s_red[2][TC_WARPS];
    tri = (u64)warp_sum_i64((long long)tri);
    elems = (u64)warp_sum_i64((long long)elems);
    if (lane == 0)
    {
        s_red[0][warp] = tri;
        s_red[1][warp] = elems;
    }
    __syncthreads();
    if (threadIdx.x == 0)
    {
        u64 a = 0, c = 0;
#pragma unroll
        for (int i = 0; i < TC_WARPS; i++)
        {
            a += s_red[0][i];
            c += s_red[1][i];
        }
        if (a) atomicAdd((u64 *)P.ctr + CTR_TC_TOTAL, a);
        if (c) atomicAdd((u64 *)P.ctr + CTR_TC_ELEMENTS, c);
    }
    for (int i = threadIdx.x; i < TC_HUB && i < P.V; i += TC_THREADS)
        if (s_hub[i]) atomicAdd(P.counts + i, s_hub[i]);
}

extern "C" int vglb_tc(vglb_ctx *ctx, vglb_graph *g, int64_t *d_counts, int64_t *h_total, vglb_stats *stats)
{
    VGLB_REQUIRE(ctx != NULL && g != NULL && d_counts != NULL && h_total != NULL, "vglb_tc: NULL argument");
    VGLB_REQUIRE(g->comm == NULL, "vglb_tc: partitioned graphs are not supported");
    CUDA_TRY(cudaSetDevice(ctx->device));
    const int32_t V = g->V;
    const int64_t E = g->E;
    const int b = vglb_key_bits(V);
    cudaStream_t st = ctx->stream;
    const int64_t launches0 = ctx->launches;
    u64 *ctr = (u64 *)ctx->d_counters;

    dev_ptr<u64> k0, k1;
    dev_ptr<int32_t> oadj;
    dev_ptr<int64_t> optr;
    dev_ptr<void> tmp;
    CUDA_TRY(vglb_dev_alloc(k0, (size_t)(E + 1) * sizeof(u64)));
    CUDA_TRY(vglb_dev_alloc(k1, (size_t)(E + 1) * sizeof(u64)));
    CUDA_TRY(vglb_dev_alloc(oadj, (size_t)(E > 0 ? E : 1) * sizeof(int32_t)));
    CUDA_TRY(vglb_dev_alloc(optr, ((size_t)V + 1) * sizeof(int64_t)));

    CUDA_TRY(cudaEventRecord(ctx->ev_start, st));
    CUDA_TRY(cudaMemsetAsync(ctr + CTR_TC_TOTAL, 0, (CTR_TC_END - CTR_TC_TOTAL) * sizeof(u64), st));
    CUDA_TRY(cudaMemsetAsync(d_counts, 0, (size_t)V * sizeof(int64_t), st));
    if (E > 0)
    {
        const int grid = (int)std::min<int64_t>((int64_t)ctx->sm_count * 8, ceil_div64(E + 1, 256));
        // 1. keys
        tc_key_kernel<<<grid, 256, 0, st>>>(g->d_out_ptr, g->d_out_adj, V, E, b, k0.get());
        KERNEL_TRY();
        ctx->launches++;
        // 2. sort over the 2b key bits
        cub::DoubleBuffer<u64> keys(k0.get(), k1.get());
        CUDA_TRY(vglb_cub(tmp, [&](void *t, size_t &bytes) {
            return cub::DeviceRadixSort::SortKeys(t, bytes, keys, E, 0, 2 * b, st);
        }));
        ctx->launches++;
        // 3. dedupe, column ids and row lengths, row pointers
        u64 *sorted = keys.Current(), *uniq = keys.Alternate();
        CUDA_TRY(vglb_cub(tmp, [&](void *t, size_t &bytes) {
            return cub::DeviceSelect::Unique(t, bytes, sorted, uniq, (int64_t *)(ctr + CTR_TC_UNIQUE), E, st);
        }));
        ctx->launches++;
        int64_t *len = (int64_t *)sorted; // the sorted keys are dead: V + 1 row lengths, then the edge costs
        dev_ptr<int64_t> len_big;
        if (V + 1 > E + 1)
        {
            CUDA_TRY(vglb_dev_alloc(len_big, ((size_t)V + 1) * sizeof(int64_t)));
            len = len_big.get();
        }
        CUDA_TRY(cudaMemsetAsync(len, 0, ((size_t)V + 1) * sizeof(int64_t), st));
        tc_ids_kernel<<<grid, 256, 0, st>>>(uniq, E, b, oadj.get(), len, ctr);
        KERNEL_TRY();
        ctx->launches++;
        CUDA_TRY(vglb_cub(tmp, [&](void *t, size_t &bytes) {
            return cub::DeviceScan::ExclusiveSum(t, bytes, (const int64_t *)len, optr.get(), V + 1, st);
        }));
        ctx->launches++;
        len_big.reset();
        // 4. edge costs and their prefix sum (into the unique keys' buffer once the costs are written)
        int64_t *cost = (int64_t *)sorted, *pre = (int64_t *)uniq;
        tc_cost_kernel<<<grid, 256, 0, st>>>(uniq, E, b, optr.get(), ctr, cost);
        KERNEL_TRY();
        ctx->launches++;
        CUDA_TRY(vglb_cub(tmp, [&](void *t, size_t &bytes) {
            return cub::DeviceScan::ExclusiveSum(t, bytes, (const int64_t *)cost, pre, E + 1, st);
        }));
        ctx->launches++;
        // 5. count
        TcCount P;
        P.optr = optr.get();
        P.oadj = oadj.get();
        P.pre = pre;
        P.V = V;
        P.ctr = ctr;
        P.counts = (u64 *)d_counts;
        CUDA_TRY(cudaFuncSetAttribute(tc_count_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TC_SMEM_BYTES));
        tc_count_kernel<<<ctx->sm_count, TC_THREADS, TC_SMEM_BYTES, st>>>(P);
        KERNEL_TRY();
        ctx->launches++;
    }
    VGLB_TRY(vglb_finish_run(ctx, launches0, stats));
    VGLB_TRY(vglb_counters_fetch(ctx, ctx->d_counters, CTR_TC_END)); // the stream is idle: no further wait
    const int64_t *h = ctx->h_counters;
    *h_total = h[CTR_TC_TOTAL];
    if (!stats) return VGLB_OK;
    stats->iterations = 1;
    stats->edges_inspected = h[CTR_TC_ELEMENTS];
    stats->vertices_processed = h[CTR_TC_ROWS];
    // the formula of include/vgl_b200.h (vglb_tc)
    stats->algorithmic_bytes = 8 * E + 12 * h[CTR_TC_EDGES] + 4 * h[CTR_TC_ELEMENTS] + 16LL * V;
    return VGLB_OK;
}
