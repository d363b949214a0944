// vgl_b200/advance.cuh — header-only, lambda-generic device side of the B200 backend (sm_100a).
//
// These templates are the "advance / compute / reduce / generate_new_frontier" operators of VGL's GraphAbstractions
// (vgl_compute_api/common/graph_abstractions.h:96-152) for ARBITRARY user functors: device lambdas cannot cross the
// C ABI of libvgl_b200, so the generic path is instantiated in the caller's translation unit (nvcc --extended-lambda) by
//   * include/vgl_b200/overlay/vgl_compute_api/gpu/graph_abstractions_gpu.h — the drop-in backend the reference's own
//     algorithms compile against, unchanged, and
//   * include/vgl_b200/graph_abstractions_b200.cuh — the stand-alone operator API over C-ABI objects,
// while the data structures, compaction and the fused algorithms live behind the C ABI.
//
// Functor contracts = the reference's (architecture_independent_api.h:17-30):
//   edge_op  (int src_id, int dst_id, int local_edge_pos, long long global_edge_pos, int vector_index)
//   vertex op(int src_id, int connections_count, int vector_index)       pre: before, post: after all edges of src
// vector_index is the lane id (0..31), also for vertex ops. The edge ops of one vertex run concurrently on up to a whole
// CTA and must be atomic where the reference's GPU lambdas are (VGL_SRC_ID_ADD, architecture_independent_api.h:47-51).
// Ordering guarantee per vertex: pre happens-before every edge op happens-before post (barriers in between) — stronger
// than the reference's GPU kernels, which run pre/post on thread 0 without a barrier (gpu/advance_csr.hpp:78-120).
//
// Load balancing (north_star (a)) replaces the reference's block / virtual-warp kernels on six streams
// (vgl_compute_api/gpu/advance_vect_csr.hpp:56-141). Ids are degree-sorted, so a degree class is an id range:
//   hub rows   (>= 4096 edges)  one CTA per row — or one CTA per 8192-edge chunk of the row when there are no vertex ops
//                               (the largest rows of a scale-26 Kronecker graph have > 10^6 edges);
//   ALL_ACTIVE, the other rows  MERGE-PATH by rows: warp w takes the complete rows whose first edge falls into the w-th
//                               2048-edge window of the adjacency array (32-ary search over the row pointers), so every warp
//                               gets the same amount of work whatever the degree distribution. Rows with >= 32 edges are
//                               walked by the whole warp, coalesced; shorter rows 32 at a time as ONE flat edge range
//                               (shuffle search over the 32 degree prefix sums), every lane busy even on degree-1 rows;
//   SPARSE                      the ascending id list splits into hub / mid / small prefixes (the frontier counts them while
//                               it compacts): hubs as above, mid rows (>= 32 edges) one warp each, small rows 32 per warp as
//                               a flat edge range;
//   rows without edges          vertex ops only (skipped when there are none).
// Every lane handles 4 independent edges per step (index loads first, then the edge ops).
#pragma once
#include <cuda_runtime.h>
#include <limits.h>
#include <stdint.h>

#include <type_traits>

namespace vglb
{

constexpr int kAdvThreads = 256;
constexpr int kAdvWarps = kAdvThreads / 32;
constexpr int kNumTiers = 8;
constexpr int kHubChunk = 8192;   // edges of a hub row handled by one CTA when the row may be split
constexpr int kWarpEdges = 2048;  // ALL_ACTIVE: edge window whose rows one warp takes
constexpr int kEdgeUnroll = 4;

struct CsrView
{
    const int64_t *ptr;
    const int32_t *adj;
    int32_t V;
    int32_t tier_border[kNumTiers]; // first id whose degree is below {4096,32,16,8,4,2,1,0}
    int32_t max_degree;
};

struct NoVertexOp
{
    __device__ __forceinline__ void operator()(int, int, int) const {}
};

template <class Op>
struct is_no_vertex_op : std::is_same<typename std::decay<Op>::type, NoVertexOp>
{
};

// ---- building blocks -----------------------------------------------------------------------------------------------

// NT cooperating threads (a CTA or a warp) walk the edges [s, e) of row `row`, kEdgeUnroll independent edges per thread and step
template <int NT, class EdgeOp>
__device__ __forceinline__ void walk_row(const CsrView &g, int32_t row, int64_t row_start, int64_t s, int64_t e, int tid, int lane,
                                         long long edge_shift, EdgeOp &edge_op)
{
    for (int64_t p0 = s + tid; p0 < e; p0 += (int64_t)NT * kEdgeUnroll)
    {
        int32_t dst[kEdgeUnroll];
#pragma unroll
        for (int k = 0; k < kEdgeUnroll; k++)
        {
            const int64_t p = p0 + (int64_t)k * NT;
            dst[k] = p < e ? g.adj[p] : -1;
        }
#pragma unroll
        for (int k = 0; k < kEdgeUnroll; k++)
        {
            const int64_t p = p0 + (int64_t)k * NT;
            if (p < e) edge_op(row, dst[k], (int)(p - row_start), edge_shift + p, lane);
        }
    }
}

// a hub row: block `chunk` of `chunks` CTAs. With vertex ops the row cannot be split (post must follow ALL edges): chunk 0
// walks the whole row between two CTA barriers. Without, every CTA walks its own kHubChunk edges.
template <class EdgeOp, class PreOp, class PostOp>
__device__ __forceinline__ void advance_hub(const CsrView &g, int32_t row, int chunk, long long edge_shift, EdgeOp &edge_op, PreOp &pre,
                                            PostOp &post)
{
    const int lane = threadIdx.x & 31;
    const int64_t s = g.ptr[row], e = g.ptr[row + 1];
    constexpr bool kSplit = is_no_vertex_op<PreOp>::value && is_no_vertex_op<PostOp>::value;
    if (kSplit)
    {
        const int64_t cs = s + (int64_t)chunk * kHubChunk;
        if (cs < e) walk_row<kAdvThreads>(g, row, s, cs, cs + kHubChunk < e ? cs + kHubChunk : e, threadIdx.x, lane, edge_shift, edge_op);
    }
    else if (chunk == 0)
    {
        const int deg = (int)(e - s);
        if (threadIdx.x == 0) pre(row, deg, lane);
        __syncthreads();
        walk_row<kAdvThreads>(g, row, s, s, e, threadIdx.x, lane, edge_shift, edge_op);
        __syncthreads();
        if (threadIdx.x == 0) post(row, deg, lane);
    }
}

// smallest r in [lo, hi] with ptr[r] >= target (ptr non-decreasing), found by the whole warp 32 probes at a time
__device__ __forceinline__ int32_t warp_lower_bound(const int64_t *__restrict__ ptr, int32_t lo, int32_t hi, int64_t target, int lane)
{
    while (lo < hi)
    {
        // candidates lo .. hi; hi is the answer when every position below it holds a value < target
        const int32_t span = hi - lo;
        const int32_t step = (span + 31) / 32;
        const int64_t pos = (int64_t)lo + (int64_t)lane * step;
        const bool ge = pos < hi ? ptr[pos] >= target : true;
        const unsigned m = __ballot_sync(0xffffffffu, ge);
        if (m == 0u)
        {
            lo = (int32_t)((int64_t)lo + 31LL * step + 1); // all 32 probes (all below hi) are too small
            continue;
        }
        const int k = __ffs(m) - 1; // first probe at or above the target (probes at or past hi count as "above")
        const int64_t found = (int64_t)lo + (int64_t)k * step;
        if (k > 0) lo = (int32_t)(found - step + 1); // the probe before it was too small
        hi = (int32_t)(found < hi ? found : hi);
        if (k == 0) break; // ptr[lo] >= target (or lo == hi)
    }
    return lo;
}

// up to 32 rows (lane k holds row k: id, start, degree; idle lanes degree 0) with < 32 edges each, walked as ONE flat range
template <class EdgeOp>
__device__ __forceinline__ void walk_flat(const CsrView &g, int32_t row, int64_t start, int deg, int lane, long long edge_shift,
                                          EdgeOp &edge_op)
{
    const unsigned FULL = 0xffffffffu;
    int incl = deg;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1)
    {
        const int up = __shfl_up_sync(FULL, incl, o);
        if (lane >= o) incl += up;
    }
    const int excl = incl - deg;
    const int total = __shfl_sync(FULL, incl, 31);
    const int start_lo = (int)(uint32_t)start, start_hi = (int)(start >> 32);
    for (int base = 0; base < total; base += 32 * kEdgeUnroll)
    {
        int32_t src[kEdgeUnroll], dst[kEdgeUnroll], local[kEdgeUnroll];
        int64_t pos[kEdgeUnroll];
#pragma unroll
        for (int k = 0; k < kEdgeUnroll; k++)
        {
            const int idx = base + k * 32 + lane;
            const int probe = idx < total ? idx : total - 1;
            // largest j with excl[j] <= probe (prefix sums are non-decreasing; rows without edges are skipped over)
            int j = 0;
#pragma unroll
            for (int s = 16; s > 0; s >>= 1)
            {
                const int cand = j + s;
                const int o = __shfl_sync(FULL, excl, cand & 31);
                if (cand < 32 && o <= probe) j = cand;
            }
            src[k] = __shfl_sync(FULL, row, j);
            local[k] = probe - __shfl_sync(FULL, excl, j);
            const int lo = __shfl_sync(FULL, start_lo, j), hi = __shfl_sync(FULL, start_hi, j);
            pos[k] = (((int64_t)hi << 32) | (uint32_t)lo) + local[k];
            dst[k] = idx < total ? g.adj[pos[k]] : -1;
        }
#pragma unroll
        for (int k = 0; k < kEdgeUnroll; k++)
            if (base + k * 32 + lane < total) edge_op(src[k], dst[k], local[k], edge_shift + pos[k], lane);
    }
}

// a batch of up to 32 rows owned by one warp (lane k: row k of the batch, `have` = the lane holds a row)
template <class EdgeOp, class PreOp, class PostOp>
__device__ __forceinline__ void advance_batch(const CsrView &g, bool have, int32_t row, int lane, long long edge_shift, EdgeOp &edge_op,
                                              PreOp &pre, PostOp &post)
{
    const unsigned FULL = 0xffffffffu;
    int64_t s = 0;
    int deg = 0;
    if (have)
    {
        s = g.ptr[row];
        deg = (int)(g.ptr[row + 1] - s);
        pre(row, deg, lane);
    }
    __syncwarp();
    // rows with >= 32 edges: the whole warp walks one row at a time (coalesced); the rest of the batch as a flat range
    unsigned long_rows = __ballot_sync(FULL, deg >= 32);
    while (long_rows)
    {
        const int k = __ffs(long_rows) - 1;
        long_rows &= long_rows - 1;
        const int32_t r = __shfl_sync(FULL, row, k);
        const int lo = __shfl_sync(FULL, (int)(uint32_t)s, k), hi = __shfl_sync(FULL, (int)(s >> 32), k);
        const int64_t rs = ((int64_t)hi << 32) | (uint32_t)lo;
        const int d = __shfl_sync(FULL, deg, k);
        walk_row<32>(g, r, rs, rs, rs + d, lane, lane, edge_shift, edge_op);
    }
    const int short_deg = deg < 32 ? deg : 0;
    if (__any_sync(FULL, short_deg > 0)) walk_flat(g, row, s, short_deg, lane, edge_shift, edge_op);
    __syncwarp();
    if (have) post(row, deg, lane);
}

// ---- ALL_ACTIVE advance (advance_worker ALL_ACTIVE branch, multicore/advance_worker.hpp:204-319) --------------------------

struct AllActivePlan
{
    int32_t hub_rows, hub_chunks;  // blocks [0, hub_blocks): hub rows — one CTA per row (vertex ops: hub_chunks = 0) or one per
                                   // kHubChunk edges of the hub region's flat edge range [0, flat_edge0) (hub_chunks CTAs)
    int32_t hub_blocks;
    int32_t flat_blocks;           // then the merge-path region: rows [hub_rows, nz_rows)
    int32_t zero_blocks;           // then rows without edges (vertex ops only)
    int32_t nz_rows;               // rows with at least one edge
    int64_t flat_edge0, flat_edges; // ptr[hub_rows] and the number of edges of the merge-path region (E - flat_edge0)
    int64_t blocks;
};

template <class PreOp, class PostOp>
inline AllActivePlan plan_all_active(const CsrView &g, int64_t edges, int64_t hub_edges)
{
    AllActivePlan P;
    P.hub_rows = g.tier_border[0];
    constexpr bool kNoOps = is_no_vertex_op<PreOp>::value && is_no_vertex_op<PostOp>::value;
    P.hub_chunks = kNoOps ? (int32_t)((hub_edges + kHubChunk - 1) / kHubChunk) : 0;
    P.hub_blocks = kNoOps ? P.hub_chunks : P.hub_rows;
    P.nz_rows = g.tier_border[kNumTiers - 2];
    P.flat_edge0 = hub_edges;
    P.flat_edges = edges - hub_edges;
    const int64_t warps = (P.flat_edges + kWarpEdges - 1) / kWarpEdges;
    P.flat_blocks = (int32_t)((warps + kAdvWarps - 1) / kAdvWarps);
    P.zero_blocks = kNoOps ? 0 : (int32_t)(((int64_t)(g.V - P.nz_rows) + kAdvThreads * 8 - 1) / (kAdvThreads * 8));
    P.blocks = (int64_t)P.hub_blocks + P.flat_blocks + P.zero_blocks;
    return P;
}

// The reference passes a second functor triple for the low-degree ("collective") region (graph_abstractions.h:96-118); its GPU
// backend ignores it (gpu/advance_vect_csr.hpp:56-141 runs edge_op everywhere) and so does this one.
template <class EdgeOp, class PreOp, class PostOp>
__global__ void __launch_bounds__(kAdvThreads)
advance_all_active_kernel(const CsrView g, const AllActivePlan P, long long edge_shift, EdgeOp edge_op, PreOp pre, PostOp post)
{
    const int64_t b = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t hub_blocks = P.hub_blocks;
    if (b < hub_blocks)
    {
        if (P.hub_chunks == 0) advance_hub(g, (int32_t)b, 0, edge_shift, edge_op, pre, post); // vertex ops: the row stays whole
        else
        {
            // no vertex ops: the hub rows' edges are the prefix [0, flat_edge0) of the adjacency array (ids are degree-sorted);
            // CTA b walks edges [b, b + 1) * kHubChunk, which span at most three rows (each has >= 4096 edges)
            const int64_t e0 = b * kHubChunk, e1 = e0 + kHubChunk < P.flat_edge0 ? e0 + kHubChunk : P.flat_edge0;
            int32_t lo = 0, hi = P.hub_rows; // largest row with ptr[row] <= e0
            while (hi - lo > 1)
            {
                const int32_t mid = lo + (hi - lo) / 2;
                if (g.ptr[mid] <= e0) lo = mid;
                else hi = mid;
            }
            for (int32_t row = lo; row < P.hub_rows; row++)
            {
                const int64_t rs = g.ptr[row], re = g.ptr[row + 1];
                if (rs >= e1) break;
                walk_row<kAdvThreads>(g, row, rs, rs > e0 ? rs : e0, re < e1 ? re : e1, threadIdx.x, lane, edge_shift, edge_op);
            }
        }
    }
    else if (b < hub_blocks + P.flat_blocks)
    {
        const int64_t w = (b - hub_blocks) * kAdvWarps + warp;
        const int64_t t0 = P.flat_edge0 + w * kWarpEdges;
        if (t0 >= P.flat_edge0 + P.flat_edges) return;
        // rows whose FIRST edge lies in [t0, t0 + kWarpEdges): complete rows, edges within kWarpEdges + 4096 of each other
        const int32_t r0 = w == 0 ? P.hub_rows : warp_lower_bound(g.ptr, P.hub_rows, P.nz_rows, t0, lane);
        const int32_t r1 = warp_lower_bound(g.ptr, r0, P.nz_rows, t0 + kWarpEdges, lane);
        for (int32_t base = r0; base < r1; base += 32)
        {
            const int32_t row = base + lane;
            advance_batch(g, row < r1, row, lane, edge_shift, edge_op, pre, post);
        }
    }
    else
    {
        const int64_t first = (int64_t)P.nz_rows + (b - hub_blocks - P.flat_blocks) * (kAdvThreads * 8);
#pragma unroll 1
        for (int j = 0; j < 8; j++)
        {
            const int64_t row = first + (int64_t)j * kAdvThreads + threadIdx.x;
            if (row < g.V)
            {
                pre((int32_t)row, 0, lane);
                post((int32_t)row, 0, lane);
            }
        }
    }
}

// ---- SPARSE advance over the ascending id list (advance_worker SPARSE branch, multicore/advance_sparse.hpp:7-249) ----------

struct SparseFrontierView
{
    const int32_t *ids; // ascending = hubs first; [0, n_hub) | [n_hub, n_hub + n_mid) | the rest
    int32_t n_hub, n_mid, n_small;
    int32_t hub_chunks, blocks_mid, blocks_small;
};

template <class PreOp, class PostOp>
inline int64_t plan_sparse(const CsrView &g, SparseFrontierView &F, int max_blocks)
{
    constexpr bool kNoOps = is_no_vertex_op<PreOp>::value && is_no_vertex_op<PostOp>::value;
    F.hub_chunks = kNoOps ? (int32_t)((g.max_degree + kHubChunk - 1) / kHubChunk) : 1;
    if (F.hub_chunks < 1) F.hub_chunks = 1;
    const int64_t bm = ((int64_t)F.n_mid + kAdvWarps - 1) / kAdvWarps, bs = ((int64_t)F.n_small + kAdvThreads - 1) / kAdvThreads;
    F.blocks_mid = (int32_t)(bm < max_blocks ? bm : max_blocks);
    F.blocks_small = (int32_t)(bs < max_blocks ? bs : max_blocks);
    return (int64_t)F.n_hub * F.hub_chunks + F.blocks_mid + F.blocks_small;
}

template <class EdgeOp, class PreOp, class PostOp>
__global__ void __launch_bounds__(kAdvThreads)
advance_sparse_kernel(const CsrView g, const SparseFrontierView F, long long edge_shift, EdgeOp edge_op, PreOp pre, PostOp post)
{
    const int64_t b = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t hub_blocks = (int64_t)F.n_hub * F.hub_chunks;
    if (b < hub_blocks)
    {
        advance_hub(g, F.ids[b / F.hub_chunks], (int)(b % F.hub_chunks), edge_shift, edge_op, pre, post);
    }
    else if (b < hub_blocks + F.blocks_mid)
    {
        const int nwarps = F.blocks_mid * kAdvWarps;
        const int32_t *ids = F.ids + F.n_hub;
        for (int i = (int)(b - hub_blocks) * kAdvWarps + warp; i < F.n_mid; i += nwarps)
        {
            const int32_t row = ids[i];
            const int64_t s = g.ptr[row], e = g.ptr[row + 1];
            if (lane == 0) pre(row, (int)(e - s), lane);
            __syncwarp();
            walk_row<32>(g, row, s, s, e, lane, lane, edge_shift, edge_op);
            __syncwarp();
            if (lane == 0) post(row, (int)(e - s), lane);
        }
    }
    else
    {
        const int nwarps = F.blocks_small * kAdvWarps;
        const int32_t *ids = F.ids + F.n_hub + F.n_mid;
        for (int i0 = ((int)(b - hub_blocks - F.blocks_mid) * kAdvWarps + warp) * 32; i0 < F.n_small; i0 += nwarps * 32)
        {
            const bool have = i0 + lane < F.n_small;
            advance_batch(g, have, have ? ids[i0 + lane] : 0, lane, edge_shift, edge_op, pre, post);
        }
    }
}

// ---- advance over a CSR whose rows are NOT degree-sorted (stand-alone API: the incoming CSR shares the outgoing numbering, so
// ids say nothing about in-degrees): warp batches of 32 rows, optionally restricted to an id list
template <class EdgeOp, class PreOp, class PostOp>
__global__ void __launch_bounds__(kAdvThreads)
advance_unsorted_kernel(const CsrView g, const int32_t *__restrict__ ids, int32_t n, long long edge_shift, EdgeOp edge_op, PreOp pre,
                        PostOp post)
{
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t i0 = warp * 32; i0 < n; i0 += nwarps * 32)
    {
        const bool have = i0 + lane < n;
        const int32_t row = have ? (ids ? ids[i0 + lane] : (int32_t)(i0 + lane)) : 0;
        advance_batch(g, have, row, lane, edge_shift, edge_op, pre, post);
    }
}

// ---- compute (common/compute.hpp:62-85): map over all vertices / over a sparse id list ------------------------------------
template <class ComputeOp>
__global__ void compute_all_active_kernel(const int64_t *__restrict__ ptr, int32_t V, ComputeOp op)
{
    for (int32_t v = blockIdx.x * blockDim.x + threadIdx.x; v < V; v += gridDim.x * blockDim.x)
        op(v, (int)(ptr[v + 1] - ptr[v]), (int)(threadIdx.x & 31));
}

template <class ComputeOp>
__global__ void compute_sparse_kernel(const int64_t *__restrict__ ptr, const int32_t *__restrict__ ids, int32_t n, ComputeOp op)
{
    for (int32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    {
        const int32_t v = ids[i];
        op(v, (int)(ptr[v + 1] - ptr[v]), (int)(threadIdx.x & 31));
    }
}

// ---- generate_new_frontier, flag pass (common/generate_new_frontier.hpp:4-43): bit v = cond(v, deg) as one bitmap word per
// warp via ballot, and — when `flags` is given — the reference frontier's int flags[] (base_frontier.h:17); the compaction
// into the ascending id list is vglb_gnf_from_bitmap behind the C ABI.
template <class Cond>
__global__ void gnf_bitmap_kernel(const int64_t *__restrict__ ptr, int32_t V, uint32_t *__restrict__ bitmap, int32_t *__restrict__ flags,
                                  Cond cond)
{
    const int32_t padded = (V + 31) & ~31;
    for (int32_t v = blockIdx.x * blockDim.x + threadIdx.x; v < padded; v += gridDim.x * blockDim.x)
    {
        const bool in = v < V && cond(v, (int)(ptr[v + 1] - ptr[v])) > 0;
        const uint32_t word = __ballot_sync(0xffffffffu, in);
        if ((threadIdx.x & 31) == 0) bitmap[v >> 5] = word;
        if (flags && v < V) flags[v] = in ? 1 : 0;
    }
}

// ---- reduce (common/reduce.hpp:4-67): block reduction + one atomic per CTA; accumulated in Acc ----------------------------
template <class Acc, class ReduceOp>
__global__ void reduce_sum_kernel(const int64_t *__restrict__ ptr, const int32_t *__restrict__ ids, int32_t n, Acc *out,
                                  ReduceOp op)
{
    __shared__ Acc s_part[32];
    Acc local = 0;
    for (int32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    {
        const int32_t v = ids ? ids[i] : i;
        local += (Acc)op(v, (int)(ptr[v + 1] - ptr[v]), (int)(threadIdx.x & 31));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) local += __shfl_xor_sync(0xffffffffu, local, o);
    if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = local;
    __syncthreads();
    if (threadIdx.x == 0)
    {
        Acc t = 0;
        for (int w = 0; w < (int)(blockDim.x + 31) / 32; w++) t += s_part[w];
        atomicAdd(out, t);
    }
}

template <class ReduceOp>
__global__ void reduce_max_kernel(const int64_t *__restrict__ ptr, const int32_t *__restrict__ ids, int32_t n, int *out,
                                  ReduceOp op)
{
    int local = INT_MIN;
    for (int32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    {
        const int32_t v = ids ? ids[i] : i;
        local = max(local, (int)op(v, (int)(ptr[v + 1] - ptr[v]), (int)(threadIdx.x & 31)));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) local = max(local, __shfl_xor_sync(0xffffffffu, local, o));
    if ((threadIdx.x & 31) == 0) atomicMax(out, local);
}

} // namespace vglb
