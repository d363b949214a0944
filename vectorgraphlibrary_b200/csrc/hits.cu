// hits.cu — HITS hub and authority scores (algorithms/hits/hits.hpp:5-100) as fused pull passes over both CSR directions.
//
// Step t = 1..steps (Kleinberg's sequential form; every CSR edge counts, duplicates and self loops included):
//     a_raw[v] = sum_{u->v} h_{t-1}[u]   a_t = a_raw / ||a_raw||_2       (pull over the incoming CSR)
//     h_raw[u] = sum_{u->v} a_t[v]       h_t = h_raw / ||h_raw||_2       (pull over the outgoing CSR)
// The vectors stay raw between passes: a pass gathers the previous pass's raw output and multiplies each row sum by that pass's
// inverse norm, which is a word in device memory; the last block of every pass writes it. After the last step one V-pass scales
// both outputs. h_0 is all ones (after the first normalisation the start vector no longer matters). A zero norm gives an inverse
// of 0, so a graph without edges yields all-zero outputs.
//
// One kernel serves both directions (hits_auth_kernel / hits_hub_kernel are the same body under two names, so that profiles tell
// the passes apart). The incoming CSR shares the SCATTER numbering, so its rows are NOT degree-sorted, and the load balance must
// not depend on row order:
//   * Merge path over rows and edges: row r starts at coordinate HITS_ROW_COST * r + ptr[r] and holds HITS_ROW_COST coordinates
//     of its own, then one per edge. The coordinates are cut into windows of HITS_WINDOW; a warp takes the rows that START in its
//     window (a 32-ary search over the start coordinates) and sums them completely. A window therefore holds at most
//     HITS_WINDOW / HITS_ROW_COST rows and its rows at most 2 x HITS_WINDOW edges, whatever the degree distribution and however
//     many rows have no edges. Warps take groups of HITS_GROUP consecutive windows, dealt round-robin, so that every warp gets
//     a share of the hub rows and of the tail.
//   * Within a window, rows are taken 32 at a time (lane = row). Rows with >= 32 edges are summed by the whole warp one after
//     another (HITS_UNROLL coalesced index loads, then as many independent gathers per lane); the shorter rows of the batch are one
//     flat edge range (a shuffle search over the degree prefix sums finds each element's row), summed with a warp segmented scan.
//   * A row with more than HITS_WINDOW edges ("long": RMAT hubs, popular vertices' in-rows) is cut at the window borders into
//     pieces, each summed by the warp of its window. Their partial sums go to a scratch slot per (window, A|B) — A: the piece that
//     starts the window, B: a long row that starts inside it; a window meets at most two long rows — and the last piece to arrive
//     (one counter per row) adds them in piece order.
// Summation order is fixed everywhere: per-lane sums in index order, then shuffle trees. The squared norm is summed in fp64:
// a per-block partial (warps in order), and the last block to finish (ticket counter) adds the partials and then the squares of
// the long rows, in the order of a list built once per call. No float atomics: two calls give the same bits.
// What bounds the pass follows the PageRank sweep's measurements (pagerank.cu header, DESIGN §4.1): the L1-miss request port.
// Indices are streamed (no L1 allocation, L2 evict-first), the gathered vector is kept L2-resident (evict-last), and no shared
// memory is used for staging.
#include <math.h>

#include <algorithm>

#include <cub/device/device_select.cuh>
#include <thrust/iterator/counting_iterator.h>

#include "common.cuh"

#define HITS_THREADS 256
#define HITS_WARPS (HITS_THREADS / 32)
#define HITS_CTAS_PER_SM 4
#define HITS_WINDOW 2048 // edges per warp window; a longer row is cut into pieces
#define HITS_UNROLL 4    // independent gathers per lane and trip
#define HITS_ROW_COST 8  // merge-path coordinates a row takes before its edges (a row costs a row-pointer round trip)
#define HITS_GROUP 8     // consecutive windows a warp takes at a time; groups are dealt to the warps in turn

struct HitsPass
{
    const int64_t *ptr;
    const int32_t *adj;
    int32_t V;
    int64_t E;
    int64_t nwin;            // ceil((HITS_ROW_COST * V + E) / HITS_WINDOW)
    const float *in;         // raw output of the previous pass (gathered)
    const float *inv_in;     // its inverse norm (device word)
    float *out;              // raw output of this pass
    float *inv_out;          // this pass's inverse norm, written by the last block
    float *piece;            // [2 * nwin] partial sums of long-row pieces
    int32_t *piece_count;    // [2 * nwin] arrival counters, indexed by the slot of a long row's first piece
    const int32_t *long_rows; // rows with > HITS_WINDOW edges, ascending
    const int32_t *n_long;
    double *block_sq;        // [gridDim.x] squared-norm partial per block
    unsigned int *ticket;    // blocks done (the last one resets it)
};

struct HitsPol
{
    uint64_t stream, keep;
};

// the whole warp sums edges [s, e) of one row: per-lane sums in index order, then the xor tree
__device__ __forceinline__ float hits_warp_range(const HitsPass &P, const HitsPol &pol, int64_t s, int64_t e, int lane)
{
    float acc[HITS_UNROLL];
#pragma unroll
    for (int u = 0; u < HITS_UNROLL; u++) acc[u] = 0.f;
    for (int64_t p0 = s + lane; p0 < e; p0 += 32 * HITS_UNROLL)
    {
        int32_t c[HITS_UNROLL];
#pragma unroll
        for (int u = 0; u < HITS_UNROLL; u++)
        {
            const int64_t p = p0 + u * 32;
            c[u] = p < e ? ld_stream_s32(P.adj + p, pol.stream) : -1;
        }
#pragma unroll
        for (int u = 0; u < HITS_UNROLL; u++) acc[u] += c[u] >= 0 ? ld_gather_f32(P.in + c[u], pol.keep) : 0.f;
    }
    float t = acc[0];
#pragma unroll
    for (int u = 1; u < HITS_UNROLL; u++) t += acc[u];
    return warp_sum_f32(t);
}

// smallest r in [lo, hi] with HITS_ROW_COST * r + ptr[r] >= target (the coordinate of row r's start), 32 probes at a time
__device__ __forceinline__ int32_t hits_lower_bound(const int64_t *__restrict__ ptr, int32_t lo, int32_t hi, int64_t target, int lane)
{
    while (lo < hi)
    {
        const int32_t step = (hi - lo + 31) / 32;
        const int64_t pos = (int64_t)lo + (int64_t)lane * step;
        const bool ge = pos < hi ? HITS_ROW_COST * pos + ptr[pos] >= target : true;
        const unsigned m = __ballot_sync(0xffffffffu, ge);
        if (m == 0u)
        {
            lo = (int32_t)((int64_t)lo + 31LL * step + 1);
            continue;
        }
        const int k = __ffs(m) - 1;
        const int64_t found = (int64_t)lo + (int64_t)k * step;
        if (k > 0) lo = (int32_t)(found - step + 1);
        hi = (int32_t)(found < hi ? found : hi);
        if (k == 0) break;
    }
    return lo;
}

// The piece of long row `row` (edges [rs, re)) that window w holds, in slot A = 0 or B = 1. Edge p of the row has coordinate
// HITS_ROW_COST * (row + 1) + p. The last piece to arrive adds the pieces in order and stores the row; its square is added by the pass's last
// block (hits_norm).
__device__ __forceinline__ void hits_long_piece(const HitsPass &P, const HitsPol &pol, int32_t row, int64_t rs, int64_t re, int64_t w,
                                                int lane, float inv)
{
    const int64_t own = (int64_t)HITS_ROW_COST * (row + 1);
    const int64_t e_lo = w * HITS_WINDOW - own, e_hi = e_lo + HITS_WINDOW; // the window's edges of this row
    const int64_t ps = rs > e_lo ? rs : e_lo, pe = re < e_hi ? re : e_hi;
    const float sum = hits_warp_range(P, pol, ps, pe, lane);
    const int64_t start = own - HITS_ROW_COST + rs;
    const int64_t a = start / HITS_WINDOW, b = (own + re - 1) / HITS_WINDOW; // windows of the row's start and last edge
    const int64_t first = 2 * a + (start == a * HITS_WINDOW ? 0 : 1);        // slot of the first piece; then 2*(a+1) .. 2*b
    const int npieces = (int)(b - a + 1);
    int last = 0;
    if (lane == 0)
    {
        __stcg(P.piece + (w == a ? first : 2 * w), sum);
        __threadfence();
        last = atomicAdd(P.piece_count + first, 1) == npieces - 1;
    }
    last = __shfl_sync(0xffffffffu, last, 0);
    if (!last) return;
    __threadfence();
    float t = 0.f;
    for (int i = lane; i < npieces; i += 32) t += __ldcg(P.piece + (i == 0 ? first : 2 * (a + i)));
    t = warp_sum_f32(t);
    if (lane == 0)
    {
        P.piece_count[first] = 0; // ready for the next pass
        __stcg(P.out + row, __fmul_rn(t, inv));
    }
}

// Rows [r0, r1) of window w (their start coordinates lie in it), 32 at a time; returns this lane's share of the squared norm
__device__ __forceinline__ double hits_window_rows(const HitsPass &P, const HitsPol &pol, int64_t w, int32_t r0, int32_t r1, int lane,
                                                   float inv)
{
    const unsigned FULL = 0xffffffffu;
    double sq = 0.0;
    for (int32_t base = r0; base < r1; base += 32)
    {
        const int32_t row = base + lane;
        const bool have = row < r1;
        int64_t s = 0, e = 0;
        if (have)
        {
            s = P.ptr[row];
            e = P.ptr[row + 1];
        }
        const int64_t deg = e - s;
        float sum = 0.f;
        // rows with 32 .. HITS_WINDOW edges: the whole warp, one row after the other
        unsigned wide = __ballot_sync(FULL, deg >= 32 && deg <= HITS_WINDOW);
        while (wide)
        {
            const int k = __ffs(wide) - 1;
            wide &= wide - 1;
            const int64_t ks = __shfl_sync(FULL, s, k), ke = __shfl_sync(FULL, e, k);
            const float t = hits_warp_range(P, pol, ks, ke, lane);
            if (lane == k) sum = t;
        }
        // at most one long row starts in a window (it runs past the window's end)
        const unsigned lng = __ballot_sync(FULL, deg > HITS_WINDOW);
        if (lng)
        {
            const int k = __ffs(lng) - 1;
            hits_long_piece(P, pol, base + k, __shfl_sync(FULL, s, k), __shfl_sync(FULL, e, k), w, lane, inv);
        }
        // rows with < 32 edges: one flat range; lane j's row holds flat elements [excl, incl)
        const int d = deg < 32 ? (int)deg : 0;
        int incl = d;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1)
        {
            const int up = __shfl_up_sync(FULL, incl, o);
            if (lane >= o) incl += up;
        }
        const int excl = incl - d;
        const int total = __shfl_sync(FULL, incl, 31);
        const int64_t s0 = __shfl_sync(FULL, s, 0);
        const int off = (int)(s - s0) - excl; // adjacency position of flat element i of this lane's row: s0 + off + i
        for (int fb = 0; fb < total; fb += 32 * HITS_UNROLL)
        {
            int key[HITS_UNROLL];
            float x[HITS_UNROLL];
            int32_t c[HITS_UNROLL];
#pragma unroll
            for (int u = 0; u < HITS_UNROLL; u++)
            {
                const int idx = fb + u * 32 + lane;
                const int probe = idx < total ? idx : total - 1;
                int j = 0; // largest j with excl[j] <= probe (rows without flat edges are stepped over)
#pragma unroll
                for (int st = 16; st > 0; st >>= 1)
                {
                    const int cand = j + st;
                    const int o = __shfl_sync(FULL, excl, cand & 31);
                    if (cand < 32 && o <= probe) j = cand;
                }
                const int oj = __shfl_sync(FULL, off, j);
                key[u] = idx < total ? j : 32;
                c[u] = idx < total ? ld_stream_s32(P.adj + s0 + oj + probe, pol.stream) : -1;
            }
#pragma unroll
            for (int u = 0; u < HITS_UNROLL; u++) x[u] = c[u] >= 0 ? ld_gather_f32(P.in + c[u], pol.keep) : 0.f;
#pragma unroll
            for (int u = 0; u < HITS_UNROLL; u++)
            {
                // inclusive segmented scan keyed by row (keys are non-decreasing over the lanes)
                float y = x[u];
#pragma unroll
                for (int o = 1; o < 32; o <<= 1)
                {
                    const float yu = __shfl_up_sync(FULL, y, o);
                    const int ku = __shfl_up_sync(FULL, key[u], o);
                    if (lane >= o && ku == key[u]) y += yu;
                }
                // lane j's row ends its part of this round in lane hi - 1 - rb
                const int rb = fb + u * 32;
                const int lo = excl > rb ? excl : rb, hi = incl < rb + 32 ? incl : rb + 32;
                const bool mine = lo < hi;
                const float t = __shfl_sync(FULL, y, mine ? hi - 1 - rb : 0);
                if (mine) sum += t;
            }
        }
        if (have && deg <= HITS_WINDOW)
        {
            const float v = __fmul_rn(sum, inv);
            st_stream_f32(P.out + row, v);
            sq += (double)v * (double)v;
        }
    }
    return sq;
}

// The pass's last block: squared norm = block partials in block order, then the long rows' squares in list order
__device__ __forceinline__ void hits_norm(const HitsPass &P, double *s_red)
{
    double t = 0.0;
    for (int i = threadIdx.x; i < (int)gridDim.x; i += HITS_THREADS) t += __ldcg(P.block_sq + i);
    const int n_long = *P.n_long;
    for (int i = threadIdx.x; i < n_long; i += HITS_THREADS)
    {
        const double v = (double)__ldcg(P.out + P.long_rows[i]);
        t += v * v;
    }
    t = warp_sum_f64(t);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = t;
    __syncthreads();
    if (threadIdx.x == 0)
    {
        double sq = 0.0;
#pragma unroll
        for (int w = 0; w < HITS_WARPS; w++) sq += s_red[w];
        *P.inv_out = sq > 0.0 ? (float)(1.0 / sqrt(sq)) : 0.f;
        *P.ticket = 0; // ready for the next pass
    }
}

__device__ __forceinline__ void hits_pass(const HitsPass &P)
{
    HitsPol pol;
    pol.stream = l2_policy_evict_first();
    pol.keep = l2_policy_evict_last();
    __shared__ double s_red[HITS_WARPS];
    __shared__ int s_last;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const float inv = *P.inv_in;
    const int64_t nw = (int64_t)gridDim.x * HITS_WARPS, gw = (int64_t)blockIdx.x * HITS_WARPS + warp;
    double sq = 0.0;
    for (int64_t w0 = gw * HITS_GROUP; w0 < P.nwin; w0 += nw * HITS_GROUP)
    {
        const int64_t w1 = w0 + HITS_GROUP < P.nwin ? w0 + HITS_GROUP : P.nwin;
        int32_t r0 = hits_lower_bound(P.ptr, 0, P.V, w0 * HITS_WINDOW, lane);
        for (int64_t w = w0; w < w1; w++)
        {
            const int64_t ws = w * HITS_WINDOW;
            // at most HITS_WINDOW / HITS_ROW_COST rows start in a window
            const int32_t near = r0 + HITS_WINDOW / HITS_ROW_COST < P.V ? r0 + HITS_WINDOW / HITS_ROW_COST : P.V;
            const int32_t r1 = hits_lower_bound(P.ptr, r0, near, ws + HITS_WINDOW, lane);
            // a long row that started in an earlier window and runs into this one (it holds coordinate ws)
            if (r0 > 0 && (int64_t)HITS_ROW_COST * r0 + P.ptr[r0] > ws)
            {
                const int64_t rs = P.ptr[r0 - 1], re = P.ptr[r0];
                if (re - rs > HITS_WINDOW) hits_long_piece(P, pol, r0 - 1, rs, re, w, lane, inv);
            }
            sq += hits_window_rows(P, pol, w, r0, r1, lane, inv);
            r0 = r1;
        }
    }
    // block partial (warps in order), then the ticket; the last block finishes the norm
    sq = warp_sum_f64(sq);
    if (lane == 0) s_red[warp] = sq;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0)
    {
        double b = 0.0;
#pragma unroll
        for (int i = 0; i < HITS_WARPS; i++) b += s_red[i];
        __stcg(P.block_sq + blockIdx.x, b);
        __threadfence();
        s_last = atomicAdd(P.ticket, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (s_last)
    {
        __threadfence();
        hits_norm(P, s_red);
    }
}

__global__ void __launch_bounds__(HITS_THREADS, HITS_CTAS_PER_SM) hits_auth_kernel(const __grid_constant__ HitsPass P) { hits_pass(P); }
__global__ void __launch_bounds__(HITS_THREADS, HITS_CTAS_PER_SM) hits_hub_kernel(const __grid_constant__ HitsPass P) { hits_pass(P); }

// h_0 = 1 everywhere, and its "inverse norm" 1
__global__ void hits_init_kernel(float *hub, int32_t V, float *inv_h)
{
    for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < V; v += (int64_t)gridDim.x * blockDim.x) hub[v] = 1.0f;
    if (blockIdx.x == 0 && threadIdx.x == 0) *inv_h = 1.0f;
}

// the outputs: a = a_raw * inv_a, h = h_raw * inv_h
__global__ void hits_scale_kernel(float *auth, float *hub, int32_t V, const float *inv_a, const float *inv_h)
{
    const float ia = *inv_a, ih = *inv_h;
    for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < V; v += (int64_t)gridDim.x * blockDim.x)
    {
        auth[v] = __fmul_rn(auth[v], ia);
        hub[v] = __fmul_rn(hub[v], ih);
    }
}

struct HitsIsLong
{
    const int64_t *ptr;
    __host__ __device__ bool operator()(int32_t r) const { return ptr[r + 1] - ptr[r] > HITS_WINDOW; }
};

extern "C" int vglb_hits(vglb_ctx *ctx, vglb_graph *g, int steps, float *d_auth, float *d_hub, vglb_stats *stats)
{
    VGLB_REQUIRE(ctx != NULL && g != NULL && d_auth != NULL && d_hub != NULL, "vglb_hits: NULL argument");
    VGLB_REQUIRE(steps >= 1 && steps < (1 << 20), "vglb_hits: steps must be in [1, 2^20)");
    VGLB_REQUIRE(g->comm == NULL, "vglb_hits: partitioned graphs are not supported");
    CUDA_TRY(cudaSetDevice(ctx->device));
    if (!g->d_in_ptr) VGLB_TRY(vglb_graph_derive_incoming(ctx, g)); // as vglb_bfs: kept with the graph
    const int32_t V = g->V;
    const int64_t E = g->E;
    const int64_t nwin = ceil_div64((int64_t)HITS_ROW_COST * V + E, HITS_WINDOW);
    const int64_t max_long = E / HITS_WINDOW + 1;
    const int grid = (int)std::min<int64_t>((int64_t)ctx->sm_count * HITS_CTAS_PER_SM, ceil_div64(nwin, HITS_WARPS * HITS_GROUP));
    cudaStream_t st = ctx->stream;
    const int64_t launches0 = ctx->launches;

    // per-call scratch from the context's cache: piece partials, piece counters, block partials, the state words
    // (ticket, inv_a, inv_h, two long-row counts) and the two long-row lists
    dev_ptr<float> piece;
    dev_ptr<int32_t> piece_count, long_rows;
    dev_ptr<double> block_sq;
    dev_ptr<unsigned int> state;
    dev_ptr<void> tmp;
    CUDA_TRY(vglb_dev_alloc(piece, (size_t)2 * nwin * sizeof(float)));
    CUDA_TRY(vglb_dev_alloc(piece_count, (size_t)2 * nwin * sizeof(int32_t)));
    CUDA_TRY(vglb_dev_alloc(block_sq, (size_t)grid * sizeof(double)));
    CUDA_TRY(vglb_dev_alloc(state, 8 * sizeof(unsigned int)));
    CUDA_TRY(vglb_dev_alloc(long_rows, (size_t)2 * max_long * sizeof(int32_t)));
    unsigned int *ticket = state.get();
    float *inv_a = (float *)(state.get() + 1), *inv_h = (float *)(state.get() + 2);
    int32_t *n_long = (int32_t *)(state.get() + 3); // [0] incoming, [1] outgoing

    CUDA_TRY(cudaEventRecord(ctx->ev_start, st));
    CUDA_TRY(cudaMemsetAsync(piece_count.get(), 0, (size_t)2 * nwin * sizeof(int32_t), st));
    CUDA_TRY(cudaMemsetAsync(state.get(), 0, 8 * sizeof(unsigned int), st));
    const int64_t *ptrs[2] = {g->d_in_ptr, g->d_out_ptr};
    for (int dir = 0; dir < 2; dir++)
    {
        int32_t *list = long_rows.get() + dir * max_long;
        const HitsIsLong pred{ptrs[dir]};
        CUDA_TRY(vglb_cub(tmp, [&](void *t, size_t &bytes) {
            return cub::DeviceSelect::If(t, bytes, thrust::counting_iterator<int32_t>(0), list, n_long + dir, V, pred, st);
        }));
        ctx->launches++;
    }
    const int fill_blocks = (int)std::min<int64_t>((int64_t)ctx->sm_count * 8, ceil_div64(V > 0 ? V : 1, 256));
    hits_init_kernel<<<fill_blocks, 256, 0, st>>>(d_hub, V, inv_h);
    KERNEL_TRY();
    ctx->launches++;

    HitsPass A;
    A.ptr = g->d_in_ptr;
    A.adj = g->d_in_adj;
    A.V = V;
    A.E = E;
    A.nwin = nwin;
    A.in = d_hub;
    A.inv_in = inv_h;
    A.out = d_auth;
    A.inv_out = inv_a;
    A.piece = piece.get();
    A.piece_count = piece_count.get();
    A.long_rows = long_rows.get();
    A.n_long = n_long;
    A.block_sq = block_sq.get();
    A.ticket = ticket;
    HitsPass H = A;
    H.ptr = g->d_out_ptr;
    H.adj = g->d_out_adj;
    H.in = d_auth;
    H.inv_in = inv_a;
    H.out = d_hub;
    H.inv_out = inv_h;
    H.long_rows = long_rows.get() + max_long;
    H.n_long = n_long + 1;
    for (int t = 0; t < steps; t++)
    {
        hits_auth_kernel<<<grid, HITS_THREADS, 0, st>>>(A);
        KERNEL_TRY();
        hits_hub_kernel<<<grid, HITS_THREADS, 0, st>>>(H);
        KERNEL_TRY();
        ctx->launches += 2;
    }
    hits_scale_kernel<<<fill_blocks, 256, 0, st>>>(d_auth, d_hub, V, inv_a, inv_h);
    KERNEL_TRY();
    ctx->launches++;
    const int rc = vglb_finish_run(ctx, launches0, stats);
    if (rc != VGLB_OK || !stats) return rc;
    stats->iterations = steps;
    stats->edges_inspected = 2 * E * steps;
    stats->vertices_processed = 2LL * V * steps;
    // the formula of include/vgl_b200.h (vglb_hits)
    stats->algorithmic_bytes = 2LL * steps * (8 * E + 12LL * V) + 16LL * V;
    return VGLB_OK;
}
