// pagerank.cu — PageRank "pull" sweep as a vectorised segmented reduction over the degree-sorted CSR (sm_100a).
//
// Reference semantics = the MULTICORE build (algorithms/pr/pr.hpp:7-148; SURVEY §3.3, App. A.12):
//     r'[u] = k + d * ( sum_{(u->v) in E, v != u} r[v] * inv[v]  +  D ),   inv[v] = 1/indeg_noloops(v) (0 if none)
//     D = sum_{v : indeg_noloops(v) == 0} r[v] / V,   r0 = 1/V,   d = 0.85f,   k = (1-d)/V,   exactly `iters` sweeps.
// The reference does this with four operator calls per sweep (compute save_old_ranks :85-90, reduce dangling :94-103,
// scatter edge_op+post :105-124, reduce ranks_sum :130-135) = 4 V-passes + one E-pass with TWO gathers per edge.
//
// B200 design: no atomics on the rank vector, no host sync inside the loop, a fixed summation order.
//   Round 2 (one GPU, 2-rank partitions): the rows with >= 32 edges go through the COLUMN BINS of pagerank_bins.cu — their edges
//   regrouped by column bin, a bin's slice of the contribution vector in shared memory, 16-bit columns — so a sweep is
//   pr_bin_kernel + pr_cold_bin_kernel + pr_sweep_kernel<false> (the sums of the heavy rows' partial sums, interleaved with
//   the rows with < 32 edges, below) (0.743 -> 0.53 ms per sweep at RMAT-24, DESIGN.md §4.1). On one GPU the rows without
//   out-edges past the bins' columns are only written by the sweep that stores the ranks (PrParams::zero_kept). What follows
//   describes the one-kernel sweep that still runs on partitions of more than 2 ranks (and with VGLB_PR_NO_BINS), and whose
//   tail / zero-row / epilogue code both forms share.
//   ONE kernel per sweep:
//   * contrib[v] = r[v]*inv[v] is produced by the epilogue of the previous sweep, so the E-pass gathers one fp32 per
//     edge (the product is the same fp32 multiply the reference does per edge, pr.hpp:112-115).
//   * What bounds the sweep (profiles/r1_pr_gather_lab*.txt): not HBM but the SM's L1-miss request port — one 128-byte
//     line request per clock per SM, whatever the number of useful bytes. Streaming the adjacency alone runs at
//     6.9 TB/s; the same stream with one random 4-byte gather per edge runs at 0.69 ms per sweep with the request port
//     95 % busy. Two things therefore decide the speed: (1) every SM must keep the request port full — many
//     independent gathers in flight per warp, no dependent pointer chasing per row; (2) nothing but the gather target
//     may live in L1 — shared memory is NOT used for staging (a 16 KB tile buffer per CTA costs 35 %, because the L1
//     that holds the hubs' contributions shrinks), adjacency / inverse degrees / results bypass L1.
//   * Load balance (replaces the ve / vc / collective tiers of multicore/advance_all_active.hpp:7-229). Rows are
//     degree-sorted, so degree classes are contiguous id ranges:
//       degree >= 32 ("heavy", 89 % of the edges of RMAT-24): the row range is cut into warp TASKS of consecutive rows
//         (<= 31 rows, ~2048 edges; rows >= 4096 edges are cut into 4096-edge pieces). A warp streams its task's edge
//         range FLAT — 128 consecutive column indices per step as coalesced int4 loads, two steps (256 gathers) in
//         flight — and assigns the gathered values to rows with a shuffle-based segmented scan keyed by row; lane k
//         owns row k of the task and pulls the row's step total with an indexed shuffle. No shared memory, no atomics,
//         a fixed summation order. Pieces of a long row leave partial sums in a scratch array; the last piece to
//         arrive (one atomic counter per long row) adds them in piece order and runs the row's epilogue.
//       degree 16..31, 8..15, 4..7, 2..3, 1 : 16 / 8 / 4 / 2 / 1 lanes per row (neighbours in id have neighbouring
//         degrees, so the rows of one warp are adjacent in the adjacency array => coalesced), two passes in flight.
//       degree 0 (56 % of the rows): no row pointers, no gathers — only the post-op, coalesced.
//   * Column indices are streamed (ld.global.nc.L1::no_allocate + L2 evict-first); the gathered contribution vector is
//     kept L2-resident (evict-last; 64 MB at scale 24 fits the 126 MB L2) and only ids below PR_COLD_ID allocate in L1.
//   * The epilogue fuses post-op (:118-121), next sweep's contribution, and the NEXT sweep's dangling mass (summed in
//     fp64: block reduction + one atomicAdd(double) per CTA), so `reduce` never returns to the host. On a partitioned
//     graph it also stores the contribution into every peer GPU's copy of the vector (NVLink P2P stores): the
//     allgather of the reference's exchange_vertices_array (mpi_exchange.hpp:155-271) happens inside the sweep.
// Row sums are fp32 trees instead of the reference's sequential fp32 (difference ~1e-7 relative, tolerance 1e-6).
// HBM roofline: algorithmic bytes per sweep = 8E (index + gathered value per edge) + 16V (row pointer, inv read,
// contribution write) [+4V rank write on the last sweep].
#include <limits.h>
#include <math.h>
#include <stdlib.h>

#include <time.h>

#include <algorithm>
#include <vector>

#include <cub/device/device_scan.cuh>

#include "common.cuh"
#include "pagerank.cuh"

// A gather in two halves (pr_zero_scale, pagerank.cuh): the load of contrib[v], or of inv[v] for a column from zero_kept on,
// then the multiply that makes the latter a contribution, applied where the value is summed
__device__ __forceinline__ float pr_gather(const PrParams &P, const L2Pol &pol, int32_t v)
{
    // hubs have the smallest local rows of every rank's slice: column = owner * vp + local row
    const uint32_t local = P.vp_mask ? ((uint32_t)v & P.vp_mask) : (P.vp ? (uint32_t)v % P.vp : (uint32_t)v);
    const float *src = (v >= P.zero_kept ? P.inv : P.contrib_in) + v;
    if (local >= P.cold_local) return ld_gather_cold_f32(src, pol.keep);
    return ld_gather_f32(src, pol.keep);
}
__device__ __forceinline__ float pr_gathered(const PrParams &P, int32_t v, float z0, float x) { return pr_zero_scale(v >= P.zero_kept, z0, x); }

__device__ __forceinline__ void pr_epilogue(const PrParams &P, const L2Pol &pol, int32_t row, float sum, float dang, double &dang_local)
{
    const float inv_r = ld_stream_f32(P.inv + row, pol.stream);
    // k + d * (rank + dangling) — pr.hpp:118-121, no FMA contraction (the x86-64 reference build has none)
    const float rank = __fadd_rn(P.k, __fmul_rn(P.d, __fadd_rn(sum, dang)));
    // a vertex nobody points to (inv == 0: 55-60 % of an RMAT graph) contributes exactly 0 in every sweep: both vectors
    // are zero-filled once and its slot is never written again — neither locally nor into the peers' copies over NVLink
    if (inv_r != 0.0f)
    {
        const float c = __fmul_rn(rank, inv_r);
        st_stream_f32(P.contrib_out + row, c);
        for (int p = 0; p < P.npeers; p++) st_stream_f32(P.peer_out[p] + row, c);
    }
    if (P.rank_out) st_stream_f32(P.rank_out + row, rank);
    if (inv_r == 0.0f) dang_local += (double)__fdiv_rn(rank, P.v_as_float); // pr.hpp:94-101
}

// ---- heavy region: one warp per task ---------------------------------------------------------------------------------

// the four gathers of one lane's int4 at relative position p, split at the row boundary nb
struct Quad
{
    float left, right; // sums of the elements before / at-or-after the boundary
};

__device__ __forceinline__ Quad pr_quad(const PrParams &P, const L2Pol &pol, float z0, const int4 a, int p, int e_lo, int e_hi, int nb, int col_cur)
{
    // element j lives at relative position p + j; valid iff e_lo <= p + j < e_hi; its row's column id is col_cur (+1 past nb)
    const int c[4] = {a.x, a.y, a.z, a.w};
    float x[4];
#pragma unroll
    for (int j = 0; j < 4; j++)
    {
        const int q = p + j;
        const int self = col_cur + (q >= nb ? 1 : 0);
        x[j] = (q >= e_lo && q < e_hi && c[j] != self) ? pr_gather(P, pol, c[j]) : 0.f;
    }
#pragma unroll
    for (int j = 0; j < 4; j++) x[j] = pr_gathered(P, c[j], z0, x[j]);
    Quad r;
    r.left = 0.f;
    r.right = 0.f;
#pragma unroll
    for (int j = 0; j < 4; j++)
    {
        if (p + j < nb) r.left += x[j];
        else r.right += x[j];
    }
    return r;
}

__device__ __forceinline__ void pr_heavy_task(const PrParams &P, const L2Pol &pol, const PrTask T, int lane, float dang, float z0, double &dang_local)
{
    const unsigned FULL = 0xffffffffu;
    const int64_t a4 = T.e0 & ~(int64_t)3;
    const int e_lo = (int)(T.e0 - a4), e_hi = e_lo + T.e_len;
    const int4 *adj4 = reinterpret_cast<const int4 *>(P.adj + a4);
    const int nsteps = (e_hi + 127) >> 7;

    if (T.nrows == 1)
    {
        // one row (or one piece of a long row): plain per-lane accumulation, four steps (512 gathers) in flight
        const int self = P.col_of_row0 + T.row0;
        float acc0 = 0.f, acc1 = 0.f, acc2 = 0.f, acc3 = 0.f;
        for (int s = 0; s < nsteps; s += 4)
        {
            int4 a[4];
#pragma unroll
            for (int u = 0; u < 4; u++)
            {
                const int p = (s + u) * 128 + lane * 4;
                a[u] = p < e_hi ? ld_stream_v4(adj4 + (s + u) * 32 + lane, pol.stream) : make_int4(self, self, self, self);
            }
#pragma unroll
            for (int u = 0; u < 4; u++)
            {
                const int p = (s + u) * 128 + lane * 4;
                const float x0 = (p + 0 >= e_lo && p + 0 < e_hi && a[u].x != self) ? pr_gather(P, pol, a[u].x) : 0.f;
                const float x1 = (p + 1 >= e_lo && p + 1 < e_hi && a[u].y != self) ? pr_gather(P, pol, a[u].y) : 0.f;
                const float x2 = (p + 2 >= e_lo && p + 2 < e_hi && a[u].z != self) ? pr_gather(P, pol, a[u].z) : 0.f;
                const float x3 = (p + 3 >= e_lo && p + 3 < e_hi && a[u].w != self) ? pr_gather(P, pol, a[u].w) : 0.f;
                acc0 += pr_gathered(P, a[u].x, z0, x0);
                acc1 += pr_gathered(P, a[u].y, z0, x1);
                acc2 += pr_gathered(P, a[u].z, z0, x2);
                acc3 += pr_gathered(P, a[u].w, z0, x3);
            }
        }
        const float acc = warp_sum_f32((acc0 + acc1) + (acc2 + acc3));
        if (T.slot < 0)
        {
            if (lane == 0) pr_epilogue(P, pol, T.row0, acc, dang, dang_local);
            return;
        }
        // piece of a long row: leave the partial sum; the last piece to arrive finishes the row
        int last = 0;
        if (lane == 0)
        {
            __stcg(P.piece_partial + T.slot, acc);
            __threadfence();
            last = atomicAdd(P.piece_count + T.row0, 1) == T.npieces - 1;
        }
        last = __shfl_sync(FULL, last, 0);
        if (!last) return;
        __threadfence();
        float t = 0.f;
        for (int i = lane; i < T.npieces; i += 32) t += __ldcg(P.piece_partial + T.slot_first + i);
        t = warp_sum_f32(t);
        if (lane == 0)
        {
            P.piece_count[T.row0] = 0; // ready for the next sweep
            pr_epilogue(P, pol, T.row0, t, dang, dang_local);
        }
        return;
    }

    // 2..31 rows, each >= 32 edges. Lane k <= nrows holds the relative boundary b_k = ptr[row0 + k] - a4.
    int bk = INT_MAX;
    if (lane <= T.nrows) bk = (int)(P.ptr[T.row0 + lane] - a4);
    int bk1 = __shfl_down_sync(FULL, bk, 1);
    if (lane == 31) bk1 = INT_MAX;
    // a lane's first element moves 128 positions per step; rows are >= minlen long, so its row index advances by at
    // most ceil(128 / minlen) per step
    const int minlen = __shfl_sync(FULL, bk, T.nrows) - __shfl_sync(FULL, bk, T.nrows - 1);
    const int rounds = min(4, 127 / max(minlen, 32) + 1);
    float acc = 0.f; // row `lane` of the task
    int cur = 0;     // row (within the task) of this lane's first element of the current step
    for (int s = 0; s < nsteps; s += 2)
    {
        int4 a[2];
        int nb[2], curs[2];
#pragma unroll
        for (int u = 0; u < 2; u++)
        {
            const int p = (s + u) * 128 + lane * 4;
            for (int r = 0; r < rounds; r++)
            {
                const int b = __shfl_sync(FULL, bk, min(cur + 1, 31));
                if (cur < T.nrows && b <= p) cur++;
            }
            curs[u] = cur;
            nb[u] = __shfl_sync(FULL, bk, min(cur + 1, 31));
            if (cur >= T.nrows) nb[u] = INT_MAX;
            a[u] = p < e_hi ? ld_stream_v4(adj4 + (s + u) * 32 + lane, pol.stream) : make_int4(0, 0, 0, 0);
        }
        Quad qd[2];
#pragma unroll
        for (int u = 0; u < 2; u++)
        {
            const int p = (s + u) * 128 + lane * 4;
            qd[u] = pr_quad(P, pol, z0, a[u], p, e_lo, e_hi, nb[u], P.col_of_row0 + T.row0 + curs[u]);
        }
#pragma unroll
        for (int u = 0; u < 2; u++)
        {
            const int sb = (s + u) * 128, p = sb + lane * 4;
            const bool inside = nb[u] <= p + 3; // a row ends inside this lane's four elements
            const int key = curs[u] + (inside ? 1 : 0);
            float y = inside ? qd[u].right : qd[u].left;
            // inclusive segmented scan of y keyed by the row of the lane's last element (keys are non-decreasing)
#pragma unroll
            for (int o = 1; o < 32; o <<= 1)
            {
                const float yu = __shfl_up_sync(FULL, y, o);
                const int ku = __shfl_up_sync(FULL, key, o);
                if (lane >= o && ku == key) y += yu;
            }
            // lane k owns row k: its elements of this step end in lane lb; pull the row's step total
            const int lo = max(bk, sb), hi = min(bk1, sb + 128);
            const bool active = lane < T.nrows && lo < hi;
            const int lb = active ? ((hi - 1 - sb) >> 2) : 0;
            const bool through = bk1 > sb + 4 * lb + 3; // row runs through lane lb's last element (or ends exactly there)
            const int src = through ? lb : max(lb - 1, 0);
            const float yv = __shfl_sync(FULL, y, src);
            const int kv = __shfl_sync(FULL, key, src);
            const float lv = __shfl_sync(FULL, qd[u].left, lb);
            if (active)
            {
                float t = (kv == lane && (through || lb >= 1)) ? yv : 0.f;
                if (!through) t += lv;
                acc += t;
            }
        }
    }
    if (lane < T.nrows) pr_epilogue(P, pol, T.row0 + lane, acc, dang, dang_local);
}

// ---- tail: rows with 1..31 edges, lane per row over the padded column-major copy -----------------------------------
// (the reference's VectorExtension, vgl_datastructures/graphs/undirected_containers/vect_csr/vector_extension/
//  vector_extension.hpp:45-106: segments of 32 consecutive rows, padded to the segment's longest row with the row's own
//  id; rows are degree-sorted, so the padding is a few per cent). No row pointers, no shuffles, every load coalesced and
//  independent; two segments are in flight per warp.
__device__ __forceinline__ void pr_tail_segments(const PrParams &P, const L2Pol &pol, int seg0, int seg1, int lane, float dang, float z0,
                                                 double &dang_local)
{
    for (int seg = seg0; seg < seg1; seg += 2)
    {
        const bool two = seg + 1 < seg1;
        const int64_t b0 = P.ve_ptr[seg], b1 = P.ve_ptr[seg + 1], b2 = two ? P.ve_ptr[seg + 2] : b1;
        const int d0 = (int)((b1 - b0) >> 5), d1 = (int)((b2 - b1) >> 5);
        const int32_t row_a = P.tail_first + seg * 32 + lane, row_b = row_a + 32;
        const int32_t self_a = P.col_of_row0 + row_a, self_b = P.col_of_row0 + row_b;
        const int32_t *pa = P.ve_adj + b0 + lane, *pb = P.ve_adj + b1 + lane;
        float acc_a = 0.f, acc_b = 0.f;
        const int dmax = max(d0, d1);
        // PR_TAIL_J neighbours of each of the two rows per trip: their index loads go out together, then their gathers (a trip
        // is two dependent round trips whatever PR_TAIL_J is)
        for (int j = 0; j < dmax; j += PR_TAIL_J)
        {
            int32_t a[PR_TAIL_J], c[PR_TAIL_J];
#pragma unroll
            for (int u = 0; u < PR_TAIL_J; u++)
            {
                a[u] = j + u < d0 ? ld_stream_s32(pa + (j + u) * 32, pol.stream) : self_a;
                c[u] = j + u < d1 ? ld_stream_s32(pb + (j + u) * 32, pol.stream) : self_b;
            }
            float x[PR_TAIL_J], y[PR_TAIL_J];
#pragma unroll
            for (int u = 0; u < PR_TAIL_J; u++)
            {
                x[u] = a[u] != self_a ? pr_gather(P, pol, a[u]) : 0.f;
                y[u] = c[u] != self_b ? pr_gather(P, pol, c[u]) : 0.f;
            }
#pragma unroll
            for (int u = 0; u < PR_TAIL_J; u += 2)
            {
                acc_a += pr_gathered(P, a[u], z0, x[u]) + pr_gathered(P, a[u + 1], z0, x[u + 1]);
                acc_b += pr_gathered(P, c[u], z0, y[u]) + pr_gathered(P, c[u + 1], z0, y[u + 1]);
            }
        }
        if (row_a < P.zero_first) pr_epilogue(P, pol, row_a, acc_a, dang, dang_local);
        if (two && row_b < P.zero_first) pr_epilogue(P, pol, row_b, acc_b, dang, dang_local);
    }
}

// ---- heavy rows whose edges went through the column bins (pagerank_bins.cu): add up the row's partial sums ---------------------------
// slot[class * nch + chunk]; a row with <= PRB_RC edges is one chunk (chunk = row + xc), the few longer ones have several.
__device__ __forceinline__ void pr_finish_binned(const PrParams &P, const L2Pol &pol, int b, int warp, int lane, float dang, double &dang_local)
{
    if (b < P.bin_long_blocks)
    {
        const int32_t row = b * PR_WARPS + warp; // one warp per long row
        if (row >= P.bin_long_rows) return;
        const int32_t c0 = P.bin_rc_ptr[row], n = (P.bin_rc_ptr[row + 1] - c0) * P.bin_nc;
        float acc = 0.f;
        for (int i = lane; i < n; i += 32)
        {
            const int cls = i % P.bin_nc, ch = c0 + i / P.bin_nc;
            acc += ld_stream_f32(P.bin_slot + (int64_t)cls * P.bin_nch + ch, pol.stream);
        }
        acc = warp_sum_f32(acc);
        if (lane == 0) pr_epilogue(P, pol, row, acc, dang, dang_local);
        return;
    }
    const int32_t row = P.bin_long_rows + (b - P.bin_long_blocks) * PR_THREADS + warp * 32 + lane;
    if (row >= P.bin_rows) return;
    const float *s = P.bin_slot + row + P.bin_xc;
    float acc0 = 0.f, acc1 = 0.f, acc2 = 0.f, acc3 = 0.f;
    for (int c = 0; c < P.bin_nc; c += 12) // 12 independent loads in flight (33 classes: three rounds)
    {
        float x[12];
#pragma unroll
        for (int i = 0; i < 12; i++) x[i] = c + i < P.bin_nc ? ld_stream_f32(s + (int64_t)(c + i) * P.bin_nch, pol.stream) : 0.f;
#pragma unroll
        for (int i = 0; i < 12; i += 4)
        {
            acc0 += x[i];
            acc1 += x[i + 1];
            acc2 += x[i + 2];
            acc3 += x[i + 3];
        }
    }
    pr_epilogue(P, pol, row, (acc0 + acc1) + (acc2 + acc3), dang, dang_local);
}

// next sweep's dangling mass: fp64 block reduction, one atomic per CTA that has any
__device__ __forceinline__ void pr_dangling_reduce(const PrParams &P, double *s_dang, double dang_local, int lane, int warp)
{
    dang_local = warp_sum_f64(dang_local);
    if (lane == 0) s_dang[warp] = dang_local;
    __syncthreads();
    if (threadIdx.x == 0)
    {
        double t = 0.0;
#pragma unroll
        for (int w = 0; w < PR_WARPS; w++) t += s_dang[w];
        if (t != 0.0) atomicAdd(P.dangling_out, t);
    }
}

// rank0 of the previous sweep: the contributions of the rows without out-edges that the gathers compute are rank0_prev * inv
__device__ __forceinline__ float pr_zero_rank_prev(const PrParams &P)
{
    return P.dangling_prev ? pr_zero_rank(P.k, P.d, (float)(*P.dangling_prev)) : P.r0;
}

// HEAVY = false: the graph's heavy rows went through the column bins, and the heavy blocks add up their partial sums
// (pr_finish_binned). That coalesced stream runs next to the latency-bound gathers of the tail rows instead of in a pass of its
// own; the kernel needs fewer registers, and more CTAs fit an SM.
template <bool HEAVY>
__global__ void __launch_bounds__(PR_THREADS, HEAVY ? PR_MIN_CTAS : PR_TAIL_MIN_CTAS) pr_sweep_kernel(const __grid_constant__ PrParams P)
{
    L2Pol pol;
    pol.stream = l2_policy_evict_first();
    pol.keep = l2_policy_evict_last();
    __shared__ double s_dang[PR_WARPS];
    int b = blockIdx.x;
    if (P.interleave)
    {
        // the tail tiers are latency-bound, the heavy region is throughput-bound: mix their blocks so that both kinds
        // are resident on every SM at any time. Block m is a tail block whenever floor((m+1)*ntail/M) advances.
        const long long ntail = (long long)gridDim.x - P.heavy_blocks, M = gridDim.x, m = b;
        const long long tails_before = m * ntail / M, tails_after = (m + 1) * ntail / M;
        b = tails_after > tails_before ? (int)(P.heavy_blocks + tails_before) : (int)(m - tails_before);
    }
    const float dang = (float)(*P.dangling_in);
    double dang_local = 0.0;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

    if (b < P.heavy_blocks)
    {
        if (HEAVY)
        {
            const int t = b * PR_WARPS + warp;
            if (t < P.ntasks) pr_heavy_task(P, pol, P.tasks[t], lane, dang, pr_zero_rank_prev(P), dang_local);
        }
        else
            pr_finish_binned(P, pol, b, warp, lane, dang, dang_local);
    }
    else if (b < P.heavy_blocks + P.tail_blocks)
    {
        const int seg0 = ((b - P.heavy_blocks) * PR_WARPS + warp) * PR_VE_SEGS_PER_WARP;
        pr_tail_segments(P, pol, seg0, min(seg0 + PR_VE_SEGS_PER_WARP, P.ve_segments), lane, dang, pr_zero_rank_prev(P), dang_local);
    }
    else
    {
        // rows without out-edges: only the post-op, coalesced
        const int32_t row0 = P.zero_first + (b - P.heavy_blocks - P.tail_blocks) * PR_ZERO_ROWS_PER_CTA;
        int32_t row1 = min(row0 + PR_ZERO_ROWS_PER_CTA, P.rows);
        if (!P.rank_out) row1 = min(row1, P.zero_kept); // (the one block a sweep of nothing else launches)
        // every such row gets the same rank: one multiply and one store per row
        const float rank0 = pr_zero_rank(P.k, P.d, dang);
        int ndang = 0;
#pragma unroll 4
        for (int32_t row = row0 + threadIdx.x; row < row1; row += PR_THREADS)
        {
            const float inv_r = ld_stream_f32(P.inv + row, pol.stream);
            if (inv_r != 0.0f)
            {
                const float c = __fmul_rn(rank0, inv_r);
                st_stream_f32(P.contrib_out + row, c);
                for (int p = 0; p < P.npeers; p++) st_stream_f32(P.peer_out[p] + row, c);
            }
            else
                ndang++;
            if (P.rank_out) st_stream_f32(P.rank_out + row, rank0);
        }
        // (n equal terms: every partial sum is an exact multiple of a 24-bit value, so n * term is what adding them one by one gives;
        // zero_kept is a block boundary, and the rows from there on are counted once per sweep, below)
        if (row0 < P.zero_kept) dang_local += (double)__fdiv_rn(rank0, P.v_as_float) * (double)ndang;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0)
        dang_local += (double)__fdiv_rn(pr_zero_rank(P.k, P.d, dang), P.v_as_float) * (double)P.zero_dangling;
    pr_dangling_reduce(P, s_dang, dang_local, lane, warp);
}

// the cold bin of the column-binned heavy rows: PR_COLD_SPU steps per warp (columns beyond the shared-memory bins, gathered from global
// memory — in a kernel of its own: it needs the L1 that pr_bin_kernel gives to shared memory, and pr_sweep_kernel must not carry
// its 4 KB of staging: every KB of shared memory there costs L1 hits of the tail rows)
__global__ void __launch_bounds__(PR_THREADS, PR_MIN_CTAS) pr_cold_bin_kernel(const __grid_constant__ PrParams P)
{
    L2Pol pol;
    pol.stream = l2_policy_evict_first();
    pol.keep = l2_policy_evict_last();
    __shared__ float s_stage[PR_WARPS][2 * PRB_STAGE];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int end_step = P.bin_nkchunks * PRB_SPC;
    const int s0 = P.bins.cold_chunk0 * PRB_SPC + (blockIdx.x * PR_WARPS + warp) * PR_COLD_SPU; // units of PR_COLD_SPU steps
    if (s0 < end_step)
        prb_unit<true>(P.bins, pol, NULL, s0, min(s0 + PR_COLD_SPU, end_step), end_step, lane, s_stage[warp], pr_zero_rank_prev(P));
}

// inv[v] = (float)(1.0 / indeg_noloops[v]) or 0 — pr.hpp:66-73 (double division then narrowing, like the reference)
__global__ void pr_inverse_degree_kernel(const int32_t *__restrict__ indeg, int32_t V, float *__restrict__ inv)
{
    int32_t v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v < V)
    {
        const int32_t d = indeg[v];
        inv[v] = d == 0 ? 0.0f : (float)(1.0 / (double)d);
    }
}

// rows [first, V) with inv == 0
__global__ void pr_count_no_inv_kernel(const float *__restrict__ inv, int32_t first, int32_t V, unsigned long long *__restrict__ count)
{
    int n = 0;
    for (int64_t v = first + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < V; v += (int64_t)gridDim.x * blockDim.x) n += inv[v] == 0.0f;
    n = __reduce_add_sync(0xffffffffu, n);
    if ((threadIdx.x & 31) == 0 && n > 0) atomicAdd(count, (unsigned long long)n);
}

// in-degree without self loops by column id, counted over this rank's rows (summed over ranks by the caller)
__global__ void pr_part_indegree_kernel(const int64_t *__restrict__ ptr, const int32_t *__restrict__ adj, int32_t rows,
                                        int32_t col0, int32_t *__restrict__ indeg)
{
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t r = warp; r < rows; r += nwarps)
    {
        const int64_t s = ptr[r], e = ptr[r + 1];
        for (int64_t p = s + (threadIdx.x & 31); p < e; p += 32)
        {
            const int32_t d = adj[p];
            if (d != col0 + (int32_t)r) atomicAdd(&indeg[d], 1);
        }
    }
}

// r0 = 1/V (pr.hpp:40-45): contrib0 = r0*inv, dangling[0] = sum over inv==0 of r0/V
__global__ void pr_init_kernel(const float *__restrict__ inv, int32_t V, float r0, float v_as_float,
                               float *__restrict__ contrib, double *__restrict__ dangling0)
{
    __shared__ double s_dang[PR_WARPS];
    double local = 0.0;
    for (int32_t v = blockIdx.x * blockDim.x + threadIdx.x; v < V; v += gridDim.x * blockDim.x)
    {
        const float i = inv[v];
        contrib[v] = __fmul_rn(r0, i);
        if (i == 0.0f) local += (double)__fdiv_rn(r0, v_as_float);
    }
    local = warp_sum_f64(local);
    if ((threadIdx.x & 31) == 0) s_dang[threadIdx.x >> 5] = local;
    __syncthreads();
    if (threadIdx.x == 0)
    {
        double t = 0.0;
        for (int w = 0; w < PR_WARPS; w++) t += s_dang[w];
        if (t != 0.0) atomicAdd(dangling0, t);
    }
}

// ---- "reference order" dangling mass (vglb_pr_opts.dangling_mode = 1) -----------------------------------------------------
// The reference sums the dangling mass in fp32: reduce<_T>(..., REDUCE_SUM) (pr.hpp:94-103) is an OpenMP
// `parallel for schedule(static) reduction(+)` over the sorted id range (multicore/reduce.hpp:18-31): T static chunks,
// sequential fp32 inside a chunk, partials combined in thread order. With ~V/2 terms of size ~1/V^2 that sum is wrong by far
// more than the 1e-6 parity tolerance (1.6e-5 at scale 16, 2e-3 at scale 22: oracle/vgl_oracle.c, vglo_pagerank_f32_tree_rows),
// so "within 1e-6 of the reference" is only reachable by summing in the same order. One warp per chunk: the lanes load 32
// consecutive values, every lane then replays the 32 sequential fp32 additions through shuffles (adding +0 for vertices
// that are not dangling is exact, as in the reference); a 1-thread kernel combines the T partials in thread order.
__global__ void pr_dangling_reference_chunks_kernel(const float *__restrict__ rank, const float *__restrict__ inv, int32_t V,
                                                    float v_as_float, int threads, float *__restrict__ partial)
{
    const int lane = threadIdx.x & 31;
    const int tid = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (tid >= threads) return;
    const int32_t q = V / threads, t = V % threads; // libgomp static schedule: the first V % T chunks are one longer
    const int32_t len = q + (tid < t ? 1 : 0);
    const int32_t start = tid < t ? tid * (q + 1) : tid * q + t;
    float part = 0.0f;
    for (int32_t base = start; base < start + len; base += 32)
    {
        const int32_t v = base + lane;
        float val = 0.0f;
        if (v < start + len && inv[v] == 0.0f) val = __fdiv_rn(rank[v], v_as_float);
        if (!__any_sync(0xffffffffu, val != 0.0f)) continue;
#pragma unroll
        for (int l = 0; l < 32; l++) part = __fadd_rn(part, __shfl_sync(0xffffffffu, val, l));
    }
    if (lane == 0) partial[tid] = part;
}

__global__ void pr_dangling_reference_combine_kernel(const float *__restrict__ partial, int threads, double *__restrict__ out)
{
    float dangling = 0.0f;
    for (int t = 0; t < threads; t++) dangling = __fadd_rn(dangling, partial[t]);
    *out = (double)dangling;
}

__global__ void pr_fill_kernel(float *a, int32_t n, float val)
{
    int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) a[i] = val;
}

// Warp tasks of the heavy region (rows with degree >= 32), built once per graph on the host from the row pointers of
// that region (a few MB): consecutive rows are packed until ~PR_TASK_EDGES edges or PR_TASK_MAX_ROWS rows; rows with
// >= PR_PIECE_EDGES edges are cut into pieces.
// `h_ptr` = the first heavy_rows + 1 row pointers on the host. vglb_graph_from_csr calls this with the caller's own array while
// the adjacency DMA is in flight (the host is idle then and the table costs 3-4 ms to build); graphs built on the device
// copy the pointers of the heavy region down first (pr_build_tasks).
int vglb_pr_build_tasks_host(vglb_ctx *ctx, vglb_graph *g, const int64_t *ptr, int32_t heavy_rows, int32_t long_rows)
{
    std::vector<PrTask> tasks;
    int32_t slots = 0;
    int32_t r = 0;
    while (r < heavy_rows)
    {
        const int64_t d = ptr[r + 1] - ptr[r];
        if (d >= PR_PIECE_EDGES)
        {
            const int32_t np = (int32_t)((d + PR_PIECE_EDGES - 1) / PR_PIECE_EDGES);
            for (int32_t i = 0; i < np; i++)
            {
                PrTask t;
                t.e0 = ptr[r] + (int64_t)i * PR_PIECE_EDGES;
                t.e_len = (int32_t)((i == np - 1) ? d - (int64_t)i * PR_PIECE_EDGES : PR_PIECE_EDGES);
                t.row0 = r;
                t.nrows = 1;
                t.slot = slots + i;
                t.slot_first = slots;
                t.npieces = np;
                tasks.push_back(t);
            }
            slots += np;
            r++;
            continue;
        }
        PrTask t;
        t.e0 = ptr[r];
        t.row0 = r;
        t.nrows = 0;
        t.slot = -1;
        t.slot_first = 0;
        t.npieces = 0;
        int64_t edges = 0;
        while (r < heavy_rows && t.nrows < PR_TASK_MAX_ROWS)
        {
            const int64_t dr = ptr[r + 1] - ptr[r];
            if (dr >= PR_PIECE_EDGES) break;
            if (t.nrows > 0 && edges + dr > PR_TASK_EDGES + PR_TASK_EDGES / 2) break;
            edges += dr;
            t.nrows++;
            r++;
            if (edges >= PR_TASK_EDGES) break;
        }
        t.e_len = (int32_t)edges;
        tasks.push_back(t);
    }
    g->pr_ntasks = (int32_t)tasks.size();
    if (!tasks.empty())
    {
        CUDA_TRY(vglb_dev_alloc(&g->d_pr_tasks, tasks.size() * sizeof(PrTask)));
        CUDA_TRY(cudaMemcpyAsync(g->d_pr_tasks, tasks.data(), tasks.size() * sizeof(PrTask), cudaMemcpyHostToDevice, ctx->stream));
    }
    CUDA_TRY(vglb_dev_alloc(&g->d_pr_piece_partial, (size_t)(slots > 0 ? slots : 1) * 4));
    const size_t counters = (size_t)(long_rows > 0 ? long_rows : 1);
    CUDA_TRY(vglb_dev_alloc(&g->d_pr_piece_count, counters * 4));
    CUDA_TRY(cudaMemsetAsync(g->d_pr_piece_count, 0, counters * 4, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return VGLB_OK;
}

static int pr_build_tasks(vglb_ctx *ctx, vglb_graph *g)
{
    const int32_t heavy_rows = g->tier_border[1];
    std::vector<int64_t> ptr((size_t)heavy_rows + 1);
    if (heavy_rows > 0)
    {
        CUDA_TRY(cudaMemcpyAsync(ptr.data(), g->d_out_ptr, ((size_t)heavy_rows + 1) * 8, cudaMemcpyDeviceToHost, ctx->stream));
        CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    }
    else
        ptr[0] = 0;
    return vglb_pr_build_tasks_host(ctx, g, ptr.data(), heavy_rows, g->tier_border[0]);
}

// ---- padded column-major copy of the tail rows (built once per graph) -------------------------------------------------
__global__ void pr_ve_seglen_kernel(const int64_t *__restrict__ ptr, int32_t tail_first, int32_t segments, int64_t *__restrict__ seglen)
{
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s < segments)
    {
        const int32_t r = tail_first + s * 32; // the first row of a segment is its longest (rows are degree-sorted)
        seglen[s] = 32 * (ptr[r + 1] - ptr[r]);
    }
    if (s == segments) seglen[s] = 0;
}

__global__ void pr_ve_fill_kernel(const int64_t *__restrict__ ptr, const int32_t *__restrict__ adj, int32_t tail_first,
                                  int32_t zero_first, int32_t col_of_row0, int32_t segments,
                                  const int64_t *__restrict__ ve_ptr, int32_t *__restrict__ ve_adj)
{
    const int lane = threadIdx.x & 31;
    const int seg = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (seg >= segments) return;
    const int32_t row = tail_first + seg * 32 + lane;
    int64_t s = 0;
    int d = 0;
    if (row < zero_first)
    {
        s = ptr[row];
        d = (int)(ptr[row + 1] - s);
    }
    const int64_t base = ve_ptr[seg];
    const int maxd = (int)((ve_ptr[seg + 1] - base) >> 5);
    for (int j = 0; j < maxd; j++) ve_adj[base + j * 32 + lane] = j < d ? adj[s + j] : col_of_row0 + row;
}

static int pr_build_tail_copy(vglb_ctx *ctx, vglb_graph *g)
{
    const int32_t tail_first = g->tier_border[1], zero_first = g->tier_border[VGLB_NUM_TIERS - 2];
    const int32_t segments = (int32_t)ceil_div64(zero_first - tail_first, 32);
    g->pr_ve_segments = segments;
    CUDA_TRY(vglb_dev_alloc(&g->d_pr_ve_ptr, ((size_t)segments + 2) * 8));
    int64_t *d_len = NULL;
    CUDA_TRY(vglb_dev_alloc(&d_len, ((size_t)segments + 2) * 8));
    pr_ve_seglen_kernel<<<(unsigned)ceil_div64(segments + 1, 256), 256, 0, ctx->stream>>>(g->d_out_ptr, tail_first, segments, d_len);
    KERNEL_TRY();
    size_t tmp_bytes = 0;
    void *tmp = NULL;
    CUDA_TRY(cub::DeviceScan::ExclusiveSum(NULL, tmp_bytes, d_len, g->d_pr_ve_ptr, segments + 1, ctx->stream));
    CUDA_TRY(vglb_dev_alloc(&tmp, tmp_bytes ? tmp_bytes : 16));
    CUDA_TRY(cub::DeviceScan::ExclusiveSum(tmp, tmp_bytes, d_len, g->d_pr_ve_ptr, segments + 1, ctx->stream));
    int64_t total = 0;
    CUDA_TRY(cudaMemcpyAsync(&total, g->d_pr_ve_ptr + segments, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    vglb_dev_free(tmp);
    vglb_dev_free(d_len);
    CUDA_TRY(vglb_dev_alloc(&g->d_pr_ve_adj, (size_t)(total > 0 ? total : 1) * 4));
    if (segments > 0)
    {
        pr_ve_fill_kernel<<<(unsigned)ceil_div64((int64_t)segments * 32, 256), 256, 0, ctx->stream>>>(
            g->d_out_ptr, g->d_out_adj, tail_first, zero_first, g->col_of_row0, segments, g->d_pr_ve_ptr, g->d_pr_ve_adj);
        KERNEL_TRY();
    }
    ctx->launches += 2;
    return VGLB_OK;
}

static double pr_now()
{
    struct timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return (double)ts.tv_sec + 1e-9 * (double)ts.tv_nsec;
}

// the column-binned heavy rows (pagerank_bins.cu); VGLB_PR_NO_BINS = developer A/B knob: warp tasks instead
int vglb_pr_bins_wanted(const vglb_graph *g)
{
    // Partitioned graphs: measured with weak scaling, 2 ranks (scale 25) 637 -> 780 GTEPS with the bins, 4 ranks (scale 26)
    // 1108 -> 1034: the bins hold a fixed number of columns, so their share of the gathers falls as the graph grows.
    // (PRB_H = 3 * 2^14 is a multiple of the rank count: a bin starts at owner 0 of a local row)
    if (g->comm && g->part_world > 2) return 0;
    return getenv("VGLB_PR_NO_BINS") == NULL;
}

int vglb_pr_prepare(vglb_ctx *ctx, vglb_graph *g, int iters)
{
    const bool trace = getenv("VGLB_PR_TRACE") != NULL; // developer aid: time of every one-off preparation stage
    double t_last = 0.0;
    auto lap = [&](const char *what) {
        if (!trace) return;
        cudaStreamSynchronize(ctx->stream);
        const double now = pr_now();
        if (t_last > 0.0) fprintf(stderr, "pr prepare: %-28s %.2f ms\n", what, (now - t_last) * 1e3);
        t_last = now;
    };
    lap("start");
    if (!g->d_pr_contrib[0])
    {
        // the gathered vector is indexed by column id: the whole (replicated) vector on a partitioned graph
        CUDA_TRY(vglb_dev_alloc(&g->d_pr_contrib[0], (size_t)g->cols * 4));
        CUDA_TRY(vglb_dev_alloc(&g->d_pr_contrib[1], (size_t)g->cols * 4));
        CUDA_TRY(cudaMemsetAsync(g->d_pr_contrib[0], 0, (size_t)g->cols * 4, ctx->stream));
        CUDA_TRY(cudaMemsetAsync(g->d_pr_contrib[1], 0, (size_t)g->cols * 4, ctx->stream));
    }
    lap("contribution vectors");
    if (!g->d_pr_inv && g->comm) // part uploaded by vglb_graph_from_csr_partitioned: count columns locally, allreduce(sum)
    {
        int32_t *d_indeg = NULL;
        CUDA_TRY(vglb_dev_alloc(&d_indeg, (size_t)g->cols * 4));
        CUDA_TRY(cudaMemsetAsync(d_indeg, 0, (size_t)g->cols * 4, ctx->stream));
        pr_part_indegree_kernel<<<ctx->sm_count * 16, 256, 0, ctx->stream>>>(g->d_out_ptr, g->d_out_adj, g->V, g->col_of_row0, d_indeg);
        KERNEL_TRY();
        int rc = vglb_comm_allreduce_async(g->comm, d_indeg, (size_t)g->cols, VGLB_DT_I32, VGLB_OP_SUM);
        if (rc != VGLB_OK) { vglb_dev_free(d_indeg); return rc; }
        CUDA_TRY(vglb_dev_alloc(&g->d_pr_inv, (size_t)g->vp * 4));
        CUDA_TRY(cudaMemsetAsync(g->d_pr_inv, 0, (size_t)g->vp * 4, ctx->stream));
        if (g->V > 0)
        {
            pr_inverse_degree_kernel<<<(unsigned)ceil_div64(g->V, 256), 256, 0, ctx->stream>>>(d_indeg + g->col_of_row0, g->V, g->d_pr_inv);
            KERNEL_TRY();
        }
        ctx->launches += 2;
        CUDA_TRY(cudaStreamSynchronize(ctx->stream));
        vglb_dev_free(d_indeg);
    }
    if (!g->d_pr_inv) // (the partitioned build fills it from its degree pass)
    {
        int32_t *d_indeg = NULL;
        CUDA_TRY(vglb_dev_alloc(&d_indeg, (size_t)g->V * 4));
        int rc = vglb_graph_indegree_noloops(ctx, g, d_indeg);
        if (rc != VGLB_OK) { vglb_dev_free(d_indeg); return rc; }
        CUDA_TRY(vglb_dev_alloc(&g->d_pr_inv, (size_t)g->V * 4));
        pr_inverse_degree_kernel<<<(unsigned)ceil_div64(g->V, 256), 256, 0, ctx->stream>>>(d_indeg, g->V, g->d_pr_inv);
        KERNEL_TRY();
        ctx->launches++;
        CUDA_TRY(cudaStreamSynchronize(ctx->stream));
        vglb_dev_free(d_indeg);
    }
    lap("inverse in-degrees");
    if (vglb_pr_bins_wanted(g) && !g->pr_bins_tried)
    {
        g->pr_bins_tried = 1;
        int rc = vglb_pr_bins_build(ctx, g);
        if (rc != VGLB_OK && rc != VGLB_ENOMEM) return rc; // (out of memory for the binned copy, +0.9 GB at scale 24: warp tasks instead)
        lap("column bins of the heavy rows");
    }
    if (!g->d_pr_piece_count && !g->pr_bins)
    {
        int rc = pr_build_tasks(ctx, g);
        if (rc != VGLB_OK) return rc;
        lap("warp tasks of the heavy rows");
    }
    if (!g->d_pr_ve_ptr)
    {
        int rc = pr_build_tail_copy(ctx, g);
        if (rc != VGLB_OK) return rc;
        lap("padded copy of the tail rows");
    }
    if (!g->comm)
    {
        // the rows without out-edges whose contributions the sweeps may leave unstored: pr_bin_kernel loads its bins' columns
        // from the stored vector, so they start past those, at a block boundary of the zero-row blocks
        const int32_t zero_first = g->tier_border[VGLB_NUM_TIERS - 2];
        const int64_t smem_cols = g->pr_bins ? std::min<int64_t>((int64_t)((const PrBins *)g->pr_bins)->nb * PRB_H, g->V) : 0;
        const int32_t kept = (int32_t)std::min<int64_t>(
            g->V, zero_first + ceil_div64(std::max<int64_t>(0, smem_cols - zero_first), PR_ZERO_ROWS_PER_CTA) * PR_ZERO_ROWS_PER_CTA);
        if (!g->pr_zero_ready || g->pr_zero_kept != kept)
        {
            unsigned long long *d_n = NULL, n = 0;
            CUDA_TRY(vglb_dev_alloc(&d_n, sizeof(*d_n)));
            CUDA_TRY(cudaMemsetAsync(d_n, 0, sizeof(*d_n), ctx->stream));
            if (kept < g->V)
            {
                pr_count_no_inv_kernel<<<(unsigned)std::min<int64_t>(ctx->sm_count * 8, ceil_div64(g->V - kept, 256)), 256, 0, ctx->stream>>>(
                    g->d_pr_inv, kept, g->V, d_n);
                KERNEL_TRY();
                ctx->launches++;
            }
            CUDA_TRY(cudaMemcpyAsync(&n, d_n, sizeof(n), cudaMemcpyDeviceToHost, ctx->stream));
            CUDA_TRY(cudaStreamSynchronize(ctx->stream));
            vglb_dev_free(d_n);
            g->pr_zero_kept = kept;
            g->pr_zero_dangling = (int32_t)n;
            g->pr_zero_ready = 1;
            lap("rows without out-edges");
        }
    }
    if (g->pr_dangling_slots < iters + 1)
    {
        vglb_dev_free(g->d_pr_dangling);
        g->d_pr_dangling = NULL;
        CUDA_TRY(vglb_dev_alloc(&g->d_pr_dangling, (size_t)(iters + 1) * sizeof(double)));
        g->pr_dangling_slots = iters + 1;
    }
    return VGLB_OK;
}

// grid layout of one sweep over `rows` local rows: heavy blocks first, then the tail tiers
int64_t vglb_pr_plan(const vglb_graph *g, int32_t rows, PrParams *P)
{
    P->ptr = g->d_out_ptr;
    P->adj = g->d_out_adj;
    P->rows = rows;
    P->tasks = (const PrTask *)g->d_pr_tasks;
    P->ntasks = g->pr_ntasks;
    P->piece_partial = g->d_pr_piece_partial;
    P->piece_count = g->d_pr_piece_count;
    P->heavy_blocks = (int32_t)ceil_div64(g->pr_ntasks, PR_WARPS);
    if (const PrBins *B = (const PrBins *)g->pr_bins)
    {
        P->bin_slot = B->d_slot;
        P->bin_rc_ptr = B->d_rc_ptr;
        P->bin_nc = B->nb + 1;
        P->bin_nch = B->nch;
        P->bin_xc = B->xc;
        P->bin_long_rows = B->long_rows;
        P->bin_rows = B->rows;
        P->bin_long_blocks = (int32_t)ceil_div64(B->long_rows, PR_WARPS);
        P->bin_finish_blocks = P->bin_long_blocks + (int32_t)ceil_div64(B->rows - B->long_rows, PR_THREADS);
        P->bin_nkchunks = B->nkchunks;
        vglb_pr_bins_params(g, NULL, &P->bins);
        P->bin_cold_blocks = (int32_t)ceil_div64(ceil_div64((int64_t)(B->nkchunks - B->cold_chunk0) * PRB_SPC, PR_COLD_SPU), PR_WARPS);
        P->ntasks = 0;
        P->heavy_blocks = P->bin_finish_blocks;
    }
    P->ve_adj = g->d_pr_ve_adj;
    P->ve_ptr = g->d_pr_ve_ptr;
    P->ve_segments = g->pr_ve_segments;
    P->tail_first = g->tier_border[1];
    P->zero_first = g->tier_border[VGLB_NUM_TIERS - 2];
    P->tail_blocks = (int32_t)ceil_div64(g->pr_ve_segments, PR_WARPS * PR_VE_SEGS_PER_WARP);
    int64_t nblocks = (int64_t)P->heavy_blocks + P->tail_blocks + ceil_div64(rows - P->zero_first, PR_ZERO_ROWS_PER_CTA);
    // developer knob for timing experiments (results are wrong when set): 1 = heavy region only, 2 = tail tiers only
    if (const char *m = getenv("VGLB_PR_ONLY"))
    {
        if (atoi(m) == 1) nblocks = P->heavy_blocks;
        if (atoi(m) == 2) P->ntasks = 0;
        if (atoi(m) == 3) { P->ntasks = 0; P->ve_segments = 0; }
    }
    P->interleave = 1;
    if (const char *m = getenv("VGLB_PR_INTERLEAVE")) P->interleave = atoi(m);
    if (getenv("VGLB_PR_ONLY")) P->interleave = 0;
    return nblocks;
}

// Shared-memory carve-outs of the sweep's kernels (a function attribute is per device: remembered per context, not per process).
static int pr_set_carveouts(vglb_ctx *ctx)
{
    if (ctx->pr_carveout_set) return VGLB_OK;
    const bool trace = getenv("VGLB_PR_TRACE") != NULL;
    auto occupancy = [&](const char *when) -> int {
        if (!trace) return VGLB_OK;
        int cold = 0, tail = 0;
        CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&cold, pr_cold_bin_kernel, PR_THREADS, 0));
        CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&tail, pr_sweep_kernel<false>, PR_THREADS, 0));
        fprintf(stderr, "pr carve-outs %s: resident CTAs per SM: pr_cold_bin_kernel %d, pr_sweep_kernel<false> %d\n", when, cold, tail);
        return VGLB_OK;
    };
    int rc = occupancy("before");
    if (rc != VGLB_OK) return rc;
    // every KB of L1 holds hub contributions: the sweep kernel asks for the smallest carve-out (64 B static are used). For
    // pr_sweep_kernel<false> it holds 7 CTAs, not the 8 its registers allow: the next larger carve-out, which holds 8, made that
    // pass 15 µs slower at RMAT-24 (DESIGN.md §4.1)
    CUDA_TRY(cudaFuncSetAttribute(pr_sweep_kernel<true>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxL1));
    CUDA_TRY(cudaFuncSetAttribute(pr_sweep_kernel<false>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxL1));
    // the cold bin's gathers hit L1 < 1 % of the time, and it is latency-bound: its carve-out must hold PR_COLD_CTAS CTAs' staging
    // (the smallest carve-out that holds one CTA's 8 KB holds only that one)
    cudaFuncAttributes fa;
    int reserved = 0, per_sm = 0;
    CUDA_TRY(cudaFuncGetAttributes(&fa, pr_cold_bin_kernel));
    CUDA_TRY(cudaDeviceGetAttribute(&reserved, cudaDevAttrReservedSharedMemoryPerBlock, ctx->device));
    CUDA_TRY(cudaDeviceGetAttribute(&per_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, ctx->device));
    const int64_t need = (int64_t)PR_COLD_CTAS * ((int64_t)fa.sharedSizeBytes + reserved);
    const int pct = (int)std::min<int64_t>(100, ceil_div64(100 * need, per_sm));
    CUDA_TRY(cudaFuncSetAttribute(pr_cold_bin_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, pct));
    rc = occupancy("after");
    if (rc != VGLB_OK) return rc;
    ctx->pr_carveout_set = 1;
    return VGLB_OK;
}

int vglb_pr_launch_sweep(vglb_ctx *ctx, const PrParams &P, int64_t nblocks)
{
    if (nblocks <= 0) return VGLB_OK;
    if (!P.bin_slot && P.heavy_blocks > 0) pr_sweep_kernel<true><<<(unsigned)nblocks, PR_THREADS, 0, ctx->stream>>>(P);
    else pr_sweep_kernel<false><<<(unsigned)nblocks, PR_THREADS, 0, ctx->stream>>>(P);
    KERNEL_TRY();
    ctx->launches++;
    return VGLB_OK;
}

extern "C" int vglb_pagerank(vglb_ctx *ctx, vglb_graph *g, int iters, float damping, float *d_ranks, vglb_stats *stats)
{
    return vglb_pagerank_ex(ctx, g, iters, damping, NULL, d_ranks, stats);
}

extern "C" int vglb_pagerank_ex(vglb_ctx *ctx, vglb_graph *g, int iters, float damping, const vglb_pr_opts *opts, float *d_ranks,
                                vglb_stats *stats)
{
    VGLB_REQUIRE(ctx != NULL && g != NULL && d_ranks != NULL, "vglb_pagerank: NULL argument");
    VGLB_REQUIRE(iters >= 0 && iters < (1 << 20), "vglb_pagerank: bad iteration count");
    const bool ref_order = opts && opts->dangling_mode == VGLB_PR_DANGLING_REFERENCE_ORDER;
    const int ref_threads = ref_order ? opts->reference_threads : 0;
    VGLB_REQUIRE(!opts || opts->dangling_mode == VGLB_PR_DANGLING_FP64 || ref_order, "vglb_pagerank_ex: bad dangling_mode");
    VGLB_REQUIRE(!ref_order || (ref_threads >= 1 && ref_threads <= 4096), "vglb_pagerank_ex: reference_threads must be in [1, 4096]");
    VGLB_REQUIRE(!ref_order || !g->comm, "vglb_pagerank_ex: the reference-order dangling sum needs the whole sorted id range (one GPU)");
    CUDA_TRY(cudaSetDevice(ctx->device));
    const int64_t launches0 = ctx->launches;
    int rc = vglb_pr_prepare(ctx, g, iters);
    if (rc != VGLB_OK) return rc;

    // On a partitioned graph (g->comm): V = this rank's rows, the vector is indexed by column id, and after every sweep
    // the owned slices are allgathered (exchange_vertices_array, mpi_exchange.hpp:155-271) and the dangling mass
    // allreduced — both enqueued on the context stream, no host synchronisation inside the loop.
    const int32_t V = g->V;
    vglb_comm *comm = g->comm;
    const int32_t col0 = g->col_of_row0;
    PrParams P;
    memset(&P, 0, sizeof(P));
    const int64_t nblocks = vglb_pr_plan(g, V, &P);
    VGLB_REQUIRE(nblocks < 0x7fffffffLL, "vglb_pagerank: grid too large");
    P.inv = g->d_pr_inv;
    P.col_of_row0 = col0;
    // The rows without out-edges from zero_kept on (PrParams). Every sweep stores them on a partitioned graph (the sweep writes
    // the peers' copies of the vector) and in reference order (its dangling sum reads every rank after each sweep), and with
    // VGLB_PR_STORE_ZERO_ROWS (developer A/B knob).
    const bool store_zero_rows = comm || ref_order || getenv("VGLB_PR_STORE_ZERO_ROWS") != NULL;
    P.zero_kept = store_zero_rows ? INT32_MAX : g->pr_zero_kept;
    P.zero_dangling = store_zero_rows ? 0 : g->pr_zero_dangling;
    P.bins.zero_col = P.zero_kept;
    // a sweep that stores no ranks launches no blocks for them (but one at least where block 0 has their dangling share to add)
    const int64_t nblocks_lean =
        store_zero_rows ? nblocks
                        : std::max<int64_t>(P.zero_dangling > 0 ? 1 : 0,
                                            std::min<int64_t>(nblocks, (int64_t)P.heavy_blocks + P.tail_blocks +
                                                                           ceil_div64(P.zero_kept - P.zero_first, PR_ZERO_ROWS_PER_CTA)));
    P.npeers = 0;
    P.d = damping;
    P.v_as_float = (float)g->V_orig;
    P.k = (float)((1.0 - (double)damping) / (double)P.v_as_float); // pr.hpp:37-38
    if (comm)
    {
        P.vp = (uint32_t)g->vp;
        P.vp_mask = (g->vp & (g->vp - 1)) == 0 ? (uint32_t)g->vp - 1u : 0u;
        P.cold_local = (uint32_t)(PR_COLD_ID / g->part_world);
    }
    else
        P.cold_local = PR_COLD_ID;
    // exchange of the owned slices after a sweep: ncclAllGather, or nothing when the sweep's epilogue already stored
    // them into the peers' vectors (then the dangling-mass allreduce is also the barrier between sweeps: a rank starts
    // sweep i+1 only after every peer finished sweep i, i.e. finished both reading buffer i and writing buffer i+1)
    const bool p2p = comm && g->pr_exchange == VGLB_EXCHANGE_P2P;
    const bool no_exchange = getenv("VGLB_PR_NO_EXCHANGE") != NULL; // developer knob: time one rank's sweeps alone (results are wrong)
    auto exchange = [&](float *vec, double *dangling, bool stored_by_peers) -> int {
        if (!comm || no_exchange) return VGLB_OK;
        if (!stored_by_peers)
        {
            int rc = vglb_comm_allgather_async(comm, vec, (size_t)g->vp * 4);
            if (rc != VGLB_OK) return rc;
        }
        return vglb_comm_allreduce_async(comm, dangling, 1, VGLB_DT_F64, VGLB_OP_SUM);
    };

    float *d_ref_partial = NULL;
    if (ref_order) CUDA_TRY(vglb_dev_alloc(&d_ref_partial, (size_t)ref_threads * sizeof(float)));
    // dangling mass of the rank vector in d_ranks, summed in the reference's order, into dangling slot `slot`
    auto reference_dangling = [&](int slot) -> int {
        pr_dangling_reference_chunks_kernel<<<(unsigned)ceil_div64((int64_t)ref_threads * 32, 256), 256, 0, ctx->stream>>>(
            d_ranks, g->d_pr_inv, V, P.v_as_float, ref_threads, d_ref_partial);
        KERNEL_TRY();
        pr_dangling_reference_combine_kernel<<<1, 1, 0, ctx->stream>>>(d_ref_partial, ref_threads, g->d_pr_dangling + slot);
        KERNEL_TRY();
        ctx->launches += 2;
        return VGLB_OK;
    };

    rc = pr_set_carveouts(ctx);
    if (rc != VGLB_OK) return rc;
    CUDA_TRY(cudaEventRecord(ctx->ev_start, ctx->stream));
    CUDA_TRY(cudaMemsetAsync(g->d_pr_dangling, 0, (size_t)(iters + 1) * sizeof(double), ctx->stream));
    const float r0 = (float)(1.0 / (double)g->V_orig); // pr.hpp:42
    P.r0 = r0;
    if (iters == 0)
    {
        if (V > 0)
        {
            pr_fill_kernel<<<(unsigned)ceil_div64(V, 256), 256, 0, ctx->stream>>>(d_ranks, V, r0);
            KERNEL_TRY();
        }
        ctx->launches++;
    }
    else
    {
        pr_init_kernel<<<ctx->sm_count * 4, PR_THREADS, 0, ctx->stream>>>(g->d_pr_inv, V, r0, P.v_as_float,
                                                                        g->d_pr_contrib[0] + col0, g->d_pr_dangling);
        KERNEL_TRY();
        ctx->launches++;
        rc = exchange(g->d_pr_contrib[0], g->d_pr_dangling, false);
        if (rc != VGLB_OK) return rc;
        if (ref_order && V > 0)
        {
            pr_fill_kernel<<<(unsigned)ceil_div64(V, 256), 256, 0, ctx->stream>>>(d_ranks, V, r0);
            KERNEL_TRY();
            ctx->launches++;
            rc = reference_dangling(0); // replaces the fp64 sum pr_init_kernel left in slot 0
            if (rc != VGLB_OK) return rc;
        }
    }
    for (int it = 0; it < iters; it++)
    {
        P.contrib_in = g->d_pr_contrib[it & 1];
        P.contrib_out = g->d_pr_contrib[(it + 1) & 1] + col0;
        P.rank_out = (it == iters - 1 || ref_order) ? d_ranks : NULL; // reference order: the next dangling sum reads the ranks
        P.dangling_in = g->d_pr_dangling + it;
        P.dangling_prev = it > 0 ? g->d_pr_dangling + it - 1 : NULL;
        P.dangling_out = g->d_pr_dangling + it + 1;
        P.npeers = 0;
        if (p2p && it < iters - 1)
            for (int p = 0; p < g->part_world; p++)
                if (p != g->part_rank) P.peer_out[P.npeers++] = g->d_pr_peer[(it + 1) & 1][p] + col0;
        if (g->pr_bins)
        {
            rc = vglb_pr_bins_launch(ctx, g, P.contrib_in); // partial sums of the heavy rows: the shared-memory bins
            if (rc != VGLB_OK) return rc;
            P.bins.contrib_in = P.contrib_in;
        }
        if (g->pr_bins && P.bin_cold_blocks > 0)
        {
            pr_cold_bin_kernel<<<(unsigned)P.bin_cold_blocks, PR_THREADS, 0, ctx->stream>>>(P); // their cold bin
            KERNEL_TRY();
            ctx->launches++;
        }
        // the heavy rows' sums (all rows without the bins), the rows with < 32 edges and the rows without out-edges
        rc = vglb_pr_launch_sweep(ctx, P, P.rank_out ? nblocks : nblocks_lean);
        if (rc != VGLB_OK) return rc;
        if (ref_order && it < iters - 1)
        {
            rc = reference_dangling(it + 1); // replaces the fp64 sum the sweep's epilogue accumulated
            if (rc != VGLB_OK) return rc;
        }
        if (it < iters - 1 || p2p)
        {
            // (with peer stores the last sweep still ends in the allreduce: no rank may start its NEXT run — which
            // rewrites buffer 0 everywhere — before every peer has finished reading)
            rc = exchange(g->d_pr_contrib[(it + 1) & 1], g->d_pr_dangling + it + 1, p2p);
            if (rc != VGLB_OK) return rc;
        }
    }
    CUDA_TRY(cudaEventRecord(ctx->ev_stop, ctx->stream));
    CUDA_TRY(cudaEventSynchronize(ctx->ev_stop));
    vglb_dev_free(d_ref_partial);
    if (stats)
    {
        float ms = 0.f;
        CUDA_TRY(cudaEventElapsedTime(&ms, ctx->ev_start, ctx->ev_stop));
        memset(stats, 0, sizeof(*stats));
        stats->seconds = ms * 1e-3;
        stats->iterations = iters;
        stats->edges_inspected = (int64_t)iters * g->E;
        stats->vertices_processed = (int64_t)iters * V;
        stats->algorithmic_bytes = (int64_t)iters * (8 * g->E + 16 * (int64_t)V) + (iters > 0 ? 4 * (int64_t)V : 0);
        if (comm) stats->frontier_bytes = (int64_t)iters * g->cols * 4; // bytes of the vector every rank receives + sends
        stats->kernel_launches = ctx->launches - launches0;
    }
    return VGLB_OK;
}

// Peer-store exchange: map every peer's two contribution vectors into this process (CUDA IPC over NVLink peer access).
// The handles travel through the communicator itself (an allgather of 2 x 64 bytes per rank).
extern "C" int vglb_graph_set_exchange(vglb_ctx *ctx, vglb_graph *g, int mode)
{
    VGLB_REQUIRE(ctx != NULL && g != NULL, "vglb_graph_set_exchange: NULL argument");
    VGLB_REQUIRE(mode == VGLB_EXCHANGE_NCCL || mode == VGLB_EXCHANGE_P2P, "vglb_graph_set_exchange: bad mode");
    if (mode == VGLB_EXCHANGE_NCCL || !g->comm || g->part_world == 1)
    {
        g->pr_exchange = VGLB_EXCHANGE_NCCL;
        return VGLB_OK;
    }
    VGLB_REQUIRE(g->part_world <= PR_MAX_PEERS, "vglb_graph_set_exchange: at most 8 ranks for the peer-store exchange");
    CUDA_TRY(cudaSetDevice(ctx->device));
    if (!g->d_pr_peer[0][(g->part_rank + 1) % g->part_world])
    {
        // Every rank goes through both handle exchanges whatever happens locally (a rank whose preparation failed offers
        // no buffer, which makes the exchange fail on every rank instead of leaving the peers inside a collective).
        const int prep = vglb_pr_prepare(ctx, g, 1);
        const int P = g->part_world, rank = g->part_rank;
        void *peers[2][64];
        int rcs[2];
        g->ipc_exported = 1;
        for (int b = 0; b < 2; b++) rcs[b] = vglb_comm_ipc_map(g->comm, prep == VGLB_OK ? (void *)g->d_pr_contrib[b] : NULL, peers[b]);
        if (prep != VGLB_OK || rcs[0] != VGLB_OK || rcs[1] != VGLB_OK)
        {
            for (int b = 0; b < 2; b++)
                for (int p = 0; p < P; p++)
                    if (rcs[b] == VGLB_OK && p != rank && peers[b][p]) cudaIpcCloseMemHandle(peers[b][p]);
            return prep != VGLB_OK ? prep : rcs[0] != VGLB_OK ? rcs[0] : rcs[1];
        }
        for (int b = 0; b < 2; b++)
            for (int p = 0; p < P; p++) g->d_pr_peer[b][p] = p == rank ? NULL : (float *)peers[b][p];
    }
    g->pr_exchange = VGLB_EXCHANGE_P2P;
    return VGLB_OK;
}
