// pagerank.cuh — internal interface of the PageRank sweep (pagerank.cu), shared with the partitioned driver
// (partition.cu). Not part of the C ABI.
#pragma once
#include "common.cuh"

#define PR_THREADS 256
#define PR_WARPS (PR_THREADS / 32)
#define PR_TASK_MAX_ROWS 31       // lanes 0..nrows hold the task's row boundaries
#define PR_MAX_PEERS 8
// tunables (profiles/r1_pr_ab.txt has the A/B runs); -D overrides are for developer A/B builds only
#ifndef PR_COLD_ID
#define PR_COLD_ID 49152          // ids at or above this are gathered without allocating in L1
#endif
#ifndef PR_TASK_EDGES
#define PR_TASK_EDGES 4096        // target edges per warp task
#endif
#ifndef PR_PIECE_EDGES
#define PR_PIECE_EDGES 8192       // rows with at least this many edges are cut into pieces of this size
#endif
#ifndef PR_MIN_CTAS
#define PR_MIN_CTAS 5             // __launch_bounds__ minimum resident CTAs per SM (48 registers)
#endif
#ifndef PR_TAIL_MIN_CTAS
#define PR_TAIL_MIN_CTAS 8        // the same for pr_sweep_kernel<false>, whose heavy blocks only add up partial sums (32 registers)
#endif
#ifndef PR_VE_SEGS_PER_WARP
#define PR_VE_SEGS_PER_WARP 8     // 32-row segments of the padded tail copy handled by one warp (r2 A/B with the column bins: 16 -> 0.611, 8 -> 0.527 ms)
#endif
#ifndef PR_TAIL_J
#define PR_TAIL_J 2               // neighbours of a tail row fetched per trip of its loop (even)
#endif
#ifndef PR_COLD_SPU
#define PR_COLD_SPU 8            // steps of the cold bin handled by one warp of pr_cold_bin_kernel (A/B at RMAT-24, ms per sweep: 1 -> 0.618, 2 -> 0.578, 4 -> 0.548, 8 -> 0.531, 16 -> 0.543, 32 -> 0.576)
#endif
#ifndef PR_COLD_CTAS
#define PR_COLD_CTAS 5            // resident CTAs of pr_cold_bin_kernel per SM that its shared-memory carve-out must hold (8 KB of staging each; A/B at RMAT-24, cold pass µs / ms per sweep: 1 -> 122.4 / 0.539, 3 -> 115.5 / 0.532, 5 -> 97.3 / 0.513; 2 is no carve-out of its own: the one that holds 2 holds 3)
#endif
#ifndef PR_ZERO_ROWS_PER_CTA
#define PR_ZERO_ROWS_PER_CTA 4096 // rows without out-edges handled by one CTA
#endif

// a warp's unit of work in the heavy region (rows with degree >= 32)
struct PrTask
{
    int64_t e0;         // first edge position
    int32_t e_len;      // number of edges
    int32_t row0;       // first row
    int32_t nrows;      // 1..31 complete rows, or 1 for a piece of a long row
    int32_t slot;       // -1: complete rows; else this piece's slot in the partial-sum array
    int32_t slot_first; // first slot of the long row
    int32_t npieces;    // pieces of the long row
};

struct vglb_ctx;
struct vglb_graph;
// ---- column-binned heavy rows (pagerank_bins.cu) --------------------------------------------------------------------------
#define PRB_H 49152     // columns per bin: its slice of the contribution vector fills 192 KB of shared memory
#define PRB_RC 4096     // a row's edges are cut into chunks of this many before binning: no (bin,row) run is longer
#define PRB_BINS 32     // shared-memory bins used (columns beyond them form the cold bin)

struct PrBins
{
    int32_t nb;          // shared-memory bins (classes 0..nb-1); class nb = the cold bin
    int32_t rows;        // binned rows = rows with >= 32 edges (ids 0..rows-1)
    int32_t long_rows;   // rows with more than one row chunk (ids 0..long_rows-1)
    int32_t nch;         // row chunks; row r >= long_rows is chunk r + xc
    int32_t xc;
    int32_t nkchunks;    // 4096-slot chunks of the binned copy
    int32_t cold_chunk0; // first chunk of the cold bin
    int64_t slots;
    int32_t nruns;
    int grid;            // persistent CTAs (one per SM)
    uint16_t *d_wcol;    // column - bin * PRB_H of every slot of the shared-memory bins (PRB_H = padding)
    int32_t *d_cold;     // column of every slot of the cold bin (-1 = padding)
    uint32_t *d_meta;    // per lane and step: static part of the segmented sum
    int32_t *d_step_run0;
    int32_t *d_run_slot;
    int32_t *d_bin_chunk0, *d_cta_chunk0;
    int32_t *d_warp_step0; // first step of every warp's piece of every (CTA, bin) (prb_warp_ranges_kernel)
    float *d_slot;       // [class][row chunk] partial sums, + 1 dummy
    int32_t *d_rc_ptr;   // first chunk of rows 0..long_rows
};

struct PrbBinParams
{
    const uint16_t *wcol;
    const int32_t *cold;
    const uint32_t *meta;
    const int32_t *step_run0, *run_slot, *bin_chunk0, *cta_chunk0, *warp_step0;
    const float *contrib_in;
    const float *inv;
    float *slot;
    int32_t nb, cold_chunk0, nruns;
    int32_t zero_col;  // the cold bin's PrParams::zero_kept (INT32_MAX in pr_bin_kernel)
    int64_t cols;      // columns of the gathered vector (sorted ids 0 .. cols-1)
    int32_t world, vp; // partitioned graph: column = owner * vp + local row, sorted id = local row * world + owner
};

int vglb_pr_bins_build(vglb_ctx *ctx, vglb_graph *g);
void vglb_pr_bins_free(vglb_graph *g);
int vglb_pr_bins_launch(vglb_ctx *ctx, vglb_graph *g, const float *contrib_in);
void vglb_pr_bins_params(const vglb_graph *g, const float *contrib_in, PrbBinParams *P);

struct PrParams
{
    const int64_t *ptr;
    const int32_t *adj;
    const float *contrib_in;       // indexed by column id (whole vector)
    const float *inv;              // indexed by local row
    float *contrib_out;            // indexed by local row (this rank's slice of the next vector)
    float *peer_out[PR_MAX_PEERS]; // the same slice inside the peers' copies of the next vector (partitioned graphs)
    float *rank_out;               // written on the final sweep only (may be NULL otherwise), indexed by local row
    const double *dangling_in;
    double *dangling_out;
    const PrTask *tasks;
    float *piece_partial;
    int32_t *piece_count;          // one arrival counter per long row (row < tier_border[0])
    int32_t ntasks;
    int32_t heavy_blocks;          // blocks [0, heavy_blocks) run warp tasks, or with the column bins finish the heavy rows
    int32_t rows;                  // local rows
    int32_t col_of_row0;           // column id of local row 0 (0 on one GPU); row r is column col_of_row0 + r
    int32_t npeers;
    uint32_t cold_local;           // gathers of local rows at or above this bypass L1 (PR_COLD_ID / ranks)
    float k, d, v_as_float;
    uint32_t vp, vp_mask;          // partitioned graphs: rows per rank (slice stride) and vp - 1 when vp is a power of two
    // tail: rows [tail_first, zero_first) have degree 1..31 and are read from the padded column-major copy
    const int32_t *ve_adj;         // segment s: ve_adj[ve_ptr[s] + j*32 + lane] = j-th neighbour of row tail_first + 32 s + lane
    const int64_t *ve_ptr;         // ve_segments + 1 offsets
    int32_t ve_segments;
    int32_t tail_first, zero_first;
    int32_t tail_blocks;           // blocks [heavy_blocks, heavy_blocks + tail_blocks) run tail segments, the rest zero rows
    // Rows without out-edges all get the same rank, rank0 = k + d * (0 + dangling). From zero_kept on (one GPU) their
    // contributions are stored only by sweeps that store the ranks: the other sweeps launch no blocks for them, a gather of
    // such a column computes rank0_prev * inv[v] (pr_zero_scale), and their share of the next dangling mass is
    // zero_dangling (their rows with inv == 0) equal terms. zero_kept is INT32_MAX where every sweep stores them.
    int32_t zero_kept;
    int32_t zero_dangling;
    const double *dangling_prev;   // the previous sweep's dangling_in, from which its rank0 follows (NULL on sweep 0)
    float r0;                      // the rank pr_init_kernel's contributions are made of (sweep 0's rank0_prev)
    // binned heavy rows (pagerank_bins.cu): pr_bin_kernel + pr_cold_bin_kernel leave partial sums, and the heavy blocks of
    // pr_sweep_kernel<false> add up every heavy row's and run its epilogue (pr_finish_binned)
    const float *bin_slot;         // NULL: the heavy blocks run warp tasks
    const int32_t *bin_rc_ptr;
    int32_t bin_nc, bin_nch, bin_xc, bin_long_rows, bin_rows;
    int32_t bin_long_blocks;       // heavy blocks [0, bin_long_blocks): one warp per long row; then one lane per row
    int32_t bin_finish_blocks;
    int32_t bin_cold_blocks;       // pr_cold_bin_kernel: one chunk of the cold bin per warp
    int32_t bin_nkchunks;          // all chunks of the binned copy; the cold bin's are bins.cold_chunk0 .. bin_nkchunks - 1
    PrbBinParams bins;
};

struct L2Pol
{
    uint64_t stream, keep;
};

#ifdef __CUDACC__
// ---- one chunk of the binned copy (shared by pr_bin_kernel: shared-memory bins, and pr_sweep_kernel: the cold bin) -------------
#define PRB_STEP 512                    // slots per warp step (16 consecutive slots per lane)
#define PRB_CHUNK 4096                  // slots per chunk
#define PRB_SPC (PRB_CHUNK / PRB_STEP)  // steps per chunk
#define PRB_ALIGN 4                     // runs start at multiples of this many slots
#define PRB_STAGE 128                   // a step closes at most PRB_STEP / PRB_ALIGN runs

__device__ __forceinline__ uint4 prb_ld_v4u(const uint4 *p, uint64_t pol)
{
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.u32 {%0,%1,%2,%3}, [%4], %5;"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p), "l"(pol));
    return r;
}

// rank of every row without out-edges: pr_epilogue with sum = 0
__device__ __forceinline__ float pr_zero_rank(float k, float d, float dang) { return __fadd_rn(k, __fmul_rn(d, __fadd_rn(0.f, dang))); }

// A column at or above PrParams::zero_kept is a row without out-edges whose contribution the previous sweep did not store: the
// gather loads inv[v] instead, and the value is z0 * inv[v], z0 being that sweep's rank0, which is the product it would have
// stored. The multiply is applied where the gathered values are summed: next to the load it would wait for the load before the
// next gather goes out.
__device__ __forceinline__ float pr_zero_scale(bool zero, float z0, float x) { return zero ? __fmul_rn(z0, x) : x; }

struct PrbStep
{
    uint4 a, b;
    unsigned m;
};

// the four 4-slot group sums of this lane's 16 slots
template <bool COLD>
__device__ __forceinline__ void prb_groups(const PrbBinParams &P, const L2Pol &pol, const float *sl, const PrbStep &cur, int64_t s, int lane,
                                           float z0, float (&g)[4])
{
    if (!COLD)
    {
        g[0] = (sl[cur.a.x & 0xffff] + sl[cur.a.x >> 16]) + (sl[cur.a.y & 0xffff] + sl[cur.a.y >> 16]);
        g[1] = (sl[cur.a.z & 0xffff] + sl[cur.a.z >> 16]) + (sl[cur.a.w & 0xffff] + sl[cur.a.w >> 16]);
        g[2] = (sl[cur.b.x & 0xffff] + sl[cur.b.x >> 16]) + (sl[cur.b.y & 0xffff] + sl[cur.b.y >> 16]);
        g[3] = (sl[cur.b.z & 0xffff] + sl[cur.b.z >> 16]) + (sl[cur.b.w & 0xffff] + sl[cur.b.w >> 16]);
    }
    else
    {
        const int4 *c4 = reinterpret_cast<const int4 *>(P.cold) + (s - (int64_t)P.cold_chunk0 * PRB_SPC) * 128 + lane;
        int4 v[4];
#pragma unroll
        for (int j = 0; j < 4; j++) v[j] = ld_stream_v4(c4 + j * 32, pol.stream);
        float x[16];
        unsigned zero = 0; // bit i: slot i is a column from zero_col on (pr_zero_scale)
#pragma unroll
        for (int j = 0; j < 4; j++)
        {
            const int c[4] = {v[j].x, v[j].y, v[j].z, v[j].w};
#pragma unroll
            for (int i = 0; i < 4; i++)
            {
                x[4 * j + i] = 0.f; // (padding: -1)
                if (c[i] >= 0)
                {
                    zero |= (c[i] >= P.zero_col ? 1u : 0u) << (4 * j + i);
                    x[4 * j + i] = ld_gather_cold_f32((c[i] >= P.zero_col ? P.inv : P.contrib_in) + c[i], pol.keep);
                }
            }
        }
#pragma unroll
        for (int i = 0; i < 16; i++) x[i] = pr_zero_scale((zero >> i) & 1, z0, x[i]);
#pragma unroll
        for (int j = 0; j < 4; j++) g[j] = (x[4 * j] + x[4 * j + 1]) + (x[4 * j + 2] + x[4 * j + 3]);
    }
}

__device__ __forceinline__ PrbStep prb_load_step(const PrbBinParams &P, const L2Pol &pol, int64_t s, int lane, bool cold)
{
    PrbStep d;
    if (!cold)
    {
        const uint4 *w = reinterpret_cast<const uint4 *>(P.wcol) + s * 64 + lane;
        d.a = prb_ld_v4u(w, pol.stream);
        d.b = prb_ld_v4u(w + 32, pol.stream);
    }
    else
        d.a = d.b = make_uint4(0, 0, 0, 0);
    d.m = __ldg(P.meta + s * 32 + lane);
    return d;
}

// One unit = the steps [s0, s1) of one bin: emits the sums of the runs that START in it. The warp ignores the leading part of a
// run that started earlier and runs on past s1 until the next start (in those steps only the lanes up to the first start
// gather). Latency: the unit is a stream — columns and metadata are fetched two steps ahead, and the sums a step closes are
// stored one step later, with slot numbers fetched meanwhile (`stage` holds 2 x PRB_STAGE floats).
template <bool COLD>
__device__ __forceinline__ void prb_unit(const PrbBinParams &P, const L2Pol &pol, const float *sl, int s0, int s1, int bin_end_step, int lane,
                                         float *stage, float z0)
{
    const unsigned FULL = 0xffffffffu;
    const int r_first = P.step_run0[s0], r_end = P.step_run0[s1]; // runs that start here
    if (r_first == r_end) return;
    float carry = 0.f;  // sum of the open run so far (lanes of earlier steps)
    int run0 = r_first; // runs started before the current step: start t of the step closes run run0 + t - 1
    PrbStep cur = prb_load_step(P, pol, s0, lane, COLD), nxt = cur;
    if (s0 + 1 < bin_end_step) nxt = prb_load_step(P, pol, s0 + 1, lane, COLD);
    int psa = -1, psb = -1, pbuf = 0; // where the sums staged by the previous step go, and the half of `stage` that holds them
    for (int s = s0; s < bin_end_step; s++)
    {
        const unsigned m = cur.m;
        const int pre = (m >> 4) & 0xff, total = (m >> 18) & 0xff;
        const bool beyond = s >= s1; // only the run that is still open matters: it ends at this step's first start
        const bool ahead2 = s + 2 <= s1 || (beyond && total == 0);
        PrbStep nx2 = nxt;
        if (ahead2 && s + 2 < bin_end_step) nx2 = prb_load_step(P, pol, s + 2, lane, COLD);
        const int ra = run0 + lane - 1, rb = ra + 32;
        const int sa = (lane < total && ra >= r_first && ra < r_end) ? __ldg(P.run_slot + ra) : -1;
        const int sb = (lane + 32 < total && rb >= r_first && rb < r_end) ? __ldg(P.run_slot + rb) : -1;
        float *st = stage + (s & 1) * PRB_STAGE;
        float g[4] = {0.f, 0.f, 0.f, 0.f};
        if (!beyond || !((m >> 17) & 1)) prb_groups<COLD>(P, pol, sl, cur, s, lane, z0, g);
        // in-lane pass: head = sum before the first start, tail = open run; the sums of the runs that close inside the lane are
        // staged in shared memory by their index within the step
        float run = 0.f, head = 0.f;
        int j = 0;
#pragma unroll
        for (int e = 0; e < 4; e++)
        {
            if ((m >> e) & 1)
            {
                if (j == 0) head = run;
                else st[pre + j] = run;
                run = 0.f;
                j++;
            }
            run += g[e];
        }
        if (j == 0) head = run;
        // segmented inclusive scan over the lanes of (lane with a start ? its tail : the whole lane), static masks
        float v = run;
#pragma unroll
        for (int o = 0; o < 5; o++)
        {
            const float vu = __shfl_up_sync(FULL, v, 1 << o);
            if ((m >> (12 + o)) & 1) v += vu;
        }
        float ex = __shfl_up_sync(FULL, v, 1);
        if (lane == 0) ex = 0.f;
        if (j > 0) st[pre] = (((m >> 17) & 1) ? ex : carry + ex) + head; // closes run run0 + pre - 1
        const float v31 = __shfl_sync(FULL, v, 31);
        carry = total > 0 ? v31 : carry + v31;
        __syncwarp();
        {
            const float *stp = stage + pbuf * PRB_STAGE; // the previous step's sums
            if (psa >= 0) P.slot[psa] = stp[lane];
            if (psb >= 0) P.slot[psb] = stp[lane + 32];
        }
        for (int t0 = 64; t0 < total; t0 += 64) // (rare: more than 64 runs closed by one step)
        {
            const int ta = t0 + lane, tb = ta + 32;
            const int qa = run0 + ta - 1, qb = run0 + tb - 1;
            const int xa = (ta < total && qa >= r_first && qa < r_end) ? __ldg(P.run_slot + qa) : -1;
            const int xb = (tb < total && qb >= r_first && qb < r_end) ? __ldg(P.run_slot + qb) : -1;
            if (xa >= 0) P.slot[xa] = st[ta];
            if (xb >= 0) P.slot[xb] = st[tb];
        }
        __syncwarp();
        psa = sa;
        psb = sb;
        pbuf = s & 1;
        run0 += total;
        if (beyond && total > 0) break; // the first start beyond the unit closed its last run
        cur = nxt;
        nxt = nx2;
        // (past the unit the stream is fetched one step ahead, and only while the last run is still open)
        if (!ahead2 && s + 2 < bin_end_step && !(s + 1 >= s1 && ((cur.m >> 18) & 0xff) > 0)) nxt = prb_load_step(P, pol, s + 2, lane, COLD);
    }
    {
        const float *stp = stage + pbuf * PRB_STAGE; // the last step's sums
        if (psa >= 0) P.slot[psa] = stp[lane];
        if (psb >= 0) P.slot[psb] = stp[lane + 32];
    }
    __syncwarp();
}

#endif

int vglb_pr_prepare(vglb_ctx *ctx, vglb_graph *g, int iters);
int64_t vglb_pr_plan(const vglb_graph *g, int32_t rows, PrParams *P);
int vglb_pr_launch_sweep(vglb_ctx *ctx, const PrParams &P, int64_t nblocks);
