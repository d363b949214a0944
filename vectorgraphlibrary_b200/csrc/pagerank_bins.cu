// pagerank_bins.cu — column-binned gather for the heavy rows of the PageRank sweep (one GPU).
//
// What it replaces: the edge_op of the pull sweep (algorithms/pr/pr.hpp:105-124) over the rows with >= 32 edges — 89 % of the
// edges of RMAT-24. Gathering contrib[v] straight from global memory is bound by the SM's L1-miss request port (one 128-byte
// line request per clock and SM: profiles/r1_pr_gather_lab*.txt): 56 % of the gathers of RMAT-24 miss the 200 KB an SM can
// keep hot, and a bigger on-SM hot set does not exist. So the edges are regrouped instead (dev/pr_bin_lab.cu,
// profiles/r2_pr_bin_lab.txt):
//   * columns are cut into NB bins of PRB_H = 49152 consecutive (degree-sorted, i.e. hottest first) ids; the edges of the
//     heavy rows are stored bin by bin, inside a bin by row: a (bin,row) RUN. While a bin is processed its slice of the
//     contribution vector sits in shared memory (192 KB), so every gather is a shared-memory read; column ids shrink to 16 bits.
//   * edges whose column lies beyond the bins (8-15 %) form a last, "cold" bin with 32-bit columns gathered from global memory.
//   * a run's sum goes to slot[class][row chunk]; pr_sweep_kernel's finish blocks add a row's slots and run the epilogue.
// The run structure is static, so everything the segmented sum needs is precomputed per lane and warp step (`meta`), runs start
// at multiples of 4 slots (padding gathers a zero) and a row's edges are cut into chunks of PRB_RC edges first, so no run is
// longer than that (the longest rows of a power-law graph would otherwise serialise one warp).
// Persistent kernel: one CTA of 32 warps per SM walks a contiguous, cost-balanced range of 4096-slot chunks; the warp that owns
// a chunk emits the runs that START in it (it runs on past the end of the chunk until the next start). No atomics, fixed
// summation order.
#include <stdlib.h>

#include <cub/device/device_scan.cuh>

#include "common.cuh"
#include "pagerank.cuh"

#define PRB_THREADS 1024
#define PRB_WARPS (PRB_THREADS / 32)
#define PRB_DROP 0xff                   // class of a self loop: not part of the sum (pr.hpp:112)
#define PRB_SMEM_BYTES ((PRB_H + 4) * 4 + PRB_WARPS * 2 * PRB_STAGE * 4)

// meta word of one lane and step:
//   bits 0..3   a run starts at slot 4 g of the lane         bits 4..11  run starts in the lanes before (this step)
//   bits 12..16 segmented-scan mask: add lane - 2^k in round k
//   bit 17      some lane before this one has a start        bits 18..25 run starts in the whole step

// Bins are ranges of the SORTED (hottest first) vertex ids. On one GPU a column id is the sorted id; on one rank's part of a
// partitioned graph column = owner * vp + local row and the sorted id is local row * ranks + owner (partition.cu).
__device__ __forceinline__ uint32_t prb_sorted_id(int32_t v, int world, uint32_t vp)
{
    return world <= 1 ? (uint32_t)v : ((uint32_t)v % vp) * (uint32_t)world + (uint32_t)v / vp;
}
__device__ __forceinline__ int prb_class(uint32_t sorted_id, int nb)
{
    const int c = (int)(sorted_id / (uint32_t)PRB_H);
    return c < nb ? c : nb;
}

// stored position of logical slot q: a step's 512 slots are stored as two 256-slot halves (16-bit columns) or four 128-slot
// quarters (32-bit columns), so that every 16-byte load of a warp is contiguous
__device__ __forceinline__ int64_t prb_phys16(int64_t q)
{
    const int i = (int)(q & (PRB_STEP - 1)), lane = i >> 4, sub = i & 15;
    return (q - i) + (sub >> 3) * 256 + lane * 8 + (sub & 7);
}
__device__ __forceinline__ int64_t prb_phys32(int64_t q)
{
    const int i = (int)(q & (PRB_STEP - 1)), lane = i >> 4, sub = i & 15;
    return (q - i) + (sub >> 2) * 128 + lane * 4 + (sub & 3);
}

// ---- build ------------------------------------------------------------------------------------------------------------------

__global__ void prb_row_chunks_kernel(const int64_t *__restrict__ ptr, int32_t rows, int32_t *__restrict__ nchunks)
{
    const int32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r < rows) nchunks[r] = (int32_t)((ptr[r + 1] - ptr[r] + PRB_RC - 1) / PRB_RC);
    if (r == rows) nchunks[r] = 0;
}

// row and edge range of row chunk ci (rows >= long_rows have one chunk each: ci = row + xc)
__device__ __forceinline__ void prb_chunk_range(const int64_t *__restrict__ ptr, const int32_t *__restrict__ rc_ptr, int32_t long_rows,
                                                int32_t xc, int32_t ci, int32_t &row, int64_t &e0, int64_t &e1)
{
    if (ci >= long_rows + xc)
    {
        row = ci - xc;
        e0 = ptr[row];
        e1 = ptr[row + 1];
        return;
    }
    int32_t lo = 0, hi = long_rows; // last row with rc_ptr[row] <= ci
    while (hi - lo > 1)
    {
        const int32_t mid = (lo + hi) >> 1;
        if (rc_ptr[mid] <= ci) lo = mid;
        else hi = mid;
    }
    row = lo;
    e0 = ptr[row] + (int64_t)(ci - rc_ptr[row]) * PRB_RC;
    e1 = min(ptr[row + 1], e0 + PRB_RC);
}

// FILL = false: cnt[class * nch + ci] = edges of row chunk ci in that class.
// FILL = true: the edges are written to their slots, in the order of the adjacency inside every run.
template <bool FILL>
__global__ void __launch_bounds__(256) prb_scatter_kernel(const int64_t *__restrict__ ptr, const int32_t *__restrict__ adj,
                                                           const int32_t *__restrict__ rc_ptr, int32_t long_rows, int32_t xc, int32_t nch,
                                                           int nb, int32_t col_of_row0, int world, uint32_t vp, int32_t *__restrict__ cnt,
                                                           const int64_t *__restrict__ run_pos, int64_t w_smem, uint16_t *__restrict__ wcol,
                                                           int32_t *__restrict__ cold)
{
    __shared__ long long s_acc[8][PRB_BINS + 1];
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nc = nb + 1;
    const int32_t ci = blockIdx.x * 8 + warp;
    if (ci >= nch) return;
    int32_t row;
    int64_t e0, e1;
    prb_chunk_range(ptr, rc_ptr, long_rows, xc, ci, row, e0, e1);
    for (int c = lane; c < nc; c += 32) s_acc[warp][c] = FILL ? run_pos[(int64_t)c * nch + ci] : 0;
    __syncwarp();
    for (int64_t p0 = e0; p0 < e1; p0 += 32)
    {
        const int64_t p = p0 + lane;
        const int32_t self = col_of_row0 + row;
        const int32_t v = p < e1 ? adj[p] : self;
        const uint32_t sid = prb_sorted_id(v, world, vp);
        const int c = v == self ? PRB_DROP : prb_class(sid, nb);
        const unsigned peers = __match_any_sync(FULL, c);
        const int rank = __popc(peers & ((1u << lane) - 1u));
        if (c != PRB_DROP)
        {
            if (FILL)
            {
                const int64_t q = s_acc[warp][c] + rank;
                if (c < nb) wcol[prb_phys16(q)] = (uint16_t)(sid - (uint32_t)c * PRB_H);
                else cold[prb_phys32(q - w_smem)] = v;
            }
        }
        __syncwarp();
        if (c != PRB_DROP && rank == 0) s_acc[warp][c] += __popc(peers);
        __syncwarp();
    }
    if (!FILL)
        for (int c = lane; c < nc; c += 32) cnt[(int64_t)c * nch + ci] = (int32_t)s_acc[warp][c];
}

__global__ void prb_lengths_kernel(const int32_t *__restrict__ cnt, int64_t n, int64_t *__restrict__ plen, int32_t *__restrict__ pflag)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n)
    {
        const int32_t c = cnt[i];
        plen[i] = (c + PRB_ALIGN - 1) / PRB_ALIGN * PRB_ALIGN;
        pflag[i] = c > 0;
    }
    if (i == n)
    {
        plen[i] = 0;
        pflag[i] = 0;
    }
}

// one thread: where every bin starts (bins are padded to whole chunks, the padding starts with a flagged dummy run)
// out[0] = all slots, out[1] = slots of the shared-memory bins, out[2] = runs (with the dummies)
__global__ void prb_bins_kernel(const int64_t *__restrict__ pos_scan, const int32_t *__restrict__ flag_scan, int32_t nch, int nc,
                                int64_t *__restrict__ bin_start, int32_t *__restrict__ bin_chunk0, int64_t *__restrict__ out)
{
    int64_t start = 0;
    for (int c = 0; c < nc; c++)
    {
        bin_start[c] = start;
        bin_chunk0[c] = (int32_t)(start / PRB_CHUNK);
        if (c == nc - 1) out[1] = start;
        const int64_t total = pos_scan[(int64_t)(c + 1) * nch] - pos_scan[(int64_t)c * nch];
        start = (start + total + PRB_ALIGN + PRB_CHUNK - 1) / PRB_CHUNK * PRB_CHUNK;
    }
    bin_start[nc] = start;
    bin_chunk0[nc] = (int32_t)(start / PRB_CHUNK);
    out[0] = start;
    out[2] = (int64_t)flag_scan[(int64_t)nc * nch] + nc;
}

// start flag and slot of every run; thread nc * nch + c handles bin c's dummy run (the first padding slot of the bin)
__global__ void prb_runs_kernel(const int32_t *__restrict__ cnt, const int64_t *__restrict__ run_pos, const int64_t *__restrict__ pos_scan,
                                const int32_t *__restrict__ flag_scan, const int64_t *__restrict__ bin_start, int32_t nch, int nc,
                                uint32_t *__restrict__ meta, int32_t *__restrict__ run_slot)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, n = (int64_t)nc * nch;
    int64_t q;
    int32_t run, slot;
    if (i < n)
    {
        if (cnt[i] == 0) return;
        q = run_pos[i];
        run = flag_scan[i] + (int32_t)(i / nch);
        slot = (int32_t)i;
    }
    else if (i < n + nc)
    {
        const int c = (int)(i - n);
        q = bin_start[c] + (pos_scan[(int64_t)(c + 1) * nch] - pos_scan[(int64_t)c * nch]);
        run = flag_scan[(int64_t)(c + 1) * nch] + c;
        slot = (int32_t)n; // never emitted
    }
    else
        return;
    run_slot[run] = slot;
    const int64_t word = (q / PRB_STEP) * 32 + ((q % PRB_STEP) >> 4);
    atomicOr(meta + word, 1u << ((q & 15) / PRB_ALIGN));
}

// run_pos[i] = first slot of run i
__global__ void prb_run_pos_kernel(const int64_t *__restrict__ pos_scan, const int64_t *__restrict__ bin_start, int32_t nch, int nc,
                                   int64_t *__restrict__ run_pos)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, n = (int64_t)nc * nch;
    if (i >= n) return;
    const int c = (int)(i / nch);
    run_pos[i] = bin_start[c] + (pos_scan[i] - pos_scan[(int64_t)c * nch]);
}

// one warp per step: the static part of the segmented sum
__global__ void prb_meta_kernel(uint32_t *__restrict__ meta, int64_t nsteps, int32_t *__restrict__ step_total)
{
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const int64_t s = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (s >= nsteps) return;
    const uint32_t f = meta[s * 32 + lane] & 15u;
    const int nst = __popc(f);
    int pre = nst;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1)
    {
        const int t = __shfl_up_sync(FULL, pre, o);
        if (lane >= o) pre += t;
    }
    const int total = __shfl_sync(FULL, pre, 31);
    pre -= nst;
    const unsigned starts = __ballot_sync(FULL, f != 0);
    const unsigned upto = starts & (lane == 31 ? FULL : ((2u << lane) - 1u)); // lanes <= this one with a start
    const int seg = upto ? 31 - __clz(upto) : 0;                              // where this lane's segment begins
    uint32_t m = f | ((uint32_t)pre << 4) | ((uint32_t)total << 18);
    if (!f)
        for (int o = 0; o < 5; o++)
            if (lane - (1 << o) >= seg) m |= 1u << (12 + o);
    if (starts & ((1u << lane) - 1u)) m |= 1u << 17;
    meta[s * 32 + lane] = m;
    if (lane == 0) step_total[s] = total;
    if (s == nsteps - 1 && lane == 0) step_total[nsteps] = 0;
}

// estimated cost of a chunk of a shared-memory bin: its 8 steps + the runs it closes
__global__ void prb_cost_kernel(const int32_t *__restrict__ step_run0, int32_t nkchunks, int64_t *__restrict__ cost)
{
    const int32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= nkchunks) return;
    const int32_t closes = step_run0[(int64_t)(k + 1) * PRB_SPC] - step_run0[(int64_t)k * PRB_SPC];
    cost[k] = 2048 + closes;
}

__global__ void prb_cta_ranges_kernel(const int64_t *__restrict__ cum, int32_t nkchunks, int grid, int32_t *__restrict__ cta_chunk0)
{
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b > grid) return;
    if (b == grid || nkchunks == 0)
    {
        cta_chunk0[b] = nkchunks;
        return;
    }
    const int64_t want = (int64_t)((double)cum[nkchunks - 1] * (double)b / (double)grid);
    int32_t lo = 0, hi = nkchunks; // first chunk whose inclusive cumulative cost exceeds `want`
    while (lo < hi)
    {
        const int32_t mid = (lo + hi) >> 1;
        if (cum[mid] > want) hi = mid;
        else lo = mid + 1;
    }
    cta_chunk0[b] = b == 0 ? 0 : lo;
}

__global__ void prb_fill_u16_kernel(uint16_t *a, int64_t n, uint16_t val)
{
    // n is a multiple of 8
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i * 8 < n)
    {
        const uint32_t w = (uint32_t)val | ((uint32_t)val << 16);
        reinterpret_cast<uint4 *>(a)[i] = make_uint4(w, w, w, w);
    }
}

// frees a PrBins and its arrays (the owner of one that is still being built, and vglb_pr_bins_free)
struct prb_deleter
{
    void operator()(PrBins *B) const
    {
        vglb_dev_free(B->d_wcol);
        vglb_dev_free(B->d_cold);
        vglb_dev_free(B->d_meta);
        vglb_dev_free(B->d_step_run0);
        vglb_dev_free(B->d_run_slot);
        vglb_dev_free(B->d_bin_chunk0);
        vglb_dev_free(B->d_cta_chunk0);
        vglb_dev_free(B->d_slot);
        vglb_dev_free(B->d_rc_ptr);
        free(B);
    }
};

void vglb_pr_bins_free(vglb_graph *g)
{
    if (g->pr_bins) prb_deleter()((PrBins *)g->pr_bins);
    g->pr_bins = NULL;
}

// Builds the binned copy of the heavy rows (degree >= 32) of a one-GPU graph. Leaves g->pr_bins NULL when there is nothing to
// bin (no heavy rows).
int vglb_pr_bins_build(vglb_ctx *ctx, vglb_graph *g) { return vglb_pr_bins_build_rows(ctx, g, g->tier_border[1]); }

// (vglb_graph_from_csr calls this before the graph is complete: only V, d_out_ptr and the adjacency of rows [0, rows) are used)
int vglb_pr_bins_build_rows(vglb_ctx *ctx, vglb_graph *g, int32_t rows)
{
    if (rows <= 0) return VGLB_OK;
    const int world = g->comm ? g->part_world : 1;
    const int64_t ncols = g->comm ? g->cols : (int64_t)g->V;
    cudaStream_t st = ctx->stream;
    int32_t long_rows = 0;
    VGLB_TRY(vglb_graph_threshold_vertex(ctx, g, PRB_RC + 1, &long_rows)); // rows with more than one chunk
    // 32 bins = the hottest 9.4 % of the columns of the BASELINE graph = 91 % of the gathers of its heavy rows. Every further bin
    // costs the finish pass one more partial sum per heavy row: 64 bins are no faster there, and on 4 GPUs (scale 26: 32 bins hold
    // 74 % of the gathers) 32 / 64 / 128 bins gave 1034 / 1075 / 939 GTEPS against 1108 with the warp tasks.
    const int nb = (int)std::min<int64_t>(PRB_BINS, ceil_div64(ncols, PRB_H));
    const int nc = nb + 1;

    std::unique_ptr<PrBins, prb_deleter> owner((PrBins *)calloc(1, sizeof(PrBins)));
    VGLB_REQUIRE(owner != NULL, "vglb_pr_bins_build: out of host memory");
    PrBins *B = owner.get();
    dev_ptr<int32_t> d_nchunks, d_rc_full, d_cnt, d_pflag, d_flag_scan, d_step_total;
    dev_ptr<int64_t> d_plen, d_pos_scan, d_bin_start, d_out, d_run_pos, d_cost;
    dev_ptr<void> tmp; // CUB temporaries, each freed where its scan has finished
    // row chunks
    CUDA_TRY(vglb_dev_alloc(d_nchunks, ((size_t)rows + 1) * 4));
    CUDA_TRY(vglb_dev_alloc(d_rc_full, ((size_t)rows + 1) * 4));
    prb_row_chunks_kernel<<<(unsigned)ceil_div64(rows + 1, 256), 256, 0, st>>>(g->d_out_ptr, rows, d_nchunks.get());
    KERNEL_TRY();
    CUDA_TRY(vglb_cub(tmp, [&](void *t, size_t &bytes) { return cub::DeviceScan::ExclusiveSum(t, bytes, (const int32_t *)d_nchunks.get(), d_rc_full.get(), (int64_t)rows + 1, st); }));
    CUDA_TRY(cudaStreamSynchronize(st));
    tmp.reset();
    int32_t nch = 0;
    CUDA_TRY(cudaMemcpyAsync(&nch, d_rc_full.get() + rows, 4, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    const int32_t xc = nch - rows; // chunks beyond one per row; all of them belong to the first long_rows rows
    CUDA_TRY(vglb_dev_alloc(&B->d_rc_ptr, ((size_t)long_rows + 1) * 4));
    CUDA_TRY(cudaMemcpyAsync(B->d_rc_ptr, d_rc_full.get(), ((size_t)long_rows + 1) * 4, cudaMemcpyDeviceToDevice, st));
    const int64_t n = (int64_t)nc * nch;
    if (n >= 0x7fffffffLL) { vglb_set_error("vglb_pr_bins_build: too many runs"); return VGLB_EINVAL; }
    // counts per (class, row chunk), scans, layout
    CUDA_TRY(vglb_dev_alloc(d_cnt, (size_t)n * 4));
    prb_scatter_kernel<false><<<(unsigned)ceil_div64(nch, 8), 256, 0, st>>>(g->d_out_ptr, g->d_out_adj, B->d_rc_ptr, long_rows, xc, nch, nb,
                                                                           g->col_of_row0, world, (uint32_t)g->vp, d_cnt.get(), NULL, 0, NULL, NULL);
    KERNEL_TRY();
    CUDA_TRY(vglb_dev_alloc(d_plen, ((size_t)n + 1) * 8));
    CUDA_TRY(vglb_dev_alloc(d_pflag, ((size_t)n + 1) * 4));
    CUDA_TRY(vglb_dev_alloc(d_pos_scan, ((size_t)n + 1) * 8));
    CUDA_TRY(vglb_dev_alloc(d_flag_scan, ((size_t)n + 1) * 4));
    prb_lengths_kernel<<<(unsigned)ceil_div64(n + 1, 256), 256, 0, st>>>(d_cnt.get(), n, d_plen.get(), d_pflag.get());
    KERNEL_TRY();
    CUDA_TRY(vglb_cub(tmp, [&](void *t, size_t &bytes) { return cub::DeviceScan::ExclusiveSum(t, bytes, (const int64_t *)d_plen.get(), d_pos_scan.get(), n + 1, st); }));
    CUDA_TRY(cudaStreamSynchronize(st));
    tmp.reset();
    CUDA_TRY(vglb_cub(tmp, [&](void *t, size_t &bytes) { return cub::DeviceScan::ExclusiveSum(t, bytes, (const int32_t *)d_pflag.get(), d_flag_scan.get(), n + 1, st); }));
    CUDA_TRY(cudaStreamSynchronize(st));
    tmp.reset();
    CUDA_TRY(vglb_dev_alloc(d_bin_start, ((size_t)nc + 1) * 8));
    CUDA_TRY(vglb_dev_alloc(&B->d_bin_chunk0, ((size_t)nc + 1) * 4));
    CUDA_TRY(vglb_dev_alloc(d_out, 3 * 8));
    prb_bins_kernel<<<1, 1, 0, st>>>(d_pos_scan.get(), d_flag_scan.get(), nch, nc, d_bin_start.get(), B->d_bin_chunk0, d_out.get());
    KERNEL_TRY();
    int64_t h_out[3];
    CUDA_TRY(cudaMemcpyAsync(h_out, d_out.get(), sizeof(h_out), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    const int64_t W = h_out[0], w_smem = h_out[1], nruns = h_out[2], nsteps = W / PRB_STEP;
    if (W / PRB_CHUNK >= 0x7fffffffLL || nruns >= 0x7fffffffLL) { vglb_set_error("vglb_pr_bins_build: graph too large for 32-bit chunk / run numbers"); return VGLB_EINVAL; }
    B->nb = nb;
    B->rows = rows;
    B->long_rows = long_rows;
    B->nch = nch;
    B->xc = xc;
    B->nkchunks = (int32_t)(W / PRB_CHUNK);
    B->cold_chunk0 = (int32_t)(w_smem / PRB_CHUNK);
    B->slots = W;
    B->nruns = (int32_t)nruns;
    B->grid = ctx->sm_count;
    // the arrays the sweep reads
    CUDA_TRY(vglb_dev_alloc(&B->d_wcol, (size_t)(w_smem > 0 ? w_smem : 8) * 2));
    CUDA_TRY(vglb_dev_alloc(&B->d_cold, (size_t)(W - w_smem) * 4));
    CUDA_TRY(vglb_dev_alloc(&B->d_meta, (size_t)nsteps * 32 * 4));
    CUDA_TRY(vglb_dev_alloc(&B->d_step_run0, ((size_t)nsteps + 1) * 4));
    CUDA_TRY(vglb_dev_alloc(&B->d_run_slot, (size_t)nruns * 4));
    CUDA_TRY(vglb_dev_alloc(&B->d_slot, ((size_t)n + 1) * 4));
    CUDA_TRY(vglb_dev_alloc(&B->d_cta_chunk0, ((size_t)B->grid + 1) * 4));
    CUDA_TRY(cudaMemsetAsync(B->d_slot, 0, ((size_t)n + 1) * 4, st));
    CUDA_TRY(cudaMemsetAsync(B->d_meta, 0, (size_t)nsteps * 32 * 4, st));
    CUDA_TRY(cudaMemsetAsync(B->d_cold, 0xFF, (size_t)(W - w_smem) * 4, st));
    if (w_smem > 0)
    {
        prb_fill_u16_kernel<<<(unsigned)ceil_div64(w_smem / 8, 256), 256, 0, st>>>(B->d_wcol, w_smem, (uint16_t)PRB_H);
        KERNEL_TRY();
    }
    // edges to their slots
    CUDA_TRY(vglb_dev_alloc(d_run_pos, (size_t)n * 8));
    prb_run_pos_kernel<<<(unsigned)ceil_div64(n, 256), 256, 0, st>>>(d_pos_scan.get(), d_bin_start.get(), nch, nc, d_run_pos.get());
    KERNEL_TRY();
    prb_scatter_kernel<true><<<(unsigned)ceil_div64(nch, 8), 256, 0, st>>>(g->d_out_ptr, g->d_out_adj, B->d_rc_ptr, long_rows, xc, nch, nb,
                                                                          g->col_of_row0, world, (uint32_t)g->vp, NULL, d_run_pos.get(), w_smem, B->d_wcol,
                                                                          B->d_cold);
    KERNEL_TRY();
    // run starts, slots, per-lane metadata, run numbers of the steps
    prb_runs_kernel<<<(unsigned)ceil_div64(n + nc, 256), 256, 0, st>>>(d_cnt.get(), d_run_pos.get(), d_pos_scan.get(), d_flag_scan.get(), d_bin_start.get(), nch, nc,
                                                                      B->d_meta, B->d_run_slot);
    KERNEL_TRY();
    CUDA_TRY(vglb_dev_alloc(d_step_total, ((size_t)nsteps + 1) * 4));
    prb_meta_kernel<<<(unsigned)ceil_div64(nsteps * 32, 256), 256, 0, st>>>(B->d_meta, nsteps, d_step_total.get());
    KERNEL_TRY();
    CUDA_TRY(vglb_cub(tmp, [&](void *t, size_t &bytes) { return cub::DeviceScan::ExclusiveSum(t, bytes, (const int32_t *)d_step_total.get(), B->d_step_run0, nsteps + 1, st); }));
    CUDA_TRY(cudaStreamSynchronize(st));
    tmp.reset();
    // cost-balanced chunk ranges of the persistent CTAs
    // (the cold bin's chunks are blocks of pr_sweep_kernel)
    if (B->cold_chunk0 > 0)
    {
        CUDA_TRY(vglb_dev_alloc(d_cost, (size_t)B->cold_chunk0 * 8));
        prb_cost_kernel<<<(unsigned)ceil_div64(B->cold_chunk0, 256), 256, 0, st>>>(B->d_step_run0, B->cold_chunk0, d_cost.get());
        KERNEL_TRY();
        CUDA_TRY(vglb_cub(tmp, [&](void *t, size_t &bytes) { return cub::DeviceScan::InclusiveSum(t, bytes, (const int64_t *)d_cost.get(), d_cost.get(), (int64_t)B->cold_chunk0, st); }));
        CUDA_TRY(cudaStreamSynchronize(st));
        tmp.reset();
    }
    prb_cta_ranges_kernel<<<(unsigned)ceil_div64(B->grid + 1, 256), 256, 0, st>>>(d_cost.get(), B->cold_chunk0, B->grid, B->d_cta_chunk0);
    KERNEL_TRY();
    CUDA_TRY(cudaStreamSynchronize(st));
    ctx->launches += 12;
    g->pr_bins = owner.release();
    return VGLB_OK;
}

// ---- the sweep's binned part ------------------------------------------------------------------------------------------------------

extern __shared__ __align__(16) float prb_smem[];

__global__ void __launch_bounds__(PRB_THREADS, 1) pr_bin_kernel(const __grid_constant__ PrbBinParams P)
{
    L2Pol pol;
    pol.stream = l2_policy_evict_first();
    pol.keep = l2_policy_evict_last();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int k_lo = P.cta_chunk0[blockIdx.x], k_hi = P.cta_chunk0[blockIdx.x + 1];
    float *stage = prb_smem + PRB_H + 4 + warp * 2 * PRB_STAGE;
    const int nc = P.nb; // (the cold bin's chunks are blocks of pr_sweep_kernel: they need the L1 this kernel gives to shared memory)
    int bin = 0;
    while (bin < nc && P.bin_chunk0[bin + 1] <= k_lo) bin++;
    for (; bin < nc && P.bin_chunk0[bin] < k_hi; bin++)
    {
        const int b_lo = max(k_lo, P.bin_chunk0[bin]), b_hi = min(k_hi, P.bin_chunk0[bin + 1]);
        const int bin_end_step = P.bin_chunk0[bin + 1] * PRB_SPC;
        {
            __syncthreads();
            // this bin's slice of the contribution vector (the last bin of a small graph is shorter)
            const int64_t c0 = (int64_t)bin * PRB_H;
            const int n = (int)min((int64_t)PRB_H, P.cols - c0);
            if (P.world <= 1)
            {
                const float4 *src = reinterpret_cast<const float4 *>(P.contrib_in + c0);
                float4 *dst = reinterpret_cast<float4 *>(prb_smem);
                for (int i = threadIdx.x; i < (n >> 2); i += PRB_THREADS) dst[i] = src[i];
                for (int i = (n & ~3) + threadIdx.x; i < n; i += PRB_THREADS) prb_smem[i] = P.contrib_in[c0 + i];
            }
            else
            {
                // sorted id c0 + i = local row * ranks + owner lives in column owner * vp + local row: one coalesced stream per owner
                // (PRB_H is a multiple of every supported rank count, so a bin starts at owner 0)
                const int per_owner = (n + P.world - 1) / P.world;
                const int64_t l0 = c0 / P.world;
                for (int o = 0; o < P.world; o++)
                    for (int l = threadIdx.x; l < per_owner; l += PRB_THREADS)
                        if (l * P.world + o < n) prb_smem[l * P.world + o] = P.contrib_in[(int64_t)o * P.vp + l0 + l];
            }
            if (threadIdx.x < 4) prb_smem[PRB_H + threadIdx.x] = 0.f; // what a padding slot gathers
            __syncthreads();
            // every warp streams one contiguous piece of this CTA's steps of the bin
            const int64_t nst = (int64_t)(b_hi - b_lo) * PRB_SPC;
            const int s0 = b_lo * PRB_SPC + (int)(nst * warp / PRB_WARPS), s1 = b_lo * PRB_SPC + (int)(nst * (warp + 1) / PRB_WARPS);
            if (s0 < s1) prb_unit<false>(P, pol, prb_smem, s0, s1, bin_end_step, lane, stage, 0.f);
        }
    }
}

void vglb_pr_bins_params(const vglb_graph *g, const float *contrib_in, PrbBinParams *P)
{
    const PrBins *B = (const PrBins *)g->pr_bins;
    P->wcol = B->d_wcol;
    P->cold = B->d_cold;
    P->meta = B->d_meta;
    P->step_run0 = B->d_step_run0;
    P->run_slot = B->d_run_slot;
    P->bin_chunk0 = B->d_bin_chunk0;
    P->cta_chunk0 = B->d_cta_chunk0;
    P->contrib_in = contrib_in;
    P->inv = g->d_pr_inv;
    P->slot = B->d_slot;
    P->nb = B->nb;
    P->cold_chunk0 = B->cold_chunk0;
    P->cols = g->comm ? g->cols : (int64_t)g->V;
    P->world = g->comm ? g->part_world : 1;
    P->vp = g->vp;
    P->nruns = B->nruns;
    P->zero_col = INT32_MAX;
}

int vglb_pr_bins_launch(vglb_ctx *ctx, vglb_graph *g, const float *contrib_in)
{
    PrBins *B = (PrBins *)g->pr_bins;
    if (!B || B->cold_chunk0 == 0) return VGLB_OK;
    if (!ctx->prb_smem_set)
    {
        CUDA_TRY(cudaFuncSetAttribute(pr_bin_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, PRB_SMEM_BYTES));
        ctx->prb_smem_set = 1;
    }
    PrbBinParams P;
    vglb_pr_bins_params(g, contrib_in, &P);
    pr_bin_kernel<<<B->grid, PRB_THREADS, PRB_SMEM_BYTES, ctx->stream>>>(P);
    KERNEL_TRY();
    ctx->launches++;
    return VGLB_OK;
}
