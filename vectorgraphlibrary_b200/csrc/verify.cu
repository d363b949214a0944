// verify.cu — device-side result verification and the EdgesArray out -> in mirror (sm_100a).
//
// verify: the reference's run-time checkers compare two vertex arrays on the host after reordering both to ORIGINAL
// (vgl_runtime/helpers/verify_results/verify_results.h): verify_results (:33-93, `error count` of elements that are not
// are_same :9-28), verify_ranking_results (:97-148, mean absolute difference against 1e-4) and equal_components (:198-254,
// two label arrays describe the same partition). Reorder + compare is 81 % of the inner wall time of a `-check` BFS run
// (SURVEY §8 f4); here the comparison is one pass on the device and only the counts come back. Both arrays must be in the
// same numbering (vglb_varray_reorder_u32 brings them there); counts do not depend on which one.
//
// EdgesArray mirror: VGL_Graph::copy_outgoing_to_incoming_edges (vgl_graph/reorder.hpp:229-233 ->
// VectorCSRGraph::reorder_edges_gather, vect_csr/reorder.hpp:61-75): per-edge values given at outgoing-CSR positions are
// copied to the positions of the same edges in the incoming CSR, so that gather-direction operators can index them with
// global_edge_pos (EdgesArray layout [outgoing | incoming], vect_csr_edges_array.hpp:49-65). The permutation
// in-position -> out-position is the stable sort of the out positions by destination — the very sort that built the
// incoming CSR (graph_build.cu: build_incoming) — computed on first use and kept with the graph.
#include <cub/device/device_radix_sort.cuh>
#include <float.h>
#include <stdlib.h>

#include "common.cuh"

namespace
{

enum { VF_I32 = 0, VF_F32 = 1 };

template <int KIND>
__global__ void verify_count_kernel(const uint32_t *__restrict__ a, const uint32_t *__restrict__ b, int64_t n, unsigned long long *out)
{
    int errors = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    {
        if (KIND == VF_I32) errors += a[i] != b[i];
        else
        {
            // are_same(float, float): fabs(a - b) <= epsilon * 100 (verify_results.h:9-13)
            const float x = __uint_as_float(a[i]), y = __uint_as_float(b[i]);
            errors += !(fabsf(x - y) <= FLT_EPSILON * 100.0f);
        }
    }
    errors = (int)warp_sum_i64(errors);
    if ((threadIdx.x & 31) == 0 && errors) atomicAdd(out, (unsigned long long)errors);
}

__global__ void verify_ranking_kernel(const float *__restrict__ a, const float *__restrict__ b, int64_t n, double *out /* [2] */)
{
    double diff = 0.0, ref = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    {
        diff += fabs((double)a[i] - (double)b[i]);
        ref += fabs((double)b[i]);
    }
    diff = warp_sum_f64(diff);
    ref = warp_sum_f64(ref);
    if ((threadIdx.x & 31) == 0)
    {
        atomicAdd(out, diff);
        atomicAdd(out + 1, ref);
    }
}

// equal_components, pass 1: the LAST index carrying each label (the reference's maps keep the last assignment)
__global__ void components_last_index_kernel(const int32_t *__restrict__ a, const int32_t *__restrict__ b, int32_t n, int32_t *__restrict__ last_a,
                                             int32_t *__restrict__ last_b, int *__restrict__ bad)
{
    for (int32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    {
        const int32_t la = a[i], lb = b[i];
        if (la < 0 || la > n + 1 || lb < 0 || lb > n + 1)
        {
            *bad = 1;
            continue;
        }
        atomicMax(&last_a[la], i);
        atomicMax(&last_b[lb], i);
    }
}

// pass 2: f_s[first[i]] != second[i] and s_f[second[i]] != first[i] each count one error (verify_results.h:228-241)
__global__ void components_compare_kernel(const int32_t *__restrict__ a, const int32_t *__restrict__ b, int32_t n,
                                          const int32_t *__restrict__ last_a, const int32_t *__restrict__ last_b, unsigned long long *out)
{
    int errors = 0;
    for (int32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    {
        errors += b[last_a[a[i]]] != b[i];
        errors += a[last_b[b[i]]] != a[i];
    }
    errors = (int)warp_sum_i64(errors);
    if ((threadIdx.x & 31) == 0 && errors) atomicAdd(out, (unsigned long long)errors);
}

__global__ void iota_u32_kernel(uint32_t *a, int64_t n)
{
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) a[i] = (uint32_t)i;
}

__global__ void gather_u32_kernel(const uint32_t *__restrict__ in, const uint32_t *__restrict__ index, int64_t n, uint32_t *__restrict__ out)
{
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) out[i] = in[index[i]];
}

int fetch_count(vglb_ctx *ctx, unsigned long long *d_out, int64_t *out)
{
    int rc = vglb_counters_fetch(ctx, d_out, 1);
    if (rc != VGLB_OK) return rc;
    *out = (int64_t)((unsigned long long *)ctx->h_counters)[0];
    return VGLB_OK;
}

} // namespace

extern "C" int vglb_verify_i32(vglb_ctx *ctx, const int32_t *d_a, const int32_t *d_b, int64_t n, int64_t *error_count)
{
    VGLB_REQUIRE(ctx != NULL && d_a != NULL && d_b != NULL && error_count != NULL && n >= 0, "vglb_verify_i32: bad argument");
    unsigned long long *d_out = (unsigned long long *)(ctx->d_counters + CTR_VERIFY_COUNT);
    CUDA_TRY(cudaMemsetAsync(d_out, 0, 8, ctx->stream));
    if (n > 0)
    {
        verify_count_kernel<VF_I32><<<ctx->sm_count * 8, 256, 0, ctx->stream>>>((const uint32_t *)d_a, (const uint32_t *)d_b, n, d_out);
        KERNEL_TRY();
        ctx->launches++;
    }
    return fetch_count(ctx, d_out, error_count);
}

extern "C" int vglb_verify_f32(vglb_ctx *ctx, const float *d_a, const float *d_b, int64_t n, int64_t *error_count)
{
    VGLB_REQUIRE(ctx != NULL && d_a != NULL && d_b != NULL && error_count != NULL && n >= 0, "vglb_verify_f32: bad argument");
    unsigned long long *d_out = (unsigned long long *)(ctx->d_counters + CTR_VERIFY_COUNT);
    CUDA_TRY(cudaMemsetAsync(d_out, 0, 8, ctx->stream));
    if (n > 0)
    {
        verify_count_kernel<VF_F32><<<ctx->sm_count * 8, 256, 0, ctx->stream>>>((const uint32_t *)d_a, (const uint32_t *)d_b, n, d_out);
        KERNEL_TRY();
        ctx->launches++;
    }
    return fetch_count(ctx, d_out, error_count);
}

extern "C" int vglb_verify_ranking_f32(vglb_ctx *ctx, const float *d_a, const float *d_ref, int64_t n, double *mean_abs_difference,
                                       double *relative_l1, int64_t *error_count)
{
    VGLB_REQUIRE(ctx != NULL && d_a != NULL && d_ref != NULL && n >= 0, "vglb_verify_ranking_f32: bad argument");
    double *d_out = (double *)(ctx->d_counters + CTR_VERIFY_SUMS);
    CUDA_TRY(cudaMemsetAsync(d_out, 0, 16, ctx->stream));
    if (n > 0)
    {
        verify_ranking_kernel<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(d_a, d_ref, n, d_out);
        KERNEL_TRY();
        ctx->launches++;
    }
    int rc = vglb_counters_fetch(ctx, d_out, 2);
    if (rc != VGLB_OK) return rc;
    double h[2];
    memcpy(h, ctx->h_counters, sizeof(h));
    const double diff = n > 0 ? h[0] / (double)n : 0.0;
    if (mean_abs_difference) *mean_abs_difference = diff;
    if (relative_l1) *relative_l1 = h[1] > 0.0 ? h[0] / h[1] : (h[0] > 0.0 ? HUGE_VAL : 0.0);
    if (error_count) *error_count = diff < 0.0001 ? 0 : n; // verify_results.h:127-130
    return VGLB_OK;
}

extern "C" int vglb_verify_components_i32(vglb_ctx *ctx, const int32_t *d_a, const int32_t *d_b, int32_t n, int64_t *error_count)
{
    VGLB_REQUIRE(ctx != NULL && d_a != NULL && d_b != NULL && error_count != NULL && n >= 0, "vglb_verify_components_i32: bad argument");
    dev_ptr<int32_t> last;
    CUDA_TRY(vglb_dev_alloc(last, 2 * ((size_t)n + 2) * 4));
    int32_t *last_a = last.get(), *last_b = last.get() + n + 2;
    unsigned long long *d_out = (unsigned long long *)(ctx->d_counters + CTR_VERIFY_COUNT);
    int *d_bad = (int *)(ctx->d_counters + CTR_BAD);
    CUDA_TRY(cudaMemsetAsync(last.get(), 0xFF, 2 * ((size_t)n + 2) * 4, ctx->stream));
    CUDA_TRY(cudaMemsetAsync(d_out, 0, 8, ctx->stream));
    CUDA_TRY(cudaMemsetAsync(d_bad, 0, 4, ctx->stream));
    if (n > 0)
    {
        components_last_index_kernel<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(d_a, d_b, n, last_a, last_b, d_bad);
        KERNEL_TRY();
        int bad = 0;
        CUDA_TRY(cudaMemcpyAsync(&bad, d_bad, 4, cudaMemcpyDeviceToHost, ctx->stream));
        CUDA_TRY(cudaStreamSynchronize(ctx->stream));
        if (bad)
        {
            vglb_set_error("vglb_verify_components_i32: labels must lie in [0, n + 1]");
            return VGLB_EINVAL;
        }
        components_compare_kernel<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(d_a, d_b, n, last_a, last_b, d_out);
        KERNEL_TRY();
        ctx->launches += 2;
    }
    VGLB_TRY(fetch_count(ctx, d_out, error_count));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return VGLB_OK;
}

// ---- EdgesArray: outgoing -> incoming mirror ---------------------------------------------------------------------------

static int edge_mirror_prepare(vglb_ctx *ctx, vglb_graph *g)
{
    if (g->d_in_to_out_pos) return VGLB_OK;
    VGLB_REQUIRE(g->comm == NULL, "vglb_earray_mirror_out_to_in: not available on a partitioned graph");
    VGLB_REQUIRE(g->E < 0xFFFFFFFFLL, "vglb_earray_mirror_out_to_in: more than 2^32 - 1 edges");
    VGLB_TRY(vglb_graph_derive_incoming(ctx, g)); // no-op when the incoming CSR exists
    const int64_t E = g->E;
    const size_t eb = (size_t)(E ? E : 1) * 4;
    dev_ptr<uint32_t> k0, k1, v0, v1;
    dev_ptr<void> tmp;
    CUDA_TRY(vglb_dev_alloc(k0, eb)); CUDA_TRY(vglb_dev_alloc(k1, eb));
    CUDA_TRY(vglb_dev_alloc(v0, eb)); CUDA_TRY(vglb_dev_alloc(v1, eb));
    if (E > 0)
    {
        // the sort that built the incoming CSR (stable, by destination, over the out positions), with the position as payload
        CUDA_TRY(cudaMemcpyAsync(k0.get(), g->d_out_adj, eb, cudaMemcpyDeviceToDevice, ctx->stream));
        iota_u32_kernel<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(v0.get(), E);
        KERNEL_TRY();
        const int bits = vglb_key_bits(g->V);
        cub::DoubleBuffer<uint32_t> keys(k0.get(), k1.get()), vals(v0.get(), v1.get());
        CUDA_TRY(vglb_cub(tmp, [&](void *t, size_t &bytes) {
            return cub::DeviceRadixSort::SortPairs(t, bytes, keys, vals, E, 0, bits, ctx->stream);
        }));
        CUDA_TRY(cudaStreamSynchronize(ctx->stream));
        g->d_in_to_out_pos = (vals.Current() == v0.get() ? v0 : v1).release();
    }
    else
        g->d_in_to_out_pos = v0.release();
    return VGLB_OK;
}

extern "C" int vglb_earray_mirror_out_to_in_u32(vglb_ctx *ctx, vglb_graph *g, const uint32_t *d_out_values, uint32_t *d_in_values)
{
    VGLB_REQUIRE(ctx != NULL && g != NULL && d_out_values != NULL && d_in_values != NULL, "vglb_earray_mirror_out_to_in_u32: NULL argument");
    VGLB_REQUIRE(d_out_values != (const uint32_t *)d_in_values, "vglb_earray_mirror_out_to_in_u32: the mirror is out-of-place");
    CUDA_TRY(cudaSetDevice(ctx->device));
    VGLB_TRY(edge_mirror_prepare(ctx, g));
    if (g->E > 0)
    {
        gather_u32_kernel<<<ctx->sm_count * 16, 256, 0, ctx->stream>>>(d_out_values, g->d_in_to_out_pos, g->E, d_in_values);
        KERNEL_TRY();
        ctx->launches++;
    }
    return VGLB_OK;
}
