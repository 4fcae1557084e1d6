// pcc_rift_batched.cu -- processRIFT's descriptor chain for every cluster of a concatenated cloud in one call.
//
// computeSimilarity runs processRIFT on every cluster of at most 700 points (src/comparator.cpp:590-684, 1224-1366).  Here one index
// over the union, one segment-restricted sorted radius pass at the largest radius (segmented_sorted_rows) and three row reductions
// (rift_segmented, pcc_radius.cu) replace the per-cluster builds and searches; the survivors are then compacted in (cluster, row)
// order.  Host round trips do not depend on the cluster count.
#include <cub/cub.cuh>
#include <algorithm>
#include <cmath>
#include <vector>

#include "pcc_internal.h"

namespace pcc {

// processRIFT's two drops (:637-646, :674-681): a row survives when its normal and every one of its nb bins are finite.  flags[rows] = 0
// so that the exclusive scan leaves the survivor count there.
__global__ void rift_survivor_kernel(const float4 *__restrict__ normals, const float *__restrict__ desc, int64_t rows, int nb, int64_t *__restrict__ flags) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t > rows) return;
    bool ok = false;
    if (t < rows) {
        const float4 m = normals[t];
        ok = finite3(m.x, m.y, m.z);
        for (int k = 0; ok && k < nb; ++k) ok = isfinite(desc[t * nb + k]);
    }
    flags[t] = ok;
}
// survivors per cluster: the scanned flags at each cluster's first row (off[n_seg] = rows gives the total)
__global__ void rift_seg_bounds_kernel(const int64_t *__restrict__ pos, const int64_t *__restrict__ off, int n_seg, int64_t *__restrict__ out) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c <= n_seg) out[c] = pos[off[c]];
}
// survivors to their place in (cluster, row) order, with cluster-local row numbers; places at or past cap are dropped
__global__ void rift_scatter_kernel(const float *__restrict__ desc, const int64_t *__restrict__ pos, int64_t rows, int nb, const int64_t *__restrict__ off,
                                    int n_seg, int64_t cap, float *__restrict__ out_desc, int32_t *__restrict__ out_rows) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= rows) return;
    const int64_t d = pos[t];
    if (pos[t + 1] == d || d >= cap) return;
    for (int k = 0; k < nb; ++k) out_desc[d * nb + k] = desc[t * nb + k];
    out_rows[d] = (int32_t)(t - off[segment_of(off, n_seg, t)]);
}

}  // namespace pcc

using namespace pcc;

extern "C" {

int pcc_rift_batched(pcc_index *idx, const void *pts, int64_t n, int stride_bytes, const float *intensity, const int64_t *cloud_offsets, int64_t n_clouds,
                     double normal_radius, double gradient_radius, double rift_radius, int n_distance_bins, int n_gradient_bins, float *out_desc,
                     int32_t *out_rows, int64_t cap, int64_t *desc_offsets, int mem, void *stream) {
    if (!idx) return fail(PCC_ERR_INVALID, "idx is NULL");
    if (n < 0 || (n > 0 && (!pts || !intensity)) || stride_bytes < 12 || (stride_bytes & 3) || cap < 0 || (cap > 0 && (!out_desc || !out_rows)) ||
        !cloud_offsets || !desc_offsets)
        return fail(PCC_ERR_INVALID, "bad arguments");
    if (n >= (1ll << 31) - 1) return fail(PCC_ERR_INVALID, "n exceeds int32 indices");
    if (n_clouds < 0 || n_clouds > (1 << 24)) return fail(PCC_ERR_INVALID, "n_clouds = %lld: 0 .. 2^24 clusters are supported", (long long)n_clouds);
    if (cloud_offsets[0] != 0 || cloud_offsets[n_clouds] != n) return fail(PCC_ERR_INVALID, "cloud_offsets must start at 0 and end at n = %lld", (long long)n);
    for (int64_t c = 0; c < n_clouds; ++c)
        if (cloud_offsets[c + 1] < cloud_offsets[c]) return fail(PCC_ERR_INVALID, "cloud_offsets decrease at cluster %lld", (long long)c);
    for (double r : {normal_radius, gradient_radius, rift_radius})
        if (!(r >= 0) || !std::isfinite(r)) return fail(PCC_ERR_INVALID, "radii must be finite and >= 0 (got %g)", r);
    if (n_distance_bins < 1 || n_gradient_bins < 1 || n_distance_bins * n_gradient_bins > 32)
        return fail(PCC_ERR_INVALID, "RIFT bins %d x %d: the histogram holds 1..32 bins (pcl::Histogram<32>)", n_distance_bins, n_gradient_bins);
    PCC_CUDA(cudaSetDevice(idx->device));
    cudaStream_t s = (cudaStream_t)stream;
    const int ns = (int)n_clouds, nb = n_distance_bins * n_gradient_bins;
    for (int c = 0; c <= ns; ++c) desc_offsets[c] = 0;
    if (n == 0) return PCC_OK;
    const double R = std::max(normal_radius, std::max(gradient_radius, rift_radius));
    PCC_TRY(pcc_build(idx, pts, n, stride_bytes, nullptr, 0, (float)R, 0, mem, stream));
    // rift_tab: cloud offsets | survivors per cluster (n_clouds + 1 each)
    PCC_TRY(idx->rift_tab.reserve((size_t)(ns + 1) * 16));
    int64_t *d_coff = idx->rift_tab.as<int64_t>(), *d_bounds = d_coff + ns + 1;
    PCC_CUDA(cudaMemcpyAsync(d_coff, cloud_offsets, (size_t)(ns + 1) * 8, cudaMemcpyHostToDevice, s));
    PCC_TRY(segment_labels(idx, d_coff, ns, s));
    const float *d_int = nullptr;
    PCC_TRY(stage_in(idx->rift_in, intensity, (size_t)n * 4, mem, s, &d_int));
    PCC_TRY(idx->rift_nrm.reserve((size_t)n * 16));
    PCC_TRY(idx->rift_grad.reserve((size_t)n * 16));
    PCC_TRY(idx->rift_desc.reserve((size_t)n * nb * 4));
    float4 *normals = idx->rift_nrm.as<float4>();
    float *desc = idx->rift_desc.as<float>();
    PCC_TRY(rift_segmented(idx, idx->seg_label.as<uint32_t>(), d_int, normal_radius, gradient_radius, rift_radius, n_distance_bins, n_gradient_bins, normals,
                           idx->rift_grad.as<float4>(), desc, s));
    PCC_TRY(idx->rift_pos.reserve((size_t)(n + 1) * 8));
    int64_t *pos = idx->rift_pos.as<int64_t>();
    rift_survivor_kernel<<<nblocks(n + 1, 256), 256, 0, s>>>(normals, desc, n, nb, pos);
    PCC_LAUNCHED();
    PCC_CUDA(cudaGetLastError());
    size_t tmp = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, tmp, pos, pos, (int)(n + 1), s);
    PCC_TRY(idx->rift_tmp.reserve(tmp));
    PCC_CUDA(cub::DeviceScan::ExclusiveSum(idx->rift_tmp.p, tmp, pos, pos, (int)(n + 1), s));
    g_launches += 2;
    rift_seg_bounds_kernel<<<nblocks(ns + 1, 256), 256, 0, s>>>(pos, d_coff, ns, d_bounds);
    PCC_LAUNCHED();
    PCC_CUDA(cudaGetLastError());
    PCC_CUDA(cudaMemcpyAsync(desc_offsets, d_bounds, (size_t)(ns + 1) * 8, cudaMemcpyDeviceToHost, s));
    PCC_CUDA(cudaStreamSynchronize(s));
    const int64_t written = std::min(desc_offsets[ns], cap);
    if (written > 0) {
        float *od = out_desc; int32_t *orow = out_rows;
        if (mem == PCC_HOST) {
            PCC_TRY(idx->rift_out.reserve((size_t)written * nb * 4)); PCC_TRY(idx->rift_row.reserve((size_t)written * 4));
            od = idx->rift_out.as<float>(); orow = idx->rift_row.as<int32_t>();
        }
        rift_scatter_kernel<<<nblocks(n, 256), 256, 0, s>>>(desc, pos, n, nb, d_coff, ns, written, od, orow);
        PCC_LAUNCHED();
        PCC_CUDA(cudaGetLastError());
        if (mem == PCC_HOST) {
            PCC_TRY(copy_out(out_desc, od, (size_t)written * nb * 4, mem, s));
            PCC_TRY(copy_out(out_rows, orow, (size_t)written * 4, mem, s));
            PCC_CUDA(cudaStreamSynchronize(s));
        }
    }
    return PCC_OK;
}

}  // extern "C"
