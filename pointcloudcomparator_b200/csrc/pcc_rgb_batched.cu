// pcc_rgb_batched.cu -- RegionGrowingRGB::findPointNeighbours and the colour segmentation of every cluster of a concatenated cloud in one
// call.
//
// computeSimilarity runs color_growing_segmentation on both clouds of every matched cluster pair (src/comparator.cpp:1457-1460 ->
// src/segmentation.cpp:161-216).  Here one index over the union, a cluster label per sorted position (segment_labels) and one
// segment-restricted selection pass (knn_select_segmented, pcc_radius.cu) replace the per-cluster index builds and k = 100 searches; the
// order-dependent grow / merge then runs on the host over each cluster's slice of the table, unchanged.  Host round trips do not depend
// on the cluster count.
#include <algorithm>
#include <memory>

#include "pcc_internal.h"

namespace pcc {

// finite points per segment: seg_n (pre-zeroed) counts the segment labels of the indexed points.  Positions are in cell order, so the
// lanes of a warp mostly share a few segments: one atomic per distinct segment of the warp, by its lowest lane, keeps one large cluster
// from serialising on a single counter.  Launched with whole warps (blockDim a multiple of 32).
__global__ void seg_count_kernel(const uint32_t *__restrict__ seg, int64_t n, uint32_t *__restrict__ seg_n) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = t < n;
    const uint32_t s = live ? __ldg(seg + t) : 0xFFFFFFFFu;
    const unsigned peers = __match_any_sync(0xFFFFFFFFu, s);
    if (live && (int)(threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(seg_n + s, (unsigned)__popc(peers));
}

static int check_batch(pcc_index *idx, const void *pts, int64_t n, int stride_bytes, const int64_t *cloud_offsets, int64_t n_clouds, int k) {
    if (!idx) return fail(PCC_ERR_INVALID, "idx is NULL");
    if (n < 0 || (n > 0 && !pts) || stride_bytes < 12 || (stride_bytes & 3) || !cloud_offsets) return fail(PCC_ERR_INVALID, "bad arguments");
    if (n >= (1ll << 31) - 1) return fail(PCC_ERR_INVALID, "n exceeds int32 indices");
    if (k < 1 || k > PCC_MAX_K) return fail(PCC_ERR_INVALID, "k=%d outside 1..%d", k, PCC_MAX_K);
    if (n_clouds < 0 || n_clouds > (1 << 24)) return fail(PCC_ERR_INVALID, "n_clouds = %lld: 0 .. 2^24 clusters are supported", (long long)n_clouds);
    if (cloud_offsets[0] != 0 || cloud_offsets[n_clouds] != n) return fail(PCC_ERR_INVALID, "cloud_offsets must start at 0 and end at n = %lld", (long long)n);
    for (int64_t c = 0; c < n_clouds; ++c)
        if (cloud_offsets[c + 1] < cloud_offsets[c]) return fail(PCC_ERR_INVALID, "cloud_offsets decrease at cluster %lld", (long long)c);
    return PCC_OK;
}

// the [n, k] table of every cluster (n > 0) into device memory: *oi / *od, or out_i / out_f when they are NULL.  k_eff (host, n_clouds)
// gets min(k, finite points) per cluster.  Leaves idx indexing the concatenated input.
static int knn_batched_table(pcc_index *idx, const void *pts, int64_t n, int stride_bytes, const int64_t *cloud_offsets, int ns, int k, int32_t **oi,
                             float **od, int32_t *k_eff, int mem, cudaStream_t s) {
    PCC_TRY(pcc_build(idx, pts, n, stride_bytes, nullptr, 0, 0.f, k, mem, s));
    // knnb_tab: cloud offsets (n_clouds + 1 int64) | finite points per cluster (n_clouds uint32)
    PCC_TRY(idx->knnb_tab.reserve((size_t)(ns + 1) * 8 + (size_t)ns * 4));
    int64_t *d_coff = idx->knnb_tab.as<int64_t>();
    uint32_t *d_cnt = reinterpret_cast<uint32_t *>(d_coff + ns + 1);
    PCC_CUDA(cudaMemcpyAsync(d_coff, cloud_offsets, (size_t)(ns + 1) * 8, cudaMemcpyHostToDevice, s));
    PCC_TRY(segment_labels(idx, d_coff, ns, s));
    const uint32_t *seg = idx->seg_label.as<uint32_t>();
    PCC_CUDA(cudaMemsetAsync(d_cnt, 0, (size_t)ns * 4, s));
    if (idx->n_indexed > 0) {
        seg_count_kernel<<<nblocks(idx->n_indexed, 256), 256, 0, s>>>(seg, idx->n_indexed, d_cnt);
        PCC_LAUNCHED();
        PCC_CUDA(cudaGetLastError());
    }
    PCC_CUDA(cudaMemcpyAsync(k_eff, d_cnt, (size_t)ns * 4, cudaMemcpyDeviceToHost, s));
    if (!*oi) {
        PCC_TRY(idx->out_i.reserve((size_t)n * k * 4)); PCC_TRY(idx->out_f.reserve((size_t)n * k * 4));
        *oi = idx->out_i.as<int32_t>(); *od = idx->out_f.as<float>();
    }
    PCC_TRY(knn_select_segmented(idx, seg, d_cnt, d_coff, k, *oi, *od, s));      // synchronises s: k_eff holds the counts
    for (int c = 0; c < ns; ++c) k_eff[c] = std::min(k_eff[c], k);
    return PCC_OK;
}

}  // namespace pcc

using namespace pcc;

extern "C" {

int pcc_knn_batched(pcc_index *idx, const void *pts, int64_t n, int stride_bytes, const int64_t *cloud_offsets, int64_t n_clouds, int k, int32_t *out_idx,
                    float *out_d2, int32_t *k_eff, int mem, void *stream) {
    PCC_TRY(check_batch(idx, pts, n, stride_bytes, cloud_offsets, n_clouds, k));
    if (!k_eff || (n > 0 && (!out_idx || !out_d2))) return fail(PCC_ERR_INVALID, "output pointers are NULL");
    PCC_CUDA(cudaSetDevice(idx->device));
    cudaStream_t s = (cudaStream_t)stream;
    const int ns = (int)n_clouds;
    std::fill(k_eff, k_eff + ns, 0);
    if (n == 0) return PCC_OK;
    int32_t *oi = mem == PCC_HOST ? nullptr : out_idx;
    float *od = mem == PCC_HOST ? nullptr : out_d2;
    PCC_TRY(knn_batched_table(idx, pts, n, stride_bytes, cloud_offsets, ns, k, &oi, &od, k_eff, mem, s));
    if (mem == PCC_HOST) {
        PCC_TRY(copy_out(out_idx, oi, (size_t)n * k * 4, mem, s));
        PCC_TRY(copy_out(out_d2, od, (size_t)n * k * 4, mem, s));
        PCC_CUDA(cudaStreamSynchronize(s));
    }
    return PCC_OK;
}

int pcc_region_growing_rgb_batched(pcc_index *idx, const void *pts, int64_t n, int stride_bytes, int rgb_offset_bytes, const int64_t *cloud_offsets,
                                   int64_t n_clouds, int k, float distance_threshold, float point_color_threshold, float region_color_threshold,
                                   int grow_neighbours, int64_t min_size, int64_t max_size, int32_t *labels, int64_t *n_clusters, int mem, void *stream) {
    PCC_TRY(check_batch(idx, pts, n, stride_bytes, cloud_offsets, n_clouds, k));
    if (rgb_offset_bytes < 12 || (rgb_offset_bytes & 3) || rgb_offset_bytes + 4 > stride_bytes) return fail(PCC_ERR_INVALID, "bad rgb offset %d", rgb_offset_bytes);
    if (grow_neighbours < 1) return fail(PCC_ERR_INVALID, "grow_neighbours=%d < 1", grow_neighbours);
    if (!n_clusters || (n > 0 && !labels)) return fail(PCC_ERR_INVALID, "output pointers are NULL");
    PCC_CUDA(cudaSetDevice(idx->device));
    cudaStream_t s = (cudaStream_t)stream;
    const int ns = (int)n_clouds;
    std::fill(n_clusters, n_clusters + ns, (int64_t)0);
    if (n == 0) return PCC_OK;
    int32_t *oi = nullptr; float *od = nullptr;
    std::unique_ptr<int32_t[]> keff(new int32_t[(size_t)ns + 1]);
    PCC_TRY(knn_batched_table(idx, pts, n, stride_bytes, cloud_offsets, ns, k, &oi, &od, keff.get(), mem, s));
    const size_t cells = (size_t)n * k;
    std::unique_ptr<int32_t[]> nb(new int32_t[cells]);
    std::unique_ptr<float[]> nd(new float[cells]);
    PCC_CUDA(cudaMemcpyAsync(nb.get(), oi, cells * 4, cudaMemcpyDeviceToHost, s));
    PCC_CUDA(cudaMemcpyAsync(nd.get(), od, cells * 4, cudaMemcpyDeviceToHost, s));
    const uint8_t *rows = static_cast<const uint8_t *>(pts);
    std::unique_ptr<uint8_t[]> staged;
    if (mem != PCC_HOST) {          // the colour words are read on the host: bring the rows over
        staged.reset(new uint8_t[(size_t)n * stride_bytes]);
        PCC_CUDA(cudaMemcpyAsync(staged.get(), pts, (size_t)n * stride_bytes, cudaMemcpyDeviceToHost, s));
        rows = staged.get();
    }
    PCC_CUDA(cudaStreamSynchronize(s));
    for (int c = 0; c < ns; ++c) {
        const int64_t b = cloud_offsets[c], m = cloud_offsets[c + 1] - b;
        PCC_TRY(pcc_region_growing_rgb(nb.get() + (size_t)b * k, nd.get() + (size_t)b * k, m, k,
                                       reinterpret_cast<const uint32_t *>(rows + (size_t)b * stride_bytes + rgb_offset_bytes), stride_bytes, distance_threshold,
                                       point_color_threshold, region_color_threshold, grow_neighbours, min_size, max_size, labels + b, n_clusters + c));
    }
    return PCC_OK;
}

}  // extern "C"
