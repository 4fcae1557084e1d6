// pcc_sift.cu -- SIFT keypoint detection: scale-space extrema and the octave loop.
//
// Replaces pcl::SIFTKeypoint<PointXYZRGB, PointWithScale>::compute as processSift calls it (src/comparator.cpp:449-465) [up].
// Per octave: VoxelGrid of the previous octave's cloud (pcc_voxel_grid) -> index on the result (pcc_build) -> difference-of-
// Gaussians scale space over sorted radius rows (pcc_sift_dog, pcc_radius.cu) -> extrema over k = 25 nearest-neighbour rows
// (pcc_knn + sift_extrema_kernel) -> keypoints.  DESIGN.md section 2 records the reading of PCL's source this restates.
#include <cub/cub.cuh>
#include <algorithm>
#include <cfloat>
#include <cmath>
#include <vector>

#include "pcc_internal.h"

namespace pcc {

static constexpr int kSiftK = 25;          // findScaleSpaceExtrema: const int k = 25
static constexpr int kSiftMaxCols = 15;    // DoG columns: nr_scales_per_octave + 2 <= 15

// findScaleSpaceExtrema: one thread per point.  min / max of every DoG column over the point's k nearest rows (std::min / std::max
// semantics, so a NaN neighbour value never replaces the running extreme), then PCL's test on columns 1 .. nc-2.  flags[row * nc + c]
// = 1 for a keypoint, so a scan over the flags keeps PCL's (point, column) output order.
__global__ void __launch_bounds__(128) sift_extrema_kernel(const int32_t *__restrict__ nbr, int k, const float *__restrict__ dog, int64_t n, int nc,
                                                           float min_contrast, uint32_t *__restrict__ flags) {
    const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= n) return;
    float mn[kSiftMaxCols], mx[kSiftMaxCols];
#pragma unroll
    for (int c = 0; c < kSiftMaxCols; ++c) { mn[c] = FLT_MAX; mx[c] = -FLT_MAX; }
    for (int j = 0; j < k; ++j) {
        const int32_t id = __ldg(nbr + row * k + j);
        if (id < 0) continue;                                   // past min(k, indexed points), or a skipped (non-finite) point
        const float *d = dog + (int64_t)id * nc;
#pragma unroll
        for (int c = 0; c < kSiftMaxCols; ++c) {
            if (c < nc) {
                const float v = __ldg(d + c);
                if (v < mn[c]) mn[c] = v;                       // std::min (min_val, d)
                if (mx[c] < v) mx[c] = v;                       // std::max (max_val, d)
            }
        }
    }
    const float *me = dog + row * nc;
    uint32_t *f = flags + row * nc;
#pragma unroll
    for (int c = 0; c < kSiftMaxCols; ++c) {
        if (c < nc) {
            uint32_t hit = 0;
            if (c >= 1 && c < nc - 1) {
                const float v = me[c];
                if (fabsf(v) >= min_contrast) {
                    if (v == mn[c] && v < mn[c - 1] && v < mn[c + 1]) hit = 1;
                    else if (v == mx[c] && v > mx[c - 1] && v > mx[c + 1]) hit = 1;
                }
            }
            f[c] = hit;
        }
    }
}
__global__ void sift_compact_kernel(const uint32_t *__restrict__ flags, const uint32_t *__restrict__ pos, int64_t m, int nc, int64_t cap,
                                    int32_t *__restrict__ out_row, int32_t *__restrict__ out_col) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m || !flags[i] || (int64_t)pos[i] >= cap) return;
    out_row[pos[i]] = (int32_t)(i / nc);
    out_col[pos[i]] = (int32_t)(i % nc);
}
// user rows -> float4 (x, y, z, packed rgb word), the layout every octave cloud uses (pcc_voxel_grid with stride 16, rgb at 12)
__global__ void sift_pack_kernel(const uint8_t *__restrict__ raw, int stride, int rgb_off, int64_t n, float4 *__restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float *p = (const float *)(raw + i * (int64_t)stride);
    out[i] = make_float4(p[0], p[1], p[2], *(const float *)(raw + i * (int64_t)stride + rgb_off));
}
// SIFTKeypointFieldSelector<PointXYZRGB>: static_cast<float> (299*p.r + 587*p.g + 114*p.b) / 1000.0f
__global__ void sift_values_kernel(const float4 *__restrict__ cloud, int64_t n, float *__restrict__ values) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t w = __float_as_uint(cloud[i].w);
    const int r = (w >> 16) & 255, g = (w >> 8) & 255, b = w & 255;
    values[i] = __fdiv_rn((float)(299 * r + 587 * g + 114 * b), 1000.0f);
}
struct SiftOctaveScales { float s[16]; };
// detectKeypointsForOctave's output: x, y, z of the octave point and scales[column]
__global__ void sift_emit_kernel(const float4 *__restrict__ cloud, const int32_t *__restrict__ rows, const int32_t *__restrict__ cols, int64_t m,
                                 SiftOctaveScales sc, float4 *__restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const float4 p = cloud[rows[i]];
    float scale = 0.f;
#pragma unroll
    for (int c = 0; c < 16; ++c) if (c == cols[i]) scale = sc.s[c];
    out[i] = make_float4(p.x, p.y, p.z, scale);
}


// ---- pcc_sift_keypoints_batched: every segment (cluster) of a concatenated cloud through one octave loop ----
// findScaleSpaceExtrema's k = 25 nearest neighbours of every indexed point among the points of its own segment (seg[sorted position]),
// exact, ties by index: rings grow around the query's cell until the 25th distance lies inside the covered radius.  Rows hold
// min(25, indexed points of the segment) indices, padded with -1 (which sift_extrema_kernel skips).
__global__ void __launch_bounds__(128) sift_seg_knn_kernel(Grid g, const uint32_t *__restrict__ seg, int32_t *__restrict__ nbr) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= g.n) return;
    const float4 q = __ldg(g.pts + t);
    const uint32_t sq = __ldg(seg + t);
    const QueryCell c = locate(g, q.x, q.y, q.z);
    RegList<kSiftK> list;
    list.init();
    int Rin = -1, R = 1;
    for (;;) {
        scan_shell(g, c, Rin, R, [&](uint32_t pos, float4 p) {
            if (__ldg(seg + pos) == sq) list.offer(make_key(dist2(q.x, q.y, q.z, p.x, p.y, p.z), __float_as_uint(p.w)));
        });
        const float cov = covered_d2(g, c, R), kth = key_d2(list.key[kSiftK - 1]);
        if (cov == CUDART_INF_F || kth < cov) break;               // an unseen point has d2 >= cov: it can neither beat nor tie the 25th
        Rin = R; R = next_ring(g, R, kth);
    }
    int32_t *o = nbr + (int64_t)__float_as_int(q.w) * kSiftK;
#pragma unroll
    for (int j = 0; j < kSiftK; ++j) o[j] = key_idx(list.key[j]);
}
// keypoints of one octave per segment: the exclusive scan of the flags at each segment's first DoG entry (off[n_seg] gives the total)
__global__ void sift_seg_bounds_kernel(const uint32_t *__restrict__ flags, const uint32_t *__restrict__ pos, int64_t m, const int64_t *__restrict__ off, int n_seg,
                                       int nc, uint32_t *__restrict__ out) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c > n_seg) return;
    const int64_t b = off[c] * nc;
    out[c] = b < m ? pos[b] : pos[m - 1] + flags[m - 1];
}
// staged keypoints (octave-major, segment-minor blocks starting at src[b]) -> (segment, octave) order: block b starts at dst[b];
// rows at or past cap are dropped
__global__ void sift_seg_reorder_kernel(const float4 *__restrict__ stage, int64_t m, const int64_t *__restrict__ src, const int64_t *__restrict__ dst, int n_blocks,
                                        int64_t cap, float4 *__restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const uint32_t b = segment_of(src, n_blocks, i);
    const int64_t d = dst[b] + (i - src[b]);
    if (d < cap) out[d] = stage[i];
}

}  // namespace pcc

using namespace pcc;

// grow `b` to `bytes`, keeping its first `used` bytes (Buf::reserve drops them)
static int reserve_keep(Buf &b, size_t used, size_t bytes, cudaStream_t s) {
    if (bytes <= b.cap) return PCC_OK;
    Buf nb;
    PCC_TRY(nb.reserve(bytes));
    if (used) PCC_CUDA(cudaMemcpyAsync(nb.p, b.p, used, cudaMemcpyDeviceToDevice, s));
    PCC_CUDA(cudaStreamSynchronize(s));
    b.release();
    b = nb;
    return PCC_OK;
}

extern "C" {

int pcc_sift_extrema(pcc_index *idx, const float *dog, int n_cols, float min_contrast, int32_t *out_row, int32_t *out_col, int64_t cap, int64_t *n_found,
                     int mem, void *stream) {
    PCC_TRY(check_index(idx, stream));
    if (n_cols < 1 || n_cols > kSiftMaxCols) return fail(PCC_ERR_INVALID, "SIFT DoG of %d columns: 1..%d are supported", n_cols, kSiftMaxCols);
    if (!n_found || cap < 0 || (cap > 0 && (!out_row || !out_col)) || !(min_contrast >= 0.f)) return fail(PCC_ERR_INVALID, "bad arguments");
    cudaStream_t s = (cudaStream_t)stream;
    *n_found = 0;
    const int64_t n = idx->n_input, m = n * n_cols;
    if (n == 0) return PCC_OK;
    if (!dog) return fail(PCC_ERR_INVALID, "dog is NULL");
    if (m >= (1ll << 31) - 1) return fail(PCC_ERR_INVALID, "%lld DoG entries exceed the 32-bit scan", (long long)m);
    const float *d_dog = nullptr;
    PCC_TRY(stage_in(idx->sift_in, dog, (size_t)m * 4, mem, s, &d_dog));
    const int k = (int)std::min<int64_t>(kSiftK, std::max<int64_t>(idx->n_indexed, 1));       // nearestKSearch returns min(k, size) rows
    PCC_TRY(idx->sift_nbr.reserve((size_t)n * k * 4));
    PCC_TRY(idx->sift_d2.reserve((size_t)n * k * 4));
    PCC_TRY(idx->sift_flag.reserve((size_t)m * 4));
    PCC_TRY(idx->sift_pos.reserve((size_t)m * 4));
    uint32_t *flags = idx->sift_flag.as<uint32_t>(), *pos = idx->sift_pos.as<uint32_t>();
    // the timed span starts at the kNN (whose own timer re-records the start event with nothing enqueued in between)
    KernelTimer timer(idx, s);
    int k_eff = 0;
    PCC_TRY(pcc_knn(idx, nullptr, 0, 16, k, idx->sift_nbr.as<int32_t>(), idx->sift_d2.as<float>(), &k_eff, PCC_DEVICE, stream));
    sift_extrema_kernel<<<nblocks(n, 128), 128, 0, s>>>(idx->sift_nbr.as<int32_t>(), k, d_dog, n, n_cols, min_contrast, flags);
    PCC_LAUNCHED();
    PCC_CUDA(cudaGetLastError());
    size_t tmp = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, tmp, flags, pos, (int)m, s);
    PCC_TRY(idx->cub_tmp.reserve(tmp));
    PCC_CUDA(cub::DeviceScan::ExclusiveSum(idx->cub_tmp.p, tmp, flags, pos, (int)m, s));
    g_launches += 2;
    uint32_t *h = (uint32_t *)idx->h_pinned;
    PCC_CUDA(cudaMemcpyAsync(h, pos + (m - 1), 4, cudaMemcpyDeviceToHost, s));
    PCC_CUDA(cudaMemcpyAsync(h + 1, flags + (m - 1), 4, cudaMemcpyDeviceToHost, s));
    PCC_CUDA(cudaStreamSynchronize(s));
    const int64_t total = (int64_t)h[0] + h[1];
    const int64_t written = std::min(total, cap);
    if (written > 0) {
        int32_t *orow = out_row, *ocol = out_col;
        if (mem == PCC_HOST) {
            PCC_TRY(idx->sift_row.reserve((size_t)written * 4)); PCC_TRY(idx->sift_col.reserve((size_t)written * 4));
            orow = idx->sift_row.as<int32_t>(); ocol = idx->sift_col.as<int32_t>();
        }
        sift_compact_kernel<<<nblocks(m, 256), 256, 0, s>>>(flags, pos, m, n_cols, written, orow, ocol);
        PCC_LAUNCHED();
        PCC_CUDA(cudaGetLastError());
        if (mem == PCC_HOST) {
            PCC_TRY(copy_out(out_row, orow, (size_t)written * 4, mem, s));
            PCC_TRY(copy_out(out_col, ocol, (size_t)written * 4, mem, s));
            PCC_CUDA(cudaStreamSynchronize(s));
        }
    }
    timer.stop();
    *n_found = total;
    return PCC_OK;
}

int pcc_sift_keypoints(pcc_index *idx, const void *pts, int64_t n, int stride_bytes, int rgb_offset_bytes, float min_scale, int nr_octaves,
                       int nr_scales_per_octave, float min_contrast, float *out4, int64_t cap, int64_t *n_keypoints, int mem, void *stream) {
    if (!idx) return fail(PCC_ERR_INVALID, "idx is NULL");
    if (n < 0 || (n > 0 && !pts) || stride_bytes < 16 || (stride_bytes & 3) || !n_keypoints || cap < 0 || (cap > 0 && !out4))
        return fail(PCC_ERR_INVALID, "bad arguments");
    if (rgb_offset_bytes < 12 || (rgb_offset_bytes & 3) || rgb_offset_bytes + 4 > stride_bytes) return fail(PCC_ERR_INVALID, "bad rgb offset %d", rgb_offset_bytes);
    // SIFTKeypoint::initCompute's checks, plus this implementation's register budget (nr_scales_per_octave + 3 <= 16 scales)
    if (!(min_scale > 0.f) || nr_octaves < 1 || nr_scales_per_octave < 1 || !(min_contrast >= 0.f))
        return fail(PCC_ERR_INVALID, "SIFT parameters: min_scale > 0, nr_octaves >= 1, nr_scales_per_octave >= 1 and min_contrast >= 0 are required");
    if (nr_scales_per_octave > 13) return fail(PCC_ERR_INVALID, "nr_scales_per_octave = %d: at most 13 are supported (16 scales)", nr_scales_per_octave);
    if (n >= (1ll << 31) - 1) return fail(PCC_ERR_INVALID, "n exceeds int32 indices");
    PCC_CUDA(cudaSetDevice(idx->device));
    cudaStream_t s = (cudaStream_t)stream;
    *n_keypoints = 0;
    if (n == 0) return PCC_OK;
    const int ns = nr_scales_per_octave + 3, nc = ns - 1;
    // octave 0's "previous cloud" is the input, repacked to the octave layout
    PCC_TRY(idx->sift_cloud[0].reserve((size_t)n * 16));
    PCC_TRY(idx->sift_cloud[1].reserve(std::max<size_t>((size_t)n * 16, (size_t)n * stride_bytes)));
    const uint8_t *raw = (const uint8_t *)pts;
    if (mem == PCC_HOST) {
        PCC_CUDA(cudaMemcpyAsync(idx->sift_cloud[1].p, pts, (size_t)n * stride_bytes, cudaMemcpyHostToDevice, s));
        raw = idx->sift_cloud[1].as<uint8_t>();
    }
    sift_pack_kernel<<<nblocks(n, 256), 256, 0, s>>>(raw, stride_bytes, rgb_offset_bytes, n, idx->sift_cloud[0].as<float4>());
    PCC_LAUNCHED();
    PCC_CUDA(cudaGetLastError());
    int cur = 0;
    int64_t n_cur = n, total = 0;
    float scale = min_scale;
    for (int octave = 0; octave < nr_octaves; ++octave) {
        const float leaf[3] = {1.0f * scale, 1.0f * scale, 1.0f * scale};
        int64_t n_next = 0;
        PCC_TRY(pcc_voxel_grid(idx, idx->sift_cloud[cur].p, n_cur, 16, 12, leaf, 0, idx->sift_cloud[1 - cur].p, &n_next, PCC_DEVICE, stream));
        cur = 1 - cur;
        n_cur = n_next;
        if (n_cur < 25) break;                                  // const size_t min_nr_points = 25
        SiftOctaveScales sc{};
        for (int i = 0; i < ns; ++i) sc.s[i] = scale * powf(2.0f, (1.0f * static_cast<float>(i) - 1.0f) / static_cast<float>(nr_scales_per_octave));
        const float4 *cloud = idx->sift_cloud[cur].as<float4>();
        PCC_TRY(pcc_build(idx, cloud, n_cur, 16, nullptr, 0, 3.0f * sc.s[ns - 1], 0, PCC_DEVICE, stream));
        PCC_TRY(idx->sift_val.reserve((size_t)n_cur * 4));
        sift_values_kernel<<<nblocks(n_cur, 256), 256, 0, s>>>(cloud, n_cur, idx->sift_val.as<float>());
        PCC_LAUNCHED();
        PCC_CUDA(cudaGetLastError());
        PCC_TRY(idx->sift_dog.reserve((size_t)n_cur * nc * 4));
        float *dog = idx->sift_dog.as<float>();
        PCC_TRY(pcc_sift_dog(idx, idx->sift_val.as<float>(), sc.s, ns, dog, PCC_DEVICE, stream));
        const int64_t cap_oct = n_cur * nc;
        PCC_TRY(idx->sift_row.reserve((size_t)cap_oct * 4)); PCC_TRY(idx->sift_col.reserve((size_t)cap_oct * 4));
        int64_t found = 0;
        PCC_TRY(pcc_sift_extrema(idx, dog, nc, min_contrast, idx->sift_row.as<int32_t>(), idx->sift_col.as<int32_t>(), cap_oct, &found, PCC_DEVICE, stream));
        const int64_t room = std::max<int64_t>(0, std::min(found, cap - total));
        if (room > 0) {
            float4 *o = (float4 *)out4 + total;
            if (mem == PCC_HOST) { PCC_TRY(idx->sift_kp.reserve((size_t)room * 16)); o = idx->sift_kp.as<float4>(); }
            sift_emit_kernel<<<nblocks(room, 128), 128, 0, s>>>(cloud, idx->sift_row.as<int32_t>(), idx->sift_col.as<int32_t>(), room, sc, o);
            PCC_LAUNCHED();
            PCC_CUDA(cudaGetLastError());
            if (mem == PCC_HOST) { PCC_TRY(copy_out(out4 + total * 4, o, (size_t)room * 16, mem, s)); PCC_CUDA(cudaStreamSynchronize(s)); }
        }
        total += found;
        scale *= 2;
    }
    if (mem != PCC_HOST) PCC_CUDA(cudaStreamSynchronize(s));
    *n_keypoints = total;
    return PCC_OK;
}

int pcc_sift_keypoints_batched(pcc_index *idx, const void *pts, int64_t n, int stride_bytes, int rgb_offset_bytes, const int64_t *cloud_offsets, int64_t n_clouds,
                               float min_scale, int nr_octaves, int nr_scales_per_octave, float min_contrast, double snap_threshold, float *out4, int32_t *snap,
                               int64_t cap, int64_t *kp_offsets, int mem, void *stream) {
    if (!idx) return fail(PCC_ERR_INVALID, "idx is NULL");
    if (n < 0 || (n > 0 && !pts) || stride_bytes < 16 || (stride_bytes & 3) || cap < 0 || (cap > 0 && !out4) || !cloud_offsets || !kp_offsets)
        return fail(PCC_ERR_INVALID, "bad arguments");
    if (rgb_offset_bytes < 12 || (rgb_offset_bytes & 3) || rgb_offset_bytes + 4 > stride_bytes) return fail(PCC_ERR_INVALID, "bad rgb offset %d", rgb_offset_bytes);
    if (!(min_scale > 0.f) || nr_octaves < 1 || nr_scales_per_octave < 1 || !(min_contrast >= 0.f))
        return fail(PCC_ERR_INVALID, "SIFT parameters: min_scale > 0, nr_octaves >= 1, nr_scales_per_octave >= 1 and min_contrast >= 0 are required");
    if (nr_scales_per_octave > 13) return fail(PCC_ERR_INVALID, "nr_scales_per_octave = %d: at most 13 are supported (16 scales)", nr_scales_per_octave);
    if (n >= (1ll << 31) - 1) return fail(PCC_ERR_INVALID, "n exceeds int32 indices");
    if (n_clouds < 0 || n_clouds > (1 << 24)) return fail(PCC_ERR_INVALID, "n_clouds = %lld: 0 .. 2^24 clusters are supported", (long long)n_clouds);
    if (cloud_offsets[0] != 0 || cloud_offsets[n_clouds] != n) return fail(PCC_ERR_INVALID, "cloud_offsets must start at 0 and end at n = %lld", (long long)n);
    for (int64_t c = 0; c < n_clouds; ++c)
        if (cloud_offsets[c + 1] < cloud_offsets[c]) return fail(PCC_ERR_INVALID, "cloud_offsets decrease at cluster %lld", (long long)c);
    if (snap && !(snap_threshold >= 0)) return fail(PCC_ERR_INVALID, "bad snap threshold");
    PCC_CUDA(cudaSetDevice(idx->device));
    cudaStream_t s = (cudaStream_t)stream;
    const int ns_ = (int)n_clouds;
    for (int c = 0; c <= ns_; ++c) kp_offsets[c] = 0;
    if (n == 0) return PCC_OK;
    const int ns = nr_scales_per_octave + 3, nc = ns - 1;
    // octave 0's "previous cloud" is the input, repacked to the octave layout (as pcc_sift_keypoints)
    PCC_TRY(idx->sift_cloud[0].reserve((size_t)n * 16));
    PCC_TRY(idx->sift_cloud[1].reserve(std::max<size_t>((size_t)n * 16, (size_t)n * stride_bytes)));
    const uint8_t *raw = (const uint8_t *)pts;
    if (mem == PCC_HOST) {
        PCC_CUDA(cudaMemcpyAsync(idx->sift_cloud[1].p, pts, (size_t)n * stride_bytes, cudaMemcpyHostToDevice, s));
        raw = idx->sift_cloud[1].as<uint8_t>();
    }
    sift_pack_kernel<<<nblocks(n, 256), 256, 0, s>>>(raw, stride_bytes, rgb_offset_bytes, n, idx->sift_cloud[0].as<float4>());
    PCC_LAUNCHED();
    PCC_CUDA(cudaGetLastError());
    std::vector<int64_t> off(cloud_offsets, cloud_offsets + ns_ + 1), next((size_t)ns_ + 1);
    std::vector<std::vector<int64_t> > counts;                   // [octave][cluster] keypoints
    std::vector<uint32_t> bounds((size_t)ns_ + 1);
    PCC_TRY(idx->seg_off.reserve((size_t)(ns_ + 1) * 12));
    int64_t *d_off = idx->seg_off.as<int64_t>();
    uint32_t *d_bounds = (uint32_t *)(d_off + ns_ + 1);
    int cur = 0;
    int64_t staged = 0;
    float scale = min_scale;
    for (int octave = 0; octave < nr_octaves; ++octave) {
        // VoxelGrid of every cluster's previous cloud; a cluster whose result has fewer than 25 points leaves the loop here, as its
        // own detectKeypoints would (const size_t min_nr_points = 25)
        PCC_TRY(segmented_voxel_grid(idx, idx->sift_cloud[cur].as<float4>(), off.data(), ns_, 1.0f * scale, 25, idx->sift_cloud[1 - cur].as<float4>(), next.data(), s));
        cur = 1 - cur;
        off.swap(next);
        const int64_t n_cur = off[ns_];
        if (n_cur == 0) break;
        SiftOctaveScales sc{};
        for (int i = 0; i < ns; ++i) sc.s[i] = scale * powf(2.0f, (1.0f * static_cast<float>(i) - 1.0f) / static_cast<float>(nr_scales_per_octave));
        const float4 *cloud = idx->sift_cloud[cur].as<float4>();
        PCC_TRY(pcc_build(idx, cloud, n_cur, 16, nullptr, 0, 3.0f * sc.s[ns - 1], 0, PCC_DEVICE, stream));
        PCC_CUDA(cudaMemcpyAsync(d_off, off.data(), (size_t)(ns_ + 1) * 8, cudaMemcpyHostToDevice, s));
        PCC_TRY(segment_labels(idx, d_off, ns_, s));
        const uint32_t *seg = idx->seg_label.as<uint32_t>();
        PCC_TRY(idx->sift_val.reserve((size_t)n_cur * 4));
        sift_values_kernel<<<nblocks(n_cur, 256), 256, 0, s>>>(cloud, n_cur, idx->sift_val.as<float>());
        PCC_LAUNCHED();
        PCC_TRY(idx->sift_dog.reserve((size_t)n_cur * nc * 4));
        float *dog = idx->sift_dog.as<float>();
        PCC_TRY(sift_dog_segmented(idx, seg, idx->sift_val.as<float>(), sc.s, ns, dog, s));
        // extrema over the clusters' own k = 25 neighbours, flags in (cluster, point, column) order
        const int64_t m = n_cur * nc;
        if (m >= (1ll << 31) - 1) return fail(PCC_ERR_INVALID, "%lld DoG entries exceed the 32-bit scan", (long long)m);
        PCC_TRY(idx->sift_nbr.reserve((size_t)n_cur * kSiftK * 4));
        int32_t *nbr = idx->sift_nbr.as<int32_t>();
        if (!idx->all_rows_indexed) PCC_CUDA(cudaMemsetAsync(nbr, 0xFF, (size_t)n_cur * kSiftK * 4, s));
        if (idx->n_indexed > 0) { sift_seg_knn_kernel<<<nblocks(idx->n_indexed, 128), 128, 0, s>>>(idx->grid(), seg, nbr); PCC_LAUNCHED(); }
        PCC_TRY(idx->sift_flag.reserve((size_t)m * 4));
        PCC_TRY(idx->sift_pos.reserve((size_t)m * 4));
        uint32_t *flags = idx->sift_flag.as<uint32_t>(), *pos = idx->sift_pos.as<uint32_t>();
        sift_extrema_kernel<<<nblocks(n_cur, 128), 128, 0, s>>>(nbr, kSiftK, dog, n_cur, nc, min_contrast, flags);
        PCC_LAUNCHED();
        PCC_CUDA(cudaGetLastError());
        size_t tmp = 0;
        cub::DeviceScan::ExclusiveSum(nullptr, tmp, flags, pos, (int)m, s);
        PCC_TRY(idx->cub_tmp.reserve(tmp));
        PCC_CUDA(cub::DeviceScan::ExclusiveSum(idx->cub_tmp.p, tmp, flags, pos, (int)m, s));
        g_launches += 2;
        sift_seg_bounds_kernel<<<nblocks(ns_ + 1, 256), 256, 0, s>>>(flags, pos, m, d_off, ns_, nc, d_bounds);
        PCC_LAUNCHED();
        PCC_CUDA(cudaGetLastError());
        PCC_CUDA(cudaMemcpyAsync(bounds.data(), d_bounds, (size_t)(ns_ + 1) * 4, cudaMemcpyDeviceToHost, s));
        PCC_CUDA(cudaStreamSynchronize(s));
        const int64_t found = (int64_t)bounds[ns_];
        counts.emplace_back((size_t)ns_);
        for (int c = 0; c < ns_; ++c) counts.back()[c] = (int64_t)bounds[c + 1] - bounds[c];
        if (found > 0) {
            PCC_TRY(idx->sift_row.reserve((size_t)found * 4)); PCC_TRY(idx->sift_col.reserve((size_t)found * 4));
            sift_compact_kernel<<<nblocks(m, 256), 256, 0, s>>>(flags, pos, m, nc, found, idx->sift_row.as<int32_t>(), idx->sift_col.as<int32_t>());
            PCC_LAUNCHED();
            PCC_TRY(reserve_keep(idx->sift_stage, (size_t)staged * 16, (size_t)(staged + found) * 16, s));
            sift_emit_kernel<<<nblocks(found, 128), 128, 0, s>>>(cloud, idx->sift_row.as<int32_t>(), idx->sift_col.as<int32_t>(), found, sc, idx->sift_stage.as<float4>() + staged);
            PCC_LAUNCHED();
            PCC_CUDA(cudaGetLastError());
            staged += found;
        }
        scale *= 2;
    }
    // (octave, cluster) blocks of the staged keypoints -> their place in (cluster, octave) order
    const int n_oct = (int)counts.size(), n_blocks = n_oct * ns_;
    std::vector<int64_t> src((size_t)n_blocks + 1), dst((size_t)n_blocks + 1);
    for (int c = 0; c < ns_; ++c) {
        int64_t k = 0;
        for (int o = 0; o < n_oct; ++o) k += counts[o][c];
        kp_offsets[c + 1] = kp_offsets[c] + k;
    }
    {
        int64_t at = 0;
        std::vector<int64_t> fill(kp_offsets, kp_offsets + ns_);
        for (int o = 0; o < n_oct; ++o)
            for (int c = 0; c < ns_; ++c) { src[(size_t)o * ns_ + c] = at; dst[(size_t)o * ns_ + c] = fill[c]; at += counts[o][c]; fill[c] += counts[o][c]; }
        src[n_blocks] = at; dst[n_blocks] = at;
    }
    const int64_t written = std::min(staged, cap);
    if (written > 0) {
        // sift_tab: src | dst (n_blocks + 1 each) | cloud offsets | keypoint offsets (n_clouds + 1 each)
        PCC_TRY(idx->sift_tab.reserve((size_t)(2 * (n_blocks + 1) + 2 * (ns_ + 1)) * 8));
        int64_t *d_src = idx->sift_tab.as<int64_t>(), *d_dst = d_src + n_blocks + 1, *d_coff = d_dst + n_blocks + 1, *d_koff = d_coff + ns_ + 1;
        PCC_CUDA(cudaMemcpyAsync(d_src, src.data(), (size_t)(n_blocks + 1) * 8, cudaMemcpyHostToDevice, s));
        PCC_CUDA(cudaMemcpyAsync(d_dst, dst.data(), (size_t)(n_blocks + 1) * 8, cudaMemcpyHostToDevice, s));
        float4 *o = (float4 *)out4;
        if (mem == PCC_HOST) { PCC_TRY(idx->sift_kp.reserve((size_t)written * 16)); o = idx->sift_kp.as<float4>(); }
        sift_seg_reorder_kernel<<<nblocks(staged, 256), 256, 0, s>>>(idx->sift_stage.as<float4>(), staged, d_src, d_dst, n_blocks, written, o);
        PCC_LAUNCHED();
        PCC_CUDA(cudaGetLastError());
        if (mem == PCC_HOST) PCC_TRY(copy_out(out4, o, (size_t)written * 16, mem, s));
        if (snap) {
            // processRIFTwithSIFT's snap, per cluster: an index over the input with segment labels, first point of the keypoint's
            // own cluster within snap_threshold
            PCC_TRY(pcc_build(idx, pts, n, stride_bytes, nullptr, 0, (float)snap_threshold, 0, mem, stream));
            PCC_CUDA(cudaMemcpyAsync(d_coff, cloud_offsets, (size_t)(ns_ + 1) * 8, cudaMemcpyHostToDevice, s));
            PCC_CUDA(cudaMemcpyAsync(d_koff, kp_offsets, (size_t)(ns_ + 1) * 8, cudaMemcpyHostToDevice, s));
            PCC_TRY(segment_labels(idx, d_coff, ns_, s));
            int32_t *sp = snap;
            if (mem == PCC_HOST) { PCC_TRY(idx->out_i.reserve((size_t)written * 4)); sp = idx->out_i.as<int32_t>(); }
            PCC_TRY(first_within_segmented(idx, idx->seg_label.as<uint32_t>(), o, written, d_koff, d_coff, ns_, snap_threshold, sp, s));
            if (mem == PCC_HOST) PCC_TRY(copy_out(snap, sp, (size_t)written * 4, mem, s));
        }
    }
    PCC_CUDA(cudaStreamSynchronize(s));
    return PCC_OK;
}

}  // extern "C"
