// pcc_voxel.cu -- VoxelGrid downsampling on the GPU (SURVEY.md section 8f, "next" row 1).
//
// Replaces pcl::VoxelGrid<PointXYZRGB>::applyFilter [up] as the reference calls it right before every segmentation
// search (src/segmentation.cpp:69-74 and :223-228, leaf 0.025): voxel key per finite point -> sort -> one centroid per
// occupied voxel, output ordered by voxel key (x fastest).  Same machinery as the grid build: keys, radix sort, scan.
// PCL's std::sort leaves the order of points inside a voxel unspecified; here the sort is stable, so a centroid is the
// fp32 sum of its points in ascending original index (the oracle sums in the same order -> bit-exact parity), and the
// r/g/b sums are exact integers in fp32 whatever the order.
#include <cub/cub.cuh>
#include <algorithm>
#include <cmath>
#include <cstring>
#include <vector>

#include "pcc_internal.h"

namespace pcc {

struct VoxelParams { float inv[3]; int min_b[3]; int mul[3]; };

__device__ __forceinline__ int f2ord_v(float f) { int i = __float_as_int(f); return i >= 0 ? i : i ^ 0x7FFFFFFF; }
// getMinMax3D over finite points
__global__ void voxel_minmax_kernel(const uint8_t *__restrict__ raw, int stride, int64_t n, int *__restrict__ bbox, unsigned long long *__restrict__ n_finite) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int lo[3] = {INT_MAX, INT_MAX, INT_MAX}, hi[3] = {INT_MIN, INT_MIN, INT_MIN};
    unsigned fin = 0;
    if (i < n) {
        const float *p = (const float *)(raw + i * (int64_t)stride);
        if (finite3(p[0], p[1], p[2])) { fin = 1; for (int d = 0; d < 3; ++d) lo[d] = hi[d] = f2ord_v(p[d]); }
    }
#pragma unroll
    for (int d = 0; d < 3; ++d) { lo[d] = __reduce_min_sync(0xffffffffu, lo[d]); hi[d] = __reduce_max_sync(0xffffffffu, hi[d]); }
    fin = __reduce_add_sync(0xffffffffu, fin);
    if ((threadIdx.x & 31) == 0 && fin) {
#pragma unroll
        for (int d = 0; d < 3; ++d) { atomicMin(bbox + d, lo[d]); atomicMax(bbox + 3 + d, hi[d]); }
        atomicAdd(n_finite, (unsigned long long)fin);
    }
}
// idx = ijk0*mul0 + ijk1*mul1 + ijk2*mul2 with ijk = int(floor(x * inv) - float(min_b)); non-finite points get key 0xFFFFFFFF (sorted last)
__global__ void voxel_key_kernel(const uint8_t *__restrict__ raw, int stride, int64_t n, VoxelParams vp, uint32_t *__restrict__ keys, uint32_t *__restrict__ rows) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float *p = (const float *)(raw + i * (int64_t)stride);
    uint32_t key = 0xFFFFFFFFu;
    if (finite3(p[0], p[1], p[2])) {
        const int i0 = (int)(floorf(__fmul_rn(p[0], vp.inv[0])) - (float)vp.min_b[0]);
        const int i1 = (int)(floorf(__fmul_rn(p[1], vp.inv[1])) - (float)vp.min_b[1]);
        const int i2 = (int)(floorf(__fmul_rn(p[2], vp.inv[2])) - (float)vp.min_b[2]);
        key = (uint32_t)(i0 * vp.mul[0] + i1 * vp.mul[1] + i2 * vp.mul[2]);
    }
    keys[i] = key; rows[i] = (uint32_t)i;
}
__global__ void voxel_heads_kernel(const uint32_t *__restrict__ keys, int64_t m, uint32_t *__restrict__ head) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < m) head[i] = (i == 0 || keys[i] != keys[i - 1]) ? 1u : 0u;
}
// head positions -> seg_start[slot]; slot = exclusive scan of head flags
__global__ void voxel_segments_kernel(const uint32_t *__restrict__ head, const uint32_t *__restrict__ slot, int64_t m, uint32_t *__restrict__ seg_start) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < m && head[i]) seg_start[slot[i]] = (uint32_t)i;
}
__global__ void voxel_keep_kernel(const uint32_t *__restrict__ seg_start, int64_t n_seg, int64_t m, uint32_t min_pts, uint32_t *__restrict__ keep) {
    int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= n_seg) return;
    const uint32_t b = seg_start[v], e = v + 1 < n_seg ? seg_start[v + 1] : (uint32_t)m;
    keep[v] = (e - b >= min_pts) ? 1u : 0u;
}
// one thread per kept voxel: sequential fp32 sums in sorted (= ascending original row) order, then / count
__global__ void voxel_centroid_kernel(const uint8_t *__restrict__ raw, int stride, int rgb_off, const uint32_t *__restrict__ rows_sorted, const uint32_t *__restrict__ seg_start,
                                      const uint32_t *__restrict__ keep, const uint32_t *__restrict__ out_slot, int64_t n_seg, int64_t m, uint8_t *__restrict__ out, int out_stride) {
    int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= n_seg || !keep[v]) return;
    const uint32_t b = seg_start[v], e = v + 1 < n_seg ? seg_start[v + 1] : (uint32_t)m;
    float sx = 0.f, sy = 0.f, sz = 0.f, sr = 0.f, sg = 0.f, sb = 0.f;
    for (uint32_t j = b; j < e; ++j) {
        const uint8_t *row = raw + (int64_t)rows_sorted[j] * stride;
        const float *p = (const float *)row;
        if (j == b) { sx = p[0]; sy = p[1]; sz = p[2]; } else { sx += p[0]; sy += p[1]; sz += p[2]; }
        if (rgb_off >= 0) { const uint8_t *c = row + rgb_off; sb += (float)c[0]; sg += (float)c[1]; sr += (float)c[2]; }    // BGRA byte order
    }
    const float cnt = (float)(e - b);
    uint8_t *o = out + (int64_t)out_slot[v] * out_stride;
    for (int k = 0; k < out_stride; k += 4) *(uint32_t *)(o + k) = 0u;
    float *q = (float *)o;
    q[0] = __fdiv_rn(sx, cnt); q[1] = __fdiv_rn(sy, cnt); q[2] = __fdiv_rn(sz, cnt);
    if (out_stride >= 16) q[3] = 1.0f;
    if (rgb_off >= 0) {
        const int r = (int)__fdiv_rn(sr, cnt), gg = (int)__fdiv_rn(sg, cnt), bb = (int)__fdiv_rn(sb, cnt);
        *(int *)(o + rgb_off) = (r << 16) | (gg << 8) | bb;
    }
}


// ---- segmented VoxelGrid (pcc::segmented_voxel_grid): every segment of a float4 (x, y, z, rgb word) cloud with its own box ----
// per segment: what pcc_voxel_grid derives from its input.  mode 0 = no rows or no finite point (empty result), 1 = voxelised with
// keys base + local voxel index, 2 = passed through (PCL's leaf-too-small test); keep = the result reaches the caller's minimum.
struct SegVoxel { VoxelParams vp; unsigned long long base; int64_t in_begin, out_begin; uint32_t vfirst; int mode, keep, pad; };
__global__ void seg_voxel_init_kernel(int *__restrict__ bbox, uint32_t *__restrict__ vcount, int n_seg) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n_seg) return;
    int *b = bbox + 8 * c;
    b[0] = b[1] = b[2] = INT_MAX; b[3] = b[4] = b[5] = INT_MIN; b[6] = 0;
    vcount[c] = 0;
}
// getMinMax3D per segment: bbox[8c .. 8c+5] = box of the finite points, bbox[8c+6] = their count; lab[i] = segment of row i.  A warp
// whose rows share one segment (the common case) reduces before its atomics.
__global__ void seg_voxel_minmax_kernel(const float4 *__restrict__ in, int64_t n, const int64_t *__restrict__ off, int n_seg, uint32_t *__restrict__ lab,
                                        int *__restrict__ bbox) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = i < n;
    uint32_t c = 0xFFFFFFFFu;
    int lo[3] = {INT_MAX, INT_MAX, INT_MAX}, hi[3] = {INT_MIN, INT_MIN, INT_MIN};
    unsigned fin = 0;
    if (live) {
        c = segment_of(off, n_seg, i);
        lab[i] = c;
        const float4 p = in[i];
        if (finite3(p.x, p.y, p.z)) { fin = 1; lo[0] = hi[0] = f2ord_v(p.x); lo[1] = hi[1] = f2ord_v(p.y); lo[2] = hi[2] = f2ord_v(p.z); }
    }
    const uint32_t c0 = __shfl_sync(0xffffffffu, c, 0);
    if (__all_sync(0xffffffffu, !live || c == c0)) {
#pragma unroll
        for (int d = 0; d < 3; ++d) { lo[d] = __reduce_min_sync(0xffffffffu, lo[d]); hi[d] = __reduce_max_sync(0xffffffffu, hi[d]); }
        fin = __reduce_add_sync(0xffffffffu, fin);
        if ((threadIdx.x & 31) != 0) return;
        c = c0;
    }
    if (!fin) return;
    int *b = bbox + 8 * (size_t)c;
#pragma unroll
    for (int d = 0; d < 3; ++d) { atomicMin(b + d, lo[d]); atomicMax(b + 3 + d, hi[d]); }
    atomicAdd((unsigned *)(b + 6), fin);
}
// composite key base[segment] + voxel_key_kernel's index with the segment's own min_b, so a segment's voxels keep the order and the
// fp32 rounding of its own call; rows that are not voxelised get ~0 (sorted last)
__global__ void seg_voxel_key_kernel(const float4 *__restrict__ in, int64_t n, const uint32_t *__restrict__ lab, const SegVoxel *__restrict__ tab,
                                     unsigned long long *__restrict__ keys, uint32_t *__restrict__ rows) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 p = in[i];
    const SegVoxel &t = tab[lab[i]];
    unsigned long long key = ~0ull;
    if (t.mode == 1 && finite3(p.x, p.y, p.z)) {
        const int i0 = (int)(floorf(__fmul_rn(p.x, t.vp.inv[0])) - (float)t.vp.min_b[0]);
        const int i1 = (int)(floorf(__fmul_rn(p.y, t.vp.inv[1])) - (float)t.vp.min_b[1]);
        const int i2 = (int)(floorf(__fmul_rn(p.z, t.vp.inv[2])) - (float)t.vp.min_b[2]);
        key = t.base + (uint32_t)(i0 * t.vp.mul[0] + i1 * t.vp.mul[1] + i2 * t.vp.mul[2]);
    }
    keys[i] = key; rows[i] = (uint32_t)i;
}
// voxel_heads_kernel on 64-bit keys, counting each segment's voxels
__global__ void seg_voxel_heads_kernel(const unsigned long long *__restrict__ keys, int64_t m, const uint32_t *__restrict__ rows, const uint32_t *__restrict__ lab,
                                       uint32_t *__restrict__ head, uint32_t *__restrict__ vcount) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const bool h = i == 0 || keys[i] != keys[i - 1];
    head[i] = h ? 1u : 0u;
    if (h) atomicAdd(vcount + lab[rows[i]], 1u);
}
// voxel v of segment c -> keep = the segment is kept, output row out_begin[c] + (v - first voxel of c)
__global__ void seg_voxel_slots_kernel(const uint32_t *__restrict__ seg_start, int64_t n_vox, const uint32_t *__restrict__ rows, const uint32_t *__restrict__ lab,
                                       const SegVoxel *__restrict__ tab, uint32_t *__restrict__ keep, uint32_t *__restrict__ out_slot) {
    const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= n_vox) return;
    const SegVoxel &t = tab[lab[rows[seg_start[v]]]];
    keep[v] = t.keep ? 1u : 0u;
    out_slot[v] = t.keep ? (uint32_t)(t.out_begin + (v - (int64_t)t.vfirst)) : 0u;
}
// kept pass-through segments: every row, the non-finite ones too
__global__ void seg_voxel_passthrough_kernel(const float4 *__restrict__ in, int64_t n, const uint32_t *__restrict__ lab, const SegVoxel *__restrict__ tab,
                                             float4 *__restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const SegVoxel &t = tab[lab[i]];
    if (t.mode == 2 && t.keep) out[t.out_begin + (i - t.in_begin)] = in[i];
}

}  // namespace pcc

using namespace pcc;

static inline float ord2f_v(int i) { int j = i >= 0 ? i : i ^ 0x7FFFFFFF; float f; memcpy(&f, &j, 4); return f; }

// getMinMax3D's box (ordered-int bits, lo[3] then hi[3]) -> PCL 1.7 VoxelGrid::applyFilter's parameters and *n_voxels = dx*dy*dz;
// false when its "leaf size is too small" test sends the input through unfiltered.  (The products are formed in double so they
// cannot wrap.)
static bool voxel_params(const int *bbox, const float leaf[3], VoxelParams *vp, int64_t *n_voxels) {
    int64_t div[3], dchk[3];
    for (int d = 0; d < 3; ++d) {
        const float mn = ord2f_v(bbox[d]), mx = ord2f_v(bbox[3 + d]);
        vp->inv[d] = 1.0f / leaf[d];
        vp->min_b[d] = (int)std::floor(mn * vp->inv[d]);
        const int max_b = (int)std::floor(mx * vp->inv[d]);
        div[d] = (int64_t)max_b - vp->min_b[d] + 1;
        dchk[d] = (int64_t)((mx - mn) * vp->inv[d]) + 1;
    }
    if ((double)dchk[0] * (double)dchk[1] * (double)dchk[2] > 2147483647.0 || (double)div[0] * (double)div[1] * (double)div[2] > 2147483647.0) return false;
    vp->mul[0] = 1; vp->mul[1] = (int)div[0]; vp->mul[2] = (int)(div[0] * div[1]);
    *n_voxels = div[0] * div[1] * div[2];
    return true;
}

extern "C" int pcc_voxel_grid(pcc_index *idx, const void *pts, int64_t n, int stride_bytes, int rgb_offset_bytes, const float leaf[3], int min_points_per_voxel,
                              void *out, int64_t *n_out, int mem, void *stream) {
    if (!idx) return fail(PCC_ERR_INVALID, "idx is NULL");
    if (n < 0 || (n > 0 && (!pts || !out)) || stride_bytes < 12 || (stride_bytes & 3) || !leaf || !n_out) return fail(PCC_ERR_INVALID, "bad arguments");
    if (!(leaf[0] > 0 && leaf[1] > 0 && leaf[2] > 0)) return fail(PCC_ERR_INVALID, "leaf size must be positive");
    if (rgb_offset_bytes >= 0 && (rgb_offset_bytes + 4 > stride_bytes || (rgb_offset_bytes & 3))) return fail(PCC_ERR_INVALID, "bad rgb offset");
    if (n >= (1ll << 31) - 1) return fail(PCC_ERR_INVALID, "n exceeds int32 indices");
    PCC_CUDA(cudaSetDevice(idx->device));
    cudaStream_t s = (cudaStream_t)stream;
    *n_out = 0;
    if (n == 0) return PCC_OK;
    const uint8_t *raw = nullptr;
    PCC_TRY(stage_in(idx->raw, (const uint8_t *)pts, (size_t)n * stride_bytes, mem, s, &raw));
    uint8_t *d_out = (uint8_t *)out;
    if (mem == PCC_HOST) { PCC_TRY(idx->stage4.reserve((size_t)n * stride_bytes)); d_out = idx->stage4.as<uint8_t>(); }
    // 1. bounding box of the finite points
    int *h = (int *)idx->h_pinned;
    PCC_TRY(idx->keys64.reserve(256));
    int *d_scal = idx->keys64.as<int>();
    {
        int init[12] = {INT_MAX, INT_MAX, INT_MAX, INT_MIN, INT_MIN, INT_MIN, 0, 0, 0, 0, 0, 0};
        memcpy(h, init, sizeof(init));
        PCC_CUDA(cudaMemcpyAsync(d_scal, h, sizeof(init), cudaMemcpyHostToDevice, s));
        PCC_CUDA(cudaStreamSynchronize(s));
    }
    voxel_minmax_kernel<<<nblocks(n, 256), 256, 0, s>>>(raw, stride_bytes, n, d_scal, (unsigned long long *)(d_scal + 8)); PCC_LAUNCHED();
    PCC_CUDA(cudaGetLastError());
    PCC_CUDA(cudaMemcpyAsync(h, d_scal, 48, cudaMemcpyDeviceToHost, s));
    PCC_CUDA(cudaStreamSynchronize(s));
    const int64_t m = (int64_t)(*(unsigned long long *)(h + 8));
    if (m == 0) return PCC_OK;
    VoxelParams vp;
    int64_t n_voxels = 0;
    // PCL 1.7 VoxelGrid::applyFilter [up]: "if (dx*dy*dz > INT_MAX) { PCL_WARN(leaf size is too small ...); output = *input_; return; }"
    // -- the input passes through UNFILTERED (every row, also the non-finite ones) and the pipeline goes on.  Same test, same
    // outcome; the warning text is left in pcc_last_error().
    if (!voxel_params(h, leaf, &vp, &n_voxels)) {
        g_error = "pcc_voxel_grid: leaf size is too small for the input dataset, integer indices would overflow -- input passed through unfiltered (PCL behaviour)";
        if (mem == PCC_HOST) memcpy(out, pts, (size_t)n * stride_bytes);
        else PCC_CUDA(cudaMemcpyAsync(out, pts, (size_t)n * stride_bytes, cudaMemcpyDeviceToDevice, s));
        if (mem != PCC_HOST) PCC_CUDA(cudaStreamSynchronize(s));
        *n_out = n;
        return PCC_OK;
    }
    // 2. keys + stable radix sort (ties keep ascending row order)
    PCC_TRY(idx->qkeys.reserve((size_t)n * 4)); PCC_TRY(idx->qkeys2.reserve((size_t)n * 4));
    PCC_TRY(idx->qperm.reserve((size_t)n * 4)); PCC_TRY(idx->qperm2.reserve((size_t)n * 4));
    voxel_key_kernel<<<nblocks(n, 256), 256, 0, s>>>(raw, stride_bytes, n, vp, idx->qkeys.as<uint32_t>(), idx->qperm.as<uint32_t>()); PCC_LAUNCHED();
    size_t tmp = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, tmp, idx->qkeys.as<uint32_t>(), idx->qkeys2.as<uint32_t>(), idx->qperm.as<uint32_t>(), idx->qperm2.as<uint32_t>(), (int)n, 0, 32, s);
    PCC_TRY(idx->cub_tmp.reserve(tmp));
    PCC_CUDA(cub::DeviceRadixSort::SortPairs(idx->cub_tmp.p, tmp, idx->qkeys.as<uint32_t>(), idx->qkeys2.as<uint32_t>(), idx->qperm.as<uint32_t>(), idx->qperm2.as<uint32_t>(), (int)n, 0, 32, s));
    g_launches += 5;
    const uint32_t *keys = idx->qkeys2.as<uint32_t>(), *rows = idx->qperm2.as<uint32_t>();
    // 3. segments (finite points are the first m entries after the sort)
    PCC_TRY(idx->misc.reserve((size_t)m * 4 * 5 + 64));
    uint32_t *head = idx->misc.as<uint32_t>(), *slot = head + m, *seg_start = slot + m, *keep = seg_start + m, *out_slot = keep + m;
    voxel_heads_kernel<<<nblocks(m, 256), 256, 0, s>>>(keys, m, head); PCC_LAUNCHED();
    cub::DeviceScan::ExclusiveSum(nullptr, tmp, head, slot, (int)m, s);
    PCC_TRY(idx->cub_tmp.reserve(tmp));
    PCC_CUDA(cub::DeviceScan::ExclusiveSum(idx->cub_tmp.p, tmp, head, slot, (int)m, s));
    g_launches += 2;
    voxel_segments_kernel<<<nblocks(m, 256), 256, 0, s>>>(head, slot, m, seg_start); PCC_LAUNCHED();
    uint32_t *hu = (uint32_t *)idx->h_pinned;
    PCC_CUDA(cudaMemcpyAsync(hu, slot + (m - 1), 4, cudaMemcpyDeviceToHost, s));
    PCC_CUDA(cudaMemcpyAsync(hu + 1, head + (m - 1), 4, cudaMemcpyDeviceToHost, s));
    PCC_CUDA(cudaStreamSynchronize(s));
    const int64_t n_seg = (int64_t)hu[0] + hu[1];
    // 4. min_points_per_voxel filter -> output slots
    voxel_keep_kernel<<<nblocks(n_seg, 256), 256, 0, s>>>(seg_start, n_seg, m, (uint32_t)std::max(min_points_per_voxel, 0), keep); PCC_LAUNCHED();
    cub::DeviceScan::ExclusiveSum(nullptr, tmp, keep, out_slot, (int)n_seg, s);
    PCC_TRY(idx->cub_tmp.reserve(tmp));
    PCC_CUDA(cub::DeviceScan::ExclusiveSum(idx->cub_tmp.p, tmp, keep, out_slot, (int)n_seg, s));
    g_launches += 2;
    PCC_CUDA(cudaMemcpyAsync(hu, out_slot + (n_seg - 1), 4, cudaMemcpyDeviceToHost, s));
    PCC_CUDA(cudaMemcpyAsync(hu + 1, keep + (n_seg - 1), 4, cudaMemcpyDeviceToHost, s));
    // 5. centroids
    voxel_centroid_kernel<<<nblocks(n_seg, 128), 128, 0, s>>>(raw, stride_bytes, rgb_offset_bytes, rows, seg_start, keep, out_slot, n_seg, m, d_out, stride_bytes); PCC_LAUNCHED();
    PCC_CUDA(cudaGetLastError());
    PCC_CUDA(cudaStreamSynchronize(s));
    const int64_t total = (int64_t)hu[0] + hu[1];
    if (mem == PCC_HOST && total > 0) { PCC_CUDA(cudaMemcpyAsync(out, d_out, (size_t)total * stride_bytes, cudaMemcpyDeviceToHost, s)); PCC_CUDA(cudaStreamSynchronize(s)); }
    *n_out = total;
    return PCC_OK;
}

// pcc_voxel_grid's steps over all segments at once: per-segment boxes (one read-back) -> per-segment parameters on the host ->
// one stable sort of (segment, voxel) keys -> heads and per-segment voxel counts (one read-back) -> the unchanged centroid kernel.
int pcc::segmented_voxel_grid(pcc_index *idx, const float4 *in, const int64_t *in_off, int n_seg, float leaf, int64_t min_rows, float4 *out, int64_t *out_off,
                              cudaStream_t s) {
    const int64_t n = in_off[n_seg];
    for (int c = 0; c <= n_seg; ++c) out_off[c] = 0;
    if (n == 0) return PCC_OK;
    const float leaf3[3] = {leaf, leaf, leaf};
    // sift_tab: SegVoxel[n_seg] | int64 offsets[n_seg + 1] | int bbox[8 n_seg] | uint32 vcount[n_seg]
    const size_t tab_bytes = (size_t)n_seg * sizeof(SegVoxel), off_at = tab_bytes, bbox_at = off_at + (size_t)(n_seg + 1) * 8, cnt_at = bbox_at + (size_t)n_seg * 32;
    PCC_TRY(idx->sift_tab.reserve(cnt_at + (size_t)n_seg * 4));
    uint8_t *tb = idx->sift_tab.as<uint8_t>();
    SegVoxel *d_tab = (SegVoxel *)tb;
    int64_t *d_off = (int64_t *)(tb + off_at);
    int *d_bbox = (int *)(tb + bbox_at);
    uint32_t *d_cnt = (uint32_t *)(tb + cnt_at);
    PCC_TRY(idx->sift_lab.reserve((size_t)n * 4));
    uint32_t *lab = idx->sift_lab.as<uint32_t>();
    PCC_CUDA(cudaMemcpyAsync(d_off, in_off, (size_t)(n_seg + 1) * 8, cudaMemcpyHostToDevice, s));
    seg_voxel_init_kernel<<<nblocks(n_seg, 256), 256, 0, s>>>(d_bbox, d_cnt, n_seg); PCC_LAUNCHED();
    seg_voxel_minmax_kernel<<<nblocks(n, 256), 256, 0, s>>>(in, n, d_off, n_seg, lab, d_bbox); PCC_LAUNCHED();
    PCC_CUDA(cudaGetLastError());
    std::vector<int> hb((size_t)n_seg * 8);
    PCC_CUDA(cudaMemcpyAsync(hb.data(), d_bbox, hb.size() * 4, cudaMemcpyDeviceToHost, s));
    PCC_CUDA(cudaStreamSynchronize(s));
    std::vector<SegVoxel> tab((size_t)n_seg);
    std::vector<int64_t> n_res((size_t)n_seg, 0);
    unsigned long long range = 0;
    int64_t m = 0;
    for (int c = 0; c < n_seg; ++c) {
        SegVoxel &t = tab[c];
        memset(&t, 0, sizeof(t));
        t.in_begin = in_off[c];
        const uint32_t fin = (uint32_t)hb[8 * c + 6];
        if (fin == 0) continue;                                     // pcc_voxel_grid: no finite point, no output
        int64_t nv = 0;
        if (!voxel_params(&hb[8 * c], leaf3, &t.vp, &nv)) { t.mode = 2; n_res[c] = in_off[c + 1] - in_off[c]; continue; }
        t.mode = 1; t.base = range; range += (unsigned long long)nv; m += fin;
    }
    std::vector<uint32_t> vcount((size_t)n_seg, 0);
    const uint32_t *rows = nullptr, *seg_start = nullptr;
    uint32_t *keep = nullptr, *out_slot = nullptr;
    int64_t n_vox = 0;
    if (m > 0) {
        PCC_CUDA(cudaMemcpyAsync(d_tab, tab.data(), tab_bytes, cudaMemcpyHostToDevice, s));
        PCC_TRY(idx->keys64.reserve((size_t)n * 8)); PCC_TRY(idx->keys64b.reserve((size_t)n * 8));
        PCC_TRY(idx->qperm.reserve((size_t)n * 4)); PCC_TRY(idx->qperm2.reserve((size_t)n * 4));
        unsigned long long *k_in = idx->keys64.as<unsigned long long>(), *k_out = idx->keys64b.as<unsigned long long>();
        seg_voxel_key_kernel<<<nblocks(n, 256), 256, 0, s>>>(in, n, lab, d_tab, k_in, idx->qperm.as<uint32_t>()); PCC_LAUNCHED();
        int bits = 1;                                              // ~0 (not voxelised) must stay above every key in the sorted bits
        while (bits < 64 && (1ull << bits) <= range) ++bits;
        size_t tmp = 0;
        cub::DeviceRadixSort::SortPairs(nullptr, tmp, k_in, k_out, idx->qperm.as<uint32_t>(), idx->qperm2.as<uint32_t>(), (int)n, 0, bits, s);
        PCC_TRY(idx->cub_tmp.reserve(tmp));
        PCC_CUDA(cub::DeviceRadixSort::SortPairs(idx->cub_tmp.p, tmp, k_in, k_out, idx->qperm.as<uint32_t>(), idx->qperm2.as<uint32_t>(), (int)n, 0, bits, s));
        g_launches += 2 * ((bits + 7) / 8) + 1;
        rows = idx->qperm2.as<uint32_t>();
        PCC_TRY(idx->misc.reserve((size_t)m * 4 * 5 + 64));
        uint32_t *head = idx->misc.as<uint32_t>(), *slot = head + m, *ss = slot + m;
        keep = ss + m; out_slot = keep + m; seg_start = ss;
        seg_voxel_heads_kernel<<<nblocks(m, 256), 256, 0, s>>>(k_out, m, rows, lab, head, d_cnt); PCC_LAUNCHED();
        cub::DeviceScan::ExclusiveSum(nullptr, tmp, head, slot, (int)m, s);
        PCC_TRY(idx->cub_tmp.reserve(tmp));
        PCC_CUDA(cub::DeviceScan::ExclusiveSum(idx->cub_tmp.p, tmp, head, slot, (int)m, s));
        g_launches += 2;
        voxel_segments_kernel<<<nblocks(m, 256), 256, 0, s>>>(head, slot, m, ss); PCC_LAUNCHED();
        PCC_CUDA(cudaGetLastError());
        PCC_CUDA(cudaMemcpyAsync(vcount.data(), d_cnt, (size_t)n_seg * 4, cudaMemcpyDeviceToHost, s));
        PCC_CUDA(cudaStreamSynchronize(s));
    }
    bool any_pass = false;
    for (int c = 0; c < n_seg; ++c) {
        SegVoxel &t = tab[c];
        if (t.mode == 1) { t.vfirst = (uint32_t)n_vox; n_vox += vcount[c]; n_res[c] = vcount[c]; }
        t.keep = n_res[c] > 0 && n_res[c] >= min_rows;
        t.out_begin = out_off[c];
        out_off[c + 1] = out_off[c] + (t.keep ? n_res[c] : 0);
        any_pass |= t.mode == 2 && t.keep;
    }
    if (out_off[n_seg] == 0) return PCC_OK;
    PCC_CUDA(cudaMemcpyAsync(d_tab, tab.data(), tab_bytes, cudaMemcpyHostToDevice, s));
    if (n_vox > 0) {
        seg_voxel_slots_kernel<<<nblocks(n_vox, 256), 256, 0, s>>>(seg_start, n_vox, rows, lab, d_tab, keep, out_slot); PCC_LAUNCHED();
        voxel_centroid_kernel<<<nblocks(n_vox, 128), 128, 0, s>>>((const uint8_t *)in, 16, 12, rows, seg_start, keep, out_slot, n_vox, m, (uint8_t *)out, 16);
        PCC_LAUNCHED();
    }
    if (any_pass) { seg_voxel_passthrough_kernel<<<nblocks(n, 256), 256, 0, s>>>(in, n, lab, d_tab, out); PCC_LAUNCHED(); }
    PCC_CUDA(cudaGetLastError());
    return PCC_OK;
}
