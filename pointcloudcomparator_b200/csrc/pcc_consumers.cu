// pcc_consumers.cu -- the O(1)/O(n) host-driven parts of the consumers: StatisticalOutlierRemoval's second pass,
// Umeyama from the ICP sums, and the ICP loop itself (SURVEY.md section 8 a5, a6).
#include <algorithm>
#include <array>
#include <limits>
#include <cfloat>
#include <cmath>
#include <cstring>
#include <vector>

#include "pcc_internal.h"

namespace pcc {

// per-block (sum d, sum d*d) with the product rounded in fp32 first, as PCL's "sq_sum += distances[i] * distances[i]" does
__global__ void sor_sums_kernel(const float *__restrict__ d, int64_t n, double *__restrict__ partials) {
    __shared__ double r0[256], r1[256];
    double a = 0, b = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) { float v = d[i]; a += (double)v; b += (double)(v * v); }
    r0[threadIdx.x] = a; r1[threadIdx.x] = b;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) { if ((int)threadIdx.x < o) { r0[threadIdx.x] += r0[threadIdx.x + o]; r1[threadIdx.x] += r1[threadIdx.x + o]; } __syncthreads(); }
    if (threadIdx.x == 0) { partials[2 * blockIdx.x] = r0[0]; partials[2 * blockIdx.x + 1] = r1[0]; }
}
__global__ void sor_final_kernel(const double *__restrict__ partials, int nb, double *__restrict__ out) {
    if (threadIdx.x < 2) { double v = 0; for (int b = 0; b < nb; ++b) v += partials[2 * b + threadIdx.x]; out[threadIdx.x] = v; }
}
__global__ void sor_keep_kernel(const float *__restrict__ d, int64_t n, double thr, uint8_t *__restrict__ keep, unsigned long long *__restrict__ kept) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    unsigned k = 0;
    if (i < n) { k = !((double)d[i] > thr); if (keep) keep[i] = (uint8_t)k; }
    k = __reduce_add_sync(0xffffffffu, k);
    if ((threadIdx.x & 31) == 0 && k) atomicAdd(kept, (unsigned long long)k);
}
__global__ void xform_kernel(const uint8_t *__restrict__ raw, int stride, int64_t n, const float *__restrict__ Tm, float4 *__restrict__ dst) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float *p = (const float *)(raw + i * (int64_t)stride);
    const float x = p[0], y = p[1], z = p[2];
    // pcl::transformPointCloud arithmetic: ((m0*x + m1*y) + m2*z) + m3 (fp32)
    dst[i] = make_float4(((Tm[0] * x + Tm[1] * y) + Tm[2] * z) + Tm[3], ((Tm[4] * x + Tm[5] * y) + Tm[6] * z) + Tm[7], ((Tm[8] * x + Tm[9] * y) + Tm[10] * z) + Tm[11], 1.f);
}

// ---- 3x3 SVD in double (Jacobi on A^T A) for Umeyama ----
static void svd3(const double A[9], double U[9], double S[3], double V[9]) {
    double B[9];
    for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) { double s = 0; for (int k = 0; k < 3; ++k) s += A[3 * k + i] * A[3 * k + j]; B[3 * i + j] = s; }
    for (int i = 0; i < 9; ++i) V[i] = (i % 4 == 0) ? 1.0 : 0.0;
    for (int sweep = 0; sweep < 60; ++sweep) {
        if (std::fabs(B[1]) + std::fabs(B[2]) + std::fabs(B[5]) < 1e-300) break;
        for (int p = 0; p < 2; ++p) for (int q = p + 1; q < 3; ++q) {
            const double apq = B[3 * p + q];
            if (std::fabs(apq) < 1e-300) continue;
            const double theta = (B[3 * q + q] - B[3 * p + p]) / (2.0 * apq);
            const double t = (theta >= 0 ? 1.0 : -1.0) / (std::fabs(theta) + std::sqrt(theta * theta + 1.0));
            const double c = 1.0 / std::sqrt(t * t + 1.0), s = t * c;
            for (int k = 0; k < 3; ++k) { double a = B[3 * k + p], b = B[3 * k + q]; B[3 * k + p] = c * a - s * b; B[3 * k + q] = s * a + c * b; }
            for (int k = 0; k < 3; ++k) { double a = B[3 * p + k], b = B[3 * q + k]; B[3 * p + k] = c * a - s * b; B[3 * q + k] = s * a + c * b; }
            for (int k = 0; k < 3; ++k) { double a = V[3 * k + p], b = V[3 * k + q]; V[3 * k + p] = c * a - s * b; V[3 * k + q] = s * a + c * b; }
        }
    }
    const double ev[3] = {B[0], B[4], B[8]};
    int ord[3] = {0, 1, 2};
    std::sort(ord, ord + 3, [&](int a, int b) { return ev[a] > ev[b]; });
    double Vs[9];
    for (int c = 0; c < 3; ++c) for (int r = 0; r < 3; ++r) Vs[3 * r + c] = V[3 * r + ord[c]];
    memcpy(V, Vs, sizeof(Vs));
    for (int c = 0; c < 3; ++c) S[c] = std::sqrt(std::max(ev[ord[c]], 0.0));
    for (int c = 0; c < 3; ++c) for (int r = 0; r < 3; ++r) { double s = 0; for (int k = 0; k < 3; ++k) s += A[3 * r + k] * V[3 * k + c]; U[3 * r + c] = s; }
    bool good[3];
    for (int c = 0; c < 3; ++c) {
        const double nrm = std::sqrt(U[c] * U[c] + U[3 + c] * U[3 + c] + U[6 + c] * U[6 + c]);
        good[c] = nrm > 1e-12 * (S[0] > 0 ? S[0] : 1.0) && nrm > 0;
        if (good[c]) for (int r = 0; r < 3; ++r) U[3 * r + c] /= nrm;
    }
    if (!good[0]) { U[0] = 1; U[3] = 0; U[6] = 0; }
    if (!good[1]) {
        const double a[3] = {U[0], U[3], U[6]};
        const int m = std::fabs(a[0]) < std::fabs(a[1]) ? (std::fabs(a[0]) < std::fabs(a[2]) ? 0 : 2) : (std::fabs(a[1]) < std::fabs(a[2]) ? 1 : 2);
        double v[3] = {-a[m] * a[0], -a[m] * a[1], -a[m] * a[2]}; v[m] += 1.0;
        const double nrm = std::sqrt(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]);
        U[1] = v[0] / nrm; U[4] = v[1] / nrm; U[7] = v[2] / nrm;
    }
    if (!good[2]) {
        const double a[3] = {U[0], U[3], U[6]}, b[3] = {U[1], U[4], U[7]};
        U[2] = a[1] * b[2] - a[2] * b[1]; U[5] = a[2] * b[0] - a[0] * b[2]; U[8] = a[0] * b[1] - a[1] * b[0];
    }
}
static double det3(const double *m) { return m[0] * (m[4] * m[8] - m[5] * m[7]) - m[1] * (m[3] * m[8] - m[5] * m[6]) + m[2] * (m[3] * m[7] - m[4] * m[6]); }
static void mat4_mul(const float *A, const float *B, float *C) {
    float r[16];
    for (int i = 0; i < 4; ++i) for (int j = 0; j < 4; ++j) { float s = 0.f; for (int k = 0; k < 4; ++k) s += A[4 * i + k] * B[4 * k + j]; r[4 * i + j] = s; }
    memcpy(C, r, sizeof(r));
}

}  // namespace pcc

using namespace pcc;

extern "C" {

// TransformationEstimationSVD -> pcl::umeyama(src, tgt, with_scaling = false) [up], evaluated from running sums in double.
int pcc_umeyama_from_sums(const double sums[16], int64_t count, float T16[16]) {
    if (!sums || !T16 || count < 1) return fail(PCC_ERR_INVALID, "bad sums / count");
    const double n = (double)count;
    double ms[3], mt[3], sigma[9];
    for (int i = 0; i < 3; ++i) { ms[i] = sums[i] / n; mt[i] = sums[3 + i] / n; }
    for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) sigma[3 * i + j] = sums[6 + 3 * i + j] / n - mt[i] * ms[j];
    double U[9], S[3], V[9];
    svd3(sigma, U, S, V);
    double Sg[3] = {1, 1, 1};
    if (det3(sigma) < 0) Sg[2] = -1;
    int rank = 0;
    for (int i = 0; i < 3; ++i) if (!(std::fabs(S[i]) <= std::fabs(S[0]) * 1e-12)) ++rank;
    if (rank == 2) Sg[2] = det3(U) * det3(V) > 0 ? 1 : -1;
    double R[9];
    for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) { double s = 0; for (int k = 0; k < 3; ++k) s += U[3 * i + k] * Sg[k] * V[3 * j + k]; R[3 * i + j] = s; }
    for (int i = 0; i < 16; ++i) T16[i] = (i % 5 == 0) ? 1.f : 0.f;
    for (int i = 0; i < 3; ++i) {
        for (int j = 0; j < 3; ++j) T16[4 * i + j] = (float)R[3 * i + j];
        T16[4 * i + 3] = (float)(mt[i] - (R[3 * i] * ms[0] + R[3 * i + 1] * ms[1] + R[3 * i + 2] * ms[2]));
    }
    return PCC_OK;
}

int pcc_sor_threshold(pcc_index *idx, const float *distances, int64_t n, int64_t n_valid, double std_mul, double stats[3], uint8_t *keep, int64_t *kept, int mem, void *stream) {
    if (!idx) return fail(PCC_ERR_INVALID, "idx is NULL");
    if (n < 0 || (n > 0 && !distances) || !stats) return fail(PCC_ERR_INVALID, "bad distances / stats");
    PCC_CUDA(cudaSetDevice(idx->device));
    cudaStream_t s = (cudaStream_t)stream;
    if (n_valid <= 0) n_valid = n;
    if (kept) *kept = 0;
    stats[0] = stats[1] = stats[2] = 0;
    if (n == 0) return PCC_OK;
    const float *d = nullptr;
    PCC_TRY(stage_in(idx->out_f, distances, (size_t)n * 4, mem, s, &d));
    const int nb = (int)std::min<int64_t>(nblocks(n, 256), 1024);
    PCC_TRY(idx->keys64b.reserve((size_t)(2 * nb + 4) * sizeof(double)));
    double *partials = idx->keys64b.as<double>(), *d_out = partials + 2 * nb;
    sor_sums_kernel<<<nb, 256, 0, s>>>(d, n, partials); PCC_LAUNCHED();
    sor_final_kernel<<<1, 32, 0, s>>>(partials, nb, d_out); PCC_LAUNCHED();
    double *h = (double *)idx->h_pinned;
    PCC_CUDA(cudaMemcpyAsync(h, d_out, 16, cudaMemcpyDeviceToHost, s));
    PCC_CUDA(cudaStreamSynchronize(s));
    const double sum = h[0], sq = h[1], nv = (double)n_valid;
    const double mean = sum / nv;
    const double var = (sq - sum * sum / nv) / (nv - 1.0);
    const double sd = std::sqrt(var);
    stats[0] = mean; stats[1] = sd; stats[2] = mean + std_mul * sd;
    uint8_t *dk = keep;
    if (keep && mem == PCC_HOST) { PCC_TRY(idx->out_i.reserve((size_t)n)); dk = idx->out_i.as<uint8_t>(); }
    unsigned long long *d_kept = (unsigned long long *)(d_out + 2);
    PCC_CUDA(cudaMemsetAsync(d_kept, 0, 8, s));
    sor_keep_kernel<<<nblocks(n, 256), 256, 0, s>>>(d, n, stats[2], dk, d_kept); PCC_LAUNCHED();
    PCC_CUDA(cudaGetLastError());
    PCC_CUDA(cudaMemcpyAsync(h, d_kept, 8, cudaMemcpyDeviceToHost, s));
    if (keep && mem == PCC_HOST) PCC_CUDA(cudaMemcpyAsync(keep, dk, (size_t)n, cudaMemcpyDeviceToHost, s));
    PCC_CUDA(cudaStreamSynchronize(s));
    if (kept) *kept = (int64_t)(*(unsigned long long *)h);
    return PCC_OK;
}

// RegionGrowing::applySmoothRegionGrowingAlgorithm + growRegion + validatePoint + assembleRegions [up] over the N x k neighbour
// table the GPU built (pcc_knn with q == NULL).  Sequential and order-dependent by definition, so it stays on the host
// (SURVEY.md section 8 a8 / 8f row 2); reference configuration: src/segmentation.cpp:249-271 (k = 100, 3 degrees, curvature 1,
// sizes 50..1000000).  Seeds are taken in ascending (curvature, index) order, NaN curvatures last (PCL's std::sort leaves ties unspecified).
int pcc_region_growing(const int32_t *neighbours, int64_t n, int k, const float *normals4, float smoothness_rad, float curvature_threshold,
                       int64_t min_size, int64_t max_size, int32_t *labels, int64_t *n_clusters) {
    if (n < 0 || k < 1 || (n > 0 && (!neighbours || !normals4 || !labels)) || !n_clusters) return fail(PCC_ERR_INVALID, "bad arguments");
    *n_clusters = 0;
    if (n == 0) return PCC_OK;
    std::vector<int32_t> order((size_t)n);
    for (int64_t i = 0; i < n; ++i) order[(size_t)i] = (int32_t)i;
    // ascending curvature, NaN curvatures last, ties by index (a strict weak order even with NaNs; PCL's comparator is not)
    std::stable_sort(order.begin(), order.end(), [&](int32_t a, int32_t b) {
        const float ca = normals4[4 * (size_t)a + 3], cb = normals4[4 * (size_t)b + 3];
        const bool na = ca != ca, nb = cb != cb;
        if (na != nb) return nb;
        return !na && ca < cb;
    });
    std::vector<int32_t> seg((size_t)n, -1), queue;
    std::vector<int64_t> seg_size;
    const float cosine_threshold = cosf(smoothness_rad);
    queue.reserve(1024);
    for (int64_t si = 0; si < n; ++si) {
        const int32_t seed0 = order[(size_t)si];
        if (seg[(size_t)seed0] != -1) continue;
        const int32_t s_id = (int32_t)seg_size.size();
        int64_t count = 1;
        seg[(size_t)seed0] = s_id;
        queue.clear(); queue.push_back(seed0);
        for (size_t head = 0; head < queue.size(); ++head) {
            const int32_t cur = queue[head];
            const float *nc = normals4 + 4 * (size_t)cur;
            const int32_t *nb = neighbours + (size_t)cur * k;
            for (int j = 0; j < k; ++j) {
                const int32_t idx = nb[j];
                if (idx < 0) break;                              // rows shorter than k end with -1
                if (seg[(size_t)idx] != -1) continue;
                const float *nn = normals4 + 4 * (size_t)idx;
                const float dot = fabsf((nn[0] * nc[0] + nn[1] * nc[1]) + nn[2] * nc[2]);
                if (dot < cosine_threshold) continue;
                seg[(size_t)idx] = s_id; ++count;
                if (!(nn[3] > curvature_threshold)) queue.push_back(idx);
            }
        }
        seg_size.push_back(count);
    }
    std::vector<int32_t> rank(seg_size.size(), -1);
    int64_t kept = 0;
    for (size_t s2 = 0; s2 < seg_size.size(); ++s2) if (seg_size[s2] >= min_size && seg_size[s2] <= max_size) rank[s2] = (int32_t)kept++;
    for (int64_t i = 0; i < n; ++i) labels[i] = rank[(size_t)seg[(size_t)i]];
    *n_clusters = kept;
    return PCC_OK;
}

// RegionGrowingRGB::extract minus findPointNeighbours (src/segmentation.cpp:179-190, called per matched cluster at
// src/comparator.cpp:1457-1460; the consumer only counts the clusters that come out) [up: segmentation/impl/region_growing_rgb.hpp
// and region_growing.hpp of PCL 1.7, restated from the published source -- NOT in /root/reference, see DESIGN.md]:
//   1. grow (RegionGrowing::applySmoothRegionGrowingAlgorithm with RegionGrowingRGB::validatePoint): normals are off in the
//      reference's configuration, so seeds are taken in index order; a neighbour joins when its colour is within
//      point_color_threshold of the CURRENT point (squared RGB distance > thr^2 rejects) and always becomes a seed.  growRegion only
//      walks the first `grow_neighbours` (RegionGrowing's neighbour_number_, 30 unless set) of the k = 100 neighbours
//      RegionGrowingRGB::findPointNeighbours asks for;
//   2. findSegmentNeighbours / findRegionsKNN: for every segment the nearest other segments by the smallest neighbour-table distance
//      (squared, as the search returns it) between their points, the k nearest kept, listed farthest first (a std::priority_queue);
//   3. applyRegionMergingAlgorithm: mean colour per segment (unsigned sums, float division, truncation); in segment order, neighbours
//      within distance_threshold^2 whose mean colour is within region_color_threshold^2 (strict <) join the homogeneous region;
//      then regions smaller than min_size are folded into their nearest neighbouring region;
//   4. assembleRegions + the size filter of extract().  labels[i] = cluster number in PCL's final order, or -1.
// Sequential and order-dependent like the plain RegionGrowing grow phase, hence host code over the GPU-built N x k table.
int pcc_region_growing_rgb(const int32_t *neighbours, const float *sqr_distances, int64_t n, int k, const uint32_t *rgba, int rgba_stride_bytes,
                           float distance_threshold, float point_color_threshold, float region_color_threshold, int grow_neighbours,
                           int64_t min_size, int64_t max_size, int32_t *labels, int64_t *n_clusters) {
    if (n < 0 || k < 1 || (n > 0 && (!neighbours || !sqr_distances || !rgba || !labels)) || !n_clusters || rgba_stride_bytes < 4 || (rgba_stride_bytes & 3) || grow_neighbours < 1)
        return fail(PCC_ERR_INVALID, "bad arguments");
    *n_clusters = 0;
    if (n == 0) return PCC_OK;
    const float dist_thr = distance_threshold * distance_threshold, p2p = point_color_threshold * point_color_threshold, r2r = region_color_threshold * region_color_threshold;
    auto colour = [&](int64_t i, unsigned c[3]) { const uint32_t v = *(const uint32_t *)((const uint8_t *)rgba + (size_t)i * rgba_stride_bytes); c[0] = (v >> 16) & 255u; c[1] = (v >> 8) & 255u; c[2] = v & 255u; };
    auto colour_diff = [](const unsigned a[3], const unsigned b[3]) {       // calculateColorimetricalDifference: unsigned products, summed in float
        float d = 0.f;
        d += (float)((a[0] - b[0]) * (a[0] - b[0])); d += (float)((a[1] - b[1]) * (a[1] - b[1])); d += (float)((a[2] - b[2]) * (a[2] - b[2]));
        return d;
    };
    auto row_len = [&](int64_t i) { int m = 0; const int32_t *r = neighbours + (size_t)i * k; while (m < k && r[m] >= 0) ++m; return m; };
    // 1. grow
    std::vector<int32_t> point_label((size_t)n, -1), queue;
    std::vector<int64_t> seg_size;
    for (int64_t seed0 = 0; seed0 < n; ++seed0) {
        if (point_label[(size_t)seed0] != -1) continue;
        const int32_t s_id = (int32_t)seg_size.size();
        int64_t count = 1;
        point_label[(size_t)seed0] = s_id;
        queue.clear(); queue.push_back((int32_t)seed0);
        for (size_t head = 0; head < queue.size(); ++head) {
            const int32_t cur = queue[head];
            unsigned cc[3]; colour(cur, cc);
            const int32_t *nb = neighbours + (size_t)cur * k;
            const int lim = std::min(grow_neighbours, row_len(cur));
            for (int j = 0; j < lim; ++j) {
                const int32_t q = nb[j];
                if (point_label[(size_t)q] != -1) continue;
                unsigned nc[3]; colour(q, nc);
                if (colour_diff(cc, nc) > p2p) continue;
                point_label[(size_t)q] = s_id; ++count;
                queue.push_back(q);
            }
        }
        seg_size.push_back(count);
    }
    const int n_seg = (int)seg_size.size();
    std::vector<std::vector<int32_t>> seg_pts((size_t)n_seg);
    for (int sg = 0; sg < n_seg; ++sg) seg_pts[(size_t)sg].reserve((size_t)seg_size[(size_t)sg]);
    for (int64_t i = 0; i < n; ++i) seg_pts[(size_t)point_label[(size_t)i]].push_back((int32_t)i);
    // 2. segment neighbours (findRegionsKNN for every segment)
    std::vector<std::vector<int>> seg_nb((size_t)n_seg);
    std::vector<std::vector<float>> seg_nd((size_t)n_seg);
    {
        const float max_dist = std::numeric_limits<float>::max();
        std::vector<float> dist((size_t)n_seg, max_dist);
        std::vector<int> stamp((size_t)n_seg, -1), touched;
        std::vector<std::pair<float, int>> cand;
        for (int sg = 0; sg < n_seg; ++sg) {
            touched.clear();
            for (int32_t p : seg_pts[(size_t)sg]) {
                const int32_t *nb = neighbours + (size_t)p * k; const float *nd = sqr_distances + (size_t)p * k;
                const int m = row_len(p);
                for (int j = 0; j < m; ++j) {
                    const int os = point_label[(size_t)nb[j]];
                    if (os == sg) continue;
                    if (stamp[(size_t)os] != sg) { stamp[(size_t)os] = sg; dist[(size_t)os] = max_dist; touched.push_back(os); }
                    if (dist[(size_t)os] > nd[j]) dist[(size_t)os] = nd[j];
                }
            }
            // PCL pushes (distance, segment) into a std::priority_queue and pops its maximum whenever it holds more than k: the k
            // smallest pairs survive (lexicographic), and they are then popped farthest first
            cand.clear();
            for (int os : touched) if (dist[(size_t)os] < max_dist) cand.push_back(std::make_pair(dist[(size_t)os], os));
            std::sort(cand.begin(), cand.end());
            if ((int)cand.size() > k) cand.resize((size_t)k);
            for (size_t c = cand.size(); c-- > 0;) { seg_nd[(size_t)sg].push_back(cand[c].first); seg_nb[(size_t)sg].push_back(cand[c].second); }
        }
    }
    // 3. merge by mean colour
    std::vector<std::array<unsigned, 3>> seg_col((size_t)n_seg, std::array<unsigned, 3>{0u, 0u, 0u});
    for (int64_t i = 0; i < n; ++i) { unsigned c[3]; colour(i, c); auto &a = seg_col[(size_t)point_label[(size_t)i]]; a[0] += c[0]; a[1] += c[1]; a[2] += c[2]; }
    for (int sg = 0; sg < n_seg; ++sg) for (int c = 0; c < 3; ++c) seg_col[(size_t)sg][c] = (unsigned)((float)seg_col[(size_t)sg][c] / (float)seg_size[(size_t)sg]);
    std::vector<int> seg_label((size_t)n_seg, -1);
    std::vector<int64_t> reg_pts; std::vector<int> reg_segs;
    for (int sg = 0; sg < n_seg; ++sg) {
        int cur;
        if (seg_label[(size_t)sg] == -1) { seg_label[(size_t)sg] = cur = (int)reg_pts.size(); reg_pts.push_back(seg_size[(size_t)sg]); reg_segs.push_back(1); }
        else cur = seg_label[(size_t)sg];
        for (size_t j = 0; j < seg_nb[(size_t)sg].size() && (int)j < k; ++j) {
            const int os = seg_nb[(size_t)sg][j];
            if (seg_nd[(size_t)sg][j] > dist_thr) continue;
            if (seg_label[(size_t)os] != -1) continue;
            if (colour_diff(seg_col[(size_t)sg].data(), seg_col[(size_t)os].data()) < r2r) { seg_label[(size_t)os] = cur; reg_pts[(size_t)cur] += seg_size[(size_t)os]; reg_segs[(size_t)cur] += 1; }
        }
    }
    const int n_reg = (int)reg_pts.size();
    std::vector<std::vector<int>> final_segs((size_t)n_reg);
    for (int sg = 0; sg < n_seg; ++sg) final_segs[(size_t)seg_label[(size_t)sg]].push_back(sg);
    // findRegionNeighbours: per region the (distance, segment) pairs of its segments' neighbours that lie in other regions, ascending by distance
    auto by_first = [](const std::pair<float, int> &a, const std::pair<float, int> &b) { return a.first < b.first; };
    std::vector<std::vector<std::pair<float, int>>> reg_nb((size_t)n_reg);
    for (int r = 0; r < n_reg; ++r) {
        for (int sg : final_segs[(size_t)r])
            for (size_t j = 0; j < seg_nb[(size_t)sg].size(); ++j)
                if (seg_label[(size_t)seg_nb[(size_t)sg][j]] != r) reg_nb[(size_t)r].push_back(std::make_pair(seg_nd[(size_t)sg][j], seg_nb[(size_t)sg][j]));
        std::stable_sort(reg_nb[(size_t)r].begin(), reg_nb[(size_t)r].end(), by_first);
    }
    for (int r = 0; r < n_reg; ++r) {
        if (reg_pts[(size_t)r] >= min_size) continue;
        if (reg_nb[(size_t)r].empty()) continue;
        if (reg_nb[(size_t)r][0].first == std::numeric_limits<float>::max()) continue;
        const int target = seg_label[(size_t)reg_nb[(size_t)r][0].second];
        for (int sg : final_segs[(size_t)r]) { final_segs[(size_t)target].push_back(sg); seg_label[(size_t)sg] = target; }
        final_segs[(size_t)r].clear();
        reg_pts[(size_t)target] += reg_pts[(size_t)r]; reg_pts[(size_t)r] = 0;
        reg_segs[(size_t)target] += reg_segs[(size_t)r]; reg_segs[(size_t)r] = 0;
        for (auto &pr : reg_nb[(size_t)target]) if (seg_label[(size_t)pr.second] == target) { pr.first = std::numeric_limits<float>::max(); pr.second = 0; }
        for (const auto &pr : reg_nb[(size_t)r]) if (seg_label[(size_t)pr.second] != target) reg_nb[(size_t)target].push_back(pr);
        reg_nb[(size_t)r].clear();
        std::stable_sort(reg_nb[(size_t)target].begin(), reg_nb[(size_t)target].end(), by_first);
    }
    // 4. assembleRegions (empty regions erased, order kept) + extract()'s size filter
    std::vector<int32_t> rank((size_t)n_reg, -1);
    int64_t kept = 0;
    for (int r = 0; r < n_reg; ++r) if (reg_pts[(size_t)r] > 0 && reg_pts[(size_t)r] >= min_size && reg_pts[(size_t)r] <= max_size) rank[(size_t)r] = (int32_t)kept++;
    for (int64_t i = 0; i < n; ++i) labels[i] = rank[(size_t)seg_label[(size_t)point_label[(size_t)i]]];
    *n_clusters = kept;
    return PCC_OK;
}

// IterativeClosestPoint::computeTransformation as the reference configures it (src/comparator.cpp:1089-1099):
// max_iter iterations, transformation_epsilon 0 (rotation threshold 1.0, translation threshold 0), absolute MSE
// threshold 1e-12, relative MSE threshold -DBL_MAX (never), no rejectors, no correspondence distance limit.
int pcc_icp_align(pcc_index *idx, const void *src, int64_t ns, int stride_bytes, int max_iter, float T16[16], int *converged, double *fitness, int *iterations, int mem, void *stream) {
    PCC_TRY(check_index(idx, stream));
    if (ns < 0 || (ns > 0 && !src) || stride_bytes < 12 || (stride_bytes & 3) || !T16) return fail(PCC_ERR_INVALID, "bad source cloud");
    cudaStream_t s = (cudaStream_t)stream;
    float Tfinal[16], Tstep[16];
    for (int i = 0; i < 16; ++i) Tfinal[i] = (i % 5 == 0) ? 1.f : 0.f;
    int it = 0, conv = 0;
    double fit = DBL_MAX;
    // device working copy of the source (float4 rows), moved in place every iteration like PCL's input_transformed
    const uint8_t *raw = nullptr;
    PCC_TRY(stage_in(idx->stage4, (const uint8_t *)src, (size_t)ns * stride_bytes, mem, s, &raw));     // stage4 is free after pcc_build
    PCC_TRY(idx->parent.reserve((size_t)std::max<int64_t>(ns, 1) * sizeof(float4) + 64));
    float4 *cur = idx->parent.as<float4>();
    float *d_T = (float *)(cur + std::max<int64_t>(ns, 1));
    if (ns > 0) {
        PCC_CUDA(cudaMemcpyAsync(d_T, Tfinal, 64, cudaMemcpyHostToDevice, s));
        xform_kernel<<<nblocks(ns, 256), 256, 0, s>>>(raw, stride_bytes, ns, d_T, cur); PCC_LAUNCHED();   // identity: plain copy to float4
        PCC_CUDA(cudaGetLastError());
    }
    double prev_mse = DBL_MAX;
    const float *apply = nullptr;
    struct OrderReset { pcc_index *i; ~OrderReset() { i->reuse_order_n = -1; i->icp_allreduce = false; } } order_reset{idx};   // also on the error returns below
    idx->icp_allreduce = idx->comm != nullptr && idx->comm_world > 1;      // with a communicator `src` is this rank's shard of the source cloud
    idx->reuse_order_n = -1;
    idx->icp_prior_n = -1;        // a new alignment starts from the untransformed source: matches left by an earlier one are loose bounds (measured: first pass 31 ms with them, 17 ms without)
    static const bool trace = getenv("PCC_ICP_TRACE") != nullptr;     // per-pass kernel time on stderr (needs pcc_set_timing)
    for (;;) {
        double sums[16]; int64_t cnt = 0;
        PCC_TRY(pcc_icp_step(idx, cur, ns, sizeof(float4), apply, sums, &cnt, nullptr, nullptr, PCC_DEVICE, s));
        idx->reuse_order_n = ns;                                  // later passes keep this pass's processing order (no key sort)
        if (trace) fprintf(stderr, "[pcc icp] pass %d: %.2f ms, %lld correspondences, mse %.3e\n", it, idx->last_ms, (long long)cnt, cnt ? sums[15] / (double)cnt : 0.0);
        if (cnt < 3) { conv = 0; break; }                        // "Not enough correspondences found"
        PCC_TRY(pcc_umeyama_from_sums(sums, cnt, Tstep));
        mat4_mul(Tstep, Tfinal, Tfinal);
        apply = Tstep;                                            // transformCloud is fused into the next pass
        ++it;
        if (it >= max_iter) { conv = 1; break; }                  // CONVERGENCE_CRITERIA_ITERATIONS
        const double cos_angle = 0.5 * ((double)Tstep[0] + (double)Tstep[5] + (double)Tstep[10] - 1);
        const double tr2 = (double)Tstep[3] * Tstep[3] + (double)Tstep[7] * Tstep[7] + (double)Tstep[11] * Tstep[11];
        if (cos_angle >= 1.0 && tr2 <= 0.0) { conv = 1; break; } // CONVERGENCE_CRITERIA_TRANSFORM
        const double mse = sums[15] / (double)cnt;
        if (std::fabs(mse - prev_mse) < 1e-12) { conv = 1; break; }   // CONVERGENCE_CRITERIA_ABS_MSE
        prev_mse = mse;
    }
    // getFitnessScore: ORIGINAL source moved by the final transform, mean 1-NN squared distance (still the same rows, near their last position)
    if (ns > 0) {
        PCC_CUDA(cudaMemcpyAsync(d_T, Tfinal, 64, cudaMemcpyHostToDevice, s));
        xform_kernel<<<nblocks(ns, 256), 256, 0, s>>>(raw, stride_bytes, ns, d_T, cur); PCC_LAUNCHED();
        PCC_CUDA(cudaGetLastError());
        double sums[16]; int64_t cnt = 0;
        PCC_TRY(pcc_icp_step(idx, cur, ns, sizeof(float4), nullptr, sums, &cnt, nullptr, nullptr, PCC_DEVICE, s));
        if (cnt > 0) fit = sums[15] / (double)cnt;
    }
    memcpy(T16, Tfinal, sizeof(Tfinal));
    if (converged) *converged = conv;
    if (fitness) *fitness = fit;
    if (iterations) *iterations = it;
    return PCC_OK;
}

}  // extern "C"
