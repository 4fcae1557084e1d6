// pcc_descriptor.cu -- descriptor-space 1-NN (SURVEY.md section 8f, "next" row 3).
//
// Replaces matchRIFTFeaturesKnn (src/comparator.cpp:560-588): pcl::KdTreeFLANN<Histogram<32>> over the descriptors of
// cloud 1, one nearestKSearch(k = 1) per descriptor of cloud 2, a match when the squared distance is below 0.05.
// N is small (hundreds to a few thousand descriptors per cluster) and the dimension is 32, so the GPU path is an exact
// brute force: one thread per query descriptor, reference descriptors staged through shared memory in tiles, squared
// L2 accumulated sequentially over the dimensions in fp32 without FMA (FLANN L2_Simple), ties broken by index.
// Non-finite reference descriptors are skipped (KdTreeFLANN::setInputCloud); a non-finite query has no match.
//
// `dim` = the number of LEADING floats of a descriptor row that take part (distance and the finiteness test); rows are
// stride_floats apart.  The reference never registers pcl::Histogram<32> as a point struct and passes no point representation, so
// PCL 1.7's DefaultPointRepresentation<PointT> applies: nr_dimensions_ = sizeof(PointT) / sizeof(float) CLAMPED TO 3
// (pcl/point_representation.h [up]) -- the reference binary builds a 3-D tree over the first three histogram bins and its
// `squaredDistances[0] < 0.05f` test sees only those.  dim = 3 is therefore the reference-exact setting and dim = 32 what the
// author presumably intended; both are instantiated, the host mirrors default to 3 (INTEGRATION.md).
#include <algorithm>
#include <cmath>

#include "pcc_internal.h"

namespace pcc {

static constexpr int kDescTile = 64, kDescThreads = 128;

template <int D>
__global__ void __launch_bounds__(kDescThreads) descriptor_nn_kernel(const float *__restrict__ ref, int64_t n_ref, int ref_stride, const float *__restrict__ qry, int64_t n_qry,
                                                                     int qry_stride, int32_t *__restrict__ out_idx, float *__restrict__ out_d2) {
    __shared__ float tile[kDescTile][D + 1];
    __shared__ int tile_ok[kDescTile];
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    float q[D];
    bool q_ok = t < n_qry;
    if (q_ok) {
#pragma unroll
        for (int i = 0; i < D; ++i) { q[i] = qry[t * qry_stride + i]; q_ok = q_ok && isfinite(q[i]); }
    } else {
#pragma unroll
        for (int i = 0; i < D; ++i) q[i] = 0.f;
    }
    float best = CUDART_INF_F; int32_t best_i = -1;
    for (int64_t base = 0; base < n_ref; base += kDescTile) {
        const int cnt = (int)min((int64_t)kDescTile, n_ref - base);
        __syncthreads();
        for (int e = threadIdx.x; e < cnt * D; e += blockDim.x) { const int r = e / D, i = e - r * D; tile[r][i] = ref[(base + r) * ref_stride + i]; }
        __syncthreads();
        if ((int)threadIdx.x < cnt) { bool ok = true; for (int i = 0; i < D; ++i) ok = ok && isfinite(tile[threadIdx.x][i]); tile_ok[threadIdx.x] = ok; }
        __syncthreads();
        if (q_ok) {
            for (int r = 0; r < cnt; ++r) {
                if (!tile_ok[r]) continue;
                float d2 = 0.f;
#pragma unroll
                for (int i = 0; i < D; ++i) { const float diff = __fsub_rn(q[i], tile[r][i]); d2 = __fadd_rn(d2, __fmul_rn(diff, diff)); }
                if (d2 < best) { best = d2; best_i = (int32_t)(base + r); }       // strict <: the lowest index wins a tie
            }
        }
    }
    if (t < n_qry) { out_idx[t] = best_i; out_d2[t] = best; }
}

}  // namespace pcc

using namespace pcc;

extern "C" int pcc_descriptor_nn(pcc_index *ws, const float *ref, int64_t n_ref, const float *qry, int64_t n_qry, int dim, int stride_floats,
                                 int32_t *out_idx, float *out_d2, int mem, void *stream) {
    if (!ws) return fail(PCC_ERR_INVALID, "workspace index is NULL");
    if (n_ref < 0 || n_qry < 0 || (n_ref > 0 && !ref) || (n_qry > 0 && (!qry || !out_idx || !out_d2)) || stride_floats < dim) return fail(PCC_ERR_INVALID, "bad arguments");
    if (dim != 32 && dim != 3) return fail(PCC_ERR_INVALID, "descriptor dimension %d is not instantiated (3 = what PCL 1.7 compares for Histogram<32>, 32 = all RIFT32 bins)", dim);
    PCC_CUDA(cudaSetDevice(ws->device));
    cudaStream_t s = (cudaStream_t)stream;
    if (n_qry == 0) return PCC_OK;
    const float *d_ref = nullptr, *d_qry = nullptr;
    PCC_TRY(stage_in(ws->raw, ref, (size_t)n_ref * stride_floats * 4, mem, s, &d_ref));
    PCC_TRY(stage_in(ws->stage4, qry, (size_t)n_qry * stride_floats * 4, mem, s, &d_qry));
    int32_t *d_oi = out_idx; float *d_od = out_d2;
    if (mem == PCC_HOST) {
        PCC_TRY(ws->out_i.reserve((size_t)n_qry * 4)); PCC_TRY(ws->out_f.reserve((size_t)n_qry * 4));
        d_oi = ws->out_i.as<int32_t>(); d_od = ws->out_f.as<float>();
    }
    const unsigned nb = (unsigned)((n_qry + kDescThreads - 1) / kDescThreads);
    if (dim == 3) descriptor_nn_kernel<3><<<nb, kDescThreads, 0, s>>>(d_ref, n_ref, stride_floats, d_qry, n_qry, stride_floats, d_oi, d_od);
    else descriptor_nn_kernel<32><<<nb, kDescThreads, 0, s>>>(d_ref, n_ref, stride_floats, d_qry, n_qry, stride_floats, d_oi, d_od);
    PCC_LAUNCHED();
    PCC_CUDA(cudaGetLastError());
    if (mem == PCC_HOST) {
        PCC_TRY(copy_out(out_idx, d_oi, (size_t)n_qry * 4, mem, s));
        PCC_TRY(copy_out(out_d2, d_od, (size_t)n_qry * 4, mem, s));
        PCC_CUDA(cudaStreamSynchronize(s));
    }
    return PCC_OK;
}
