// pcc_internal.h -- host-side state behind the opaque pcc_index of include/pcc/search.h.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <algorithm>
#include <atomic>
#include <string>

#include "../../include/pcc/search.h"
#include "pcc_device.cuh"

namespace pcc {

extern thread_local std::string g_error;
extern std::atomic<int64_t> g_launches;
int fail(int code, const char *fmt, ...);

#define PCC_CUDA(expr)                                                                                   \
    do {                                                                                                 \
        cudaError_t e__ = (expr);                                                                        \
        if (e__ != cudaSuccess) return pcc::fail(PCC_ERR_CUDA, "%s:%d %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(e__)); \
    } while (0)
#define PCC_TRY(expr)                 \
    do {                              \
        int r__ = (expr);             \
        if (r__ != PCC_OK) return r__; \
    } while (0)
#define PCC_LAUNCHED() (++pcc::g_launches)

// grow-only device buffer
struct Buf {
    void *p = nullptr;
    size_t cap = 0;
    int reserve(size_t bytes) {
        if (bytes <= cap) return PCC_OK;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) { p = nullptr; return fail(PCC_ERR_CUDA, "cudaMalloc(%zu) -> %s", want, cudaGetErrorString(e)); }
        cap = want;
        return PCC_OK;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <class T> T *as() const { return (T *)p; }
};

struct GridHost {
    float ox = 0, oy = 0, oz = 0, cell = 1, inv_cell = 1;
    int nx = 1, ny = 1, nz = 1;
    double occupancy = 0;      // mean points per non-empty cell
    double block_fill = 0;     // occupied cells per 3x3x3 block around a point, measured on the first auto-tune grid (0 = not measured)
    int64_t n_cells = 1;
};

}  // namespace pcc

struct pcc_index {
    int device = 0;
    bool built = false;
    int64_t n_input = 0;      // rows handed to pcc_build (label / self-query row count)
    int64_t n_indexed = 0;    // finite rows
    bool all_rows_indexed = false;   // every input row is in the index exactly once (no `indices` list, no non-finite row): self-query outputs need no pre-fill
    pcc::GridHost gh;
    pcc::Buf pts;             // float4 [n_indexed], sorted by cell
    pcc::Buf cell_start;      // uint32 [n_cells + 1]
    pcc::Buf occ;             // uint32 [n_cells / 32 + 2]: one bit per cell, set when the cell holds a point (derived from cell_start)
    pcc::Buf occ2, cstart;    // compact cell table (pcc_device.cuh cell_begin): uint2 per 32 cells, uint32 per non-empty cell
    bool occ_valid = false;
    // scratch (grow-only, reused by every call on this index; calls on one index are serialised by the caller per stream)
    pcc::Buf raw, stage4, cellrank, qbuf, qkeys, qkeys2, qperm, qperm2, cub_tmp, out_i, out_f, out_l, keys64, keys64b, misc, parent, inv_pos, sel_params, icp_prior, calib;
    // pcc_sift_*: the octave clouds (ping-pong, float4 x, y, z, packed rgb) live outside the scratch pcc_voxel_grid and pcc_build reuse
    pcc::Buf sift_cloud[2], sift_val, sift_dog, sift_in, sift_nbr, sift_d2, sift_flag, sift_pos, sift_row, sift_col, sift_kp;
    // pcc_sift_keypoints_batched: segment label per sorted position of the current grid (segment_labels), the octave's segment
    // offsets, per-segment tables, per-row segment labels of the segmented VoxelGrid and the keypoints staged across octaves
    pcc::Buf seg_label, seg_off, sift_tab, sift_lab, sift_stage;
    // pcc_rift_batched: one stage's rows derived from the master rows (offsets, keys, scan scratch), the staged intensity, per-row
    // normals, gradients and descriptors, the survivor scan, the cluster offsets and bounds, and the compacted rows of a PCC_HOST call
    pcc::Buf rift_off, rift_keys, rift_tmp, rift_in, rift_nrm, rift_grad, rift_desc, rift_pos, rift_tab, rift_out, rift_row;
    // pcc_knn_batched: the cluster offsets and the finite points per cluster
    pcc::Buf knnb_tab;
    uint64_t grid_gen = 0;     // bumped by pcc_build / pcc_adopt
    void *comm = nullptr;      // ncclComm_t handed to pcc_comm_init (not owned); rank / world of this process in it
    int comm_rank = 0, comm_world = 1;
    // host-side launch cost matters once a rank's shard is ~1 M queries (0.5 ms of GPU work per call): CUB's temp-size queries and
    // the per-function attributes are done once, not per call
    int64_t sel_tmp_nq = -1; size_t sel_tmp_bytes = 0; int64_t sort_tmp_nq = -1; int sort_tmp_bits = 0; size_t sort_tmp_bytes = 0;
    bool icp_allreduce = false;   // pcc_icp_step sums its 17 doubles over the ranks (set by pcc_icp_align while it runs on a sharded source)
    int calib_k = -1;          // k the logging-threshold table in `calib` was calibrated for (-1: none), on grid generation calib_gen of the grid owner
    uint64_t calib_gen = 0;
    int64_t calib_nq = 0;      // batch size of the call that last ran the block kernel (fallback monitor, see launch_knn_fast)
    int64_t reuse_order_n = -1;  // pcc_icp_align: the processing order of the previous pass is kept for this many rows (points move by millimetres between passes; the order only matters for locality)
    int64_t icp_prior_n = -1;  // rows of icp_prior that hold sorted positions into the CURRENT grid (-1: none; reset by pcc_build / pcc_adopt)
    bool inv_valid = false;   // inv_pos (original row -> sorted position) is built lazily by the consumers that need it
    void *h_pinned = nullptr;  // 4 KiB pinned scratch for scalar read-backs
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    bool timing = false;
    double last_ms = -1;

    // host-buffer calls on large batches are pipelined over two slots (this index and a scratch-only shadow that borrows
    // the grid): chunk i copies in / searches / copies out on stream i & 1, so PCIe traffic of one chunk overlaps the
    // kernels of the other
    pcc_index *shadow = nullptr;
    const pcc_index *grid_owner = nullptr;
    cudaStream_t pipe_stream[2] = {nullptr, nullptr};
    // the wide pass of pcc_knn runs beside the ring pass on this stream (both are latency-bound and touch different rows)
    cudaStream_t aux_stream = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;

    pcc::Grid grid() const {
        const pcc_index *o = grid_owner ? grid_owner : this;
        pcc::Grid g;
        g.pts = o->pts.as<float4>(); g.cell_start = o->cell_start.as<uint32_t>(); g.occ = o->occ.as<uint32_t>(); g.occ2 = o->occ2.as<uint2>(); g.cstart = o->cstart.as<uint32_t>();
        g.ox = o->gh.ox; g.oy = o->gh.oy; g.oz = o->gh.oz; g.inv_cell = o->gh.inv_cell; g.cell = o->gh.cell;
        g.nx = o->gh.nx; g.ny = o->gh.ny; g.nz = o->gh.nz; g.n = (uint32_t)o->n_indexed;
        return g;
    }
};

namespace pcc {
// prepared query batch: float4 queries on device + the processing order
struct Queries {
    const float4 *q = nullptr;     // [nq] (x, y, z, _)
    const uint32_t *order = nullptr;  // [nq] query rows sorted by grid cell (non-finite last); nullptr in self mode
    int64_t nq = 0;
    bool self = false;             // queries are the indexed cloud itself: thread t handles sorted point t, row = original index
    int64_t rows = 0;              // number of output rows (nq, or n_input in self mode)
};
static inline QueryView view_of(const Queries &q) { return QueryView{q.q, q.order, q.nq, q.self}; }
static inline unsigned nblocks(int64_t n, int threads) { return (unsigned)std::max<int64_t>(1, (n + threads - 1) / threads); }
// block size of the kernels that keep k keys per thread in dynamic shared memory (up to 96 KB of keys a block)
static inline int heap_threads(int k) {
    int t = (int)((96 * 1024) / ((size_t)k * sizeof(nkey_t)));
    t = std::min(128, (t / 32) * 32);
    return std::max(32, t);
}
template <class Kern>
static int set_heap_smem(Kern kern) {
    PCC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));   // per device: set on every launch (cheap)
    return PCC_OK;
}
// an entry's input array on the device: the caller's pointer (PCC_DEVICE), or a copy in `buf` (PCC_HOST)
template <class T>
static int stage_in(Buf &buf, const T *src, size_t bytes, int mem, cudaStream_t s, const T **dev) {
    *dev = src;
    if (mem != PCC_HOST) return PCC_OK;
    PCC_TRY(buf.reserve(std::max<size_t>(bytes, 16)));
    if (bytes) PCC_CUDA(cudaMemcpyAsync(buf.p, src, bytes, cudaMemcpyHostToDevice, s));
    *dev = buf.as<T>();
    return PCC_OK;
}
// per-row results are written to the caller's pointer (PCC_DEVICE) or to out_f (PCC_HOST); deliver_rows copies the
// latter back and returns with them on the host
template <class T>
static int output_rows(pcc_index *idx, T *out, size_t bytes, int mem, T **dev) {
    *dev = out;
    if (mem == PCC_HOST) { PCC_TRY(idx->out_f.reserve(bytes)); *dev = idx->out_f.as<T>(); }
    return PCC_OK;
}
int copy_out(void *dst, const void *src_dev, size_t bytes, int mem, cudaStream_t s);
static inline int deliver_rows(void *out, const void *dev, size_t bytes, int mem, cudaStream_t s) {
    if (mem == PCC_HOST) { PCC_TRY(copy_out(out, dev, bytes, mem, s)); PCC_CUDA(cudaStreamSynchronize(s)); }
    return PCC_OK;
}
// every entry that searches the grid: idx is a built index, its device is current, and after pcc_adopt the occupancy bitmap is
// derived on the caller's stream (ordered after the caller's fill of cell_start, before its next kernel)
int check_index(pcc_index *idx, void *stream);
int prepare_queries(pcc_index *idx, const void *q, int64_t nq, int stride_bytes, int mem, cudaStream_t s, Queries *out);
int rebuild_inverse(pcc_index *idx, cudaStream_t s);
int comm_allreduce_f64(pcc_index *idx, double *d_buf, int n, cudaStream_t s);   // pcc_comm.cu; no-op without a communicator
// k > 32: neighbours by selection (pcc_radius.cu); rows are sorted by (d2, index), oi / od are device pointers
int knn_select(pcc_index *idx, const Queries &qs, int k, int32_t *oi, float *od, cudaStream_t s);
// ---- segmented clouds: segment c is rows [off[c], off[c+1]) of a concatenation (pcc_sift_keypoints_batched) ----
// idx->seg_label[sorted position] = segment of the point's original row; d_off is a device array of n_seg + 1 offsets
int segment_labels(pcc_index *idx, const int64_t *d_off, int n_seg, cudaStream_t s);
// the indexed cloud's own radius rows with neighbours of the query's segment only, sorted by (d2, index): offsets (n_input + 1,
// in idx->out_l) and keys (idx->keys64); rows of unindexed points are empty
int segmented_sorted_rows(pcc_index *idx, const uint32_t *seg, double radius, const int64_t **d_off, const nkey_t **keys, cudaStream_t s);
// pcc_knn(q == NULL, k) of every segment alone, for any 1 <= k <= PCC_MAX_K, over the selection path: the dense [n_input, k] table
// oi / od with segment-LOCAL indices (row - seg_off[segment]), (d2, index) order, rows past min(k, seg_n[segment]) and rows of
// unindexed points (-1, +inf).  seg_n (finite points per segment), seg_off (n_seg + 1), oi and od are device pointers.
int knn_select_segmented(pcc_index *idx, const uint32_t *seg, const uint32_t *seg_n, const int64_t *seg_off, int k, int32_t *oi, float *od, cudaStream_t s);
// pcc_sift_dog over segmented_sorted_rows (device pointers, no checks); rows of unindexed points are NaN
int sift_dog_segmented(pcc_index *idx, const uint32_t *seg, const float *values, const float *scales, int n_scales, float *out, cudaStream_t s);
// processRIFT's normals, gradient and RIFT stages over one segmented_sorted_rows pass at the largest radius (pcc_rift_batched): each
// stage's rows are a prefix of the master rows, less the neighbours with a non-finite normal for the gradient and RIFT stages, and
// empty for a query whose own normal is not finite.  normals / gradient (float4) and desc (nd * ng floats) have one row per input row;
// rows of unindexed points get NaN normals and undefined gradients and descriptors.  All pointers are device pointers.
int rift_segmented(pcc_index *idx, const uint32_t *seg, const float *intensity, double normal_radius, double gradient_radius, double rift_radius,
                   int nd, int ng, float4 *normals, float4 *gradient, float *desc, cudaStream_t s);
// pcc_first_within restricted to the query's segment: query t belongs to segment segment_of(d_qoff, t), the indexed points carry
// their segment in seg, and out[t] is relative to that segment's first row (d_poff).  q, d_qoff, d_poff and out are device pointers.
int first_within_segmented(pcc_index *idx, const uint32_t *seg, const float4 *q, int64_t nq, const int64_t *d_qoff, const int64_t *d_poff, int n_seg,
                           double thr, int32_t *out, cudaStream_t s);
// VoxelGrid (leaf in every axis, rgb averaged) of every segment of a float4 (x, y, z, rgb word) cloud, each segment with its own
// bounding box, exactly as pcc_voxel_grid on that segment alone.  in_off / out_off are host arrays of n_seg + 1 offsets.  A
// segment whose result has fewer than min_rows rows is dropped (no rows in `out`); the others are written in segment order.
int segmented_voxel_grid(pcc_index *idx, const float4 *in, const int64_t *in_off, int n_seg, float leaf, int64_t min_rows, float4 *out, int64_t *out_off,
                         cudaStream_t s);
struct KernelTimer {
    pcc_index *idx; cudaStream_t s;
    KernelTimer(pcc_index *i, cudaStream_t st) : idx(i), s(st) { if (idx->timing) cudaEventRecord(idx->ev0, s); }
    void stop() { if (idx->timing) { cudaEventRecord(idx->ev1, s); cudaEventSynchronize(idx->ev1); float ms = 0; cudaEventElapsedTime(&ms, idx->ev0, idx->ev1); idx->last_ms = ms; } }
};
}  // namespace pcc
