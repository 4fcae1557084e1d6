// pcc_build.cu -- index lifetime, uniform-grid build (cell keys -> counting sort -> cell-start scan) and
// query-batch preparation (cell keys -> radix sort) for libpcc_search.so.
//
// Replaces pcl::search::KdTree::setInputCloud -> KdTreeFLANN::setInputCloud -> flann::KDTreeSingleIndex::buildIndex
// (reference call sites: src/segmentation.cpp:122 and implicitly every consumer, SURVEY.md section 8 a1).
#include <cub/cub.cuh>
#include <stdarg.h>
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <vector>

#include <cstring>
#include "pcc_internal.h"

namespace pcc {

thread_local std::string g_error;
std::atomic<int64_t> g_launches{0};

int fail(int code, const char *fmt, ...) {
    char buf[1024];
    va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof(buf), fmt, ap); va_end(ap);
    g_error = buf;
    return code;
}

static constexpr int kMaxDim = 2048;                 // covered_d2()'s rounding margin assumes this cap
static constexpr int64_t kMaxCellsDefault = 1ll << 28;      // hard cap: knn_rings_kernel packs (first cell | (cells - 1) << 28) in one uint32 (pcc_knn.cu)

__device__ __forceinline__ int f2ord(float f) { int i = __float_as_int(f); return i >= 0 ? i : i ^ 0x7FFFFFFF; }
static inline float ord2f(int i) { int j = i >= 0 ? i : i ^ 0x7FFFFFFF; float f; memcpy(&f, &j, 4); return f; }

// raw strided rows -> float4 (x, y, z, original row as int bits; NaN w marks a skipped row) + bbox + finite count
__global__ void extract_kernel(const uint8_t *__restrict__ raw, int stride, const int32_t *__restrict__ indices, int64_t m,
                               int64_t n_rows, float4 *__restrict__ stage, int *__restrict__ bbox, unsigned long long *__restrict__ n_finite) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int lo[3] = {INT_MAX, INT_MAX, INT_MAX}, hi[3] = {INT_MIN, INT_MIN, INT_MIN};
    int fin = 0;
    if (i < m) {
        int64_t row = indices ? (int64_t)indices[i] : i;
        float x = CUDART_NAN_F, y = x, z = x;
        if (row >= 0 && row < n_rows) {
            const float *p = (const float *)(raw + row * (int64_t)stride);
            x = p[0]; y = p[1]; z = p[2];
        }
        fin = finite3(x, y, z);
        stage[i] = make_float4(x, y, z, fin ? __int_as_float((int)row) : CUDART_NAN_F);
        if (fin) { lo[0] = hi[0] = f2ord(x); lo[1] = hi[1] = f2ord(y); lo[2] = hi[2] = f2ord(z); }
    }
#pragma unroll
    for (int d = 0; d < 3; ++d) { lo[d] = __reduce_min_sync(0xffffffffu, lo[d]); hi[d] = __reduce_max_sync(0xffffffffu, hi[d]); }
    unsigned nf = __reduce_add_sync(0xffffffffu, (unsigned)fin);
    if ((threadIdx.x & 31) == 0 && nf) {
#pragma unroll
        for (int d = 0; d < 3; ++d) { atomicMin(bbox + d, lo[d]); atomicMax(bbox + 3 + d, hi[d]); }
        atomicAdd(n_finite, (unsigned long long)nf);
    }
}

struct BinParams { float ox, oy, oz, inv; int nx, ny, nz; };
constexpr int64_t kFillSamples = 1 << 17;                 // points sampled by blockfill_kernel
constexpr double kFillSurface = 15.0, kFillVolume = 21.0;  // occupied cells per 3x3x3 block: at or below = surface target, at or above = volume target, linear between
__device__ __forceinline__ uint32_t cell_of(const BinParams &b, float x, float y, float z) {
    int cx = grid_c(grid_u(x, b.ox, b.inv), b.nx), cy = grid_c(grid_u(y, b.oy, b.inv), b.ny), cz = grid_c(grid_u(z, b.oz, b.inv), b.nz);
    return (uint32_t)(((size_t)cz * b.ny + cy) * b.nx + cx);
}
// counting sort pass 1: per-cell histogram; the atomic's return value is the point's rank inside its cell
__global__ void bin_kernel(const float4 *__restrict__ stage, int64_t m, BinParams b, uint32_t *__restrict__ counts, uint2 *__restrict__ cellrank) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    float4 p = stage[i];
    if (p.w != p.w) { if (cellrank) cellrank[i] = make_uint2(0xFFFFFFFFu, 0u); return; }
    uint32_t c = cell_of(b, p.x, p.y, p.z);
    uint32_t r = atomicAdd(counts + c, 1u);
    if (cellrank) cellrank[i] = make_uint2(c, r);
}
// How many of the 27 cells around a point's cell hold a point, summed over every `stride`-th staged point: ~27 for a cloud that fills
// its volume, 9-13 for a surface.  `counts` is the per-cell histogram (before the scan).  out[0] += occupied neighbours, out[1] += samples.
__global__ void blockfill_kernel(const float4 *__restrict__ stage, int64_t m, int64_t stride, BinParams b, const uint32_t *__restrict__ counts, unsigned long long *__restrict__ out) {
    const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * stride;
    unsigned filled = 0, sample = 0;
    if (i < m) {
        const float4 p = stage[i];
        if (p.w == p.w) {
            const int cx = grid_c(grid_u(p.x, b.ox, b.inv), b.nx), cy = grid_c(grid_u(p.y, b.oy, b.inv), b.ny), cz = grid_c(grid_u(p.z, b.oz, b.inv), b.nz);
            sample = 1;
            for (int z = max(cz - 1, 0); z <= min(cz + 1, b.nz - 1); ++z)
                for (int y = max(cy - 1, 0); y <= min(cy + 1, b.ny - 1); ++y)
                    for (int x = max(cx - 1, 0); x <= min(cx + 1, b.nx - 1); ++x)
                        filled += counts[((size_t)z * b.ny + y) * b.nx + x] > 0u ? 1u : 0u;
        }
    }
    filled = __reduce_add_sync(0xffffffffu, filled); sample = __reduce_add_sync(0xffffffffu, sample);
    if ((threadIdx.x & 31) == 0 && sample) { atomicAdd(out, (unsigned long long)filled); atomicAdd(out + 1, (unsigned long long)sample); }
}
__global__ void nonzero_kernel(const uint32_t *__restrict__ counts, int64_t n, unsigned long long *__restrict__ out) {
    unsigned local = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) local += counts[i] != 0;
    local = __reduce_add_sync(0xffffffffu, local);
    if ((threadIdx.x & 31) == 0 && local) atomicAdd(out, (unsigned long long)local);
}
// counting sort pass 2: scatter to cell_start[cell] + rank
__global__ void scatter_kernel(const float4 *__restrict__ stage, const uint2 *__restrict__ cellrank, int64_t m,
                               const uint32_t *__restrict__ cell_start, float4 *__restrict__ pts) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    uint2 cr = cellrank[i];
    if (cr.x == 0xFFFFFFFFu) return;
    pts[cell_start[cr.x] + cr.y] = stage[i];
}
// inv_pos[original row] = position in the sorted array (0xFFFFFFFF for rows that are not indexed)
__global__ void inverse_kernel(const float4 *__restrict__ pts, int64_t n, uint32_t *__restrict__ inv_pos) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) inv_pos[__float_as_int(pts[i].w)] = (uint32_t)i;
}
// occ bit c = cell c is not empty.  The dense cell_start table is far larger than L2 on big grids (56 M cells = 225 MB at
// the 10 M-point headline size) while the bitmap is 7 MB, so the ring passes that mostly verify EMPTY cells around a block
// test the bitmap first and touch cell_start only where there is something to read.
__global__ void occupancy_kernel(const uint32_t *__restrict__ cell_start, int64_t n_cells, uint32_t *__restrict__ occ) {
    const int64_t words = (n_cells + 31) / 32 + 1;
    for (int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; c < words * 32; c += (int64_t)gridDim.x * blockDim.x) {
        const bool full = c < n_cells && cell_start[c + 1] > cell_start[c];
        const unsigned w = __ballot_sync(0xffffffffu, full);
        if ((threadIdx.x & 31) == 0) occ[c >> 5] = w;
    }
}
struct PopcOp { __device__ __forceinline__ uint32_t operator()(uint32_t w) const { return (uint32_t)__popc(w); } };
// compact table: occ2[w] = {occ word, non-empty cells before it}; cstart[rank] = cell_start of the rank-th non-empty cell; cstart[total] = n
__global__ void compact_table_kernel(const uint32_t *__restrict__ occ, const uint32_t *__restrict__ wprefix, int64_t words, const uint32_t *__restrict__ cell_start,
                                     int64_t n_cells, uint2 *__restrict__ occ2, uint32_t *__restrict__ cstart) {
    const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= words) return;
    uint32_t bits = occ[w], r = wprefix[w];
    occ2[w] = make_uint2(bits, r);
    while (bits) { const int b = __ffs(bits) - 1; bits &= bits - 1; cstart[r++] = cell_start[w * 32 + b]; }
    if (w == words - 1) cstart[r] = cell_start[n_cells];
}
// occ bitmap from cell_start (after pcc_build / pcc_adopt)
static int rebuild_occupancy(pcc_index *idx, cudaStream_t s) {
    const int64_t n_cells = std::max<int64_t>(idx->gh.n_cells, 1);
    const int64_t words = (n_cells + 31) / 32 + 1;
    PCC_TRY(idx->occ.reserve((size_t)words * 4));
    const int64_t threads = words * 32;
    occupancy_kernel<<<(unsigned)std::min<int64_t>((threads + 255) / 256, 148 * 32), 256, 0, s>>>(idx->cell_start.as<uint32_t>(), idx->gh.n_cells, idx->occ.as<uint32_t>());
    PCC_LAUNCHED();
    PCC_CUDA(cudaGetLastError());
#if PCC_COMPACT_TABLE      // measurement build (DESIGN.md section 5): parity-clean, 8 % slower than the dense table on the headline workload
    PCC_TRY(idx->occ2.reserve((size_t)(words + 1) * sizeof(uint2)));
    PCC_TRY(idx->cstart.reserve((size_t)(std::min<int64_t>(n_cells, std::max<int64_t>(idx->n_indexed, 0)) + 2) * 4));
    PCC_TRY(idx->qkeys2.reserve((size_t)words * 4));          // scratch: per-word prefix
    size_t tmp = 0;
    cub::TransformInputIterator<uint32_t, PopcOp, const uint32_t *> pc(idx->occ.as<uint32_t>(), PopcOp());
    cub::DeviceScan::ExclusiveSum(nullptr, tmp, pc, idx->qkeys2.as<uint32_t>(), (int)words, s);
    PCC_TRY(idx->cub_tmp.reserve(tmp));
    PCC_CUDA(cub::DeviceScan::ExclusiveSum(idx->cub_tmp.p, tmp, pc, idx->qkeys2.as<uint32_t>(), (int)words, s));
    g_launches += 2;
    PCC_CUDA(cudaMemsetAsync(idx->occ2.as<uint2>() + words, 0, sizeof(uint2), s));
    compact_table_kernel<<<(unsigned)((words + 255) / 256), 256, 0, s>>>(idx->occ.as<uint32_t>(), idx->qkeys2.as<uint32_t>(), words, idx->cell_start.as<uint32_t>(), idx->gh.n_cells,
                                                                 idx->occ2.as<uint2>(), idx->cstart.as<uint32_t>());
    PCC_LAUNCHED();
    PCC_CUDA(cudaGetLastError());
#endif
    idx->occ_valid = true;
    return PCC_OK;
}
int check_index(pcc_index *idx, void *stream) {
    if (!idx) return fail(PCC_ERR_INVALID, "idx is NULL");
    if (!idx->built) return fail(PCC_ERR_STATE, "index not built (call pcc_build first)");
    PCC_CUDA(cudaSetDevice(idx->device));
    if (!idx->occ_valid) PCC_TRY(rebuild_occupancy(idx, (cudaStream_t)stream));     // first query after pcc_adopt
    return PCC_OK;
}
int rebuild_inverse(pcc_index *idx, cudaStream_t s) {
    PCC_TRY(idx->inv_pos.reserve((size_t)std::max<int64_t>(idx->n_input, 1) * 4));
    PCC_CUDA(cudaMemsetAsync(idx->inv_pos.p, 0xFF, (size_t)std::max<int64_t>(idx->n_input, 1) * 4, s));
    if (idx->n_indexed > 0) {
        inverse_kernel<<<(unsigned)((idx->n_indexed + 255) / 256), 256, 0, s>>>(idx->pts.as<float4>(), idx->n_indexed, idx->inv_pos.as<uint32_t>());
        PCC_LAUNCHED();
        PCC_CUDA(cudaGetLastError());
    }
    idx->inv_valid = true;
    return PCC_OK;
}

// query rows -> float4 + cell key (n_cells for non-finite rows so they sort last) + identity permutation
__global__ void qprep_kernel(const uint8_t *__restrict__ raw, int stride, int64_t nq, BinParams b, uint32_t bad_key,
                             float4 *__restrict__ qbuf, uint32_t *__restrict__ keys, uint32_t *__restrict__ perm) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nq) return;
    const float *p = (const float *)(raw + i * (int64_t)stride);
    float x = p[0], y = p[1], z = p[2];
    qbuf[i] = make_float4(x, y, z, 0.f);
    if (keys) { keys[i] = finite3(x, y, z) ? cell_of(b, x, y, z) : bad_key; perm[i] = (uint32_t)i; }
}

// Target points per NON-EMPTY cell.  PCC_OCC overrides it (measurement knob).
// Surface-like clouds, measured on B200 (10 M queries on a 10 M-point surface cloud, kNN ms at target 4 / 6 / 8 / 10 / 12): k = 4: 3.46 / 2.60 /
// 2.21 / - / -, k = 8: 4.31 / 3.14 / 2.71 / 2.76 / -, k = 16: - / 4.89 / 4.13 / 4.17 / 4.15, k = 32 at 12 / 16 / 20: 9.47 / 9.52 /
// 10.4; k = 1 (own kernel) at 3 / 4 / 8: 2.68 / 2.36 / 1.80.  With ~8 points per occupied cell the 3x3x3 block settles >80 % of the queries for k <= 16; smaller cells send too
// many of them to the ring passes, larger ones make the block walk longer.
static double occupancy_target(int k_hint) {
    int k = k_hint > 0 ? k_hint : 16;
    if (k == 1) return 12.0;       // k = 1 at 8 / 10 / 12 / 16 / 20: 1.79 / 1.74 / 1.62 / 1.64 / 1.70 ms (k = 2, 4, 8 are best at 8; profiles/r2/occupancy_surface_small_k.txt)
    return std::max(8.0, 0.5 * k);
}
// Volume-filling clouds: all 27 cells of a block are occupied (a surface fills 9-13), so the same block population needs
// a third of the points per cell.  Measured on a 10 M-point uniform cube, 10 M queries (profiles/r2/occupancy_uniform_cloud.txt), best
// target / kNN ms there vs ms at 8 per cell: k = 1: 1.3-1.9 / 0.99 vs 1.37; k = 2: 1.9 / 1.58 vs 2.16; k = 4: 1.9 / 1.66 vs 2.31 (1.3: 2.50);
// k = 8: 2.3-3.1 / 2.32 vs 3.02; k = 16: 4 / 3.63 vs 4.48; k = 32: 5-6 / 11.2 vs 12.4 (16, the surface target: 15.7; 3: 24.0).
// k > 32 (selection path) is flat in the target (k = 50: 20.4 ms at 4 and at 25).
static double occupancy_target_volume(int k_hint) {
    int k = k_hint > 0 ? k_hint : 16;
    if (k > 32) return 0.5 * k;
    return std::max(1.9, std::min(k / 3.5, 4.0 + (k - 16) / 10.0));
}
static bool occupancy_override(double *v) {
    const char *e = getenv("PCC_OCC");
    if (e && atof(e) > 0) { *v = atof(e); return true; }
    return false;
}

static void dims_for(const double ext[3], double cell, int dims[3]) {
    for (int d = 0; d < 3; ++d) dims[d] = (int)std::min<double>(kMaxDim, std::floor(ext[d] / cell) + 1);
}
static double clamp_cell(const double ext[3], double cell, int64_t max_cells) {
    double mx = std::max(ext[0], std::max(ext[1], ext[2]));
    if (!(cell > 0) || !std::isfinite(cell)) cell = mx > 0 ? mx : 1.0;
    cell = std::max(cell, mx / (kMaxDim - 1));
    for (int it = 0; it < 64; ++it) {
        int d[3]; dims_for(ext, cell, d);
        double total = (double)d[0] * d[1] * d[2];
        if (total <= (double)max_cells) break;
        cell *= std::max(1.02, std::cbrt(total / (double)max_cells));
    }
    return cell;
}

int prepare_queries(pcc_index *idx, const void *q, int64_t nq, int stride_bytes, int mem, cudaStream_t s, Queries *out) {
    if (!idx->built) return fail(PCC_ERR_STATE, "index not built (call pcc_build first)");
    if (q == nullptr) { out->self = true; out->nq = idx->n_indexed; out->rows = idx->n_input; out->q = nullptr; out->order = nullptr; return PCC_OK; }
    if (nq < 0 || nq >= (1ll << 31) - 1 || stride_bytes < 12 || (stride_bytes & 3)) return fail(PCC_ERR_INVALID, "bad query batch (nq=%lld stride=%d; nq must be below 2^31 - 1: row counts go to CUB as 32-bit ints)", (long long)nq, stride_bytes);
    out->self = false; out->nq = nq; out->rows = nq;
    if (nq == 0) return PCC_OK;
    const uint8_t *raw = (const uint8_t *)q;
    if (mem == PCC_HOST) {
        PCC_TRY(idx->raw.reserve((size_t)nq * stride_bytes));
        PCC_CUDA(cudaMemcpyAsync(idx->raw.p, q, (size_t)nq * stride_bytes, cudaMemcpyHostToDevice, s));
        raw = idx->raw.as<uint8_t>();
    }
    PCC_TRY(idx->qbuf.reserve((size_t)nq * sizeof(float4)));
    if (idx->reuse_order_n == nq && nq > 2048) {          // same rows as the previous pass, slightly moved: keep its order
        BinParams b0{idx->gh.ox, idx->gh.oy, idx->gh.oz, idx->gh.inv_cell, idx->gh.nx, idx->gh.ny, idx->gh.nz};
        qprep_kernel<<<nblocks(nq, 256), 256, 0, s>>>(raw, stride_bytes, nq, b0, (uint32_t)idx->gh.n_cells, idx->qbuf.as<float4>(), nullptr, nullptr);
        PCC_LAUNCHED();
        PCC_CUDA(cudaGetLastError());
        out->q = idx->qbuf.as<float4>();
        out->order = idx->qperm2.as<uint32_t>();
        return PCC_OK;
    }
    const bool sort = nq > 2048;
    BinParams b{idx->gh.ox, idx->gh.oy, idx->gh.oz, idx->gh.inv_cell, idx->gh.nx, idx->gh.ny, idx->gh.nz};
    if (sort) {
        PCC_TRY(idx->qkeys.reserve((size_t)nq * 4)); PCC_TRY(idx->qkeys2.reserve((size_t)nq * 4));
        PCC_TRY(idx->qperm.reserve((size_t)nq * 4)); PCC_TRY(idx->qperm2.reserve((size_t)nq * 4));
    }
    qprep_kernel<<<nblocks(nq, 256), 256, 0, s>>>(raw, stride_bytes, nq, b, (uint32_t)idx->gh.n_cells, idx->qbuf.as<float4>(),
                                                     sort ? idx->qkeys.as<uint32_t>() : nullptr, sort ? idx->qperm.as<uint32_t>() : nullptr);
    PCC_LAUNCHED();
    PCC_CUDA(cudaGetLastError());
    out->q = idx->qbuf.as<float4>();
    out->order = nullptr;
    if (sort) {
        int bits = 1; while ((1ll << bits) <= idx->gh.n_cells && bits < 32) ++bits;
        // The order only serves locality, so the lowest key bits (runs of 2^low adjacent x-cells) may stay unsorted: PCC_SORT_LOW_BITS
        // (measurement knob, default 0 = full order; 26-bit keys take four 8-bit radix passes, 24 bits three).
        static const int low_env = getenv("PCC_SORT_LOW_BITS") ? atoi(getenv("PCC_SORT_LOW_BITS")) : 0;
        const int low = std::max(0, std::min(low_env, bits - 8));
        size_t tmp = idx->sort_tmp_bytes;
        if (idx->sort_tmp_nq != nq || idx->sort_tmp_bits != bits) {
            cub::DeviceRadixSort::SortPairs(nullptr, tmp, idx->qkeys.as<uint32_t>(), idx->qkeys2.as<uint32_t>(), idx->qperm.as<uint32_t>(), idx->qperm2.as<uint32_t>(), (int)nq, low, bits, s);
            idx->sort_tmp_nq = nq; idx->sort_tmp_bits = bits; idx->sort_tmp_bytes = tmp;
        }
        PCC_TRY(idx->cub_tmp.reserve(tmp));
        PCC_CUDA(cub::DeviceRadixSort::SortPairs(idx->cub_tmp.p, tmp, idx->qkeys.as<uint32_t>(), idx->qkeys2.as<uint32_t>(), idx->qperm.as<uint32_t>(), idx->qperm2.as<uint32_t>(), (int)nq, low, bits, s));
        g_launches += 4;
        out->order = idx->qperm2.as<uint32_t>();
    }
    return PCC_OK;
}

int copy_out(void *dst, const void *src_dev, size_t bytes, int mem, cudaStream_t s) {
    if (!bytes || dst == src_dev) return PCC_OK;
    PCC_CUDA(cudaMemcpyAsync(dst, src_dev, bytes, mem == PCC_HOST ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice, s));
    return PCC_OK;
}

}  // namespace pcc

using namespace pcc;

extern "C" {

const char *pcc_last_error(void) { return g_error.c_str(); }
int pcc_version(void) { return 100; }
int64_t pcc_launch_count(void) { return g_launches.load(); }

int pcc_create(int device, pcc_index **out) {
    if (!out) return fail(PCC_ERR_INVALID, "out is NULL");
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) return fail(PCC_ERR_CUDA, "no usable CUDA device (%s); this library has no CPU fallback", cudaGetErrorString(e));
    if (device < 0 || device >= n) return fail(PCC_ERR_INVALID, "device %d out of range (0..%d)", device, n - 1);
    PCC_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    PCC_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) return fail(PCC_ERR_CUDA, "device %d is sm_%d%d; libpcc_search is built for sm_100a only", device, prop.major, prop.minor);
    pcc_index *idx = new pcc_index();
    idx->device = device;
    PCC_CUDA(cudaMallocHost(&idx->h_pinned, 4096));
    memset(idx->h_pinned, 0, 4096);
    PCC_CUDA(cudaEventCreate(&idx->ev0));
    PCC_CUDA(cudaEventCreate(&idx->ev1));
    *out = idx;
    return PCC_OK;
}

void pcc_destroy(pcc_index *idx) {
    if (!idx) return;
    cudaSetDevice(idx->device);
    if (idx->shadow) { pcc_index *sh = idx->shadow; idx->shadow = nullptr; pcc_destroy(sh); }
    for (int i = 0; i < 2; ++i) if (idx->pipe_stream[i]) cudaStreamDestroy(idx->pipe_stream[i]);
    Buf *bufs[] = {&idx->pts, &idx->cell_start, &idx->occ, &idx->occ2, &idx->cstart, &idx->raw, &idx->stage4, &idx->cellrank, &idx->qbuf, &idx->qkeys, &idx->qkeys2, &idx->qperm, &idx->qperm2,
                   &idx->cub_tmp, &idx->out_i, &idx->out_f, &idx->out_l, &idx->keys64, &idx->keys64b, &idx->misc, &idx->parent, &idx->inv_pos, &idx->sel_params, &idx->icp_prior, &idx->calib,
                   &idx->sift_cloud[0], &idx->sift_cloud[1], &idx->sift_val, &idx->sift_dog, &idx->sift_in, &idx->sift_nbr, &idx->sift_d2, &idx->sift_flag, &idx->sift_pos,
                   &idx->sift_row, &idx->sift_col, &idx->sift_kp, &idx->seg_label, &idx->seg_off, &idx->sift_tab, &idx->sift_lab, &idx->sift_stage,
                   &idx->rift_off, &idx->rift_keys, &idx->rift_tmp, &idx->rift_in, &idx->rift_nrm, &idx->rift_grad, &idx->rift_desc, &idx->rift_pos,
                   &idx->rift_tab, &idx->rift_out, &idx->rift_row, &idx->knnb_tab};
    for (Buf *b : bufs) b->release();
    if (idx->h_pinned) cudaFreeHost(idx->h_pinned);
    if (idx->aux_stream) cudaStreamDestroy(idx->aux_stream);
    if (idx->ev_fork) cudaEventDestroy(idx->ev_fork);
    if (idx->ev_join) cudaEventDestroy(idx->ev_join);
    if (idx->ev0) cudaEventDestroy(idx->ev0);
    if (idx->ev1) cudaEventDestroy(idx->ev1);
    delete idx;
}

int64_t pcc_size(const pcc_index *idx) { return idx ? idx->n_indexed : 0; }

int pcc_grid_info(const pcc_index *idx, double out[5]) {
    if (!idx || !idx->built) return fail(PCC_ERR_STATE, "index not built");
    out[0] = idx->gh.nx; out[1] = idx->gh.ny; out[2] = idx->gh.nz; out[3] = idx->gh.cell; out[4] = idx->gh.occupancy;
    return PCC_OK;
}

int pcc_set_timing(pcc_index *idx, int enable) { if (!idx) return fail(PCC_ERR_INVALID, "idx is NULL"); idx->timing = enable != 0; idx->last_ms = -1; return PCC_OK; }
double pcc_last_kernel_ms(const pcc_index *idx) { return idx ? idx->last_ms : -1; }

int pcc_build(pcc_index *idx, const void *pts, int64_t n, int stride_bytes, const int32_t *indices, int64_t n_idx,
              float cell_hint, int k_hint, int mem, void *stream) {
    if (!idx) return fail(PCC_ERR_INVALID, "idx is NULL");
    if (n < 0 || (n > 0 && !pts) || stride_bytes < 12 || (stride_bytes & 3)) return fail(PCC_ERR_INVALID, "bad cloud (n=%lld stride=%d)", (long long)n, stride_bytes);
    if (n >= (1ll << 31) - 1) return fail(PCC_ERR_INVALID, "n=%lld exceeds int32 indices", (long long)n);
    if (indices && (n_idx < 0 || n_idx >= (1ll << 31) - 1)) return fail(PCC_ERR_INVALID, "n_idx=%lld out of range", (long long)n_idx);
    cudaStream_t s = (cudaStream_t)stream;
    PCC_CUDA(cudaSetDevice(idx->device));
    idx->built = false;
    idx->inv_valid = false;
    idx->occ_valid = false;
    idx->icp_prior_n = -1;
    ++idx->grid_gen;
    const int64_t m = indices ? n_idx : n;
    idx->n_input = n;                 // labels / self-query rows are addressed by ORIGINAL row number
    idx->n_indexed = 0;
    idx->gh = GridHost();

    const uint8_t *raw = (const uint8_t *)pts;
    const int32_t *d_indices = indices;
    if (mem == PCC_HOST && m > 0) {
        PCC_TRY(idx->raw.reserve((size_t)n * stride_bytes));
        PCC_CUDA(cudaMemcpyAsync(idx->raw.p, pts, (size_t)n * stride_bytes, cudaMemcpyHostToDevice, s));
        raw = idx->raw.as<uint8_t>();
        if (indices) {
            PCC_TRY(idx->misc.reserve((size_t)n_idx * 4));
            PCC_CUDA(cudaMemcpyAsync(idx->misc.p, indices, (size_t)n_idx * 4, cudaMemcpyHostToDevice, s));
            d_indices = idx->misc.as<int32_t>();
        }
    }
    // 1. strided rows -> float4 staging + bbox + finite count
    int *h = (int *)idx->h_pinned;            // [0..5] bbox, [8..9] n_finite, [10..11] nonzero
    PCC_TRY(idx->stage4.reserve((size_t)std::max<int64_t>(m, 1) * sizeof(float4)));
    PCC_TRY(idx->keys64.reserve(256));
    int *d_scal = idx->keys64.as<int>();      // 6 ints bbox + 2 x u64
    {
        int init[12] = {INT_MAX, INT_MAX, INT_MAX, INT_MIN, INT_MIN, INT_MIN, 0, 0, 0, 0, 0, 0};
        memcpy(h, init, sizeof(init));
        PCC_CUDA(cudaMemcpyAsync(d_scal, h, sizeof(init), cudaMemcpyHostToDevice, s));
        PCC_CUDA(cudaStreamSynchronize(s));    // h is reused below
    }
    if (m > 0) {
        extract_kernel<<<nblocks(m, 256), 256, 0, s>>>(raw, stride_bytes, d_indices, m, n, idx->stage4.as<float4>(), d_scal, (unsigned long long *)(d_scal + 8));
        PCC_LAUNCHED();
        PCC_CUDA(cudaGetLastError());
    }
    PCC_CUDA(cudaMemcpyAsync(h, d_scal, 48, cudaMemcpyDeviceToHost, s));
    PCC_CUDA(cudaStreamSynchronize(s));
    const int64_t nfin = (int64_t)(*(unsigned long long *)(h + 8));
    idx->n_indexed = nfin;
    idx->all_rows_indexed = !indices && nfin == n;       // an `indices` list may repeat or skip rows even when the counts agree
    if (nfin == 0) {   // empty index: every query returns nothing
        PCC_TRY(idx->pts.reserve(sizeof(float4)));
        PCC_TRY(idx->cell_start.reserve(2 * sizeof(uint32_t)));
        PCC_CUDA(cudaMemsetAsync(idx->cell_start.p, 0, 2 * sizeof(uint32_t), s));
        idx->gh = GridHost();
        PCC_TRY(rebuild_occupancy(idx, s));
        idx->built = true;
        return PCC_OK;
    }
    double lo[3], ext[3];
    for (int d = 0; d < 3; ++d) { lo[d] = ord2f(h[d]); ext[d] = (double)ord2f(h[3 + d]) - lo[d]; }

    // 2. cell size: caller's hint, or iterate on the measured occupancy of non-empty cells
    int64_t max_cells = kMaxCellsDefault;
    if (const char *e = getenv("PCC_MAX_CELLS")) { long long v = atoll(e); if (v >= 1) max_cells = std::min<long long>(v, kMaxCellsDefault); }   // never above 2^28: knn_rings_kernel packs a cell index in 28 bits
    const double mx = std::max(ext[0], std::max(ext[1], ext[2]));
    double cell;
    const bool autotune = !(cell_hint > 0);
    double target = occupancy_target(k_hint);
    const bool target_fixed = occupancy_override(&target);
    if (!autotune) cell = cell_hint;
    else {
        int live = 0; double vol = 1;
        for (int d = 0; d < 3; ++d) if (ext[d] > 1e-6 * mx && ext[d] > 0) { ++live; vol *= ext[d]; }
        cell = live ? std::pow(vol * target / (double)nfin, 1.0 / live) : 1.0;
    }
    cell = clamp_cell(ext, cell, max_cells);

    PCC_TRY(idx->cellrank.reserve((size_t)m * sizeof(uint2)));
    BinParams b{};
    int dims[3]; int64_t n_cells = 0; double occ = 0;
    double prev_cell = 0, prev_occ = 0, dim_first = 2.0;
    for (int it = 0; it < 5; ++it) {
        dims_for(ext, cell, dims);
        n_cells = (int64_t)dims[0] * dims[1] * dims[2];
        const float cellf = (float)cell;
        b = BinParams{(float)lo[0], (float)lo[1], (float)lo[2], 1.0f / cellf, dims[0], dims[1], dims[2]};
        PCC_TRY(idx->cell_start.reserve((size_t)(n_cells + 1) * sizeof(uint32_t)));
        PCC_CUDA(cudaMemsetAsync(idx->cell_start.p, 0, (size_t)(n_cells + 1) * sizeof(uint32_t), s));
        PCC_CUDA(cudaMemsetAsync(d_scal + 10, 0, 24, s));
        bin_kernel<<<nblocks(m, 256), 256, 0, s>>>(idx->stage4.as<float4>(), m, b, idx->cell_start.as<uint32_t>(), idx->cellrank.as<uint2>());
        PCC_LAUNCHED();
        nonzero_kernel<<<(unsigned)std::min<int64_t>(nblocks(n_cells, 256), 148 * 16), 256, 0, s>>>(idx->cell_start.as<uint32_t>(), n_cells, (unsigned long long *)(d_scal + 10));
        PCC_LAUNCHED();
        const bool probe_fill = autotune && !target_fixed && it == 0;     // surface or volume?  decided once, on the first grid
        if (probe_fill) {
            const int64_t stride = std::max<int64_t>(1, m / kFillSamples);
            blockfill_kernel<<<nblocks((m + stride - 1) / stride, 256), 256, 0, s>>>(idx->stage4.as<float4>(), m, stride, b, idx->cell_start.as<uint32_t>(), (unsigned long long *)(d_scal + 12));
            PCC_LAUNCHED();
        }
        PCC_CUDA(cudaGetLastError());
        PCC_CUDA(cudaMemcpyAsync(h + 10, d_scal + 10, 24, cudaMemcpyDeviceToHost, s));
        PCC_CUDA(cudaStreamSynchronize(s));
        const int64_t nonempty = (int64_t)(*(unsigned long long *)(h + 10));
        occ = (double)nfin / (double)std::max<int64_t>(nonempty, 1);
        if (probe_fill) {
            const unsigned long long filled = *(unsigned long long *)(h + 12), samples = *(unsigned long long *)(h + 14);
            const double nb = samples ? (double)filled / (double)samples : 0.0;      // occupied cells of a 3x3x3 block, mean over the sample
            const double w = std::min(1.0, std::max(0.0, (nb - kFillSurface) / (kFillVolume - kFillSurface)));
            target = (1.0 - w) * target + w * occupancy_target_volume(k_hint);
            dim_first = 2.0 + w;
            idx->gh.block_fill = nb;
        }
        if (!autotune || it == 4) break;
        if (occ > 0.9 * target && occ < 1.4 * target) break;      // the cost curve is steep below the target (ring passes), shallow above it
        double dim_est = dim_first;   // first correction: 2 for a surface, 3 for a filled volume; afterwards the measured scaling exponent
        if (prev_cell > 0 && prev_occ > 0 && std::fabs(std::log(cell / prev_cell)) > 1e-3) {
            dim_est = std::log(occ / prev_occ) / std::log(cell / prev_cell);
            dim_est = std::min(3.0, std::max(1.0, dim_est));
        }
        prev_cell = cell; prev_occ = occ;
        double next = clamp_cell(ext, cell * std::pow(target / occ, 1.0 / dim_est), max_cells);
        if (std::fabs(next / cell - 1.0) < 0.02) break;   // clamped: cannot get closer
        cell = next;
    }
    idx->gh.ox = b.ox; idx->gh.oy = b.oy; idx->gh.oz = b.oz;
    idx->gh.cell = (float)cell; idx->gh.inv_cell = b.inv;
    idx->gh.nx = dims[0]; idx->gh.ny = dims[1]; idx->gh.nz = dims[2];
    idx->gh.n_cells = n_cells; idx->gh.occupancy = occ;

    // 3. cell-start scan (in place over the histogram) and scatter
    size_t tmp = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, tmp, idx->cell_start.as<uint32_t>(), idx->cell_start.as<uint32_t>(), (int)(n_cells + 1), s);
    PCC_TRY(idx->cub_tmp.reserve(tmp));
    PCC_CUDA(cub::DeviceScan::ExclusiveSum(idx->cub_tmp.p, tmp, idx->cell_start.as<uint32_t>(), idx->cell_start.as<uint32_t>(), (int)(n_cells + 1), s));
    g_launches += 2;
    PCC_TRY(idx->pts.reserve((size_t)nfin * sizeof(float4)));
    scatter_kernel<<<nblocks(m, 256), 256, 0, s>>>(idx->stage4.as<float4>(), idx->cellrank.as<uint2>(), m, idx->cell_start.as<uint32_t>(), idx->pts.as<float4>());
    PCC_LAUNCHED();
    PCC_CUDA(cudaGetLastError());
    PCC_TRY(rebuild_occupancy(idx, s));
    if (mem == PCC_HOST) PCC_CUDA(cudaStreamSynchronize(s));
    idx->built = true;
    return PCC_OK;
}

int pcc_export(const pcc_index *idx, double meta[16], void *ptrs[2]) {
    if (!idx || !idx->built) return fail(PCC_ERR_STATE, "index not built");
    meta[0] = (double)idx->n_indexed; meta[1] = (double)idx->n_input;
    meta[2] = idx->gh.nx; meta[3] = idx->gh.ny; meta[4] = idx->gh.nz;
    meta[5] = idx->gh.ox; meta[6] = idx->gh.oy; meta[7] = idx->gh.oz;
    meta[8] = idx->gh.cell; meta[9] = idx->gh.inv_cell; meta[10] = idx->gh.occupancy; meta[11] = (double)idx->gh.n_cells;
    meta[12] = idx->all_rows_indexed ? 1.0 : 0.0; meta[13] = meta[14] = meta[15] = 0;
    ptrs[0] = idx->pts.p; ptrs[1] = idx->cell_start.p;
    return PCC_OK;
}

int pcc_adopt(pcc_index *idx, const double meta[16], void *stream) {
    if (!idx) return fail(PCC_ERR_INVALID, "idx is NULL");
    (void)stream;
    PCC_CUDA(cudaSetDevice(idx->device));
    if (!(meta[0] >= 0 && meta[1] >= 0 && meta[0] < 2147483647.0 && meta[1] < 2147483647.0 && meta[2] >= 1 && meta[3] >= 1 && meta[4] >= 1 && meta[2] <= 2048 && meta[3] <= 2048 && meta[4] <= 2048 &&
          meta[11] >= 1 && meta[11] <= (double)kMaxCellsDefault && meta[11] == meta[2] * meta[3] * meta[4] && meta[8] > 0))
        return fail(PCC_ERR_INVALID, "pcc_adopt: grid description out of range (n=%g dims=%gx%gx%g cells=%g cell=%g)", meta[0], meta[2], meta[3], meta[4], meta[11], meta[8]);
    idx->n_indexed = (int64_t)meta[0]; idx->n_input = (int64_t)meta[1]; idx->all_rows_indexed = meta[12] == 1.0;
    idx->gh.nx = (int)meta[2]; idx->gh.ny = (int)meta[3]; idx->gh.nz = (int)meta[4];
    idx->gh.ox = (float)meta[5]; idx->gh.oy = (float)meta[6]; idx->gh.oz = (float)meta[7];
    idx->gh.cell = (float)meta[8]; idx->gh.inv_cell = (float)meta[9]; idx->gh.occupancy = meta[10]; idx->gh.n_cells = (int64_t)meta[11];
    PCC_TRY(idx->pts.reserve((size_t)std::max<int64_t>(idx->n_indexed, 1) * sizeof(float4)));
    PCC_TRY(idx->cell_start.reserve((size_t)(idx->gh.n_cells + 1) * sizeof(uint32_t)));
    idx->built = true;
    idx->inv_valid = false;
    idx->icp_prior_n = -1;
    ++idx->grid_gen;
    idx->occ_valid = false;       // the caller fills the arrays after this call: the bitmap is derived on the first query
    return PCC_OK;
}

}  // extern "C"
