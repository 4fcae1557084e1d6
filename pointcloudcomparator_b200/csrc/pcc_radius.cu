// pcc_radius.cu -- batched fixed-radius queries (CSR output) and the consumers built on them.
//
// Replaces (SURVEY.md section 8): a3 Search::radiusSearch batched, a4 NormalEstimation with setRadiusSearch,
// a7 EuclideanClusterExtraction (GPU union-find over the radius graph), a9 the SIFT keypoint snap loop.
#include <cub/cub.cuh>
#include <algorithm>
#include <cmath>
#include <cstring>

#include "pcc_internal.h"

namespace pcc {

// rows_query for the searching kernels: false for tail threads and for external queries that are not finite or meet an empty index.
// rows_query is called on each side of the v.self test so that each inlined copy folds to one branch (a single call that branches
// again on v.self compiles to a different block layout).
__device__ __forceinline__ bool load_query(const Grid &g, const QueryView &v, int64_t t, float &x, float &y, float &z, int64_t &row) {
    if (t >= v.nq) return false;
    if (v.self) { row = rows_query(g, v, t, x, y, z); return true; }
    row = rows_query(g, v, t, x, y, z);
    return finite3(x, y, z) && g.n > 0;
}

// visit every indexed point with d2 < r2 (strict, KdTreeFLANN::radiusSearch [up]); R0 = ceil(r / cell)
template <class F>
__device__ __forceinline__ void radius_visit(const Grid &g, float x, float y, float z, float r2, int R0, F &&f) {
    const QueryCell c = locate(g, x, y, z);
    int Rin = -1, R = R0;
    for (;;) {
        scan_shell(g, c, Rin, R, [&](uint32_t pos, float4 p) { const float d2 = dist2(x, y, z, p.x, p.y, p.z); if (d2 < r2) f(pos, p, d2); });
        if (covered_d2(g, c, R) >= r2) break;
        Rin = R; ++R;
    }
}

__global__ void __launch_bounds__(128) radius_count_kernel(Grid g, QueryView v, float r2, int R0, unsigned max_nn, int64_t *__restrict__ counts) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    float x, y, z; int64_t row;
    if (!load_query(g, v, t, x, y, z, row)) return;      // counts are pre-zeroed
    unsigned n = 0;
    radius_visit(g, x, y, z, r2, R0, [&](uint32_t, float4, float) { ++n; });
    if (max_nn && n > max_nn) n = max_nn;
    counts[row] = n;
}
// rows as packed (d2, idx) keys in visit order
__global__ void __launch_bounds__(128) radius_fill_kernel(Grid g, QueryView v, float r2, int R0, const int64_t *__restrict__ offsets, nkey_t *__restrict__ keys) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    float x, y, z; int64_t row;
    if (!load_query(g, v, t, x, y, z, row)) return;
    nkey_t *o = keys + offsets[row];
    // One 8-byte store per neighbour made this kernel store-bound (every lane writes into its own row: 32 sectors per
    // request).  Keys leave four at a time as one 32-byte aligned piece; the 0-3 keys before the row's first aligned
    // address and the 0-3 left at the end are stored singly.
    int lead = (int)((4u - (unsigned)(((uintptr_t)o >> 3) & 3u)) & 3u);
    nkey_t p0 = 0, p1 = 0, p2 = 0, p3 = 0;
    int n = 0;
    radius_visit(g, x, y, z, r2, R0, [&](uint32_t, float4 p, float d2) {
        const nkey_t key = make_key(d2, __float_as_uint(p.w));
        if (lead > 0) { *o++ = key; --lead; return; }
        const int slot = n & 3;
        if (slot == 0) p0 = key; else if (slot == 1) p1 = key; else if (slot == 2) p2 = key; else p3 = key;
        ++n;
        if (slot == 3) { reinterpret_cast<ulonglong2 *>(o)[0] = make_ulonglong2(p0, p1); reinterpret_cast<ulonglong2 *>(o)[1] = make_ulonglong2(p2, p3); o += 4; }
    });
    const int rest = n & 3;
    if (rest > 0) o[0] = p0;
    if (rest > 1) o[1] = p1;
    if (rest > 2) o[2] = p2;
}
// max_nn-capped rows: keep the max_nn smallest keys in a shared-memory heap, emit them sorted
__global__ void radius_capped_kernel(Grid g, QueryView v, float r2, int R0, int max_nn, const int64_t *__restrict__ offsets, nkey_t *__restrict__ keys) {
    extern __shared__ nkey_t smem_keys[];
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    float x, y, z; int64_t row;
    if (!load_query(g, v, t, x, y, z, row)) return;
    HeapList list; list.init(smem_keys + threadIdx.x, blockDim.x, max_nn);
    radius_visit(g, x, y, z, r2, R0, [&](uint32_t, float4 p, float d2) { list.offer(make_key(d2, __float_as_uint(p.w))); });
    list.finish();
    nkey_t *o = keys + offsets[row];
    for (int j = 0; j < list.cnt; ++j) o[j] = list.at(j);
}
// ---- per-row sort of the CSR rows by the packed (d2, idx) key ----
// cub::DeviceSegmentedSort took 475 ms for 722 M keys in 5 M rows of ~144 (its large-segment path, one block per row);
// radius rows are short, so one WARP sorts one row: <= 32 keys in registers with shuffles, <= 1024 keys with a bitonic
// network in the warp's shared-memory slice.  Longer rows are listed and sorted by the library afterwards.
// bitonic network over 32 * KPL keys held KPL per lane (element e = r * 32 + lane): partners below stride 32 through
// shuffles, above it inside the lane
template <int KPL>
__device__ __forceinline__ void warp_sort_regs(nkey_t (&v)[KPL], int lane) {
    constexpr int N = 32 * KPL;
#pragma unroll
    for (int kk = 2; kk <= N; kk <<= 1) {
#pragma unroll
        for (int j = kk >> 1; j > 0; j >>= 1) {
            if (j >= 32) {
                const int jj = j >> 5;
#pragma unroll
                for (int r = 0; r < KPL; ++r) {
                    if ((r & jj) == 0) {
                        const nkey_t a = v[r], b = v[r | jj];
                        const bool up = (((r << 5) | lane) & kk) == 0;
                        const bool sw = (b < a) == up;
                        v[r] = sw ? b : a; v[r | jj] = sw ? a : b;
                    }
                }
            } else {
#pragma unroll
                for (int r = 0; r < KPL; ++r) {
                    const nkey_t o = __shfl_xor_sync(0xffffffffu, v[r], j);
                    const bool up = (((r << 5) | lane) & kk) == 0, lower = (lane & j) == 0;
                    v[r] = ((lower == up) == (o < v[r])) ? o : v[r];
                }
            }
        }
    }
}
template <int KPL>
__device__ __forceinline__ void sort_row_in_place(nkey_t *__restrict__ k, int n, int lane) {
    nkey_t v[KPL];
#pragma unroll
    for (int r = 0; r < KPL; ++r) v[r] = (r * 32 + lane) < n ? k[r * 32 + lane] : PCC_EMPTY_KEY;
    warp_sort_regs<KPL>(v, lane);
#pragma unroll
    for (int r = 0; r < KPL; ++r) if ((r * 32 + lane) < n) k[r * 32 + lane] = v[r];
}
static constexpr int kRowSortWarps = 4, kRowSortCap = 1024;
__global__ void __launch_bounds__(kRowSortWarps * 32) sort_rows_kernel(const int64_t *__restrict__ offsets, int64_t rows, nkey_t *__restrict__ keys,
                                                                       uint32_t *__restrict__ big_rows, unsigned *__restrict__ n_big) {
    __shared__ nkey_t sm_all[kRowSortWarps][kRowSortCap];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * kRowSortWarps + warp;
    if (row >= rows) return;
    const int64_t b = offsets[row];
    const int64_t n64 = offsets[row + 1] - b;
    if (n64 <= 1) return;
    if (n64 > kRowSortCap) { if (lane == 0) big_rows[atomicAdd(n_big, 1u)] = (uint32_t)row; return; }
    const int n = (int)n64;
    nkey_t *k = keys + b;
    if (n <= 32) {                                    // one key per lane, compare-exchange through shuffles
        nkey_t v = lane < n ? k[lane] : PCC_EMPTY_KEY;
#pragma unroll
        for (int kk = 2; kk <= 32; kk <<= 1) {
#pragma unroll
            for (int j = kk >> 1; j > 0; j >>= 1) {
                const nkey_t o = __shfl_xor_sync(0xffffffffu, v, j);
                const bool up = (lane & kk) == 0, lower = (lane & j) == 0;
                const nkey_t mn = v < o ? v : o, mx = v < o ? o : v;
                v = (lower == up) ? mn : mx;
            }
        }
        if (lane < n) k[lane] = v;
        return;
    }
    // up to 256 keys: registers and shuffles, no shared memory and no barriers (measured on the selection path: 2.7 ms
    // -> 0.95 ms for 2 M rows of ~55 keys); longer rows: bitonic network in the warp's shared-memory slice
    if (n <= 64) { sort_row_in_place<2>(k, n, lane); return; }
    if (n <= 128) { sort_row_in_place<4>(k, n, lane); return; }
    if (n <= 256) { sort_row_in_place<8>(k, n, lane); return; }
    nkey_t *sm = sm_all[warp];
    int P = 64; while (P < n) P <<= 1;
    for (int i = lane; i < P; i += 32) sm[i] = i < n ? k[i] : PCC_EMPTY_KEY;
    __syncwarp();
    for (int kk = 2; kk <= P; kk <<= 1) {
        for (int j = kk >> 1; j > 0; j >>= 1) {
            for (int t = lane; t < (P >> 1); t += 32) {
                const int i = ((t & ~(j - 1)) << 1) | (t & (j - 1));
                const nkey_t a = sm[i], c = sm[i + j];
                const bool up = (i & kk) == 0;
                if ((c < a) == up) { sm[i] = c; sm[i + j] = a; }
            }
            __syncwarp();
        }
    }
    for (int i = lane; i < n; i += 32) k[i] = sm[i];
}
// ---- k nearest neighbours by SELECTION, 32 < k <= PCC_MAX_K (the reference's own k: 50, 51, 100) ----
// A per-thread heap of k 64-bit keys in shared memory (knn_heap_kernel) pays a log(k) sift of 8-byte entries per
// accepted candidate.  Here the k-th distance is bracketed first and the neighbours are then produced like a radius
// search whose radius is per query:
//   bound  -- histogram of the block's squared distances below the covered radius (64 buckets, shared memory, one
//             load-add-store per candidate); the first bucket B whose cumulative count reaches k brackets the k-th
//             distance, and that count m (>= k, a few percent above) is the row length.  Too few points below the
//             covered radius -> the block grows and the histogram is rebuilt,
//   fill   -- after a prefix sum over m: re-walk the block clipped to the ball of bucket B's upper edge and emit the
//             packed (d2, idx) keys of every point whose bucket is <= B (the same expression as in `bound`),
//   sort   -- one warp per row (sort_csr_rows), the CSR machinery of the radius search,
// and the consumer takes the first k keys of each row: exact, canonical (d2, index) order.
constexpr int kSelBuckets = 64;
struct SelParam { float scale; int bucket; int R; int pad; };
#ifndef PCC_SELB
#define PCC_SELB 6          // measured: 116 registers -> 80, k = 50 2.86 -> 2.70 ms, k = 100 5.27 -> 5.01 ms (2 M queries)
#endif
__global__ void __launch_bounds__(128, PCC_SELB) select_bound_kernel(Grid g, QueryView v, int k, int64_t *__restrict__ counts, SelParam *__restrict__ params) {
    __shared__ uint32_t hist_all[kSelBuckets * 128];
    uint32_t *hist = hist_all + threadIdx.x;
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    float x, y, z; int64_t row;
    if (!load_query(g, v, t, x, y, z, row)) return;      // counts are pre-zeroed
    const QueryCell c = locate(g, x, y, z);
    int R = 1, B = -1;
    unsigned m = 0;
    float scale = 0.f;
    for (;;) {
        const float cov = covered_d2(g, c, R);
        float hi = cov;
        if (cov == CUDART_INF_F) {          // the block holds the whole cloud: bracket by the largest distance instead
            float mx = 0.f;
            scan_shell(g, c, -1, R, [&](uint32_t, float4 p) { mx = fmaxf(mx, dist2(x, y, z, p.x, p.y, p.z)); });
            hi = fmaxf(mx * 1.0001f, 1e-30f);
            if (!(hi < CUDART_INF_F)) hi = 3.0e38f;
        }
        unsigned seen = 0;
        if (hi > 0.f) {
            scale = (float)kSelBuckets / hi;
#pragma unroll 8
            for (int b = 0; b < kSelBuckets; ++b) hist[b * 128] = 0u;
            scan_shell(g, c, -1, R, [&](uint32_t, float4 p) {
                const float fb = __fmul_rn(dist2(x, y, z, p.x, p.y, p.z), scale);
                if (fb < (float)kSelBuckets) hist[(int)fb * 128] += 1u;
            });
            for (int b = 0; b < kSelBuckets; ++b) { seen += hist[b * 128]; if (seen >= (unsigned)k) { B = b; break; } }
        }
        if (B >= 0) { m = seen; break; }
        if (cov == CUDART_INF_F) { B = kSelBuckets - 1; m = seen; break; }      // fewer than k points in the cloud: all of them
        R = seen > 0 ? R + 1 : next_ring(g, R, CUDART_INF_F);
    }
    counts[row] = (m + 3u) & ~3u;          // rows are padded with empty keys to a multiple of 4: 32-byte aligned 32-byte stores in the fill
    SelParam sp; sp.scale = scale; sp.bucket = B; sp.R = R; sp.pad = 0;
    params[row] = sp;
}
__global__ void __launch_bounds__(128) select_fill_kernel(Grid g, QueryView v, const int64_t *__restrict__ offsets, const SelParam *__restrict__ params, nkey_t *__restrict__ keys) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    float x, y, z; int64_t row;
    if (!load_query(g, v, t, x, y, z, row)) return;
    if (offsets[row + 1] == offsets[row]) return;
    const SelParam sp = params[row];
    const QueryCell c = locate(g, x, y, z);
    ulonglong2 *o = reinterpret_cast<ulonglong2 *>(keys + offsets[row]);       // offsets are multiples of 4 keys
    const float edge = (float)(sp.bucket + 1) / sp.scale;          // every selected point has d2 * scale < bucket + 1
    const float limit = (float)(sp.bucket + 1);
    // four keys are gathered in registers and leave as one aligned 32-byte piece: one key per store made this kernel
    // store-bound (9 sectors per request, 3.3 GB of L2 write traffic for 0.9 GB of keys)
    nkey_t p0 = PCC_EMPTY_KEY, p1 = PCC_EMPTY_KEY, p2 = PCC_EMPTY_KEY, p3 = PCC_EMPTY_KEY;
    int n = 0;
    scan_clipped(g, c, -1, sp.R, to_cell_units(g, edge * 1.00001f), [&](uint32_t, float4 p) {
        const float d2 = dist2(x, y, z, p.x, p.y, p.z);
        const float fb = __fmul_rn(d2, sp.scale);
        if (fb < (float)kSelBuckets && (float)(int)fb < limit) {
            const nkey_t key = make_key(d2, __float_as_uint(p.w));
            const int slot = n & 3;
            if (slot == 0) p0 = key; else if (slot == 1) p1 = key; else if (slot == 2) p2 = key; else p3 = key;
            ++n;
            if (slot == 3) { o[0] = make_ulonglong2(p0, p1); o[1] = make_ulonglong2(p2, p3); o += 2; p0 = p1 = p2 = p3 = PCC_EMPTY_KEY; }
        }
    });
    if (n & 3) { o[0] = make_ulonglong2(p0, p1); o[1] = make_ulonglong2(p2, p3); }
}
// first k keys of every row -> the dense [rows, k] result, (-1, +inf) padded
__global__ void select_unpack_kernel(const int64_t *__restrict__ offsets, const nkey_t *__restrict__ keys, int64_t rows, int k, int32_t *__restrict__ idx, float *__restrict__ d2) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows * k) return;
    const int64_t row = i / k; const int j = (int)(i - row * k);
    const int64_t b = offsets[row], e = offsets[row + 1];
    const nkey_t key = b + j < e ? keys[b + j] : PCC_EMPTY_KEY;
    idx[i] = key_idx(key); d2[i] = key_d2(key);
}
// Rows of the selection path are k plus a few keys long: sort them in REGISTERS (warp_sort_regs, 2 / 4 / 8 keys per lane)
// and write the first k straight into the dense result -- no shared memory, no barriers, no second pass over the keys.
// Rows above 256 keys (k > ~240, heavy ties) are counted and left to the generic row sort.
template <int KPL>
__device__ __forceinline__ void sort_unpack_row(const nkey_t *__restrict__ k_in, int n, int k, int lane, int32_t *__restrict__ oi, float *__restrict__ od) {
    nkey_t v[KPL];
#pragma unroll
    for (int r = 0; r < KPL; ++r) v[r] = (r * 32 + lane) < n ? k_in[r * 32 + lane] : PCC_EMPTY_KEY;
    warp_sort_regs<KPL>(v, lane);
#pragma unroll
    for (int r = 0; r < KPL; ++r) { const int e = r * 32 + lane; if (e < k) { oi[e] = key_idx(v[r]); od[e] = key_d2(v[r]); } }
}
__global__ void __launch_bounds__(128) select_sort_unpack_kernel(const int64_t *__restrict__ offsets, const nkey_t *__restrict__ keys, int64_t rows, int k,
                                                                 int32_t *__restrict__ idx, float *__restrict__ d2, unsigned *__restrict__ n_long) {
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * 4 + (threadIdx.x >> 5);
    if (row >= rows) return;
    const int64_t b = offsets[row], n64 = offsets[row + 1] - b;
    int32_t *oi = idx + row * k; float *od = d2 + row * k;
    if (n64 > 256) { if (lane == 0) atomicAdd(n_long, 1u); return; }
    const int n = (int)n64;
    if (n <= 32) {
        nkey_t v[1] = {lane < n ? keys[b + lane] : PCC_EMPTY_KEY};
        warp_sort_regs<1>(v, lane);
        for (int e = lane; e < k; e += 32) { oi[e] = e < 32 ? key_idx(v[0]) : -1; od[e] = e < 32 ? key_d2(v[0]) : CUDART_INF_F; }
    } else if (n <= 64) {
        sort_unpack_row<2>(keys + b, n, k, lane, oi, od);
        for (int e = 64 + lane; e < k; e += 32) { oi[e] = -1; od[e] = CUDART_INF_F; }
    } else if (n <= 128) {
        sort_unpack_row<4>(keys + b, n, k, lane, oi, od);
        for (int e = 128 + lane; e < k; e += 32) { oi[e] = -1; od[e] = CUDART_INF_F; }
    } else {
        sort_unpack_row<8>(keys + b, n, k, lane, oi, od);
        for (int e = 256 + lane; e < k; e += 32) { oi[e] = -1; od[e] = CUDART_INF_F; }
    }
}
__global__ void big_row_bounds_kernel(const int64_t *__restrict__ offsets, const uint32_t *__restrict__ big_rows, unsigned n_big, int64_t *__restrict__ begin, int64_t *__restrict__ end) {
    const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_big) { begin[i] = offsets[big_rows[i]]; end[i] = offsets[big_rows[i] + 1]; }
}
__global__ void big_row_copy_kernel(const int64_t *__restrict__ begin, const int64_t *__restrict__ end, const nkey_t *__restrict__ src, nkey_t *__restrict__ dst) {
    for (int64_t i = begin[blockIdx.x] + threadIdx.x; i < end[blockIdx.x]; i += blockDim.x) dst[i] = src[i];
}
__global__ void unpack_kernel(const nkey_t *__restrict__ keys, int64_t n, int32_t *__restrict__ idx, float *__restrict__ d2) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    nkey_t k = keys[i];
    idx[i] = (int32_t)(uint32_t)k; d2[i] = __uint_as_float((uint32_t)(k >> 32));
}

// NormalEstimation(radius): accumulate the (d2, idx)-sorted row in order, exactly like the kNN variant
__global__ void __launch_bounds__(128) normals_rows_kernel(Grid g, QueryView v, const int64_t *__restrict__ offsets, const nkey_t *__restrict__ keys,
                                                           const uint32_t *__restrict__ inv_pos, float vx, float vy, float vz, float4 *__restrict__ out) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= v.nq) return;
    float x, y, z;
    const int64_t row = rows_query(g, v, t, x, y, z);
    const int64_t b = offsets[row], e = offsets[row + 1];
    float a[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    for (int64_t j = b; j < e; ++j) { float4 p = __ldg(g.pts + __ldg(inv_pos + (uint32_t)keys[j])); accu_add(a, p.x, p.y, p.z); }
    out[row] = normal_from_accu(a, (int)min((int64_t)INT_MAX, e - b), x, y, z, vx, vy, vz);
}

// IntensityGradientEstimation(radius), is_dense branch: centroid and mean intensity over the sorted row, then
// A = sum (p-c)(p-c)^T (upper triangle) and b = sum (p-c)(I-mean) in row order, x = colPivHouseholderQr(A).solve(b),
// gradient = (I - n n^T) x.  Intensity is read by original index, the normal by the query's row.
__global__ void __launch_bounds__(128) gradient_rows_kernel(Grid g, QueryView v, const int64_t *__restrict__ offsets, const nkey_t *__restrict__ keys,
                                                            const uint32_t *__restrict__ inv_pos, const float *__restrict__ intensity,
                                                            const float4 *__restrict__ normals, float4 *__restrict__ out) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= v.nq) return;
    float qx, qy, qz;
    const int64_t row = rows_query(g, v, t, qx, qy, qz);
    const int64_t b = offsets[row], e = offsets[row + 1];
    const float qnan = CUDART_NAN_F;
    if (e - b < 3) { out[row] = make_float4(qnan, qnan, qnan, 0.f); return; }
    float cx = 0.f, cy = 0.f, cz = 0.f, mi = 0.f;
    for (int64_t j = b; j < e; ++j) {
        const uint32_t id = (uint32_t)keys[j];
        const float4 p = __ldg(g.pts + __ldg(inv_pos + id));
        cx += p.x; cy += p.y; cz += p.z;
        mi += __ldg(intensity + id);
    }
    const float fn = (float)(e - b);
    cx = __fdiv_rn(cx, fn); cy = __fdiv_rn(cy, fn); cz = __fdiv_rn(cz, fn); mi = __fdiv_rn(mi, fn);
    float a00 = 0.f, a01 = 0.f, a02 = 0.f, a11 = 0.f, a12 = 0.f, a22 = 0.f, b0 = 0.f, b1 = 0.f, b2 = 0.f;
    for (int64_t j = b; j < e; ++j) {
        const uint32_t id = (uint32_t)keys[j];
        const float4 p = __ldg(g.pts + __ldg(inv_pos + id));
        const float in = __ldg(intensity + id);
        if (!isfinite(in)) continue;                 // indexed points are finite; a non-finite intensity is skipped like PCL
        const float x = p.x - cx, y = p.y - cy, z = p.z - cz, w = in - mi;
        a00 += x * x; a01 += x * y; a02 += x * z;
        a11 += y * y; a12 += y * z;
        a22 += z * z;
        b0 += x * w; b1 += y * w; b2 += z * w;
    }
    float A[9] = {a00, a01, a02, a01, a11, a12, a02, a12, a22};
    const float rhs[3] = {b0, b1, b2};
    float xs[3];
    colpiv_qr_solve(A, rhs, xs);
    const float4 n = __ldg(normals + row);
    const float nn[3] = {n.x, n.y, n.z};
    float gr[3];
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        const float m0 = (r == 0 ? 1.f : 0.f) - nn[r] * nn[0];
        const float m1 = (r == 1 ? 1.f : 0.f) - nn[r] * nn[1];
        const float m2 = (r == 2 ? 1.f : 0.f) - nn[r] * nn[2];
        gr[r] = sum3(m0 * xs[0], m1 * xs[1], m2 * xs[2]);
    }
    out[row] = make_float4(gr[0], gr[1], gr[2], 0.f);
}

// Eigen 3.3's SSE squared-norm reduction (MatrixXf::normalize) over the first nb of 32 register-resident bins: packets of 4 in
// two accumulators, predux (l0 + l2) + (l1 + l3), then the scalar tail.  Loops are unrolled over all 32 slots so h stays in registers.
__device__ __forceinline__ float rift_sq_norm(const float (&h)[32], int nb) {
    if (nb < 4) {
        float s = h[0] * h[0];
#pragma unroll
        for (int i = 1; i < 3; ++i) if (i < nb) s = s + h[i] * h[i];
        return s;
    }
    const int aligned = nb & ~3, aligned2 = nb & ~7;
    float r0[4], r1[4];
#pragma unroll
    for (int l = 0; l < 4; ++l) r0[l] = h[l] * h[l];
    if (aligned > 4) {
#pragma unroll
        for (int l = 0; l < 4; ++l) r1[l] = h[4 + l] * h[4 + l];
#pragma unroll
        for (int idx = 8; idx < 32; idx += 8) {
            if (idx < aligned2) {
#pragma unroll
                for (int l = 0; l < 4; ++l) { r0[l] = r0[l] + h[idx + l] * h[idx + l]; r1[l] = r1[l] + h[idx + 4 + l] * h[idx + 4 + l]; }
            }
        }
#pragma unroll
        for (int l = 0; l < 4; ++l) r0[l] = r0[l] + r1[l];
        if (aligned > aligned2) {
#pragma unroll
            for (int idx = 0; idx < 32; idx += 8) {
                if (idx == aligned2) {
#pragma unroll
                    for (int l = 0; l < 4; ++l) r0[l] = r0[l] + h[idx + l] * h[idx + l];
                }
            }
        }
    }
    float s = (r0[0] + r0[2]) + (r0[1] + r0[3]);
#pragma unroll
    for (int i = 4; i < 32; ++i) if (i >= aligned && i < nb) s = s + h[i] * h[i];
    return s;
}

// RIFTEstimation(radius): one thread per query walks its (d2, idx)-sorted row; per neighbour the gradient magnitude and the angle
// to (p - p0), the bilinear spread over (distance, gradient) bins in PCL's loop order; the nd x ng histogram (<= 32 floats) is kept
// in registers -- bin indices are run-time values, so every add goes through an unrolled compare over the 32 slots -- then
// normalised and written in PCL's order, bin = gradient_bin * nd + distance_bin (the column-major storage of Eigen's nd x ng matrix).
__global__ void __launch_bounds__(128) rift_rows_kernel(Grid g, QueryView v, const int64_t *__restrict__ offsets, const nkey_t *__restrict__ keys,
                                                        const uint32_t *__restrict__ inv_pos, const float4 *__restrict__ gradient, float radius,
                                                        int nd, int ng, float *__restrict__ out) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= v.nq) return;
    float qx, qy, qz;
    const int64_t row = rows_query(g, v, t, qx, qy, qz);
    const int nb = nd * ng;
    float *o = out + row * nb;
    const int64_t b = offsets[row], e = offsets[row + 1];
    if (e == b) { for (int k = 0; k < nb; ++k) o[k] = CUDART_NAN_F; return; }
    float h[32];
#pragma unroll
    for (int k = 0; k < 32; ++k) h[k] = 0.f;
    const float rden = radius + 1.1920929e-07f, gden = 3.14159274f + 1.1920929e-07f;       // float(M_PI) + FLT_EPSILON
    const float fnd = (float)nd, fng = (float)ng;
    for (int64_t j = b; j < e; ++j) {
        const nkey_t key = keys[j];
        const uint32_t id = (uint32_t)key;
        const float4 p = __ldg(g.pts + __ldg(inv_pos + id));
        const float4 gv = __ldg(gradient + id);
        const float mag = sqrtf(sum3(gv.x * gv.x, gv.y * gv.y, gv.z * gv.z));
        float ux = p.x - qx, uy = p.y - qy, uz = p.z - qz;
        const float z = sum3(ux * ux, uy * uy, uz * uz);
        if (z > 0.f) { const float s = sqrtf(z); ux = __fdiv_rn(ux, s); uy = __fdiv_rn(uy, s); uz = __fdiv_rn(uz, s); }
        float ang = acosf(__fdiv_rn(sum3(gv.x * ux, gv.y * uy, gv.z * uz), mag));
        if (!isfinite(ang)) ang = 0.f;
        const float dist = __fdiv_rn(fnd * sqrtf(__uint_as_float((uint32_t)(key >> 32))), rden);
        const float grad = __fdiv_rn(fng * ang, gden);
        const int dmin = max((int)ceilf(dist - 1.f), 0), dmax = min((int)floorf(dist + 1.f), nd - 1);
        const int gmin = (int)ceilf(grad - 1.f), gmax = (int)floorf(grad + 1.f);
        for (int gi = gmin; gi <= gmax; ++gi) {
            const int gw = (gi + ng) % ng;
            const float wg = 1.0f - fabsf(grad - (float)gi);
            for (int di = dmin; di <= dmax; ++di) {
                const float w = (1.0f - fabsf(dist - (float)di)) * wg;
                const float add = w * mag;
                const int bin = gw * nd + di;
#pragma unroll
                for (int k = 0; k < 32; ++k) if (k == bin) h[k] += add;
            }
        }
    }
    const float z = rift_sq_norm(h, nb);
    if (z > 0.f) {
        const float s = sqrtf(z);
#pragma unroll
        for (int k = 0; k < 32; ++k) h[k] = __fdiv_rn(h[k], s);
    }
#pragma unroll
    for (int k = 0; k < 32; ++k) if (k < nb) o[k] = h[k];
}

// per-scale constants of SIFTKeypoint::computeScaleSpace, computed on the host with PCL's libm calls (pcc_sift_dog)
struct SiftScales { float sigma_sqr[16]; float cutoff[16]; };

// SIFTKeypoint::computeScaleSpace: one thread per point walks its (d2, idx)-sorted row once.  PCL sums each scale over the row
// prefix with d2 <= 9 sigma^2 (it breaks at the first neighbour beyond); the cutoffs grow with the scale, so a neighbour feeds a
// suffix of the scales and every (num, den) pair sees the same terms in the same order as PCL's per-scale loop.
__global__ void __launch_bounds__(128) sift_dog_rows_kernel(Grid g, QueryView v, const int64_t *__restrict__ offsets, const nkey_t *__restrict__ keys,
                                                            const float *__restrict__ values, SiftScales sc, int ns, float *__restrict__ out) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= v.nq) return;
    float qx, qy, qz;
    const int64_t row = rows_query(g, v, t, qx, qy, qz);
    const int64_t b = offsets[row], e = offsets[row + 1];
    float num[16], den[16];
#pragma unroll
    for (int s = 0; s < 16; ++s) { num[s] = 0.f; den[s] = 0.f; }
    for (int64_t j = b; j < e; ++j) {
        const nkey_t key = keys[j];
        const float d2 = __uint_as_float((uint32_t)(key >> 32));
        const float val = __ldg(values + (uint32_t)key);
#pragma unroll
        for (int s = 0; s < 16; ++s) {
            if (s < ns && d2 <= sc.cutoff[s]) {
                const float w = sift_expf(__fdiv_rn(__fmul_rn(-0.5f, d2), sc.sigma_sqr[s]));
                num[s] = __fadd_rn(num[s], __fmul_rn(val, w));
                den[s] = __fadd_rn(den[s], w);
            }
        }
    }
    float *o = out + row * (ns - 1);
    float prev = 0.f;
#pragma unroll
    for (int s = 0; s < 16; ++s) {
        if (s < ns) {
            const float resp = __fdiv_rn(num[s], den[s]);
            if (s > 0) o[s - 1] = __fsub_rn(resp, prev);
            prev = resp;
        }
    }
}

// SIFT keypoint snap: lowest original index with sqrt(double(dx)^2 + double(dy)^2 + double(dz)^2) < thr
__global__ void __launch_bounds__(128) first_within_kernel(Grid g, QueryView v, double thr, float r2_cover, int R0, int32_t *__restrict__ out) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= v.nq) return;
    const uint32_t qi = v.order ? __ldg(v.order + t) : (uint32_t)t;
    const float4 q = __ldg(v.q + qi);
    int32_t best = INT_MAX;
    if (finite3(q.x, q.y, q.z) && g.n > 0) {
        const QueryCell c = locate(g, q.x, q.y, q.z);
        int Rin = -1, R = R0;
        for (;;) {
            scan_shell(g, c, Rin, R, [&](uint32_t, float4 p) {
                const double dx = (double)(q.x - p.x), dy = (double)(q.y - p.y), dz = (double)(q.z - p.z);
                if (sqrt(dx * dx + dy * dy + dz * dz) < thr) best = min(best, __float_as_int(p.w));
            });
            if (covered_d2(g, c, R) >= r2_cover) break;
            Rin = R; ++R;
        }
    }
    out[qi] = best == INT_MAX ? -1 : best;
}

// ---- EuclideanClusterExtraction: lock-free union-find over sorted positions ----
// Loads bypass L1 (__ldcg) so a root that another SM has just hooked is seen in L2; a stale value is still
// an ancestor in the same set, so following it is safe, and the CAS below is the only way a root changes.
__device__ __forceinline__ uint32_t uf_find(uint32_t *parent, uint32_t x) {
    uint32_t p = __ldcg(parent + x);
    while (p != x) { uint32_t gp = __ldcg(parent + p); if (gp != p) parent[x] = gp; x = p; p = gp; }   // path halving
    return x;
}
__device__ __forceinline__ void uf_union(uint32_t *parent, uint32_t a, uint32_t b) {
    for (;;) {
        a = uf_find(parent, a); b = uf_find(parent, b);
        if (a == b) return;
        if (a < b) { uint32_t t = a; a = b; b = t; }      // hook the larger root under the smaller
        const uint32_t old = atomicCAS(parent + a, a, b);
        if (old == a) return;
        a = old;                                            // lost the race: continue from the true parent
    }
}
__global__ void iota_kernel(uint32_t *p, int64_t n) { int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; if (i < n) p[i] = (uint32_t)i; }
__global__ void __launch_bounds__(128) ece_link_kernel(Grid g, float r2, int R0, uint32_t *__restrict__ parent) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= g.n) return;
    const float4 q = __ldg(g.pts + t);
    // `ra` is an ancestor of t (its root when last looked up).  Most neighbours already hang directly under it after the
    // first few unions, so one load of parent[pos] settles them without the two root walks of a full union.
    uint32_t ra = uf_find(parent, (uint32_t)t);
    radius_visit(g, q.x, q.y, q.z, r2, R0, [&](uint32_t pos, float4, float) {
        if (pos >= (uint32_t)t) return;
        if (pos == ra || __ldcg(parent + pos) == ra) return;
        uf_union(parent, ra, pos);
        ra = uf_find(parent, ra);
    });
}
// sharded clustering: link only the edges whose query endpoint lies in [begin, end) of the sorted order
__global__ void __launch_bounds__(128) ece_link_range_kernel(Grid g, float r2, int R0, uint32_t begin, uint32_t end, uint32_t *__restrict__ parent) {
    const int64_t t = (int64_t)begin + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= end) return;
    const float4 q = __ldg(g.pts + t);
    uint32_t ra = uf_find(parent, (uint32_t)t);
    radius_visit(g, q.x, q.y, q.z, r2, R0, [&](uint32_t pos, float4, float) {
        if (pos == (uint32_t)t || pos == ra || __ldcg(parent + pos) == ra) return;
        uf_union(parent, ra, pos);
        ra = uf_find(parent, ra);
    });
}
// merge another rank's knowledge: node i and other[i] are in the same component
__global__ void ece_absorb_kernel(uint32_t n, const uint32_t *__restrict__ other, uint32_t *__restrict__ parent) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    const uint32_t o = other[t];
    if (o != (uint32_t)t && o < n) uf_union(parent, (uint32_t)t, o);
}
__global__ void ece_compress_kernel(uint32_t n, uint32_t *__restrict__ parent) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n) parent[t] = uf_find(parent, (uint32_t)t);
}
__global__ void ece_flatten_kernel(Grid g, uint32_t *__restrict__ parent, uint32_t *__restrict__ size, uint32_t *__restrict__ min_orig) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= g.n) return;
    const uint32_t r = uf_find(parent, (uint32_t)t);
    parent[t] = r;      // safe: r is a root, roots never change in this kernel
    atomicAdd(size + r, 1u);
    atomicMin(min_orig + r, (uint32_t)__float_as_int(__ldg(g.pts + t).w));
}
// kept roots -> (sort key, root) list; key orders by size descending then smallest member index
__global__ void ece_select_kernel(uint32_t n, const uint32_t *__restrict__ parent, const uint32_t *__restrict__ size, const uint32_t *__restrict__ min_orig,
                                  uint32_t min_size, uint32_t max_size, nkey_t *__restrict__ keys, uint32_t *__restrict__ roots, unsigned long long *__restrict__ n_kept) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n || parent[t] != (uint32_t)t) return;
    const uint32_t s = size[t];
    if (s < min_size || s > max_size) return;
    const unsigned long long slot = atomicAdd(n_kept, 1ull);
    keys[slot] = ((nkey_t)(0xFFFFFFFFu - s) << 32) | min_orig[t];
    roots[slot] = (uint32_t)t;
}
__global__ void ece_rank_kernel(const nkey_t *__restrict__ keys_sorted, const uint32_t *__restrict__ roots_sorted, int64_t n_kept, uint32_t *__restrict__ rank_of_root, int64_t *__restrict__ sizes, int64_t sizes_cap) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_kept) return;
    rank_of_root[roots_sorted[i]] = (uint32_t)i;
    if (sizes && i < sizes_cap) sizes[i] = (int64_t)(0xFFFFFFFFu - (uint32_t)(keys_sorted[i] >> 32));
}
__global__ void ece_label_kernel(Grid g, const uint32_t *__restrict__ parent, const uint32_t *__restrict__ rank_of_root, int32_t *__restrict__ labels) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= g.n) return;
    labels[__float_as_int(__ldg(g.pts + t).w)] = (int32_t)rank_of_root[parent[t]];
}
__global__ void fill_u32_kernel(uint32_t *p, int64_t n, uint32_t v) { int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; if (i < n) p[i] = v; }
__global__ void fill_f4_kernel(float4 *p, int64_t n, float4 v) { int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; if (i < n) p[i] = v; }

static inline int ring0(const pcc_index *idx, double radius) { return std::max(1, (int)std::ceil(radius / (double)idx->gh.cell)); }

// shared by pcc_radius_count and the internal consumers: counts (device, zeroed, rows+1) -> inclusive CSR offsets
static int radius_offsets(pcc_index *idx, const Queries &qs, double radius, unsigned max_nn, int64_t *d_offsets, cudaStream_t s) {
    const float r2 = (float)(radius * radius);
    PCC_CUDA(cudaMemsetAsync(d_offsets, 0, (size_t)(qs.rows + 1) * sizeof(int64_t), s));
    if (qs.nq > 0) {
        radius_count_kernel<<<nblocks(qs.nq, 128), 128, 0, s>>>(idx->grid(), view_of(qs), r2, ring0(idx, radius), max_nn, d_offsets);
        PCC_LAUNCHED();
        PCC_CUDA(cudaGetLastError());
    }
    size_t tmp = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, tmp, d_offsets, d_offsets, (int)(qs.rows + 1), s);
    PCC_TRY(idx->cub_tmp.reserve(tmp));
    PCC_CUDA(cub::DeviceScan::ExclusiveSum(idx->cub_tmp.p, tmp, d_offsets, d_offsets, (int)(qs.rows + 1), s));
    g_launches += 2;
    return PCC_OK;
}
// every CSR row sorted by its packed (d2, idx) key: one warp per row, rows above 1024 keys by the library afterwards
static int sort_csr_rows(pcc_index *idx, int64_t rows, const int64_t *d_offsets, int64_t total, nkey_t *keys, cudaStream_t s) {
    Queries qs; qs.rows = rows;
    {
        PCC_TRY(idx->misc.reserve((size_t)qs.rows * 4 + 64));
        unsigned *n_big = idx->misc.as<unsigned>();
        uint32_t *big_rows = idx->misc.as<uint32_t>() + 16;
        PCC_CUDA(cudaMemsetAsync(n_big, 0, 4, s));
        sort_rows_kernel<<<nblocks(qs.rows, kRowSortWarps), kRowSortWarps * 32, 0, s>>>(d_offsets, qs.rows, keys, big_rows, n_big);
        PCC_LAUNCHED();
        PCC_CUDA(cudaGetLastError());
        unsigned *h = (unsigned *)idx->h_pinned;
        PCC_CUDA(cudaMemcpyAsync(h, n_big, 4, cudaMemcpyDeviceToHost, s));
        PCC_CUDA(cudaStreamSynchronize(s));
        const unsigned nb = h[0];
        if (nb > 0) {       // rows longer than 1024 neighbours: library segmented sort over just those rows
            if (total >= (1ll << 31)) return fail(PCC_ERR_INVALID, "radius result of %lld neighbours exceeds the segmented-sort limit", (long long)total);
            PCC_TRY(idx->keys64b.reserve((size_t)total * sizeof(nkey_t)));
            PCC_TRY(idx->parent.reserve((size_t)nb * 16));
            int64_t *bb = idx->parent.as<int64_t>(), *be = bb + nb;
            big_row_bounds_kernel<<<nblocks(nb, 256), 256, 0, s>>>(d_offsets, big_rows, nb, bb, be); PCC_LAUNCHED();
            size_t tmp = 0;
            cub::DeviceSegmentedSort::SortKeys(nullptr, tmp, keys, idx->keys64b.as<nkey_t>(), (int)total, (int)nb, bb, be, s);
            PCC_TRY(idx->cub_tmp.reserve(tmp));
            PCC_CUDA(cub::DeviceSegmentedSort::SortKeys(idx->cub_tmp.p, tmp, keys, idx->keys64b.as<nkey_t>(), (int)total, (int)nb, bb, be, s));
            g_launches += 3;
            big_row_copy_kernel<<<nb, 256, 0, s>>>(bb, be, idx->keys64b.as<nkey_t>(), keys); PCC_LAUNCHED();
            PCC_CUDA(cudaGetLastError());
        }
    }
    return PCC_OK;
}
// rows as packed keys into idx->keys64 (sorted in place when requested); total = offsets[rows]
static int radius_rows(pcc_index *idx, const Queries &qs, double radius, unsigned max_nn, int sorted, const int64_t *d_offsets, int64_t total, nkey_t **keys_out, cudaStream_t s) {
    const float r2 = (float)(radius * radius);
    PCC_TRY(idx->keys64.reserve((size_t)std::max<int64_t>(total, 1) * sizeof(nkey_t)));
    nkey_t *keys = idx->keys64.as<nkey_t>();
    *keys_out = keys;
    if (qs.nq == 0 || total == 0) return PCC_OK;
    const bool capped = max_nn != 0 && (int64_t)max_nn < idx->n_indexed;
    if (capped) {
        if (max_nn > PCC_MAX_K) return fail(PCC_ERR_INVALID, "max_nn=%u above %d is only supported when it is >= the indexed point count", max_nn, PCC_MAX_K);
        const int th = heap_threads((int)max_nn);
        PCC_TRY(set_heap_smem(radius_capped_kernel));
        radius_capped_kernel<<<nblocks(qs.nq, th), th, (size_t)max_nn * th * sizeof(nkey_t), s>>>(idx->grid(), view_of(qs), r2, ring0(idx, radius), (int)max_nn, d_offsets, keys);
        PCC_LAUNCHED();
        PCC_CUDA(cudaGetLastError());
        return PCC_OK;   // already sorted
    }
    radius_fill_kernel<<<nblocks(qs.nq, 128), 128, 0, s>>>(idx->grid(), view_of(qs), r2, ring0(idx, radius), d_offsets, keys);
    PCC_LAUNCHED();
    PCC_CUDA(cudaGetLastError());
    if (sorted) PCC_TRY(sort_csr_rows(idx, qs.rows, d_offsets, total, keys, s));
    return PCC_OK;
}

// sorted neighbour rows for k > 32: d_offsets (rows + 1, device) and keys (idx->keys64); every row holds >= min(k, cloud) keys
int knn_select_rows(pcc_index *idx, const Queries &qs, int k, int64_t *d_offsets, nkey_t **keys_out, int64_t *total_out, bool sort_rows, cudaStream_t s) {
    PCC_TRY(idx->sel_params.reserve((size_t)std::max<int64_t>(qs.rows, 1) * sizeof(SelParam)));
    SelParam *params = idx->sel_params.as<SelParam>();
    PCC_CUDA(cudaMemsetAsync(d_offsets, 0, (size_t)(qs.rows + 1) * sizeof(int64_t), s));
    if (qs.nq > 0) {
        select_bound_kernel<<<nblocks(qs.nq, 128), 128, 0, s>>>(idx->grid(), view_of(qs), k, d_offsets, params);
        PCC_LAUNCHED();
        PCC_CUDA(cudaGetLastError());
    }
    size_t tmp = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, tmp, d_offsets, d_offsets, (int)(qs.rows + 1), s);
    PCC_TRY(idx->cub_tmp.reserve(tmp));
    PCC_CUDA(cub::DeviceScan::ExclusiveSum(idx->cub_tmp.p, tmp, d_offsets, d_offsets, (int)(qs.rows + 1), s));
    g_launches += 2;
    int64_t *h = (int64_t *)idx->h_pinned;
    PCC_CUDA(cudaMemcpyAsync(h, d_offsets + qs.rows, 8, cudaMemcpyDeviceToHost, s));
    PCC_CUDA(cudaStreamSynchronize(s));
    const int64_t total = h[0];
    *total_out = total;
    PCC_TRY(idx->keys64.reserve((size_t)std::max<int64_t>(total, 1) * sizeof(nkey_t)));
    nkey_t *keys = idx->keys64.as<nkey_t>();
    *keys_out = keys;
    if (qs.nq == 0 || total == 0) return PCC_OK;
    select_fill_kernel<<<nblocks(qs.nq, 128), 128, 0, s>>>(idx->grid(), view_of(qs), d_offsets, params, keys);
    PCC_LAUNCHED();
    PCC_CUDA(cudaGetLastError());
    return sort_rows ? sort_csr_rows(idx, qs.rows, d_offsets, total, keys, s) : PCC_OK;
}
// pcc_knn for k > 32
int knn_select(pcc_index *idx, const Queries &qs, int k, int32_t *oi, float *od, cudaStream_t s) {
    PCC_TRY(idx->out_l.reserve((size_t)(qs.rows + 1) * 8));
    int64_t *d_off = idx->out_l.as<int64_t>();
    nkey_t *keys = nullptr; int64_t total = 0;
    PCC_TRY(knn_select_rows(idx, qs, k, d_off, &keys, &total, false, s));
    if (qs.rows == 0) return PCC_OK;
    PCC_TRY(idx->misc.reserve(256));
    unsigned *n_long = idx->misc.as<unsigned>();
    PCC_CUDA(cudaMemsetAsync(n_long, 0, 4, s));
    select_sort_unpack_kernel<<<nblocks(qs.rows, 4), 128, 0, s>>>(d_off, keys, qs.rows, k, oi, od, n_long);
    PCC_LAUNCHED();
    PCC_CUDA(cudaGetLastError());
    unsigned *h = (unsigned *)idx->h_pinned;
    PCC_CUDA(cudaMemcpyAsync(h, n_long, 4, cudaMemcpyDeviceToHost, s));
    PCC_CUDA(cudaStreamSynchronize(s));
    if (h[0] > 0) {         // rows above 256 keys (large k, or many points tied inside the bracketing bucket): generic row sort, then unpack everything
        PCC_TRY(sort_csr_rows(idx, qs.rows, d_off, total, keys, s));
        select_unpack_kernel<<<nblocks(qs.rows * (int64_t)k, 256), 256, 0, s>>>(d_off, keys, qs.rows, k, oi, od);
        PCC_LAUNCHED();
        PCC_CUDA(cudaGetLastError());
    }
    return PCC_OK;
}

}  // namespace pcc

using namespace pcc;

// The sorted-radius-row consumers (normals, intensity gradient, RIFT, SIFT DoG) after their own checks and input staging: the
// batch's radius rows sorted by (d2, index) (offsets in idx->out_l, keys in idx->keys64), the output (the caller's pointer, or out_f
// for PCC_HOST) with the rows of unindexed points pre-filled -- 0xFF bytes (NaN), or (NaN, NaN, NaN, 0) for the gradient -- and
// launch(offsets, keys, out) when there are queries.  Host inputs are staged in stage4 (free after pcc_build) and sel_params (only
// used inside the k > 32 kNN selection); the rows touch neither.  A PCC_HOST call returns with its results on the host.
template <class Launch>
static int sorted_rows_consumer(pcc_index *idx, const Queries &qs, double radius, void *out, size_t row_bytes, bool fill_nan_w0, int mem, cudaStream_t s,
                                Launch &&launch) {
    KernelTimer timer(idx, s);
    if (!idx->inv_valid) PCC_TRY(rebuild_inverse(idx, s));
    PCC_TRY(idx->out_l.reserve((size_t)(qs.rows + 1) * 8));
    int64_t *d_off = idx->out_l.as<int64_t>();
    PCC_TRY(radius_offsets(idx, qs, radius, 0, d_off, s));
    int64_t *h = (int64_t *)idx->h_pinned;
    PCC_CUDA(cudaMemcpyAsync(h, d_off + qs.rows, 8, cudaMemcpyDeviceToHost, s));
    PCC_CUDA(cudaStreamSynchronize(s));
    nkey_t *keys = nullptr;
    PCC_TRY(radius_rows(idx, qs, radius, 0, 1, d_off, h[0], &keys, s));
    const size_t bytes = (size_t)qs.rows * row_bytes;
    void *od = nullptr;
    PCC_TRY(output_rows(idx, out, bytes, mem, &od));
    if (qs.self && !idx->all_rows_indexed) {
        if (fill_nan_w0) { fill_f4_kernel<<<nblocks(qs.rows, 256), 256, 0, s>>>((float4 *)od, qs.rows, make_float4(NAN, NAN, NAN, 0.f)); PCC_LAUNCHED(); }
        else PCC_CUDA(cudaMemsetAsync(od, 0xFF, bytes, s));
    }
    if (qs.nq > 0) {
        launch(d_off, keys, od);
        PCC_LAUNCHED();
        PCC_CUDA(cudaGetLastError());
    }
    timer.stop();
    return deliver_rows(out, od, bytes, mem, s);
}

extern "C" {

int pcc_radius_count(pcc_index *idx, const void *q, int64_t nq, int stride_bytes, double radius, unsigned max_nn, int64_t *offsets, int64_t *total, int mem, void *stream) {
    PCC_TRY(check_index(idx, stream));
    if (!(radius >= 0) || !offsets) return fail(PCC_ERR_INVALID, "bad radius / offsets");
    cudaStream_t s = (cudaStream_t)stream;
    Queries qs;
    PCC_TRY(prepare_queries(idx, q, nq, stride_bytes, mem, s, &qs));
    int64_t *d_off = offsets;
    if (mem == PCC_HOST) { PCC_TRY(idx->out_l.reserve((size_t)(qs.rows + 1) * 8)); d_off = idx->out_l.as<int64_t>(); }
    KernelTimer timer(idx, s);
    PCC_TRY(radius_offsets(idx, qs, radius, max_nn, d_off, s));
    timer.stop();
    int64_t *h = (int64_t *)idx->h_pinned;
    PCC_CUDA(cudaMemcpyAsync(h, d_off + qs.rows, 8, cudaMemcpyDeviceToHost, s));
    if (mem == PCC_HOST) PCC_TRY(copy_out(offsets, d_off, (size_t)(qs.rows + 1) * 8, mem, s));
    PCC_CUDA(cudaStreamSynchronize(s));
    if (total) *total = h[0];
    return PCC_OK;
}

int pcc_radius_fill(pcc_index *idx, const void *q, int64_t nq, int stride_bytes, double radius, unsigned max_nn, int sorted, const int64_t *offsets,
                    int32_t *out_idx, float *out_d2, int mem, void *stream) {
    PCC_TRY(check_index(idx, stream));
    if (!(radius >= 0) || !offsets) return fail(PCC_ERR_INVALID, "bad radius / offsets");
    cudaStream_t s = (cudaStream_t)stream;
    Queries qs;
    PCC_TRY(prepare_queries(idx, q, nq, stride_bytes, mem, s, &qs));
    const int64_t *d_off = offsets;
    int64_t total = 0;
    if (mem == PCC_HOST) {
        PCC_TRY(idx->out_l.reserve((size_t)(qs.rows + 1) * 8));
        PCC_CUDA(cudaMemcpyAsync(idx->out_l.p, offsets, (size_t)(qs.rows + 1) * 8, cudaMemcpyHostToDevice, s));
        d_off = idx->out_l.as<int64_t>();
        total = offsets[qs.rows];
    } else {
        int64_t *h = (int64_t *)idx->h_pinned;
        PCC_CUDA(cudaMemcpyAsync(h, offsets + qs.rows, 8, cudaMemcpyDeviceToHost, s));
        PCC_CUDA(cudaStreamSynchronize(s));
        total = h[0];
    }
    if (total == 0) return PCC_OK;
    if (!out_idx || !out_d2) return fail(PCC_ERR_INVALID, "output pointers are NULL");
    nkey_t *keys = nullptr;
    KernelTimer timer(idx, s);
    PCC_TRY(radius_rows(idx, qs, radius, max_nn, sorted, d_off, total, &keys, s));
    int32_t *oi = out_idx; float *od = out_d2;
    if (mem == PCC_HOST) { PCC_TRY(idx->out_i.reserve((size_t)total * 4)); PCC_TRY(idx->out_f.reserve((size_t)total * 4)); oi = idx->out_i.as<int32_t>(); od = idx->out_f.as<float>(); }
    unpack_kernel<<<nblocks(total, 256), 256, 0, s>>>(keys, total, oi, od);
    PCC_LAUNCHED();
    PCC_CUDA(cudaGetLastError());
    timer.stop();
    if (mem == PCC_HOST) {
        PCC_TRY(copy_out(out_idx, oi, (size_t)total * 4, mem, s));
        PCC_TRY(copy_out(out_d2, od, (size_t)total * 4, mem, s));
        PCC_CUDA(cudaStreamSynchronize(s));
    }
    return PCC_OK;
}

int pcc_normals_radius(pcc_index *idx, const void *q, int64_t nq, int stride_bytes, double radius, const float viewpoint[3], float *out, int mem, void *stream) {
    PCC_TRY(check_index(idx, stream));
    if (!(radius >= 0)) return fail(PCC_ERR_INVALID, "bad radius");
    cudaStream_t s = (cudaStream_t)stream;
    Queries qs;
    PCC_TRY(prepare_queries(idx, q, nq, stride_bytes, mem, s, &qs));
    if (qs.rows == 0) return PCC_OK;
    if (!out) return fail(PCC_ERR_INVALID, "output pointer is NULL");
    const float vx = viewpoint ? viewpoint[0] : 0.f, vy = viewpoint ? viewpoint[1] : 0.f, vz = viewpoint ? viewpoint[2] : 0.f;
    return sorted_rows_consumer(idx, qs, radius, out, 16, false, mem, s, [&](const int64_t *d_off, const nkey_t *keys, void *od) {
        normals_rows_kernel<<<nblocks(qs.nq, 128), 128, 0, s>>>(idx->grid(), view_of(qs), d_off, keys, idx->inv_pos.as<uint32_t>(), vx, vy, vz, (float4 *)od);
    });
}

int pcc_intensity_gradient(pcc_index *idx, const void *q, int64_t nq, int stride_bytes, double radius, const float *intensity, const float *normals4,
                           float *out, int mem, void *stream) {
    PCC_TRY(check_index(idx, stream));
    if (!(radius >= 0)) return fail(PCC_ERR_INVALID, "bad radius");
    cudaStream_t s = (cudaStream_t)stream;
    Queries qs;
    PCC_TRY(prepare_queries(idx, q, nq, stride_bytes, mem, s, &qs));
    if (qs.rows == 0) return PCC_OK;
    if (!out || !intensity || !normals4) return fail(PCC_ERR_INVALID, "intensity / normals / output pointer is NULL");
    const float *d_int = nullptr, *d_nrm = nullptr;
    PCC_TRY(stage_in(idx->stage4, intensity, (size_t)idx->n_input * 4, mem, s, &d_int));
    PCC_TRY(stage_in(idx->sel_params, normals4, (size_t)qs.rows * 16, mem, s, &d_nrm));
    return sorted_rows_consumer(idx, qs, radius, out, 16, true, mem, s, [&](const int64_t *d_off, const nkey_t *keys, void *od) {
        gradient_rows_kernel<<<nblocks(qs.nq, 128), 128, 0, s>>>(idx->grid(), view_of(qs), d_off, keys, idx->inv_pos.as<uint32_t>(), d_int, (const float4 *)d_nrm,
                                                                 (float4 *)od);
    });
}

int pcc_rift(pcc_index *idx, const void *q, int64_t nq, int stride_bytes, double radius, const float *gradient4, int n_distance_bins, int n_gradient_bins,
             float *out, int mem, void *stream) {
    PCC_TRY(check_index(idx, stream));
    if (!(radius >= 0)) return fail(PCC_ERR_INVALID, "bad radius");
    if (n_distance_bins < 1 || n_gradient_bins < 1 || n_distance_bins * n_gradient_bins > 32)
        return fail(PCC_ERR_INVALID, "RIFT bins %d x %d: the histogram holds 1..32 bins (pcl::Histogram<32>)", n_distance_bins, n_gradient_bins);
    cudaStream_t s = (cudaStream_t)stream;
    Queries qs;
    PCC_TRY(prepare_queries(idx, q, nq, stride_bytes, mem, s, &qs));
    if (qs.rows == 0) return PCC_OK;
    if (!out || !gradient4) return fail(PCC_ERR_INVALID, "gradient / output pointer is NULL");
    const float *d_grad = nullptr;
    PCC_TRY(stage_in(idx->stage4, gradient4, (size_t)idx->n_input * 16, mem, s, &d_grad));
    return sorted_rows_consumer(idx, qs, radius, out, (size_t)n_distance_bins * n_gradient_bins * 4, false, mem, s, [&](const int64_t *d_off, const nkey_t *keys, void *od) {
        rift_rows_kernel<<<nblocks(qs.nq, 128), 128, 0, s>>>(idx->grid(), view_of(qs), d_off, keys, idx->inv_pos.as<uint32_t>(), (const float4 *)d_grad,
                                                             (float)radius, n_distance_bins, n_gradient_bins, (float *)od);
    });
}

int pcc_sift_dog(pcc_index *idx, const float *values, const float *scales, int n_scales, float *out, int mem, void *stream) {
    PCC_TRY(check_index(idx, stream));
    if (!scales || n_scales < 2 || n_scales > 16) return fail(PCC_ERR_INVALID, "SIFT scale space of %d scales: 2..16 are supported", n_scales);
    SiftScales sc{};
    for (int i = 0; i < n_scales; ++i) {
        if (!(scales[i] > 0.f) || !std::isfinite(scales[i]) || (i > 0 && !(scales[i] >= scales[i - 1])))
            return fail(PCC_ERR_INVALID, "SIFT scales must be positive, finite and ascending (scale %d = %g)", i, (double)scales[i]);
        sc.sigma_sqr[i] = powf(scales[i], 2.0f);                 // computeScaleSpace: sigma_sqr = powf (scales[i_scale], 2.0f)
        sc.cutoff[i] = 9 * sc.sigma_sqr[i];                      // if (dist_sqr <= 9*sigma_sqr)
    }
    const double radius = (double)(3.0f * scales[n_scales - 1]);      // max_radius = 3.0f * scales.back (), a float handed to radiusSearch
    cudaStream_t s = (cudaStream_t)stream;
    Queries qs;
    PCC_TRY(prepare_queries(idx, nullptr, 0, 16, mem, s, &qs));
    if (qs.rows == 0) return PCC_OK;
    if (!out || !values) return fail(PCC_ERR_INVALID, "values / output pointer is NULL");
    const float *d_val = nullptr;
    PCC_TRY(stage_in(idx->stage4, values, (size_t)idx->n_input * 4, mem, s, &d_val));
    return sorted_rows_consumer(idx, qs, radius, out, (size_t)(n_scales - 1) * 4, false, mem, s, [&](const int64_t *d_off, const nkey_t *keys, void *od) {
        sift_dog_rows_kernel<<<nblocks(qs.nq, 128), 128, 0, s>>>(idx->grid(), view_of(qs), d_off, keys, d_val, sc, n_scales, (float *)od);
    });
}

int pcc_first_within(pcc_index *idx, const void *q, int64_t nq, int stride_bytes, double thr, int32_t *out, int mem, void *stream) {
    PCC_TRY(check_index(idx, stream));
    if (!(thr >= 0) || !q) return fail(PCC_ERR_INVALID, "bad threshold / queries");
    cudaStream_t s = (cudaStream_t)stream;
    Queries qs;
    PCC_TRY(prepare_queries(idx, q, nq, stride_bytes, mem, s, &qs));
    if (qs.rows == 0) return PCC_OK;
    int32_t *oi = out;
    if (mem == PCC_HOST) { PCC_TRY(idx->out_i.reserve((size_t)nq * 4)); oi = idx->out_i.as<int32_t>(); }
    const float r2_cover = (float)(thr * thr * (1.0 + 1e-5));
    first_within_kernel<<<nblocks(nq, 128), 128, 0, s>>>(idx->grid(), view_of(qs), thr, r2_cover, ring0(idx, thr), oi);
    PCC_LAUNCHED();
    PCC_CUDA(cudaGetLastError());
    if (mem == PCC_HOST) { PCC_TRY(copy_out(out, oi, (size_t)nq * 4, mem, s)); PCC_CUDA(cudaStreamSynchronize(s)); }
    return PCC_OK;
}

// sizes, PCL ordering and labels from a parent forest over sorted positions (any forest whose trees are the components)
static int ece_finish(pcc_index *idx, uint32_t *parent, int64_t min_size, int64_t max_size, int32_t *labels, int64_t *n_clusters, int64_t *sizes,
                      int64_t sizes_cap, int mem, cudaStream_t s) {
    const int64_t n = idx->n_indexed, rows = idx->n_input;
    int32_t *d_labels = labels;
    if (mem == PCC_HOST) { PCC_TRY(idx->out_i.reserve((size_t)rows * 4)); d_labels = idx->out_i.as<int32_t>(); }
    PCC_CUDA(cudaMemsetAsync(d_labels, 0xFF, (size_t)rows * 4, s));
    int64_t kept = 0;
    int64_t *d_sizes = sizes;
    if (n > 0) {
        const Grid g = idx->grid();
        // size | min_orig | rank_of_root | roots | roots_sorted : 5 x uint32[n]; keys | keys_sorted : 2 x u64[n]
        PCC_TRY(idx->misc.reserve((size_t)n * 4 * 5));
        PCC_TRY(idx->keys64.reserve((size_t)n * 8 + 64)); PCC_TRY(idx->keys64b.reserve((size_t)n * 8));
        uint32_t *size = idx->misc.as<uint32_t>(), *min_orig = size + n, *rank_of_root = min_orig + n, *roots = rank_of_root + n, *roots_sorted = roots + n;
        nkey_t *keys = idx->keys64.as<nkey_t>(), *keys_sorted = idx->keys64b.as<nkey_t>();
        unsigned long long *d_kept = (unsigned long long *)(keys + n);
        const unsigned nb256 = nblocks(n, 256);
        PCC_CUDA(cudaMemsetAsync(size, 0, (size_t)n * 4, s));
        PCC_CUDA(cudaMemsetAsync(min_orig, 0xFF, (size_t)n * 4, s));
        PCC_CUDA(cudaMemsetAsync(rank_of_root, 0xFF, (size_t)n * 4, s));
        PCC_CUDA(cudaMemsetAsync(d_kept, 0, 8, s));
        ece_flatten_kernel<<<nb256, 256, 0, s>>>(g, parent, size, min_orig); PCC_LAUNCHED();
        const uint32_t mn = (uint32_t)std::min<int64_t>(std::max<int64_t>(min_size, 0), 0xFFFFFFFFll), mxs = (uint32_t)std::min<int64_t>(std::max<int64_t>(max_size, 0), 0xFFFFFFFFll);
        ece_select_kernel<<<nb256, 256, 0, s>>>((uint32_t)n, parent, size, min_orig, mn, mxs, keys, roots, d_kept); PCC_LAUNCHED();
        PCC_CUDA(cudaGetLastError());
        unsigned long long *h = (unsigned long long *)idx->h_pinned;
        PCC_CUDA(cudaMemcpyAsync(h, d_kept, 8, cudaMemcpyDeviceToHost, s));
        PCC_CUDA(cudaStreamSynchronize(s));
        kept = (int64_t)h[0];
        if (kept > 0) {
            size_t tmp = 0;
            cub::DeviceRadixSort::SortPairs(nullptr, tmp, keys, keys_sorted, roots, roots_sorted, (int)kept, 0, 64, s);
            PCC_TRY(idx->cub_tmp.reserve(tmp));
            PCC_CUDA(cub::DeviceRadixSort::SortPairs(idx->cub_tmp.p, tmp, keys, keys_sorted, roots, roots_sorted, (int)kept, 0, 64, s));
            g_launches += 8;
            if (sizes && mem == PCC_HOST) { PCC_TRY(idx->out_l.reserve((size_t)std::min(kept, sizes_cap) * 8 + 8)); d_sizes = idx->out_l.as<int64_t>(); }
            ece_rank_kernel<<<nblocks(kept, 256), 256, 0, s>>>(keys_sorted, roots_sorted, kept, rank_of_root, d_sizes, sizes_cap); PCC_LAUNCHED();
        }
        ece_label_kernel<<<nb256, 256, 0, s>>>(g, parent, rank_of_root, d_labels); PCC_LAUNCHED();
        PCC_CUDA(cudaGetLastError());
    }
    if (mem == PCC_HOST) {
        PCC_TRY(copy_out(labels, d_labels, (size_t)rows * 4, mem, s));
        if (sizes && kept > 0) PCC_TRY(copy_out(sizes, d_sizes, (size_t)std::min(kept, sizes_cap) * 8, mem, s));
    }
    PCC_CUDA(cudaStreamSynchronize(s));
    *n_clusters = kept;
    return PCC_OK;
}

int pcc_euclidean_labels(pcc_index *idx, double tolerance, int64_t min_size, int64_t max_size, int32_t *labels, int64_t *n_clusters, int64_t *sizes,
                         int64_t sizes_cap, int mem, void *stream) {
    PCC_TRY(check_index(idx, stream));
    if (!(tolerance >= 0) || !labels || !n_clusters) return fail(PCC_ERR_INVALID, "bad tolerance / outputs");
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t n = idx->n_indexed;
    *n_clusters = 0;
    if (idx->n_input == 0) return PCC_OK;
    PCC_TRY(idx->parent.reserve((size_t)std::max<int64_t>(n, 1) * 4));
    uint32_t *parent = idx->parent.as<uint32_t>();
    KernelTimer timer(idx, s);
    if (n > 0) {
        iota_kernel<<<nblocks(n, 256), 256, 0, s>>>(parent, n); PCC_LAUNCHED();
        ece_link_kernel<<<nblocks(n, 128), 128, 0, s>>>(idx->grid(), (float)(tolerance * tolerance), ring0(idx, tolerance), parent); PCC_LAUNCHED();
        PCC_CUDA(cudaGetLastError());
    }
    const int rc = ece_finish(idx, parent, min_size, max_size, labels, n_clusters, sizes, sizes_cap, mem, s);
    timer.stop();
    return rc;
}

// ---- sharded clustering (SURVEY.md section 8e): parent forests over SORTED positions, device memory only ----
int pcc_ece_init(pcc_index *idx, uint32_t *parent, void *stream) {
    PCC_TRY(check_index(idx, stream));
    if (!parent) return fail(PCC_ERR_INVALID, "parent is NULL");
    if (idx->n_indexed > 0) { iota_kernel<<<nblocks(idx->n_indexed, 256), 256, 0, (cudaStream_t)stream>>>(parent, idx->n_indexed); PCC_LAUNCHED(); PCC_CUDA(cudaGetLastError()); }
    return PCC_OK;
}
int pcc_ece_link_range(pcc_index *idx, double tolerance, int64_t begin, int64_t end, uint32_t *parent, void *stream) {
    PCC_TRY(check_index(idx, stream));
    if (!(tolerance >= 0) || !parent || begin < 0 || end > idx->n_indexed || begin > end) return fail(PCC_ERR_INVALID, "bad range [%lld, %lld) of %lld", (long long)begin, (long long)end, (long long)idx->n_indexed);
    if (end > begin) {
        ece_link_range_kernel<<<nblocks(end - begin, 128), 128, 0, (cudaStream_t)stream>>>(idx->grid(), (float)(tolerance * tolerance), ring0(idx, tolerance), (uint32_t)begin, (uint32_t)end, parent);
        PCC_LAUNCHED(); PCC_CUDA(cudaGetLastError());
    }
    return PCC_OK;
}
int pcc_ece_absorb(pcc_index *idx, const uint32_t *other, uint32_t *parent, void *stream) {
    PCC_TRY(check_index(idx, stream));
    if (!other || !parent) return fail(PCC_ERR_INVALID, "NULL forest");
    if (idx->n_indexed > 0) {
        ece_absorb_kernel<<<nblocks(idx->n_indexed, 256), 256, 0, (cudaStream_t)stream>>>((uint32_t)idx->n_indexed, other, parent); PCC_LAUNCHED();
        ece_compress_kernel<<<nblocks(idx->n_indexed, 256), 256, 0, (cudaStream_t)stream>>>((uint32_t)idx->n_indexed, parent); PCC_LAUNCHED();
        PCC_CUDA(cudaGetLastError());
    }
    return PCC_OK;
}
int pcc_ece_finish(pcc_index *idx, uint32_t *parent, int64_t min_size, int64_t max_size, int32_t *labels, int64_t *n_clusters, int64_t *sizes, int64_t sizes_cap, void *stream) {
    PCC_TRY(check_index(idx, stream));
    if (!parent || !labels || !n_clusters) return fail(PCC_ERR_INVALID, "NULL argument");
    *n_clusters = 0;
    if (idx->n_input == 0) return PCC_OK;
    return ece_finish(idx, parent, min_size, max_size, labels, n_clusters, sizes, sizes_cap, PCC_DEVICE, (cudaStream_t)stream);
}

}  // extern "C"
