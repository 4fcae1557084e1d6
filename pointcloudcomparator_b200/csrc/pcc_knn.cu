// pcc_knn.cu -- batched exact k-nearest-neighbour kernels and the consumers fused onto them.
//
// Replaces (SURVEY.md section 8): a2 Search::nearestKSearch batched over all query points, a5 the first pass of
// StatisticalOutlierRemoval, a4 NormalEstimation with setKSearch, a6 the ICP correspondence + sums pass,
// a8 RegionGrowing(RGB)::findPointNeighbours (= pcc_knn with q == NULL).
//
// One thread owns one query.  Queries are processed in grid-cell order (the indexed cloud is already
// sorted; external batches are radix-sorted by cell key) so the 32 lanes of a warp walk overlapping
// float4 runs that stay in L1.  The search starts with the 3x3x3 block and grows ring by ring until the
// k-th distance is provably inside the scanned block (covered_d2), so results are exact for any density.
#include <algorithm>
#include <cmath>
#include <cstring>

#include <cub/device/device_select.cuh>
#include <cub/iterator/counting_input_iterator.cuh>

#include "pcc_internal.h"
#include "pcc_fastknn.cuh"

namespace pcc {

// rows_query for the kNN kernels: false for tail threads and non-finite queries; write_empty = the row still gets (-1, +inf).
// rows_query is called on each side of the v.self test, as in pcc_radius.cu's load_query.
__device__ __forceinline__ bool load_query(const Grid &g, const QueryView &v, int64_t t, float &x, float &y, float &z, int64_t &row, bool &write_empty) {
    write_empty = false;
    if (t >= v.nq) return false;
    if (v.self) { row = rows_query(g, v, t, x, y, z); return true; }
    row = rows_query(g, v, t, x, y, z);
#ifdef PCC_EXP_SEQROWS        // measurement build only (results land in processing order): what do the scattered 128-byte row writes cost?
    row = t;
#endif
#ifdef PCC_EXP_SEQQ           // measurement build only: queries read in processing order instead of gathered through `order`
    { float4 p = __ldg(v.q + t); x = p.x; y = p.y; z = p.z; }
#endif
    if (!finite3(x, y, z) || g.n == 0) { write_empty = true; return false; }
    return true;
}

// exact kNN driver: scan the 3x3x3 block, then shells, until the k-th key is inside the covered radius
template <class List>
__device__ __forceinline__ void knn_search(const Grid &g, float x, float y, float z, int k, List &list) {
    const QueryCell c = locate(g, x, y, z);
    int Rin = -1, R = 1;
    for (;;) {
        scan_progressive(g, c, Rin, R, [&]() { return to_cell_units(g, key_d2(list.at(k - 1))); },
                         [&](uint32_t, float4 p) { list.offer(make_key(dist2(x, y, z, p.x, p.y, p.z), __float_as_uint(p.w))); });
        const float cov = covered_d2(g, c, R);
        if (cov == CUDART_INF_F) break;
        const nkey_t kth = list.at(k - 1);
        if (kth != PCC_EMPTY_KEY && key_d2(kth) < cov) break;
        Rin = R; R = next_ring(g, R, key_d2(kth));
    }
}

template <int K>
__device__ __forceinline__ void write_row(const nkey_t (&key)[K], int k, int32_t *__restrict__ oi, float *__restrict__ od, int vec4) {
    if (vec4 && K >= 4 && k == K) {
#pragma unroll
        for (int j = 0; j + 3 < K; j += 4) {
            reinterpret_cast<int4 *>(oi)[j >> 2] = make_int4(key_idx(key[j]), key_idx(key[j + 1]), key_idx(key[j + 2]), key_idx(key[j + 3]));
            reinterpret_cast<float4 *>(od)[j >> 2] = make_float4(key_d2(key[j]), key_d2(key[j + 1]), key_d2(key[j + 2]), key_d2(key[j + 3]));
        }
    } else {
#pragma unroll
        for (int j = 0; j < K; ++j) if (j < k) { oi[j] = key_idx(key[j]); od[j] = key_d2(key[j]); }
    }
}
// exact path for one query slot t: insertion-sorted 64-bit keys + ring expansion (any density, any tie pattern)
template <int K>
__device__ __forceinline__ void knn_reg_body(const Grid &g, const QueryView &v, int64_t t, int k, int32_t *__restrict__ out_idx, float *__restrict__ out_d2, int vec4) {
    float x, y, z; int64_t row; bool empty;
    RegList<K> list; list.init();
    const bool live = load_query(g, v, t, x, y, z, row, empty);
    if (!live && !empty) return;
    if (live) knn_search(g, x, y, z, k, list);
    write_row<K>(list.key, k, out_idx + row * k, out_d2 + row * k, vec4);
}
template <int K>
__global__ void __launch_bounds__(128) knn_reg_kernel(Grid g, QueryView v, int k, int32_t *__restrict__ out_idx, float *__restrict__ out_d2, int vec4) {
    knn_reg_body<K>(g, v, (int64_t)blockIdx.x * blockDim.x + threadIdx.x, k, out_idx, out_d2, vec4);
}
constexpr unsigned kTiedToWide = 4096;   // a tied-query list this short is finished by knn_wide_kernel instead of knn_fixup_kernel
// queries the fast path could not prove exact (listed by knn_fast_kernel)
// `ring_flag[t]` = 1 for the queries whose 3x3x3 block did not prove the k-th distance; a stream compaction turns the flags
// into `ring_list` / `ring_count` IN PROCESSING ORDER (neighbouring lanes stay neighbours in space) for knn_rings_kernel.
struct FixList { uint32_t *list; unsigned *count; unsigned long long *stats; uint32_t *ring_list; unsigned *ring_count; uint8_t *ring_flag; uint32_t *wide_list; unsigned *wide_count; uint32_t *late_list; unsigned *late_count; uint32_t *retry_list; unsigned *retry_count; };   // stats: optional debug counters (PCC_STATS=1)
// append `value` to a device list, one atomic per warp
__device__ __forceinline__ void push_list(uint32_t *list, unsigned *count, uint32_t value) {
    const unsigned mask = __activemask();
    const int leader = __ffs(mask) - 1, lane = threadIdx.x & 31;
    unsigned base = 0;
    if (lane == leader) base = atomicAdd(count, (unsigned)__popc(mask));
    base = __shfl_sync(mask, base, leader);
    list[base + __popc(mask & ((1u << lane) - 1))] = value;
}
template <int K>
__global__ void __launch_bounds__(128) knn_fixup_kernel(Grid g, QueryView v, int k, int32_t *__restrict__ out_idx, float *__restrict__ out_d2, int vec4, FixList fix) {
    const unsigned n = *fix.count;
    if (fix.wide_list && n <= kTiedToWide) return;          // a short list was taken by knn_wide_kernel
    for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) knn_reg_body<K>(g, v, (int64_t)fix.list[i], k, out_idx, out_d2, vec4);
}

// ---- two-phase path for 2 <= k <= 32 ----
// phase 1: distances only, over the 3x3x3 block (rows clipped progressively to the ball of the running k-th distance).
// Every candidate that is not beyond the current k-th distance is also LOGGED (its position in the sorted array, 4 bytes,
// slot-major shared memory): the final neighbours are a subset of the logged candidates (the k-th distance only shrinks),
// and a query logs ~k(1 + ln(M/k)) of its M candidates, so phase 2 re-visits ~45 points instead of re-walking ~105.
// Returns tau = k-th smallest d2 inside the block (+inf if it holds fewer than k points), whether the block PROVES it
// (tau < covered_d2(1)), and the number of logged candidates (> L means the log overflowed and is incomplete).
// An unproved query (~18 % on the headline workload) still gets its row from the block, and is then listed for
// knn_rings_kernel, which merges the outer rings into that row.  Measured on B200: growing rings inside this kernel cost
// 1.3 ms of 4.7 ms because nearly every warp holds a few such queries and pays each 25-row pass with ~5 lanes active;
// listed and compacted, the same queries run with all lanes busy.
// launch shape per list size: 32 KB of log per block either way (64 slots x 128 threads, or 128 slots x 64 threads)
#ifndef PCC_LOG16
#define PCC_LOG16 48
#endif
#ifndef PCC_MB16
#define PCC_MB16 9
#endif
#ifndef PCC_LOG32
#define PCC_LOG32 80
#endif
#ifndef PCC_MB32
#define PCC_MB32 5
#endif
constexpr int64_t kSmallBatch = 1024, kSmallBatchBigK = 64;   // measured: k = 16 28 us (1 query) / 56 us (1023) vs 78 us staged; k = 50 heap 55 us (1 query) but 300 us at 512 vs 260 us selection
constexpr int kRingMaxR = 3;      // widest block knn_rings_kernel settles; beyond that a query is "wide" (knn_wide_kernel)
template <int K> struct FastCfg { static constexpr int threads = 128, log_slots = K <= 16 ? PCC_LOG16 : PCC_LOG32, min_blocks = K <= 16 ? PCC_MB16 : PCC_MB32; };
}  // namespace pcc
#include "pcc_knn_thr.cuh"
namespace pcc {
template <int K>
__device__ __forceinline__ float kth_distance(const Grid &g, const QueryCell &c, float x, float y, float z, int k, RegDist<K> &list, bool &proved,
                                              uint32_t *__restrict__ slog, int &nlog, const int R0) {
    scan_progressive(g, c, -1, R0, [&]() { return to_cell_units(g, (k == K) ? list.d[K - 1] : list.at(k - 1)); }, [&](uint32_t pos, float4 p) {
        const float d2 = dist2(x, y, z, p.x, p.y, p.z);
        if (d2 <= list.d[K - 1]) {            // "<=": a candidate tied with the final k-th distance must be in the log too
            if (nlog < FastCfg<K>::log_slots) slog[nlog * FastCfg<K>::threads] = pos;
            ++nlog;
            list.insert(d2);
        }
    });
    const float kth = (k == K) ? list.d[K - 1] : list.at(k - 1);
    const float cov = covered_d2(g, c, R0);
    proved = cov == CUDART_INF_F || kth < cov;
    return kth;
}
// One query through the two-phase path over the block of radius R0 (= 1) around its cell.  An unproved query is flagged
// for knn_rings_kernel when one more ring can settle it (its row is written first); otherwise it is listed as "wide" for
// knn_wide_kernel.  More than K candidates tied at the k-th distance -> the exact per-thread kernel.
template <int K>
__device__ __forceinline__ void knn_fast_body(const Grid &g, const QueryView &v, const int64_t t, int k, int32_t *__restrict__ out_idx, float *__restrict__ out_d2, int vec4,
                                              const FixList &fix, uint32_t *__restrict__ slog, const int R0) {
    constexpr int kFastThreads = FastCfg<K>::threads, kLogSlots = FastCfg<K>::log_slots;
    float x, y, z; int64_t row; bool empty;
    const bool live = load_query(g, v, t, x, y, z, row, empty);
    if (!live) {
        if (R0 == 1 && t < v.nq) fix.ring_flag[t] = 0;
        if (empty) { nkey_t e[K];
#pragma unroll
            for (int j = 0; j < K; ++j) e[j] = PCC_EMPTY_KEY;
            write_row<K>(e, k, out_idx + row * k, out_d2 + row * k, vec4); }
        return;
    }
    const QueryCell c = locate(g, x, y, z);
    RegDist<K> list; list.init();
    int nlog = 0; bool proved;
    const float tau = kth_distance<K>(g, c, x, y, z, k, list, proved, slog, nlog, R0);
    // phase 2: keep the logged candidates with d2 <= tau (compacted in place: the m-th survivor never overtakes the read index)
    int m = 0;
    if (nlog <= kLogSlots) {
        for (int i = 0; i < nlog; ++i) {
            const uint32_t pos = slog[i * kFastThreads];
            const float4 p = __ldg(g.pts + pos);
            if (dist2(x, y, z, p.x, p.y, p.z) <= tau) { slog[m * kFastThreads] = pos; ++m; }
        }
    } else {
        // log overflow (adversarial visiting order or heavy ties): re-walk the block inside the tau-ball instead
        scan_clipped(g, c, -1, R0, to_cell_units(g, tau), [&](uint32_t pos, float4 p) {
            if (dist2(x, y, z, p.x, p.y, p.z) <= tau) { if (m < kLogSlots) slog[m * kFastThreads] = pos; ++m; }
        });
    }
    if (fix.stats && R0 == 1) { atomicAdd(fix.stats + 0, 1ull); atomicAdd(fix.stats + 1, (unsigned long long)nlog); atomicAdd(fix.stats + 4, proved ? 0ull : 1ull); atomicAdd(fix.stats + 5, m > K ? 1ull : 0ull); atomicAdd(fix.stats + 6, (unsigned long long)m); atomicAdd(fix.stats + 3, nlog > kLogSlots ? 1ull : 0ull); }
    // where an unproved query goes next: one more ring (flag), the wide pass, or the exact kernel
    const bool tied = m > K;                                                       // more than K candidates tied at tau: exact path
    const bool wide = !tied && !proved && (tau == CUDART_INF_F || next_ring(g, 1, tau) > kRingMaxR);
    if (R0 == 1) fix.ring_flag[t] = (!tied && !proved && !wide) ? 1 : 0;
    if (tied) { push_list(fix.list, fix.count, (uint32_t)t); return; }
    if (wide) { push_list(fix.wide_list, fix.wide_count, (uint32_t)t); return; }
    nkey_t e[K];
#pragma unroll
    for (int j = 0; j < K; ++j) {
        e[j] = PCC_EMPTY_KEY;
        if (j < m) { const float4 p = __ldg(g.pts + slog[j * kFastThreads]); e[j] = make_key(dist2(x, y, z, p.x, p.y, p.z), __float_as_uint(p.w)); }
    }
    bitonic_sort_key<K>(e);
    write_row<K>(e, k, out_idx + row * k, out_d2 + row * k, vec4);
}
// measured on B200 (10 M queries, k = 16): 96 registers / 5 blocks per SM 6.44 ms, 79 / 6 blocks 5.85 ms, 64 / 8 blocks 5.51 ms --
// the kernel is latency- and issue-bound, so occupancy is worth a few spilled words
template <int K>
__global__ void __launch_bounds__(FastCfg<K>::threads, FastCfg<K>::min_blocks) knn_fast_kernel(Grid g, QueryView v, int k, int32_t *__restrict__ out_idx, float *__restrict__ out_d2, int vec4, FixList fix) {
    __shared__ uint32_t slog_all[FastCfg<K>::log_slots * FastCfg<K>::threads];
    knn_fast_body<K>(g, v, (int64_t)blockIdx.x * blockDim.x + threadIdx.x, k, out_idx, out_d2, vec4, fix, slog_all + threadIdx.x, 1);
}
// The "wide" queries (fewer than k points in the 3x3x3 block, a ball wider than two cells, or whatever knn_rings_kernel
// could not settle): few, but each needs many rows -- as one thread per query they are a serial chain of dependent loads
// hundreds of rows long (measured: 35 k such queries cost 0.9 ms).  Here ONE WARP owns a query.  A pass takes its rows 32
// at a time: each lane plans one row (run bounds), the occupied runs are appended to a run list with their length prefix
// sums, and the points of all listed runs are then dealt round-robin to the lanes (point q -> lane q % 32), so every lane
// is busy whatever the run lengths.  The best keys so far live one per lane, sorted (lane j = j-th smallest 64-bit
// (d2, index) key); a step whose points reach inside the current ball sorts them across the warp and merges them in
// with a bitonic network of shuffles (about 200 instructions), which also tightens the ball.  Passes grow ring by ring
// exactly like the per-thread search (covered_d2 / next_ring), so the result is exact for any density.
// warp-wide bitonic network over one 64-bit key per lane (ascending by lane)
__device__ __forceinline__ nkey_t warp_sort_keys(nkey_t v, int lane) {
#pragma unroll
    for (int size = 2; size <= 32; size <<= 1) {
#pragma unroll
        for (int j = size >> 1; j > 0; j >>= 1) {
            const nkey_t o = __shfl_xor_sync(0xffffffffu, v, j);
            const bool keep_min = ((lane & j) == 0) == ((lane & size) == 0);
            v = (keep_min == (o < v)) ? o : v;
        }
    }
    return v;
}
// best (ascending by lane) and batch (any order) -> the 32 smallest of both, ascending by lane
__device__ __forceinline__ nkey_t warp_merge_keys(nkey_t best, nkey_t batch, int lane) {
    batch = warp_sort_keys(batch, lane);
    const nkey_t r = __shfl_sync(0xffffffffu, batch, 31 - lane);
    nkey_t v = r < best ? r : best;                      // bitonic sequence holding the 32 smallest
#pragma unroll
    for (int j = 16; j > 0; j >>= 1) {
        const nkey_t o = __shfl_xor_sync(0xffffffffu, v, j);
        v = (((lane & j) == 0) == (o < v)) ? o : v;
    }
    return v;
}
constexpr int kWideRuns = 64;                    // runs planned per chunk of 32 rows (two strips per row at most)
__device__ __forceinline__ uint32_t warp_inclusive_scan(uint32_t v, int lane) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const uint32_t w = __shfl_up_sync(0xffffffffu, v, o); if (lane >= o) v += w; }
    return v;
}
__global__ void __launch_bounds__(128, 5) knn_wide_kernel(Grid g, QueryView v, int k, int32_t *__restrict__ out_idx, float *__restrict__ out_d2, FixList fix,
                                                         const uint32_t *__restrict__ wlist, const unsigned *__restrict__ wcount, int take_tied) {
    __shared__ uint32_t srun_j[4 * kWideRuns], srun_len[4 * kWideRuns], srun_off[4 * (kWideRuns + 1)];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    uint32_t *run_j = srun_j + wib * kWideRuns, *run_len = srun_len + wib * kWideRuns, *run_off = srun_off + wib * (kWideRuns + 1);
    // a SHORT list of tied queries (more than K candidates at the k-th distance) is taken along: as a handful of single
    // threads in knn_fixup_kernel they are a 0.1 ms latency tail; a long one (lattice data) stays with that kernel
    const unsigned n_wide = *wcount, n_tied = (take_tied && *fix.count <= kTiedToWide) ? *fix.count : 0u, n = n_wide + n_tied;
    const unsigned full = 0xffffffffu, lt = (1u << lane) - 1u;
    for (unsigned i = blockIdx.x * 4 + wib; i < n; i += gridDim.x * 4) {
        float x, y, z; int64_t row; bool empty;
        if (!load_query(g, v, (int64_t)(i < n_wide ? wlist[i] : fix.list[i - n_wide]), x, y, z, row, empty)) continue;      // warp-uniform
        const QueryCell c = locate(g, x, y, z);
        int Rin = -1, R = 3;                     // a listed query is known not to be settled by the 3x3x3 block
        nkey_t best = PCC_EMPTY_KEY;             // lane j: the j-th smallest (d2, index) key seen so far
        float tau = CUDART_INF_F;                // d2 of the k-th of them: later points must beat or tie it
        unsigned long long steps = 0;
        for (;;) {
            const int n1 = 2 * R + 1, nrows = n1 * n1;
            const float tau_u = to_cell_units(g, tau);
            const int per = Rin < 0 ? 2 : 1;     // a whole-block pass has one run per row: plan two rows per lane
            for (int row0 = 0; row0 < nrows; row0 += 32 * per) {
                // plan: rows -> occupied runs, appended to the warp's run list (at most two per lane)
                RowRuns r; r.j1 = r.e1 = r.j2 = r.e2 = 0;
                if (row0 + lane < nrows) r = row_runs(g, c, Rin, R, tau_u, (row0 + lane) / n1, (row0 + lane) % n1);
                if (per == 2 && row0 + 32 + lane < nrows) {
                    const RowRuns r2 = row_runs(g, c, Rin, R, tau_u, (row0 + 32 + lane) / n1, (row0 + 32 + lane) % n1);
                    r.j2 = r2.j1; r.e2 = r2.e1;
                }
                const unsigned m1 = __ballot_sync(full, r.j1 < r.e1), m2 = __ballot_sync(full, r.j2 < r.e2);
                const int nrun = __popc(m1) + __popc(m2);
                if (nrun == 0) continue;
                if (r.j1 < r.e1) { const int q = __popc(m1 & lt); run_j[q] = r.j1; run_len[q] = r.e1 - r.j1; }
                if (r.j2 < r.e2) { const int q = __popc(m1) + __popc(m2 & lt); run_j[q] = r.j2; run_len[q] = r.e2 - r.j2; }
                __syncwarp();
                const uint32_t la = lane < nrun ? run_len[lane] : 0u, lb = lane + 32 < nrun ? run_len[lane + 32] : 0u;
                const uint32_t ia = warp_inclusive_scan(la, lane), ib = warp_inclusive_scan(lb, lane);
                const uint32_t ta = __shfl_sync(full, ia, 31), P = ta + __shfl_sync(full, ib, 31);
                run_off[lane] = ia - la; run_off[lane + 32] = ta + ib - lb;
                if (lane == 0) run_off[kWideRuns] = P;
                __syncwarp();
                // flat walk: point q of the concatenated runs belongs to lane q % 32 -- every lane busy whatever the run
                // lengths; two points per lane and step so two loads are in flight
                int rc = 0;
                for (uint32_t q0 = 0; q0 < P; q0 += 64) {
                    bool has[2] = {false, false}; nkey_t key[2] = {PCC_EMPTY_KEY, PCC_EMPTY_KEY}; float4 p[2];
#pragma unroll
                    for (int u = 0; u < 2; ++u) {
                        const uint32_t q = q0 + 32 * u + lane;
                        has[u] = q < P;
                        if (has[u]) { while (q >= run_off[rc + 1]) ++rc; p[u] = __ldg(g.pts + run_j[rc] + (q - run_off[rc])); }
                    }
#pragma unroll
                    for (int u = 0; u < 2; ++u) {
                        if (has[u]) { const float d2 = dist2(x, y, z, p[u].x, p[u].y, p[u].z); has[u] = d2 <= tau; key[u] = has[u] ? make_key(d2, __float_as_uint(p[u].w)) : PCC_EMPTY_KEY; }
                        if (__ballot_sync(full, has[u])) {
                            best = warp_merge_keys(best, key[u], lane);
                            tau = key_d2(__shfl_sync(full, best, k - 1));
                        }
                    }
                    ++steps;
                }
                __syncwarp();
            }
            const float cov = covered_d2(g, c, R);
            if (cov == CUDART_INF_F || tau < cov) break;
            Rin = R; R = next_ring(g, R, tau);
        }
        if (fix.stats && lane == 0) { atomicAdd(fix.stats + 2, 1ull); atomicAdd(fix.stats + 7, steps); atomicAdd(fix.stats + 8 + (R <= 1 ? 0 : R == 2 ? 1 : R == 3 ? 2 : R < 8 ? 3 : R < 16 ? 4 : 5), 1ull); }
        if (lane < k) { out_idx[row * k + lane] = key_idx(best); out_d2[row * k + lane] = key_d2(best); }
        __syncwarp();
    }
}
// Finishes the queries knn_fast_kernel could not prove inside the 3x3x3 block and whose ball fits a block of radius
// kRingMaxR.  One thread per listed query (the list is in processing order, so the lanes of a warp are neighbours in
// space).  The kernel is bound by load latency, not by arithmetic, so the work is cut into stages whose loads are
// independent of each other and issued four at a time:
//   plan   -- (no loads) the rows outside the block that the ball of the k-th distance reaches -- a clipped box, not all 25
//             or 49 -- and their x-ranges, packed into the thread's log column,
//   probe  -- the occupancy bitmap for each range: most of those cells are EMPTY and are dismissed here without touching
//             the (32x larger, DRAM-resident) cell table; the occupied ranges go to the thread's run table,
//   bounds -- the cell_start pair of every run,
//   walk   -- the points of the runs, four per step across run boundaries; those inside the ball are logged.
// Only the k-th distance of the row the fast kernel wrote is read up front.  If nothing was logged (the usual outcome: the
// ball pokes into empty space) the row already is the answer; otherwise the row is loaded, the logged points are
// inserted with the exact 64-bit path and the row is rewritten.  Whatever does not fit this shape (fewer than k points in
// the block, more ranges or logged points than the tables hold, not proved afterwards) goes to knn_wide_kernel.
constexpr int kRingLog = 24, kRingRuns = 12;
#ifndef PCC_RINGS_MB
#define PCC_RINGS_MB 6
#endif
template <int K>
__global__ void __launch_bounds__(128, K <= 16 ? PCC_RINGS_MB : 4) knn_rings_kernel(Grid g, QueryView v, int k, int32_t *__restrict__ out_idx, float *__restrict__ out_d2, int vec4, FixList fix) {
    __shared__ uint32_t slog_all[kRingLog * 128];
    __shared__ uint2 srun_all[kRingRuns * 128];
    uint32_t *slog = slog_all + threadIdx.x;
    uint2 *srun = srun_all + threadIdx.x;
    const unsigned n = *fix.ring_count;
    for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const uint32_t t = fix.ring_list[i];
        float x, y, z; int64_t row; bool empty;
        if (!load_query(g, v, (int64_t)t, x, y, z, row, empty)) continue;
        int32_t *oi = out_idx + row * k; float *od = out_d2 + row * k;
        float kth = od[k - 1];                                    // +inf when the block held fewer than k points
        const QueryCell c = locate(g, x, y, z);
        const int R = kth == CUDART_INF_F ? kRingMaxR + 1 : next_ring(g, 1, kth);
        bool defer = R > kRingMaxR;
        int ncand = 0, nrun = 0, nlog = 0;
        if (!defer) {
            // plan: same conservative margins as row_runs; a range is (first cell | (cells - 1) << 28), at most 7 cells long
            const float tau_u = to_cell_units(g, kth), rad = sqrtf(tau_u) + 2e-3f;
            const int z0 = max(max(c.cz - R, 0), (int)floorf(c.uz - rad)), z1 = min(min(c.cz + R, g.nz - 1), (int)floorf(c.uz + rad));
            const int y0 = max(max(c.cy - R, 0), (int)floorf(c.uy - rad)), y1 = min(min(c.cy + R, g.ny - 1), (int)floorf(c.uy + rad));
            for (int zz = z0; zz <= z1; ++zz) {
                const float gz = fmaxf(fmaxf((float)zz - c.uz, c.uz - (float)(zz + 1)) - 2e-3f, 0.f);
                for (int yy = y0; yy <= y1; ++yy) {
                    const float gy = fmaxf(fmaxf((float)yy - c.uy, c.uy - (float)(yy + 1)) - 2e-3f, 0.f);
                    const float D = gy * gy + gz * gz;
                    if (D > tau_u) continue;
                    const float w = sqrtf(tau_u - D) + 2e-3f;
                    const int xlo = max(max(c.cx - R, 0), (int)floorf(c.ux - w)), xhi = min(min(c.cx + R, g.nx - 1), (int)floorf(c.ux + w));
                    const uint32_t base = (uint32_t)(((size_t)zz * g.ny + yy) * g.nx);
                    const bool shell = max(abs(zz - c.cz), abs(yy - c.cy)) > 1;
                    // shell row: one range; inner row: the cells left and right of the 3x3x3 block
                    const int xa1 = xlo, xb1 = shell ? xhi : min(xhi, c.cx - 2);
                    const int xa2 = max(xlo, c.cx + 2), xb2 = shell ? -1 : xhi;
                    if (xa1 <= xb1) { if (ncand < kRingLog) slog[ncand * 128] = (base + (uint32_t)xa1) | ((uint32_t)(xb1 - xa1) << 28); ++ncand; }
                    if (xa2 <= xb2) { if (ncand < kRingLog) slog[ncand * 128] = (base + (uint32_t)xa2) | ((uint32_t)(xb2 - xa2) << 28); ++ncand; }
                }
            }
            defer = ncand > kRingLog;
        }
        if (!defer) {
            // probe: four ranges per step, bitmap words first, tests after
            for (int r0 = 0; r0 < ncand; r0 += 4) {
                uint32_t cw[4], w0[4], w1[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    cw[u] = slog[min(r0 + u, ncand - 1) * 128];
                    const uint32_t b = cw[u] & 0x0fffffffu;
                    w0[u] = __ldg(g.occ + (b >> 5)); w1[u] = __ldg(g.occ + (b >> 5) + 1);
                }
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const uint32_t b = cw[u] & 0x0fffffffu, len = (cw[u] >> 28) + 1u;
                    const uint32_t bits = __funnelshift_r(w0[u], w1[u], b & 31u) & ((1u << len) - 1u);
                    if (r0 + u < ncand && bits != 0u) { if (nrun < kRingRuns) srun[nrun * 128] = make_uint2(b, b + len); ++nrun; }
                }
            }
            defer = nrun > kRingRuns;
        }
        if (!defer && nrun > 0) {
            // bounds: cell ranges -> point ranges
            for (int r0 = 0; r0 < nrun; r0 += 4) {
                uint2 pr[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) { const uint2 cr = srun[min(r0 + u, nrun - 1) * 128]; pr[u] = make_uint2(__ldg(g.cell_start + cr.x), __ldg(g.cell_start + cr.y)); }
#pragma unroll
                for (int u = 0; u < 4; ++u) if (r0 + u < nrun) srun[(r0 + u) * 128] = pr[u];
            }
            // walk: four points per step, taken across run boundaries (every run is non-empty: the bitmap is exact)
            int r = 0;
            uint2 cur = srun[0];
            bool more = true;
            while (more) {
                uint32_t pos[4]; bool ok[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    if (cur.x >= cur.y && r + 1 < nrun) { ++r; cur = srun[r * 128]; }
                    ok[u] = cur.x < cur.y; pos[u] = ok[u] ? cur.x : 0u;
                    if (ok[u]) ++cur.x;
                }
                more = cur.x < cur.y || r + 1 < nrun;
                float4 p[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) p[u] = __ldg(g.pts + pos[u]);
#pragma unroll
                for (int u = 0; u < 4; ++u)
                    if (ok[u] && dist2(x, y, z, p[u].x, p[u].y, p[u].z) <= kth) { if (nlog < kRingLog) slog[nlog * 128] = pos[u]; ++nlog; }
            }
            defer = nlog > kRingLog;
        }
        RegList<K> list;
        if (!defer && nlog > 0) {
            if (vec4 && K >= 4 && k == K) {
#pragma unroll
                for (int j = 0; j + 3 < K; j += 4) {
                    const int4 a = reinterpret_cast<const int4 *>(oi)[j >> 2]; const float4 d = reinterpret_cast<const float4 *>(od)[j >> 2];
                    list.key[j] = a.x < 0 ? PCC_EMPTY_KEY : make_key(d.x, (uint32_t)a.x); list.key[j + 1] = a.y < 0 ? PCC_EMPTY_KEY : make_key(d.y, (uint32_t)a.y);
                    list.key[j + 2] = a.z < 0 ? PCC_EMPTY_KEY : make_key(d.z, (uint32_t)a.z); list.key[j + 3] = a.w < 0 ? PCC_EMPTY_KEY : make_key(d.w, (uint32_t)a.w);
                }
            } else {
#pragma unroll
                for (int j = 0; j < K; ++j) { list.key[j] = PCC_EMPTY_KEY; if (j < k) { const int32_t a = oi[j]; if (a >= 0) list.key[j] = make_key(od[j], (uint32_t)a); } }
            }
            for (int q = 0; q < nlog; ++q) { const float4 p = __ldg(g.pts + slog[q * 128]); list.offer(make_key(dist2(x, y, z, p.x, p.y, p.z), __float_as_uint(p.w))); }
            kth = key_d2((k == K) ? list.key[K - 1] : list.at(k - 1));
        }
        if (!defer) {
            const float cov = covered_d2(g, c, R);
            defer = !(cov == CUDART_INF_F || kth < cov);
        }
        if (defer) push_list(fix.late_list, fix.late_count, t);
        else if (nlog > 0) write_row<K>(list.key, k, oi, od, vec4);
    }
}

// ---- warp-owns-a-cell variant: the 3x3x3 stencil is staged in shared memory with TMA bulk copies ----
// Used when a grid cell holds many queries (Q >> N, e.g. the 100 M-query point of the BASELINE sweep): the lanes of a warp
// that fall into the same cell share one stencil, so the warp (a) computes the 9 run bounds once, (b) pulls the runs into
// its shared-memory tile with cp.async.bulk (one elected lane, completion on an mbarrier), and (c) walks the tile with
// UNIFORM trip counts and broadcast 16-byte shared loads -- no per-lane address math, no run-length divergence.  Ring >= 2,
// the logged phase 2, the sort and the write are the per-lane code of knn_fast_kernel.  With few queries per cell the
// lanes of a warp belong to ~4 different cells and this variant loses to the per-thread walk; measured on B200 it also loses
// at 80 queries per cell (single-buffered tiles expose the bulk-copy latency), so it is opt-in only (DESIGN.md section 5).
namespace tma {
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long *bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long *bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, unsigned bytes, unsigned long long *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long *bar, unsigned parity) {
    asm volatile("{\n\t.reg .pred p;\n\tWAIT_%=:\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t@p bra DONE_%=;\n\tbra WAIT_%=;\n\tDONE_%=:\n\t}"
                 ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
}  // namespace tma

static constexpr int kCellWarps = 4, kCellCap = 320, kCellLog = 48;   // 20 KB tiles + 24 KB logs per block (static shared memory limit 48 KB)
template <int K>
__global__ void __launch_bounds__(kCellWarps * 32, 5) knn_cell_kernel(Grid g, QueryView v, int k, int32_t *__restrict__ out_idx, float *__restrict__ out_d2, int vec4, FixList fix) {
    __shared__ __align__(128) float4 s_tile[kCellWarps][kCellCap];
    __shared__ uint32_t s_log_all[kCellWarps][kCellLog][32];
    __shared__ __align__(8) unsigned long long s_bar[kCellWarps];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float4 *tile = s_tile[warp];
    uint32_t *slog = &s_log_all[warp][0][lane];           // slot stride = 32 words
    unsigned long long *bar = &s_bar[warp];
    if (lane == 0) tma::mbar_init(bar, 1);
    __syncwarp();
    unsigned parity = 0;

    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    float x = 0.f, y = 0.f, z = 0.f; int64_t row = 0; bool empty = false;
    const bool live = load_query(g, v, t, x, y, z, row, empty);
    QueryCell c; c.cx = c.cy = c.cz = 0; c.ux = c.uy = c.uz = 0.f;
    if (live) c = locate(g, x, y, z);
    const int cell_id = live ? (c.cz * g.ny + c.cy) * g.nx + c.cx : -1;
    RegDist<K> list; list.init();
    int nlog = 0;

    // ring 1, cooperatively per distinct cell among the warp's lanes
    unsigned todo = __ballot_sync(0xffffffffu, live);
    while (todo) {
        const int leader = __ffs(todo) - 1;
        const int cid = __shfl_sync(0xffffffffu, cell_id, leader);
        const bool mine = live && cell_id == cid;
        const unsigned group = __ballot_sync(0xffffffffu, mine);
        const int lcx = __shfl_sync(0xffffffffu, c.cx, leader), lcy = __shfl_sync(0xffffffffu, c.cy, leader), lcz = __shfl_sync(0xffffffffu, c.cz, leader);
        // lane r < 9 owns row r of the stencil (centre-out order); bounds are then broadcast with shuffles
        uint32_t my_s = 0, my_e = 0;
        if (lane < 9) {
            const int dz = centre_out(lane / 3), dy = centre_out(lane % 3);
            const int zz = lcz + dz, yy = lcy + dy;
            if (zz >= 0 && zz < g.nz && yy >= 0 && yy < g.ny) {
                const uint32_t *rowp = g.cell_start + ((size_t)zz * g.ny + yy) * g.nx;
                my_s = __ldg(rowp + max(lcx - 1, 0)); my_e = __ldg(rowp + min(lcx + 1, g.nx - 1) + 1);
            }
        }
        int r = 0; uint32_t off_in_run = 0;               // progress through the 9 runs (uniform across the warp)
        while (r < 9) {
            // plan one tile: whole runs while they fit, else a slice of the run that does not fit.  Every lane computes the same
            // plan; lane q keeps the (start, count) of run q so later loops can fetch it with a runtime-indexed shuffle.
            uint32_t my_ts = 0, my_tn = 0, fill = 0;
            int r_next = 9; uint32_t off_next = 0; bool open = true;
#pragma unroll
            for (int q = 0; q < 9; ++q) {
                const uint32_t s_q = __shfl_sync(0xffffffffu, my_s, q), e_q = __shfl_sync(0xffffffffu, my_e, q);
                if (open && q >= r) {
                    const uint32_t begin = s_q + (q == r ? off_in_run : 0u);
                    const uint32_t avail = e_q - begin;
                    const uint32_t take = min(avail, (uint32_t)kCellCap - fill);
                    if (lane == q) { my_ts = begin; my_tn = take; }
                    fill += take;
                    if (take == avail) { r_next = q + 1; off_next = 0; }
                    else { r_next = q; off_next = (q == r ? off_in_run : 0u) + take; open = false; }
                    if (fill == (uint32_t)kCellCap) open = false;
                }
            }
            r = r_next; off_in_run = off_next;
            if (fill == 0) continue;
            // stage the tile: one elected lane posts the byte count and issues one bulk copy per run
            if (lane == 0) { tma::fence_proxy_async(); tma::mbar_expect_tx(bar, fill * 16u); }
            {
                uint32_t off = 0;
#pragma unroll
                for (int q = 0; q < 9; ++q) {
                    const uint32_t ts = __shfl_sync(0xffffffffu, my_ts, q), tn = __shfl_sync(0xffffffffu, my_tn, q);
                    if (lane == 0 && tn) tma::bulk_g2s(tile + off, g.pts + ts, tn * 16u, bar);
                    off += tn;
                }
            }
            tma::mbar_wait(bar, parity); parity ^= 1u;
            // walk the tile: uniform trip counts, broadcast 16-byte shared loads
            uint32_t off = 0;
#pragma unroll 1
            for (int q = 0; q < 9; ++q) {
                const uint32_t ts = __shfl_sync(0xffffffffu, my_ts, q), tn = __shfl_sync(0xffffffffu, my_tn, q);
                for (uint32_t jj = 0; jj < tn; ++jj) {
                    const float4 p = tile[off + jj];
                    if (mine) {
                        const float d2 = dist2(x, y, z, p.x, p.y, p.z);
                        if (d2 <= list.d[K - 1]) {
                            if (nlog < kCellLog) slog[nlog * 32] = ts + jj;
                            ++nlog;
                            list.insert(d2);
                        }
                    }
                }
                off += tn;
            }
            __syncwarp();
        }
        todo &= ~group;
    }
    if (!live) {
        if (empty) { nkey_t e[K];
#pragma unroll
            for (int j = 0; j < K; ++j) e[j] = PCC_EMPTY_KEY;
            write_row<K>(e, k, out_idx + row * k, out_d2 + row * k, vec4); }
        return;
    }
    // rings >= 2 per lane (ball-clipped), same as knn_fast_kernel
    int R = 1;
    float tau = (k == K) ? list.d[K - 1] : list.at(k - 1);
    for (;;) {
        const float cov = covered_d2(g, c, R);
        if (cov == CUDART_INF_F || tau < cov) break;
        const int Rin = R; R = next_ring(g, R, tau);
        scan_progressive(g, c, Rin, R, [&]() { return to_cell_units(g, (k == K) ? list.d[K - 1] : list.at(k - 1)); }, [&](uint32_t pos, float4 p) {
            const float d2 = dist2(x, y, z, p.x, p.y, p.z);
            if (d2 <= list.d[K - 1]) { if (nlog < kCellLog) slog[nlog * 32] = pos; ++nlog; list.insert(d2); }
        });
        tau = (k == K) ? list.d[K - 1] : list.at(k - 1);
    }
    int m = 0;
    if (nlog <= kCellLog) {
        for (int i = 0; i < nlog; ++i) {
            const uint32_t pos = slog[i * 32];
            const float4 p = __ldg(g.pts + pos);
            if (dist2(x, y, z, p.x, p.y, p.z) <= tau) { slog[m * 32] = pos; ++m; }
        }
    } else {
        scan_clipped(g, c, -1, R, to_cell_units(g, tau), [&](uint32_t pos, float4 p) {
            if (dist2(x, y, z, p.x, p.y, p.z) <= tau) { if (m < kCellLog) slog[m * 32] = pos; ++m; }
        });
    }
    if (m > K) { fix.list[atomicAdd(fix.count, 1u)] = (uint32_t)t; return; }
    nkey_t e[K];
#pragma unroll
    for (int j = 0; j < K; ++j) {
        e[j] = PCC_EMPTY_KEY;
        if (j < m) { const float4 p = __ldg(g.pts + slog[j * 32]); e[j] = make_key(dist2(x, y, z, p.x, p.y, p.z), __float_as_uint(p.w)); }
    }
    bitonic_sort_key<K>(e);
    write_row<K>(e, k, out_idx + row * k, out_d2 + row * k, vec4);
}

// 32 < k <= PCC_MAX_K: per-thread max-heap in dynamic shared memory
__global__ void knn_heap_kernel(Grid g, QueryView v, int k, int32_t *__restrict__ out_idx, float *__restrict__ out_d2) {
    extern __shared__ nkey_t smem_keys[];
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    float x, y, z; int64_t row; bool empty;
    HeapList list; list.init(smem_keys + threadIdx.x, blockDim.x, k);
    const bool live = load_query(g, v, t, x, y, z, row, empty);
    if (!live && !empty) return;
    if (live) {
        const QueryCell c = locate(g, x, y, z);
        int Rin = -1, R = 1;
        for (;;) {
            scan_progressive(g, c, Rin, R, [&]() { return list.full() ? to_cell_units(g, key_d2(list.worst())) : CUDART_INF_F; },
                             [&](uint32_t, float4 p) { list.offer(make_key(dist2(x, y, z, p.x, p.y, p.z), __float_as_uint(p.w))); });
            const float cov = covered_d2(g, c, R);
            if (cov == CUDART_INF_F) break;
            if (list.full() && key_d2(list.worst()) < cov) break;
            Rin = R; R = next_ring(g, R, list.full() ? key_d2(list.worst()) : CUDART_INF_F);
        }
    }
    list.finish();
    int32_t *oi = out_idx + row * k; float *od = out_d2 + row * k;
    for (int j = 0; j < k; ++j) { nkey_t e = list.at(j); oi[j] = key_idx(e); od[j] = key_d2(e); }
}

// ---- fused: StatisticalOutlierRemoval first pass (mean distance to the mean_k nearest, self dropped) ----
// EXACT: mean_k == K - 1 (the instantiated sizes match mean_k = 1, 4, 8, 16, 32, 50), every list index is static.
template <int K, bool EXACT>
__global__ void __launch_bounds__(128, (K <= 17 ? 8 : (K <= 33 ? 6 : 4))) mean_dist_reg_kernel(Grid g, QueryView v, int mean_k, float *__restrict__ out) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    float x, y, z; int64_t row; bool empty;
    const bool live = load_query(g, v, t, x, y, z, row, empty);
    if (!live) { if (empty) out[row] = 0.f; return; }
    RegDist<K> list; list.init();
    const QueryCell c = locate(g, x, y, z);
    int Rin = -1, R = 1;
    for (;;) {
        scan_progressive(g, c, Rin, R, [&]() { return to_cell_units(g, EXACT ? list.d[K - 1] : list.at(mean_k)); }, [&](uint32_t, float4 p) { list.offer(dist2(x, y, z, p.x, p.y, p.z)); });
        const float cov = covered_d2(g, c, R);
        if (cov == CUDART_INF_F) break;
        const float kth = EXACT ? list.d[K - 1] : list.at(mean_k);
        if (kth < cov) break;
        Rin = R; R = next_ring(g, R, kth);
    }
    double s = 0.0;
    if (EXACT) {
#pragma unroll
        for (int j = 1; j < K; ++j) s += sqrt((double)list.d[j]);
    } else {
#pragma unroll 1
        for (int j = 1; j <= mean_k; ++j) s += sqrt((double)list.at(j));
    }
    out[row] = (float)(s / (double)mean_k);
}
__global__ void mean_dist_heap_kernel(Grid g, QueryView v, int mean_k, float *__restrict__ out) {
    extern __shared__ nkey_t smem_keys[];
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    float x, y, z; int64_t row; bool empty;
    const bool live = load_query(g, v, t, x, y, z, row, empty);
    if (!live) { if (empty) out[row] = 0.f; return; }
    HeapList list; list.init(smem_keys + threadIdx.x, blockDim.x, mean_k + 1);
    const QueryCell c = locate(g, x, y, z);
    int Rin = -1, R = 1;
    for (;;) {
        scan_progressive(g, c, Rin, R, [&]() { return list.full() ? to_cell_units(g, key_d2(list.worst())) : CUDART_INF_F; },
                             [&](uint32_t, float4 p) { list.offer(make_key(dist2(x, y, z, p.x, p.y, p.z), __float_as_uint(p.w))); });
        const float cov = covered_d2(g, c, R);
        if (cov == CUDART_INF_F) break;
        if (list.full() && key_d2(list.worst()) < cov) break;
        Rin = R; R = next_ring(g, R, list.full() ? key_d2(list.worst()) : CUDART_INF_F);
    }
    list.finish();
    double s = 0.0;
    for (int j = 1; j <= mean_k; ++j) s += sqrt((double)key_d2(list.at(j)));
    out[row] = (float)(s / (double)mean_k);
}

// ---- fused: NormalEstimation with setKSearch(k) ----
template <int K>
__global__ void __launch_bounds__(128) normals_knn_reg_kernel(Grid g, QueryView v, int k, const uint32_t *__restrict__ inv_pos, float vx, float vy, float vz, float4 *__restrict__ out) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    float x, y, z; int64_t row; bool empty;
    const bool live = load_query(g, v, t, x, y, z, row, empty);
    if (!live) { if (empty) out[row] = make_float4(CUDART_NAN_F, CUDART_NAN_F, CUDART_NAN_F, CUDART_NAN_F); return; }
    RegList<K> list; list.init();
    knn_search(g, x, y, z, k, list);
    float a[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0}; int cnt = 0;
#pragma unroll
    for (int j = 0; j < K; ++j) if (j < k && list.key[j] != PCC_EMPTY_KEY) { float4 p = __ldg(g.pts + __ldg(inv_pos + (uint32_t)list.key[j])); accu_add(a, p.x, p.y, p.z); ++cnt; }
    out[row] = normal_from_accu(a, cnt, x, y, z, vx, vy, vz);
}
__global__ void normals_knn_heap_kernel(Grid g, QueryView v, int k, const uint32_t *__restrict__ inv_pos, float vx, float vy, float vz, float4 *__restrict__ out) {
    extern __shared__ nkey_t smem_keys[];
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    float x, y, z; int64_t row; bool empty;
    const bool live = load_query(g, v, t, x, y, z, row, empty);
    if (!live) { if (empty) out[row] = make_float4(CUDART_NAN_F, CUDART_NAN_F, CUDART_NAN_F, CUDART_NAN_F); return; }
    HeapList list; list.init(smem_keys + threadIdx.x, blockDim.x, k);
    const QueryCell c = locate(g, x, y, z);
    int Rin = -1, R = 1;
    for (;;) {
        scan_progressive(g, c, Rin, R, [&]() { return list.full() ? to_cell_units(g, key_d2(list.worst())) : CUDART_INF_F; },
                             [&](uint32_t, float4 p) { list.offer(make_key(dist2(x, y, z, p.x, p.y, p.z), __float_as_uint(p.w))); });
        const float cov = covered_d2(g, c, R);
        if (cov == CUDART_INF_F) break;
        if (list.full() && key_d2(list.worst()) < cov) break;
        Rin = R; R = next_ring(g, R, list.full() ? key_d2(list.worst()) : CUDART_INF_F);
    }
    list.finish();
    float a[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0}; int cnt = 0;
    for (int j = 0; j < list.cnt; ++j) { float4 p = __ldg(g.pts + __ldg(inv_pos + (uint32_t)list.at(j))); accu_add(a, p.x, p.y, p.z); ++cnt; }
    out[row] = normal_from_accu(a, cnt, x, y, z, vx, vy, vz);
}

// ---- fused: ICP correspondence pass ----
struct Mat34 { float m[12]; };
static constexpr int kIcpThreads = 128, kIcpMaxPriorR = 16;
// One thread per source point: move it by T (IterativeClosestPoint::transformCloud arithmetic), find its nearest
// target point, and reduce the 16 sums Umeyama needs + the correspondence count to one row of doubles per block.
// `prior[row]` = sorted position of the target point this source row matched in the previous pass (0xFFFFFFFF = none).  ANY
// target point is a valid upper bound for the nearest-neighbour distance, so the result does not depend on it; but between
// two ICP iterations a point moves little, the old match is (nearly) the new one, and the search starts as ONE pass over
// the block that covers the ball of that distance, clipped to the ball -- instead of doubling blocks outwards through
// empty space until something is found (first iterations), or walking the whole 3x3x3 block (converged iterations).
// (Seeding the first pass -- every 16th source point answered first, its match handed to the 15 after it as their starting
// bound -- was measured on the 10 M pair and is slower: 23.6 vs 17.5 ms.  One pass over the whole ball of a loose bound costs
// more than shells that double until the first point is seen and are clipped from there on.)
__global__ void __launch_bounds__(kIcpThreads) icp_step_kernel(Grid g, float4 *__restrict__ src, const uint32_t *__restrict__ order, int64_t ns, Mat34 T, int apply,
                                                               double *__restrict__ partials, int32_t *__restrict__ corr_idx, float *__restrict__ corr_d2,
                                                               uint32_t *__restrict__ prior) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    double acc[17];
#pragma unroll
    for (int i = 0; i < 17; ++i) acc[i] = 0.0;
    if (t < ns) {
        const uint32_t qi = order ? __ldg(order + t) : (uint32_t)t;
        float4 p = src[qi];
        int32_t bi = -1; float bd = CUDART_INF_F;
        uint32_t acc_pos = 0xFFFFFFFFu;
        if (finite3(p.x, p.y, p.z)) {
            if (apply) {   // ((m0*x + m1*y) + m2*z) + m3 in fp32; -fmad=false keeps the products separately rounded
                float nx = ((T.m[0] * p.x + T.m[1] * p.y) + T.m[2] * p.z) + T.m[3];
                float ny = ((T.m[4] * p.x + T.m[5] * p.y) + T.m[6] * p.z) + T.m[7];
                float nz = ((T.m[8] * p.x + T.m[9] * p.y) + T.m[10] * p.z) + T.m[11];
                p.x = nx; p.y = ny; p.z = nz;
                src[qi] = p;
            }
            if (g.n > 0 && finite3(p.x, p.y, p.z)) {
                Nearest1 nn; nn.init(p.x, p.y, p.z);
                const QueryCell c = locate(g, p.x, p.y, p.z);
                int R = 1;
                const uint32_t pv = prior ? prior[qi] : 0xFFFFFFFFu;
                if (pv < g.n) {
                    const float4 m = __ldg(g.pts + pv);
                    nn.bd = dist2(p.x, p.y, p.z, m.x, m.y, m.z); nn.bidx = __float_as_uint(m.w); nn.bpos = pv;
                    R = next_ring(g, 0, nn.bd);
                    // a bound wider than kIcpMaxPriorR cells does not help (a pass costs O(R^2) rows): forget it and search
                    // outwards as usual (the source cloud changed between calls).
                    if (R > kIcpMaxPriorR) { nn.init(p.x, p.y, p.z); R = 1; }
                }
                nearest1_search(g, c, R, nn);
                bi = nn.found() ? (int32_t)nn.bidx : -1; bd = nn.bd;
                const uint32_t bpos = nn.bpos;
                if (bi >= 0) {
                    acc_pos = bpos;
                    const float4 m = __ldg(g.pts + bpos);
                    const double sx = p.x, sy = p.y, sz = p.z, tx = m.x, ty = m.y, tz = m.z;
                    acc[0] = sx; acc[1] = sy; acc[2] = sz; acc[3] = tx; acc[4] = ty; acc[5] = tz;
                    acc[6] = tx * sx; acc[7] = tx * sy; acc[8] = tx * sz;
                    acc[9] = ty * sx; acc[10] = ty * sy; acc[11] = ty * sz;
                    acc[12] = tz * sx; acc[13] = tz * sy; acc[14] = tz * sz;
                    acc[15] = (double)bd; acc[16] = 1.0;
                }
            }
        }
        if (corr_idx) corr_idx[qi] = bi;
        if (corr_d2) corr_d2[qi] = bd;
        if (prior) prior[qi] = bi >= 0 ? acc_pos : 0xFFFFFFFFu;
    }
    __shared__ double red[kIcpThreads / 32][17];
#pragma unroll
    for (int i = 0; i < 17; ++i) {
        double v = acc[i];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5][i] = v;
    }
    __syncthreads();
    if (threadIdx.x < 17) {
        double v = 0.0;
#pragma unroll
        for (int w = 0; w < kIcpThreads / 32; ++w) v += red[w][threadIdx.x];
        partials[(size_t)blockIdx.x * 17 + threadIdx.x] = v;
    }
}
// fixed-order final reduction of the per-block rows (deterministic run to run)
__global__ void icp_reduce_kernel(const double *__restrict__ partials, int64_t n_blocks, double *__restrict__ out) {
    __shared__ double red[256];
    const int comp = blockIdx.x;    // 0..16
    double v = 0.0;
    for (int64_t b = threadIdx.x; b < n_blocks; b += blockDim.x) v += partials[(size_t)b * 17 + comp];
    red[threadIdx.x] = v;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) { if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o]; __syncthreads(); }
    if (threadIdx.x == 0) out[comp] = red[0];
}
// strided rows -> float4 working copy of the source cloud
__global__ void icp_load_kernel(const uint8_t *__restrict__ raw, int stride, int64_t ns, float4 *__restrict__ dst) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= ns) return;
    const float *p = (const float *)(raw + i * (int64_t)stride);
    dst[i] = make_float4(p[0], p[1], p[2], 1.0f);
}
__global__ void icp_store_kernel(const float4 *__restrict__ srcw, int64_t ns, uint8_t *__restrict__ raw, int stride) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= ns) return;
    float *p = (float *)(raw + i * (int64_t)stride);
    float4 v = srcw[i];
    p[0] = v.x; p[1] = v.y; p[2] = v.z;
}

__global__ void fill_f32_kernel(float *p, int64_t n, float v) { int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; if (i < n) p[i] = v; }

template <int K>
static void launch_knn_reg(const Grid &g, const QueryView &v, int k, int32_t *oi, float *od, int vec4, cudaStream_t s) {
    knn_reg_kernel<K><<<nblocks(v.nq, 128), 128, 0, s>>>(g, v, k, oi, od, vec4);
    PCC_LAUNCHED();
}
template <int K>
static void launch_knn_cell(const Grid &g, const QueryView &v, int k, int32_t *oi, float *od, int vec4, FixList fix, cudaStream_t s) {
    fix.wide_list = nullptr;            // this variant grows its rings in the kernel; every listed query goes to knn_fixup_kernel
    cudaMemsetAsync(fix.count, 0, sizeof(unsigned), s);
    knn_cell_kernel<K><<<nblocks(v.nq, kCellWarps * 32), kCellWarps * 32, 0, s>>>(g, v, k, oi, od, vec4, fix);
    PCC_LAUNCHED();
    knn_fixup_kernel<K><<<148 * 4, 128, 0, s>>>(g, v, k, oi, od, vec4, fix);
    PCC_LAUNCHED();
}
// logging-threshold table of knn_thr_kernel for (this grid, k): calibrated from a strided sample of the batch, cached in the index
constexpr int64_t kCalibSample = 1 << 15;
constexpr float kCalibQuantile = 0.99f;
template <int K>
static int calibrate_thr(pcc_index *idx, const Grid &g, const QueryView &v, int k, cudaStream_t s) {
    PCC_TRY(idx->calib.reserve((size_t)kCalibBuckets * kCalibBins * 4 + kCalibBuckets * 4));
    unsigned *hist = idx->calib.as<unsigned>();
    float *ratio = (float *)(hist + kCalibBuckets * kCalibBins);
    PCC_CUDA(cudaMemsetAsync(hist, 0, (size_t)kCalibBuckets * kCalibBins * 4, s));
    const int64_t stride = std::max<int64_t>(1, v.nq / kCalibSample), ns = (v.nq + stride - 1) / stride;
    knn_calib_kernel<K><<<nblocks(ns, 128), 128, 0, s>>>(g, v, k, stride, hist);
    PCC_LAUNCHED();
    static const float quantile = getenv("PCC_THR_QUANTILE") ? (float)atof(getenv("PCC_THR_QUANTILE")) : kCalibQuantile;      // measurement knob
    knn_calib_finish_kernel<<<1, kCalibBuckets, 0, s>>>(hist, ratio, quantile);
    PCC_LAUNCHED();
    return PCC_OK;
}
template <int K>
static int launch_knn_fast(pcc_index *idx, const Grid &g, const QueryView &v, int k, int32_t *oi, float *od, int vec4, FixList fix, cudaStream_t s) {
    size_t tmp = idx->sel_tmp_bytes;
    if (idx->sel_tmp_nq != v.nq) {
        cub::DeviceSelect::Flagged(nullptr, tmp, cub::CountingInputIterator<uint32_t>(0), fix.ring_flag, fix.ring_list, fix.ring_count, (int)v.nq, s);
        idx->sel_tmp_nq = v.nq; idx->sel_tmp_bytes = tmp;
    }
    PCC_TRY(idx->cub_tmp.reserve(tmp));
    if (!idx->aux_stream) {
        PCC_CUDA(cudaStreamCreateWithFlags(&idx->aux_stream, cudaStreamNonBlocking));
        PCC_CUDA(cudaEventCreateWithFlags(&idx->ev_fork, cudaEventDisableTiming));
        PCC_CUDA(cudaEventCreateWithFlags(&idx->ev_join, cudaEventDisableTiming));
    }
    if (fix.stats) { cudaMemsetAsync(fix.count, 0, sizeof(unsigned), s); cudaMemsetAsync(fix.wide_count, 0, 3 * sizeof(unsigned), s); }      // the stats words sit between the counters
    else cudaMemsetAsync(fix.count, 0, 33 * sizeof(unsigned), s);           // count [0] ... wide_count, late_count, retry_count [30..32] in one go
    static const bool old_fast_env = getenv("PCC_OLD_FAST") != nullptr;   // measurement aid: the round-1 block kernel (sorted insertion + candidate log)
    // Measured on B200, 10 M queries vs the 10 M-point surface cloud (profiles/r2/sweep_k_blockkernel.txt): the threshold kernel wins at
    // K = 16 (3.50 vs 3.81 ms), ties at K = 8 (2.53 / 2.51) and loses at K = 4 (2.28 / 2.07: ~10 logged candidates do not pay for a
    // 16-wide network) and K = 32 (10.96 / 9.17: two 32-wide networks per block of the log), so it serves 8 < k <= 16 only.
    static const bool thr_all = getenv("PCC_THR_ALL") != nullptr;
    const bool old_fast = old_fast_env || (K != 16 && !thr_all) || v.nq >= (1ll << 31);     // the retry list keeps a flag bit beside the query number
    if (old_fast) {
        knn_fast_kernel<K><<<nblocks(v.nq, FastCfg<K>::threads), FastCfg<K>::threads, 0, s>>>(g, v, k, oi, od, vec4, fix);
        PCC_LAUNCHED();
    } else {
        // the table only steers how many candidates a query logs (the result is exact whatever it holds), so it is kept
        // across calls; it is re-made when the previous call sent more than 4 % of its queries to the exact path
        // (the count is read back without a sync, so it is at worst one call late)
        const pcc_index *owner = idx->grid_owner ? idx->grid_owner : idx;
        unsigned *h_fb = (unsigned *)((char *)idx->h_pinned + 2048);
        if (idx->calib_k == k && idx->calib_gen == owner->grid_gen && idx->calib_nq > 0 && (double)h_fb[0] > 0.04 * (double)idx->calib_nq) idx->calib_k = -1;
        if (idx->calib_k != k || idx->calib_gen != owner->grid_gen) {
            PCC_TRY(calibrate_thr<K>(idx, g, v, k, s));
            idx->calib_k = k; idx->calib_gen = owner->grid_gen;
        }
        const float *ratio = (const float *)(idx->calib.as<unsigned>() + kCalibBuckets * kCalibBins);
        static std::atomic<unsigned long long> attr_done{0};            // per device, once per process (5-10 us each otherwise, every call)
        if (!((attr_done.load() >> (idx->device & 63)) & 1ull)) {
            PCC_CUDA(cudaFuncSetAttribute(knn_thr_kernel<K, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ThrCfg<K>::smem));
            PCC_CUDA(cudaFuncSetAttribute(knn_thr_kernel<K, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ThrCfg<K>::smem));
            PCC_CUDA(cudaFuncSetAttribute(knn_thr_retry_kernel<K, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ThrCfg<K>::smem));
            PCC_CUDA(cudaFuncSetAttribute(knn_thr_retry_kernel<K, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ThrCfg<K>::smem));
            attr_done.fetch_or(1ull << (idx->device & 63));
        }
        const char *staged_env = getenv("PCC_THR_STAGED");              // TMA-staged variant: opt-in, read per call so a test can switch it (measured slower, DESIGN.md section 5)
        const bool staged = staged_env && atoi(staged_env) != 0;
        if (staged && k == K) {
            static std::atomic<unsigned long long> sattr_done{0};
            if (!((sattr_done.load() >> (idx->device & 63)) & 1ull)) {
                PCC_CUDA(cudaFuncSetAttribute(knn_thr_staged_kernel<K, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ThrStagedCfg<K>::smem));
                sattr_done.fetch_or(1ull << (idx->device & 63));
            }
            knn_thr_staged_kernel<K, true><<<nblocks(v.nq, ThrCfg<K>::threads), ThrCfg<K>::threads, ThrStagedCfg<K>::smem, s>>>(g, v, k, oi, od, vec4, fix, ratio);
            PCC_LAUNCHED();
            knn_thr_retry_kernel<K, true><<<148 * 4, ThrCfg<K>::threads, ThrCfg<K>::smem, s>>>(g, v, k, oi, od, vec4, fix, ratio);
            PCC_LAUNCHED();
        } else if (k == K) {
            knn_thr_kernel<K, true><<<nblocks(v.nq, ThrCfg<K>::threads), ThrCfg<K>::threads, ThrCfg<K>::smem, s>>>(g, v, k, oi, od, vec4, fix, ratio);
            PCC_LAUNCHED();
            knn_thr_retry_kernel<K, true><<<148 * 4, ThrCfg<K>::threads, ThrCfg<K>::smem, s>>>(g, v, k, oi, od, vec4, fix, ratio);
            PCC_LAUNCHED();
        } else {
            knn_thr_kernel<K, false><<<nblocks(v.nq, ThrCfg<K>::threads), ThrCfg<K>::threads, ThrCfg<K>::smem, s>>>(g, v, k, oi, od, vec4, fix, ratio);
            PCC_LAUNCHED();
            knn_thr_retry_kernel<K, false><<<148 * 4, ThrCfg<K>::threads, ThrCfg<K>::smem, s>>>(g, v, k, oi, od, vec4, fix, ratio);
            PCC_LAUNCHED();
        }
        h_fb[0] = 0; idx->calib_nq = v.nq;
        PCC_CUDA(cudaMemcpyAsync(h_fb, fix.retry_count, sizeof(unsigned), cudaMemcpyDeviceToHost, s));
    }
    // fork: the wide queries (and a short tied list) on the aux stream, beside the compaction + ring pass on `s`
    PCC_CUDA(cudaEventRecord(idx->ev_fork, s));
    PCC_CUDA(cudaStreamWaitEvent(idx->aux_stream, idx->ev_fork, 0));
    knn_wide_kernel<<<148 * 6, 128, 0, idx->aux_stream>>>(g, v, k, oi, od, fix, fix.wide_list, fix.wide_count, old_fast ? 1 : 0);
    PCC_LAUNCHED();
    PCC_CUDA(cudaEventRecord(idx->ev_join, idx->aux_stream));
    PCC_CUDA(cub::DeviceSelect::Flagged(idx->cub_tmp.p, tmp, cub::CountingInputIterator<uint32_t>(0), fix.ring_flag, fix.ring_list, fix.ring_count, (int)v.nq, s));
    PCC_LAUNCHED();
    knn_rings_kernel<K><<<148 * 16, 128, 0, s>>>(g, v, k, oi, od, vec4, fix);
    PCC_LAUNCHED();
    PCC_CUDA(cudaStreamWaitEvent(s, idx->ev_join, 0));
    knn_wide_kernel<<<148 * 2, 128, 0, s>>>(g, v, k, oi, od, fix, fix.late_list, fix.late_count, 0);      // what the ring pass handed on (rare)
    PCC_LAUNCHED();
    if (old_fast) {                  // the threshold kernel settles its ties in knn_thr_retry_kernel: nothing is listed for the fix-up kernel
        knn_fixup_kernel<K><<<148 * 4, 128, 0, s>>>(g, v, k, oi, od, vec4, fix);
        PCC_LAUNCHED();
    }
    return PCC_OK;
}

}  // namespace pcc

using namespace pcc;

// one batch on one stream; `sync` = wait for the host copies before returning (PCC_HOST only)
static int knn_impl(pcc_index *idx, const void *q, int64_t nq, int stride_bytes, int k, int32_t *out_idx, float *out_d2, int *k_eff, int mem, cudaStream_t s, bool sync) {
    Queries qs;
    PCC_TRY(prepare_queries(idx, q, nq, stride_bytes, mem, s, &qs));
    if (k_eff) *k_eff = (int)std::min<int64_t>(k, idx->n_indexed);
    if (qs.rows == 0) return PCC_OK;
    if (!out_idx || !out_d2) return fail(PCC_ERR_INVALID, "output pointers are NULL");
    int32_t *oi = out_idx; float *od = out_d2;
    const size_t cells = (size_t)qs.rows * k;
    if (mem == PCC_HOST) {
        PCC_TRY(idx->out_i.reserve(cells * 4)); PCC_TRY(idx->out_f.reserve(cells * 4));
        oi = idx->out_i.as<int32_t>(); od = idx->out_f.as<float>();
    }
    if (qs.self && !idx->all_rows_indexed) {   // rows of skipped (non-finite) points stay empty: (-1, +inf)
        PCC_CUDA(cudaMemsetAsync(oi, 0xFF, cells * 4, s));
        fill_f32_kernel<<<nblocks((int64_t)cells, 256), 256, 0, s>>>(od, (int64_t)cells, INFINITY);
        PCC_LAUNCHED();
    }
    const Grid g = idx->grid();
    const QueryView v = view_of(qs);
    const int vec4 = ((((uintptr_t)oi) | ((uintptr_t)od)) & 15) == 0 && (k % 4 == 0);
    KernelTimer timer(idx, s);
    if (qs.nq > 0) {
        // A small batch (the per-point calls of a PCL consumer that only swapped its tree, INTEGRATION.md level 1) is all launch
        // latency: it takes the single-kernel exact path instead of the seven launches of the staged one (k <= 32), or the
        // heap kernel instead of the selection path with its two read-backs (k > 32).
        static const bool exact_env = getenv("PCC_EXACT_ONLY") != nullptr;      // debugging aid: force the ring-expansion path
        const bool exact_only = exact_env || v.nq < (k <= 32 ? kSmallBatch : kSmallBatchBigK);
        static const bool want_stats = getenv("PCC_STATS") != nullptr;
        // warp-owns-a-cell TMA variant: opt-in (PCC_CELL_KERNEL=1).  Measured on B200 it is exact but 1.6-2.8x slower than the
        // per-thread walk even at 80 queries per cell (profiles/r1/cell_kernel_probe.jsonl), so it is never chosen automatically.
        const char *cell_env = getenv("PCC_CELL_KERNEL");
        const bool use_cell = cell_env && atoi(cell_env) != 0;
        FixList fix{nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
        if (k > 1 && k <= 32 && !exact_only) {
            PCC_TRY(idx->misc.reserve((size_t)v.nq * 21 + 512));
            fix.count = idx->misc.as<unsigned>(); fix.ring_count = fix.count + 1; fix.wide_count = fix.count + 30; fix.late_count = fix.count + 31; fix.retry_count = fix.count + 32;
            fix.list = idx->misc.as<uint32_t>() + 64; fix.ring_list = fix.list + v.nq; fix.wide_list = fix.ring_list + v.nq; fix.late_list = fix.wide_list + v.nq; fix.retry_list = fix.late_list + v.nq; fix.ring_flag = (uint8_t *)(fix.retry_list + v.nq);
            if (want_stats) { fix.stats = (unsigned long long *)(idx->misc.as<uint32_t>() + 2); PCC_CUDA(cudaMemsetAsync(fix.stats, 0, 112, s)); }
        }
        if (k == 1) launch_knn_reg<1>(g, v, k, oi, od, vec4, s);
        else if (exact_only && k <= 2) launch_knn_reg<2>(g, v, k, oi, od, vec4, s);
        else if (exact_only && k <= 4) launch_knn_reg<4>(g, v, k, oi, od, vec4, s);
        else if (exact_only && k <= 8) launch_knn_reg<8>(g, v, k, oi, od, vec4, s);
        else if (exact_only && k <= 16) launch_knn_reg<16>(g, v, k, oi, od, vec4, s);
        else if (exact_only && k <= 32) launch_knn_reg<32>(g, v, k, oi, od, vec4, s);
        else if (use_cell && k <= 8) launch_knn_cell<8>(g, v, k, oi, od, vec4, fix, s);
        else if (use_cell && k <= 16) launch_knn_cell<16>(g, v, k, oi, od, vec4, fix, s);
        else if (use_cell && k <= 32) launch_knn_cell<32>(g, v, k, oi, od, vec4, fix, s);
        else if (k <= 4) PCC_TRY(launch_knn_fast<4>(idx, g, v, k, oi, od, vec4, fix, s));
        else if (k <= 8) PCC_TRY(launch_knn_fast<8>(idx, g, v, k, oi, od, vec4, fix, s));
        else if (k <= 16) PCC_TRY(launch_knn_fast<16>(idx, g, v, k, oi, od, vec4, fix, s));
        else if (k <= 32) PCC_TRY(launch_knn_fast<32>(idx, g, v, k, oi, od, vec4, fix, s));
        else if (!exact_only) PCC_TRY(knn_select(idx, qs, k, oi, od, s));      // 32 < k: bracket the k-th distance, then fill + sort rows
        else {
            const int th = heap_threads(k);
            PCC_TRY(set_heap_smem(knn_heap_kernel));
            knn_heap_kernel<<<nblocks(v.nq, th), th, (size_t)k * th * sizeof(nkey_t), s>>>(g, v, k, oi, od);
            PCC_LAUNCHED();
        }
        PCC_CUDA(cudaGetLastError());
    }
    timer.stop();
    if (getenv("PCC_STATS") && k > 1 && k <= 32) {
        unsigned long long h[14];
        cudaMemcpyAsync(h, idx->misc.as<uint32_t>() + 2, 112, cudaMemcpyDeviceToHost, s); cudaStreamSynchronize(s);
        const double q = (double)std::max<unsigned long long>(h[0], 1);
        fprintf(stderr, "[pcc stats] queries=%llu logged/q=%.1f log_overflow=%.5f need_ring2=%.3f fixup=%.5f members/q=%.2f\n",
                h[0], h[1] / q, h[3] / q, h[4] / q, h[5] / q, h[6] / q);
        fprintf(stderr, "[pcc stats] wide queries=%llu steps/q=%.1f final R: <=1 %llu, 2 %llu, 3 %llu, 4-7 %llu, 8-15 %llu, 16+ %llu\n", h[2], h[7] / (double)std::max<unsigned long long>(h[2], 1), h[8], h[9], h[10], h[11], h[12], h[13]);
    }
    if (mem == PCC_HOST) {
        PCC_TRY(copy_out(out_idx, oi, cells * 4, mem, s));
        PCC_TRY(copy_out(out_d2, od, cells * 4, mem, s));
        if (sync) PCC_CUDA(cudaStreamSynchronize(s));
    }
    return PCC_OK;
}

extern "C" {

int pcc_knn(pcc_index *idx, const void *q, int64_t nq, int stride_bytes, int k, int32_t *out_idx, float *out_d2, int *k_eff, int mem, void *stream) {
    PCC_TRY(check_index(idx, stream));
    if (k < 1 || k > PCC_MAX_K) return fail(PCC_ERR_INVALID, "k=%d outside 1..%d", k, PCC_MAX_K);
    cudaStream_t s = (cudaStream_t)stream;
    // Large host batches: two-slot pipeline, 1 Mi queries per chunk (16 MB in, k x 8 MB out), so the device->host copy of
    // chunk i overlaps the search of chunk i+1 and the host->device copy of chunk i+2 (PCIe is full duplex).
    static const int64_t kChunk = getenv("PCC_PIPE_CHUNK_LOG2") ? (1ll << std::max(16, std::min(24, atoi(getenv("PCC_PIPE_CHUNK_LOG2"))))) : (1ll << 20);      // measured on B200 (profiles/r2/e2e_chunk_probe.txt): 2^20 wins
    if (mem == PCC_HOST && q && nq >= 2 * kChunk && !idx->timing && stride_bytes >= 12 && !(stride_bytes & 3)) {
        if (!out_idx || !out_d2) return fail(PCC_ERR_INVALID, "output pointers are NULL");
        if (!idx->shadow) {
            idx->shadow = new pcc_index();
            idx->shadow->device = idx->device;
            idx->shadow->grid_owner = idx;
            PCC_CUDA(cudaMallocHost(&idx->shadow->h_pinned, 4096));
            for (int i = 0; i < 2; ++i) PCC_CUDA(cudaStreamCreateWithFlags(&idx->pipe_stream[i], cudaStreamNonBlocking));
        }
        pcc_index *sh = idx->shadow;
        sh->built = true; sh->n_input = idx->n_input; sh->n_indexed = idx->n_indexed; sh->gh = idx->gh;
        PCC_CUDA(cudaStreamSynchronize(s));                      // work queued on the caller's stream comes first
        int rc = PCC_OK;
        int64_t c0 = 0;
        for (int i = 0; c0 < nq && rc == PCC_OK; ++i, c0 += kChunk) {
            const int64_t n = std::min(kChunk, nq - c0);
            rc = knn_impl((i & 1) ? sh : idx, (const uint8_t *)q + c0 * stride_bytes, n, stride_bytes, k, out_idx + c0 * k, out_d2 + c0 * k, k_eff, PCC_HOST, idx->pipe_stream[i & 1], false);
        }
        cudaStreamSynchronize(idx->pipe_stream[0]);
        cudaStreamSynchronize(idx->pipe_stream[1]);
        return rc;
    }
    return knn_impl(idx, q, nq, stride_bytes, k, out_idx, out_d2, k_eff, mem, s, true);
}

int pcc_knn_mean_dist(pcc_index *idx, const void *q, int64_t nq, int stride_bytes, int mean_k, float *out_mean, int mem, void *stream) {
    PCC_TRY(check_index(idx, stream));
    if (mean_k < 1 || mean_k + 1 > PCC_MAX_K) return fail(PCC_ERR_INVALID, "mean_k=%d outside 1..%d", mean_k, PCC_MAX_K - 1);
    cudaStream_t s = (cudaStream_t)stream;
    Queries qs;
    PCC_TRY(prepare_queries(idx, q, nq, stride_bytes, mem, s, &qs));
    if (qs.rows == 0) return PCC_OK;
    if (!out_mean) return fail(PCC_ERR_INVALID, "output pointer is NULL");
    float *od = nullptr;
    PCC_TRY(output_rows(idx, out_mean, (size_t)qs.rows * 4, mem, &od));
    if (qs.self && !idx->all_rows_indexed) PCC_CUDA(cudaMemsetAsync(od, 0, (size_t)qs.rows * 4, s));
    const Grid g = idx->grid();
    const QueryView v = view_of(qs);
    const int need = mean_k + 1;
    KernelTimer timer(idx, s);
    if (qs.nq > 0) {
        const unsigned nb = nblocks(v.nq, 128);
#define PCC_MD(KK)                                                                            \
    if (need == KK) mean_dist_reg_kernel<KK, true><<<nb, 128, 0, s>>>(g, v, mean_k, od);          \
    else mean_dist_reg_kernel<KK, false><<<nb, 128, 0, s>>>(g, v, mean_k, od)
        if (need <= 2) { PCC_MD(2); }
        else if (need <= 5) { PCC_MD(5); }
        else if (need <= 9) { PCC_MD(9); }
        else if (need <= 17) { PCC_MD(17); }
        else if (need <= 33) { PCC_MD(33); }
        else if (need <= 51) { PCC_MD(51); }
#undef PCC_MD
        else {
            const int th = heap_threads(need);
            PCC_TRY(set_heap_smem(mean_dist_heap_kernel));
            mean_dist_heap_kernel<<<nblocks(v.nq, th), th, (size_t)need * th * sizeof(nkey_t), s>>>(g, v, mean_k, od);
        }
        PCC_LAUNCHED();
        PCC_CUDA(cudaGetLastError());
    }
    timer.stop();
    return deliver_rows(out_mean, od, (size_t)qs.rows * 4, mem, s);
}

int pcc_normals_knn(pcc_index *idx, const void *q, int64_t nq, int stride_bytes, int k, const float viewpoint[3], float *out, int mem, void *stream) {
    PCC_TRY(check_index(idx, stream));
    if (k < 1 || k > PCC_MAX_K) return fail(PCC_ERR_INVALID, "k=%d outside 1..%d", k, PCC_MAX_K);
    cudaStream_t s = (cudaStream_t)stream;
    Queries qs;
    PCC_TRY(prepare_queries(idx, q, nq, stride_bytes, mem, s, &qs));
    if (qs.rows == 0) return PCC_OK;
    if (!out) return fail(PCC_ERR_INVALID, "output pointer is NULL");
    if (!idx->inv_valid) PCC_TRY(rebuild_inverse(idx, s));
    float4 *od = nullptr;
    PCC_TRY(output_rows(idx, (float4 *)out, (size_t)qs.rows * 16, mem, &od));
    if (qs.self && !idx->all_rows_indexed) PCC_CUDA(cudaMemsetAsync(od, 0xFF, (size_t)qs.rows * 16, s));   // 0xFFFFFFFF = NaN
    const float vx = viewpoint ? viewpoint[0] : 0.f, vy = viewpoint ? viewpoint[1] : 0.f, vz = viewpoint ? viewpoint[2] : 0.f;
    const Grid g = idx->grid();
    const QueryView v = view_of(qs);
    const uint32_t *inv = idx->inv_pos.as<uint32_t>();
    KernelTimer timer(idx, s);
    if (qs.nq > 0) {
        const unsigned nb = nblocks(v.nq, 128);
        if (k <= 8) normals_knn_reg_kernel<8><<<nb, 128, 0, s>>>(g, v, k, inv, vx, vy, vz, od);
        else if (k <= 16) normals_knn_reg_kernel<16><<<nb, 128, 0, s>>>(g, v, k, inv, vx, vy, vz, od);
        else if (k <= 32) normals_knn_reg_kernel<32><<<nb, 128, 0, s>>>(g, v, k, inv, vx, vy, vz, od);
        else {
            const int th = heap_threads(k);
            PCC_TRY(set_heap_smem(normals_knn_heap_kernel));
            normals_knn_heap_kernel<<<nblocks(v.nq, th), th, (size_t)k * th * sizeof(nkey_t), s>>>(g, v, k, inv, vx, vy, vz, od);
        }
        PCC_LAUNCHED();
        PCC_CUDA(cudaGetLastError());
    }
    timer.stop();
    return deliver_rows(out, od, (size_t)qs.rows * 16, mem, s);
}

// src working copy lives in idx->stage4-independent buffer `parent` is reserved for clustering; ICP uses qbuf-sized `keys64b`
int pcc_icp_step(pcc_index *idx, void *src_inout, int64_t ns, int stride_bytes, const float *T_apply, double sums[16], int64_t *count,
                 int32_t *corr_idx, float *corr_d2, int mem, void *stream) {
    PCC_TRY(check_index(idx, stream));
    if (ns < 0 || stride_bytes < 12 || (stride_bytes & 3)) return fail(PCC_ERR_INVALID, "bad source cloud (ns=%lld stride=%d)", (long long)ns, stride_bytes);
    if (!sums || !count) return fail(PCC_ERR_INVALID, "sums / count are NULL");
    cudaStream_t s = (cudaStream_t)stream;
    for (int i = 0; i < 16; ++i) sums[i] = 0;
    *count = 0;
    if (ns == 0) return PCC_OK;
    // working float4 copy + cell-sorted processing order of the (untransformed) source
    Queries qs;
    PCC_TRY(prepare_queries(idx, src_inout, ns, stride_bytes, mem, s, &qs));
    float4 *work = idx->qbuf.as<float4>();
    Mat34 T; int apply = 0;
    if (T_apply) { memcpy(T.m, T_apply, sizeof(T.m)); apply = 1; } else memset(&T, 0, sizeof(T));
    const unsigned nb = nblocks(ns, kIcpThreads);
    PCC_TRY(idx->keys64b.reserve(((size_t)nb * 17 + 32) * sizeof(double)));
    double *partials = idx->keys64b.as<double>();
    double *d_out = partials + (size_t)nb * 17;
    int32_t *ci = corr_idx; float *cd = corr_d2;
    if (mem == PCC_HOST) {
        if (corr_idx) { PCC_TRY(idx->out_i.reserve((size_t)ns * 4)); ci = idx->out_i.as<int32_t>(); }
        if (corr_d2) { PCC_TRY(idx->out_f.reserve((size_t)ns * 4)); cd = idx->out_f.as<float>(); }
    }
    KernelTimer timer(idx, s);
    static const bool no_prior = getenv("PCC_ICP_NO_PRIOR") != nullptr;      // measurement aid
    uint32_t *prior = nullptr;
    if (!no_prior) {
        const bool fresh = idx->icp_prior_n != ns;        // first pass over this source cloud (or a new index): no bounds yet
        if (fresh) {
            PCC_TRY(idx->icp_prior.reserve((size_t)std::max<int64_t>(ns, 1) * 4));
            PCC_CUDA(cudaMemsetAsync(idx->icp_prior.p, 0xFF, (size_t)std::max<int64_t>(ns, 1) * 4, s));
            idx->icp_prior_n = ns;
        }
        prior = idx->icp_prior.as<uint32_t>();
    }
    icp_step_kernel<<<nb, kIcpThreads, 0, s>>>(idx->grid(), work, qs.order, ns, T, apply, partials, ci, cd, prior);
    PCC_LAUNCHED();
    icp_reduce_kernel<<<17, 256, 0, s>>>(partials, nb, d_out);
    PCC_LAUNCHED();
    if (idx->icp_allreduce) PCC_TRY(comm_allreduce_f64(idx, d_out, 17, s));      // sharded source cloud: the sums of every rank's shard (NCCL)
    PCC_CUDA(cudaGetLastError());
    timer.stop();
    double *h = (double *)idx->h_pinned;
    PCC_CUDA(cudaMemcpyAsync(h, d_out, 17 * sizeof(double), cudaMemcpyDeviceToHost, s));
    if (apply) {   // hand the moved points back in the caller's layout
        if (mem == PCC_DEVICE) {
            icp_store_kernel<<<nblocks(ns, 256), 256, 0, s>>>(work, ns, (uint8_t *)src_inout, stride_bytes);
            PCC_LAUNCHED();
        } else {
            icp_store_kernel<<<nblocks(ns, 256), 256, 0, s>>>(work, ns, idx->raw.as<uint8_t>(), stride_bytes);
            PCC_LAUNCHED();
            PCC_CUDA(cudaMemcpyAsync(src_inout, idx->raw.p, (size_t)ns * stride_bytes, cudaMemcpyDeviceToHost, s));
        }
    }
    if (mem == PCC_HOST) {
        if (corr_idx) PCC_TRY(copy_out(corr_idx, ci, (size_t)ns * 4, mem, s));
        if (corr_d2) PCC_TRY(copy_out(corr_d2, cd, (size_t)ns * 4, mem, s));
    }
    PCC_CUDA(cudaStreamSynchronize(s));
    for (int i = 0; i < 16; ++i) sums[i] = h[i];
    *count = (int64_t)llround(h[16]);
    return PCC_OK;
}

}  // extern "C"
