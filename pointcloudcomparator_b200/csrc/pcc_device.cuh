// pcc_device.cuh -- device-side building blocks shared by every query kernel.
//
// Data layout in HBM (see DESIGN.md): the indexed cloud is ONE float4 array sorted by grid cell
// (x, y, z, original index bit-cast into .w) plus ONE dense uint32 cell_start table in row-major
// (z, y, x) order, so the cells x-R..x+R of a row are one contiguous run of points: a 3x3x3 stencil
// is 9 coalesced float4 runs, not 27 cell lookups.
#pragma once
#include <type_traits>
#include <cuda_runtime.h>
#include <stdint.h>
#include <math_constants.h>

namespace pcc {

struct Grid {
    const float4 *pts;            // sorted by cell; .w = original index (int bits)
    const uint32_t *cell_start;   // n_cells + 1
    const uint32_t *occ;          // n_cells bits (+ one padding word): cell holds at least one point
    const uint2 *occ2;            // per 32 cells: {the occ word, number of non-empty cells before it}
    const uint32_t *cstart;       // first sorted position of every NON-EMPTY cell, in cell order (+ one entry = n)
    float ox, oy, oz;             // origin = bbox min
    float inv_cell, cell;
    int nx, ny, nz;
    uint32_t n;                   // indexed points
};

#ifndef PCC_COMPACT_TABLE
#define PCC_COMPACT_TABLE 0
#endif
// first sorted position of cell c (= of the next non-empty cell when c is empty; c = n_cells gives n).  Dense: one load from the
// n_cells-entry table.  Compact: the rank of c among the non-empty cells from the bitmap word + its prefix, then one load from
// the table of non-empty cells -- two dependent loads, but 19 MB of tables instead of 225 MB at the headline size.
__device__ __forceinline__ uint32_t cell_begin(const Grid &g, size_t c) {
#if PCC_COMPACT_TABLE
    const uint2 w = __ldg(g.occ2 + (c >> 5));
    return __ldg(g.cstart + w.y + __popc(w.x & ((1u << (c & 31)) - 1u)));
#else
    return __ldg(g.cell_start + c);
#endif
}

// Squared L2 exactly as FLANN L2_Simple evaluates it in fp32: ((dx*dx + dy*dy) + dz*dz), no FMA.
__device__ __forceinline__ float dist2(float qx, float qy, float qz, float px, float py, float pz) {
    float dx = __fsub_rn(qx, px), dy = __fsub_rn(qy, py), dz = __fsub_rn(qz, pz);
    return __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
}
// continuous grid coordinate; the SAME expression bins points at build time and queries at search time
__device__ __forceinline__ float grid_u(float x, float o, float inv) { return __fmul_rn(__fsub_rn(x, o), inv); }
__device__ __forceinline__ int grid_c(float u, int n) { return (int)fminf(fmaxf(floorf(u), 0.f), (float)(n - 1)); }
__device__ __forceinline__ bool finite3(float x, float y, float z) { return isfinite(x) && isfinite(y) && isfinite(z); }

// a prepared query batch as the kernels see it (pcc_internal.h Queries)
struct QueryView { const float4 *q; const uint32_t *order; int64_t nq; bool self; };
// thread t (< v.nq) -> query coordinates; returns the output row.  Self mode: sorted point t, row = its original index.
__device__ __forceinline__ int64_t rows_query(const Grid &g, const QueryView &v, int64_t t, float &x, float &y, float &z) {
    if (v.self) { float4 p = __ldg(g.pts + t); x = p.x; y = p.y; z = p.z; return __float_as_int(p.w); }
    uint32_t qi = v.order ? __ldg(v.order + t) : (uint32_t)t; float4 p = __ldg(v.q + qi); x = p.x; y = p.y; z = p.z; return qi;
}

struct QueryCell {
    float ux, uy, uz;
    int cx, cy, cz;
};
__device__ __forceinline__ QueryCell locate(const Grid &g, float x, float y, float z) {
    QueryCell c;
    c.ux = grid_u(x, g.ox, g.inv_cell); c.uy = grid_u(y, g.oy, g.inv_cell); c.uz = grid_u(z, g.oz, g.inv_cell);
    c.cx = grid_c(c.ux, g.nx); c.cy = grid_c(c.uy, g.ny); c.cz = grid_c(c.uz, g.nz);
    return c;
}
// Squared world distance below which every indexed point is guaranteed to lie inside the block of
// Chebyshev radius R around the query's cell (+inf once the block covers the whole grid).
// Margins: 2e-3 cells absolute + 1e-5 relative cover the fp32 rounding of grid_u (dims are capped
// at 2048 cells per axis, so |u| rounding <= 2048 * 2^-23 = 2.5e-4) and of cell = 1 / inv_cell.
__device__ __forceinline__ float covered_d2(const Grid &g, const QueryCell &c, int R) {
    float b = CUDART_INF_F;
    if (c.cx - R > 0) b = fminf(b, c.ux - (float)(c.cx - R));
    if (c.cx + R < g.nx - 1) b = fminf(b, (float)(c.cx + R + 1) - c.ux);
    if (c.cy - R > 0) b = fminf(b, c.uy - (float)(c.cy - R));
    if (c.cy + R < g.ny - 1) b = fminf(b, (float)(c.cy + R + 1) - c.uy);
    if (c.cz - R > 0) b = fminf(b, c.uz - (float)(c.cz - R));
    if (c.cz + R < g.nz - 1) b = fminf(b, (float)(c.cz + R + 1) - c.uz);
    if (b == CUDART_INF_F) return b;
    b = (b * (1.0f - 1e-5f) - 2e-3f) * g.cell;
    return b > 0.f ? b * b : 0.f;
}

// Visit every indexed point in the cells with Chebyshev ring index in (Rin, Rout] around (cx,cy,cz)
// (Rin = -1 visits the whole block).  f(pos, float4 point).
template <class F>
__device__ __forceinline__ void scan_shell(const Grid &g, const QueryCell &c, int Rin, int Rout, F &&f) {
    const int z0 = max(c.cz - Rout, 0), z1 = min(c.cz + Rout, g.nz - 1);
    const int y0 = max(c.cy - Rout, 0), y1 = min(c.cy + Rout, g.ny - 1);
    const int xa = max(c.cx - Rout, 0), xb = min(c.cx + Rout, g.nx - 1);
    for (int z = z0; z <= z1; ++z) {
        for (int y = y0; y <= y1; ++y) {
            const uint32_t *row = g.cell_start + ((size_t)z * g.ny + y) * g.nx;
            const bool outer = max(abs(z - c.cz), abs(y - c.cy)) > Rin;
            if (outer) {
                uint32_t j = __ldg(row + xa), e = __ldg(row + xb + 1);
                for (; j < e; ++j) f(j, __ldg(g.pts + j));
            } else {
                int xl = c.cx - Rin - 1;             // left strip [xa, xl]
                if (xl >= xa) { uint32_t j = __ldg(row + xa), e = __ldg(row + xl + 1); for (; j < e; ++j) f(j, __ldg(g.pts + j)); }
                int xr = c.cx + Rin + 1;             // right strip [xr, xb]
                if (xr <= xb) { uint32_t j = __ldg(row + xr), e = __ldg(row + xb + 1); for (; j < e; ++j) f(j, __ldg(g.pts + j)); }
            }
        }
    }
}

// world d2 -> cell units, rounded up (used as the clipping radius of scan_clipped)
__device__ __forceinline__ float to_cell_units(const Grid &g, float d2) { return d2 == CUDART_INF_F ? d2 : d2 * g.inv_cell * g.inv_cell * (1.0f + 4e-5f); }

// Next block radius of an exact search whose k-th distance is not yet covered by radius R.  While fewer than k points
// have been seen the block doubles (a shell row costs ONE run lookup whatever its x-length, so a pass is O(R^2), not
// O(R^3)); once k points are known the block jumps straight to the radius that covers their ball.
__device__ __forceinline__ int next_ring(const Grid &g, int R, float kth_d2) {
    const int cap = max(g.nx, max(g.ny, g.nz));
    if (kth_d2 == CUDART_INF_F) return min(2 * R + 1, max(cap, R + 1));
    const float need = sqrtf(to_cell_units(g, kth_d2)) + 0.01f;
    return max(R + 1, (int)fminf(ceilf(need), (float)cap));
}

// one contiguous float4 run: points are fetched four at a time (independent 16-byte loads in flight together) and
// then processed in order, which hides most of the L1/L2 latency a one-at-a-time walk exposes
// A visitor derived from group_visitor takes the four points of a full group at once (f.four(j, p0, p1, p2, p3)) so that it can
// test the group with one branch; f(j, p) still serves the tail of a run.
struct group_visitor {};
template <class F>
__device__ __forceinline__ void walk_run(const Grid &g, uint32_t j, uint32_t e, F &&f) {
    for (; j + 4 <= e; j += 4) {
        const float4 p0 = __ldg(g.pts + j), p1 = __ldg(g.pts + j + 1), p2 = __ldg(g.pts + j + 2), p3 = __ldg(g.pts + j + 3);
#ifndef PCC_GROUP_VISIT
#define PCC_GROUP_VISIT 1
#endif
        if constexpr (PCC_GROUP_VISIT && std::is_base_of<group_visitor, typename std::remove_reference<F>::type>::value) f.four(j, p0, p1, p2, p3);
        else { f(j, p0); f(j + 1, p1); f(j + 2, p2); f(j + 3, p3); }
    }
    if (j < e) {
        const float4 p0 = __ldg(g.pts + j);
        const float4 p1 = __ldg(g.pts + min(j + 1, e - 1)), p2 = __ldg(g.pts + min(j + 2, e - 1));
        f(j, p0);
        if (j + 1 < e) f(j + 1, p1);
        if (j + 2 < e) f(j + 2, p2);
    }
}

// scan_shell restricted to the ball of squared radius tau_u (CELL units, +inf = no restriction) around the query:
// a row is skipped when its (y, z) gap alone exceeds the ball and the x-range of a kept row is cut to the cells the
// ball can reach.  Every test is conservative (2e-3 cell slack + the 4e-5 relative slack of to_cell_units, the same
// rounding budget as covered_d2), so no point with d2 <= tau is ever skipped.  This is what makes ring >= 2 cheap:
// a query that misses the 3x3x3 guarantee by a little only touches the one or two cells the ball pokes into.
// Rows are visited centre-out (offsets 0, -1, +1, -2, +2, ...): the nearest rows come first, so the running k-th distance
// tightens early and fewer later candidates pass the insertion guard.
__device__ __forceinline__ int centre_out(int a) { return (a & 1) ? -((a + 1) >> 1) : (a >> 1); }
struct RowRuns { uint32_t j1, e1, j2, e2; };
// does any of the cells [xa, xb] of the row whose first cell has linear index `base` hold a point?  One bit per cell
// (Grid::occ); ranges longer than 32 cells are not tested.  Rings beyond the first mostly verify EMPTY cells, and the
// bitmap answers that from L1/L2 where the dense cell_start table (32x larger) would go to DRAM.
__device__ __forceinline__ bool row_occupied(const Grid &g, size_t base, int xa, int xb) {
    if (xb - xa >= 32) return true;
    const size_t b = base + (size_t)xa;
#if PCC_COMPACT_TABLE
    const uint32_t w0 = __ldg(&g.occ2[b >> 5].x), w1 = __ldg(&g.occ2[(b >> 5) + 1].x);
#else
    const uint32_t w0 = __ldg(g.occ + (b >> 5)), w1 = __ldg(g.occ + (b >> 5) + 1);
#endif
    const uint32_t bits = __funnelshift_r(w0, w1, (uint32_t)(b & 31));
    const int len = xb - xa + 1;
    return (bits & (len == 32 ? 0xffffffffu : ((1u << len) - 1u))) != 0u;
}
// run bounds of row (az, ay) of the block (centre-out numbering); empty runs (j == e) for skipped rows
__device__ __forceinline__ RowRuns row_runs(const Grid &g, const QueryCell &c, int Rin, int Rout, float tau_u, int az, int ay) {
    RowRuns r; r.j1 = r.e1 = r.j2 = r.e2 = 0;
    const int dz = centre_out(az), z = c.cz + dz, dy = centre_out(ay), y = c.cy + dy;
    if (z < 0 || z >= g.nz || y < 0 || y >= g.ny) return r;
    const float gz = fmaxf(fmaxf((float)z - c.uz, c.uz - (float)(z + 1)) - 2e-3f, 0.f);
    const float gy = fmaxf(fmaxf((float)y - c.uy, c.uy - (float)(y + 1)) - 2e-3f, 0.f);
    const float D = gy * gy + gz * gz;
    if (D > tau_u) return r;
    int xlo = c.cx - Rout, xhi = c.cx + Rout;
    if (tau_u < CUDART_INF_F) {
        const float w = sqrtf(tau_u - D) + 2e-3f;
        xlo = max(xlo, (int)floorf(c.ux - w)); xhi = min(xhi, (int)floorf(c.ux + w));
    }
    xlo = max(xlo, 0); xhi = min(xhi, g.nx - 1);
    const size_t base = ((size_t)z * g.ny + y) * g.nx;
    const bool probe = Rin >= 0;                     // first pass (whole block): the table rows are hot, read them directly
    if (max(abs(dz), abs(dy)) > Rin) {
        if (xlo <= xhi && (!probe || row_occupied(g, base, xlo, xhi))) { r.j1 = cell_begin(g, base + xlo); r.e1 = cell_begin(g, base + xhi + 1); }
    } else {
        const int xl = min(xhi, c.cx - Rin - 1);     // left strip [xlo, xl]
        if (xlo <= xl && row_occupied(g, base, xlo, xl)) { r.j1 = cell_begin(g, base + xlo); r.e1 = cell_begin(g, base + xl + 1); }
        const int xr = max(xlo, c.cx + Rin + 1);     // right strip [xr, xhi]
        if (xr <= xhi && row_occupied(g, base, xr, xhi)) { r.j2 = cell_begin(g, base + xr); r.e2 = cell_begin(g, base + xhi + 1); }
    }
    return r;
}
// The row loop is software-pipelined: the cell_start loads of row i+1 are issued before row i is walked, so the
// dependent load chain (table -> points) of the next row overlaps the arithmetic of the current one.
// The clipping ball is re-read before every row (`tau_now()` returns the current squared radius in cell units).  It pays when a
// pass is large: a far query (ICP's first iterations, outliers) doubles its block until it sees the first point, and from that
// row on the rest of the SAME pass is clipped to the ball of the best distance so far instead of scanning the whole block.
// (The bounds of row i+1 are fetched before row i is walked, so a row is clipped with the radius known one row earlier --
// conservative, never wrong.)  Ending the row / plane loops at the last row the ball reaches (instead of rejecting the rows
// beyond it one by one) was measured on the 10 M ICP pair and is SLOWER (102 vs 92 ms): a caller with a bound already asks for
// the block that just covers its ball, so few rows lie beyond it, and the extra loop state costs every row.
template <class T, class F>
__device__ __forceinline__ void scan_progressive(const Grid &g, const QueryCell &c, int Rin, int Rout, T &&tau_now, F &&f) {
    const int n1 = 2 * Rout + 1;
    int az = 0, ay = 0;
    RowRuns nxt = row_runs(g, c, Rin, Rout, tau_now(), 0, 0);
    for (;;) {
        const RowRuns cur = nxt;
        if (++ay == n1) { ay = 0; ++az; }
        const bool more = az < n1;
        if (more) nxt = row_runs(g, c, Rin, Rout, tau_now(), az, ay);
        walk_run(g, cur.j1, cur.e1, f);
        walk_run(g, cur.j2, cur.e2, f);
        if (!more) break;
    }
}
// the same walk with a fixed ball
template <class F>
__device__ __forceinline__ void scan_clipped(const Grid &g, const QueryCell &c, int Rin, int Rout, float tau_u, F &&f) {
    scan_progressive(g, c, Rin, Rout, [&]() { return tau_u; }, f);
}

// Nearest point so far in the canonical (d2, original index) order.  A full group of four candidates is tested with ONE branch
// (min of the four against the best): after the first few points almost no group improves the best, so a candidate costs its
// distance and a quarter of a compare instead of a 64-bit compare + five selects (15 % of the pass's instructions before).
struct Nearest1 : group_visitor {
    float x, y, z, bd; uint32_t bidx, bpos;
    __device__ __forceinline__ void init(float qx, float qy, float qz) { x = qx; y = qy; z = qz; bd = CUDART_INF_F; bidx = 0xFFFFFFFFu; bpos = 0; }
    __device__ __forceinline__ bool found() const { return bidx != 0xFFFFFFFFu; }
    __device__ __forceinline__ void take(uint32_t pos, const float4 &r, float d2) {          // given d2 <= bd
        const uint32_t ri = __float_as_uint(r.w);
        if (d2 < bd || ri < bidx) { bd = d2; bidx = ri; bpos = pos; }
    }
    __device__ __forceinline__ void operator()(uint32_t pos, const float4 &r) { const float d2 = dist2(x, y, z, r.x, r.y, r.z); if (d2 <= bd) take(pos, r, d2); }
    __device__ __forceinline__ void four(uint32_t j, const float4 &p0, const float4 &p1, const float4 &p2, const float4 &p3) {
        const float d0 = dist2(x, y, z, p0.x, p0.y, p0.z), d1 = dist2(x, y, z, p1.x, p1.y, p1.z), d2 = dist2(x, y, z, p2.x, p2.y, p2.z), d3 = dist2(x, y, z, p3.x, p3.y, p3.z);
        if (fminf(fminf(d0, d1), fminf(d2, d3)) <= bd) {
            if (d0 <= bd) take(j, p0, d0);
            if (d1 <= bd) take(j + 1, p1, d1);
            if (d2 <= bd) take(j + 2, p2, d2);
            if (d3 <= bd) take(j + 3, p3, d3);
        }
    }
};
// exact 1-NN driver: one pass over the block of radius R (the caller's bound, if any, already sits in `nn`), then shells until the
// best distance is inside the covered radius
__device__ __forceinline__ void nearest1_search(const Grid &g, const QueryCell &c, int R, Nearest1 &nn) {
    int Rin = -1;
    for (;;) {
        scan_progressive(g, c, Rin, R, [&]() { return to_cell_units(g, nn.bd); }, nn);
        const float cov = covered_d2(g, c, R);
        if (cov == CUDART_INF_F) break;
        if (nn.found() && nn.bd < cov) break;
        Rin = R; R = next_ring(g, R, nn.bd);
    }
}

// ---------------------------------------------------------------------------------------------
// top-k containers.  Entries are 64-bit keys (fp32 d2 bits << 32 | payload): d2 >= +0 so the
// unsigned order of the bits is the numeric order, and one 64-bit compare gives the canonical
// (d2, original index) tie rule.  Empty slots hold ~0 (decodes to idx -1, d2 +inf on output).
typedef unsigned long long nkey_t;
#define PCC_EMPTY_KEY 0xFFFFFFFFFFFFFFFFull
__device__ __forceinline__ nkey_t make_key(float d2, uint32_t payload) { return ((nkey_t)__float_as_uint(d2) << 32) | payload; }
__device__ __forceinline__ float key_d2(nkey_t k) { return k == PCC_EMPTY_KEY ? CUDART_INF_F : __uint_as_float((uint32_t)(k >> 32)); }
__device__ __forceinline__ int32_t key_idx(nkey_t k) { return k == PCC_EMPTY_KEY ? -1 : (int32_t)(uint32_t)k; }

// k <= K entries kept sorted in registers (all indexing is compile-time after unrolling)
template <int K>
struct RegList {
    nkey_t key[K];
    __device__ __forceinline__ void init() {
#pragma unroll
        for (int i = 0; i < K; ++i) key[i] = PCC_EMPTY_KEY;
    }
    __device__ __forceinline__ void offer(nkey_t c) {
        if (c < key[K - 1]) {
#pragma unroll
            for (int i = 0; i < K; ++i) { const nkey_t t = key[i]; const bool lt = c < t; key[i] = lt ? c : t; c = lt ? t : c; }
        }
    }
    __device__ __forceinline__ nkey_t at(int j) const {   // j runtime, resolved with selects
        nkey_t r = key[0];
#pragma unroll
        for (int i = 1; i < K; ++i) r = (i == j) ? key[i] : r;
        return r;
    }
    __device__ __forceinline__ void finish() {}
};

// k entries as a binary max-heap in shared memory, slot-major ([slot][thread]) so that the 32 lanes
// of a warp always hit 32 different banks whatever slot each lane is at.  Used for 32 < k <= PCC_MAX_K.
struct HeapList {
    nkey_t *h; int stride; int k; int cnt;
    __device__ __forceinline__ nkey_t &a(int i) { return h[(size_t)i * stride]; }
    __device__ __forceinline__ void init(nkey_t *base, int stride_, int k_) { h = base; stride = stride_; k = k_; cnt = 0; }
    __device__ __forceinline__ void offer(nkey_t c) {
        if (cnt < k) {                       // sift up
            int i = cnt++;
            while (i > 0) { int p = (i - 1) >> 1; nkey_t pv = a(p); if (!(pv < c)) break; a(i) = pv; i = p; }
            a(i) = c;
        } else if (c < a(0)) {               // replace the root, sift down
            sift_down(c, cnt);
        }
    }
    __device__ __forceinline__ void sift_down(nkey_t c, int n) {
        int i = 0;
        for (;;) {
            int l = 2 * i + 1; if (l >= n) break;
            nkey_t lv = a(l); int m = l;
            if (l + 1 < n) { nkey_t rv = a(l + 1); if (lv < rv) { lv = rv; m = l + 1; } }
            if (!(c < lv)) break;
            a(i) = lv; i = m;
        }
        a(i) = c;
    }
    __device__ __forceinline__ bool full() const { return cnt == k; }
    __device__ __forceinline__ nkey_t worst() { return cnt == k ? a(0) : PCC_EMPTY_KEY; }
    // heap -> ascending order in slots [0, cnt); slots [cnt, k) = empty
    __device__ __forceinline__ void finish() {
        for (int n = cnt - 1; n > 0; --n) { nkey_t last = a(n); a(n) = a(0); sift_down(last, n); }
        for (int i = cnt; i < k; ++i) a(i) = PCC_EMPTY_KEY;
    }
    __device__ __forceinline__ nkey_t at(int j) { return a(j); }
};

// distances only (no payload): k smallest d2 kept sorted in registers with min/max only.
template <int K>
struct RegDist {
    float d[K];
    __device__ __forceinline__ void init() {
#pragma unroll
        for (int i = 0; i < K; ++i) d[i] = CUDART_INF_F;
    }
    __device__ __forceinline__ void insert(float c) {          // unguarded: a no-op when c >= d[K-1]
#pragma unroll
        for (int i = K - 1; i > 0; --i) d[i] = fminf(d[i], fmaxf(d[i - 1], c));
        d[0] = fminf(d[0], c);
    }
    __device__ __forceinline__ void offer(float c) { if (c < d[K - 1]) insert(c); }
    __device__ __forceinline__ float at(int j) const {
        float r = d[0];
#pragma unroll
        for (int i = 1; i < K; ++i) r = (i == j) ? d[i] : r;
        return r;
    }
};

// -------------------------------------------------------------------------------------------------
// pcl::eigen33 smallest eigenpair + curvature, fp32, same operation order as the PCL 1.7 source the
// oracle restates (common/impl/eigen.hpp [up]); compiled with -fmad=false so nothing is contracted.
__device__ __forceinline__ void roots2(float b, float c, float *r) {
    r[0] = 0.f;
    float d = (float)((double)b * (double)b - 4.0 * (double)c);
    if (d < 0.0f) d = 0.0f;
    float sd = sqrtf(d);
    r[2] = 0.5f * (b + sd);
    r[1] = 0.5f * (b - sd);
}
__device__ __forceinline__ void roots3(const float *m, float *r) {
    float c0 = m[0] * m[4] * m[8] + 2.0f * m[1] * m[2] * m[5] - m[0] * m[5] * m[5] - m[4] * m[2] * m[2] - m[8] * m[1] * m[1];
    float c1 = m[0] * m[4] - m[1] * m[1] + m[0] * m[8] - m[2] * m[2] + m[4] * m[8] - m[5] * m[5];
    float c2 = m[0] + m[4] + m[8];
    if (fabsf(c0) < 1.1920929e-07f) { roots2(c2, c1, r); return; }
    const float s_inv3 = (float)(1.0 / 3.0);
    const float s_sqrt3 = sqrtf(3.0f);
    float c2_over_3 = c2 * s_inv3;
    float a_over_3 = (c1 - c2 * c2_over_3) * s_inv3;
    if (a_over_3 > 0.f) a_over_3 = 0.f;
    float half_b = 0.5f * (c0 + c2_over_3 * (2.0f * c2_over_3 * c2_over_3 - c1));
    float q = half_b * half_b + a_over_3 * a_over_3 * a_over_3;
    if (q > 0.f) q = 0.f;
    float rho = sqrtf(-a_over_3);
    float theta = atan2f(sqrtf(-q), half_b) * s_inv3;
    float cos_theta = cosf(theta), sin_theta = sinf(theta);
    r[0] = c2_over_3 + 2.0f * rho * cos_theta;
    r[1] = c2_over_3 - rho * (cos_theta + s_sqrt3 * sin_theta);
    r[2] = c2_over_3 - rho * (cos_theta - s_sqrt3 * sin_theta);
    float t;
    if (r[0] >= r[1]) { t = r[0]; r[0] = r[1]; r[1] = t; }
    if (r[1] >= r[2]) { t = r[1]; r[1] = r[2]; r[2] = t; if (r[0] >= r[1]) { t = r[0]; r[0] = r[1]; r[1] = t; } }
    if (r[0] <= 0.f) roots2(c2, c1, r);
}
// accu[9] = sums in neighbour order (xx xy xz yy yz zz x y z), cnt neighbours -> normal + curvature, flipped to viewpoint
__device__ __forceinline__ float4 normal_from_accu(float *a, int cnt, float px, float py, float pz, float vx, float vy, float vz) {
    const float qnan = CUDART_NAN_F;
    if (cnt < 3) return make_float4(qnan, qnan, qnan, qnan);
    const float fn = (float)cnt;
#pragma unroll
    for (int i = 0; i < 9; ++i) a[i] = __fdiv_rn(a[i], fn);
    float cov[9];
    cov[0] = a[0] - a[6] * a[6]; cov[1] = a[1] - a[6] * a[7]; cov[2] = a[2] - a[6] * a[8];
    cov[4] = a[3] - a[7] * a[7]; cov[5] = a[4] - a[7] * a[8]; cov[8] = a[5] - a[8] * a[8];
    cov[3] = cov[1]; cov[6] = cov[2]; cov[7] = cov[5];
    float scale = 0.f;
#pragma unroll
    for (int i = 0; i < 9; ++i) scale = fmaxf(scale, fabsf(cov[i]));
    if (scale <= 1.17549435e-38f) scale = 1.0f;
    float m[9];
#pragma unroll
    for (int i = 0; i < 9; ++i) m[i] = __fdiv_rn(cov[i], scale);
    float r[3]; roots3(m, r);
    const float ev = r[0] * scale;
    m[0] -= r[0]; m[4] -= r[0]; m[8] -= r[0];
    float v1[3] = {m[1] * m[5] - m[2] * m[4], m[2] * m[3] - m[0] * m[5], m[0] * m[4] - m[1] * m[3]};
    float v2[3] = {m[1] * m[8] - m[2] * m[7], m[2] * m[6] - m[0] * m[8], m[0] * m[7] - m[1] * m[6]};
    float v3[3] = {m[4] * m[8] - m[5] * m[7], m[5] * m[6] - m[3] * m[8], m[3] * m[7] - m[4] * m[6]};
    float l1 = v1[0] * v1[0] + v1[1] * v1[1] + v1[2] * v1[2];
    float l2 = v2[0] * v2[0] + v2[1] * v2[1] + v2[2] * v2[2];
    float l3 = v3[0] * v3[0] + v3[1] * v3[1] + v3[2] * v3[2];
    float nx, ny, nz, l;
    if (l1 >= l2 && l1 >= l3) { nx = v1[0]; ny = v1[1]; nz = v1[2]; l = l1; }
    else if (l2 >= l1 && l2 >= l3) { nx = v2[0]; ny = v2[1]; nz = v2[2]; l = l2; }
    else { nx = v3[0]; ny = v3[1]; nz = v3[2]; l = l3; }
    const float s = sqrtf(l);
    nx = __fdiv_rn(nx, s); ny = __fdiv_rn(ny, s); nz = __fdiv_rn(nz, s);
    const float eig_sum = cov[0] + cov[4] + cov[8];
    const float curv = eig_sum != 0.f ? fabsf(__fdiv_rn(ev, eig_sum)) : 0.f;
    const float wx = vx - px, wy = vy - py, wz = vz - pz;
    const float cos_theta = (wx * nx + wy * ny + wz * nz);
    if (cos_theta < 0) { nx *= -1; ny *= -1; nz *= -1; }
    return make_float4(nx, ny, nz, curv);
}
__device__ __forceinline__ void accu_add(float *a, float x, float y, float z) {
    a[0] += x * x; a[1] += x * y; a[2] += x * z; a[3] += y * y; a[4] += y * z; a[5] += z * z; a[6] += x; a[7] += y; a[8] += z;
}

// Eigen's completely unrolled reduction of a fixed-size 3-vector (norm, dot, 3x3 * vector): a0 + (a1 + a2)
__device__ __forceinline__ float sum3(float a0, float a1, float a2) { return a0 + (a1 + a2); }

// x = A.colPivHouseholderQr().solve(b) for a 3x3 fp32 system, Eigen 3.3's ColPivHouseholderQR restated (DESIGN.md section 2):
// largest-remaining-norm pivot (first on ties) with the LAPACK norm downdate, makeHouseholderInPlace, rank = pivots before the
// first column whose squared norm falls below (max norm * eps)^2 / 3 * (3 - k), back substitution over those pivots, zeros for
// the rest.  a is column-major (a[r + 3c]); with -fmad=false every operation below is one correctly rounded fp32 op.
__device__ __forceinline__ void colpiv_qr_solve(float a[9], const float b[3], float x[3]) {
    const float eps = 1.1920929e-07f;
    float hc[3], nu[3], nd[3];
    int perm[3] = {0, 1, 2};
#pragma unroll
    for (int k = 0; k < 3; ++k) { nd[k] = sqrtf(sum3(a[3 * k] * a[3 * k], a[3 * k + 1] * a[3 * k + 1], a[3 * k + 2] * a[3 * k + 2])); nu[k] = nd[k]; }
    float mx = nu[0];
    if (nu[1] > mx) mx = nu[1];
    if (nu[2] > mx) mx = nu[2];
    const float te = mx * eps;
    const float threshold_helper = __fdiv_rn(te * te, 3.0f);
    const float norm_downdate_threshold = sqrtf(eps);
    int np = 3;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        int bi = k;
#pragma unroll
        for (int j = k + 1; j < 3; ++j) if (nu[j] > nu[bi]) bi = j;
        const float bsq = nu[bi] * nu[bi];
        if (np == 3 && bsq < threshold_helper * (float)(3 - k)) np = k;
        if (bi != k) {        // bi is a run-time index: swap through selects so everything stays in registers
#pragma unroll
            for (int j = k + 1; j < 3; ++j) {
                if (j == bi) {
#pragma unroll
                    for (int r = 0; r < 3; ++r) { const float t = a[r + 3 * k]; a[r + 3 * k] = a[r + 3 * j]; a[r + 3 * j] = t; }
                    float t = nu[k]; nu[k] = nu[j]; nu[j] = t;
                    t = nd[k]; nd[k] = nd[j]; nd[j] = t;
                    const int ti = perm[k]; perm[k] = perm[j]; perm[j] = ti;
                }
            }
        }
        const float c0 = a[k + 3 * k];
        float tail_sq = 0.f;
#pragma unroll
        for (int r = k + 1; r < 3; ++r) tail_sq = (r == k + 1) ? a[r + 3 * k] * a[r + 3 * k] : tail_sq + a[r + 3 * k] * a[r + 3 * k];
        float tau, beta;
        if (tail_sq <= 1.17549435e-38f) {
            tau = 0.f; beta = c0;
#pragma unroll
            for (int r = k + 1; r < 3; ++r) a[r + 3 * k] = 0.f;
        } else {
            beta = sqrtf(c0 * c0 + tail_sq);
            if (c0 >= 0.f) beta = -beta;
            const float den = c0 - beta;
#pragma unroll
            for (int r = k + 1; r < 3; ++r) a[r + 3 * k] = __fdiv_rn(a[r + 3 * k], den);
            tau = __fdiv_rn(beta - c0, beta);
        }
        hc[k] = tau;
        a[k + 3 * k] = beta;
        if (tau != 0.f) {
#pragma unroll
            for (int j = k + 1; j < 3; ++j) {
                float t = 0.f;
#pragma unroll
                for (int r = k + 1; r < 3; ++r) t += a[r + 3 * k] * a[r + 3 * j];
                t = t + a[k + 3 * j];
                a[k + 3 * j] = a[k + 3 * j] - tau * t;
#pragma unroll
                for (int r = k + 1; r < 3; ++r) a[r + 3 * j] = a[r + 3 * j] - t * (tau * a[r + 3 * k]);
            }
        }
#pragma unroll
        for (int j = k + 1; j < 3; ++j) {
            if (nu[j] != 0.f) {
                float t = __fdiv_rn(fabsf(a[k + 3 * j]), nu[j]);
                t = (1.f + t) * (1.f - t);
                t = t < 0.f ? 0.f : t;
                const float q = __fdiv_rn(nu[j], nd[j]);
                const float t2 = t * (q * q);
                if (t2 <= norm_downdate_threshold) {
                    float s = 0.f;
#pragma unroll
                    for (int r = k + 1; r < 3; ++r) s = (r == k + 1) ? a[r + 3 * j] * a[r + 3 * j] : s + a[r + 3 * j] * a[r + 3 * j];
                    nd[j] = sqrtf(s);
                    nu[j] = nd[j];
                } else {
                    nu[j] *= sqrtf(t);
                }
            }
        }
    }
    x[0] = x[1] = x[2] = 0.f;
    if (np == 0) return;
    float c[3] = {b[0], b[1], b[2]};
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        if (k < np) {
            if (k == 2) { c[2] = c[2] * (1.f - hc[2]); }
            else if (hc[k] != 0.f) {
                float t = a[k + 1 + 3 * k] * c[k + 1];
#pragma unroll
                for (int r = k + 2; r < 3; ++r) t = t + a[r + 3 * k] * c[r];
                t = t + c[k];
                c[k] = c[k] - hc[k] * t;
#pragma unroll
                for (int r = k + 1; r < 3; ++r) c[r] = c[r] - t * (hc[k] * a[r + 3 * k]);
            }
        }
    }
#pragma unroll
    for (int i = 2; i >= 0; --i) {
        if (i < np && c[i] != 0.f) {
            c[i] = __fdiv_rn(c[i], a[i + 3 * i]);
#pragma unroll
            for (int s = 0; s < i; ++s) c[s] = c[s] - c[i] * a[s + 3 * i];
        }
    }
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        if (i < np) {
#pragma unroll
            for (int j = 0; j < 3; ++j) if (perm[i] == j) x[j] = c[i];
        }
    }
}

// expf for SIFTKeypoint's Gaussian weights, restated so that the CPU oracle (descriptor_oracle.c orc_sift_expf) computes the same
// bits: fp64 with every operation separately rounded -- Cody-Waite reduction x = k ln2 + r (fdlibm's split of ln2), Horner Taylor
// polynomial to r^11 on |r| <= ln2/2, exact scaling by 2^k -- then ONE rounding to fp32.  The fp64 error (~1e-15 relative) makes
// the result the correctly rounded expf except within ~1e-15 of an fp32 rounding midpoint, so it can differ by one ulp from a
// libm expf.  Valid for x in [-80, 80]; SIFT only calls it on [-4.6, 0].
__device__ __forceinline__ float sift_expf(float x) {
    const double xd = (double)x;
    const double k = rint(__dmul_rn(xd, 1.4426950408889634));
    const double r = __dsub_rn(__dsub_rn(xd, __dmul_rn(k, 0.6931471803691238)), __dmul_rn(k, 1.9082149292705877e-10));
    double p = 2.505210838544172e-08;
    p = __dadd_rn(__dmul_rn(p, r), 2.755731922398589e-07);
    p = __dadd_rn(__dmul_rn(p, r), 2.7557319223985893e-06);
    p = __dadd_rn(__dmul_rn(p, r), 2.48015873015873e-05);
    p = __dadd_rn(__dmul_rn(p, r), 0.0001984126984126984);
    p = __dadd_rn(__dmul_rn(p, r), 0.001388888888888889);
    p = __dadd_rn(__dmul_rn(p, r), 0.008333333333333333);
    p = __dadd_rn(__dmul_rn(p, r), 0.041666666666666664);
    p = __dadd_rn(__dmul_rn(p, r), 0.16666666666666666);
    p = __dadd_rn(__dmul_rn(p, r), 0.5);
    p = __dadd_rn(__dmul_rn(p, r), 1.0);
    p = __dadd_rn(__dmul_rn(p, r), 1.0);
    const double two_k = __hiloint2double(((int)k + 1023) << 20, 0);
    return __double2float_rn(__dmul_rn(p, two_k));
}

}  // namespace pcc
