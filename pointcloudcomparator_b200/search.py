"""Python host mirror of the reference's search plug-in, over the C ABI (include/pcc/search.h).

`GridSearch` keeps pcl::search::Search<PointT>'s vocabulary -- setInputCloud / nearestKSearch /
radiusSearch, batched over all query points -- plus the fused per-query reductions of its consumers
(reference call sites: src/segmentation.cpp:120-131,169-190,232-271; src/comparator.cpp:1089-1110,
1523-1541).  numpy arrays go through the PCC_HOST path (copies inside the call, like PCL's
std::vector outputs); torch CUDA tensors go through PCC_DEVICE (no copies, current stream).

The C++ twin that a PCL build would actually link is include/pcc/grid_search.hpp.
"""
from __future__ import annotations

import ctypes as C
import ctypes.util as ctypes_util

import numpy as np

from . import _lib
from ._lib import DEVICE, HOST, PccError, check

try:  # torch is plumbing only (device memory + streams)
    import torch
except Exception:  # pragma: no cover
    torch = None


def _is_cuda(t) -> bool:
    return torch is not None and isinstance(t, torch.Tensor) and t.is_cuda


def _rows(a):
    """(pointer, n, stride_bytes, mem, keepalive) for a [n, >=3] float32 numpy array or CUDA tensor."""
    if _is_cuda(a):
        assert a.dtype == torch.float32 and a.dim() == 2 and a.shape[1] >= 3 and a.stride(1) == 1
        return a.data_ptr(), a.shape[0], a.stride(0) * 4, DEVICE, a
    a = np.asarray(a)
    if a.dtype != np.float32 or a.ndim != 2 or a.shape[1] < 3 or a.strides[1] != 4 or (a.shape[0] > 1 and a.strides[0] % 4):
        a = np.ascontiguousarray(a, np.float32)
        assert a.ndim == 2 and a.shape[1] >= 3
    return a.ctypes.data, a.shape[0], (a.strides[0] if a.shape[0] > 1 else a.shape[1] * 4), HOST, a


def _stream(device=None):
    """torch's current stream ON THE INDEX'S DEVICE (the library launches there whatever torch's current device is)."""
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream) if torch is not None and torch.cuda.is_available() else None


class GridSearch:
    """pcl::search::KdTree<PointT> stand-in backed by the sm_100a uniform-grid engine."""

    def __init__(self, device: int = 0, sorted: bool = True):
        self._L = _lib.lib()
        self._h = C.c_void_p()
        check(self._L.pcc_create(int(device), C.byref(self._h)))
        self.device = int(device)
        self._sorted = bool(sorted)
        self._cloud = None
        self._mem = HOST
        self._n_input = 0

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            self._L.pcc_destroy(h)

    # ---- pcl::search::Search interface -------------------------------------------------------
    def getName(self) -> str:
        return "pcc::search::GridSearch"

    def setSortedResults(self, sorted: bool):
        self._sorted = bool(sorted)

    def getSortedResults(self) -> bool:
        return self._sorted

    def setInputCloud(self, cloud, indices=None, cell_hint: float = 0.0, k_hint: int = 0):
        """Search::setInputCloud(cloud, indices): index the finite points (original row numbers are kept)."""
        ptr, n, stride, mem, keep = _rows(cloud)
        ip, ni, ikeep = None, 0, None
        if indices is not None:
            if mem == DEVICE:
                ikeep = indices.to(torch.int32).contiguous()
                ip, ni = ikeep.data_ptr(), ikeep.numel()
            else:
                ikeep = np.ascontiguousarray(indices, np.int32)
                ip, ni = ikeep.ctypes.data, ikeep.size
        check(self._L.pcc_build(self._h, ptr, n, stride, ip, ni, float(cell_hint), int(k_hint), mem, _stream(self.device)))
        self._cloud, self._mem, self._n_input = keep, mem, n
        return self

    def getInputCloud(self):
        return self._cloud

    def _adopt_input(self, cloud, mem, n: int):
        """A batched entry rebuilt this index on `cloud` (n rows): self-queries (queries=None) now mean its rows.  n = 0 leaves the
        index, and so this state, untouched."""
        if n > 0:
            self._cloud, self._mem, self._n_input = cloud, mem, n

    @property
    def size(self) -> int:
        return int(self._L.pcc_size(self._h))

    def grid_info(self) -> dict:
        out = (C.c_double * 5)()
        check(self._L.pcc_grid_info(self._h, out))
        return dict(dims=(int(out[0]), int(out[1]), int(out[2])), cell=out[3], occupancy=out[4])

    def _queries(self, q):
        if q is None:
            return None, 0, 16, self._mem, None, self._n_input
        ptr, n, stride, mem, keep = _rows(q)
        return ptr, n, stride, mem, keep, n

    def _alloc(self, mem, shape, dtype):
        if mem == DEVICE:
            t = torch.empty(shape, dtype={np.int32: torch.int32, np.float32: torch.float32, np.int64: torch.int64, np.uint8: torch.uint8}[dtype], device=f"cuda:{self.device}")
            return t, t.data_ptr()
        a = np.empty(shape, dtype)
        return a, a.ctypes.data

    def nearestKSearch(self, queries, k: int):
        """Batched Search::nearestKSearch.  queries=None means every point of the input cloud.
        Returns (indices[n, k] int32, sqr_distances[n, k] float32, k_eff)."""
        ptr, nq, stride, mem, keep, rows = self._queries(queries)
        idx, ip = self._alloc(mem, (rows, k), np.int32)
        d2, dp = self._alloc(mem, (rows, k), np.float32)
        keff = C.c_int()
        check(self._L.pcc_knn(self._h, ptr, nq, stride, int(k), ip, dp, C.byref(keff), mem, _stream(self.device)))
        return idx, d2, keff.value

    def radiusSearch(self, queries, radius: float, max_nn: int = 0):
        """Batched Search::radiusSearch as CSR: (offsets[n+1] int64, indices int32, sqr_distances float32)."""
        ptr, nq, stride, mem, keep, rows = self._queries(queries)
        off, op = self._alloc(mem, (rows + 1,), np.int64)
        total = C.c_int64()
        check(self._L.pcc_radius_count(self._h, ptr, nq, stride, float(radius), int(max_nn), op, C.byref(total), mem, _stream(self.device)))
        idx, ip = self._alloc(mem, (max(total.value, 1),), np.int32)
        d2, dp = self._alloc(mem, (max(total.value, 1),), np.float32)
        check(self._L.pcc_radius_fill(self._h, ptr, nq, stride, float(radius), int(max_nn), int(self._sorted), op, ip, dp, mem, _stream(self.device)))
        return off, idx[: total.value], d2[: total.value]

    # ---- fused consumers -----------------------------------------------------------------------
    def meanNeighbourDistance(self, queries, mean_k: int):
        """StatisticalOutlierRemoval first pass: mean distance to the mean_k nearest (self dropped)."""
        ptr, nq, stride, mem, keep, rows = self._queries(queries)
        out, op = self._alloc(mem, (rows,), np.float32)
        check(self._L.pcc_knn_mean_dist(self._h, ptr, nq, stride, int(mean_k), op, mem, _stream(self.device)))
        return out

    def sorThreshold(self, distances, n_valid: int, std_mul: float):
        mem = DEVICE if _is_cuda(distances) else HOST
        if mem == HOST:
            distances = np.ascontiguousarray(distances, np.float32)
        n = distances.shape[0]
        keep, kp = self._alloc(mem, (n,), np.uint8)
        stats = (C.c_double * 3)()
        kept = C.c_int64()
        dp = distances.data_ptr() if mem == DEVICE else distances.ctypes.data
        check(self._L.pcc_sor_threshold(self._h, dp, n, int(n_valid), float(std_mul), stats, kp, C.byref(kept), mem, _stream(self.device)))
        return dict(mean=stats[0], stddev=stats[1], threshold=stats[2], kept=kept.value, keep=keep)

    def normalsKnn(self, queries, k: int, viewpoint=(0.0, 0.0, 0.0)):
        ptr, nq, stride, mem, keep, rows = self._queries(queries)
        out, op = self._alloc(mem, (rows, 4), np.float32)
        vp = (C.c_float * 3)(*[float(v) for v in viewpoint])
        check(self._L.pcc_normals_knn(self._h, ptr, nq, stride, int(k), vp, op, mem, _stream(self.device)))
        return out

    def normalsRadius(self, queries, radius: float, viewpoint=(0.0, 0.0, 0.0)):
        ptr, nq, stride, mem, keep, rows = self._queries(queries)
        out, op = self._alloc(mem, (rows, 4), np.float32)
        vp = (C.c_float * 3)(*[float(v) for v in viewpoint])
        check(self._L.pcc_normals_radius(self._h, ptr, nq, stride, float(radius), vp, op, mem, _stream(self.device)))
        return out

    def _per_row(self, a, mem, rows: int, cols: int, dtype=np.float32):
        """An input table of the descriptor consumers in the memory kind of the call: [rows, cols] float32, contiguous."""
        if mem == DEVICE:
            t = a if _is_cuda(a) else torch.as_tensor(np.asarray(a), device=f"cuda:{self.device}")
            t = t.to(device=f"cuda:{self.device}", dtype=torch.float32).reshape(rows, -1)
            if t.shape[1] < cols:
                t = torch.nn.functional.pad(t, (0, cols - t.shape[1]))
            t = t[:, :cols].contiguous()
            return t, t.data_ptr()
        h = a.detach().cpu().numpy() if _is_cuda(a) else np.asarray(a)
        h = np.asarray(h, dtype).reshape(rows, -1)
        out = np.zeros((rows, cols), dtype)
        out[:, : min(cols, h.shape[1])] = h[:, :cols]
        return out, out.ctypes.data

    def intensityGradient(self, queries, radius: float, intensity, normals):
        """IntensityGradientEstimation (src/comparator.cpp:649-656): intensity[n_input] per input row of the indexed cloud,
        normals[rows, >=3] of the queries (rows = n_input for queries=None).  Returns [rows, 4] = gx, gy, gz, 0."""
        ptr, nq, stride, mem, keep, rows = self._queries(queries)
        it, ip = self._per_row(intensity, mem, self._n_input, 1)
        nm, nmp = self._per_row(normals, mem, rows, 4)
        out, op = self._alloc(mem, (rows, 4), np.float32)
        check(self._L.pcc_intensity_gradient(self._h, ptr, nq, stride, float(radius), ip, nmp, op, mem, _stream(self.device)))
        return out

    def rift(self, queries, radius: float, gradients, nr_distance_bins: int = 4, nr_gradient_bins: int = 8):
        """RIFTEstimation (src/comparator.cpp:659-673): gradients[n_input, >=3] per input row of the indexed cloud.  Returns
        [rows, nd*ng] in PCL's histogram order (gradient bin outer, distance bin inner); NaN rows for queries without neighbours."""
        ptr, nq, stride, mem, keep, rows = self._queries(queries)
        gt, gp = self._per_row(gradients, mem, self._n_input, 4)
        out, op = self._alloc(mem, (rows, max(int(nr_distance_bins) * int(nr_gradient_bins), 1)), np.float32)
        check(self._L.pcc_rift(self._h, ptr, nq, stride, float(radius), gp, int(nr_distance_bins), int(nr_gradient_bins), op, mem, _stream(self.device)))
        return out

    def siftDoG(self, values, scales):
        """SIFTKeypoint::computeScaleSpace over the indexed cloud itself (src/comparator.cpp:449-465): values[n_input] (one field
        value per input row), scales = one octave's ascending scale table (2..16 entries).  Returns [n_input, len(scales) - 1]
        float32, dog[:, s-1] = response_s - response_{s-1}; NaN rows for skipped (non-finite) points."""
        sc = np.ascontiguousarray(scales, np.float32).reshape(-1)
        mem = self._mem
        vt, vp = self._per_row(values, mem, self._n_input, 1)
        out, op = self._alloc(mem, (self._n_input, max(sc.size - 1, 1)), np.float32)
        check(self._L.pcc_sift_dog(self._h, vp, sc.ctypes.data, int(sc.size), op, mem, _stream(self.device)))
        return out

    def siftExtrema(self, dog, min_contrast: float = 0.001):
        """SIFTKeypoint::findScaleSpaceExtrema over the indexed cloud: dog[n_input, n_cols] -> (rows, columns) int32 in (row,
        column) order, the points that are DoG extrema among their 25 nearest neighbours."""
        mem = self._mem
        n_cols = int(dog.shape[1])
        dt, dp = self._per_row(dog, mem, self._n_input, n_cols)
        cap = max(self._n_input * max(n_cols - 2, 0), 1)
        rows, rp = self._alloc(mem, (cap,), np.int32)
        cols, cp = self._alloc(mem, (cap,), np.int32)
        found = C.c_int64()
        check(self._L.pcc_sift_extrema(self._h, dp, n_cols, float(min_contrast), rp, cp, cap, C.byref(found), mem, _stream(self.device)))
        return rows[: found.value], cols[: found.value]

    def icpStep(self, source, T_apply=None, want_correspondences: bool = False):
        """One correspondence pass against the indexed (target) cloud; `source` is moved in place by T_apply."""
        ptr, ns, stride, mem, keep = _rows(source)
        sums = (C.c_double * 16)()
        cnt = C.c_int64()
        Tp = None
        if T_apply is not None:
            Tp = (C.c_float * 16)(*np.asarray(T_apply, np.float32).reshape(-1).tolist())
        ci = cd = None
        ip = dp = None
        if want_correspondences:
            ci, ip = self._alloc(mem, (ns,), np.int32)
            cd, dp = self._alloc(mem, (ns,), np.float32)
        check(self._L.pcc_icp_step(self._h, ptr, ns, stride, Tp, sums, C.byref(cnt), ip, dp, mem, _stream(self.device)))
        return cnt.value, np.array(sums[:], np.float64), ci, cd

    def icpAlign(self, source, max_iter: int = 20):
        """IterativeClosestPoint::align + getFitnessScore against the indexed (target) cloud."""
        ptr, ns, stride, mem, keep = _rows(source)
        T = (C.c_float * 16)()
        conv, it, fit = C.c_int(), C.c_int(), C.c_double()
        check(self._L.pcc_icp_align(self._h, ptr, ns, stride, int(max_iter), T, C.byref(conv), C.byref(fit), C.byref(it), mem, _stream(self.device)))
        return dict(T=np.array(T[:], np.float32).reshape(4, 4), converged=bool(conv.value), fitness=fit.value, iterations=it.value)

    def euclideanClusters(self, tolerance: float, min_size: int = 1, max_size: int = 2**31 - 1):
        """EuclideanClusterExtraction over the input cloud: (labels[n] int32, sizes int64)."""
        mem = self._mem
        labels, lp = self._alloc(mem, (max(self._n_input, 1),), np.int32)
        cap = max(self._n_input // max(int(min_size), 1) + 1, 1)
        sizes, sp = self._alloc(mem, (cap,), np.int64)
        nc = C.c_int64()
        check(self._L.pcc_euclidean_labels(self._h, float(tolerance), int(min_size), int(max_size), lp, C.byref(nc), sp, cap, mem, _stream(self.device)))
        return labels[: self._n_input], sizes[: nc.value]

    # ---- sharded clustering primitives (device tensors; forests over SORTED positions, see include/pcc/search.h) ----
    def eceNewForest(self):
        parent = torch.empty(max(self.size, 1), dtype=torch.int32, device=f"cuda:{self.device}")
        check(self._L.pcc_ece_init(self._h, parent.data_ptr(), _stream(self.device)))
        return parent

    def eceLinkRange(self, parent, tolerance: float, begin: int, end: int):
        check(self._L.pcc_ece_link_range(self._h, float(tolerance), int(begin), int(end), parent.data_ptr(), _stream(self.device)))

    def eceAbsorb(self, parent, other):
        check(self._L.pcc_ece_absorb(self._h, other.data_ptr(), parent.data_ptr(), _stream(self.device)))

    def eceFinish(self, parent, min_size: int = 1, max_size: int = 2**31 - 1):
        labels = torch.empty(max(self._n_input, 1), dtype=torch.int32, device=f"cuda:{self.device}")
        cap = max(self._n_input // max(int(min_size), 1) + 1, 1)
        sizes = torch.empty(cap, dtype=torch.int64, device=f"cuda:{self.device}")
        nc = C.c_int64()
        check(self._L.pcc_ece_finish(self._h, parent.data_ptr(), int(min_size), int(max_size), labels.data_ptr(), C.byref(nc), sizes.data_ptr(), cap, _stream(self.device)))
        return labels[: self._n_input], sizes[: nc.value]

    def firstWithin(self, queries, thr: float):
        ptr, nq, stride, mem, keep = _rows(queries)
        out, op = self._alloc(mem, (nq,), np.int32)
        check(self._L.pcc_first_within(self._h, ptr, nq, stride, float(thr), op, mem, _stream(self.device)))
        return out

    # ---- measurement + multi-GPU plumbing ----------------------------------------------------------
    # ---- multi-GPU (include/pcc/search.h: pcc_comm_init / pcc_broadcast_index / pcc_gather) ----------------------
    def commInit(self, nccl_comm, rank: int, world: int):
        """Attach the caller's ncclComm_t (an integer handle, e.g. from shard.nccl_comm) to this index."""
        check(self._L.pcc_comm_init(self._h, C.c_void_p(int(nccl_comm) if nccl_comm else 0), int(rank), int(world)))
        return self

    def broadcastIndex(self, root: int = 0):
        """Every rank but `root` adopts the grid `root` built (NCCL broadcast straight into the device arrays)."""
        check(self._L.pcc_broadcast_index(self._h, int(root), _stream(self.device)))
        self._mem = DEVICE
        self._n_input = int(self._meta()[1])
        return self

    def _meta(self):
        meta = (C.c_double * 16)()
        ptrs = (C.c_void_p * 2)()
        check(self._L.pcc_export(self._h, meta, ptrs))
        return np.array(meta[:], np.float64)

    def gather(self, local, rows, n_total: int):
        """All-gather of per-shard result rows (CUDA tensors): `local` [n_local, ...] 4-byte elements, `rows` the original row number
        of each local row (int32/int64 tensor) or None (rank-order concatenation).  Returns the full [n_total, ...] table."""
        assert _is_cuda(local) and local.is_contiguous() and local.element_size() == 4
        row_bytes = int(np.prod(local.shape[1:], dtype=np.int64)) * 4 if local.dim() > 1 else 4
        out = torch.empty((int(n_total),) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
        r32 = None if rows is None else rows.to(torch.int32).contiguous()
        check(self._L.pcc_gather(self._h, local.data_ptr(), local.shape[0], row_bytes, None if r32 is None else r32.data_ptr(), out.data_ptr(), int(n_total), _stream(self.device)))
        return out

    def setTiming(self, enable: bool):
        check(self._L.pcc_set_timing(self._h, int(enable)))

    def lastKernelMs(self) -> float:
        return float(self._L.pcc_last_kernel_ms(self._h))

    def export(self):
        """(meta[16] float64, points float4 tensor view, cell_start tensor view) of the built grid (device memory)."""
        meta = (C.c_double * 16)()
        ptrs = (C.c_void_p * 2)()
        check(self._L.pcc_export(self._h, meta, ptrs))
        return np.array(meta[:], np.float64), int(ptrs[0] or 0), int(ptrs[1] or 0)

    def adopt(self, meta):
        m = (C.c_double * 16)(*[float(v) for v in meta])
        check(self._L.pcc_adopt(self._h, m, _stream(self.device)))
        self._n_input, self._mem = int(meta[1]), DEVICE
        return self.export()


def voxel_grid(rows, leaf, rgb_offset_bytes: int = -1, min_points: int = 0, device: int = 0, workspace: "GridSearch | None" = None):
    """pcl::VoxelGrid::applyFilter (src/segmentation.cpp:69-74, 223-228) on the GPU: rows[n, stride] float32 (numpy or CUDA
    tensor, colour as a packed BGRA word at rgb_offset_bytes) -> one centroid row per occupied voxel, ordered by voxel index."""
    ws = workspace or GridSearch(device)
    ptr, n, stride, mem, keep = _rows(rows)
    lf = (C.c_float * 3)(*np.broadcast_to(np.asarray(leaf, np.float32), (3,)).tolist())
    if mem == DEVICE:
        out = torch.empty_like(rows)
        op = out.data_ptr()
    else:
        out = np.zeros((n, stride // 4), np.float32)
        op = out.ctypes.data
    n_out = C.c_int64()
    check(ws._L.pcc_voxel_grid(ws._h, ptr, n, stride, int(rgb_offset_bytes), lf, int(min_points), op, C.byref(n_out), mem, _stream(ws.device)))
    return out[: n_out.value]


def region_growing(neighbours, normals, smoothness_rad: float = 3.0 / 180.0 * np.pi, curvature_threshold: float = 1.0, min_size: int = 50, max_size: int = 1000000):
    """RegionGrowing::extract over a GPU-built neighbour table (src/segmentation.cpp:249-271): labels[n] (creation order, -1 = dropped), count."""
    nb = np.ascontiguousarray(neighbours.cpu().numpy() if _is_cuda(neighbours) else neighbours, np.int32)
    nm = np.ascontiguousarray(normals.cpu().numpy() if _is_cuda(normals) else normals, np.float32)
    labels = np.empty(nb.shape[0], np.int32)
    nc = C.c_int64()
    check(_lib.lib().pcc_region_growing(nb.ctypes.data, nb.shape[0], nb.shape[1], nm.ctypes.data, float(smoothness_rad), float(curvature_threshold), int(min_size), int(max_size), labels.ctypes.data, C.byref(nc)))
    return labels, nc.value


def region_growing_rgb(neighbours, sqr_distances, rgba, distance_threshold: float = 10.0, point_color_threshold: float = 6.0, region_color_threshold: float = 5.0,
                       grow_neighbours: int = 30, min_size: int = 200, max_size: int = 2**31 - 1):
    """RegionGrowingRGB::extract over the GPU-built N x k table (color_growing_segmentation, src/segmentation.cpp:161-216): returns
    (labels[n] int32, n_clusters).  rgba = packed 0x00RRGGBB words (uint32[n])."""
    nb = np.ascontiguousarray(neighbours, np.int32)
    nd = np.ascontiguousarray(sqr_distances, np.float32)
    col = np.ascontiguousarray(rgba, np.uint32)
    assert nb.shape == nd.shape and col.shape[0] == nb.shape[0]
    labels = np.empty(nb.shape[0], np.int32)
    nc = C.c_int64()
    check(_lib.lib().pcc_region_growing_rgb(nb.ctypes.data, nd.ctypes.data, nb.shape[0], nb.shape[1], col.ctypes.data, 4, float(distance_threshold), float(point_color_threshold),
                                            float(region_color_threshold), int(grow_neighbours), int(min_size), int(max_size), labels.ctypes.data, C.byref(nc)))
    return labels, int(nc.value)


def knn_batched(xyz, offsets, k: int, device: int = 0, workspace: "GridSearch | None" = None):
    """RegionGrowingRGB::findPointNeighbours on every cluster [offsets[c], offsets[c+1]) of xyz in one pcc_knn_batched call: returns
    (idx [n, k] int32, d2 [n, k] float32, k_eff int32 [n_clouds]); the rows of cluster c are GridSearch().setInputCloud(cluster, k_hint=k)
    .nearestKSearch(None, k) of that cluster alone, bit for bit, with cluster-LOCAL indices.  numpy inputs go through PCC_HOST; a CUDA
    tensor xyz keeps the call and the table on the device, on the current stream.  `workspace` is left indexing the concatenation."""
    off = np.ascontiguousarray(np.asarray(offsets), np.int64)
    n_clouds = off.shape[0] - 1
    k_eff = np.zeros(max(n_clouds, 0) + 1, np.int32)
    ws = workspace or GridSearch(device)
    ptr, n, stride, mem, keep = _rows(xyz if _is_cuda(xyz) else np.asarray(xyz, np.float32))
    idx, ip = ws._alloc(mem, (n, int(k)), np.int32)
    d2, dp = ws._alloc(mem, (n, int(k)), np.float32)
    check(ws._L.pcc_knn_batched(ws._h, ptr, n, stride, off.ctypes.data, n_clouds, int(k), ip, dp, k_eff.ctypes.data, mem, _stream(ws.device)))
    ws._adopt_input(keep, mem, n)
    return idx, d2, k_eff[:n_clouds]


def region_growing_rgb_batched(xyz, rgb, offsets, k: int = 100, distance_threshold: float = 10.0, point_color_threshold: float = 6.0,
                               region_color_threshold: float = 5.0, grow_neighbours: int = 30, min_size: int = 200, max_size: int = 2**31 - 1,
                               device: int = 0, workspace: "GridSearch | None" = None):
    """color_growing_segmentation (src/segmentation.cpp:161-216) on every cluster [offsets[c], offsets[c+1]) of xyz / rgb in one
    pcc_region_growing_rgb_batched call: returns (labels int32 [n], n_clusters int64 [n_clouds]); labels of cluster c are cluster-LOCAL and
    equal region_growing_rgb over knn_batched's table of that cluster alone.  rgb is uint8 [n, 3] (r, g, b).  The reference's "more than
    10 points" test (src/segmentation.cpp:167) stays with the caller.  A CUDA tensor xyz runs the search on the device, on the current
    stream; the grow runs on the host either way."""
    off = np.ascontiguousarray(np.asarray(offsets), np.int64)
    n_clouds = off.shape[0] - 1
    rows, ptr, n, mem = _xyzrgb_rows(xyz, rgb)
    labels = np.empty(max(n, 1), np.int32)
    n_clusters = np.zeros(max(n_clouds, 0) + 1, np.int64)
    ws = workspace or GridSearch(device)
    check(ws._L.pcc_region_growing_rgb_batched(ws._h, ptr, n, 16, 12, off.ctypes.data, n_clouds, int(k), float(distance_threshold), float(point_color_threshold),
                                               float(region_color_threshold), int(grow_neighbours), int(min_size), int(max_size), labels.ctypes.data,
                                               n_clusters.ctypes.data, mem, _stream(ws.device)))
    ws._adopt_input(rows, mem, n)
    return labels[:n], n_clusters[:n_clouds]


def descriptor_nn(ref, qry, dims: int | None = None, device: int = 0, workspace: "GridSearch | None" = None):
    """1-NN in descriptor space (matchRIFTFeaturesKnn, src/comparator.cpp:560-588): (index into ref or -1, squared distance).
    `dims` = leading floats of a row that take part (None = all columns; 3 = what PCL 1.7 compares for Histogram<32>, see search.h)."""
    ws = workspace or GridSearch(device)
    dims = int(ref.shape[1] if dims is None else dims)
    if _is_cuda(ref):
        assert ref.dtype == torch.float32 and qry.dtype == torch.float32 and ref.stride(1) == 1 and qry.stride(1) == 1 and ref.stride(0) == qry.stride(0)
        idx = torch.empty(qry.shape[0], dtype=torch.int32, device=ref.device); d2 = torch.empty(qry.shape[0], dtype=torch.float32, device=ref.device)
        check(ws._L.pcc_descriptor_nn(ws._h, ref.data_ptr(), ref.shape[0], qry.data_ptr(), qry.shape[0], dims, ref.stride(0), idx.data_ptr(), d2.data_ptr(), DEVICE, _stream(ws.device)))
        return idx, d2
    ref, qry = np.ascontiguousarray(ref, np.float32), np.ascontiguousarray(qry, np.float32)
    idx, d2 = np.empty(qry.shape[0], np.int32), np.empty(qry.shape[0], np.float32)
    check(ws._L.pcc_descriptor_nn(ws._h, ref.ctypes.data, ref.shape[0], qry.ctypes.data, qry.shape[0], dims, ref.shape[1], idx.ctypes.data, d2.ctypes.data, HOST, _stream(ws.device)))
    return idx, d2


def match_rift_features_knn(desc1, desc2, threshold: float = 0.05, match_dims: int = 3, **kw):
    """The reference's correspondence vector: one leading 0 (its `std::vector<int> correspondence(1)`), then the matched indices.
    match_dims = 3 reproduces the reference binary (PCL 1.7 clamps an unregistered Histogram<32> to its first 3 floats);
    match_dims = 32 matches on the whole RIFT histogram."""
    idx, d2 = descriptor_nn(desc1, desc2, dims=match_dims, **kw)
    if _is_cuda(idx):
        idx, d2 = idx.cpu().numpy(), d2.cpu().numpy()
    keep = (idx >= 0) & (d2 < np.float32(threshold))
    return [0] + idx[keep].tolist()


def rgb_to_intensity(rgb):
    """PCL 1.7 PointXYZRGBtoXYZI (src/comparator.cpp:597): 0.299f r + 0.587f g + 0.114f b, evaluated left to right in fp32.
    rgb[n, 3] uint8 (r, g, b) -> float32[n]."""
    c = np.asarray(rgb.cpu().numpy() if _is_cuda(rgb) else rgb).reshape(-1, 3).astype(np.float32)
    return ((np.float32(0.299) * c[:, 0] + np.float32(0.587) * c[:, 1]) + np.float32(0.114) * c[:, 2]).astype(np.float32)


def process_rift(xyz, rgb, normal_radius: float = 0.03, gradient_radius: float = 0.03, rift_radius: float = 0.05, nr_distance_bins: int = 4,
                 nr_gradient_bins: int = 8, device: int = 0, stages: dict | None = None):
    """processRIFT (src/comparator.cpp:590-684) on the GPU: intensity (:597) -> NormalEstimation r 0.03 (:628-635) -> drop the rows
    whose normal is NaN (:637-646) -> IntensityGradientEstimation r 0.03 (:649-656) -> RIFTEstimation r 0.05, 4 x 8 bins (:659-673)
    -> drop the rows with a non-finite bin (:674-681).  The gradient and RIFT stages search the filtered cloud, so the index is
    rebuilt on it.  Returns (descriptors [m, nd*ng] float32, kept_rows int64 into xyz); m is the reference's "Number of
    descriptors".  `stages` (a dict) receives the intermediate arrays."""
    xyz = np.ascontiguousarray(np.asarray(xyz.cpu().numpy() if _is_cuda(xyz) else xyz, np.float32)[:, :3])
    inten = rgb_to_intensity(rgb)
    s0 = GridSearch(device).setInputCloud(xyz, cell_hint=normal_radius)
    normals = s0.normalsRadius(None, normal_radius)
    keep1 = np.flatnonzero(np.isfinite(normals[:, :3]).all(1))
    xyz1 = np.ascontiguousarray(xyz[keep1])
    s1 = GridSearch(device).setInputCloud(xyz1, cell_hint=rift_radius)
    grad = s1.intensityGradient(None, gradient_radius, inten[keep1], normals[keep1])
    desc = s1.rift(None, rift_radius, grad, nr_distance_bins, nr_gradient_bins)
    keep2 = np.flatnonzero(np.isfinite(desc).all(1))
    if stages is not None:
        stages.update(intensity=inten, normals=normals, kept_normals=keep1, gradients=grad, descriptors_all=desc)
    return desc[keep2], keep1[keep2].astype(np.int64)


def process_rift_batched(xyz, rgb, offsets, normal_radius: float = 0.03, gradient_radius: float = 0.03, rift_radius: float = 0.05,
                         nr_distance_bins: int = 4, nr_gradient_bins: int = 8, device: int = 0):
    """process_rift on every cluster [offsets[c], offsets[c+1]) of xyz / rgb in one pcc_rift_batched call: returns (descriptors [m, nd*ng],
    desc_offsets int64 [n_clouds + 1], kept_rows int64 [m]); rows desc_offsets[c]:desc_offsets[c+1] are process_rift of cluster c, bit for
    bit, with cluster-LOCAL kept rows.  numpy inputs go through PCC_HOST; a CUDA tensor xyz keeps the call and its outputs on the device,
    on the current stream."""
    off = np.ascontiguousarray(np.asarray(offsets), np.int64)
    n_clouds = off.shape[0] - 1
    desc_off = np.zeros(max(n_clouds, 0) + 1, np.int64)
    nb = int(nr_distance_bins) * int(nr_gradient_bins)
    inten = rgb_to_intensity(rgb)
    if _is_cuda(xyz):
        ptr, n, stride, mem, keep = _rows(xyz)
        it = torch.as_tensor(inten, device=xyz.device)
        ip = it.data_ptr()
        alloc = lambda shape, dt: torch.empty(shape, dtype=dt, device=xyz.device)      # noqa: E731
        f32, i32 = torch.float32, torch.int32
    else:
        ptr, n, stride, mem, keep = _rows(np.asarray(xyz, np.float32))
        ip = inten.ctypes.data
        alloc = lambda shape, dt: np.empty(shape, dt)                                   # noqa: E731
        f32, i32 = np.float32, np.int32
    L = _lib.lib()
    ws = GridSearch(device)
    cap = max(n, 1)
    while True:
        out = alloc((cap, max(nb, 1)), f32)
        rows = alloc((cap,), i32)
        op, rp = (out.data_ptr(), rows.data_ptr()) if mem == DEVICE else (out.ctypes.data, rows.ctypes.data)
        check(L.pcc_rift_batched(ws._h, ptr, n, stride, ip, off.ctypes.data, n_clouds, float(normal_radius), float(gradient_radius), float(rift_radius),
                                 int(nr_distance_bins), int(nr_gradient_bins), op, rp, cap, desc_off.ctypes.data, mem, _stream(ws.device)))
        total = int(desc_off[-1])
        if total <= cap:
            break
        cap = total
    kept = rows[:total].to(torch.int64) if mem == DEVICE else rows[:total].astype(np.int64)
    return out[:total], desc_off, kept


def sift_field_values(rgb):
    """PCL 1.7 SIFTKeypointFieldSelector<PointXYZRGB>: float(299 r + 587 g + 114 b) / 1000.0f (integer sum, one fp32 division).
    Not the XYZRGB -> XYZI weights of rgb_to_intensity.  rgb[n, 3] uint8 (r, g, b) -> float32[n]."""
    c = np.asarray(rgb.cpu().numpy() if _is_cuda(rgb) else rgb).reshape(-1, 3).astype(np.int64)
    return ((299 * c[:, 0] + 587 * c[:, 1] + 114 * c[:, 2]).astype(np.float32) / np.float32(1000.0)).astype(np.float32)


_libm = None


def sift_scales(base_scale: float, nr_scales_per_octave: int = 5):
    """One octave's scale table as detectKeypointsForOctave builds it: base_scale * powf(2.0f, (1.0f * i - 1.0f) / nr_scales_per_octave)
    for i < nr_scales_per_octave + 3, with the C library's powf (the one libpcc_search calls), float32."""
    global _libm
    if _libm is None:
        _libm = C.CDLL(ctypes_util.find_library("m"))
        _libm.powf.argtypes, _libm.powf.restype = [C.c_float, C.c_float], C.c_float
    nsp = np.float32(nr_scales_per_octave)
    e = [(np.float32(1.0) * np.float32(i) - np.float32(1.0)) / nsp for i in range(int(nr_scales_per_octave) + 3)]
    return np.array([np.float32(base_scale) * np.float32(_libm.powf(2.0, float(x))) for x in e], np.float32)


def _sift_rows(xyz, rgb):
    """[n, 4] float32 (x, y, z, packed 0x00RRGGBB word): the layout pcc_sift_keypoints and every octave cloud use."""
    xyz = np.asarray(xyz.cpu().numpy() if _is_cuda(xyz) else xyz, np.float32)
    c = np.asarray(rgb.cpu().numpy() if _is_cuda(rgb) else rgb).reshape(-1, 3).astype(np.uint32)
    rows = np.empty((xyz.shape[0], 4), np.float32)
    rows[:, :3] = xyz[:, :3]
    rows[:, 3] = ((c[:, 0] << 16) | (c[:, 1] << 8) | c[:, 2]).view(np.float32)
    return rows


def _xyzrgb_rows(xyz, rgb):
    """_sift_rows in the memory kind of xyz: (rows, pointer, n, mem); a CUDA tensor xyz gets CUDA rows (PCC_DEVICE), else numpy (PCC_HOST)."""
    if _is_cuda(xyz):
        c = torch.as_tensor(np.asarray(rgb.cpu().numpy() if _is_cuda(rgb) else rgb).reshape(-1, 3).astype(np.int32), device=xyz.device)
        rows = torch.empty((xyz.shape[0], 4), dtype=torch.float32, device=xyz.device)
        rows[:, :3] = xyz[:, :3]
        rows[:, 3] = ((c[:, 0] << 16) | (c[:, 1] << 8) | c[:, 2]).view(torch.float32)
        return rows, rows.data_ptr(), rows.shape[0], DEVICE
    rows = _sift_rows(xyz, rgb)
    return rows, rows.ctypes.data, rows.shape[0], HOST


def sift_keypoints(xyz, rgb, min_scale: float = 0.005, nr_octaves: int = 5, nr_scales_per_octave: int = 5, min_contrast: float = 0.001,
                   device: int = 0, stages: dict | None = None):
    """SIFTKeypoint<PointXYZRGB, PointWithScale>::compute as processSift configures it (src/comparator.cpp:449-465), one
    pcc_sift_keypoints call: returns float32 [m, 4] = (x, y, z, scale) in (octave, point, column) order.  `stages` (a dict)
    receives stages["octaves"], one dict per octave (cloud, scales, dog, rows, cols, keypoints), recomputed through the public
    pieces (voxel_grid, GridSearch.siftDoG / siftExtrema); their keypoints concatenate to the returned array."""
    rows = _sift_rows(xyz, rgb)
    ws = GridSearch(device)
    cap = max(rows.shape[0], 1)
    while True:
        out = np.empty((cap, 4), np.float32)
        found = C.c_int64()
        check(ws._L.pcc_sift_keypoints(ws._h, rows.ctypes.data, rows.shape[0], 16, 12, float(min_scale), int(nr_octaves), int(nr_scales_per_octave),
                                       float(min_contrast), out.ctypes.data, cap, C.byref(found), HOST, _stream(ws.device)))
        if found.value <= cap:
            break
        cap = found.value
    if stages is not None:
        cloud, scale, octs = rows, np.float32(min_scale), []
        for _ in range(int(nr_octaves)):
            cloud = voxel_grid(cloud, scale, rgb_offset_bytes=12, workspace=ws)
            if cloud.shape[0] < 25:
                break
            scales = sift_scales(scale, nr_scales_per_octave)
            s = GridSearch(device).setInputCloud(cloud, cell_hint=float(np.float32(3) * scales[-1]))
            dog = s.siftDoG(sift_field_values(np.stack([(cloud[:, 3].view(np.uint32) >> sh) & 255 for sh in (16, 8, 0)], 1)), scales)
            r, c = s.siftExtrema(dog, min_contrast)
            kp = np.column_stack([cloud[r, :3], scales[c]]).astype(np.float32)
            octs.append(dict(cloud=cloud, scales=scales, dog=dog, rows=r, cols=c, keypoints=kp))
            scale = np.float32(scale * np.float32(2))
        stages["octaves"] = octs
    return out[: found.value]


def process_sift(xyz, rgb, snap_threshold: float = 0.05, device: int = 0, **sift_kw):
    """processSift + the snap of processRIFTwithSIFT (src/comparator.cpp:435-469, 696-713): SIFT keypoints of the cluster, then for
    every keypoint the first cloud point (lowest index) within 0.05 of it, -1 if none.  Returns (keypoints [m, 4], snap int32[m]):
    what processRIFTwithSIFT holds before its descriptor chain."""
    kp = sift_keypoints(xyz, rgb, device=device, **sift_kw)
    if kp.shape[0] == 0:
        return kp, np.empty(0, np.int32)
    xyz = np.ascontiguousarray(np.asarray(xyz.cpu().numpy() if _is_cuda(xyz) else xyz, np.float32)[:, :3])
    s = GridSearch(device).setInputCloud(xyz, cell_hint=snap_threshold)
    return kp, s.firstWithin(np.ascontiguousarray(kp[:, :3]), snap_threshold)


def _sift_batched(xyz, rgb, offsets, snap_threshold, min_scale, nr_octaves, nr_scales_per_octave, min_contrast, device):
    """pcc_sift_keypoints_batched over the clusters [offsets[c], offsets[c+1]) of xyz: numpy inputs go through PCC_HOST, a CUDA
    tensor xyz through PCC_DEVICE on the current stream.  Returns (keypoints [m, 4], kp_offsets int64 [n_clouds + 1], snap or None)."""
    off = np.ascontiguousarray(np.asarray(offsets), np.int64)
    n_clouds = off.shape[0] - 1
    kp_off = np.zeros(max(n_clouds, 0) + 1, np.int64)
    want_snap = snap_threshold is not None
    rows, ptr, n, mem = _xyzrgb_rows(xyz, rgb)
    if mem == DEVICE:
        alloc = lambda shape, dt: torch.empty(shape, dtype=dt, device=xyz.device)   # noqa: E731
        f32, i32 = torch.float32, torch.int32
    else:
        alloc = lambda shape, dt: np.empty(shape, dt)                                 # noqa: E731
        f32, i32 = np.float32, np.int32
    L = _lib.lib()
    ws = GridSearch(device)
    cap = max(n, 1)
    while True:
        out = alloc((cap, 4), f32)
        snap = alloc((cap,), i32) if want_snap else None
        op = out.data_ptr() if mem == DEVICE else out.ctypes.data
        sp = None if snap is None else (snap.data_ptr() if mem == DEVICE else snap.ctypes.data)
        check(L.pcc_sift_keypoints_batched(ws._h, ptr, n, 16, 12, off.ctypes.data, n_clouds, float(min_scale), int(nr_octaves), int(nr_scales_per_octave),
                                           float(min_contrast), float(snap_threshold if want_snap else 0.0), op, sp, cap, kp_off.ctypes.data, mem,
                                           _stream(ws.device)))
        total = int(kp_off[-1])
        if total <= cap:
            break
        cap = total
    return out[:total], kp_off, (None if snap is None else snap[:total])


def sift_keypoints_batched(xyz, rgb, offsets, min_scale: float = 0.005, nr_octaves: int = 5, nr_scales_per_octave: int = 5, min_contrast: float = 0.001,
                           device: int = 0):
    """sift_keypoints on every cluster [offsets[c], offsets[c+1]) of xyz / rgb in one pcc_sift_keypoints_batched call: returns
    (keypoints float32 [m, 4], kp_offsets int64 [n_clouds + 1]); keypoints[kp_offsets[c]:kp_offsets[c+1]] is sift_keypoints of cluster c,
    bit for bit.  A CUDA tensor xyz keeps the call and its outputs in device memory."""
    kp, kp_off, _ = _sift_batched(xyz, rgb, offsets, None, min_scale, nr_octaves, nr_scales_per_octave, min_contrast, device)
    return kp, kp_off


def process_sift_batched(xyz, rgb, offsets, snap_threshold: float = 0.05, device: int = 0, **sift_kw):
    """process_sift on every cluster of xyz / rgb in one call: (keypoints [m, 4], kp_offsets int64 [n_clouds + 1], snap int32 [m]); snap
    holds cluster-LOCAL rows (the lowest-index point of the keypoint's own cluster within snap_threshold, -1 if none)."""
    kw = dict(min_scale=0.005, nr_octaves=5, nr_scales_per_octave=5, min_contrast=0.001)
    kw.update(sift_kw)
    return _sift_batched(xyz, rgb, offsets, float(snap_threshold), kw["min_scale"], kw["nr_octaves"], kw["nr_scales_per_octave"], kw["min_contrast"], device)


def umeyama_from_sums(sums, count: int):
    T = (C.c_float * 16)()
    s = (C.c_double * 16)(*[float(v) for v in sums])
    check(_lib.lib().pcc_umeyama_from_sums(s, int(count), T))
    return np.array(T[:], np.float32).reshape(4, 4)


def launch_count() -> int:
    return int(_lib.lib().pcc_launch_count())
