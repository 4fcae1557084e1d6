"""ctypes front-end of the descriptor-stage and SIFT-keypoint CPU oracle (descriptor_oracle/descriptor_oracle.c).

TEST INFRASTRUCTURE ONLY, like oracle/: the product package (pointcloudcomparator_b200) never imports it.  The
neighbour rows come from oracle.KdTree.radius (sorted by (fp32 d2, original index)), so the chain below is
CPU code end to end.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libdescriptor_oracle.so")
_lib = None


def build(force: bool = False) -> str:
    src = os.path.join(_HERE, "descriptor_oracle.c")
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _HERE, "-s"], env={**os.environ, "CC": "/usr/bin/gcc"})
    return _SO


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_SO)
        f32p, i32p, i64p, i64, i32 = C.POINTER(C.c_float), C.POINTER(C.c_int32), C.POINTER(C.c_int64), C.c_int64, C.c_int
        L.orc_colpiv_qr_solve3.argtypes = [f32p, f32p, f32p]
        L.orc_colpiv_qr_solve3.restype = None
        L.orc_intensity_gradient_from_lists.argtypes = [f32p, i32, f32p, f32p, i64, i64p, i32p, f32p]
        L.orc_intensity_gradient_from_lists.restype = None
        L.orc_rift_from_lists.argtypes = [f32p, i32, f32p, i64, i32, i64p, i32p, f32p, f32p, C.c_float, i32, i32, f32p]
        L.orc_rift_from_lists.restype = i32
        L.orc_rgb_to_intensity.argtypes = [C.POINTER(C.c_uint8), i64, f32p]
        L.orc_rgb_to_intensity.restype = None
        L.orc_desc_num_threads.restype = i32
        L.orc_sift_expf.argtypes = [f32p, i64, f32p]
        L.orc_sift_expf.restype = None
        L.orc_sift_scales.argtypes = [C.c_float, i32, f32p]
        L.orc_sift_scales.restype = None
        L.orc_sift_field_values.argtypes = [C.POINTER(C.c_uint8), i64, f32p]
        L.orc_sift_field_values.restype = None
        L.orc_sift_dog_from_lists.argtypes = [f32p, i64, i64p, i32p, f32p, f32p, i32, f32p]
        L.orc_sift_dog_from_lists.restype = None
        L.orc_sift_extrema_from_lists.argtypes = [f32p, i64, i32, i32p, i32, C.c_float, i32p, i32p, i64]
        L.orc_sift_extrema_from_lists.restype = i64
        _lib = L
    return _lib


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t))


def _f32(a, min_cols=3):
    a = np.ascontiguousarray(a, dtype=np.float32)
    assert a.ndim == 2 and a.shape[1] >= min_cols
    return a


def num_threads() -> int:
    return int(lib().orc_desc_num_threads())


def colpiv_qr_solve(A, b):
    """x = A.colPivHouseholderQr().solve(b) for one 3x3 fp32 system (Eigen 3.3 restated)."""
    A = np.ascontiguousarray(np.asarray(A, np.float32).T)       # column-major
    b = np.ascontiguousarray(b, np.float32)
    x = np.empty(3, np.float32)
    lib().orc_colpiv_qr_solve3(_p(A, C.c_float), _p(b, C.c_float), _p(x, C.c_float))
    return x


def rgb_to_intensity(rgb):
    rgb = np.ascontiguousarray(rgb, np.uint8).reshape(-1, 3)
    out = np.empty(rgb.shape[0], np.float32)
    lib().orc_rgb_to_intensity(_p(rgb, C.c_uint8), rgb.shape[0], _p(out, C.c_float))
    return out


def intensity_gradient(pts, offsets, nbr, intensity, normals):
    """IntensityGradientEstimation over the radius rows (offsets, nbr) of one query each; normals[nq, >=3] of the queries."""
    pts = _f32(pts)
    offsets = np.ascontiguousarray(offsets, np.int64)
    nbr = np.ascontiguousarray(nbr, np.int32).reshape(-1)
    intensity = np.ascontiguousarray(intensity, np.float32).reshape(-1)
    nq = offsets.shape[0] - 1
    nrm = np.zeros((nq, 4), np.float32)
    nrm[:, :3] = np.asarray(normals, np.float32)[:, :3]
    out = np.empty((nq, 4), np.float32)
    lib().orc_intensity_gradient_from_lists(_p(pts, C.c_float), pts.shape[1], _p(intensity, C.c_float), _p(nrm, C.c_float), nq,
                                            _p(offsets, C.c_int64), _p(nbr, C.c_int32), _p(out, C.c_float))
    return out


def rift(pts, qpts, offsets, nbr, d2, gradients, radius: float, nr_distance_bins: int = 4, nr_gradient_bins: int = 8):
    """RIFTEstimation over the radius rows (offsets, nbr, d2) of the queries qpts; gradients[n_surface, >=3]."""
    pts, qpts = _f32(pts), _f32(qpts)
    offsets = np.ascontiguousarray(offsets, np.int64)
    nbr = np.ascontiguousarray(nbr, np.int32).reshape(-1)
    d2 = np.ascontiguousarray(d2, np.float32).reshape(-1)
    g = np.zeros((np.asarray(gradients).shape[0], 4), np.float32)
    g[:, :3] = np.asarray(gradients, np.float32)[:, :3]
    nb = nr_distance_bins * nr_gradient_bins
    out = np.empty((qpts.shape[0], max(nb, 1)), np.float32)
    rc = lib().orc_rift_from_lists(_p(pts, C.c_float), pts.shape[1], _p(qpts, C.c_float), qpts.shape[0], qpts.shape[1], _p(offsets, C.c_int64),
                                   _p(nbr, C.c_int32), _p(d2, C.c_float), _p(g, C.c_float), float(radius), int(nr_distance_bins),
                                   int(nr_gradient_bins), _p(out, C.c_float))
    if rc != 0:
        raise ValueError(f"nr_distance_bins * nr_gradient_bins = {nb} is outside 1..32")
    return out


def process_rift(xyz, rgb, normal_radius=0.03, gradient_radius=0.03, rift_radius=0.05, nr_distance_bins=4, nr_gradient_bins=8, stages=None):
    """processRIFT (src/comparator.cpp:590-684) on the CPU: intensity -> normals r 0.03 -> drop NaN normals -> gradient r 0.03
    -> RIFT r 0.05 -> drop non-finite descriptors, both later stages over the filtered cloud.  Returns (descriptors, kept_rows);
    `stages` (a dict) receives the intermediate arrays."""
    import oracle
    xyz = np.ascontiguousarray(np.asarray(xyz, np.float32)[:, :3])
    inten = rgb_to_intensity(rgb)
    normals = oracle.normals_radius(xyz, normal_radius)
    keep1 = np.flatnonzero(np.isfinite(normals[:, :3]).all(1))
    xyz1, inten1, nrm1 = xyz[keep1], inten[keep1], normals[keep1]
    tree = oracle.KdTree(xyz1)
    off, idx, _ = tree.radius(xyz1, gradient_radius)
    grad = intensity_gradient(xyz1, off, idx, inten1, nrm1)
    off, idx, d2 = tree.radius(xyz1, rift_radius)
    desc = rift(xyz1, xyz1, off, idx, d2, grad, rift_radius, nr_distance_bins, nr_gradient_bins)
    keep2 = np.flatnonzero(np.isfinite(desc).all(1))
    if stages is not None:
        stages.update(intensity=inten, normals=normals, kept_normals=keep1, gradients=grad, descriptors_all=desc)
    return desc[keep2], keep1[keep2]


def sift_expf(x):
    """The fp64-evaluated expf both the oracle and the kernels use for SIFT's Gaussian weights (float32 in, float32 out)."""
    x = np.ascontiguousarray(x, np.float32).reshape(-1)
    out = np.empty_like(x)
    lib().orc_sift_expf(_p(x, C.c_float), x.size, _p(out, C.c_float))
    return out


def sift_scales(base_scale: float, nr_scales_per_octave: int):
    """One octave's scale table, float32[nr_scales_per_octave + 3], with PCL's powf."""
    out = np.empty(int(nr_scales_per_octave) + 3, np.float32)
    lib().orc_sift_scales(float(np.float32(base_scale)), int(nr_scales_per_octave), _p(out, C.c_float))
    return out


def sift_field_values(rgb):
    """SIFTKeypointFieldSelector<PointXYZRGB>: float(299 r + 587 g + 114 b) / 1000.0f; rgb[n, 3] uint8."""
    rgb = np.ascontiguousarray(rgb, np.uint8).reshape(-1, 3)
    out = np.empty(rgb.shape[0], np.float32)
    lib().orc_sift_field_values(_p(rgb, C.c_uint8), rgb.shape[0], _p(out, C.c_float))
    return out


def sift_dog(values, offsets, nbr, d2, scales):
    """computeScaleSpace over sorted radius rows (offsets, nbr, d2) at 3.0f * scales[-1]: float32[nq, len(scales) - 1]."""
    values = np.ascontiguousarray(values, np.float32).reshape(-1)
    offsets = np.ascontiguousarray(offsets, np.int64)
    nbr = np.ascontiguousarray(nbr, np.int32).reshape(-1)
    d2 = np.ascontiguousarray(d2, np.float32).reshape(-1)
    scales = np.ascontiguousarray(scales, np.float32)
    nq = offsets.shape[0] - 1
    out = np.empty((nq, scales.size - 1), np.float32)
    lib().orc_sift_dog_from_lists(_p(values, C.c_float), nq, _p(offsets, C.c_int64), _p(nbr, C.c_int32), _p(d2, C.c_float),
                                  _p(scales, C.c_float), scales.size, _p(out, C.c_float))
    return out


def sift_extrema(dog, nn, min_contrast: float = 0.001):
    """findScaleSpaceExtrema over neighbour rows nn[n, k] (entries < 0 absent): (rows, columns) int32 in (row, column) order."""
    dog = np.ascontiguousarray(dog, np.float32)
    nn = np.ascontiguousarray(nn, np.int32)
    n, nc = dog.shape
    cap = max(n * max(nc - 2, 0), 1)
    rows, cols = np.empty(cap, np.int32), np.empty(cap, np.int32)
    m = lib().orc_sift_extrema_from_lists(_p(dog, C.c_float), n, nc, _p(nn, C.c_int32), nn.shape[1], float(min_contrast),
                                          _p(rows, C.c_int32), _p(cols, C.c_int32), cap)
    return rows[:m].copy(), cols[:m].copy()


def pack_rgb(xyz, rgb):
    """[n, 4] float32 rows (x, y, z, packed 0x00RRGGBB word), the layout the octave loop voxelises."""
    rgb = np.asarray(rgb, np.uint32).reshape(-1, 3)
    rows = np.empty((rgb.shape[0], 4), np.float32)
    rows[:, :3] = np.asarray(xyz, np.float32)[:, :3]
    rows[:, 3] = ((rgb[:, 0] << 16) | (rgb[:, 1] << 8) | rgb[:, 2]).view(np.float32)
    return rows


def unpack_rgb(rows):
    w = np.ascontiguousarray(rows[:, 3], np.float32).view(np.uint32)
    return np.stack([(w >> 16) & 255, (w >> 8) & 255, w & 255], 1).astype(np.uint8)


def sift_keypoints(xyz, rgb, min_scale=0.005, nr_octaves=5, nr_scales_per_octave=5, min_contrast=0.001, stages=None):
    """SIFTKeypoint<PointXYZRGB, PointWithScale>::compute (src/comparator.cpp:449-465) on the CPU: per octave oracle.voxel_grid of
    the previous octave's cloud, stop below 25 points, oracle.KdTree radius rows at 3 * scales[-1] -> DoG, k = 25 rows -> extrema.
    Returns float32[m, 4] = (x, y, z, scale); `stages` (a dict) receives a list of per-octave dicts."""
    import oracle
    cloud = pack_rgb(xyz, rgb)
    scale = np.float32(min_scale)
    out = []
    for octave in range(int(nr_octaves)):
        cloud = oracle.voxel_grid(cloud, scale, rgb_offset_floats=3)
        if cloud.shape[0] < 25:
            break
        scales = sift_scales(scale, nr_scales_per_octave)
        fin = np.isfinite(cloud[:, :3]).all(1)
        tree = oracle.KdTree(cloud)
        off, idx, d2 = tree.radius(cloud, float(np.float32(3.0) * scales[-1]))
        dog = sift_dog(sift_field_values(unpack_rgb(cloud)), off, idx, d2, scales)
        dog[~fin] = np.nan
        nn, _, _ = tree.knn(cloud, min(25, max(tree.size, 1)))
        nn[~fin] = -1
        rows, cols = sift_extrema(dog, nn, min_contrast)
        kp = np.empty((rows.size, 4), np.float32)
        kp[:, :3] = cloud[rows, :3]
        kp[:, 3] = scales[cols]
        out.append(kp)
        if stages is not None:
            stages.setdefault("octaves", []).append(dict(cloud=cloud, scales=scales, dog=dog, rows=rows, cols=cols, keypoints=kp))
        scale = np.float32(scale * np.float32(2))
    return np.concatenate(out) if out else np.empty((0, 4), np.float32)
