"""ctypes binding of libpcc_search.so (the C ABI declared in include/pcc/search.h).

There is no fallback of any kind: if the shared library is missing or no sm_100 device is
usable, every entry point raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.abspath(os.environ["PCC_SO"]) if os.environ.get("PCC_SO") else os.path.join(_HERE, "libpcc_search.so")     # PCC_SO: developer builds from scripts/build_variant.sh

HOST, DEVICE = 0, 1
MAX_K = 512

_lib = None

# every symbol include/pcc/search.h declares (tests check the .so exports each one)
SYMBOLS = [
    "pcc_last_error", "pcc_version", "pcc_launch_count", "pcc_create", "pcc_destroy", "pcc_build", "pcc_size", "pcc_grid_info",
    "pcc_knn", "pcc_radius_count", "pcc_radius_fill", "pcc_knn_mean_dist", "pcc_sor_threshold", "pcc_normals_knn",
    "pcc_normals_radius", "pcc_icp_step", "pcc_icp_align", "pcc_umeyama_from_sums", "pcc_euclidean_labels", "pcc_first_within",
    "pcc_export", "pcc_adopt", "pcc_set_timing", "pcc_last_kernel_ms", "pcc_ece_init", "pcc_ece_link_range", "pcc_ece_absorb", "pcc_ece_finish", "pcc_voxel_grid", "pcc_descriptor_nn", "pcc_region_growing",
    "pcc_region_growing_rgb", "pcc_intensity_gradient", "pcc_rift", "pcc_sift_dog", "pcc_sift_extrema", "pcc_sift_keypoints", "pcc_comm_init", "pcc_comm_info", "pcc_broadcast_index", "pcc_gather", "pcc_allreduce_f64",
]


class PccError(RuntimeError):
    pass


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise PccError(f"{SO_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                       "(make -C pointcloudcomparator_b200/csrc); there is no CPU fallback")
    L = C.CDLL(SO_PATH)
    vp, i64, i32, dbl, u32 = C.c_void_p, C.c_int64, C.c_int, C.c_double, C.c_uint
    L.pcc_last_error.restype = C.c_char_p
    L.pcc_launch_count.restype = i64
    L.pcc_create.argtypes = [i32, C.POINTER(vp)]
    L.pcc_destroy.argtypes = [vp]
    L.pcc_destroy.restype = None
    L.pcc_build.argtypes = [vp, vp, i64, i32, vp, i64, C.c_float, i32, i32, vp]
    L.pcc_size.argtypes = [vp]
    L.pcc_size.restype = i64
    L.pcc_grid_info.argtypes = [vp, C.POINTER(dbl)]
    L.pcc_knn.argtypes = [vp, vp, i64, i32, i32, vp, vp, C.POINTER(i32), i32, vp]
    L.pcc_radius_count.argtypes = [vp, vp, i64, i32, dbl, u32, vp, C.POINTER(i64), i32, vp]
    L.pcc_radius_fill.argtypes = [vp, vp, i64, i32, dbl, u32, i32, vp, vp, vp, i32, vp]
    L.pcc_knn_mean_dist.argtypes = [vp, vp, i64, i32, i32, vp, i32, vp]
    L.pcc_sor_threshold.argtypes = [vp, vp, i64, i64, dbl, C.POINTER(dbl), vp, C.POINTER(i64), i32, vp]
    L.pcc_normals_knn.argtypes = [vp, vp, i64, i32, i32, C.POINTER(C.c_float), vp, i32, vp]
    L.pcc_normals_radius.argtypes = [vp, vp, i64, i32, dbl, C.POINTER(C.c_float), vp, i32, vp]
    L.pcc_intensity_gradient.argtypes = [vp, vp, i64, i32, dbl, vp, vp, vp, i32, vp]
    L.pcc_rift.argtypes = [vp, vp, i64, i32, dbl, vp, i32, i32, vp, i32, vp]
    L.pcc_sift_dog.argtypes = [vp, vp, vp, i32, vp, i32, vp]
    L.pcc_sift_extrema.argtypes = [vp, vp, i32, C.c_float, vp, vp, i64, C.POINTER(i64), i32, vp]
    L.pcc_sift_keypoints.argtypes = [vp, vp, i64, i32, i32, C.c_float, i32, i32, C.c_float, vp, i64, C.POINTER(i64), i32, vp]
    L.pcc_icp_step.argtypes = [vp, vp, i64, i32, C.POINTER(C.c_float), C.POINTER(dbl), C.POINTER(i64), vp, vp, i32, vp]
    L.pcc_icp_align.argtypes = [vp, vp, i64, i32, i32, C.POINTER(C.c_float), C.POINTER(i32), C.POINTER(dbl), C.POINTER(i32), i32, vp]
    L.pcc_umeyama_from_sums.argtypes = [C.POINTER(dbl), i64, C.POINTER(C.c_float)]
    L.pcc_euclidean_labels.argtypes = [vp, dbl, i64, i64, vp, C.POINTER(i64), vp, i64, i32, vp]
    L.pcc_first_within.argtypes = [vp, vp, i64, i32, dbl, vp, i32, vp]
    L.pcc_ece_init.argtypes = [vp, vp, vp]
    L.pcc_ece_link_range.argtypes = [vp, dbl, i64, i64, vp, vp]
    L.pcc_ece_absorb.argtypes = [vp, vp, vp, vp]
    L.pcc_ece_finish.argtypes = [vp, vp, i64, i64, vp, C.POINTER(i64), vp, i64, vp]
    L.pcc_voxel_grid.argtypes = [vp, vp, i64, i32, i32, C.POINTER(C.c_float), i32, vp, C.POINTER(i64), i32, vp]
    L.pcc_descriptor_nn.argtypes = [vp, vp, i64, vp, i64, i32, i32, vp, vp, i32, vp]
    L.pcc_region_growing.argtypes = [vp, i64, i32, vp, C.c_float, C.c_float, i64, i64, vp, C.POINTER(i64)]
    L.pcc_export.argtypes = [vp, C.POINTER(dbl), C.POINTER(vp)]
    L.pcc_adopt.argtypes = [vp, C.POINTER(dbl), vp]
    L.pcc_region_growing_rgb.argtypes = [vp, vp, i64, i32, vp, i32, C.c_float, C.c_float, C.c_float, i32, i64, i64, vp, C.POINTER(i64)]
    L.pcc_comm_init.argtypes = [vp, vp, i32, i32]
    L.pcc_comm_info.argtypes = [vp, C.POINTER(i32), C.POINTER(i32)]
    L.pcc_broadcast_index.argtypes = [vp, i32, vp]
    L.pcc_gather.argtypes = [vp, vp, i64, i32, vp, vp, i64, vp]
    L.pcc_allreduce_f64.argtypes = [vp, vp, i32, vp]
    L.pcc_set_timing.argtypes = [vp, i32]
    L.pcc_last_kernel_ms.argtypes = [vp]
    L.pcc_last_kernel_ms.restype = dbl
    _lib = L
    return L


def check(rc: int):
    if rc != 0:
        raise PccError(f"libpcc_search error {rc}: {lib().pcc_last_error().decode(errors='replace')}")
