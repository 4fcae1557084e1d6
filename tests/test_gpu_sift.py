"""GPU parity of SIFT keypoint detection (pcc_sift_dog, pcc_sift_extrema, pcc_sift_keypoints, process_sift) against the CPU oracle
(descriptor_oracle/ over oracle.KdTree rows), plus the C++ mirror self-test.  Every bar is bit-identity, NaN patterns included: the
extremum test is == and strict <, so keypoint lists admit no tolerance.  Run on the B200 box with `-m gpu`."""
import os
import subprocess

import numpy as np
import pytest

import descriptor_oracle as D
import oracle
from conftest import bits
from pointcloudcomparator_b200 import synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


def same(a, b):
    """bit-identical, NaN payloads aside"""
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    na, nb = np.isnan(a), np.isnan(b)
    return a.shape == b.shape and np.array_equal(na, nb) and np.array_equal(bits(np.where(na, 0, a)), bits(np.where(nb, 0, b)))


@pytest.fixture(scope="module")
def room():
    xyz = synth.room(100000, 51)[:, :3].copy()
    rgb = synth.rgb_for(xyz, 52)
    xyz[::997] = np.nan                                             # skipped by the index: NaN DoG rows
    return xyz, rgb


def _cluster(n, radius):
    base = (synth.room(60000, 41)[:, :3] * 0.12).astype(np.float32)
    a = base[np.flatnonzero(np.linalg.norm(base - base[0], axis=1) < radius)[:n]]
    return a, synth.rgb_for(a * 8, 43)


@pytest.mark.parametrize("base_scale", [0.005, 0.04])               # the octave-0 and octave-3 scale tables
def test_sift_dog_bit_identical(torch_cuda, room, base_scale):
    from pointcloudcomparator_b200.search import GridSearch, sift_field_values, sift_scales
    xyz, rgb = room
    scales = sift_scales(base_scale, 5)
    assert np.array_equal(scales, D.sift_scales(base_scale, 5))
    values = sift_field_values(rgb)
    r = float(np.float32(3) * scales[-1])
    off, idx, d2 = oracle.KdTree(xyz).radius(xyz, r)
    want = D.sift_dog(values, off, idx, d2, scales)
    bad = ~np.isfinite(xyz).all(1)
    want[bad] = np.nan
    s = GridSearch().setInputCloud(xyz, cell_hint=r)
    got = s.siftDoG(values, scales)
    assert same(got, want)
    assert np.isnan(got[bad]).all() and np.isfinite(got[~bad]).all() and (got[~bad] != 0).any()
    torch = torch_cuda
    sd = GridSearch().setInputCloud(torch.as_tensor(xyz, device="cuda"), cell_hint=r)
    gd = sd.siftDoG(torch.as_tensor(values, device="cuda"), scales)
    torch.cuda.synchronize()
    assert same(gd.cpu().numpy(), want)
    print(f"DoG at base scale {base_scale}: {xyz.shape[0]} rows, mean row {np.diff(off).mean():.1f}, bit-identical in host and device memory")


def test_sift_extrema_bit_identical(torch_cuda):
    from pointcloudcomparator_b200.search import GridSearch, sift_field_values
    xyz = synth.room(100000, 53)[:, :3]
    cloud = oracle.voxel_grid(D.pack_rgb(xyz, synth.rgb_for(xyz, 54)), np.float32(0.01), rgb_offset_floats=3)
    scales = D.sift_scales(0.01, 5)
    values = sift_field_values(D.unpack_rgb(cloud))
    tree = oracle.KdTree(cloud)
    off, idx, d2 = tree.radius(cloud, float(np.float32(3) * scales[-1]))
    dog = D.sift_dog(values, off, idx, d2, scales)
    nn, _, _ = tree.knn(cloud, 25)
    want_r, want_c = D.sift_extrema(dog, nn, 0.001)
    assert want_r.size > 100
    s = GridSearch().setInputCloud(cloud[:, :3].copy(), cell_hint=0.05)
    r, c = s.siftExtrema(dog, 0.001)                                 # the oracle's DoG: the kernel alone
    assert np.array_equal(r, want_r) and np.array_equal(c, want_c)
    own = s.siftDoG(values, scales)                                  # and the whole pair
    assert same(own, dog)
    r2, c2 = s.siftExtrema(own, 0.001)
    assert np.array_equal(r2, want_r) and np.array_equal(c2, want_c)
    torch = torch_cuda
    sd = GridSearch().setInputCloud(torch.as_tensor(cloud[:, :3].copy(), device="cuda"), cell_hint=0.05)
    rd, cd = sd.siftExtrema(torch.as_tensor(dog, device="cuda"), 0.001)
    assert np.array_equal(rd.cpu().numpy(), want_r) and np.array_equal(cd.cpu().numpy(), want_c)
    print(f"extrema over {cloud.shape[0]} octave points: {want_r.size} keypoints, identical lists")


def _clouds():
    a7, c7 = _cluster(700, 0.12)
    a5, c5 = _cluster(5000, 0.4)
    room = synth.room(100000, 55)[:, :3].copy()
    wide = synth.room(60000, 57, size=(30.0, 30.0, 3.0))[:, :3].copy()      # 30 m: VoxelGrid's leaf-too-small pass-through
    wide[::1009] = np.nan
    return [("cluster-700", a7, c7), ("cluster-5000", a5, c5), ("room-100k", room, synth.rgb_for(room, 56)),
            ("wide-30m", wide, synth.rgb_for(np.nan_to_num(wide), 58))]


@pytest.mark.parametrize("case", range(4))
def test_sift_keypoints_identical(torch_cuda, case):
    from pointcloudcomparator_b200.search import sift_keypoints
    label, xyz, rgb = _clouds()[case]
    st_o, st_g = {}, {}
    want = D.sift_keypoints(xyz, rgb, stages=st_o)
    got = sift_keypoints(xyz, rgb, stages=st_g)
    sizes = [o["cloud"].shape[0] for o in st_o["octaves"]]
    print(f"{label}: {xyz.shape[0]} points, octaves {sizes}, {want.shape[0]} keypoints")
    assert got.dtype == np.float32 and got.shape == want.shape and np.array_equal(bits(got), bits(want))
    assert [o["cloud"].shape[0] for o in st_g["octaves"]] == sizes
    for og, oo in zip(st_g["octaves"], st_o["octaves"]):
        assert np.array_equal(og["scales"], oo["scales"]) and same(og["dog"], oo["dog"])
        assert np.array_equal(og["rows"], oo["rows"]) and np.array_equal(og["cols"], oo["cols"])
    assert np.array_equal(np.concatenate([o["keypoints"] for o in st_g["octaves"]] + [np.empty((0, 4), np.float32)]), got)
    if label == "cluster-700":
        assert len(sizes) == 4                                       # 5 octaves asked, the fifth grid has < 25 points
    if label == "wide-30m":
        assert sizes[0] == xyz.shape[0]                              # octave 0 passed the cloud through unfiltered, NaN rows included
    assert want.shape[0] > 0


def test_sift_keypoints_cap_and_arguments(torch_cuda):
    import ctypes as C
    from pointcloudcomparator_b200._lib import HOST, PccError
    from pointcloudcomparator_b200.search import GridSearch, _sift_rows, sift_keypoints
    xyz, rgb = _cluster(5000, 0.4)
    full = sift_keypoints(xyz, rgb)
    ws = GridSearch()
    rows = _sift_rows(xyz, rgb)
    out = np.full((5, 4), -7.0, np.float32)
    found = C.c_int64()
    rc = ws._L.pcc_sift_keypoints(ws._h, rows.ctypes.data, rows.shape[0], 16, 12, 0.005, 5, 5, 0.001, out.ctypes.data, 3, C.byref(found), HOST, None)
    assert rc == 0 and found.value == full.shape[0] > 3
    assert np.array_equal(out[:3], full[:3]) and (out[3:] == -7.0).all()
    with pytest.raises(PccError):
        sift_keypoints(xyz, rgb, nr_scales_per_octave=14)
    with pytest.raises(PccError):
        sift_keypoints(xyz, rgb, min_scale=0.0)


def test_process_sift_snap(torch_cuda):
    from pointcloudcomparator_b200.search import process_sift
    xyz, rgb = _cluster(5000, 0.4)
    kp, snap = process_sift(xyz, rgb)
    assert np.array_equal(bits(kp), bits(D.sift_keypoints(xyz, rgb)))
    assert np.array_equal(snap, oracle.first_within(xyz, np.ascontiguousarray(kp[:, :3]), 0.05))
    assert kp.shape[0] > 0 and snap.dtype == np.int32 and (snap >= 0).any()


def test_cpp_sift_mirror(torch_cuda):
    exe = os.path.join(ROOT, "tests", "cpp", "test_sift")
    assert os.path.exists(exe), "run __graft_entry__.build() first"
    out = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "PASS" in out.stdout, out.stdout + out.stderr
