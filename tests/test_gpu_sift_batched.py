"""GPU parity of batched SIFT keypoint detection (pcc_sift_keypoints_batched, sift_keypoints_batched, process_sift_batched): every
cluster of a batch must get exactly what the per-cluster sift_keypoints / process_sift calls return and what the CPU oracle
(descriptor_oracle.sift_keypoints, oracle.first_within) computes on that cluster alone.  Bit-identity throughout: the extremum test is
== and strict <, so keypoint lists admit no tolerance.  Run on the B200 box with `-m gpu`."""
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
PCC_ERR_INVALID = -1                                                  # include/pcc/search.h


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


def _patch(n, radius, seed=41):
    base = (synth.room(60000, seed)[:, :3] * 0.12).astype(np.float32)
    a = base[np.flatnonzero(np.linalg.norm(base - base[0], axis=1) < radius)[:n]]
    return np.ascontiguousarray(a)


def _concat(clusters):
    """[(xyz, rgb), ...] -> (xyz, rgb, offsets)"""
    xyz = np.concatenate([c[0] for c in clusters] + [np.empty((0, 3), np.float32)]).astype(np.float32)
    rgb = np.concatenate([c[1] for c in clusters] + [np.empty((0, 3), np.uint8)]).astype(np.uint8)
    off = np.concatenate([[0], np.cumsum([c[0].shape[0] for c in clusters])]).astype(np.int64)
    return xyz, rgb, off


def shared_space():
    """one room patch split into three clusters by a seeded random label: every neighbourhood mixes clusters"""
    xyz = _patch(3000, 0.3)
    rgb = synth.rgb_for(xyz * 8, 61)
    lab = np.random.default_rng(62).integers(0, 3, xyz.shape[0])
    return _concat([(xyz[lab == c], rgb[lab == c]) for c in range(3)])


def scene():
    """the Euclidean clusters (tolerance 0.05, at least 100 points) of a synth.scene cloud after a 0.025 VoxelGrid, kept above 700
    points (the reference's -e path also removes planes first; that step is not part of this fixture)"""
    p = synth.scene(800000, 73, extent=14.0, n_objects=120)[0][:, :3].copy()
    v = np.ascontiguousarray(oracle.voxel_grid(p, np.float32(0.025))[:, :3])
    lab, sizes = oracle.KdTree(v).ece(0.05, 100, 10**9)
    rgb = synth.rgb_for(v, 74)
    keep = np.flatnonzero(sizes > 700)
    return _concat([(v[lab == c], rgb[lab == c]) for c in keep])


def edges():
    """a 700-point cluster (4 octaves) beside a 5000-point one (5), a 10-point cluster, an empty one, a 30 m cluster with NaN rows
    that VoxelGrid passes through, and a second 700-point cluster"""
    a7 = _patch(700, 0.12)
    a5 = _patch(5000, 0.4)
    tiny = _patch(10, 0.05)
    wide = synth.room(20000, 57, size=(30.0, 30.0, 3.0))[:, :3].astype(np.float32)
    wide[::1009] = np.nan
    b7 = _patch(700, 0.12, seed=45)
    return _concat([(a7, synth.rgb_for(a7 * 8, 43)), (a5, synth.rgb_for(a5 * 8, 44)), (tiny, synth.rgb_for(tiny, 46)),
                    (np.empty((0, 3), np.float32), np.empty((0, 3), np.uint8)), (wide, synth.rgb_for(np.nan_to_num(wide), 58)),
                    (b7, synth.rgb_for(b7 * 8, 47))])


BATCHES = {"shared-space": shared_space, "scene": scene, "edges": edges}
_cache = {}


def batch(name):
    if name not in _cache:
        _cache[name] = BATCHES[name]()
    return _cache[name]


def per_cluster_gpu(xyz, rgb, off):
    from pointcloudcomparator_b200.search import process_sift
    kps, snaps = [], []
    for c in range(off.size - 1):
        kp, sn = process_sift(xyz[off[c]:off[c + 1]], rgb[off[c]:off[c + 1]])
        kps.append(kp), snaps.append(sn)
    return kps, snaps


def per_cluster_oracle(xyz, rgb, off):
    kps, snaps, octaves = [], [], []
    for c in range(off.size - 1):
        x, r = xyz[off[c]:off[c + 1]], rgb[off[c]:off[c + 1]]
        if x.shape[0] == 0:
            kps.append(np.empty((0, 4), np.float32)), snaps.append(np.empty(0, np.int32)), octaves.append(0)
            continue
        st = {}
        kp = D.sift_keypoints(x, r, stages=st)
        kps.append(kp)
        snaps.append(oracle.first_within(x, np.ascontiguousarray(kp[:, :3]), 0.05) if kp.shape[0] else np.empty(0, np.int32))
        octaves.append(len(st.get("octaves", [])))             # no entry when the first VoxelGrid leaves fewer than 25 points
    return kps, snaps, octaves


def split(a, kp_off):
    return [a[kp_off[c]:kp_off[c + 1]] for c in range(kp_off.size - 1)]


def assert_per_cluster(kp, kp_off, snap, want_kp, want_snap):
    assert kp.dtype == np.float32 and kp_off[0] == 0 and kp_off[-1] == kp.shape[0] and (np.diff(kp_off) >= 0).all()
    assert len(want_kp) == kp_off.size - 1
    for c, (g, w) in enumerate(zip(split(kp, kp_off), want_kp)):
        assert g.shape == w.shape and np.array_equal(bits(g), bits(w)), f"cluster {c}: {g.shape[0]} keypoints, want {w.shape[0]}"
    if snap is not None:
        for c, (g, w) in enumerate(zip(split(snap, kp_off), want_snap)):
            assert g.dtype == np.int32 and np.array_equal(g, w), f"cluster {c}: snap differs"


@pytest.mark.parametrize("name", list(BATCHES))
def test_batched_equals_per_cluster_and_oracle(torch_cuda, name):
    from pointcloudcomparator_b200.search import process_sift_batched, sift_keypoints_batched
    xyz, rgb, off = batch(name)
    kp, kp_off, snap = process_sift_batched(xyz, rgb, off)
    g_kp, g_snap = per_cluster_gpu(xyz, rgb, off)
    assert_per_cluster(kp, kp_off, snap, g_kp, g_snap)
    o_kp, o_snap, octaves = per_cluster_oracle(xyz, rgb, off)
    assert_per_cluster(kp, kp_off, snap, o_kp, o_snap)
    kp2, kp_off2 = sift_keypoints_batched(xyz, rgb, off)
    assert np.array_equal(kp_off2, kp_off) and np.array_equal(bits(kp2), bits(kp))
    sizes = np.diff(off)
    print(f"{name}: {off.size - 1} clusters of {sizes.min()}..{sizes.max()} points, octaves {octaves}, {kp.shape[0]} keypoints, "
          f"{int((snap >= 0).sum())} snapped")
    assert kp.shape[0] > 0 and (snap >= 0).any()
    if name == "scene":
        assert ((sizes > 700) & (sizes <= 1500)).sum() >= 16
    if name == "edges":
        assert octaves[0] == 4 and octaves[1] == 5                   # the 700-point cluster retires one octave before its neighbour
        assert octaves[2] == 0 and kp_off[3] == kp_off[2]            # fewer than 25 points: the first VoxelGrid already ends it
        assert kp_off[4] == kp_off[3]                                # the empty cluster
        assert kp_off[5] > kp_off[4]                                 # the pass-through cluster has keypoints


def test_batch_of_one_equals_single_call(torch_cuda):
    from pointcloudcomparator_b200.search import sift_keypoints, sift_keypoints_batched
    xyz = _patch(5000, 0.4)
    rgb = synth.rgb_for(xyz * 8, 44)
    kp, kp_off = sift_keypoints_batched(xyz, rgb, [0, xyz.shape[0]])
    want = sift_keypoints(xyz, rgb)
    assert kp_off.tolist() == [0, want.shape[0]] and np.array_equal(bits(kp), bits(want))


def test_memory_kinds_and_streams(torch_cuda):
    torch = torch_cuda
    from pointcloudcomparator_b200.search import process_sift_batched
    xyz, rgb, off = batch("edges")
    kp, kp_off, snap = process_sift_batched(xyz, rgb, off)
    t = torch.as_tensor(xyz, device="cuda")
    dk, doff, dsnap = process_sift_batched(t, rgb, off)
    torch.cuda.synchronize()
    assert dk.is_cuda and dsnap.is_cuda
    assert np.array_equal(doff, kp_off) and np.array_equal(bits(dk.cpu().numpy()), bits(kp)) and np.array_equal(dsnap.cpu().numpy(), snap)
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        t2 = torch.as_tensor(xyz, device="cuda")
        sk, soff, ssnap = process_sift_batched(t2, rgb, off)
        sk_h, ssnap_h = sk.cpu(), ssnap.cpu()
    side.synchronize()
    assert np.array_equal(soff, kp_off) and np.array_equal(bits(sk_h.numpy()), bits(kp)) and np.array_equal(ssnap_h.numpy(), snap)


def _call(xyz, rgb, off, cap, out, snap, kp_off, min_scale=0.005, nr_scales=5):
    from pointcloudcomparator_b200 import _lib
    from pointcloudcomparator_b200.search import GridSearch, _sift_rows
    ws = GridSearch()
    rows = _sift_rows(xyz, rgb)
    off = np.ascontiguousarray(off, np.int64)
    rc = ws._L.pcc_sift_keypoints_batched(ws._h, rows.ctypes.data, rows.shape[0], 16, 12, off.ctypes.data, off.size - 1, float(min_scale), 5, int(nr_scales),
                                          0.001, 0.05, None if out is None else out.ctypes.data, None if snap is None else snap.ctypes.data, cap,
                                          kp_off.ctypes.data, _lib.HOST, None)
    return rc, ws


def test_cap_writes_leading_rows_and_full_offsets(torch_cuda):
    from pointcloudcomparator_b200.search import process_sift_batched
    xyz, rgb, off = batch("shared-space")
    kp, kp_off, snap = process_sift_batched(xyz, rgb, off)
    cap = int(kp_off[1]) + 2                                         # ends inside the second cluster
    assert kp.shape[0] > cap
    out = np.full((cap + 3, 4), -7.0, np.float32)
    sn = np.full(cap + 3, -9, np.int32)
    ko = np.full(off.size, -5, np.int64)
    rc, _ = _call(xyz, rgb, off, cap, out, sn, ko)
    assert rc == 0 and np.array_equal(ko, kp_off)
    assert np.array_equal(bits(out[:cap]), bits(kp[:cap])) and (out[cap:] == -7.0).all()
    assert np.array_equal(sn[:cap], snap[:cap]) and (sn[cap:] == -9).all()
    ko0 = np.full(off.size, -5, np.int64)
    rc, _ = _call(xyz, rgb, off, 0, None, None, ko0)                 # cap 0: counting only
    assert rc == 0 and np.array_equal(ko0, kp_off)


@pytest.mark.parametrize("bad", ["start", "end", "decrease", "scales14", "min_scale0"])
def test_argument_errors(torch_cuda, bad):
    xyz, rgb, off = batch("shared-space")
    off = off.copy()
    kw = {}
    if bad == "start":
        off[0] = 1
    elif bad == "end":
        off[-1] -= 1
    elif bad == "decrease":
        off[1], off[2] = off[2], off[1]
    elif bad == "scales14":
        kw["nr_scales"] = 14
    else:
        kw["min_scale"] = 0.0
    out = np.empty((16, 4), np.float32)
    ko = np.zeros(off.size, np.int64)
    rc, ws = _call(xyz, rgb, off, 16, out, None, ko, **kw)
    assert rc == PCC_ERR_INVALID
    assert ws._L.pcc_last_error()


def test_cpp_sift_batched_mirror(torch_cuda):
    exe = os.path.join(ROOT, "tests", "cpp", "test_sift_batched")
    assert os.path.exists(exe), "run __graft_entry__.build() first"
    out = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "PASS" in out.stdout, out.stdout + out.stderr
