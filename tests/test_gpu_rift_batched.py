"""GPU parity of batched processRIFT (pcc_rift_batched, process_rift_batched): every cluster of a batch must get exactly what the
per-cluster process_rift returns on that cluster alone, bit for bit (same kernels over the same rows in the same order), and the same
shapes and kept rows as the CPU oracle (descriptor_oracle.process_rift; GPU normals are within 1e-5 of the oracle's, not bit-equal, so
the bins are compared with a printed difference).  Run on the B200 box with `-m gpu`."""
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
    return np.ascontiguousarray(base[np.flatnonzero(np.linalg.norm(base - base[0], axis=1) < radius)[:n]])


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
    """the Euclidean clusters (tolerance 0.05) of 100 to 700 points of a synth.scene cloud after a 0.025 VoxelGrid: the clusters
    computeSimilarity sends through processRIFT"""
    p = synth.scene(800000, 73, extent=14.0, n_objects=120)[0][:, :3].copy()
    v = np.ascontiguousarray(oracle.voxel_grid(p, np.float32(0.025))[:, :3])
    lab, sizes = oracle.KdTree(v).ece(0.05, 100, 10**9)
    rgb = synth.rgb_for(v, 74)
    keep = np.flatnonzero(sizes <= 700)
    return _concat([(v[lab == c], rgb[lab == c]) for c in keep])


def sparse():
    """a thin cluster: many points have fewer than 3 neighbours at 0.03 (dropped at the normals) or NaN gradients (dropped at the end)"""
    return _patch(3000, 0.3, 47)[::9]


def edges():
    """an empty, a 1-point and a 2-point cluster, a cluster with NaN rows, the sparse cluster, and two clusters 1 km apart (the union's
    extent forces the grid's 2048-cell cap, so cells are far larger than the radius)"""
    a = _patch(700, 0.12)
    nan = _patch(700, 0.12, 45).copy()
    nan[::37] = np.nan
    sp = sparse()
    far = _patch(400, 0.12, 49) + np.float32([1000.0, 0, 0])
    near = _patch(400, 0.12, 51)
    rgb = lambda x, s: synth.rgb_for(np.nan_to_num(x) * 8, s)            # noqa: E731
    e = np.empty((0, 3), np.float32)
    return _concat([(e, rgb(e, 1)), (a[:1], rgb(a[:1], 2)), (a[:2], rgb(a[:2], 3)), (nan, rgb(nan, 4)), (sp, rgb(sp, 5)), (near, rgb(near, 6)),
                    (far, rgb(far, 7)), (a, rgb(a, 8))])


BATCHES = {"shared-space": shared_space, "scene": scene, "edges": edges}
_cache = {}


def batch(name):
    if name not in _cache:
        _cache[name] = BATCHES[name]()
    return _cache[name]


def split(a, off):
    return [a[off[c]:off[c + 1]] for c in range(off.size - 1)]


def assert_per_cluster_gpu(desc, d_off, kept, xyz, rgb, off, **kw):
    from pointcloudcomparator_b200.search import process_rift
    assert desc.dtype == np.float32 and kept.dtype == np.int64 and d_off[0] == 0 and d_off[-1] == desc.shape[0] and (np.diff(d_off) >= 0).all()
    assert d_off.size == off.size
    for c, (dg, kg) in enumerate(zip(split(desc, d_off), split(kept, d_off))):
        x, r = xyz[off[c]:off[c + 1]], rgb[off[c]:off[c + 1]]
        if x.shape[0] < 3:                  # no point has the 3 neighbours a normal needs: nothing survives (and process_rift has no
            assert dg.shape[0] == 0         # filtered cloud to index)
            continue
        dw, kw_ = process_rift(x, r, **kw)
        assert dg.shape == dw.shape and np.array_equal(kg, kw_), f"cluster {c}: {dg.shape[0]} descriptors, alone {dw.shape[0]}"
        assert np.array_equal(bits(dg), bits(dw)), f"cluster {c}: descriptors differ"


def assert_per_cluster_oracle(desc, d_off, kept, xyz, rgb, off, name):
    worst = 0.0
    for c, (dg, kg) in enumerate(zip(split(desc, d_off), split(kept, d_off))):
        x, r = xyz[off[c]:off[c + 1]], rgb[off[c]:off[c + 1]]
        if x.shape[0] == 0 or not np.isfinite(x).all():           # the oracle's KdTree takes finite clouds only
            continue
        do, ko = D.process_rift(x, r)
        assert dg.shape == do.shape and np.array_equal(kg, ko), f"cluster {c}: {dg.shape[0]} descriptors, oracle {do.shape[0]}"
        if dg.size:
            worst = max(worst, float(np.abs(dg - do).max()))
    print(f"{name}: max per-bin |batched gpu - oracle| = {worst:.3g}")


@pytest.mark.parametrize("name", list(BATCHES))
def test_batched_equals_per_cluster_and_oracle(torch_cuda, name):
    from pointcloudcomparator_b200.search import process_rift_batched
    xyz, rgb, off = batch(name)
    desc, d_off, kept = process_rift_batched(xyz, rgb, off)
    assert desc.shape[1] == 32
    assert_per_cluster_gpu(desc, d_off, kept, xyz, rgb, off)
    assert_per_cluster_oracle(desc, d_off, kept, xyz, rgb, off, name)
    sizes = np.diff(off)
    print(f"{name}: {off.size - 1} clusters of {sizes.min()}..{sizes.max()} points, {desc.shape[0]} descriptors")
    assert desc.shape[0] > 0
    if name == "scene":
        assert off.size - 1 >= 16 and sizes.min() >= 100 and sizes.max() <= 700
    if name == "edges":
        assert d_off[1] == d_off[0] and d_off[2] == d_off[1] and d_off[3] == d_off[2]      # empty, 1 and 2 points: no descriptor
        assert d_off[4] > d_off[3] and d_off[7] > d_off[6]                                 # the NaN-row cluster and the far cluster
        # the sparse cluster drops points at the normals that lie within the RIFT radius of kept points, and drops rows at the end
        sp = sparse()
        st = {}
        dw, kw_ = D.process_rift(sp, rgb[off[4]:off[5]], stages=st)
        k1 = st["kept_normals"]
        dropped = np.setdiff1d(np.arange(sp.shape[0]), k1)
        assert dropped.size > 0 and kw_.size < k1.size
        assert oracle.KdTree(sp[dropped]).radius(np.ascontiguousarray(sp[k1]), 0.05)[0][-1] > 0


def test_union_grid_is_capped(torch_cuda):
    """the far pair makes the union 1 km wide: the grid hits its 2048-cell cap, cells grow far past the radius"""
    xyz, rgb, off = batch("edges")
    rc, ws, ko = _call(xyz, rgb, off, 0, None, None)
    assert rc == 0
    info = ws.grid_info()
    assert max(info["dims"]) <= 2048 and info["cell"] > 0.4, info


def test_batch_of_one_equals_single_call(torch_cuda):
    from pointcloudcomparator_b200.search import process_rift, process_rift_batched
    xyz = _patch(700, 0.12)
    rgb = synth.rgb_for(xyz * 8, 43)
    desc, d_off, kept = process_rift_batched(xyz, rgb, [0, xyz.shape[0]])
    dw, kw = process_rift(xyz, rgb)
    assert d_off.tolist() == [0, dw.shape[0]] and np.array_equal(kept, kw) and np.array_equal(bits(desc), bits(dw))


def test_bins_3x7(torch_cuda):
    from pointcloudcomparator_b200.search import process_rift_batched
    xyz, rgb, off = batch("shared-space")
    desc, d_off, kept = process_rift_batched(xyz, rgb, off, nr_distance_bins=3, nr_gradient_bins=7)
    assert desc.shape[1] == 21
    assert_per_cluster_gpu(desc, d_off, kept, xyz, rgb, off, nr_distance_bins=3, nr_gradient_bins=7)


def test_memory_kinds_and_streams(torch_cuda):
    torch = torch_cuda
    from pointcloudcomparator_b200.search import process_rift_batched
    xyz, rgb, off = batch("edges")
    desc, d_off, kept = process_rift_batched(xyz, rgb, off)
    t = torch.as_tensor(xyz, device="cuda")
    dd, doff, dk = process_rift_batched(t, rgb, off)
    torch.cuda.synchronize()
    assert dd.is_cuda and dk.is_cuda and dk.dtype == torch.int64
    assert np.array_equal(doff, d_off) and np.array_equal(bits(dd.cpu().numpy()), bits(desc)) and np.array_equal(dk.cpu().numpy(), kept)
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        t2 = torch.as_tensor(xyz, device="cuda")
        sd, soff, sk = process_rift_batched(t2, rgb, off)
        sd_h, sk_h = sd.cpu(), sk.cpu()
    side.synchronize()
    assert np.array_equal(soff, d_off) and np.array_equal(bits(sd_h.numpy()), bits(desc)) and np.array_equal(sk_h.numpy(), kept)


def _call(xyz, rgb, off, cap, out, rows, n=None, n_clouds=None, radii=(0.03, 0.03, 0.05), bins=(4, 8)):
    from pointcloudcomparator_b200 import _lib
    from pointcloudcomparator_b200.search import GridSearch, rgb_to_intensity
    ws = GridSearch()
    xyz = np.ascontiguousarray(xyz, np.float32)
    inten = rgb_to_intensity(rgb)
    off = np.ascontiguousarray(off, np.int64)
    ko = np.full(off.size, -5, np.int64)
    rc = ws._L.pcc_rift_batched(ws._h, xyz.ctypes.data, xyz.shape[0] if n is None else n, 12, inten.ctypes.data, off.ctypes.data,
                                off.size - 1 if n_clouds is None else n_clouds, *[float(r) for r in radii], int(bins[0]), int(bins[1]),
                                None if out is None else out.ctypes.data, None if rows is None else rows.ctypes.data, cap, ko.ctypes.data, _lib.HOST, None)
    return rc, ws, ko


def test_cap_writes_leading_rows_and_full_offsets(torch_cuda):
    from pointcloudcomparator_b200.search import process_rift_batched
    xyz, rgb, off = batch("shared-space")
    desc, d_off, kept = process_rift_batched(xyz, rgb, off)
    cap = int(d_off[1]) + 2                                          # ends inside the second cluster
    assert desc.shape[0] > cap
    out = np.full((cap + 3, 32), -7.0, np.float32)
    rows = np.full(cap + 3, -9, np.int32)
    rc, _, ko = _call(xyz, rgb, off, cap, out, rows)
    assert rc == 0 and np.array_equal(ko, d_off)
    assert np.array_equal(bits(out[:cap]), bits(desc[:cap])) and (out[cap:] == -7.0).all()
    assert np.array_equal(rows[:cap], kept[:cap]) and (rows[cap:] == -9).all()
    rc, _, ko0 = _call(xyz, rgb, off, 0, None, None)                 # cap 0: counting only
    assert rc == 0 and np.array_equal(ko0, d_off)


@pytest.mark.parametrize("bad", ["start", "end", "decrease", "n_clouds", "n", "radius_nan", "radius_neg", "radius_inf", "bins0", "bins33"])
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
    elif bad == "n_clouds":
        kw["n_clouds"] = (1 << 24) + 1
    elif bad == "n":
        kw["n"] = (1 << 31) - 1
    elif bad == "radius_nan":
        kw["radii"] = (0.03, float("nan"), 0.05)
    elif bad == "radius_neg":
        kw["radii"] = (-0.03, 0.03, 0.05)
    elif bad == "radius_inf":
        kw["radii"] = (0.03, 0.03, float("inf"))
    elif bad == "bins0":
        kw["bins"] = (0, 8)
    else:
        kw["bins"] = (4, 9)
    out = np.empty((16, 32), np.float32)
    rows = np.empty(16, np.int32)
    rc, ws, _ = _call(xyz, rgb, off, 16, out, rows, **kw)
    assert rc == PCC_ERR_INVALID
    assert ws._L.pcc_last_error()


def test_fixed_cost_does_not_grow_with_cluster_count(torch_cuda):
    """the same launches for 8 and for 64 clusters of 700 points: one build, one sorted pass, three reductions, one compaction"""
    from pointcloudcomparator_b200.search import launch_count, process_rift_batched
    a = _patch(700, 0.12)
    rgb = synth.rgb_for(a * 8, 43)

    def tiles(k):
        return _concat([(a + np.float32([0.5 * (i % 8), 0.5 * (i // 8), 0]), rgb) for i in range(k)])

    deltas = []
    for k in (8, 64):
        xyz, rg, off = tiles(k)
        process_rift_batched(xyz, rg, off)                           # warm-up
        before = launch_count()
        desc, d_off, _ = process_rift_batched(xyz, rg, off)
        deltas.append(launch_count() - before)
        assert d_off.size == k + 1 and (np.diff(d_off) > 0).all()
    print(f"launches per call: 8 clusters {deltas[0]}, 64 clusters {deltas[1]}")
    assert deltas[0] == deltas[1]


def test_cpp_rift_batched_mirror(torch_cuda):
    exe = os.path.join(ROOT, "tests", "cpp", "test_rift_batched")
    assert os.path.exists(exe), "run __graft_entry__.build() first"
    out = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "PASS" in out.stdout, out.stdout + out.stderr
