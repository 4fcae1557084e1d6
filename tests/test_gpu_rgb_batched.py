"""GPU parity of batched colour segmentation (pcc_knn_batched / knn_batched, pcc_region_growing_rgb_batched / region_growing_rgb_batched):
every cluster of a batch must get exactly what the per-cluster calls return on that cluster alone -- the N x k table bit for bit (cluster-
local indices, d2 bits, (d2, index) order, (-1, +inf) padding) and the same colour labels and counts -- and the same as the CPU oracle's
tables where the oracle applies.  Run on the B200 box with `-m gpu`."""
import os
import subprocess

import numpy as np
import pytest

import oracle
from conftest import bits
from oracle import rgb_region_growing
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


def _rgb(x, seed):
    return synth.rgb_for(np.nan_to_num(x) * 8, seed)


def shared_space():
    """one room patch split into three clusters by a seeded random label: every neighbourhood mixes clusters"""
    xyz = _patch(3000, 0.3)
    rgb = _rgb(xyz, 61)
    lab = np.random.default_rng(62).integers(0, 3, xyz.shape[0])
    return _concat([(xyz[lab == c], rgb[lab == c]) for c in range(3)])


def _scene_clusters():
    """computeSimilarity's clusters of a synth.scene cloud: 0.025 VoxelGrid, then RegionGrowing (k = 100 table, k = 50 normals, 3 degrees,
    curvature 1, at least 50 points; src/segmentation.cpp:223-271), on the CPU oracle"""
    p = synth.scene(400000, 73, extent=10.0, n_objects=60)[0][:, :3].copy()
    v = np.ascontiguousarray(oracle.voxel_grid(p, np.float32(0.025))[:, :3])
    tree = oracle.KdTree(v)
    nb, _, _ = tree.knn(v, 100)
    lab, nc = oracle.region_growing(nb, oracle.normals_knn(v, 50, tree=tree), 3.0 / 180.0 * np.pi, 1.0, 50, 1000000)
    return v, [np.flatnonzero(lab == c) for c in range(nc)]


def scene():
    v, members = _scene_clusters()
    rgb = synth.rgb_for(v, 74)
    return _concat([(v[m], rgb[m]) for m in members])


def overlap():
    """both clouds of every matched pair in one call: the scene's clusters and the same clusters of a noisy copy, which overlap them in
    space, so half of every visited point belongs to the other cloud"""
    v, members = _scene_clusters()
    w = synth.noisy_copy(v, 75, 0.002)[:, :3]
    rgb, rgb2 = synth.rgb_for(v, 74), synth.rgb_for(v, 76)
    return _concat([(v[m], rgb[m]) for m in members] + [(w[m], rgb2[m]) for m in members])


def edges():
    """an empty, a 1-, a 2- and a 60-point cluster, a cluster with NaN rows, an all-NaN cluster, one point set split into two clusters
    (every point has an exact duplicate in the other, which must never appear), a lattice (ties broken by index), and two clusters 1 km
    apart (the union's extent forces the grid's 2048-cell cap)"""
    a = _patch(700, 0.12)
    nan = _patch(700, 0.12, 45).copy()
    nan[::37] = np.nan
    allnan = np.full((5, 3), np.nan, np.float32)
    dup = _patch(300, 0.12, 47)
    g = np.arange(6, dtype=np.float32) * np.float32(0.25)                  # exact coordinates: exactly tied distances
    lattice = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3) + np.float32([3.0, 0.0, 0.0])
    far = _patch(400, 0.12, 49) + np.float32([1000.0, 0, 0])
    near = _patch(400, 0.12, 51)
    e = np.empty((0, 3), np.float32)
    parts = [e, a[:1], a[:2], a[:60], nan, allnan, dup, dup[::-1].copy(), lattice, near, far, a]
    return _concat([(x, _rgb(x, 10 + i)) for i, x in enumerate(parts)])


BATCHES = {"shared-space": shared_space, "scene": scene, "overlap": overlap, "edges": edges}
SMALL = ("shared-space", "edges")
_cache = {}


def batch(name):
    if name not in _cache:
        _cache[name] = BATCHES[name]()
    return _cache[name]


def pack(rgb):
    c = np.asarray(rgb).reshape(-1, 3).astype(np.uint32)
    return (c[:, 0] << 16) | (c[:, 1] << 8) | c[:, 2]


def alone(x, k):
    """pcc_knn(q = NULL, k) on one cluster: (idx, d2, k_eff)"""
    from pointcloudcomparator_b200.search import GridSearch
    if not np.isfinite(x).all(1).any():                      # nothing to index: every row is empty
        return np.full((x.shape[0], k), -1, np.int32), np.full((x.shape[0], k), np.inf, np.float32), 0
    return GridSearch().setInputCloud(np.ascontiguousarray(x), k_hint=k).nearestKSearch(None, k)


@pytest.mark.parametrize("k", [1, 16, 25, 100, 300])
@pytest.mark.parametrize("name", list(BATCHES))
def test_knn_batched_equals_per_cluster(torch_cuda, name, k):
    from pointcloudcomparator_b200.search import knn_batched
    xyz, _, off = batch(name)
    idx, d2, k_eff = knn_batched(xyz, off, k)
    assert idx.shape == (xyz.shape[0], k) and d2.shape == idx.shape and k_eff.shape == (off.size - 1,)
    for c in range(off.size - 1):
        x = xyz[off[c]:off[c + 1]]
        if x.shape[0] == 0:
            assert k_eff[c] == 0
            continue
        ai, ad, ak = alone(x, k)
        assert k_eff[c] == ak == min(k, int(np.isfinite(x).all(1).sum())), f"cluster {c}: k_eff {k_eff[c]}, alone {ak}"
        gi, gd = idx[off[c]:off[c + 1]], d2[off[c]:off[c + 1]]
        assert np.array_equal(gi, ai) and np.array_equal(bits(gd), bits(ad)), f"cluster {c} ({x.shape[0]} points): rows differ"
        assert ((gi == -1) | ((gi >= 0) & (gi < x.shape[0]))).all()
        if k == 100 and np.isfinite(x).all():
            oi, od, _ = oracle.KdTree(x).knn(x, k)
            assert np.array_equal(gi, oi) and np.array_equal(bits(gd), bits(od)), f"cluster {c}: rows differ from the oracle"
    sizes = np.diff(off)
    print(f"{name} k={k}: {off.size - 1} clusters of {sizes.min()}..{sizes.max()} points")


def test_edges_batch_is_what_it_claims(torch_cuda):
    """the duplicates never cross, the lattice has ties, NaN rows are empty, the union grid is at its cap"""
    from pointcloudcomparator_b200.search import GridSearch, knn_batched
    xyz, _, off = batch("edges")
    ws = GridSearch()
    idx, d2, k_eff = knn_batched(xyz, off, 16, workspace=ws)
    assert k_eff.tolist()[:6] == [0, 1, 2, 16, 16, 0]
    d6, d7 = idx[off[6]:off[7]], idx[off[7]:off[8]]
    n6 = off[7] - off[6]
    assert (d2[off[6]:off[8], 0] == 0).all() and (d2[off[6]:off[8], 1] > 0).all()      # each duplicate sees itself at 0, not its twin
    assert (d6[:, 0] == np.arange(n6)).all() and (d7[:, 0] == np.arange(n6)).all()
    lat = d2[off[8]:off[9]]
    assert (lat[:, 1:] == lat[:, :-1]).any()                                           # tied distances inside rows
    bad = ~np.isfinite(xyz).all(1)
    assert (idx[bad] == -1).all() and np.isinf(d2[bad]).all()
    info = ws.grid_info()
    assert max(info["dims"]) <= 2048 and info["cell"] > 0.4, info


def assert_rgb_per_cluster(labels, counts, xyz, rgb, off, with_oracle, **kw):
    from pointcloudcomparator_b200.search import region_growing_rgb
    k = kw.pop("k", 100)
    for c in range(off.size - 1):
        x, col = xyz[off[c]:off[c + 1]], pack(rgb[off[c]:off[c + 1]])
        if x.shape[0] == 0:
            assert counts[c] == 0
            continue
        ai, ad, _ = alone(x, k)
        lab, nc = region_growing_rgb(ai, ad, col, **kw)
        assert counts[c] == nc and np.array_equal(labels[off[c]:off[c + 1]], lab), f"cluster {c}: {counts[c]} colour clusters, alone {nc}"
        if with_oracle and np.isfinite(x).all():
            oi, od, _ = oracle.KdTree(x).knn(x, k)
            ol, onc = rgb_region_growing.extract(oi, od, col, kw.get("distance_threshold", 10.0), kw.get("point_color_threshold", 6.0),
                                                 kw.get("region_color_threshold", 5.0), kw.get("grow_neighbours", 30), None, kw.get("min_size", 200))
            assert onc == nc and np.array_equal(ol, lab), f"cluster {c}: differs from the oracle"


@pytest.mark.parametrize("min_size", [200, 20])
@pytest.mark.parametrize("name", list(BATCHES))
def test_region_growing_rgb_batched_equals_per_cluster(torch_cuda, name, min_size):
    from pointcloudcomparator_b200.search import region_growing_rgb_batched
    xyz, rgb, off = batch(name)
    labels, counts = region_growing_rgb_batched(xyz, rgb, off, min_size=min_size)
    assert labels.shape == (xyz.shape[0],) and counts.shape == (off.size - 1,)
    assert_rgb_per_cluster(labels, counts, xyz, rgb, off, name in SMALL, min_size=min_size)
    print(f"{name} min {min_size}: colour clusters per cluster {np.bincount(counts).tolist()}, {int((labels == -1).sum())} of {labels.size} points unlabelled")
    assert (counts >= 2).any() or (labels == -1).any()
    if name in ("scene", "overlap") and min_size == 200:            # the reference configuration splits clusters and drops points
        assert (counts >= 2).any() and (labels == -1).any()


def test_memory_kinds_streams_and_workspaces(torch_cuda):
    torch = torch_cuda
    from pointcloudcomparator_b200.search import GridSearch, knn_batched, region_growing_rgb_batched
    xyz, rgb, off = batch("edges")
    hi, hd, hk = knn_batched(xyz, off, 100)
    hl, hc = region_growing_rgb_batched(xyz, rgb, off, min_size=20)
    t = torch.as_tensor(xyz, device="cuda")
    di, dd, dk = knn_batched(t, off, 100)
    dl, dc = region_growing_rgb_batched(t, rgb, off, min_size=20)
    torch.cuda.synchronize()
    assert di.is_cuda and dd.is_cuda
    assert np.array_equal(di.cpu().numpy(), hi) and np.array_equal(bits(dd.cpu().numpy()), bits(hd)) and np.array_equal(dk, hk)
    assert np.array_equal(dl, hl) and np.array_equal(dc, hc)
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        t2 = torch.as_tensor(xyz, device="cuda")
        si, sd, sk = knn_batched(t2, off, 100)
        si_h, sd_h = si.cpu(), sd.cpu()
        sl, sc = region_growing_rgb_batched(t2, rgb, off, min_size=20)
    side.synchronize()
    assert np.array_equal(si_h.numpy(), hi) and np.array_equal(bits(sd_h.numpy()), bits(hd)) and np.array_equal(sk, hk)
    assert np.array_equal(sl, hl) and np.array_equal(sc, hc)
    # a workspace indexing another cloud (with its own kNN state) before the call, then two batched calls in a row on it
    ws = GridSearch().setInputCloud(synth.room(20000, 5)[:, :3], k_hint=16)
    ws.nearestKSearch(None, 16)
    wi, wd, wk = knn_batched(xyz, off, 100, workspace=ws)
    assert np.array_equal(wi, hi) and np.array_equal(bits(wd), bits(hd)) and np.array_equal(wk, hk)
    xs, rs, offs = batch("shared-space")
    si2, sd2, _ = knn_batched(xs, offs, 100)
    wi2, wd2, _ = knn_batched(xs, offs, 100, workspace=ws)
    assert np.array_equal(wi2, si2) and np.array_equal(bits(wd2), bits(sd2))
    wl, wc = region_growing_rgb_batched(xyz, rgb, off, min_size=20, workspace=ws)
    assert np.array_equal(wl, hl) and np.array_equal(wc, hc)


def test_workspace_self_queries_follow_the_batch(torch_cuda):
    """after a batched call the workspace indexes the concatenation: its self-queries (queries=None), size and input cloud describe the
    batch, whether the cloud it indexed before was larger or smaller, on host arrays and on CUDA tensors"""
    torch = torch_cuda
    from pointcloudcomparator_b200.search import GridSearch, knn_batched, region_growing_rgb_batched

    def alone_all(x, k=16):
        return GridSearch().setInputCloud(np.ascontiguousarray(x), k_hint=k).nearestKSearch(None, k)

    for before, name in ((20000, "edges"), (1000, "shared-space")):      # a larger, then a smaller cloud indexed before the batch
        xyz, rgb, off = batch(name)
        want = alone_all(xyz)
        for call in ("knn", "rgb"):
            ws = GridSearch().setInputCloud(synth.room(before, 5)[:, :3], k_hint=16)
            ws.nearestKSearch(None, 16)
            if call == "knn":
                knn_batched(xyz, off, 100, workspace=ws)
            else:
                region_growing_rgb_batched(xyz, rgb, off, workspace=ws)
            gi, gd, gk = ws.nearestKSearch(None, 16)
            assert ws.getInputCloud().shape[0] == xyz.shape[0] and ws.size == int(np.isfinite(xyz).all(1).sum())
            assert gi.shape == want[0].shape and np.array_equal(gi, want[0]) and np.array_equal(bits(gd), bits(want[1])) and gk == want[2], (name, call)
        t = torch.as_tensor(xyz, device="cuda")
        wsd = GridSearch().setInputCloud(torch.as_tensor(synth.room(before, 5)[:, :3], device="cuda"), k_hint=16)
        knn_batched(t, off, 100, workspace=wsd)
        di, dd, dk = wsd.nearestKSearch(None, 16)
        torch.cuda.synchronize()
        assert di.is_cuda and np.array_equal(di.cpu().numpy(), want[0]) and np.array_equal(bits(dd.cpu().numpy()), bits(want[1])) and dk == want[2]
    # an empty batch leaves the workspace as it was
    ws = GridSearch().setInputCloud(synth.room(1000, 5)[:, :3], k_hint=16)
    e = np.empty((0, 3), np.float32)
    knn_batched(e, [0, 0], 16, workspace=ws)
    region_growing_rgb_batched(e, np.empty((0, 3), np.uint8), [0], workspace=ws)
    assert ws.getInputCloud().shape[0] == 1000 and ws.nearestKSearch(None, 16)[0].shape == (1000, 16)


def test_fixed_cost_does_not_grow_with_cluster_count(torch_cuda):
    """the same launches for 8 and for 64 clusters of 2000 points"""
    from pointcloudcomparator_b200.search import knn_batched, launch_count, region_growing_rgb_batched
    a = _patch(2000, 0.3)
    rgb = _rgb(a, 43)

    def tiles(k):
        return _concat([(a + np.float32([0.7 * (i % 8), 0.7 * (i // 8), 0]), rgb) for i in range(k)])

    deltas = []
    for k in (8, 64):
        xyz, rg, off = tiles(k)
        region_growing_rgb_batched(xyz, rg, off)                     # warm-up
        before = launch_count()
        knn_batched(xyz, off, 100)
        mid = launch_count()
        labels, counts = region_growing_rgb_batched(xyz, rg, off)
        deltas.append((mid - before, launch_count() - mid))
        assert counts.size == k
    print(f"launches per call (knn, rgb): 8 clusters {deltas[0]}, 64 clusters {deltas[1]}")
    assert deltas[0] == deltas[1]


def _call(entry, xyz, off, k=100, n=None, n_clouds=None, stride=16, rgb_off=12, null_out=False):
    from pointcloudcomparator_b200 import _lib
    from pointcloudcomparator_b200.search import GridSearch
    ws = GridSearch()
    rows = np.zeros((xyz.shape[0], 4), np.float32)
    rows[:, :3] = xyz
    off = np.ascontiguousarray(off, np.int64)
    n = rows.shape[0] if n is None else n
    n_clouds = off.size - 1 if n_clouds is None else n_clouds
    a = np.empty((rows.shape[0], max(k, 1)), np.int32)
    b = np.empty((rows.shape[0], max(k, 1)), np.float32)
    c = np.empty(max(off.size, 1), np.int64)
    out = [None if null_out else a.ctypes.data, None if null_out else b.ctypes.data, None if null_out else c.ctypes.data]
    if entry == "knn":
        rc = ws._L.pcc_knn_batched(ws._h, rows.ctypes.data, n, stride, off.ctypes.data, n_clouds, k, out[0], out[1], out[2], _lib.HOST, None)
    else:
        rc = ws._L.pcc_region_growing_rgb_batched(ws._h, rows.ctypes.data, n, stride, rgb_off, off.ctypes.data, n_clouds, k, 10.0, 6.0, 5.0, 30, 200,
                                                  2**31 - 1, out[0], out[2], _lib.HOST, None)
    return rc, ws


@pytest.mark.parametrize("entry", ["knn", "rgb"])
@pytest.mark.parametrize("bad", ["start", "end", "decrease", "n_clouds", "k0", "k513", "null_out", "stride", "rgb_offset"])
def test_argument_errors(torch_cuda, entry, bad):
    xyz, _, off = batch("shared-space")
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
    elif bad == "k0":
        kw["k"] = 0
    elif bad == "k513":
        kw["k"] = 513
    elif bad == "null_out":
        kw["null_out"] = True
    elif bad == "stride":
        kw["stride"] = 10
    else:
        if entry == "knn":
            pytest.skip("pcc_knn_batched reads no colour")
        kw["rgb_off"] = 14
    rc, ws = _call(entry, xyz, off, **kw)
    assert rc == PCC_ERR_INVALID
    assert ws._L.pcc_last_error()


def test_cpp_rgb_batched_mirror(torch_cuda):
    exe = os.path.join(ROOT, "tests", "cpp", "test_rgb_batched")
    assert os.path.exists(exe), "run __graft_entry__.build() first"
    out = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "PASS" in out.stdout, out.stdout + out.stderr
