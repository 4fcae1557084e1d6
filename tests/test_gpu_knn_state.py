"""kNN exactness against the state an index carries from call to call: the cached logging-threshold table of the k <= 16 block
kernel, a handle rebuilt or re-adopted in place, the two-slot pipelined host path (index + shadow, each with its own table), the
dispatch boundaries of pcc_knn, the process-wide switches (read once per process, so each runs in a subprocess of this file) and
the grid-size extremes.  Bar: bit-exact indices and fp32 squared distances against oracle.KdTree / oracle.brute_knn, keff equal.

Run as a script (`python tests/test_gpu_knn_state.py <case>`) this file is the worker the switch tests start."""
import functools
import os
import re
import subprocess
import sys
import zlib

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for _p in (ROOT, HERE):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import oracle                                      # noqa: E402
from conftest import bits                          # noqa: E402
from pointcloudcomparator_b200 import synth        # noqa: E402

pytestmark = pytest.mark.gpu

CALIB_LAUNCHES = 2          # knn_calib_kernel + knn_calib_finish_kernel
SORTED_PREP = 1 + 4         # a batch of > 2048 rows: qprep_kernel + four radix-sort passes
BLOCK_PATH = 6              # block kernel, its retry (threshold) or fix-up (round-1) pass, wide, ring compaction, ring, late wide


@pytest.fixture(scope="module")
def GS():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from pointcloudcomparator_b200.search import GridSearch
    return GridSearch


# ---------------------------------------------------------------- helpers
def assert_knn_equal(gi, gd, oi, od, what=""):
    assert gi.shape == oi.shape, (what, gi.shape, oi.shape)
    assert np.array_equal(gi, oi), f"{what}: index mismatch in rows {np.unique(np.argwhere(gi != oi)[:, 0])[:8].tolist()}"
    assert np.array_equal(bits(gd), bits(od)), f"{what}: d2 mismatch in rows {np.unique(np.argwhere(bits(gd) != bits(od))[:, 0])[:8].tolist()}"


def knn_checked(s, q, k, tree, what=""):
    """One nearestKSearch, checked against the oracle; returns the number of kernel launches it took."""
    from pointcloudcomparator_b200.search import launch_count
    n0 = launch_count()
    gi, gd, keff = s.nearestKSearch(q, k)
    delta = launch_count() - n0
    oi, od, okeff = tree.knn(q, k)
    assert keff == okeff, (what, keff, okeff)
    assert_knn_equal(gi, gd, oi, od, what)
    return delta


def radius_checked(s, q, r, tree, what=""):
    off, idx, d2 = s.radiusSearch(q, r)
    ooff, oidx, od2 = tree.radius(q, r)
    assert np.array_equal(off, ooff) and np.array_equal(idx, oidx) and np.array_equal(bits(d2), bits(od2)), what


def mean_dist_checked(s, q, mean_k, tree, what=""):
    got = s.meanNeighbourDistance(q, mean_k)
    _, d2, _ = tree.knn(s.getInputCloud() if q is None else q, mean_k + 1)
    assert np.array_equal(bits(got), bits(oracle.sor_mean_dist(d2, mean_k))), what


def normals_checked(s, q, k, ref, tree, what=""):
    """Normals of q (None: the indexed cloud) from the k nearest.  eigen33's last-ulp rounding differs between glibc and CUDA
    (tests/test_gpu_parity.py test_normals_knn_vs_oracle), so the 1e-5 bar applies where the neighbourhood is a plane
    (curvature < 0.02: a well separated smallest eigenvalue); there wrong neighbours give a visibly different normal."""
    qp = ref if q is None else q
    got = s.normalsKnn(q, k)
    idx, _, _ = tree.knn(qp, k)
    want = oracle.normals_from_lists(ref, qp, np.arange(len(qp) + 1, dtype=np.int64) * k, np.where(idx < 0, 0, idx))
    empty = idx[:, 0] < 0
    want[empty] = np.nan
    assert np.array_equal(np.isnan(got[:, 0]), np.isnan(want[:, 0])), what
    planar = ~empty & (want[:, 3] < 0.02)
    assert planar.mean() > 0.5, (what, planar.mean())
    err = np.linalg.norm(got[planar, :3] - want[planar, :3], axis=1)
    assert err.max() < 1e-5, (what, err.max(), np.flatnonzero(planar)[np.argmax(err)])


# ---------------------------------------------------------------- the mixed cloud (A, C, D, E, F)
@functools.lru_cache(maxsize=None)
def mixed():
    """A room surface, a dense uniform volume floating inside it (no surface in it), a 3000-point clump inside one cell and
    exact duplicates of both.  Query batches: P noisy surface, V inside the volume, F mostly non-finite + far, N all
    non-finite (empty calibration sample), C inside the clump.  Every batch is > 2048 rows (sorted path, threshold kernel)."""
    rng = np.random.default_rng(2024)
    surf = synth.room(150_000, 3101)
    vol = (np.array([2.5, 1.3, 1.0]) + rng.random((50_000, 3)) * [1.0, 1.0, 1.2]).astype(np.float32)
    centre = surf[123]
    clump = (centre + rng.normal(0, 2e-4, (3000, 3))).astype(np.float32)
    dup = np.concatenate([surf[rng.choice(len(surf), 30, replace=False)], vol[rng.choice(len(vol), 400, replace=False)]])
    ref = np.concatenate([surf, vol, clump, dup]).astype(np.float32)
    ref = np.ascontiguousarray(ref[rng.permutation(len(ref))])
    P = (surf[rng.choice(len(surf), 20_000, replace=False)] + rng.normal(0, 0.005, (20_000, 3))).astype(np.float32)
    V = (np.array([2.5, 1.3, 1.0]) + rng.random((8000, 3)) * [1.0, 1.0, 1.2]).astype(np.float32)
    F = np.full((3000, 3), np.nan, np.float32)
    F[::3, 1] = np.inf
    F[::3, 0] = 0.0
    far = rng.uniform(-60, 60, (150, 3)).astype(np.float32)
    F[rng.choice(3000, 150, replace=False)] = far
    N = np.full((3000, 3), np.nan, np.float32)
    N[1::2] = [np.inf, 1.0, 1.0]
    C = (centre + rng.normal(0, 3e-4, (3000, 3))).astype(np.float32)
    return dict(ref=ref, surf=surf, P=P, V=V, F=F, N=N, C=C, vol_lo=np.array([2.5, 1.3, 1.0]), vol_hi=np.array([3.5, 2.3, 2.2]))


@functools.lru_cache(maxsize=None)
def mixed_tree():
    return oracle.KdTree(mixed()["ref"])


# ---------------------------------------------------------------- A. a stale table on one handle
def test_stale_threshold_table_one_handle(GS):
    m, tree = mixed(), mixed_tree()
    ref = m["ref"]
    s = GS().setInputCloud(ref)
    seq = [("P", 12), ("P", 12), ("P", 12), ("V", 12), ("V", 12), ("V", 12), ("P", 12), ("P", 16), ("F", 16), ("P", 16),
           ("N", 9), ("P", 9), ("C", 16), ("P", 16), ("V", 9), ("C", 12), ("P", 16)]
    between = [lambda: mean_dist_checked(s, m["P"][:5000], 8, tree, "mean_k 8"),
               lambda: radius_checked(s, m["P"][:5000], 0.05, tree, "radius 0.05"),
               lambda: normals_checked(s, m["P"][:5000], 16, ref, tree, "normals k 16"),
               lambda: mean_dist_checked(s, m["V"][:3000], 16, tree, "mean_k 16 volume"),
               lambda: radius_checked(s, m["C"][:500], 0.002, tree, "radius in the clump")]
    deltas = []
    for i, (name, k) in enumerate(seq):
        deltas.append(knn_checked(s, m[name], k, tree, f"call {i}: {name} k={k}"))
        between[i % len(between)]()
    base = SORTED_PREP + BLOCK_PATH
    cal = [d == base + CALIB_LAUNCHES for d in deltas]
    print("launch deltas", deltas, "calibrated", [f"{i}:{n}{k}" for i, ((n, k), c) in enumerate(zip(seq, cal)) if c])
    assert deltas[1] == deltas[2] == base, f"a warm repeated call takes a fixed number of launches: {deltas}"
    assert set(deltas) <= {base, base + CALIB_LAUNCHES}, deltas
    assert cal[0], "a fresh index calibrates on its first block-kernel call"
    assert not cal[1] and not cal[2], "the table calibrated on P must be reused for the next P calls"
    assert cal[4] or cal[5], "the P table sent > 4 % of the volume batch to the retry pass: one of the next two calls must recalibrate"
    for i, ((_, k), (_, k0)) in enumerate(zip(seq[1:], seq[:-1]), 1):
        if k != k0:
            assert cal[i], f"call {i}: k changed {k0} -> {k}, the table must be re-made"


# ---------------------------------------------------------------- B. rebuilding one handle
def test_rebuild_one_handle(GS):
    rng = np.random.default_rng(7)
    A = synth.room(80_000, 501)
    qA = synth.sweep_queries(A, 5000, seed=502, sigma=0.01)
    srcA = (A[rng.permutation(len(A))[:20_000]] + rng.normal(0, 0.02, (20_000, 3))).astype(np.float32)
    Bf = (synth.room(60_000, 503, size=(2.0, 1.5, 1.0)) + np.float32([10.0, -5.0, 3.0])).astype(np.float32)
    B = np.insert(Bf, rng.choice(len(Bf), 300, replace=False), np.float32(np.nan), axis=0)
    B[rng.choice(len(B), 50, replace=False), 2] = np.inf
    bad = ~np.isfinite(B).all(1)
    qB = synth.sweep_queries(Bf, 5000, seed=504, sigma=0.005)
    srcB = (Bf[rng.permutation(len(Bf))[:20_000]] + rng.normal(0, 0.01, (20_000, 3))).astype(np.float32)
    tA, tB = oracle.KdTree(A), oracle.KdTree(B)

    def icp_checked(s, src, tree, what):
        cnt, sums, ci, cd = s.icpStep(src.copy(), None, want_correspondences=True)
        ocnt, osums, oci, ocd = tree.icp_pass(src)
        assert cnt == ocnt, (what, cnt, ocnt)
        assert np.array_equal(ci, oci), f"{what}: correspondence mismatch in rows {np.flatnonzero(ci != oci)[:8].tolist()}"
        assert np.array_equal(bits(cd), bits(ocd)), f"{what}: d2 mismatch in rows {np.flatnonzero(bits(cd) != bits(ocd))[:8].tolist()}"
        assert np.allclose(sums, osums, rtol=1e-12, atol=1e-9), (what, (sums - osums).tolist())

    s = GS().setInputCloud(A)
    assert s.export()[0][12] == 1.0
    knn_checked(s, qA, 16, tA, "A external")
    normals_checked(s, None, 16, A, tA, "A normals")
    icp_checked(s, srcA, tA, "A icp")

    s.setInputCloud(B)                                               # new extent, density, row count; NaN rows
    meta = s.export()[0]
    assert meta[12] == 0.0 and meta[0] == len(B) - bad.sum() and meta[1] == len(B)
    knn_checked(s, qB, 16, tB, "B external")
    gi, gd, keff = s.nearestKSearch(None, 16)
    oi, od, _ = tB.knn(B, 16)
    assert keff == 16
    assert_knn_equal(gi, gd, oi, od, "B self")
    assert (gi[bad] == -1).all() and np.isinf(gd[bad]).all() and (gi[~bad] >= 0).all(), "rows of unindexed points must be (-1, +inf)"
    normals_checked(s, None, 16, B, tB, "B normals (new inverse permutation)")
    icp_checked(s, srcB, tB, "B icp, source of the size used on A")
    lab, sizes = s.euclideanClusters(0.03, 50, 250_000)
    olab, osizes = tB.ece(0.03, 50, 250_000)
    assert np.array_equal(sizes, osizes), ("B clusters", sizes[:8].tolist(), osizes[:8].tolist())
    assert np.array_equal(lab, olab), f"B cluster labels differ in rows {np.flatnonzero(lab != olab)[:8].tolist()}"

    sub = np.sort(rng.choice(np.flatnonzero(~bad), 25_000, replace=False)).astype(np.int32)
    s.setInputCloud(B, indices=sub)
    tS = oracle.KdTree(B[sub])
    gi, gd, _ = s.nearestKSearch(qB, 16)
    oi, od, _ = tS.knn(qB, 16)
    assert_knn_equal(gi, gd, sub[oi], od, "B subset external")
    gi, gd, _ = s.nearestKSearch(None, 12)
    oi, od, _ = tS.knn(B[sub], 12)
    assert_knn_equal(gi[sub], gd[sub], sub[oi], od, "B subset self")
    rest = np.setdiff1d(np.arange(len(B)), sub)
    assert (gi[rest] == -1).all() and np.isinf(gd[rest]).all()

    s.setInputCloud(B)
    knn_checked(s, qB, 12, tB, "B again")
    s.setInputCloud(A)
    assert s.export()[0][12] == 1.0
    knn_checked(s, qA, 16, tA, "back to A")
    gi, gd, _ = s.nearestKSearch(None, 16)
    oi, od, _ = tA.knn(A, 16)
    assert_knn_equal(gi, gd, oi, od, "A self after rebuilds")
    normals_checked(s, None, 16, A, tA, "A normals after rebuilds")
    icp_checked(s, srcA, tA, "A icp after rebuilds")


# ---------------------------------------------------------------- C. the pipelined host path with unlike chunks
def test_pipelined_host_path_unlike_chunks(GS):
    import torch
    m, tree = mixed(), mixed_tree()
    rng = np.random.default_rng(11)
    chunk = 1 << 20
    surf_q = synth.sweep_queries(m["surf"], chunk, seed=12, sigma=0.01)
    vol_q = (m["vol_lo"] + rng.random((chunk, 3)) * (m["vol_hi"] - m["vol_lo"])).astype(np.float32)
    vol_q[rng.choice(chunk, chunk // 8, replace=False)] = rng.uniform(-30, 30, (chunk // 8, 3)).astype(np.float32)     # far rows
    last = m["P"][:1]
    sel = np.random.default_rng(13).choice(2 * chunk + 1, 20_000, replace=False)
    from pointcloudcomparator_b200.search import launch_count
    s = GS().setInputCloud(m["ref"])
    for phase in ("surface first", "volume first", "rebuilt"):
        if phase == "rebuilt":
            s.setInputCloud(m["ref"], k_hint=4)                  # another grid: both slots must drop their tables
        first, second = (vol_q, surf_q) if phase == "volume first" else (surf_q, vol_q)
        qry = np.ascontiguousarray(np.concatenate([first, second, last]))
        dq = torch.from_numpy(qry).cuda()
        for j, k in enumerate((16, 12, 1, 40, 16)):
            n0 = launch_count()
            hi, hd, keff = s.nearestKSearch(qry, k)                      # host buffer -> two-slot pipeline
            n1 = launch_count()
            di, dd, _ = s.nearestKSearch(dq, k)                          # one launch sequence over the whole batch
            dh, dd_ = n1 - n0, launch_count() - n1
            print(f"{phase} k={k}: launches pipelined {dh}, one-shot {dd_}")
            assert keff == k
            assert dh > dd_, (phase, k, dh, dd_)                         # one launch sequence per chunk
            if j == 0 and phase != "volume first":
                # a fresh or rebuilt index: the index (chunk 0, surface queries) and its shadow (chunk 1, volume and far
                # queries) each calibrate their own table; the 1-row chunk 2 takes the exact single-kernel path
                assert dh == 2 * (SORTED_PREP + BLOCK_PATH + CALIB_LAUNCHES) + 2, (phase, dh)
            assert torch.equal(torch.from_numpy(hi).cuda(), di), (phase, k)
            assert torch.equal(torch.from_numpy(hd).cuda().view(torch.int32), dd.view(torch.int32)), (phase, k)
            oi, od, _ = tree.knn(qry[sel], k)
            assert_knn_equal(hi[sel], hd[sel], oi, od, f"{phase} k={k}")
            del hi, hd, di, dd


# ---------------------------------------------------------------- D. adopted grids
def _view(ptr, nbytes):
    import torch

    class _Mem:
        pass
    mem = _Mem()
    mem.__cuda_array_interface__ = {"shape": (nbytes // 4,), "typestr": "<f4", "data": (int(ptr), False), "version": 3}
    return torch.as_tensor(mem, device="cuda:0")


def _adopt_copy(dst, src):
    import torch
    meta, s_pts, s_cells = src.export()
    _, d_pts, d_cells = dst.adopt(meta)
    _view(d_pts, int(meta[0]) * 16).copy_(_view(s_pts, int(meta[0]) * 16))
    _view(d_cells, (int(meta[11]) + 1) * 4).copy_(_view(s_cells, (int(meta[11]) + 1) * 4))
    torch.cuda.synchronize()
    return meta


def test_adopted_grid_every_path_and_readoption(GS):
    import torch
    ref = synth.room(50_000, 12)
    rng = np.random.default_rng(2)
    qry = np.concatenate([ref[::5] + np.float32(0.004), rng.uniform(-1, 6, (2000, 3)).astype(np.float32), [[np.nan, 0, 0]]]).astype(np.float32)
    a = GS().setInputCloud(torch.from_numpy(ref).cuda(), k_hint=8)
    b = GS()
    meta_a = _adopt_copy(b, a)
    tree = oracle.KdTree(ref)
    for k in (1, 5, 12, 16, 32, 40, 200):
        knn_checked(b, qry, k, tree, f"adopted k={k}")
    radius_checked(b, qry, 0.04, tree, "adopted radius")
    gi, gd, _ = b.nearestKSearch(None, 16)
    oi, od, _ = tree.knn(ref, 16)
    assert_knn_equal(gi.cpu().numpy(), gd.cpu().numpy(), oi, od, "adopted self")

    other = np.concatenate([synth.uniform(70_000, 14, extent=3.0), synth.room(30_000, 15, size=(3.0, 3.0, 3.0))]).astype(np.float32)
    q2 = np.concatenate([synth.sweep_queries(other, 9000, seed=16, sigma=0.01), rng.uniform(-1, 4, (1000, 3)).astype(np.float32)]).astype(np.float32)
    c = GS().setInputCloud(torch.from_numpy(other).cuda())
    meta = _adopt_copy(b, c)                                                 # a different grid into the same handle
    assert meta[11] != meta_a[11] and meta[0] != meta_a[0]               # another cell table and another point count
    tree2 = oracle.KdTree(other)
    for k in (16, 12, 5, 1, 32, 40, 200):
        knn_checked(b, q2, k, tree2, f"re-adopted k={k}")
    radius_checked(b, q2, 0.05, tree2, "re-adopted radius")


# ---------------------------------------------------------------- E. dispatch boundaries
def test_dispatch_boundaries(GS):
    m = mixed()
    rng = np.random.default_rng(21)
    pool = np.concatenate([m["P"], m["V"], m["C"][:2000], synth.sweep_queries(m["surf"], 34_000, seed=22, sigma=0.02),
                           rng.uniform(-8, 12, (1500, 3)).astype(np.float32), np.full((37, 3), np.nan, np.float32)]).astype(np.float32)
    assert len(pool) == 65_537
    pool = np.ascontiguousarray(pool[rng.permutation(len(pool))])
    ref, tree = m["ref"], mixed_tree()
    for k, sizes in ((9, None), (16, None), (32, None), (33, (63, 64, 65)), (50, (63, 64, 65))):
        sizes = sizes or (1, 31, 32, 33, 1023, 1024, 1025, 32767, 32768, 65535, 65536, 65537)
        oi, od, _ = tree.knn(pool[: max(sizes)], k)
        s = GS().setInputCloud(ref)
        deltas = {}
        for nq in sizes:
            from pointcloudcomparator_b200.search import launch_count
            n0 = launch_count()
            gi, gd, keff = s.nearestKSearch(pool[:nq], k)
            deltas[nq] = launch_count() - n0
            assert keff == k
            assert_knn_equal(gi, gd, oi[:nq], od[:nq], f"k={k} nq={nq}")
        small = 1024 if k <= 32 else 64
        assert deltas[small - 1] < deltas[small], (k, deltas)            # below the boundary: the single-kernel exact path


# ---------------------------------------------------------------- G. grid extremes
def test_largest_grid_far_corner(GS):
    rng = np.random.default_rng(31)
    hi = np.array([20.47, 20.47, 0.40])
    dense = np.array([20.0, 20.0, 0.0]) + rng.random((20_000, 3)) * [0.47, 0.47, 0.40]
    sparse = np.array([19.0, 19.0, 0.0]) + rng.random((3000, 3)) * [1.0, 1.47, 0.40]
    origin = rng.random((5000, 3)) * [0.5, 0.5, 0.40]
    ref = np.concatenate([[[0, 0, 0], hi], dense, sparse, origin]).astype(np.float32)
    ref = ref[rng.permutation(len(ref))]
    s = GS().setInputCloud(ref, cell_hint=0.002)
    meta = s.export()[0]
    dims = meta[2:5]
    print("largest grid: dims", dims.tolist(), "cells", int(meta[11]), "cell", meta[8])
    assert meta[11] >= 2 ** 27 and meta[11] <= 2 ** 28 and dims.max() <= 2048, meta[:12].tolist()
    qry = np.concatenate([dense[::5] + rng.normal(0, 0.01, (4000, 3)), sparse[::3] + rng.normal(0, 0.02, (1000, 3)),
                          np.array([19.0, 19.0, -0.05]) + rng.random((2000, 3)) * [1.6, 1.6, 0.5], origin[:500]]).astype(np.float32)
    tree = oracle.KdTree(ref)
    for k in (5, 16, 32):
        knn_checked(s, qry, k, tree, f"largest grid k={k}")
    radius_checked(s, qry, 0.03, tree, "largest grid radius")
    del s


@pytest.mark.parametrize("env", [{"PCC_MAX_CELLS": "4096"}, {"PCC_OCC": "200"}])
def test_very_coarse_grid(GS, env):
    """Thousands of points per block: the block kernels' logs overflow and the retry pass compresses (PCC_STATS, so a
    subprocess; both grid variables are read per build)."""
    st = _stats_by_label(_run_worker("coarse", {**env, "PCC_STATS": "1"}).stderr)
    print(env, {k: (v["overflow"], v["fixup"]) for k, v in st.items()})
    assert len(st) == 4, sorted(st)
    assert all(v["overflow"] > 0.2 for v in st.values()), st                # measured on B200: 0.43 .. 1.0 of the queries per call


# ---------------------------------------------------------------- F. process-wide switches (one subprocess each)
STATS_RE = re.compile(r"\[pcc stats\] queries=(\d+) logged/q=([\d.]+) log_overflow=([\d.]+) need_ring2=([\d.]+) fixup=([\d.]+) members/q=([\d.]+)")


def _run_worker(case, env_add, timeout=900):
    env = {k: v for k, v in os.environ.items() if not k.startswith("PCC_")}
    env.update(env_add)
    r = subprocess.run([sys.executable, os.path.abspath(__file__), case], env=env, cwd=ROOT, timeout=timeout, capture_output=True, text=True)
    assert r.returncode == 0 and "PASS" in r.stdout.splitlines(), f"worker {case} {env_add} rc={r.returncode}\n{r.stdout[-3000:]}\n{r.stderr[-3000:]}"
    return r


def _stats_by_label(stderr):
    out, label = {}, None
    for line in stderr.splitlines():
        if line.startswith("[case] "):
            label = line[7:].strip()
        mt = STATS_RE.search(line)
        if mt and label is not None:
            out[label] = dict(queries=int(mt[1]), logged=float(mt[2]), overflow=float(mt[3]), fixup=float(mt[5]))
    return out


def _weighted(st, key):
    q = sum(v["queries"] for v in st.values())
    return sum(v[key] * v["queries"] for v in st.values()) / max(q, 1)


@pytest.fixture(scope="module")
def default_stats(GS):
    st = _stats_by_label(_run_worker("stats", {"PCC_STATS": "1"}).stderr)
    assert len(st) == 2 * 5 * 3, sorted(st)
    return st


def test_switch_quantile_zero_tightest_table(default_stats):
    st = _stats_by_label(_run_worker("stats", {"PCC_STATS": "1", "PCC_THR_QUANTILE": "0"}).stderr)
    assert sorted(st) == sorted(default_stats)
    fd, f0 = _weighted(default_stats, "fixup"), _weighted(st, "fixup")
    print(f"retry (fixup) fraction: default {fd:.4f}, PCC_THR_QUANTILE=0 {f0:.4f}; per call (default, quantile 0):",
          {k: (default_stats[k]["fixup"], v["fixup"]) for k, v in st.items()})
    assert f0 > 4 * fd and f0 > fd + 0.2, (fd, f0)


def test_switch_quantile_one_loosest_table(default_stats):
    st = _stats_by_label(_run_worker("stats", {"PCC_STATS": "1", "PCC_THR_QUANTILE": "1"}).stderr)
    assert sorted(st) == sorted(default_stats)
    ld, l1 = _weighted(default_stats, "logged"), _weighted(st, "logged")
    clump = {k: v["overflow"] for k, v in st.items() if "clump" in k}
    print(f"logged/q: default {ld:.2f}, PCC_THR_QUANTILE=1 {l1:.2f}; log_overflow on the clump {clump}; per call (default, quantile 1):",
          {k: (default_stats[k]["logged"], v["logged"]) for k, v in st.items()})
    assert l1 > 1.05 * ld, (ld, l1)          # logged/q saturates at the log size (the clump overflows in every run)
    assert clump and all(v > 0 for v in clump.values()), clump


@pytest.mark.parametrize("case,env", [("thr_all", {"PCC_THR_ALL": "1"}), ("old_fast", {"PCC_OLD_FAST": "1"}),
                                      ("exact_only", {"PCC_EXACT_ONLY": "1"}), ("pipe16", {"PCC_PIPE_CHUNK_LOG2": "16"})])
def test_switch_worker(GS, case, env):
    r = _run_worker(case, env)
    print(r.stdout[-800:])


# ---------------------------------------------------------------- worker side
def _stress_cloud(rng, kind, n):
    if kind == "surface":
        return synth.room(n, int(rng.integers(1 << 30)))
    if kind == "volume":
        return (rng.random((n, 3)) * 4.0).astype(np.float32)
    if kind == "clustered":                       # very uneven density + far outliers (tests/test_gpu_parity.py _stress_cloud)
        c = rng.normal(0, 1.0, (8, 3))
        p = c[rng.integers(0, 8, n)] + rng.normal(0, 0.01, (n, 3)) * rng.choice([1.0, 10.0], (n, 1))
        p[: n // 100] = rng.uniform(-30, 30, (n // 100, 3))
        return p.astype(np.float32)
    if kind == "quantized":                       # millimetre-quantized: many exact ties and duplicates
        return (np.round(rng.random((n, 3)) * [2.0, 2.0, 0.5] * 200) / 200).astype(np.float32)
    raise ValueError(kind)


def _label(text):
    sys.stderr.write(f"[case] {text}\n")
    sys.stderr.flush()


def _worker_stats(GS):
    """k in {9, 12, 16} on four cloud kinds and the clump of the mixed cloud, with the per-lane and the staged block kernel."""
    for staged in (False, True):
        if staged:
            os.environ["PCC_THR_STAGED"] = "1"
        for kind in ("surface", "volume", "clustered", "quantized", "clump"):
            if kind == "clump":
                ref, qry = mixed()["ref"], mixed()["C"]
                tree = mixed_tree()
            else:
                rng = np.random.default_rng(zlib.crc32(kind.encode()))
                ref = _stress_cloud(rng, kind, 80_000)
                spread = np.maximum(ref.max(0) - ref.min(0), 1e-9)
                qry = (ref[rng.integers(0, len(ref), 8000)] + rng.normal(0, 2e-3, (8000, 3)) * spread).astype(np.float32)
                tree = oracle.KdTree(ref)
            s = GS().setInputCloud(ref)
            for k in (16, 9, 12):
                _label(f"{'staged/' if staged else ''}{kind} k={k}")
                knn_checked(s, qry, k, tree, f"{kind} k={k} staged={staged}")
    os.environ.pop("PCC_THR_STAGED", None)


def _worker_thr_all(GS):
    m, tree = mixed(), mixed_tree()
    s = GS().setInputCloud(m["ref"])
    for k in (2, 3, 4, 5, 8, 17, 24, 32):
        first = knn_checked(s, m["P"], k, tree, f"P k={k}")
        again = knn_checked(s, m["P"], k, tree, f"P k={k} again")
        assert first == SORTED_PREP + BLOCK_PATH + CALIB_LAUNCHES, (k, first)      # new k: the threshold kernel calibrates its table
        knn_checked(s, m["V"], k, tree, f"V k={k}")
        knn_checked(s, m["C"], k, tree, f"C k={k}")
        print(f"k={k}: launches {first} (calibrating) / {again}")


def _worker_old_fast(GS):
    m, tree = mixed(), mixed_tree()
    g = np.arange(20, dtype=np.float32) * 0.25
    lattice = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3)
    lattice = np.ascontiguousarray(lattice[np.random.default_rng(5).permutation(len(lattice))])
    lat = GS().setInputCloud(lattice)
    s = GS().setInputCloud(m["ref"])
    for k in (9, 16):
        gi, gd, _ = lat.nearestKSearch(lattice, k)                      # 8000 tied queries: knn_fixup_kernel after the round-1 kernel
        oi, od, _ = oracle.brute_knn(lattice, lattice, k)
        assert_knn_equal(gi, gd, oi, od, f"lattice k={k}")
        first = knn_checked(s, m["P"], k, tree, f"P k={k}")
        again = knn_checked(s, m["P"], k, tree, f"P k={k} again")
        assert first == SORTED_PREP + BLOCK_PATH, (k, first)            # new k, but the round-1 kernel has no table to calibrate
        knn_checked(s, m["V"], k, tree, f"V k={k}")
        knn_checked(s, m["C"], k, tree, f"C k={k}")
        print(f"k={k}: launches {first} / {again}")


def _worker_exact_only(GS):
    m, tree = mixed(), mixed_tree()
    rng = np.random.default_rng(41)
    qry = np.concatenate([m["P"], m["V"], m["C"], m["F"], synth.sweep_queries(m["surf"], 80_000, seed=42, sigma=0.01),
                          rng.uniform(-2, 8, (2000, 3)).astype(np.float32)]).astype(np.float32)
    assert len(qry) >= 100_000
    s = GS().setInputCloud(m["ref"])
    for k in (2, 8, 16, 32, 40, 200):
        d = knn_checked(s, qry, k, tree, f"k={k}")
        assert d == SORTED_PREP + 1, (k, d)      # ONE search kernel (register list or heap), not the staged or selection path
        print(f"k={k}: {d} launches")


def _worker_pipe16(GS):
    import torch
    m, tree = mixed(), mixed_tree()
    rng = np.random.default_rng(51)
    chunk = 1 << 16
    pool = np.concatenate([synth.sweep_queries(m["surf"], 3 * chunk, seed=52, sigma=0.01),
                           (m["vol_lo"] + rng.random((2 * chunk + 1000, 3)) * (m["vol_hi"] - m["vol_lo"]))]).astype(np.float32)
    from pointcloudcomparator_b200.search import launch_count
    s = GS().setInputCloud(m["ref"])
    for nq in (2 * chunk + 5, 5 * chunk + 1000):
        qry = np.ascontiguousarray(pool[:nq] if nq < 3 * chunk else pool[rng.permutation(len(pool))][:nq])
        for k in (12, 16):
            n0 = launch_count()
            hi, hd, keff = s.nearestKSearch(qry, k)
            dh = launch_count() - n0
            n0 = launch_count()
            di, dd, _ = s.nearestKSearch(torch.from_numpy(qry).cuda(), k)
            dd_ = launch_count() - n0
            assert keff == k and np.array_equal(hi, di.cpu().numpy()) and np.array_equal(bits(hd), bits(dd.cpu().numpy())), (nq, k)
            oi, od, _ = tree.knn(qry, k)
            assert_knn_equal(hi, hd, oi, od, f"nq={nq} k={k}")
            assert dh > dd_ + SORTED_PREP, (nq, k, dh, dd_)               # several chunks, each its own launch sequence
            print(f"nq={nq} k={k}: launches pipelined {dh}, one-shot {dd_}")


def _worker_coarse(GS):
    m, tree = mixed(), mixed_tree()
    s = GS().setInputCloud(m["ref"])
    meta, info = s.export()[0], s.grid_info()
    print("cells", int(meta[11]), "occupancy", info["occupancy"])
    if "PCC_MAX_CELLS" in os.environ:
        assert meta[11] <= int(os.environ["PCC_MAX_CELLS"]), meta[11]
    else:
        assert info["occupancy"] >= 100, info
    qry = np.concatenate([m["P"][:4000], m["V"][:2000], m["C"][:1000], m["F"][:500]])
    for k in (9, 16, 32, 12):
        _label(f"coarse k={k}")
        knn_checked(s, qry, k, tree, f"coarse k={k}")


WORKERS = {"coarse": _worker_coarse, "stats": _worker_stats, "thr_all": _worker_thr_all, "old_fast": _worker_old_fast, "exact_only": _worker_exact_only, "pipe16": _worker_pipe16}


if __name__ == "__main__":
    import torch
    assert torch.cuda.is_available(), "the worker needs a CUDA device"
    from pointcloudcomparator_b200.search import GridSearch
    WORKERS[sys.argv[1]](GridSearch)
    print("PASS", flush=True)
