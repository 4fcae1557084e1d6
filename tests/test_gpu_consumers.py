"""GPU tests of the fused per-query consumers (pcc_normals_knn, pcc_knn_mean_dist, pcc_normals_radius, pcc_intensity_gradient,
pcc_rift, pcc_sift_dog, pcc_first_within, pcc_sor_threshold) at every kernel instantiation their dispatch can pick, with self and
external queries, over `indices` subsets, in host and device memory, on side streams and on an adopted grid.

References: the CPU oracle (oracle.KdTree rows -> normals_from_lists / sor_mean_dist / sor_threshold; descriptor_oracle for
gradients, RIFT and DoG) and, for the SOR statistics, plain fp64 numpy and scipy.  Bars: mean distances, gradients and DoG
bit-identical (NaN payloads aside); unit normals within 1e-5 on every row, curvature rtol 1e-3 / atol 5e-7; RIFT bins within 1e-5;
SOR statistics within 1e-9 relative.  NaN patterns match exactly.  Run on the B200 box with `-m gpu`."""
import ctypes as C

import numpy as np
import pytest

import descriptor_oracle as D
import oracle
from conftest import bits
from pointcloudcomparator_b200 import synth

pytestmark = pytest.mark.gpu

VP = (1.5, -2.0, 10.0)                 # a viewpoint off the origin, outside the room: every flip is decided against the query point
SENTINEL_F = np.float32(-1234.5)       # neither NaN nor 0: a row still holding it was never written
SENTINEL_I = 0x5A5A5A5A
SENTINEL_B = 0x5A


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


@pytest.fixture(scope="module")
def GS(torch_cuda):
    from pointcloudcomparator_b200.search import GridSearch
    return GridSearch


def same(a, b):
    """bit-identical, NaN payloads aside (the C oracle's NAN and CUDA's differ in payload only)"""
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    na, nb = np.isnan(a), np.isnan(b)
    return a.shape == b.shape and np.array_equal(na, nb) and np.array_equal(bits(np.where(na, 0, a)), bits(np.where(nb, 0, b)))


def check_normals(got, want, qpts, vp=(0.0, 0.0, 0.0)):
    """NaN rows identical; every other unit normal within 1e-5 and curvature within rtol 1e-3 / atol 5e-7.  Where the viewpoint lies
    within 1e-5 rad of a row's tangent plane the flip is decided by the last bits of the normal, so there either sign passes."""
    got, want = np.asarray(got, np.float32), np.asarray(want, np.float32)
    assert got.shape == want.shape
    assert np.array_equal(np.isnan(got), np.isnan(want)), np.argwhere(np.isnan(got) != np.isnan(want))[:5].tolist()
    ok = ~np.isnan(want[:, 0])
    g, w = got[ok], want[ok]
    err = np.linalg.norm(g[:, :3] - w[:, :3], axis=1)
    v = np.asarray(vp, np.float64) - np.asarray(qpts, np.float64)[ok, :3]
    tangent = np.abs(np.einsum("ij,ij->i", v, w[:, :3].astype(np.float64))) <= 1e-5 * np.linalg.norm(v, axis=1)
    err = np.where(tangent, np.minimum(err, np.linalg.norm(g[:, :3] + w[:, :3], axis=1)), err)
    assert err.max(initial=0.0) < 1e-5, err.max()
    assert np.allclose(g[:, 3], w[:, 3], rtol=1e-3, atol=5e-7)
    return int(ok.sum())


def check_rift(got, want):
    """1e-5 absolute per bin (acosf is not correctly rounded on either side), identical NaN bins"""
    got, want = np.asarray(got, np.float32), np.asarray(want, np.float32)
    assert got.shape == want.shape and np.array_equal(np.isnan(got), np.isnan(want))
    fin = ~np.isnan(want)
    assert np.abs(got[fin] - want[fin]).max(initial=0.0) <= 1e-5


def oracle_normals_knn(pts, tree, qpts, k, vp):
    idx, _, _ = tree.knn(qpts, k)
    return oracle.normals_from_lists(pts, qpts, np.arange(len(qpts) + 1, dtype=np.int64) * k, idx, vp)


def oracle_mean_dist(tree, qpts, mean_k):
    _, d2, _ = tree.knn(qpts, mean_k + 1)
    return oracle.sor_mean_dist(d2, mean_k)


def query_mix(s, ref, seed, n_noisy=3000):
    """External queries in 32-byte rows (x, y, z, 5 floats of padding): noisy copies of cloud points, points exactly on cell faces of
    the index's grid, far queries outside the bounding box, NaN / inf rows.  Returns (rows [n, 8], xyz [n, 3] contiguous)."""
    rng = np.random.default_rng(seed)
    meta, _, _ = s.export()
    origin, cell = meta[5:8].astype(np.float32), np.float32(meta[8])
    dims = meta[2:5].astype(np.int64)
    faces = (origin + cell * rng.integers(0, dims, (400, 3)).astype(np.float32)).astype(np.float32)
    fin = ref[np.isfinite(ref[:, :3]).all(1), :3]
    noisy = (fin[rng.integers(0, len(fin), n_noisy)] + rng.normal(0, 0.004, (n_noisy, 3))).astype(np.float32)
    far = rng.uniform(-60, 60, (100, 3)).astype(np.float32)
    bad = np.array([[np.nan, 1, 1], [1, np.nan, 1], [1, 1, np.inf], [np.nan, np.nan, np.nan]], np.float32)
    xyz = np.concatenate([noisy[: n_noisy // 2], faces, bad[:2], far, noisy[n_noisy // 2:], bad[2:]]).astype(np.float32)
    rows = rng.normal(0, 100, (len(xyz), 8)).astype(np.float32)           # padding holds junk: only the first 12 bytes of a row are read
    rows[:, :3] = xyz
    return rows, np.ascontiguousarray(xyz)


@pytest.fixture(scope="module")
def room20k():
    ref = synth.room(20000, 61)
    return ref, oracle.KdTree(ref)


# ---------------------------------------------------------------- 1. every kernel size, self and external queries
# pcc_normals_knn: normals_knn_reg_kernel<8> (k <= 8), <16>, <32>, normals_knn_heap_kernel (k > 32; k = 512 = PCC_MAX_K runs it with
# 32 threads a block and 128 KB of shared memory).  k < 3: every row NaN.
@pytest.mark.parametrize("k", [1, 2, 3, 5, 8, 9, 16, 17, 31, 32, 33, 64, 200, 512])
def test_normals_knn_every_kernel_size(GS, room20k, k):
    ref, tree = room20k
    s = GS().setInputCloud(ref, k_hint=k)
    got = s.normalsKnn(None, k, viewpoint=VP)
    want = oracle_normals_knn(ref, tree, ref, k, VP)
    n_ok = check_normals(got, want, ref, VP)
    assert n_ok == (len(ref) if k >= 3 else 0)
    rows, xyz = query_mix(s, ref, 100 + k)
    got = s.normalsKnn(rows, k, viewpoint=VP)
    want = oracle_normals_knn(ref, tree, xyz, k, VP)
    check_normals(got, want, xyz, VP)
    assert np.isnan(got[~np.isfinite(xyz).all(1)]).all()


# pcc_knn_mean_dist: mean_dist_reg_kernel<K, EXACT> for need = mean_k + 1 <= K in {2, 5, 9, 17, 33, 51}, EXACT when need == K, else
# mean_dist_heap_kernel.  Pairs reached below: <2,T> 1; <5,F> 2, 3; <5,T> 4; <9,T> 8; <17,F> 12; <17,T> 16; <33,F> 24; <33,T> 32;
# <51,F> 40; <51,T> 50; <9,F> 6; heap 51, 100, 511 (need = 512 = PCC_MAX_K).
@pytest.mark.parametrize("mean_k", [1, 2, 3, 4, 6, 8, 12, 16, 24, 32, 40, 50, 51, 100, 511])
def test_mean_distance_every_kernel_size(GS, room20k, mean_k):
    ref, tree = room20k
    s = GS().setInputCloud(ref, k_hint=mean_k + 1)
    got = s.meanNeighbourDistance(None, mean_k)
    assert np.array_equal(bits(got), bits(oracle_mean_dist(tree, ref, mean_k)))
    assert (got > 0).all() and np.isfinite(got).all()
    rows, xyz = query_mix(s, ref, 200 + mean_k)
    got = s.meanNeighbourDistance(rows, mean_k)
    assert np.array_equal(bits(got), bits(oracle_mean_dist(tree, xyz, mean_k)))
    assert (got[~np.isfinite(xyz).all(1)] == 0).all()


@pytest.mark.parametrize("n", [2, 10, 100])
def test_cloud_smaller_than_k(GS, n):
    """Fewer indexed points than k: normals over the short rows (NaN below 3 points), +inf mean distances, at every kernel kind."""
    ref = synth.room(n, 63)
    tree = oracle.KdTree(ref)
    q = np.concatenate([ref, synth.noisy_copy(ref, 64, 0.05)]).astype(np.float32)
    for k in (3, 8, 16, 32, 200, 512):
        s = GS().setInputCloud(ref, k_hint=k)
        for qq in (None, q):
            qp = ref if qq is None else q
            check_normals(s.normalsKnn(qq, k, viewpoint=VP), oracle_normals_knn(ref, tree, qp, k, VP), qp, VP)
    for mean_k in (4, 12, 32, 50, 150, 511):
        s = GS().setInputCloud(ref, k_hint=mean_k + 1)
        for qq in (None, q):
            qp = ref if qq is None else q
            got = s.meanNeighbourDistance(qq, mean_k)
            want = oracle_mean_dist(tree, qp, mean_k)
            assert np.array_equal(bits(got), bits(want))
            if mean_k + 1 > n:
                assert np.isinf(got).all()


def test_consumer_argument_rejections(GS):
    from pointcloudcomparator_b200._lib import PccError
    s = GS().setInputCloud(synth.room(2000, 65))
    for k in (0, 513, -1):
        with pytest.raises(PccError):
            s.normalsKnn(None, k)
    for mean_k in (0, 512, -1):
        with pytest.raises(PccError):
            s.meanNeighbourDistance(None, mean_k)
    assert np.isfinite(s.meanNeighbourDistance(None, 511)).all()      # the limits themselves are accepted
    assert np.isfinite(s.normalsKnn(None, 512)[:, :3]).all()


# ---------------------------------------------------------------- 2. external queries through the radius normals
@pytest.mark.parametrize("radius", [0.03, 0.08])
def test_normals_radius_external_queries_and_viewpoint(GS, torch_cuda, radius):
    ref = synth.room(60000, 66)
    tree = oracle.KdTree(ref)
    s = GS().setInputCloud(ref, cell_hint=radius)
    rows, xyz = query_mix(s, ref, 67, n_noisy=20000)
    off, idx, _ = tree.radius(xyz, radius)
    want = oracle.normals_from_lists(ref, xyz, off, idx, VP)
    got = s.normalsRadius(rows, radius, viewpoint=VP)
    check_normals(got, want, xyz, VP)
    counts = np.diff(off)
    assert (counts == 0).any() and (counts >= 3).sum() > 1000
    assert radius > 0.05 or ((counts > 0) & (counts < 3)).any()          # 1 or 2 neighbours: NaN rows from the kernel, not a pre-fill
    gd = s.normalsRadius(torch_cuda.from_numpy(rows).cuda(), radius, viewpoint=VP)
    assert np.array_equal(bits(gd.cpu().numpy()), bits(got))
    got = s.normalsRadius(None, radius, viewpoint=VP)
    off, idx, _ = tree.radius(ref, radius)
    check_normals(got, oracle.normals_from_lists(ref, ref, off, idx, VP), ref, VP)


# ---------------------------------------------------------------- 3. `indices` subsets: oracle over pts[sub], pre-filled rows elsewhere
def _subset_like(n, seed):
    """[n, 4] room rows with 1 % NaN rows, a sorted random 40 % `indices` subset (so the oracle's tie order over pts[sub] is the GPU's
    order by original index), the mask of indexed rows, and per-row intensity and gradient inputs."""
    rng = np.random.default_rng(seed)
    pts = np.zeros((n, 4), np.float32)
    pts[:, :3] = synth.room(n, seed + 1)
    pts[:, 3] = 1.0
    pts[rng.choice(n, n // 100, replace=False), rng.integers(0, 3, n // 100)] = np.nan
    sub = np.sort(rng.choice(n, int(0.4 * n), replace=False)).astype(np.int32)
    indexed = np.zeros(n, bool)
    indexed[sub] = True
    indexed &= np.isfinite(pts[:, :3]).all(1)
    grad = rng.normal(0, 50, (n, 4)).astype(np.float32)
    grad[:, 3] = 0
    grad[::7, :3] = 0
    return pts, sub, indexed, (rng.random(n) * 255).astype(np.float32), grad


@pytest.fixture(scope="module")
def subset_cloud():
    pts, sub, indexed, inten, grad = _subset_like(30000, 70)
    P = np.ascontiguousarray(pts[sub])
    return pts, sub, P, oracle.KdTree(P), indexed, inten, grad


def _unit_rows(rng, m):
    v = rng.normal(size=(m, 4)).astype(np.float32)
    v[:, :3] /= np.linalg.norm(v[:, :3], axis=1, keepdims=True)
    v[:, 3] = 0
    return v


def _is_ff(a):
    return (np.ascontiguousarray(a, np.float32).view(np.uint32) == 0xFFFFFFFF).all()


def test_indices_subset_every_consumer(GS, subset_cloud):
    pts, sub, P, tree, indexed, inten, grad = subset_cloud
    n = len(pts)
    rn, rg, rr = 0.15, 0.15, 0.2
    s = GS().setInputCloud(pts, indices=sub, cell_hint=rr)
    assert s.size == indexed.sum()
    rows, xyz = query_mix(s, pts, 72)
    rng = np.random.default_rng(73)
    Pq = np.ascontiguousarray(P[:, :3])

    def to_rows(local):                                           # oracle over the queries P -> one row per input row of pts
        out = np.empty((n,) + local.shape[1:], local.dtype)
        out[sub] = local
        return out

    # kNN normals and mean distance
    for k in (16, 50):
        got = s.normalsKnn(None, k, viewpoint=VP)
        idx, _, _ = tree.knn(Pq, k)
        want = to_rows(oracle.normals_from_lists(pts, Pq, np.arange(len(P) + 1, dtype=np.int64) * k, np.where(idx >= 0, sub[idx], -1), VP))
        check_normals(got[indexed], want[indexed], pts[indexed], VP)
        assert _is_ff(got[~indexed])
        qn = s.normalsKnn(rows, k, viewpoint=VP)
        idx, _, _ = tree.knn(xyz, k)
        check_normals(qn, oracle.normals_from_lists(pts, xyz, np.arange(len(xyz) + 1, dtype=np.int64) * k, np.where(idx >= 0, sub[idx], -1), VP), xyz, VP)
    for mean_k in (8, 50):
        got = s.meanNeighbourDistance(None, mean_k)
        want = to_rows(oracle_mean_dist(tree, Pq, mean_k))
        assert np.array_equal(bits(got[indexed]), bits(want[indexed])) and (bits(got[~indexed]) == 0).all()
        assert np.array_equal(bits(s.meanNeighbourDistance(rows, mean_k)), bits(oracle_mean_dist(tree, xyz, mean_k)))

    # radius normals
    off, idx, _ = tree.radius(Pq, rn)
    got = s.normalsRadius(None, rn, viewpoint=VP)
    want = to_rows(oracle.normals_from_lists(pts, Pq, off, sub[idx], VP))
    check_normals(got[indexed], want[indexed], pts[indexed], VP)
    assert _is_ff(got[~indexed])
    offq, idxq, _ = tree.radius(xyz, rn)
    check_normals(s.normalsRadius(rows, rn, viewpoint=VP), oracle.normals_from_lists(pts, xyz, offq, sub[idxq], VP), xyz, VP)

    # intensity gradient: intensity per input row, normals per query row; pre-fill (NaN, NaN, NaN, 0)
    nrm = _unit_rows(rng, n)
    off, idx, _ = tree.radius(Pq, rg)
    got = s.intensityGradient(None, rg, inten, nrm)
    want = to_rows(D.intensity_gradient(pts, off, sub[idx], inten, nrm[sub]))
    assert same(got[indexed], want[indexed])
    assert np.isnan(got[~indexed, :3]).all() and (bits(got[~indexed, 3]) == 0).all() and (got[:, 3] == 0).all()
    nq = _unit_rows(rng, len(xyz))
    offq, idxq, _ = tree.radius(xyz, rg)
    assert same(s.intensityGradient(rows, rg, inten, nq), D.intensity_gradient(pts, offq, sub[idxq], inten, nq))

    # RIFT: gradients per input row; pre-fill 0xFF bytes
    off, idx, d2 = tree.radius(Pq, rr)
    got = s.rift(None, rr, grad)
    want = to_rows(D.rift(pts, Pq, off, sub[idx], d2, grad, rr))
    check_rift(got[indexed], want[indexed])
    assert _is_ff(got[~indexed])
    offq, idxq, d2q = tree.radius(xyz, rr)
    check_rift(s.rift(rows, rr, grad), D.rift(pts, xyz, offq, sub[idxq], d2q, grad, rr))

    # SIFT DoG (self only): field values per input row; pre-fill 0xFF bytes
    scales = D.sift_scales(0.02, 5)
    r = float(np.float32(3) * scales[-1])
    off, idx, d2 = tree.radius(Pq, r)
    got = s.siftDoG(inten, scales)
    want = to_rows(D.sift_dog(inten, off, sub[idx], d2, scales))
    assert same(got[indexed], want[indexed])
    assert _is_ff(got[~indexed])


def test_duplicated_indices_descriptor_consumers(GS):
    """An `indices` list that repeats rows: each copy is a point of its own in every neighbourhood (as in pcl::search over such a list),
    both copies write the same output row, and the rows left out keep their pre-fill."""
    rng = np.random.default_rng(74)
    pts = np.concatenate([rng.normal(0, 0.02, (6, 3)), [[3, 3, 3], [np.nan, 0, 0]]]).astype(np.float32)
    sub = np.array([0, 0, 1, 1, 2, 3, 3, 4, 6, 7], np.int32)            # row 5 left out, row 7 NaN
    indexed = np.zeros(len(pts), bool)
    indexed[[0, 1, 2, 3, 4, 6]] = True
    P = np.ascontiguousarray(pts[sub])
    tree = oracle.KdTree(P)
    s = GS().setInputCloud(pts, indices=sub, cell_hint=0.1)
    assert s.size == 9
    r = 0.2
    inten = (rng.random(len(pts)) * 255).astype(np.float32)
    nrm = _unit_rows(rng, len(pts))
    grad = rng.normal(0, 50, (len(pts), 4)).astype(np.float32)
    off, idx, d2 = tree.radius(P, r)
    assert np.diff(off)[0] == 8 and np.diff(off)[8] == 1                # 5 cluster rows indexed 8 times; the far row sees itself
    gi = D.intensity_gradient(pts, off, sub[idx], inten, nrm[sub])
    ri = D.rift(pts, P, off, sub[idx], d2, grad, r)
    scales = D.sift_scales(0.01, 5)
    rd = float(np.float32(3) * scales[-1])
    offd, idxd, d2d = tree.radius(P, rd)
    di = D.sift_dog(inten, offd, sub[idxd], d2d, scales)
    fin = np.isfinite(P).all(1)
    for j in np.flatnonzero(fin):                                       # both copies of a row give the same answer
        first = np.flatnonzero((sub == sub[j]) & fin)[0]
        assert same(gi[j], gi[first]) and same(ri[j], ri[first]) and same(di[j], di[first])
    want_g, want_r, want_d = np.empty((len(pts), 4), np.float32), np.empty((len(pts), 32), np.float32), np.empty((len(pts), 7), np.float32)
    want_g[sub], want_r[sub], want_d[sub] = gi, ri, di
    g = s.intensityGradient(None, r, inten, nrm)
    assert same(g[indexed], want_g[indexed]) and np.isnan(g[~indexed, :3]).all() and (bits(g[~indexed, 3]) == 0).all()
    assert np.isfinite(g[0, :3]).all()
    rf = s.rift(None, r, grad)
    check_rift(rf[indexed], want_r[indexed])
    assert _is_ff(rf[~indexed])
    dg = s.siftDoG(inten, scales)
    assert same(dg[indexed], want_d[indexed]) and _is_ff(dg[~indexed])


# ---------------------------------------------------------------- 4./5. every row written, both memory kinds, side streams
def _run_entries(s, torch, mem, rows, inputs, mean_k=8, k=16, r=0.15):
    """Every per-row consumer through its C entry, outputs pre-filled with a sentinel (numpy for PCC_HOST, CUDA tensors for PCC_DEVICE),
    inputs in the same memory kind, on torch's current stream.  rows=None: self queries.  Returns host copies."""
    from pointcloudcomparator_b200._lib import DEVICE, check
    L, h = s._L, s._h
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    n_in = s._n_input
    nrows = n_in if rows is None else len(rows)

    def out(shape, dtype, fill):
        if mem == DEVICE:
            t = torch.full(shape, fill, dtype={np.float32: torch.float32, np.int32: torch.int32, np.uint8: torch.uint8}[dtype], device="cuda")
            return t, t.data_ptr()
        a = np.full(shape, fill, dtype)
        return a, a.ctypes.data

    def inp(a):
        a = np.ascontiguousarray(a)
        if mem == DEVICE:
            t = torch.from_numpy(a).cuda()
            return t, t.data_ptr()
        return a, a.ctypes.data

    keep = []
    if rows is None:
        qp, nq, stride = None, 0, 16
    else:
        qt, qp = inp(rows)
        nq, stride = len(rows), rows.shape[1] * 4
        keep.append(qt)
    vp = (C.c_float * 3)(*VP)
    res = {}
    o, op = out((nrows,), np.float32, SENTINEL_F)
    check(L.pcc_knn_mean_dist(h, qp, nq, stride, mean_k, op, mem, st)); res["mean"] = o
    o, op = out((nrows, 4), np.float32, SENTINEL_F)
    check(L.pcc_normals_knn(h, qp, nq, stride, k, vp, op, mem, st)); res["normals_knn"] = o
    o, op = out((nrows, 4), np.float32, SENTINEL_F)
    check(L.pcc_normals_radius(h, qp, nq, stride, r, vp, op, mem, st)); res["normals_radius"] = o
    it, ip = inp(inputs["intensity"][:n_in]); nt, np_ = inp(inputs["normals"][:nrows]); gt, gp = inp(inputs["gradient"][:n_in])
    keep += [it, nt, gt]
    o, op = out((nrows, 4), np.float32, SENTINEL_F)
    check(L.pcc_intensity_gradient(h, qp, nq, stride, r, ip, np_, op, mem, st)); res["gradient"] = o
    o, op = out((nrows, 32), np.float32, SENTINEL_F)
    check(L.pcc_rift(h, qp, nq, stride, r, gp, 4, 8, op, mem, st)); res["rift"] = o
    if rows is None:
        sc = D.sift_scales(0.02, 5)                                        # the scale table is read on the host in both memory kinds
        o, op = out((n_in, 7), np.float32, SENTINEL_F)
        check(L.pcc_sift_dog(h, ip, sc.ctypes.data, sc.size, op, mem, st)); res["dog"] = o
        dist, dp = res["mean"], (res["mean"].data_ptr() if mem == DEVICE else res["mean"].ctypes.data)
        o, op = out((n_in,), np.uint8, SENTINEL_B)
        stats, kept = (C.c_double * 3)(), C.c_int64()
        check(L.pcc_sor_threshold(h, dp, n_in, s.size, 1.5, stats, op, C.byref(kept), mem, st)); res["keep"] = o
        res["sor_stats"] = np.array(list(stats) + [kept.value], np.float64)
    else:
        o, op = out((nrows,), np.int32, SENTINEL_I)
        check(L.pcc_first_within(h, qp, nq, stride, 0.05, op, mem, st)); res["first_within"] = o
    return {key: (v.cpu().numpy() if hasattr(v, "cpu") else np.array(v)) for key, v in res.items()}


@pytest.fixture(scope="module")
def entry_setup(GS):
    pts, sub, indexed, inten, grad = _subset_like(20000, 80)
    s = GS().setInputCloud(pts, indices=sub, cell_hint=0.15)
    rows, xyz = query_mix(s, pts, 81)
    rng = np.random.default_rng(82)
    inputs = dict(intensity=inten, normals=_unit_rows(rng, max(len(pts), len(rows))), gradient=grad)
    return s, pts, rows, inputs


def _sentinel_free(key, a):
    if a.dtype == np.float32:
        return not (bits(a) == bits(np.array([SENTINEL_F]))[0]).any()
    if a.dtype == np.uint8:
        return not (a == SENTINEL_B).any() and set(np.unique(a).tolist()) <= {0, 1}
    if a.dtype == np.int32:
        return not (a == SENTINEL_I).any()
    return True


@pytest.mark.parametrize("self_query", [True, False])
def test_every_row_written_host_and_device(torch_cuda, entry_setup, self_query):
    from pointcloudcomparator_b200._lib import DEVICE, HOST
    s, pts, rows, inputs = entry_setup
    q = None if self_query else rows
    host = _run_entries(s, torch_cuda, HOST, q, inputs)
    dev = _run_entries(s, torch_cuda, DEVICE, q, inputs)
    assert host.keys() == dev.keys()
    for key in host:
        assert _sentinel_free(key, host[key]), f"{key}: host rows left unwritten"
        assert _sentinel_free(key, dev[key]), f"{key}: device rows left unwritten"
        if host[key].dtype == np.float32:
            assert np.array_equal(bits(host[key]), bits(dev[key])), key
        else:
            assert np.array_equal(host[key], dev[key]), key
    if self_query:
        assert host["keep"].sum() == host["sor_stats"][3] < len(pts)
        assert (host["mean"][~np.isfinite(pts[:, :3]).all(1)] == 0).all()


def test_side_stream_matches_default_stream(torch_cuda, entry_setup):
    from pointcloudcomparator_b200._lib import DEVICE, HOST
    torch = torch_cuda
    s, pts, rows, inputs = entry_setup
    base = {(mem, sq): _run_entries(s, torch, mem, None if sq else rows, inputs) for mem in (HOST, DEVICE) for sq in (True, False)}
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for (mem, sq), want in base.items():
            got = _run_entries(s, torch, mem, None if sq else rows, inputs)
            for key in want:
                assert np.array_equal(np.ascontiguousarray(got[key]).view(np.uint8), np.ascontiguousarray(want[key]).view(np.uint8)), (mem, sq, key)
    torch.cuda.synchronize()


def _view(torch, ptr, nbytes):
    class _Mem:
        pass
    m = _Mem()
    m.__cuda_array_interface__ = {"shape": (nbytes // 4,), "typestr": "<f4", "data": (int(ptr), False), "version": 3}
    return torch.as_tensor(m, device="cuda:0")


def test_adopted_grid_filled_on_side_stream(GS, torch_cuda):
    """pcc_adopt, the arrays filled with copy_ on a non-blocking side stream and no synchronize, then every grid consumer on that
    stream: the occupancy bitmap and the inverse positions are derived on the caller's stream, after the fill."""
    torch = torch_cuda
    pts, sub, indexed, inten, grad = _subset_like(40000, 90)
    rng = np.random.default_rng(91)
    r = 0.05
    a = GS().setInputCloud(torch.from_numpy(pts).cuda(), indices=torch.from_numpy(sub).cuda(), cell_hint=r)
    rows, xyz = query_mix(a, pts, 92)
    qd = torch.from_numpy(rows).cuda()
    nrm = torch.from_numpy(_unit_rows(rng, len(pts))).cuda()
    dint, dgrad = torch.from_numpy(inten).cuda(), torch.from_numpy(grad).cuda()
    scales = D.sift_scales(0.01, 5)

    def run(s):
        off, idx, d2 = s.radiusSearch(qd, r)
        lab, sizes = s.euclideanClusters(r, 10, 1 << 30)
        return dict(off=off, idx=idx, d2=d2, normals_radius=s.normalsRadius(None, r, viewpoint=VP), gradient=s.intensityGradient(None, r, dint, nrm),
                    rift=s.rift(None, r, dgrad), dog=s.siftDoG(dint, scales), first=s.firstWithin(qd, r), labels=lab, sizes=sizes,
                    normals_knn=s.normalsKnn(None, 16, viewpoint=VP), mean=s.meanNeighbourDistance(None, 8), normals_knn_q=s.normalsKnn(qd, 50, viewpoint=VP))

    want = {key: v.cpu() for key, v in run(a).items()}
    meta, a_pts, a_cells = a.export()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        b = GS()
        _, b_pts, b_cells = b.adopt(meta)
        _view(torch, b_pts, int(meta[0]) * 16).copy_(_view(torch, a_pts, int(meta[0]) * 16))
        _view(torch, b_cells, (int(meta[11]) + 1) * 4).copy_(_view(torch, a_cells, (int(meta[11]) + 1) * 4))
        got = {key: v.cpu() for key, v in run(b).items()}
    torch.cuda.synchronize()
    for key in want:
        assert want[key].shape == got[key].shape and torch.equal(want[key].view(torch.uint8) if want[key].dtype == torch.float32 else want[key],
                                                                 got[key].view(torch.uint8) if got[key].dtype == torch.float32 else got[key]), key
    assert len(want["sizes"]) > 0 and len(want["idx"]) > 0


# ---------------------------------------------------------------- 6. SOR threshold at 1 M rows with NaN rows
def test_sor_threshold_million_rows_nan_rows_device(GS, torch_cuda):
    """n = 1 M distances: sor_sums_kernel's grid-stride loop runs 4 times (1024 blocks of 256).  1 % NaN rows carry a 0 distance and
    n_valid = s.size < n.  Host and device distances give identical statistics and masks, equal to oracle.sor; an fp64 numpy restatement
    (PCL's fp32-rounded squares) agrees within 1e-9, and the mean distances agree with a float64 scipy cKDTree within 1e-6 relative."""
    from scipy.spatial import cKDTree
    n, mean_k, mul = 1_000_000, 8, 1.5
    ref = synth.room(n, 95)
    bad = np.random.default_rng(96).choice(n, n // 100, replace=False)
    ref[bad, 2] = np.nan
    valid = np.isfinite(ref).all(1)
    s = GS().setInputCloud(ref, k_hint=mean_k + 1)
    assert s.size == valid.sum() < n
    dist = s.meanNeighbourDistance(None, mean_k)
    o = oracle.sor(ref, mean_k, mul)
    assert np.array_equal(bits(dist), bits(o["distances"])) and (dist[~valid] == 0).all()
    rh = s.sorThreshold(dist, s.size, mul)
    rd = s.sorThreshold(torch_cuda.from_numpy(dist).cuda(), s.size, mul)
    for key in ("mean", "stddev", "threshold"):
        assert abs(rh[key] - o[key]) <= 1e-9 * abs(o[key]), key
        assert rh[key] == rd[key], key                                     # same kernels, same reduction order
    assert rh["kept"] == rd["kept"] == o["kept"] < n
    assert np.array_equal(rh["keep"].astype(bool), o["keep"]) and np.array_equal(rd["keep"].cpu().numpy(), rh["keep"])
    d = dist.astype(np.float64)
    nv = float(valid.sum())
    sq = (dist * dist).astype(np.float64)                                   # PCL: sq_sum += distances[i] * distances[i] in fp32
    mean = d.sum() / nv
    sd = np.sqrt((sq.sum() - d.sum() ** 2 / nv) / (nv - 1.0))
    assert abs(rh["mean"] - mean) <= 1e-9 * mean and abs(rh["stddev"] - sd) <= 1e-9 * sd
    assert abs(rh["threshold"] - (mean + mul * sd)) <= 1e-9 * (mean + mul * sd)
    ref64 = ref[valid].astype(np.float64)
    dd, _ = cKDTree(ref64).query(ref64, mean_k + 1, workers=-1)
    md = dd[:, 1:].mean(1)
    rel = np.abs(dist[valid].astype(np.float64) - md) / md
    assert rel.max() <= 1e-6, rel.max()
