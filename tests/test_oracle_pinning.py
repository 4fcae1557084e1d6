"""Pins the CPU oracle (oracle/pcc_oracle.c) before anything is compared against it.

The reference has no tests or golden vectors for this path (SURVEY.md section 4) and PCL/FLANN are not
installable here, so the pins are: (1) committed golden vectors produced by OpenCV's bundled
FLANN KDTreeSingleIndex (tests/golden/make_golden.py), (2) the same library's answers on larger
and 32-D inputs, recorded by the same script, (3) scipy cKDTree at set level, (4) hand-derived
known answers.
"""
import hashlib
import os

import numpy as np
import pytest

import oracle
from conftest import bits
from pointcloudcomparator_b200 import synth


@pytest.fixture(scope="module")
def flann():
    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "opencv_flann_pins.npz"))


def _recorded(flann, name, ref, qry):
    """(idx, d2) of OpenCV's FLANN KDTreeSingleIndex (leaf 15, exact, sorted) on these inputs, as tests/golden/make_golden.py recorded them."""
    ref, qry = np.ascontiguousarray(ref, np.float32), np.ascontiguousarray(qry, np.float32)
    assert str(flann[f"{name}_inputs_sha256"]) == hashlib.sha256(ref.tobytes() + qry.tobytes()).hexdigest(), f"{name}: inputs differ from the recorded ones"
    return flann[f"{name}_idx"], flann[f"{name}_d2"]


def test_golden_knn(golden):
    ref, qry = golden["ref"], golden["qry"]
    tree = oracle.KdTree(ref)
    for k in (1, 16, 50):
        for idx, d2, _ in (tree.knn(qry, k), oracle.brute_knn(ref, qry, k)):
            assert np.array_equal(idx, golden[f"knn{k}_idx"])
            assert np.array_equal(bits(d2), bits(golden[f"knn{k}_d2"]))
    ti, td, _ = oracle.KdTree(golden["uref"]).knn(golden["uqry"], 16)
    assert np.array_equal(ti, golden["uknn16_idx"]) and np.array_equal(bits(td), bits(golden["uknn16_d2"]))


def test_golden_radius(golden):
    ref, qry, r = golden["ref"], golden["qry"], float(golden["radius"])
    for off, idx, d2 in (oracle.KdTree(ref).radius(qry, r), oracle.brute_radius(ref, qry, r)):
        assert np.array_equal(off, golden["rad_off"])
        assert np.array_equal(idx, golden["rad_idx"])
        assert np.array_equal(bits(d2), bits(golden["rad_d2"]))


def test_recorded_opencv_flann_knn(flann):
    ref = synth.room(60000, 1001)
    qry = synth.sweep_queries(ref, 3000, seed=9)[::3]
    ci, cd = _recorded(flann, "room60k_knn16", ref, qry)
    ti, td, _ = oracle.KdTree(ref).knn(qry, 16)
    assert np.array_equal(ci, ti) and np.array_equal(bits(cd), bits(td))


def test_lattice_ties_distance_multiset_matches_flann(flann):
    """FLANN keeps visit order among equal d2; the canonical order is (d2, idx).  Distances agree always."""
    g = np.arange(12, dtype=np.float32)
    ref = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3)
    qry = np.ascontiguousarray(ref[::7])
    _, cd = _recorded(flann, "lattice_knn8", ref, qry)
    ti, td, _ = oracle.KdTree(ref).knn(qry, 8)
    bi, bd, _ = oracle.brute_knn(ref, qry, 8)
    assert np.array_equal(bits(cd), bits(td))
    assert np.array_equal(ti, bi) and np.array_equal(bits(td), bits(bd))
    # canonical order: rows sorted by (d2, idx)
    key = td.astype(np.float64) * 1e7 + ti
    assert (np.diff(key, axis=1) > 0).all()


def test_scipy_set_level():
    from scipy.spatial import cKDTree
    ref = synth.uniform(30000, 5001, extent=2.0)
    qry = synth.sweep_queries(ref, 1000, seed=3, sigma=0.05)
    ti, _, _ = oracle.KdTree(ref).knn(qry, 10)
    _, si = cKDTree(ref.astype(np.float64)).query(qry.astype(np.float64), 10)
    same = np.mean([set(a) == set(b) for a, b in zip(ti, si)])
    assert same > 0.999   # float64 vs fp32 rounding may swap a near-tie at rank 10


def test_nan_rows_k_gt_n_and_duplicates():
    ref = np.array([[0, 0, 0], [np.nan, 0, 0], [1, 0, 0], [1, 0, 0], [0, 2, 0], [np.inf, 1, 1]], np.float32)
    qry = np.array([[0.9, 0, 0], [np.nan, 0, 0]], np.float32)
    for idx, d2, keff in (oracle.KdTree(ref).knn(qry, 6), oracle.brute_knn(ref, qry, 6)):
        assert keff == 4
        assert idx[0].tolist() == [2, 3, 0, 4, -1, -1]          # duplicates tie -> lower index first
        assert np.isinf(d2[0, 4:]).all() and (idx[1] == -1).all()
    assert oracle.KdTree(ref).size == 4


def test_radius_strict_boundary_and_max_nn():
    ref = np.array([[0, 0, 0], [0.5, 0, 0], [1.0, 0, 0], [0, 0.25, 0]], np.float32)
    qry = np.zeros((1, 3), np.float32)
    for fn in (lambda r, m: oracle.KdTree(ref).radius(qry, r, m), lambda r, m: oracle.brute_radius(ref, qry, r, m)):
        off, idx, d2 = fn(0.5, 0)            # d2 == r2 exactly -> excluded (strict <)
        assert idx.tolist() == [0, 3]
        off, idx, d2 = fn(0.5000001, 0)
        assert idx.tolist() == [0, 3, 1]
        off, idx, d2 = fn(2.0, 2)            # max_nn keeps the closest
        assert idx.tolist() == [0, 3]
        off, idx, d2 = fn(1e-3, 0)
        assert idx.tolist() == [0]


def test_normals_planar_patch_and_degenerate():
    rng = np.random.default_rng(0)
    p = np.zeros((400, 3), np.float32)
    p[:, :2] = rng.random((400, 2)) * 0.2 + 1.0
    p[:, 2] = 3.0
    n = oracle.normals_knn(p, 20)
    assert np.allclose(np.abs(n[:, 2]), 1.0, atol=1e-3) and (n[:, 2] < 0).all()      # flipped towards the origin; fp32 single-pass covariance is only ~1e-3 accurate here (PCL behaviour)
    assert np.all(n[:, 3] < 5e-3)
    # fewer than 3 neighbours -> NaN
    off, idx, _ = oracle.KdTree(p[:2]).radius(p[:2], 10.0)
    out = oracle.normals_from_lists(p[:2], p[:2], off, idx)
    assert np.isnan(out).all()


def test_sor_known_answer():
    g = np.arange(10, dtype=np.float32)
    ref = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3)
    ref = np.concatenate([ref, np.array([[30, 30, 30]], np.float32)])
    r = oracle.sor(ref, mean_k=6, std_mul=1.5)
    assert not r["keep"][-1] and r["keep"][555]
    assert np.isclose(r["distances"][555], 1.0)       # interior lattice point: 6 neighbours at distance 1


def test_ece_two_blobs_gap_and_size_filter():
    rng = np.random.default_rng(1)
    a = rng.random((300, 3)).astype(np.float32) * 0.1
    b = a + np.array([0.1 + 0.06, 0, 0], np.float32)          # nearest gap 0.06
    small = np.array([[5, 5, 5], [5.01, 5, 5]], np.float32)
    pts = np.concatenate([a, b, small])
    lab, sizes = oracle.KdTree(pts).ece(0.05, 100, 250000)
    assert sizes.tolist() == [300, 300] and set(lab[:300]) == {0} and set(lab[300:600]) == {1} and (lab[600:] == -1).all()
    lab, sizes = oracle.KdTree(pts).ece(0.07, 100, 250000)
    assert sizes.tolist() == [600]
    lab, sizes = oracle.KdTree(pts).ece(0.07, 100, 500)        # over max -> dropped whole
    assert sizes.tolist() == [] and (lab == -1).all()


def test_ece_scene_known_cluster_count():
    pts, ids = synth.scene(80000, 3001, extent=6.0, n_objects=25)
    lab, sizes = oracle.KdTree(pts).ece(0.05, 100, 250000)
    assert len(sizes) == 25
    # one label per object
    for o in range(25):
        assert len(set(lab[ids == o])) == 1
    assert (np.diff(sizes) <= 0).all()


def test_icp_recovers_rigid_transform():
    src, tgt, T = synth.icp_pair(40000, 4001, size=(5, 5, 3))
    r = oracle.icp(src, tgt, 20)
    assert r["converged"] and r["iterations"] <= 20
    Tinv = np.linalg.inv(T)
    assert np.allclose(r["T"], Tinv, atol=2e-4)
    assert r["fitness"] < 1e-5


def test_umeyama_reflection_guard():
    rng = np.random.default_rng(5)
    s = rng.normal(size=(50, 3))
    R = np.array([[0, -1, 0], [1, 0, 0], [0, 0, 1.0]])
    t = s @ R.T + np.array([1, 2, 3.0])
    sums = np.zeros(16)
    sums[0:3], sums[3:6], sums[6:15] = s.sum(0), t.sum(0), (t.T @ s).reshape(-1)
    T = oracle.umeyama_from_sums(sums, 50)
    assert np.allclose(T[:3, :3], R, atol=1e-6) and np.allclose(T[:3, 3], [1, 2, 3], atol=1e-5)


def test_first_within():
    pts = np.array([[0, 0, 0], [0.04, 0, 0], [0.01, 0, 0]], np.float32)
    q = np.array([[0.03, 0, 0], [1, 1, 1]], np.float32)
    assert oracle.first_within(pts, q, 0.05).tolist() == [0, -1]


def test_voxel_grid_known_answers():
    # two points in one 1 m voxel, one alone; colour averaged and truncated; output ordered by voxel index (x fastest)
    rows = np.zeros((3, 8), np.float32)
    rows[:, :3] = [[2.25, 0.5, 0.5], [0.25, 0.25, 0.25], [0.75, 0.5, 0.75]]
    rows[:, 3] = 1.0
    col = rows[:, 4:5].view(np.uint8)                       # BGRA bytes
    col[0] = [10, 20, 30, 0]; col[1] = [0, 100, 255, 0]; col[2] = [1, 101, 0, 0]
    out = oracle.voxel_grid(rows, 1.0, rgb_offset_floats=4)
    assert out.shape[0] == 2
    assert np.allclose(out[0, :3], [0.5, 0.375, 0.5]) and np.allclose(out[1, :3], [2.25, 0.5, 0.5])
    assert out[0, 4:5].view(np.uint8).tolist() == [0, 100, 127, 0] and out[1, 4:5].view(np.uint8).tolist() == [10, 20, 30, 0]
    assert (out[:, 3] == 1.0).all()
    # distinct-voxel count equals numpy's, NaN rows are ignored
    p = synth.room(50000, 1001, stride4=True)
    p[7, 0] = np.nan
    o = oracle.voxel_grid(p, 0.025)
    fin = np.isfinite(p[:, :3]).all(1)
    ijk = np.floor(p[fin, :3] * np.float32(1 / np.float32(0.025))).astype(np.int64)
    assert o.shape[0] == len(np.unique(ijk, axis=0))
    vox = np.floor(o[:, :3] * np.float32(1 / np.float32(0.025)) + 1e-4).astype(np.int64)
    assert len(np.unique(vox, axis=0)) >= 0.999 * o.shape[0]      # every centroid stays inside its own voxel (up to fp32 rounding on faces)


def test_descriptor_nn_matches_opencv_flann_32d(flann):
    rng = np.random.default_rng(3)
    ref = rng.random((700, 32), dtype=np.float32) * 0.3
    qry = (ref[rng.integers(0, 700, 400)] + rng.normal(0, 0.02, (400, 32))).astype(np.float32)
    ci, cd = _recorded(flann, "desc32_nn", ref, qry)                       # same index family KdTreeFLANN<Histogram<32>> builds
    oi, od = oracle.descriptor_nn(ref, qry)
    # OpenCV's FLANN uses the 4-way unrolled cvflann::L2 functor (sums four squared differences per step); PCL's KdTreeFLANN
    # uses L2_Simple (one dimension at a time), which the oracle restates.  Same neighbours, distances equal to a few ulp.
    assert np.array_equal(ci[:, 0], oi) and np.allclose(cd[:, 0], od, rtol=1e-6, atol=0)
    ref[5, 7] = np.nan; qry[3, 0] = np.inf
    oi, od = oracle.descriptor_nn(ref, qry)
    assert (oi != 5).all() and oi[3] == -1 and np.isinf(od[3])


# ---------------------------------------------------------------------------------------------------------------------
# Independent pins of the CONSUMER restatements (round 2).  Each check below compares the oracle with code that shares
# nothing with oracle/pcc_oracle.c or the CUDA product: numpy/scipy library routines, or a plain-Python restatement written
# from the published PCL 1.7 / Eigen algorithm.  A shared misreading between product and oracle can no longer pass unseen.

def _eigh_normals(ref, idx_rows):
    """fp64 covariance of each neighbour list + numpy.linalg.eigh: smallest eigenvector, curvature = l0 / (l0 + l1 + l2)."""
    out = np.zeros((len(idx_rows), 4)); gap = np.zeros(len(idx_rows))
    for i, nb in enumerate(idx_rows):
        p = ref[nb].astype(np.float64)
        c = np.cov(p.T, bias=True)
        w, v = np.linalg.eigh(c)
        out[i, :3], out[i, 3] = v[:, 0], abs(w[0] / w.sum())
        gap[i] = (w[1] - w[0]) / w.sum()
    return out, gap


def test_normals_vs_numpy_eigh():
    """NormalEstimation (src/segmentation.cpp:236-240, k = 50; src/comparator.cpp:628-635, r = 0.03) vs LAPACK's symmetric eigensolver
    in fp64 on the same neighbour lists: direction within 1e-4 rad wherever the smallest eigenvalue is separated, curvature rtol 1e-3."""
    ref = synth.room(30000, 1001, size=(1.5, 1.0, 0.7))     # ~4600 points per m2: a 3 cm ball holds ~13 points
    tree = oracle.KdTree(ref)
    sel = np.arange(0, 30000, 15)
    for name, rows, nrm in (
        ("k50", tree.knn(ref, 50)[0][sel], oracle.normals_knn(ref, 50, tree=tree)[sel]),
        ("r03", None, oracle.normals_radius(ref, 0.03, tree=tree)[sel]),
    ):
        if rows is None:
            off, idx, _ = tree.radius(ref, 0.03)
            rows = [idx[off[i]:off[i + 1]] for i in sel]
        ok = np.array([len(r) >= 3 for r in rows])
        big = np.array([len(r) >= 8 for r in rows])[ok]
        exp, gap = _eigh_normals(ref, [r for r, o in zip(rows, ok) if o])
        got = nrm[ok].astype(np.float64)
        assert np.isnan(nrm[~ok]).all(), name
        well = (gap > 1e-3) & big
        assert well.mean() > 0.8, name
        cosang = np.abs((got[:, :3] * exp[:, :3]).sum(1))
        # PCL accumulates the covariance in ONE fp32 pass (E[pp^T] - mu mu^T) on raw room coordinates (|p| up to 7 m, neighbour
        # spread ~5 cm): that cancellation costs ~1e-3 rad against the fp64 two-pass answer and is reference behaviour (the tight
        # fp32 parity of product vs oracle is tested on the GPU); what is pinned here is the algorithm: which eigenvector, its
        # sign convention, and the curvature formula.
        ang = np.arccos(np.clip(cosang[well], 0, 1))
        assert np.quantile(ang, 0.99) < 2e-2 and np.median(ang) < 2e-3, (name, np.quantile(ang, 0.99), np.median(ang))
        # flipped towards the viewpoint (origin): n . (vp - p) >= 0
        assert ((got[:, :3] * (-ref[sel][ok])).sum(1) >= -1e-6).all(), name
        assert np.allclose(np.linalg.norm(got[:, :3], axis=1), 1.0, atol=1e-5), name
    # the same comparison where fp32 cancellation is negligible (cloud centred at the origin, 2 cm patch): tight agreement
    rng = np.random.default_rng(3)
    small = (rng.normal(size=(4000, 3)) * np.array([0.02, 0.02, 0.002])).astype(np.float32)
    R, _ = np.linalg.qr(rng.normal(size=(3, 3)))
    small = (small @ R.T.astype(np.float32)).astype(np.float32)
    t2 = oracle.KdTree(small)
    rows = t2.knn(small, 30)[0]
    got = oracle.normals_knn(small, 30, tree=t2).astype(np.float64)
    exp, gap = _eigh_normals(small, rows)
    well = gap > 1e-3
    ang = np.linalg.norm(np.cross(got[:, :3], exp[:, :3]), axis=1)       # sin(angle): resolves below the 3e-4 rad floor of arccos on fp32 unit vectors
    # eigenvector perturbation theory: an fp32 covariance (relative error ~1e-6 of the trace) moves the eigenvector by error / gap
    assert well.mean() > 0.95 and (ang * gap)[well].max() < 3e-5 and np.median(ang) < 2e-5, ((ang * gap)[well].max(), np.median(ang))
    assert ang[gap > 0.1].max() < 2e-4
    assert np.allclose(got[well, 3], exp[well, 3], rtol=1e-3, atol=1e-7)


def test_ece_vs_scipy_connected_components():
    """EuclideanClusterExtraction (src/segmentation.cpp:125-131) = connected components of the radius graph, size-filtered, largest
    first, indices ascending inside a cluster -- against scipy.sparse.csgraph over cKDTree.query_pairs."""
    from scipy.sparse import coo_matrix
    from scipy.sparse.csgraph import connected_components
    from scipy.spatial import cKDTree
    pts, _ = synth.scene(60000, 3001, extent=5.0, n_objects=18)
    rng = np.random.default_rng(11)
    pts = np.concatenate([pts, rng.random((300, 3)).astype(np.float32) * 5.0])          # stray points: tiny clusters that the size filter drops
    tol = 0.05
    tr = cKDTree(pts.astype(np.float64))
    n = len(pts)
    parts = []
    for r in (tol - 1e-6, tol + 1e-6):                      # the components do not depend on the edges at the strict `<` boundary,
        pairs = tr.query_pairs(r, output_type="ndarray")    # so fp64 (scipy) and fp32 (FLANN arithmetic) must agree on them
        parts.append(connected_components(coo_matrix((np.ones(len(pairs)), (pairs[:, 0], pairs[:, 1])), shape=(n, n)), directed=False))
    assert parts[0][0] == parts[1][0] and np.array_equal(parts[0][1], parts[1][1])
    ncomp, comp = parts[0]
    size = np.bincount(comp, minlength=ncomp)
    lab, sizes = oracle.KdTree(pts).ece(tol, 100, 250000)
    keep = np.flatnonzero((size >= 100) & (size <= 250000))
    assert sorted(sizes.tolist(), reverse=True) == sizes.tolist() == sorted(size[keep].tolist(), reverse=True)
    assert ((lab >= 0) == np.isin(comp, keep)).all()
    # same partition: one oracle label per scipy component and vice versa
    m = lab >= 0
    assert len(set(zip(lab[m].tolist(), comp[m].tolist()))) == len(keep) == len(sizes)
    # the over-max rule drops a component whole
    lab2, sizes2 = oracle.KdTree(pts).ece(tol, 100, int(sizes[0]) - 1)
    assert sizes2.tolist() == sizes[1:].tolist() and (lab2[lab == 0] == -1).all()


def _eigen_umeyama(src, dst, dtype):
    """Eigen::umeyama(src, dst, with_scaling = false) as published (Eigen/src/Geometry/Umeyama.h), which PCL 1.7's
    TransformationEstimationSVD::estimateRigidTransformation calls on 3 x n matrices; numpy SVD instead of JacobiSVD."""
    src, dst = np.asarray(src, dtype), np.asarray(dst, dtype)
    n = src.shape[0]
    one_over_n = dtype(1) / dtype(n)
    sm, dm = src.sum(0, dtype=dtype) * one_over_n, dst.sum(0, dtype=dtype) * one_over_n
    sd, dd = src - sm, dst - dm
    sigma = (one_over_n * (dd.T @ sd)).astype(dtype)
    U, d, Vt = np.linalg.svd(sigma)
    S = np.ones(3, dtype)
    if np.linalg.det(sigma) < 0:
        S[2] = -1
    rank = int((np.abs(d) > np.finfo(dtype).eps * np.abs(d[0])).sum())
    if rank == 2:
        if np.linalg.det(U) * np.linalg.det(Vt) > 0:
            Rm = U @ Vt
        else:
            S2 = S.copy(); S2[2] = -1
            Rm = U @ np.diag(S2) @ Vt
    else:
        Rm = U @ np.diag(S) @ Vt
    T = np.eye(4, dtype=dtype)
    T[:3, :3] = Rm
    T[:3, 3] = dm - Rm @ sm
    return T


def test_umeyama_vs_numpy_svd():
    """TransformationEstimationSVD (ICP, src/comparator.cpp:1089-1099): the oracle's closed-form 3x3 SVD + reflection guard vs
    numpy's LAPACK SVD driving Eigen's published umeyama(), in fp64 and in fp32 (PCL's Scalar)."""
    rng = np.random.default_rng(21)
    for case in range(6):
        n = 500
        s = rng.normal(size=(n, 3)) * [1.0, 0.7, 0.4] + rng.normal(size=3) * 3
        a = rng.normal(size=3); a /= np.linalg.norm(a); th = rng.uniform(0.01, 2.5)
        K = np.array([[0, -a[2], a[1]], [a[2], 0, -a[0]], [-a[1], a[0], 0]])
        R = np.eye(3) + np.sin(th) * K + (1 - np.cos(th)) * K @ K
        t = s @ R.T + rng.normal(size=3) + rng.normal(size=(n, 3)) * 1e-3
        if case == 4:                                       # planar source (rank 2): the branch with the determinant test
            s[:, 2] = 0.0; t = s @ R.T + [0.3, -0.2, 0.1]
        if case == 5:                                       # mirrored target: the reflection guard must return a proper rotation
            t = s * [1, 1, -1] + rng.normal(size=(n, 3)) * 1e-3
        s32, t32 = s.astype(np.float32), t.astype(np.float32)
        sums = np.zeros(16)
        sums[0:3], sums[3:6] = s32.astype(np.float64).sum(0), t32.astype(np.float64).sum(0)
        sums[6:15] = (t32.astype(np.float64).T @ s32.astype(np.float64)).reshape(-1)
        T = oracle.umeyama_from_sums(sums, n).astype(np.float64)
        T64 = _eigen_umeyama(s32, t32, np.float64)
        T32 = _eigen_umeyama(s32, t32, np.float32).astype(np.float64)
        assert abs(np.linalg.det(T[:3, :3]) - 1) < 1e-5, case
        assert np.allclose(T, T64, atol=2e-6, rtol=1e-6), (case, np.abs(T - T64).max())
        # fp32 Eigen arithmetic (what PCL's Scalar = float runs) agrees with the fp64-sum restatement to fp32 accumulation error:
        # the reference's own result moves by this much with Eigen's (unspecified, vectorised) summation order
        assert np.allclose(T, T32, atol=5e-5, rtol=1e-4), (case, np.abs(T - T32).max())


def test_voxel_grid_vs_numpy_lexsort():
    """VoxelGrid::applyFilter (src/segmentation.cpp:69-74, 223-228; leaf 0.025): voxel index from floor(p * inv_leaf) - min index,
    output ordered by linear voxel index (x fastest), centroid = mean of x, y, z -- against numpy lexsort + add.reduceat in fp64."""
    p = synth.room(80000, 1001, stride4=True)
    p[11, 1] = np.nan
    leaf = np.float32(0.025)
    inv = np.float32(1.0) / leaf
    fin = np.isfinite(p[:, :3]).all(1)
    q = p[fin]
    lo, hi = q[:, :3].min(0), q[:, :3].max(0)
    mn = np.floor(lo * inv).astype(np.int64)
    ijk = np.floor(q[:, :3] * inv).astype(np.int64) - mn
    div = np.floor(hi * inv).astype(np.int64) - mn + 1
    lin = ijk[:, 0] + ijk[:, 1] * div[0] + ijk[:, 2] * div[0] * div[1]
    order = np.lexsort((np.arange(len(lin)), lin))
    starts = np.flatnonzero(np.r_[True, np.diff(lin[order]) != 0])
    cnt = np.diff(np.r_[starts, len(lin)])
    cen = np.add.reduceat(q[order, :3].astype(np.float64), starts, axis=0) / cnt[:, None]
    out = oracle.voxel_grid(p, float(leaf))
    assert out.shape[0] == len(starts)
    assert np.allclose(out[:, :3], cen, rtol=2e-6, atol=2e-6)          # fp32 running sums vs fp64
    assert (out[:, 3] == 1.0).all()
    # min_points_per_voxel drops sparse voxels
    out3 = oracle.voxel_grid(p, float(leaf), min_points=3)
    assert out3.shape[0] == int((cnt >= 3).sum()) and np.allclose(out3[:, :3], cen[cnt >= 3], rtol=2e-6, atol=2e-6)


def _py_region_growing(nb, normals, theta, curv_thr, min_size, max_size):
    """pcl::RegionGrowing::extract restated in plain Python from the published PCL 1.7 algorithm (region_growing.hpp:
    applySmoothRegionGrowingAlgorithm / growRegion / validatePoint, smooth mode on, curvature test on, residual test off)."""
    from collections import deque
    n = len(nb)
    label = [-1] * n
    cos_thr = np.float32(np.cos(np.float32(theta)))
    curv = normals[:, 3]
    order = sorted(range(n), key=lambda i: (np.inf if np.isnan(curv[i]) else curv[i], i))
    nrm = normals[:, :3]
    seg = 0; sizes = []
    for seed in order:
        if label[seed] != -1:
            continue
        label[seed] = seg; cnt = 1
        dq = deque([seed])
        while dq:
            cur = dq.popleft()
            for j in nb[cur]:
                if j < 0 or label[j] != -1:
                    continue
                a, b = nrm[j], nrm[cur]
                dot = np.float32(abs(np.float32(np.float32(np.float32(a[0] * b[0]) + np.float32(a[1] * b[1])) + np.float32(a[2] * b[2]))))
                if not dot >= cos_thr:          # "dot < threshold -> reject"; a NaN dot product is not < threshold, PCL keeps it
                    if dot < cos_thr:
                        continue
                label[j] = seg; cnt += 1
                if not curv[j] > curv_thr:
                    dq.append(j)
        sizes.append(cnt); seg += 1
    keep = [s for s in range(seg) if min_size <= sizes[s] <= max_size]
    remap = {s: i for i, s in enumerate(keep)}
    return np.array([remap.get(l, -1) for l in label], np.int32), len(keep)


def test_region_growing_vs_python_fifo():
    """RegionGrowing as configured at src/segmentation.cpp:249-271 (k = 30 here to keep the Python loop short)."""
    ref = synth.room(6000, 1001, size=(2.0, 1.5, 1.0))
    tree = oracle.KdTree(ref)
    nb = tree.knn(ref, 30)[0]
    normals = oracle.normals_knn(ref, 20, tree=tree)
    for theta, cthr, mn in ((3.0 / 180 * np.pi, 1.0, 50), (8.0 / 180 * np.pi, 0.05, 20)):
        lab, nc = oracle.region_growing(nb, normals, theta, cthr, mn, 1000000)
        plab, pnc = _py_region_growing(nb, normals, theta, cthr, mn, 1000000)
        assert nc == pnc and nc > 3
        assert np.array_equal(lab, plab)


def test_sor_vs_numpy():
    """StatisticalOutlierRemoval (src/comparator.cpp:1523-1527): mean of sqrt(d2[1..k]) in double -> float; mean / (n-1)-variance of
    those in double; keep dist <= mean + mul * stddev -- against numpy on scipy's neighbour distances."""
    from scipy.spatial import cKDTree
    ref = synth.room(20000, 2001)
    ref[::997] += 0.4                                       # a few outliers
    k = 50
    r = oracle.sor(ref, k, 1.5)
    d, _ = cKDTree(ref.astype(np.float64)).query(ref.astype(np.float64), k + 1)
    md = d[:, 1:].mean(1)
    assert np.allclose(r["distances"], md, rtol=2e-6)
    dist = r["distances"].astype(np.float64)
    n = len(dist)
    mean = dist.sum() / n
    var = ((dist ** 2).sum() - dist.sum() ** 2 / n) / (n - 1)
    thr = mean + 1.5 * np.sqrt(var)
    assert np.isclose(r["mean"], mean, rtol=1e-12) and np.isclose(r["stddev"], np.sqrt(var), rtol=1e-9) and np.isclose(r["threshold"], thr, rtol=1e-9)
    assert np.array_equal(r["keep"], dist <= thr) and 0 < (~r["keep"]).sum() < 0.2 * n


def test_icp_vs_numpy_loop():
    """IterativeClosestPoint::computeTransformation + DefaultConvergenceCriteria + getFitnessScore (src/comparator.cpp:1089-1099):
    the oracle's loop against a numpy / scipy restatement of the published PCL 1.7 algorithm (cKDTree correspondences, Eigen's
    umeyama through numpy SVD, the rotation / translation / relative-MSE criteria, max 20 iterations)."""
    from scipy.spatial import cKDTree
    src, tgt, _ = synth.icp_pair(20000, 4001, size=(4, 4, 2))
    r = oracle.icp(src, tgt, 20)
    tr = cKDTree(tgt.astype(np.float64))
    cur = src.astype(np.float32)
    final = np.eye(4, dtype=np.float32)
    prev_mse, it, conv = None, 0, False
    similar = 0
    while True:
        d, j = tr.query(cur.astype(np.float64), 1)
        T = _eigen_umeyama(cur, tgt[j], np.float64).astype(np.float32)
        cur = (cur.astype(np.float32) @ T[:3, :3].T + T[:3, 3]).astype(np.float32)
        final = (T @ final).astype(np.float32)
        it += 1
        mse = float((d.astype(np.float64) ** 2).sum() / len(d))
        cos_angle = 0.5 * (T[0, 0] + T[1, 1] + T[2, 2] - 1)
        trans2 = float((T[:3, 3].astype(np.float64) ** 2).sum())
        if it >= 20:
            conv = True; break
        if cos_angle >= 1.0 and trans2 <= 0.0:      # PCL defaults: rotation threshold 1.0 (cos), translation threshold 0 (ICP sets transformation_epsilon_ = 0)
            similar += 1
            if similar >= 1: conv = True; break
        else:
            similar = 0
        if prev_mse is not None and abs(mse - prev_mse) < 1e-12:
            conv = True; break
        prev_mse = mse
    d, _ = tr.query(cur.astype(np.float64), 1)
    fit = float((d ** 2).mean())
    assert r["converged"] == conv
    assert abs(r["iterations"] - it) <= 1
    assert np.allclose(r["T"], final, atol=5e-5)
    assert np.isclose(r["fitness"], fit, rtol=2e-3)


def test_descriptor_nn_three_dims_matches_flann_on_first_three_bins(flann):
    """PCL 1.7's DefaultPointRepresentation clamps an unregistered point type to its first 3 floats, so the reference's
    KdTreeFLANN<Histogram<32>> (src/comparator.cpp:564-577) is a 3-D tree over bins 0..2: the oracle's dims = 3 mode against a
    FLANN KDTreeSingleIndex built on exactly those columns."""
    rng = np.random.default_rng(8)
    ref = rng.random((900, 32), dtype=np.float32) * 0.3
    qry = (ref[rng.integers(0, 900, 500)] + rng.normal(0, 0.02, (500, 32))).astype(np.float32)
    ci, cd = _recorded(flann, "desc3_nn", ref[:, :3], qry[:, :3])
    oi, od = oracle.descriptor_nn(ref, qry, dims=3)
    assert np.array_equal(ci[:, 0], oi) and np.allclose(cd[:, 0], od, rtol=1e-6, atol=0)
    o32, _ = oracle.descriptor_nn(ref, qry)
    assert (o32 != oi).any()                               # the two modes really differ on this data
