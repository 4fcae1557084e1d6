"""CPU pins of the descriptor-stage oracle (descriptor_oracle/): IntensityGradientEstimation, RIFTEstimation and PCL's
PointXYZRGBtoXYZI, against known answers and independent numpy restatements.  No GPU needed."""
import numpy as np
import pytest

import descriptor_oracle as D
import oracle
from pointcloudcomparator_b200 import synth
from pointcloudcomparator_b200.search import rgb_to_intensity

EPS32 = float(np.finfo(np.float32).eps)


# ---------------------------------------------------------------- intensity
def test_rgb_to_intensity_hand_values():
    rgb = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, 1], [255, 255, 255], [100, 50, 200]], np.uint8)
    f = np.float32
    want = np.array([0.0, f(0.299), f(0.587), f(0.114),
                     (f(0.299) * f(255) + f(0.587) * f(255)) + f(0.114) * f(255),
                     (f(0.299) * f(100) + f(0.587) * f(50)) + f(0.114) * f(200)], np.float32)
    for got in (rgb_to_intensity(rgb), D.rgb_to_intensity(rgb)):
        assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    assert abs(float(want[4]) - 255.0) < 1e-4 and abs(float(want[5]) - (29.9 + 29.35 + 22.8)) < 1e-4


def test_rgb_to_intensity_mirror_equals_oracle_everywhere():
    rgb = np.random.default_rng(5).integers(0, 256, (200000, 3)).astype(np.uint8)
    assert np.array_equal(rgb_to_intensity(rgb).view(np.uint32), D.rgb_to_intensity(rgb).view(np.uint32))


# ---------------------------------------------------------------- column-pivoting QR
def test_colpiv_qr_full_rank_matches_lstsq():
    rng = np.random.default_rng(1)
    for _ in range(200):
        Q = rng.normal(size=(3, 3))
        A = (Q @ Q.T + 0.5 * np.eye(3)).astype(np.float32)
        b = rng.normal(size=3).astype(np.float32)
        x = D.colpiv_qr_solve(A, b)
        ref = np.linalg.solve(A.astype(np.float64), b.astype(np.float64))
        assert np.abs(x - ref).max() <= 1e-4 * np.linalg.cond(A.astype(np.float64)) * np.abs(ref).max()


def test_colpiv_qr_rank_two_zeroes_the_free_unknown():
    """A planar neighbourhood on z = const: row and column 2 of A are exactly zero, the rank is decided as 2 and the unknown
    of the zero column is returned as 0 (Eigen: back substitution over the nonzero pivots, zeros for the rest)."""
    rng = np.random.default_rng(2)
    for _ in range(50):
        Q = rng.normal(size=(2, 2))
        A = np.zeros((3, 3), np.float32)
        A[:2, :2] = Q @ Q.T + 0.3 * np.eye(2)
        b = np.array([rng.normal(), rng.normal(), 0.0], np.float32)
        x = D.colpiv_qr_solve(A, b)
        assert x[2] == 0.0
        assert np.allclose(x[:2], np.linalg.solve(A[:2, :2].astype(np.float64), b[:2].astype(np.float64)), rtol=1e-4, atol=1e-6)
    assert np.array_equal(D.colpiv_qr_solve(np.zeros((3, 3)), np.zeros(3)), np.zeros(3, np.float32))


# ---------------------------------------------------------------- gradient: known answer
def _patch(rng, m, normal, noise):
    n = np.asarray(normal, np.float64); n /= np.linalg.norm(n)
    u = np.cross(n, [1.0, 0.0, 0.0] if abs(n[0]) < 0.9 else [0.0, 1.0, 0.0]); u /= np.linalg.norm(u)
    v = np.cross(n, u)
    st = rng.uniform(-0.02, 0.02, (m, 2))
    p = np.array([1.0, 2.0, 0.5]) + st[:, :1] * u + st[:, 1:] * v + rng.normal(0, noise, (m, 1)) * n
    return p, n


@pytest.mark.parametrize("planar", [True, False])
def test_gradient_linear_intensity_known_answer(planar):
    """I = c + a.p: in exact arithmetic b = A a, so every solver gives the in-plane part of a and the gradient is (I - n n^T) a.
    fp32 bound: the centred coordinates, A and b carry a relative rounding error of about m * eps each (sequential sums of m
    terms), the solve multiplies it by the in-plane condition kappa of A; 50 * m * eps * kappa * |a| leaves a 10x margin over
    what the noisy patch shows.  planar=True: an exactly planar z = 0.5 patch (rank-2 branch, the normal component of x is
    undetermined and the projection removes it)."""
    rng = np.random.default_rng(3 if planar else 4)
    a = np.array([3.0, -2.0, 5.0])
    for _ in range(20):
        m = int(rng.integers(12, 60))
        if planar:
            st = rng.uniform(-0.02, 0.02, (m, 2))
            p = np.column_stack([1.0 + st[:, 0], 2.0 + st[:, 1], np.full(m, 0.5)])
            n = np.array([0.0, 0.0, 1.0])
        else:
            p, n = _patch(rng, m, rng.normal(size=3), 0.002)
        pts = p.astype(np.float32)
        inten = (0.25 + pts.astype(np.float64) @ a * 0.01).astype(np.float32) * 100.0
        inten = inten.astype(np.float32)
        off = np.array([0, m], np.int64)
        nbr = np.arange(m, dtype=np.int32)
        g = D.intensity_gradient(pts, off, nbr, inten, n[None].astype(np.float32))[0, :3].astype(np.float64)
        want = a - n * (n @ a)
        P = pts.astype(np.float64) - pts.astype(np.float64).mean(0)
        w = np.linalg.eigvalsh(P.T @ P)
        kappa = w[2] / w[1]
        assert np.abs(g - want).max() <= 50 * m * EPS32 * kappa * np.linalg.norm(a), (g, want)


def test_gradient_nan_below_three_neighbours_and_zero_fourth_component():
    pts = np.array([[0, 0, 0], [0.01, 0, 0], [0, 0.01, 0]], np.float32)
    inten = np.array([1, 2, 3], np.float32)
    off = np.array([0, 0, 1, 3, 6], np.int64)
    nbr = np.array([0, 0, 1, 0, 1, 2], np.int32)
    g = D.intensity_gradient(pts, off, nbr, inten, np.tile([[0, 0, 1]], (4, 1)))
    assert np.isnan(g[:3, :3]).all() and np.isfinite(g[3]).all() and (g[:, 3] == 0).all()


# ---------------------------------------------------------------- gradient: independent pin
@pytest.fixture(scope="module")
def room_rows():
    xyz = synth.room(400000, 11)[:, :3]
    inten = rgb_to_intensity(synth.rgb_for(xyz, 12))
    tree = oracle.KdTree(xyz)
    off, idx, d2 = tree.radius(xyz, 0.03)
    nrm = oracle.normals_from_lists(xyz, xyz, off, idx)
    return xyz, inten, tree, off, idx, nrm


def test_gradient_pinned_to_fp64_lstsq_on_room(room_rows):
    """numpy fp64: A and b from the oracle's own rows, np.linalg.lstsq, then the projection with the oracle's normal.  Tolerance
    1e-5 relative times the in-plane condition kappa = l_max / l_mid of A (the normals pin scales by the eigen-gap the same way).
    Pinned where the rank is unambiguous: neighbourhoods that are exactly planar IN FP32 (on an axis-aligned box face whose fp32
    centroid equals the face coordinate, so a row and column of A are exactly zero and the rank is 2) and clearly
    three-dimensional ones (l_min / l_max >= 1e-3).  Elsewhere -- faces whose fp32 centroid is off by one rounding, the sphere,
    edges -- the rank decision rests on a pivot of rounding size, the normal component of x is then large and the projection
    with an fp32 normal leaks it: that is the reference algorithm's own sensitivity (the rank decision the QR has to reproduce),
    not a restatement error."""
    xyz, inten, tree, off, idx, nrm = room_rows
    g = D.intensity_gradient(xyz, off, idx, inten, nrm)
    sel = np.random.default_rng(0).choice(len(xyz), 3000, replace=False)
    checked = {"planar": 0, "volume": 0}
    for i in sel:
        l = idx[off[i]:off[i + 1]]
        if len(l) < 3:
            assert np.isnan(g[i, :3]).all()
            continue
        P = xyz[l].astype(np.float64)
        v = inten[l].astype(np.float64)
        Q = P - P.mean(0)
        A, b = Q.T @ Q, Q.T @ (v - v.mean())
        w = np.linalg.eigvalsh(A)
        P32 = xyz[l]
        c32 = np.cumsum(P32, axis=0, dtype=np.float32)[-1] / np.float32(len(l))      # the oracle's sequential fp32 centroid
        planar = bool(((P32 - c32) == 0).all(0).any())
        if not planar and w[0] / w[2] < 1e-3:
            continue
        n = nrm[i, :3].astype(np.float64)
        x = np.linalg.lstsq(A, b, rcond=None)[0]
        ref = x - n * (n @ x)
        assert np.abs(g[i, :3] - ref).max() <= 1e-5 * (w[2] / w[1]) * max(np.linalg.norm(ref), 1e-6), i
        checked["planar" if planar else "volume"] += 1
    assert checked["planar"] > 500 and checked["volume"] > 50, checked


# ---------------------------------------------------------------- RIFT: independent pin
def rift_np(pts, qpts, off, nbr, d2, grad, radius, nd, ng):
    """computeRIFT restated in fp64 with np.add.at; histogram order gradient bin outer, distance bin inner."""
    pts, qpts, grad = (np.asarray(a, np.float64)[:, :3] for a in (pts, qpts, grad))
    out = np.full((qpts.shape[0], nd * ng), np.nan)
    for i in range(qpts.shape[0]):
        l = nbr[off[i]:off[i + 1]]
        if len(l) == 0:
            continue
        h = np.zeros((nd, ng))
        g = grad[l]
        mag = np.linalg.norm(g, axis=1)
        u = pts[l] - qpts[i]
        un = np.linalg.norm(u, axis=1)
        u = np.where(un[:, None] > 0, u / np.where(un > 0, un, 1)[:, None], 0.0)
        with np.errstate(invalid="ignore", divide="ignore"):
            ang = np.arccos((g * u).sum(1) / mag)
        ang = np.where(np.isfinite(ang), ang, 0.0)
        d = nd * np.sqrt(np.asarray(d2[off[i]:off[i + 1]], np.float64)) / (radius + EPS32)
        gb = ng * ang / (np.pi + EPS32)
        for j in range(len(l)):
            for gi in range(int(np.ceil(gb[j] - 1)), int(np.floor(gb[j] + 1)) + 1):
                for di in range(max(int(np.ceil(d[j] - 1)), 0), min(int(np.floor(d[j] + 1)), nd - 1) + 1):
                    np.add.at(h, (di, gi % ng), (1 - abs(d[j] - di)) * (1 - abs(gb[j] - gi)) * mag[j])
        z = np.sqrt((h ** 2).sum())
        if z > 0:
            h /= z
        out[i] = h.T.reshape(-1)          # column-major: index g * nd + d
    return out


def _rift_case(seed=7, n=3000):
    rng = np.random.default_rng(seed)
    xyz = synth.room(n, seed)[:, :3][:600].copy()
    xyz = (xyz * 0.05).astype(np.float32)          # dense patch: tens of neighbours at r = 0.05
    grad = rng.normal(size=(xyz.shape[0], 4)).astype(np.float32)
    grad[:, 3] = 0
    grad[::7, :3] = 0                              # zero gradients: angle NaN -> 0, weight 0
    return xyz, grad


@pytest.mark.parametrize("nd,ng", [(4, 8), (2, 5)])
def test_rift_pinned_to_numpy(nd, ng):
    xyz, grad = _rift_case()
    tree = oracle.KdTree(xyz)
    q = np.vstack([xyz, [[50.0, 50.0, 50.0]]]).astype(np.float32)       # last query: no neighbour
    off, idx, d2 = tree.radius(q, 0.05)
    got = D.rift(xyz, q, off, idx, d2, grad, 0.05, nd, ng)
    want = rift_np(xyz, q, off, idx, d2, grad, 0.05, nd, ng)
    assert got.shape == (q.shape[0], nd * ng)
    assert np.isnan(got[-1]).all() and np.isnan(want[-1]).all()
    assert np.abs(got[:-1] - want[:-1]).max() < 2e-5
    assert np.allclose(np.linalg.norm(got[:-1].astype(np.float64), axis=1), 1.0, atol=1e-5)


def test_rift_wraparound_self_neighbour_zero_and_empty():
    p0 = np.zeros((1, 3), np.float32)
    pts = np.array([[0, 0, 0], [0.02, 0, 0], [0, 0.03, 0]], np.float32)
    # neighbour 1's gradient points back at the query: angle = pi -> gradient bin ~ ng, wrapped onto bin 0
    grad = np.array([[0, 0, 1, 0], [-2, 0, 0, 0], [0, -1, 1e-3, 0]], np.float32)
    off, idx, d2 = oracle.brute_radius(pts, p0, 0.05)
    got = D.rift(pts, p0, off, idx, d2, grad, 0.05, 4, 8)[0]
    want = rift_np(pts, p0, off, idx, d2, grad, 0.05, 4, 8)[0]
    assert np.abs(got - want).max() < 2e-5
    h = want.reshape(8, 4)                          # [gradient bin, distance bin]
    assert h[0].sum() > 0 and h[7].sum() > 0        # the angle-pi neighbours land at both ends of the gradient range
    # self-neighbour (d = 0) with a nonzero gradient: angle = pi/2 -> gradient bin ~4 (3.9999998 or just above 4 in fp32), distance bin 0
    off1, idx1, d21 = oracle.brute_radius(pts[:1], p0, 0.05)
    h1 = D.rift(pts[:1], p0, off1, idx1, d21, grad[:1], 0.05, 4, 8)[0].reshape(8, 4)
    assert int(np.argmax(h1.sum(1))) in (3, 4) and h1[3:5].sum() > 0.999 and set(np.flatnonzero(h1.sum(0))) == {0}
    # all-zero gradients: the histogram stays zero (normalize() of a zero matrix is a no-op), not NaN
    z = D.rift(pts, p0, off, idx, d2, np.zeros_like(grad), 0.05, 4, 8)[0]
    assert (z == 0).all()
    # no neighbour: NaN row
    far = np.array([[9, 9, 9]], np.float32)
    offf, idxf, d2f = oracle.brute_radius(pts, far, 0.05)
    assert np.isnan(D.rift(pts, far, offf, idxf, d2f, grad, 0.05, 4, 8)).all()


def test_rift_histogram_order_gradient_outer_distance_inner():
    """One neighbour at distance bin ~1 whose gradient makes 45 degrees with (p - p0): gradient bin ~2.  PCL's order puts the
    peak at g * nd + d = 2 * 4 + 1 = 9 (distance-outer would be 1 * 8 + 2 = 10)."""
    r = 0.05
    dist = (r + EPS32) / 4
    pts = np.array([[dist, 0, 0]], np.float32)
    grad = np.array([[1, 1, 0, 0]], np.float32)
    q = np.zeros((1, 3), np.float32)
    off, idx, d2 = oracle.brute_radius(pts, q, r)
    h = D.rift(pts, q, off, idx, d2, grad, r, 4, 8)[0]
    assert int(np.argmax(h)) == 9 and h[9] > 0.99


def test_rift_rejects_more_than_32_bins():
    pts = np.zeros((1, 3), np.float32)
    with pytest.raises(ValueError):
        D.rift(pts, pts, np.array([0, 1]), np.array([0], np.int32), np.zeros(1, np.float32), np.zeros((1, 4)), 0.05, 4, 9)


def test_process_rift_oracle_chain_shapes():
    xyz = (synth.room(20000, 21)[:700, :3] * 0.1).astype(np.float32)
    rgb = synth.rgb_for(xyz * 10, 22)
    stages = {}
    desc, kept = D.process_rift(xyz, rgb, stages=stages)
    assert desc.shape[1] == 32 and desc.shape[0] == kept.shape[0] > 0
    assert np.isfinite(desc).all() and np.all(np.diff(kept) > 0)
    assert set(kept.tolist()) <= set(stages["kept_normals"].tolist())
