"""CPU pins of the SIFT-keypoint oracle (descriptor_oracle/: orc_sift_*) against code that shares nothing with it: hand-computed
field values, numpy's fp64 exp, numpy restatements of computeScaleSpace over scipy cKDTree rows and of findScaleSpaceExtrema, and
known answers (a constant cloud, a plane with a bright and a dark Gaussian blob, an octave loop that runs out of points)."""
import numpy as np
import pytest
from scipy.spatial import cKDTree

import descriptor_oracle as D
import oracle
from pointcloudcomparator_b200 import synth


def test_field_selector_hand_computed():
    v = D.sift_field_values(np.array([[255, 255, 255], [1, 2, 3], [1, 1, 1], [0, 0, 0]], np.uint8))
    assert v[0] == np.float32(255.0)
    assert v[1] == np.float32(1.815)                     # (299 + 1174 + 342) / 1000
    assert v[2] == np.float32(1.0) and v[3] == 0.0       # 1000 / 1000 exactly


def test_sift_expf_within_one_ulp_of_fp64_exp():
    x = np.concatenate([np.linspace(-4.6, 0.0, 1_000_001, dtype=np.float64).astype(np.float32),
                        np.random.default_rng(3).uniform(-4.6, 0.0, 200_000).astype(np.float32),
                        np.array([-4.6, -4.5, -0.0, 0.0, np.nextafter(np.float32(0), np.float32(-1))], np.float32)])
    got = D.sift_expf(x)
    want = np.exp(x.astype(np.float64)).astype(np.float32)
    ulps = np.abs(got.view(np.int32).astype(np.int64) - want.view(np.int32).astype(np.int64))
    equal = float((ulps == 0).mean())
    print(f"sift_expf: {x.size} arguments on [-4.6, 0], {equal * 100:.5f} % bit-equal to fp64 exp rounded to fp32, max {ulps.max()} ulp")
    assert ulps.max() <= 1
    assert equal > 0.9999
    assert D.sift_expf(np.array([0.0], np.float32))[0] == 1.0


def _octave(n=20000, seed=11, leaf=0.01):
    xyz = synth.room(n, seed)[:, :3]
    rgb = synth.rgb_for(xyz, seed + 1)
    cloud = oracle.voxel_grid(D.pack_rgb(xyz, rgb), np.float32(leaf), rgb_offset_floats=3)
    return cloud, D.sift_scales(leaf, 5)


def test_dog_matches_numpy_fp64_restatement_on_room_octave():
    cloud, scales = _octave()
    values = D.sift_field_values(D.unpack_rgb(cloud))
    r = float(np.float32(3.0) * scales[-1])
    off, idx, d2 = oracle.KdTree(cloud).radius(cloud, r)
    got = D.sift_dog(values, off, idx, d2, scales)
    # numpy: cKDTree rows, fp32 squared distances (PCL's) for the radius and cutoff tests, fp64 weights and sums
    p = cloud[:, :3]
    r2 = np.float32(r * r)
    sig2 = scales.astype(np.float64) ** 2
    cut = np.float32(9) * (scales * scales)
    want = np.empty_like(got, dtype=np.float64)
    for i, row in enumerate(cKDTree(p.astype(np.float64)).query_ball_point(p.astype(np.float64), r * 1.001)):
        row = np.asarray(row)
        dd = p[row] - p[i]
        dd2 = (dd[:, 0] * dd[:, 0] + dd[:, 1] * dd[:, 1]) + dd[:, 2] * dd[:, 2]
        keep = dd2 < r2
        dd2, vals = dd2[keep].astype(np.float64), values[row[keep]].astype(np.float64)
        resp = []
        for s in range(scales.size):
            m = dd2 <= cut[s]
            w = np.exp(-0.5 * dd2[m] / sig2[s])
            resp.append((vals[m] * w).sum() / w.sum())
        want[i] = np.diff(resp)
    err = np.abs(got - want).max()
    print(f"DoG over {cloud.shape[0]} octave points: max |oracle - numpy fp64| = {err:.3g} (values up to {values.max():.1f})")
    assert err <= 2e-5 * float(values.max())
    assert np.abs(want).max() > 1.0                      # the room's colour edges give a real scale-space signal


def _extrema_numpy(dog, nn, c):
    n, nc = dog.shape
    out = []
    for i in range(n):
        rows = nn[i][nn[i] >= 0]
        mn, mx = dog[rows].min(0), dog[rows].max(0)
        for s in range(1, nc - 1):
            v = dog[i, s]
            if abs(v) >= c and ((v == mn[s] and v < mn[s - 1] and v < mn[s + 1]) or (v == mx[s] and v > mx[s - 1] and v > mx[s + 1])):
                out.append((i, s))
    return out


def test_extrema_rule_matches_numpy_restatement():
    rng = np.random.default_rng(21)
    p = rng.uniform(0, 1, (6000, 3))
    _, nn = cKDTree(p).query(p, 25)                       # continuous random points: no distance ties
    dog = rng.normal(0, 0.01, (p.shape[0], 7)).astype(np.float32)
    dog[::7] *= np.float32(0.01)                          # a share of values below min_contrast
    nn = nn.astype(np.int32)
    nn[5, 20:] = -1                                       # absent entries are skipped
    rows, cols = D.sift_extrema(dog, nn, 0.001)
    want = _extrema_numpy(dog, nn, np.float32(0.001))
    assert list(zip(rows.tolist(), cols.tolist())) == want
    assert len(want) > 50 and set(cols.tolist()) <= set(range(1, 6))
    assert (np.abs(dog[rows, cols]) >= np.float32(0.001)).all()


def test_constant_cloud_has_zero_dog_and_no_keypoints():
    xyz = synth.room(30000, 13)[:, :3]
    rgb = np.ones((xyz.shape[0], 3), np.uint8)            # value 1.0: fl(1 w) = w, so every response is exactly den / den = 1
    st = {}
    kp = D.sift_keypoints(xyz, rgb, stages=st)
    assert kp.shape == (0, 4) and len(st["octaves"]) == 5
    for o in st["octaves"]:
        assert (o["dog"] == 0).all()


def blob_plane(sb=0.02, h=0.004, L=0.4, seed=5):
    """A dense jittered grid on z = 0.5 whose grey value carries a bright (+100) and a dark (-100) Gaussian blob of sigma sb."""
    rng = np.random.default_rng(seed)
    g = np.arange(0, L, h)
    X, Y = np.meshgrid(g, g, indexing="ij")
    xy = np.stack([X.ravel(), Y.ravel()], 1) + rng.uniform(-0.1 * h, 0.1 * h, (X.size, 2))
    c1, c2 = np.array([0.12, 0.2]), np.array([0.28, 0.2])
    v = 128 + 100 * np.exp(-((xy - c1) ** 2).sum(1) / (2 * sb * sb)) - 100 * np.exp(-((xy - c2) ** 2).sum(1) / (2 * sb * sb))
    c = np.clip(np.rint(v), 0, 255).astype(np.uint8)
    return np.column_stack([xy, np.full(len(xy), 0.5)]).astype(np.float32), np.stack([c, c, c], 1), c1, c2


@pytest.mark.parametrize("sb", [0.02, 0.04])
def test_blob_plane_extrema_at_blob_centres_and_scale(sb):
    """dog[:, s-1] = response_s - response_{s-1} (coarser minus finer smoothing), so a bright blob's centre is a DoG MINIMUM and a
    dark blob's a MAXIMUM; both are found at the octave whose base scale equals the blob's sigma, at a scale within one step."""
    xyz, rgb, c1, c2 = blob_plane(sb)
    st = {}
    kp = D.sift_keypoints(xyz, rgb, stages=st)
    step = 2.0 ** (1.0 / 5)
    for centre, sign in ((c1, -1), (c2, +1)):
        hits = []
        for o in st["octaves"]:
            tree = oracle.KdTree(o["cloud"])
            nn, _, _ = tree.knn(o["cloud"], 25)
            for r, c in zip(o["rows"], o["cols"]):
                p, scale = o["cloud"][r, :2], float(o["scales"][c])
                if np.linalg.norm(p - centre) <= float(o["scales"][1]) and abs(np.log(scale / sb)) <= np.log(step) * 1.01:
                    v = o["dog"][r, c]
                    branch = -1 if v == o["dog"][nn[r], c].min() else (+1 if v == o["dog"][nn[r], c].max() else 0)
                    hits.append((branch, np.sign(v), scale))
        assert hits, (centre, sb)
        assert all(b == sign and s == sign for b, s, _ in hits), hits
    # the octave / column -> scale bookkeeping: every keypoint's scale is an entry of its octave's table, octaves in order
    m = 0
    for o in st["octaves"]:
        k = o["keypoints"]
        assert np.array_equal(k, kp[m : m + len(k)]) and np.isin(k[:, 3], o["scales"][1:-2]).all()
        m += len(k)
    assert m == len(kp)


def test_octave_loop_stops_below_25_points():
    rng = np.random.default_rng(17)
    g = np.arange(12) * 0.0113 + 0.00137
    X, Y = np.meshgrid(g, g, indexing="ij")
    xyz = np.column_stack([X.ravel(), Y.ravel(), np.full(X.size, 0.00371)]).astype(np.float32)
    rgb = rng.integers(0, 256, (xyz.shape[0], 3)).astype(np.uint8)
    # numpy restatement of the counts: voxel ids floor(x * (1 / leaf)) of the previous octave's centroids
    pts, leaf, want = xyz.astype(np.float64), np.float32(0.005), []
    while len(want) < 5:
        inv = np.float32(1) / leaf
        ids = np.floor(pts.astype(np.float32) * inv).astype(np.int64)
        _, inverse = np.unique(ids, axis=0, return_inverse=True)
        inverse = inverse.reshape(-1)
        pts = np.stack([np.bincount(inverse, pts[:, d]) / np.bincount(inverse) for d in range(3)], 1)
        if len(pts) < 25:
            break
        want.append(len(pts))
        leaf = np.float32(leaf * 2)
    st = {}
    D.sift_keypoints(xyz, rgb, stages=st)
    got = [o["cloud"].shape[0] for o in st["octaves"]]
    print(f"octave sizes {got}, numpy prediction {want}")
    assert got == want and len(got) < 5
