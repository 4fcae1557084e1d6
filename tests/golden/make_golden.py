"""Generates tests/golden/flann_single_index.npz and opencv_flann_pins.npz with OpenCV's bundled FLANN (KDTreeSingleIndex,
algorithm=4, leaf_max_size=15, checks=-1, eps=0, sorted) -- the same index family PCL 1.7's
KdTreeFLANN drives (SURVEY.md section 8c).  PCL/FLANN themselves are not installable here, so these
are stand-in golden vectors, NOT outputs of the reference binary.  Run from the repo root:

    python tests/golden/make_golden.py
"""
import hashlib
import os
import sys

import cv2
import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "..", ".."))
from pointcloudcomparator_b200 import synth  # noqa: E402

out = {}
ref = synth.room(4096, 1001)
qry = np.concatenate([synth.sweep_queries(ref, 192, seed=5002, sigma=0.01), ref[:64]]).astype(np.float32)
fl = cv2.flann_Index(ref, dict(algorithm=4, leaf_max_size=15))
out["ref"], out["qry"] = ref, qry
for k in (1, 16, 50):
    idx, d2 = fl.knnSearch(qry, k, params=dict(checks=-1, eps=0.0, sorted=True))
    out[f"knn{k}_idx"], out[f"knn{k}_d2"] = idx.astype(np.int32), d2.astype(np.float32)
radius = 0.25
r2 = np.float32(radius * radius)
off, ridx, rd2 = [0], [], []
for j in range(qry.shape[0]):
    n, ii, dd = fl.radiusSearch(qry[j : j + 1], float(r2), 4096, params=dict(checks=-1, eps=0.0, sorted=True))
    off.append(off[-1] + n), ridx.append(ii[0, :n].astype(np.int32)), rd2.append(dd[0, :n].astype(np.float32))
out["radius"] = np.float64(radius)
out["rad_off"], out["rad_idx"], out["rad_d2"] = np.asarray(off, np.int64), np.concatenate(ridx), np.concatenate(rd2)
# uniform volume cloud too (different tree shape)
ref2 = synth.uniform(4096, 5001, extent=1.0)
q2 = synth.sweep_queries(ref2, 128, seed=77, sigma=0.02)
fl2 = cv2.flann_Index(ref2, dict(algorithm=4, leaf_max_size=15))
i2, d2 = fl2.knnSearch(q2, 16, params=dict(checks=-1, eps=0.0, sorted=True))
out["uref"], out["uqry"], out["uknn16_idx"], out["uknn16_d2"] = ref2, q2, i2.astype(np.int32), d2.astype(np.float32)
np.savez_compressed(os.path.join(os.path.dirname(__file__), "flann_single_index.npz"), **out)
print({k: v.shape for k, v in out.items()})

# FLANN's answers for the FLANN pins in tests/test_oracle_pinning.py.  Their inputs are too large to store, so the tests rebuild
# them from the same seeds; the SHA-256 of the inputs is kept so that a changed generator fails instead of comparing other data.
pins = {}


def record(name, ref, qry, k):
    ref, qry = np.ascontiguousarray(ref, np.float32), np.ascontiguousarray(qry, np.float32)
    idx, d2 = cv2.flann_Index(ref, dict(algorithm=4, leaf_max_size=15)).knnSearch(qry, k, params=dict(checks=-1, eps=0.0, sorted=True))
    pins[f"{name}_idx"], pins[f"{name}_d2"] = idx.astype(np.int32), d2.astype(np.float32)
    pins[f"{name}_inputs_sha256"] = np.str_(hashlib.sha256(ref.tobytes() + qry.tobytes()).hexdigest())


ref = synth.room(60000, 1001)
record("room60k_knn16", ref, synth.sweep_queries(ref, 3000, seed=9)[::3], 16)          # every third query keeps the file small
g = np.arange(12, dtype=np.float32)
lattice = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3)
record("lattice_knn8", lattice, lattice[::7], 8)
rng = np.random.default_rng(3)
ref = rng.random((700, 32), dtype=np.float32) * 0.3
record("desc32_nn", ref, ref[rng.integers(0, 700, 400)] + rng.normal(0, 0.02, (400, 32)), 1)
rng = np.random.default_rng(8)
ref = rng.random((900, 32), dtype=np.float32) * 0.3
qry = ref[rng.integers(0, 900, 500)] + rng.normal(0, 0.02, (500, 32))
record("desc3_nn", ref[:, :3], qry[:, :3], 1)
np.savez_compressed(os.path.join(os.path.dirname(__file__), "opencv_flann_pins.npz"), **pins)
print({k: v.shape for k, v in pins.items()})
