"""SIFT keypoint probe: pcc_sift_keypoints as processSift calls it (min_scale 0.005, 5 octaves, 5 scales per octave, min_contrast
0.001) on a 700-point and a 5000-point cluster (processRIFTwithSIFT runs it on clusters above 700 points), the C1 room at 100 k points
and a 1 M-point room.  One JSON line per case.  Per octave: point count, mean radius row at 3 * scales[-1], and the device time of
pcc_sift_dog (radius count, fill, row sort, DoG kernel) and of pcc_sift_extrema (k = 25 kNN, extremum kernel, scan, compaction),
best of 10 after warm-up (pcc_set_timing), on device arrays.  Per call: wall_ms = mean host time of the whole sift_keypoints call
(host arrays in and out, 10 calls after 2 warm-up calls), the CPU oracle's time for the same keypoints (descriptor_oracle/), and
whether the two keypoint arrays are bit-identical.  usage: python scripts/sift_probe.py"""
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import descriptor_oracle as D
from pointcloudcomparator_b200 import synth
from pointcloudcomparator_b200.search import GridSearch, sift_field_values, sift_keypoints


def card():
    name, limit = torch.cuda.get_device_name(0), None
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True, timeout=30)
        if out.returncode == 0 and out.stdout.strip():
            name, limit = [v.strip() for v in out.stdout.strip().split(",")[:2]]
    except (OSError, subprocess.SubprocessError):
        pass
    return name, limit


def best_ms(fn, s, reps=10):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    s.setTiming(True)
    best = 1e30
    for _ in range(reps):
        fn()
        best = min(best, s.lastKernelMs())
    s.setTiming(False)
    return best


def case(label, xyz, rgb):
    st = {}
    kp = sift_keypoints(xyz, rgb, stages=st)
    sift_keypoints(xyz, rgb)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(10):
        sift_keypoints(xyz, rgb)
    wall = (time.perf_counter() - t0) / 10 * 1e3
    t0 = time.perf_counter()
    want = D.sift_keypoints(xyz, rgb)
    cpu = (time.perf_counter() - t0) * 1e3
    octaves = []
    for o in st["octaves"]:
        cloud, scales = o["cloud"], o["scales"]
        r = float(np.float32(3) * scales[-1])
        dx = torch.as_tensor(np.ascontiguousarray(cloud[:, :3]), device="cuda")
        s = GridSearch(0).setInputCloud(dx, cell_hint=r)
        vals = torch.as_tensor(sift_field_values(D.unpack_rgb(cloud)), device="cuda")
        dog = s.siftDoG(vals, scales)
        off, _, _ = s.radiusSearch(None, r)
        mean_row = float((off[1:] - off[:-1]).double().mean())
        kd = best_ms(lambda: s.siftDoG(vals, scales), s)
        ke = best_ms(lambda: s.siftExtrema(dog, 0.001), s)
        octaves.append(dict(points=int(cloud.shape[0]), radius=round(r, 5), mean_row=round(mean_row, 2), dog_ms=round(kd, 4), extrema_ms=round(ke, 4),
                            keypoints=int(o["rows"].shape[0])))
    name, limit = card()
    same = bool(kp.shape == want.shape and np.array_equal(kp.view(np.uint32), want.view(np.uint32)))
    return dict(case=label, n=int(xyz.shape[0]), gpu=name, power_limit=limit, keypoints=int(kp.shape[0]), octaves=octaves,
                wall_ms=round(wall, 3), cpu_oracle_ms=round(cpu, 1), cpu_oracle_threads=D.num_threads(), bit_identical=same)


def main():
    if not torch.cuda.is_available():
        raise SystemExit("sift_probe.py measures the GPU path: no CUDA device")
    base = (synth.room(60000, 41)[:, :3] * 0.12).astype(np.float32)
    cases = []
    for n, rad in ((700, 0.12), (5000, 0.4)):
        cl = base[np.flatnonzero(np.linalg.norm(base - base[0], axis=1) < rad)[:n]]
        cases.append((f"cluster-{n}", cl, synth.rgb_for(cl * 8, 43)))
    for label, n, seed in (("C1 room-100k", 100_000, 1001), ("room-1M", 1_000_000, 2001)):
        xyz = synth.room(n, seed)[:, :3].copy()
        cases.append((label, xyz, synth.rgb_for(xyz, seed + 1)))
    for label, xyz, rgb in cases:
        print(json.dumps(case(label, xyz, rgb)), flush=True)


if __name__ == "__main__":
    main()
