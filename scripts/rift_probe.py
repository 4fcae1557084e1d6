"""Descriptor-stage probe: pcc_intensity_gradient (r = 0.03) and pcc_rift (r = 0.05, 4 x 8) over the indexed cloud itself, as
processRIFT calls them.  One JSON line per case: a 700-point cluster (the largest processRIFT handles), the C1 room at 100 k points
and a 1 M-point room.  kernel_ms = best of 10 after warm-up of the call's device work (radius count, fill, row sort and the fused
reduction; pcc_set_timing), wall_ms = mean host time per call on device arrays ending in a synchronise.  Algorithmic bytes per query
follow SURVEY.md section 8d's fused-epilogue rule: gradient 16 N/Q + 4 N/Q + 16 + 16 + 16 (points, intensities, query, normal in,
gradient out), RIFT 16 N/Q + 16 N/Q + 16 + 4 nd ng (points, gradients, query, histogram out), as a fraction of the 6533.8 GB/s
measured HBM copy rate.  The CPU oracle (descriptor_oracle/) is timed on the same rows.  usage: python scripts/rift_probe.py"""
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import descriptor_oracle as D
import oracle
from pointcloudcomparator_b200 import synth
from pointcloudcomparator_b200.search import GridSearch, rgb_to_intensity

PEAK = 6533.8e9
ND, NG = 4, 8


def card():
    name, limit = torch.cuda.get_device_name(0), None
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True, timeout=30)
        if out.returncode == 0 and out.stdout.strip():
            name, limit = [v.strip() for v in out.stdout.strip().split(",")[:2]]
    except (OSError, subprocess.SubprocessError):
        pass
    return name, limit


def timed(fn, s, reps=10):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    s.setTiming(True)
    best = 1e30
    for _ in range(reps):
        fn()
        best = min(best, s.lastKernelMs())
    s.setTiming(False)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        fn()
    torch.cuda.synchronize()
    return best, (time.perf_counter() - t0) / reps * 1e3


def case(label, xyz, rgb):
    n = xyz.shape[0]
    inten = rgb_to_intensity(rgb)
    tree = oracle.KdTree(xyz)
    off_g, idx_g, _ = tree.radius(xyz, 0.03)
    normals = oracle.normals_from_lists(xyz, xyz, off_g, idx_g)
    t0 = time.perf_counter()
    grad_o = D.intensity_gradient(xyz, off_g, idx_g, inten, normals)
    cpu_grad_ms = (time.perf_counter() - t0) * 1e3
    off_r, idx_r, d2_r = tree.radius(xyz, 0.05)
    t0 = time.perf_counter()
    rift_o = D.rift(xyz, xyz, off_r, idx_r, d2_r, grad_o, 0.05, ND, NG)
    cpu_rift_ms = (time.perf_counter() - t0) * 1e3

    dx = torch.as_tensor(xyz, device="cuda")
    di, dn, dg = (torch.as_tensor(a, device="cuda") for a in (inten, normals, grad_o))
    s = GridSearch(0).setInputCloud(dx, cell_hint=0.05)
    kg, wg = timed(lambda: s.intensityGradient(None, 0.03, di, dn), s)
    kr, wr = timed(lambda: s.rift(None, 0.05, dg, ND, NG), s)
    g = s.intensityGradient(None, 0.03, di, dn).cpu().numpy()
    h = s.rift(None, 0.05, dg, ND, NG).cpu().numpy()
    same_nan = np.array_equal(np.isnan(g), np.isnan(grad_o))
    grad_bitexact = bool(same_nan and np.array_equal(np.where(np.isnan(g), 0, g).view(np.uint32), np.where(np.isnan(grad_o), 0, grad_o).view(np.uint32)))
    clean = np.isfinite(rift_o).all(1)               # unit-norm rows (a NaN gradient nearby leaves a row unnormalised and partly NaN)
    rift_err = float(np.abs(h[clean] - rift_o[clean]).max()) if clean.any() else 0.0
    same_rift_nan = bool(np.array_equal(np.isnan(h), np.isnan(rift_o)))
    mg, mr = float(np.diff(off_g).mean()), float(np.diff(off_r).mean())
    bg = 16 * mg + 4 * mg + 16 + 16 + 16          # N/Q neighbours per query: every neighbour read once per query (no reuse credit)
    br = 16 * mr + 16 * mr + 16 + 4 * ND * NG
    name, limit = card()
    return dict(case=label, n=n, gpu=name, power_limit=limit,
                gradient=dict(radius=0.03, mean_row=round(mg, 2), kernel_ms=round(kg, 4), wall_ms=round(wg, 4), bytes_per_query=round(bg, 1),
                              frac_hbm=round(n * bg / (kg * 1e-3) / PEAK, 5), cpu_oracle_ms=round(cpu_grad_ms, 2), bit_identical=grad_bitexact),
                rift=dict(radius=0.05, bins=[ND, NG], mean_row=round(mr, 2), kernel_ms=round(kr, 4), wall_ms=round(wr, 4), bytes_per_query=round(br, 1),
                          frac_hbm=round(n * br / (kr * 1e-3) / PEAK, 5), cpu_oracle_ms=round(cpu_rift_ms, 2), max_bin_err_unit_rows=rift_err,
                          unit_rows=int(clean.sum()), same_nan_pattern=same_rift_nan),
                cpu_oracle_threads=D.num_threads())


def main():
    if not torch.cuda.is_available():
        raise SystemExit("rift_probe.py measures the GPU path: no CUDA device")
    base = (synth.room(60000, 41)[:, :3] * 0.12).astype(np.float32)
    cl = base[np.flatnonzero(np.linalg.norm(base - base[0], axis=1) < 0.12)[:700]]
    cases = [("cluster-700", cl, synth.rgb_for(cl * 8, 43))]
    for label, n, seed in (("C1 room-100k", 100_000, 1001), ("room-1M", 1_000_000, 2001)):
        xyz = synth.room(n, seed)[:, :3].copy()
        cases.append((label, xyz, synth.rgb_for(xyz, seed + 1)))
    for label, xyz, rgb in cases:
        print(json.dumps(case(label, xyz, rgb)), flush=True)


if __name__ == "__main__":
    main()
