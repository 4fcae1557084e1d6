"""Batched RIFT probe: computeSimilarity's processRIFT stage on every cluster of a batch, as one pcc_rift_batched call against the
per-cluster loop of process_rift.  Batches: (a) 16 and 64 clusters of 700 points (the largest clusters processRIFT takes), each a patch
of the room cloud moved 2 m apart, and (b) the Euclidean clusters of 100 to 700 points of the tests' synth.scene cloud (0.025 VoxelGrid,
tolerance 0.05, min 100 points).  One JSON line per batch:
  loop_ms / batched_ms   mean host time of the per-cluster process_rift loop and of one process_rift_batched call (host arrays in and
                         out, 10 repetitions after 2 warm-up ones)
  device                 the batched call's kernels from torch.profiler: count, busy_ms = summed kernel time, span_ms = first kernel
                         start to last kernel end
  cpu_oracle_ms          descriptor_oracle.process_rift per cluster
  bit_identical          batched descriptors, offsets and kept rows equal the per-cluster loop's
The card's name and power limit are read in the same run.  usage: python scripts/rift_batch_probe.py [out.jsonl]
(default profiles/r6/rift_batch_probe.jsonl)"""
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch

import descriptor_oracle as D
import oracle
from pointcloudcomparator_b200 import synth
from pointcloudcomparator_b200.search import process_rift, process_rift_batched


def card():
    name, limit = torch.cuda.get_device_name(0), None
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True, timeout=30)
        if out.returncode == 0 and out.stdout.strip():
            name, limit = [v.strip() for v in out.stdout.strip().split(",")[:2]]
    except (OSError, subprocess.SubprocessError):
        pass
    return name, limit


def concat(clusters):
    xyz = np.concatenate([c[0] for c in clusters]).astype(np.float32)
    rgb = np.concatenate([c[1] for c in clusters]).astype(np.uint8)
    off = np.concatenate([[0], np.cumsum([c[0].shape[0] for c in clusters])]).astype(np.int64)
    return xyz, rgb, off


def small_clusters(k):
    base = (synth.room(60000, 41)[:, :3] * 0.12).astype(np.float32)
    rng = np.random.default_rng(5)
    out = []
    for i in range(k):
        centre = base[rng.integers(0, base.shape[0])]
        cl = base[np.flatnonzero(np.linalg.norm(base - centre, axis=1) < 0.12)[:700]] + np.float32([2.0 * i, 0, 0])
        out.append((cl, synth.rgb_for(cl * 8, 43 + i)))
    return concat(out)


def scene_clusters():
    p = synth.scene(800000, 73, extent=14.0, n_objects=120)[0][:, :3].copy()
    v = np.ascontiguousarray(oracle.voxel_grid(p, np.float32(0.025))[:, :3])
    lab, sizes = oracle.KdTree(v).ece(0.05, 100, 10**9)
    rgb = synth.rgb_for(v, 74)
    return concat([(v[lab == c], rgb[lab == c]) for c in np.flatnonzero(sizes <= 700)])


def mean_ms(fn, reps=10):
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / reps * 1e3


def loop(xyz, rgb, off):
    return [process_rift(xyz[off[c]:off[c + 1]], rgb[off[c]:off[c + 1]]) for c in range(off.size - 1)]


def device_time(xyz, rgb, off):
    from torch.profiler import ProfilerActivity, profile
    process_rift_batched(xyz, rgb, off)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        process_rift_batched(xyz, rgb, off)
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            ev = json.load(f)["traceEvents"]
    k = sorted((e for e in ev if e.get("cat") == "kernel"), key=lambda e: e["ts"])
    return dict(kernels=len(k), busy_ms=round(sum(e["dur"] for e in k) / 1e3, 4), span_ms=round((max(e["ts"] + e["dur"] for e in k) - k[0]["ts"]) / 1e3, 4))


def case(label, xyz, rgb, off):
    desc, d_off, kept = process_rift_batched(xyz, rgb, off)
    ref = loop(xyz, rgb, off)
    same = bool(np.array_equal(np.diff(d_off), [r[0].shape[0] for r in ref])
                and np.array_equal(desc.view(np.uint32), np.concatenate([r[0] for r in ref]).view(np.uint32))
                and np.array_equal(kept, np.concatenate([r[1] for r in ref])))
    loop_ms = mean_ms(lambda: loop(xyz, rgb, off))
    batched_ms = mean_ms(lambda: process_rift_batched(xyz, rgb, off))
    dev = device_time(xyz, rgb, off)
    t0 = time.perf_counter()
    for c in range(off.size - 1):
        D.process_rift(xyz[off[c]:off[c + 1]], rgb[off[c]:off[c + 1]])
    cpu = (time.perf_counter() - t0) * 1e3
    name, limit = card()
    sizes = np.diff(off)
    return dict(case=label, clusters=int(off.size - 1), points=int(off[-1]), cluster_min=int(sizes.min()), cluster_max=int(sizes.max()), gpu=name,
                power_limit=limit, descriptors=int(desc.shape[0]), loop_ms=round(loop_ms, 3), batched_ms=round(batched_ms, 3), device=dev,
                cpu_oracle_ms=round(cpu, 1), cpu_oracle_threads=D.num_threads(), bit_identical=same)


def main():
    if not torch.cuda.is_available():
        raise SystemExit("rift_batch_probe.py measures the GPU path: no CUDA device")
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r6", "rift_batch_probe.jsonl")
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    with open(out, "w") as f:
        for label, make in (("16 x 700", lambda: small_clusters(16)), ("64 x 700", lambda: small_clusters(64)), ("scene ECE 100..700", scene_clusters)):
            line = json.dumps(case(label, *make()))
            print(line, flush=True)
            f.write(line + "\n")


if __name__ == "__main__":
    main()
