"""Batched colour-segmentation probe: computeSimilarity's color_growing_segmentation on every cluster of a batch, as one
region_growing_rgb_batched call against the per-cluster loop (GridSearch + nearestKSearch(None, 100) + region_growing_rgb).  Batches:
(a) the region-growing clusters (>= 50 points) of the tests' synth.scene cloud after a 0.025 VoxelGrid, synth.rgb_for colours;
(b) those clusters plus the same clusters of a noisy second copy in one call (both clouds of every matched pair: the clusters overlap in
space, so half of every visited point belongs to the other cloud); (c) 64 clusters of 2000 points.  One JSON line per batch:
  loop_ms / batched_ms   mean host time of the per-cluster loop and of one region_growing_rgb_batched call (host arrays in and out,
                         10 repetitions after 2 warm-up ones)
  knn_batched_ms         mean host time of one knn_batched call (the table only, host arrays out)
  host_grow_ms           the per-cluster host grows over the batched table (region_growing_rgb, one cluster after another), and
  host_grow_share        that time over batched_ms
  device                 the batched call's kernels from torch.profiler, in a run of its own: count, busy_ms = summed kernel time,
                         span_ms = first kernel start to last kernel end
  cpu_oracle_ms          oracle.KdTree(cluster).knn(cluster, 100) per cluster plus the same host grow
  identical              batched labels and counts equal the per-cluster loop's (asserted)
The card's name and power limit are read in the same run.  usage: python scripts/rgb_batch_probe.py [out.jsonl]
(default profiles/r7/rgb_batch_probe.jsonl)"""
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

import oracle
from pointcloudcomparator_b200 import synth
from pointcloudcomparator_b200.search import GridSearch, knn_batched, region_growing_rgb, region_growing_rgb_batched

K = 100


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


def pack(rgb):
    c = np.asarray(rgb).reshape(-1, 3).astype(np.uint32)
    return (c[:, 0] << 16) | (c[:, 1] << 8) | c[:, 2]


def scene_clusters():
    """RegionGrowing's clusters (k = 100 table, k = 50 normals, 3 degrees, curvature 1, >= 50 points) of the voxelised scene"""
    p = synth.scene(400000, 73, extent=10.0, n_objects=60)[0][:, :3].copy()
    v = np.ascontiguousarray(oracle.voxel_grid(p, np.float32(0.025))[:, :3])
    tree = oracle.KdTree(v)
    nb, _, _ = tree.knn(v, 100)
    lab, nc = oracle.region_growing(nb, oracle.normals_knn(v, 50, tree=tree), 3.0 / 180.0 * np.pi, 1.0, 50, 1000000)
    return v, [np.flatnonzero(lab == c) for c in range(nc)]


def batch_scene():
    v, members = scene_clusters()
    rgb = synth.rgb_for(v, 74)
    return concat([(v[m], rgb[m]) for m in members])


def batch_pairs():
    v, members = scene_clusters()
    w = synth.noisy_copy(v, 75, 0.002)[:, :3]
    rgb, rgb2 = synth.rgb_for(v, 74), synth.rgb_for(v, 76)
    return concat([(v[m], rgb[m]) for m in members] + [(w[m], rgb2[m]) for m in members])


def batch_tiles(k=64, n=2000):
    base = (synth.room(60000, 41)[:, :3] * 0.12).astype(np.float32)
    rng = np.random.default_rng(5)
    out = []
    for i in range(k):
        centre = base[rng.integers(0, base.shape[0])]
        cl = base[np.flatnonzero(np.linalg.norm(base - centre, axis=1) < 0.3)[:n]] + np.float32([2.0 * i, 0, 0])
        out.append((cl, synth.rgb_for(cl * 8, 43 + i)))
    return concat(out)


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
    out = []
    for c in range(off.size - 1):
        x = xyz[off[c]:off[c + 1]]
        nb, nd, _ = GridSearch().setInputCloud(x, k_hint=K).nearestKSearch(None, K)
        out.append(region_growing_rgb(nb, nd, pack(rgb[off[c]:off[c + 1]])))
    return out


def grows(nb, nd, rgb, off):
    return [region_growing_rgb(nb[off[c]:off[c + 1]], nd[off[c]:off[c + 1]], pack(rgb[off[c]:off[c + 1]])) for c in range(off.size - 1)]


def device_time(xyz, rgb, off):
    from torch.profiler import ProfilerActivity, profile
    region_growing_rgb_batched(xyz, rgb, off)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        region_growing_rgb_batched(xyz, rgb, off)
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            ev = json.load(f)["traceEvents"]
    k = sorted((e for e in ev if e.get("cat") == "kernel"), key=lambda e: e["ts"])
    return dict(kernels=len(k), busy_ms=round(sum(e["dur"] for e in k) / 1e3, 4), span_ms=round((max(e["ts"] + e["dur"] for e in k) - k[0]["ts"]) / 1e3, 4))


def case(label, xyz, rgb, off):
    labels, counts = region_growing_rgb_batched(xyz, rgb, off)
    ref = loop(xyz, rgb, off)
    same = bool(np.array_equal(counts, [r[1] for r in ref]) and np.array_equal(labels, np.concatenate([r[0] for r in ref])))
    assert same, f"{label}: batched labels differ from the per-cluster loop"
    loop_ms = mean_ms(lambda: loop(xyz, rgb, off))
    batched_ms = mean_ms(lambda: region_growing_rgb_batched(xyz, rgb, off))
    knn_ms = mean_ms(lambda: knn_batched(xyz, off, K))
    nb, nd, _ = knn_batched(xyz, off, K)
    grow_ms = mean_ms(lambda: grows(nb, nd, rgb, off))
    dev = device_time(xyz, rgb, off)
    t0 = time.perf_counter()
    for c in range(off.size - 1):
        x = np.ascontiguousarray(xyz[off[c]:off[c + 1]])
        oi, od, _ = oracle.KdTree(x).knn(x, K)
        region_growing_rgb(oi, od, pack(rgb[off[c]:off[c + 1]]))
    cpu = (time.perf_counter() - t0) * 1e3
    name, limit = card()
    sizes = np.diff(off)
    return dict(case=label, clusters=int(off.size - 1), points=int(off[-1]), cluster_min=int(sizes.min()), cluster_max=int(sizes.max()), gpu=name,
                power_limit=limit, colour_clusters=int(counts.sum()), loop_ms=round(loop_ms, 3), batched_ms=round(batched_ms, 3),
                knn_batched_ms=round(knn_ms, 3), host_grow_ms=round(grow_ms, 3), host_grow_share=round(grow_ms / batched_ms, 3), device=dev,
                cpu_oracle_ms=round(cpu, 1), cpu_oracle_threads=oracle.num_threads(), identical=same)


def main():
    if not torch.cuda.is_available():
        raise SystemExit("rgb_batch_probe.py measures the GPU path: no CUDA device")
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r7", "rgb_batch_probe.jsonl")
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    with open(out, "w") as f:
        for label, make in (("(a) scene RG clusters", batch_scene), ("(b) scene RG clusters + noisy copy", batch_pairs), ("(c) 64 x 2000", batch_tiles)):
            line = json.dumps(case(label, *make()))
            print(line, flush=True)
            f.write(line + "\n")


if __name__ == "__main__":
    main()
