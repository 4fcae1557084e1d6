#!/usr/bin/env python
"""bench.py -- the driver's measurement contract for the batched kNN hot path.

Metric (BASELINE.json): kNN queries/s, k = 16, 10 M-point clouds, at 1/2/4/8 B200.

  python bench.py --gpus N --steps K --warmup W          (N > 1: launched under torch.distributed.run)
  python bench.py --impl reference ...                   (the CPU path on the box's host cores, rank 0 only)
  python bench.py ... --dump-outputs DIR                 (also writes a fixed sample of the last timed step's result rows to DIR/*.npy)

One "step" = one pass of the hot path over one batch: pcc_knn (query cell keys -> radix sort -> fused kNN kernel)
for ONE set of Q = 10 M query points against the 10 M-point indexed reference cloud, everything resident in HBM.
`value` is device-timed (CUDA events on the launch stream, max over ranks).  `e2e` is the same call through the
C ABI with pinned HOST buffers: the host->device copy of the step's queries and the device->host read of the
(idx, d2) table are inside the timed region.  Multi-GPU (strong scaling): reference grid built on rank 0 and broadcast through the
C ABI (pcc_broadcast_index), the common query set is split by grid-cell range and every rank answers Q/N of it; the gather of the result
table (pcc_gather) and the round-1 weak-scaling number are reported as separate fields.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "knn_queries_per_s_k16_10M"
UNIT = "queries/s"
K = 16
DUMP_BYTES = 64_000_000
DUMP_SEED = 20240601


def workload_config(args, world):
    return {
        "workload": f"raw kNN sweep point (BASELINE configs[4], the split of configs[3]): k={args.k}, ONE set of Q={args.nq} queries vs N={args.n} reference points, "
                    f"{args.cloud} cloud (S5/S4 generators, seeds 4001/5002), queries = reference points + N(0, 1 cm), shuffled",
        "n_ref": args.n, "n_query_total": args.nq, "n_query_per_gpu": args.nq // max(world, 1), "k": args.k, "cloud": args.cloud,
        "parallelism": f"query-sharded x{world} by grid-cell range (blocks of {args.shard_block} queries of the cell order dealt round-robin; strong scaling: the same {args.nq} queries at every GPU count), reference grid replicated "
                       "(built on rank 0, pcc_broadcast_index = ncclBroadcast); no collective inside the timed region -- the gather of the result table "
                       "(pcc_gather) is timed separately as gather_ms / value_with_gather",
        "l2": "inputs larger than L2 (160 MB grid + 225 MB cell table + 160 MB queries + 1.28 GB output per step, split over the ranks, vs 126 MB L2); no explicit flush",
        "timed_region": "pcc_knn on this rank's device-resident shard: cell keys + radix sort of the queries + kNN kernels; index build and broadcast excluded (build_ms, broadcast_ms)",
    }


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled every 50 ms from before the warm-up until after the kernel-timing re-run."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu: int):
        self.gpu, self.proc, self.lines = gpu, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=lambda: self.lines.extend(self.proc.stdout), daemon=True).start()
        except Exception:
            self.proc = None

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])), mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm)}


def make_clouds(args, rank):
    from pointcloudcomparator_b200 import synth
    if args.cloud == "surface":
        ref = synth.room(args.n, 4001, size=(10.0, 10.0, 3.0), stride4=True)
    else:
        ref = synth.uniform(args.n, 5001, 10.0, stride4=True)
    qry = synth.sweep_queries(ref, args.nq, seed=5002 + rank, sigma=0.01, stride4=True)
    return ref, qry


def dump_rows(n: int, k: int):
    """Positions of the result rows --dump-outputs writes: all n when they fit in DUMP_BYTES, else a fixed seeded sample
    (ascending).  A row costs k float64 indices, k float32 squared distances and its float64 query row number."""
    fit = max(1, (DUMP_BYTES - 4096) // (12 * k + 8))
    if n <= fit:
        return np.arange(n)
    return np.sort(np.random.default_rng(DUMP_SEED).choice(n, fit, replace=False))


def dump_outputs(path: str, query_rows, idx, d2):
    """Result rows of the timed path as <path>/<name>.npy; indices as float64, which holds every int32 exactly."""
    os.makedirs(path, exist_ok=True)
    for name, a in (("query_rows", np.asarray(query_rows, np.float64)), ("knn_indices", np.asarray(idx, np.float64)),
                    ("knn_sqr_distances", np.asarray(d2, np.float32))):
        np.save(os.path.join(path, f"{name}.npy"), a)


def host_threads() -> int:
    """Threads the CPU arm uses: every core this process may run on.  Set explicitly on each call -- torch.distributed.run
    exports OMP_NUM_THREADS=1, which made the round-1 reference arm single-threaded at N >= 2."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return max(1, os.cpu_count() or 1)


def cpu_baseline(ref, qry, k, budget_s=12.0, threads=0, tree=None):
    """The oracle's restated FLANN KDTreeSingleIndex (OpenMP over queries) on a bounded sample of the same workload."""
    import oracle
    t0 = time.perf_counter()
    tree = tree or oracle.KdTree(ref)
    build_s = time.perf_counter() - t0
    threads = threads if threads > 0 else host_threads()
    cores = threads
    chunk, done, spent = 200_000, 0, 0.0
    while spent < budget_s and done < qry.shape[0]:
        q = qry[done: done + chunk]
        t0 = time.perf_counter()
        tree.knn(q, k, threads=threads)
        spent += time.perf_counter() - t0
        done += q.shape[0]
    return {"value": done / spent, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"first {done} of the {qry.shape[0]} queries against the full {ref.shape[0]}-point kd-tree (leaf 15, exact), "
                      f"{cores} OpenMP threads over queries, {spent:.1f} s; tree build {build_s:.1f} s not included"}, spent, done


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    ref, qry = make_clouds(args, 0)
    import oracle
    tree = oracle.KdTree(ref)
    cores = host_threads()
    sample = min(args.nq, 500_000)
    total = args.warmup + args.steps
    times = []
    for s in range(total):
        start = (s * sample) % max(args.nq - sample, 1)
        q = qry[start:][:sample]
        t0 = time.perf_counter()
        idx, d2, _ = tree.knn(q, args.k, threads=cores)
        times.append(time.perf_counter() - t0)
    if args.dump_outputs:
        pick = dump_rows(len(q), args.k)
        dump_outputs(args.dump_outputs, start + pick, idx[pick], d2[pick])
    t = sum(times[args.warmup:])
    value = sample * args.steps / t
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * t / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args, args.gpus),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": f"each step = {sample} of the {args.nq} queries against the full {args.n}-point kd-tree; restated FLANN KDTreeSingleIndex "
                                       f"(PCL 1.7 / FLANN cannot be built in this image), {cores} OpenMP threads"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


def _dbg(msg):
    if os.environ.get("PCC_BENCH_DEBUG"):
        print(f"[bench rank {os.environ.get('RANK', '0')}] {msg}", file=sys.stderr, flush=True)


def _events_ms(fn, reps, barrier, world, dist, torch):
    """max-over-ranks device time of `reps` calls of fn (CUDA events on the current stream, barrier + sync on both sides)."""
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def run_ours(args):
    import torch
    import torch.distributed as dist
    from pointcloudcomparator_b200 import shard
    from pointcloudcomparator_b200.search import GridSearch, launch_count

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    dev = torch.device(f"cuda:{local}")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    _dbg("process group up")
    ref, qry = make_clouds(args, 0)          # ONE common query set: every rank generates the same arrays (fixed seeds)
    _dbg("clouds generated")
    s = GridSearch(local)
    if world > 1:
        shard.attach(s)                      # our own ncclComm_t, handed to libpcc_search (pcc_comm_init)
    torch.cuda.synchronize()
    build_ms = build2_ms = 0.0
    if rank == 0:
        dref = torch.from_numpy(ref).cuda()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        s.setInputCloud(dref, k_hint=args.k)
        torch.cuda.synchronize()
        build_ms = 1e3 * (time.perf_counter() - t0)           # first call: includes every scratch allocation
        t0 = time.perf_counter()
        s.setInputCloud(dref, k_hint=args.k)
        torch.cuda.synchronize()
        build2_ms = 1e3 * (time.perf_counter() - t0)          # steady state: what a pipeline that rebuilds per consumer pays
    _dbg("index built")
    broadcast_ms = 0.0
    if world > 1:
        barrier()
        t0 = time.perf_counter()
        s.broadcastIndex(0)
        barrier()
        broadcast_ms = 1e3 * (time.perf_counter() - t0)
    grid = s.grid_info()
    meta = s._meta()
    _dbg(f"grid ready {grid}")

    # ---- this rank's shard of the common query set (contiguous range of the cell order) ------------
    if world > 1:
        mine, rows = shard.shard_queries(qry, rank, world, meta[5:8], grid["cell"], grid["dims"], block=args.shard_block)
    else:
        mine, rows = qry, None
    nq_local = mine.shape[0]
    dqry = torch.from_numpy(mine).cuda()
    drows = None if rows is None else torch.from_numpy(rows).to(dev)

    # ---- device-resident steps (strong scaling) ----------------------------------------------------------
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()                      # samples cover warm-up + timed steps + the kernel-timing re-run
        time.sleep(0.4)                      # let nvidia-smi attach before the first launch
    out = None
    for _ in range(args.warmup):
        out = s.nearestKSearch(dqry, args.k)
    barrier()
    l0 = launch_count()

    def step():
        nonlocal out
        out = s.nearestKSearch(dqry, args.k)

    ms = _events_ms(step, args.steps, barrier, world, dist, torch)
    launches = launch_count() - l0
    if args.dump_outputs:                    # `out` is the last timed step's result; N > 1: each rank holds its shard, gathered into query order
        ti, td = out[0], out[1]
        if world > 1:
            ti, td = s.gather(ti, drows, args.nq), s.gather(td, drows, args.nq)
        if rank == 0:
            pick = dump_rows(args.nq, args.k)
            sel = torch.from_numpy(pick).to(dev)
            dump_outputs(args.dump_outputs, pick, ti[sel].cpu().numpy(), td[sel].cpu().numpy())
        del ti, td
    rank_ms = None
    if world > 1:                # per-rank time of the same steps (load balance of the shards), gathered for the JSON line
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier(); e0.record()
        for _ in range(args.steps):
            step()
        e1.record(); torch.cuda.synchronize()
        mine_ms = torch.tensor([e0.elapsed_time(e1) / args.steps], dtype=torch.float64, device="cuda")
        allms = [torch.zeros_like(mine_ms) for _ in range(world)]
        dist.all_gather(allms, mine_ms)
        rank_ms = [round(float(x.item()), 4) for x in allms]
    value = args.nq * args.steps / (ms * 1e-3)
    _dbg(f"timed steps done {ms:.2f} ms")

    # ---- the dominant kernel alone (library-side CUDA events on the launch stream) -------------
    s.setTiming(True)
    kms = []
    for _ in range(args.steps):
        s.nearestKSearch(dqry, args.k)
        kms.append(s.lastKernelMs())
    s.setTiming(False)
    clocks = sampler.stop() if rank == 0 else None
    kernel_ms = float(np.mean(kms))
    peak, peak_src = measured_peak()
    bytes_per_query = 16.0 * args.n / args.nq + 16 + 8 * args.k
    achieved = nq_local * bytes_per_query / (kernel_ms * 1e-3) / 1e9
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        try:
            traffic = json.load(open(tpath)).get(f"knn_k{args.k}_{args.cloud}_{args.n}")
        except Exception:
            traffic = None

    # ---- correctness gate on the bench workload itself: sampled rows vs the CPU oracle, bit-exact ---------------
    parity = None
    tree = None
    gi, gd, _ = out
    if rank == 0 and not args.no_parity:
        import oracle
        tree = oracle.KdTree(ref)
        pick = np.random.default_rng(7).choice(nq_local, size=min(args.parity_rows, nq_local), replace=False)
        oi, od, _ = tree.knn(mine[pick], args.k, threads=host_threads())
        pidx = torch.from_numpy(pick).to(dev)
        ci, cd = gi[pidx].cpu().numpy(), gd[pidx].cpu().numpy()
        bad = int(((ci != oi) | (cd.view(np.uint32) != od.view(np.uint32))).any(axis=1).sum())
        parity = {"rows": int(len(pick)), "mismatches": bad, "checker": "oracle.KdTree.knn (restated FLANN KDTreeSingleIndex), indices and fp32 d2 bit-exact"}
        _dbg(f"parity sample {parity}")
    barrier()

    # ---- gather of the result table (the one optional collective), timed on its own -----------------------------
    gather_ms = None
    if world > 1:
        def gather():
            s.gather(gi, drows, args.nq)
            s.gather(gd, drows, args.nq)
        gather()
        gather_ms = _events_ms(gather, 3, barrier, world, dist, torch) / 3
        full_i = s.gather(gi, drows, args.nq)
        chk = int(full_i[:: max(args.nq // 1000, 1), 0].long().sum())
        del full_i
    else:
        chk = int(gi[:: max(args.nq // 1000, 1), 0].long().sum())

    # ---- weak scaling for comparison: every rank answers its OWN Q queries (round 1's number) -------------------
    weak_value = None
    if world > 1 and not args.no_weak:
        own = torch.from_numpy(make_clouds(args, rank)[1]).cuda()
        s.nearestKSearch(own, args.k)
        wsteps = max(1, min(args.steps, 5))
        wms = _events_ms(lambda: s.nearestKSearch(own, args.k), wsteps, barrier, world, dist, torch)
        weak_value = world * args.nq * wsteps / (wms * 1e-3)
        del own
    del out, gi, gd

    # ---- end to end through the C ABI with pinned host buffers ---------------------------------
    import ctypes as C
    from pointcloudcomparator_b200 import _lib
    L = _lib.lib()
    hq = torch.from_numpy(mine).pin_memory().numpy()
    e2e_steps = max(1, min(args.steps, 5))
    hidx = torch.empty((nq_local, args.k), dtype=torch.int32).pin_memory()
    hd2 = torch.empty((nq_local, args.k), dtype=torch.float32).pin_memory()
    hmd = torch.empty((nq_local,), dtype=torch.float32).pin_memory()
    keff = C.c_int()

    def e2e_step():
        _lib.check(L.pcc_knn(s._h, hq.ctypes.data, nq_local, hq.strides[0], args.k, hidx.data_ptr(), hd2.data_ptr(), C.byref(keff), _lib.HOST, None))

    def e2e_fused_step():      # the same search with the consumer's reduction fused on the device: 4 bytes per query come back
        _lib.check(L.pcc_knn_mean_dist(s._h, hq.ctypes.data, nq_local, hq.strides[0], args.k, hmd.data_ptr(), _lib.HOST, None))

    def wall(fn, reps):
        fn()
        barrier()
        t0 = time.perf_counter()
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
        t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    e2e_s = wall(e2e_step, e2e_steps)
    e2e_value = args.nq * e2e_steps / e2e_s
    fused_s = wall(e2e_fused_step, e2e_steps)
    checksum = int(hidx[:: max(nq_local // 1000, 1), 0].long().sum())
    h2d = int(nq_local * hq.strides[0]); d2h = int(nq_local * args.k * 8)
    _dbg("e2e done")

    # ---- BASELINE configs[3]: ICP pre-alignment, 10 M vs 10 M, source sharded over the ranks -------------------
    icp = None
    if not args.no_c4:
        from pointcloudcomparator_b200 import synth
        src, tgt, _ = synth.icp_pair(args.n, 4001, size=(10.0, 10.0, 3.0), stride4=True)
        t = GridSearch(local)
        if world > 1:
            shard.attach(t)
        if rank == 0:
            t.setInputCloud(torch.from_numpy(tgt).cuda(), k_hint=32)
        if world > 1:
            t.broadcastIndex(0)
        b, e = shard.shard_ranges(src.shape[0], world)[rank]
        dsrc = torch.from_numpy(np.ascontiguousarray(src[b:e])).cuda()
        r = t.icpAlign(dsrc.clone(), 20)                       # warm-up (scratch allocation)
        barrier()
        t0 = time.perf_counter()
        r = t.icpAlign(dsrc.clone(), 20)
        barrier()
        icp_s = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(icp_s, op=dist.ReduceOp.MAX)
        icp = {"ms": 1e3 * float(icp_s.item()), "iterations": int(r["iterations"]), "converged": bool(r["converged"]), "fitness": float(r["fitness"]),
               "source_points_total": int(src.shape[0]), "target_points": int(tgt.shape[0]),
               "how": "pcc_icp_align on this rank's shard of the source; 17 doubles all-reduced per pass (ncclAllReduce inside pcc_icp_step); wall clock, max over ranks"}
        del t, dsrc

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args, world),
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d * world, "d2h_bytes_per_step": d2h * world,
                    "steps": e2e_steps, "how": "pcc_knn(PCC_HOST) on every rank's shard with pinned host query / result buffers; H2D + sort + kernels + D2H inside the timed region; max over ranks",
                    "pcie_gbs_per_gpu": (h2d + d2h) * e2e_steps / e2e_s / 1e9, "checksum": checksum,
                    "fused_consumer": {"value": args.nq * e2e_steps / fused_s, "unit": UNIT, "d2h_bytes_per_step": int(nq_local * 4) * world,
                                       "how": "pcc_knn_mean_dist(PCC_HOST): same search, the SOR reduction fused on the device, 4 bytes per query returned -- shows what is left of e2e once the 128-byte result row does not cross PCIe"}},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                         "kernel": f"pcc::knn_thr_kernel<{args.k}> + the passes that finish what it lists (knn_thr_retry_kernel, DeviceSelect, knn_rings_kernel, knn_wide_kernel x2), timed together on rank 0's shard",
                         "kernel_ms": kernel_ms, "bytes_per_query": bytes_per_query, "queries_per_launch": int(nq_local), "peak_source": peak_src,
                         "how": "algorithmic bytes q*(16*N/Q + 16 + 8k) of this rank's q queries / mean kernel time over the same steps re-run with library-side CUDA events around the launches"},
            "parity_sample": parity, "result_checksum": chk,
            "build_ms": build_ms, "build_steady_ms": build2_ms,
            "build_roofline": {"algorithmic_bytes": int(args.n * (16 + 16 + 4)), "achieved_gbs": args.n * 36 / (build2_ms * 1e-3) / 1e9 if build2_ms else None, "peak": peak,
                               "frac": (args.n * 36 / (build2_ms * 1e-3) / 1e9 / peak) if build2_ms else None,
                               "how": "N*(stride_in 16 + float4 16 + cell id 4) bytes / steady-state pcc_build wall time (includes the occupancy auto-tune passes)"},
            "broadcast_ms": broadcast_ms, "grid": grid,
        }
        if world > 1:
            line["rank_ms_per_step"] = rank_ms
            line["gather_ms"] = gather_ms
            line["value_with_gather"] = args.nq / ((ms / args.steps + gather_ms) * 1e-3)
            line["gather_bytes_per_rank"] = int(args.nq * args.k * 8)
            line["weak_value"] = weak_value
        if icp is not None:
            line["icp_c4"] = icp
        if world == 1 and not args.no_cpu:
            cb, _, _ = cpu_baseline(ref, qry, args.k, tree=tree)
            line["cpu_baseline"] = cb
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


_REAL_STDOUT = None


def _claim_stdout():
    """Route everything libraries print on fd 1 (e.g. NCCL's version banner) to stderr; the JSON line alone goes to stdout."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def emit(line: dict):
    _REAL_STDOUT.write(json.dumps(line) + "\n")
    _REAL_STDOUT.flush()


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--ref-points", dest="n", type=int, default=10_000_000, help="reference points")
    ap.add_argument("--queries", dest="nq", type=int, default=10_000_000, help="queries per GPU")
    ap.add_argument("--k", type=int, default=K)
    ap.add_argument("--cloud", default="surface", choices=["surface", "uniform"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-parity", action="store_true", help="skip the sampled bit-exact check against the CPU oracle")
    ap.add_argument("--parity-rows", type=int, default=20000)
    ap.add_argument("--no-c4", action="store_true", help="skip the ICP 10 M vs 10 M arm (BASELINE configs[3])")
    ap.add_argument("--no-weak", action="store_true", help="skip the weak-scaling comparison steps at N > 1")
    ap.add_argument("--shard-block", type=int, default=8192, help="queries per block of the cell order dealt round-robin to the ranks (0 = one contiguous range per rank)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the last step's result rows (all of them, or a fixed seeded "
                                                             "sample within 64 MB) as DIR/query_rows.npy, DIR/knn_indices.npy and DIR/knn_sqr_distances.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
