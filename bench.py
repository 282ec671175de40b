#!/usr/bin/env python
"""bench.py — TrueKNN hot path on N B200s (one process per GPU).

    python bench.py --gpus 1 --steps 10 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...        # the CPU arm (oracle port, all host cores; rank 0 only under torchrun)

Metric (BASELINE.json): kNN queries/s, k = 10, 3-D.  A step = one full search (start-radius estimate + every
radius-doubling round) over the prebuilt LBVH, inputs resident in HBM; BVH build ms is reported beside it (the
reference's own split: "Build time" vs "True KNN time", samples/s01-trueknn/hostCode.cpp:201-212 vs :279-347).
`e2e` is the same metric through the C ABI with pinned HOST buffers: H2D of the points + build + search + D2H of
the results inside the timed region, with a per-phase split from CUDA events.  After the timed region every rank
checks sampled result rows against the exact GPU brute force (`verified`).

Workloads (--workload; the default "auto" is cfg2 at N = 1 and cfg4 at N > 1):
  cfg2  10 M uniform points (seed 42), every point is a query — BASELINE.json configs[1], the N = 1 headline.
        With --workload cfg2 at N > 1 it is weak-scaled (10 M x N points replicated, 10 M queries per GPU).
  cfg4  100 M uniform points at EVERY N, queries sharded by Morton slice over a replicated BVH — strong scaling,
        BASELINE.json configs[3] and the >= 6.5x target; the default for N > 1.  At N > 1 rank 0 also times the whole
        workload on its own GPU (`single_gpu_same_workload`) so the speed-up is measured inside one job.
  cfg5  2 B uniform points partitioned by Morton range over the ranks (BASELINE.json configs[4]; 8 GPUs); every rank
        generates its index slice on the device; checked by the distributed brute force (tknn_partition_verify).
  cfg1 / cfg3  parity-test shapes, runnable for completeness (100 K k=5; 10 M LiDAR-like k=64).
All multi-GPU collectives run inside libtrueknn over NCCL; torch.distributed carries the NCCL unique id and the
max-over-ranks reductions of the timings.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

WORKLOADS = {
    "cfg1": dict(n=100_000, k=5, cloud="uniform", seed=42, scaling="weak", mode="shard",
                 name="cfg1: TrueKNN k=5 on 100K uniform 3-D points (seed 42), all points are queries"),
    "cfg2": dict(n=10_000_000, k=10, cloud="uniform", seed=42, scaling="weak", mode="shard",
                 name="cfg2: TrueKNN k=10 on 10M uniform 3-D points (seed 42), all points are queries"),
    "cfg3": dict(n=10_000_000, k=64, cloud="lidar", seed=7, scaling="weak", mode="shard",
                 name="cfg3: TrueKNN k=64 on 10M clustered LiDAR-like 3-D points (seed 7)"),
    "cfg4": dict(n=100_000_000, k=10, cloud="uniform", seed=42, scaling="strong", mode="shard",
                 name="cfg4: query-sharded kNN k=10 on 100M uniform 3-D points, BVH replicated per GPU"),
    "cfg5": dict(n=2_000_000_000, k=10, cloud="uniform", seed=42, scaling="strong", mode="partition",
                 name="cfg5: point-partitioned kNN k=10 on 2B uniform 3-D points (Morton-range ownership, boundary-query "
                      "exchange + partial top-k merge over NCCL)"),
}


def resolve_workload(args) -> str:
    if args.workload != "auto":
        return args.workload
    return "cfg2" if args.gpus == 1 else "cfg4"


def _peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu, self.proc, self.lines = gpu_index, None, []
        self.t_begin = self.t_end = None

    def mark_begin(self):
        self.t_begin = time.time()

    def mark_end(self):
        self.t_end = time.time()

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def sm_mhz_so_far(self):
        vals = []
        for ts, ln in self.lines:
            f = ln.split(",")
            if len(f) >= 9 and self.t_begin and ts >= self.t_begin - 0.05 and (not self.t_end or ts <= self.t_end + 0.15):
                try:
                    vals.append(float(f[1]))
                except ValueError:
                    pass
        return float(np.median(vals)) if vals else None

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            # samples from the first warm-up step to the end of the timed region count as "under load"
            if self.t_begin and ts < self.t_begin - 0.05:
                continue
            if self.t_end and ts > self.t_end + 0.15:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------------------------------
# CPU arm: the oracle port timed on ALL host cores (the reference has no CPU implementation of its own and cannot be
# compiled here — OptiX — so `kind` is "port").  Queries are runs of consecutive positions of the kd-tree's own point
# order, i.e. spatially coherent like the GPU arm's Morton order; the cloud is the GPU arm's cloud.
# --------------------------------------------------------------------------------------------------
def _cpu_cloud(cfg: dict, n_points: int):
    from owlraytracing_b200 import datasets

    return datasets.uniform(n_points, cfg["seed"]) if cfg["cloud"] == "uniform" else datasets.lidar_like(n_points, cfg["seed"])


def _coherent_positions(n_points: int, m: int, it: int, run: int = 4096) -> np.ndarray:
    """m tree positions as evenly spread runs of `run` consecutive positions (a different offset every step)."""
    if n_points <= run or m >= n_points:
        return np.arange(m, dtype=np.int64) % n_points
    runs = max(1, (m + run - 1) // run)
    stride = max(1, (n_points - run) // runs)
    starts = np.arange(runs, dtype=np.int64) * stride + (it * 7919) % stride
    return (starts[:, None] + np.arange(run, dtype=np.int64)[None, :]).reshape(-1)[:m]


def cpu_arm(cfg: dict, n_points: int, steps: int, warmup: int, sample_queries: int, label: str, with_scipy: bool = False):
    os.environ["OMP_NUM_THREADS"] = str(os.cpu_count() or 1)   # torchrun exports 1 to its workers
    from oracle import oracle as O

    O.set_num_threads(os.cpu_count() or 1)   # liboracle.so comes from build(): the benchmark compiles nothing in the tree
    x = _cpu_cloud(cfg, n_points)
    t0 = time.perf_counter()
    tree = O.KdTree(x, leaf=8)
    build_s = time.perf_counter() - t0
    m = min(sample_queries, n_points)
    times = []
    for it in range(warmup + steps):
        pos = _coherent_positions(n_points, m, it)
        t0 = time.perf_counter()
        tree.query_positions(pos, cfg["k"])
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    tree.close()
    per_step = float(np.mean(times)) if times else float("nan")
    res = {
        "value": m / per_step, "unit": "queries/s", "cores": O.num_threads(), "kind": "port",
        "sample": f"{label}: {m} queries per step, taken as runs of 4096 consecutive points of the kd-tree's own order "
                  f"(spatially coherent, like the GPU arm's Morton order), against the full {n_points}-point exact kd-tree "
                  f"(oracle/knn_oracle.c, OpenMP on all {O.num_threads()} threads; tree build {build_s:.2f} s excluded like the GPU build)",
        "build_s": build_s, "ms_per_step": per_step * 1e3,
    }
    if with_scipy:
        try:
            from scipy.spatial import cKDTree

            t0 = time.perf_counter()
            st = cKDTree(x.astype(np.float64), leafsize=16)
            sb = time.perf_counter() - t0
            ms = min(m, 500_000)
            pos = _coherent_positions(n_points, ms, 0)
            q = x[pos % n_points].astype(np.float64)
            t0 = time.perf_counter()
            st.query(q, k=cfg["k"] + 1, workers=-1)
            sq = time.perf_counter() - t0
            res["second"] = {"value": ms / sq, "unit": "queries/s", "cores": os.cpu_count(), "kind": "scipy.spatial.cKDTree",
                             "sample": f"{ms} queries (k+1 with self, float64, leafsize 16, workers=-1) against the full "
                                       f"{n_points}-point tree; tree build {sb:.2f} s excluded"}
        except Exception as e:  # noqa: BLE001
            res["second"] = {"unavailable": f"scipy cKDTree: {e}"}
    return res


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = resolve_workload(args)
    cfg = WORKLOADS[wl]
    n_points = cfg["n"]
    if wl == "cfg2" and args.gpus > 1:
        n_points = cfg["n"] * args.gpus
    if args.points:
        n_points = args.points
    note = None
    if n_points > 200_000_000:  # no host kd-tree at 2 B points: the CPU arm answers over the first 100 M indices
        note = f"CPU tree over the first 100000000 of {n_points} points (a 2 B-point host kd-tree does not fit the run)"
        n_points = 100_000_000
    res = cpu_arm(cfg, n_points, args.steps, args.warmup, args.cpu_sample, "reference arm")
    line = {
        "impl": "reference", "metric": "knn_queries_per_s", "value": res["value"], "unit": "queries/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": res["ms_per_step"], "higher_is_better": True,
        "scaling": cfg["scaling"] if not (wl == "cfg2") else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": cfg["name"], "n_points": n_points, "k": cfg["k"], "queries_per_step": min(args.cpu_sample, n_points),
                   "note": note},
        "cpu_baseline": {k: res[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": res["value"], "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------------
# roofline of the dominant kernel (tknn::trav::traverse_kernel)
# --------------------------------------------------------------------------------------------------
def _ncu_profile(workload: str):
    """Per-workload ncu capture of the traversal kernel (tools/ncu_profile.py writes it): instruction count, DRAM bytes,
    l1tex / issue-slot utilisation of round 1 at the workload's full size."""
    path = os.path.join(ROOT, "profiles", f"r2_traverse_{workload}_ncu.json")
    try:
        return json.load(open(path)), os.path.relpath(path, ROOT)
    except Exception:
        return None, None


def roofline_block(t, wl, cfg, cs, nq, n_points, n_nodes, kern_ms_per_step, ms_per_step, sm_mhz, round1_ms_per_step):
    k = cfg["k"]
    alg_bytes = nq * (16 + 8 * k) + 64 * cs["nodes_visited"] + 16 * cs["points_tested"]
    warp_bytes = nq * (16 + 8 * k) + 64 * cs["warp_node_visits"] + 16 * cs["warp_point_loads"]
    kt = kern_ms_per_step * 1e-3
    hbm_peak, hbm_src = _peaks()
    achieved = alg_bytes / kt / 1e9
    sm = t.measure_smem_bandwidth()          # live: ~12 launches of ~1 ms
    smem_peak = sm["smem_conflict_free_gbs"]
    # compulsory HBM traffic (SURVEY.md §8d B_min): every point, node and query once, every result row once
    b_min = 16 * n_points + 64 * n_nodes + 16 * nq + 8 * k * nq
    prof, prof_path = _ncu_profile(wl)
    traffic = issue = l1tex = None
    if prof:
        traffic = prof["dram_bytes_per_query"] * nq
        sm_hz = (sm_mhz or 1965.0) * 1e6
        winst = prof["warp_instructions_per_query"] * nq
        peak_issue = 148 * 4 * sm_hz             # one warp instruction per SM sub-partition per cycle
        k1 = max(round1_ms_per_step, 1e-6) * 1e-3   # the capture is round 1's launch: divide by round 1's live time
        issue = {"warp_instructions_per_query": prof["warp_instructions_per_query"],
                 "achieved_warp_inst_per_s": winst / k1, "peak_warp_inst_per_s": peak_issue, "frac": winst / k1 / peak_issue,
                 "round1_kernel_ms": round1_ms_per_step,
                 "ncu_issue_active_pct": prof.get("issue_active_pct"), "ncu_threads_per_inst": prof.get("threads_per_inst"),
                 "note": "warp instructions of round 1's traverse_kernel launch from the ncu capture of THIS workload (full size) "
                         "over that launch's live time and the SM clock sampled during the run"}
        l1tex = prof.get("l1tex_throughput_pct")
    return {
        "bound": "smem", "achieved": achieved, "peak": smem_peak, "unit": "GB/s", "frac": achieved / smem_peak,
        "traffic": traffic, "kernel": "tknn::trav::traverse_kernel", "kernel_ms_per_step": kern_ms_per_step,
        "kernel_share_of_step": kern_ms_per_step / ms_per_step,
        "peak_source": "measured live: tknn_measure_smem_bandwidth, conflict-free LDS.128, bytes delivered to lanes "
                       "(the 128 B/clk/SM shared-memory / L1 data path the kernel's node and leaf reads go through)",
        "smem_broadcast_peak_gbs": sm["smem_broadcast_gbs"],
        "algorithmic_bytes_per_query": alg_bytes / max(nq, 1),
        "bytes_per_query_loaded_once_per_warp": warp_bytes / max(nq, 1),
        "hbm": {"compulsory_bytes": b_min, "achieved_gbs": b_min / kt / 1e9, "peak_gbs": hbm_peak, "peak_source": hbm_src,
                "frac": b_min / kt / 1e9 / hbm_peak,
                "ncu_dram_traffic_over_compulsory": (traffic / b_min) if traffic else None,
                "ncu_dram_gbs": (traffic / kt / 1e9) if traffic else None,
                "note": "the kernel cannot be HBM-bound: a warp loads each node / leaf once for 32 queries"},
        "ncu_l1tex_throughput_pct": l1tex, "issue_slots": issue, "ncu_profile": prof_path,
        "nodes_per_query": cs["nodes_visited"] / max(nq, 1), "points_tested_per_query": cs["points_tested"] / max(nq, 1),
        "note": "SURVEY.md §8d's algorithmic bytes (every query billed for its own node and point reads) against the measured "
                "shared-memory/L1 bandwidth: the reads are served once per warp from L1/shared memory and broadcast, so this — "
                "with the issue-slot fraction — is the roof that binds; `hbm` holds the compulsory-traffic view",
    }


# --------------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------------
DUMP_BYTES = 60_000_000   # array bytes of --dump-outputs: with the .npy headers, under 64 MB


def dump_outputs(path, qid, idx, dist, rank, world):
    """Write the rows one search step returned (query ids, neighbour indices, distances) as DIR/<name>.npy, for comparing
    two builds output for output.  Rows are taken in query-id order, so the files do not depend on the order the engine
    emits rows in; when all rows exceed DUMP_BYTES (over all ranks), a fixed seeded sample of them is written.  Ids and
    indices are stored as float64, which holds every int32 exactly.  With several ranks each writes its own files."""
    import torch

    n, k = int(idx.shape[0]), int(idx.shape[1])
    m = min(n, DUMP_BYTES // ((8 + 8 * k + 4 * k) * world))
    pick = torch.from_numpy(np.sort(np.random.default_rng(0).choice(n, m, replace=False))).to(qid.device)
    rows = torch.argsort(qid.long())[pick]
    suffix = f"_rank{rank}" if world > 1 else ""
    os.makedirs(path, exist_ok=True)
    for name, a in (("query_ids", qid[rows].double()), ("neighbour_indices", idx[rows].double()),
                    ("neighbour_distances", dist[rows].float())):
        np.save(os.path.join(path, f"{name}{suffix}.npy"), a.cpu().numpy())


def run_gpu(args):
    # ONE JSON line on stdout: whatever libraries print there (NCCL announces its version on stdout when a communicator
    # is created) goes to stderr; the line itself is written to the saved descriptor at the end
    json_fd = os.dup(1)
    sys.stdout.flush()
    os.dup2(2, 1)

    import torch
    import torch.distributed as dist

    from owlraytracing_b200 import TrueKNN, datasets

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world == 1 and args.gpus > 1:
        raise SystemExit("--gpus N > 1 must be launched with torch.distributed.run --nproc-per-node N")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(vals):
        tm = torch.tensor(vals, dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        return [float(v) for v in tm.tolist()]

    def sum_over_ranks(vals):
        tm = torch.tensor(vals, dtype=torch.int64, device=dev)
        if world > 1:
            dist.all_reduce(tm, op=dist.ReduceOp.SUM)
        return [int(v) for v in tm.tolist()]

    wl = resolve_workload(args)
    cfg = WORKLOADS[wl]
    k = cfg["k"]
    partition = cfg["mode"] == "partition"
    weak_grow = wl == "cfg2" and world > 1
    n_points = cfg["n"] * world if weak_grow else cfg["n"]
    if args.points:
        n_points = args.points
    scaling = "weak" if wl in ("cfg1", "cfg2", "cfg3") else "strong"

    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()  # nvidia-smi needs ~1 s to start streaming; it runs through warm-up and the timed region
    t = TrueKNN(local_rank, **{kv.split("=")[0]: int(kv.split("=")[1]) for kv in args.opt})
    stream = torch.cuda.current_stream()
    t.set_stream(stream.cuda_stream)
    if world > 1:
        t.comm_init_torch()      # NCCL communicator inside the library; torch only carries the unique id

    # ---- synthetic input ----
    if partition:
        lo, hi = n_points * rank // world, n_points * (rank + 1) // world
        xd = torch.empty((hi - lo, 3), dtype=torch.float32, device=dev)
        t.generate_uniform(cfg["seed"], lo, hi - lo, out=xd)     # this rank's index slice, generated on the device
    elif cfg["cloud"] == "uniform":
        xd = torch.empty((n_points, 3), dtype=torch.float32, device=dev)
        t.generate_uniform(cfg["seed"], 0, n_points, out=xd)
    else:
        xd = torch.from_numpy(datasets.lidar_like(n_points, cfg["seed"])).to(dev)
    torch.cuda.synchronize()

    # ---- build (timed separately) ----
    build_ms, dstats_build = [], None
    for _ in range(3):
        if partition:
            barrier()
            t.partition_build(xd, lo)
            dstats_build = t.dist_stats()
            build_ms.append(dstats_build["build_total_ms"])
        else:
            t.build(xd)
            build_ms.append(t.stats()["build_ms"])
    bstats = t.stats()
    if partition:
        del xd                                  # the owned points live in the library now
        torch.cuda.empty_cache()
        cap = t.partition_owned()
    else:
        cap = t.shard_capacity(world)
    qid = torch.empty((cap,), dtype=torch.int32, device=dev)
    idx = torch.empty((cap, k), dtype=torch.int32, device=dev)
    dst = torch.empty((cap, k), dtype=torch.float32, device=dev)

    def step():
        if partition:
            return t.partition_search(k, args.start_radius, out=(qid, idx, dst))
        return t.search_shard(k, rank, world, start_radius=args.start_radius, out=(qid, idx, dst))

    if sampler:
        sampler.mark_begin()
    for _ in range(max(args.warmup, 0)):
        step()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches, kernel_ms_sum, kernel_ms_round1 = 0, 0.0, 0.0
    ev0.record(stream)
    for _ in range(args.steps):
        q_r, i_r, d_r = step()
        s = t.stats()
        launches += s["kernel_launches"]
        kernel_ms_sum += sum(s["kernel_ms"])   # the traversal kernels of every round (CUDA events inside the library)
        kernel_ms_round1 += s["kernel_ms"][0] if s["kernel_ms"] else 0.0
    ev1.record(stream)
    barrier()
    if sampler:
        sampler.mark_end()
    elapsed_ms = max_over_ranks([ev0.elapsed_time(ev1)])[0]
    my_queries = int(q_r.shape[0])
    sstats = t.stats()
    dstats = t.dist_stats() if partition else None
    total_queries = sum_over_ranks([my_queries])[0]
    ms_per_step = elapsed_ms / args.steps
    value = total_queries / (ms_per_step * 1e-3)
    sm_mhz = sampler.sm_mhz_so_far() if sampler else None
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, q_r, i_r, d_r, rank, world)   # before any later search reuses the buffers

    # ---- in-bench correctness: sampled rows against the exact GPU brute force, at every N ----
    if partition:
        checked, bad = t.partition_verify(k, min(args.verify_samples_partition, my_queries), q_r, i_r, d_r)
        verify = {"method": "tknn_partition_verify: every rank brute-forces all sampled queries against its own points, "
                            "partial lists all-gathered and merged on (d2, global index)", "samples_per_rank":
                  min(args.verify_samples_partition, my_queries), "checked": checked, "bad": bad}
    else:
        m = min(args.verify_samples, my_queries)
        rows = (torch.arange(m, device=dev, dtype=torch.int64) * my_queries) // max(m, 1)
        ids = q_r[rows].contiguous()
        bi, bd = t.brute_force(ids, k)
        bad_local = int(((bi != i_r[rows]).any(1) | (bd != d_r[rows]).any(1)).sum().item())
        checked, bad = sum_over_ranks([m, bad_local])
        verify = {"method": "tknn_brute_force (exact tiled GPU brute force over the replicated cloud) on evenly spaced rows of "
                            "every rank's shard, indices and distances compared bit for bit", "samples_per_rank": m,
                  "checked": checked, "bad": bad}
    verified = bool(checked > 0 and bad == 0)

    # ---- strong scaling: the same workload on ONE GPU, measured inside this job (rank 0; the others wait) ----
    single = None
    if world > 1 and scaling == "strong" and not partition and not args.no_single:
        if rank == 0:
            cap1 = t.shard_capacity(1)
            q1 = torch.empty((cap1,), dtype=torch.int32, device=dev)
            i1 = torch.empty((cap1, k), dtype=torch.int32, device=dev)
            d1 = torch.empty((cap1, k), dtype=torch.float32, device=dev)
            t.search_shard(k, 0, 1, start_radius=args.start_radius, out=(q1, i1, d1))
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = max(2, min(args.steps, 4))
            e0.record(stream)
            for _ in range(reps):
                t.search_shard(k, 0, 1, start_radius=args.start_radius, out=(q1, i1, d1))
            e1.record(stream)
            torch.cuda.synchronize()
            ms1 = e0.elapsed_time(e1) / reps
            single = {"n_gpus": 1, "ms_per_step": ms1, "value": n_points / (ms1 * 1e-3), "steps": reps,
                      "speedup_of_this_run": value / (n_points / (ms1 * 1e-3))}
            del q1, i1, d1
            torch.cuda.empty_cache()
        barrier()

    # ---- roofline of the dominant kernel ----
    roofline = None
    t.set_option("counters", 1)   # one counting step on every rank (in partition mode a step is collective)
    step()
    cs = t.stats()
    t.set_option("counters", 0)
    if rank == 0:
        roofline = roofline_block(t, wl, cfg, cs, my_queries, int(bstats["n_points"]), bstats["n_nodes"],
                                  kernel_ms_sum / args.steps, ms_per_step, sm_mhz, kernel_ms_round1 / args.steps)

    # ---- end to end through the C ABI with pinned host buffers ----
    e2e = None
    if not args.no_e2e:
        e2e = run_e2e(args, t, torch, dist, dev, stream, world, rank, wl, cfg, n_points, cap, total_queries, barrier,
                      max_over_ranks, xd if not partition else None, partition, lo if partition else 0,
                      (hi - lo) if partition else 0)

    # ---- CPU baseline beside it (rank 0, N = 1 only) ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cpu = cpu_arm(cfg, n_points, steps=2, warmup=1, sample_queries=args.cpu_sample, label="cpu_baseline", with_scipy=True)
        cpu = {kk: cpu[kk] for kk in ("value", "unit", "cores", "kind", "sample", "second") if kk in cpu}

    clocks = sampler.stop() if sampler else None
    if rank == 0:
        if weak_grow:
            wname = (f"cfg2 weak-scaled: query-sharded kNN k=10, {n_points} uniform points replicated per GPU, "
                     f"10M queries per GPU")
        else:
            wname = cfg["name"]
        line = {
            "metric": "knn_queries_per_s", "value": value, "unit": "queries/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": scaling,
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "verified": verified, "verify": verify,
            "config": {
                "workload": wname, "n_points": n_points, "k": k, "queries_total": total_queries, "queries_per_gpu": my_queries,
                "sharding": ("points partitioned by Morton range (cell-aligned splitters), boundary queries exchanged, partial "
                             "top-k merged — NCCL inside libtrueknn" if partition else
                             "queries sharded by contiguous Morton slice, BVH replicated, no data-path collective"),
                "start_radius": "auto (sampled k-th-neighbour distance)" if args.start_radius <= 0 else args.start_radius,
                "l2_policy": f"inputs larger than L2: {int(bstats['n_points']) * 16 / 1e6:.0f} MB points + "
                             f"{bstats['n_nodes'] * 64 / 1e6:.0f} MB nodes + {my_queries * k * 8 / 1e6:.0f} MB results per step per GPU "
                             f"vs 126 MB L2",
                "timed_region": "search only (estimate + all rounds" + (" + exchange + remote search + merge" if partition else "") +
                                "), CUDA events on the launching stream, max over ranks; build reported separately",
            },
            "build_ms": float(np.median(build_ms)), "build_ms_all": [float(v) for v in build_ms],
            "build_phases_ms": ({p: dstats_build[p] for p in ("box_ms", "codes_ms", "splitters_ms", "bucket_ms", "exchange_ms",
                                                              "lbvh_ms", "summaries_ms")} if partition else
                                {p: bstats[p] for p in ("bounds_ms", "morton_ms", "sort_ms", "leaves_ms", "hierarchy_ms", "refit_ms")}),
            "rounds": int(sstats["rounds"]), "round_queries": sstats["round_queries"], "round_ms": sstats["round_ms"],
            "start_radius": sstats["start_radius"],
            "queries_per_s_incl_build": total_queries / ((ms_per_step + float(np.median(build_ms))) * 1e-3),
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu,
        }
        if single:
            line["single_gpu_same_workload"] = single
        if partition:
            line["partition"] = {p: dstats[p] for p in ("n_owned", "local_search_ms", "reach_ms", "exchange_out_ms",
                                                        "remote_search_ms", "exchange_back_ms", "merge_ms", "finish_ms",
                                                        "search_total_ms", "boundary_sent", "boundary_received",
                                                        "bytes_sent_search")}
            line["partition"]["bytes_sent_build"] = dstats_build["bytes_sent_build"]
        sys.stdout.flush()
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    t.close()
    if world > 1:
        dist.destroy_process_group()


def run_e2e(args, t, torch, dist, dev, stream, world, rank, wl, cfg, n_points, cap, total_queries, barrier, max_over_ranks, xd,
            partition, p_lo, p_n):
    """The same metric through the C ABI with pinned HOST buffers, every step: H2D of this rank's points, build, search,
    D2H of its result rows.  Phases from the library's CUDA events (tknn_stats / tknn_dist_stats)."""
    import psutil

    k = cfg["k"]
    out_bytes = cap * k * 8 + cap * 4
    in_rows = p_n if partition else (n_points if world == 1 else (n_points + world - 1) // world)
    need = out_bytes + in_rows * 12
    avail = psutil.virtual_memory().available
    if need * world * 1.5 > avail:
        return {"skipped": f"pinned host buffers of {need / 1e9:.1f} GB per rank x {world} ranks exceed the host memory "
                           f"available to this run ({avail / 1e9:.0f} GB)"}
    if partition:
        xh = torch.empty((p_n, 3), dtype=torch.float32, pin_memory=True)
        t.generate_uniform(cfg["seed"], p_lo, p_n, out=xh.numpy())
        my_slice = xh
    else:
        xh = torch.empty((in_rows, 3), dtype=torch.float32, pin_memory=True)
        per = (n_points + world - 1) // world
        first = min(n_points, per * rank) if world > 1 else 0
        xh.copy_(xd[first: first + in_rows])
        my_slice = xh
    qid_h = torch.empty((cap,), dtype=torch.int32, pin_memory=True)
    idx_h = torch.empty((cap, k), dtype=torch.int32, pin_memory=True)
    dst_h = torch.empty((cap, k), dtype=torch.float32, pin_memory=True)
    out_np = (qid_h.numpy(), idx_h.numpy(), dst_h.numpy())
    full_np = (idx_h.numpy()[:n_points], dst_h.numpy()[:n_points]) if world == 1 and not partition else None
    phases = {"h2d_ms": 0.0, "allgather_ms": 0.0, "build_ms": 0.0, "search_ms": 0.0, "d2h_ms": 0.0}

    def e2e_step(record):
        if partition:
            t.partition_build(my_slice.numpy(), p_lo)
            ds = t.dist_stats()
            t.partition_search(k, args.start_radius, out=out_np)
            ss, ds2 = t.stats(), t.dist_stats()
            if record:
                phases["h2d_ms"] += ds["h2d_ms"]
                phases["build_ms"] += ds["build_total_ms"] - ds["h2d_ms"]
                phases["search_ms"] += ds2["search_total_ms"]
                phases["d2h_ms"] += ds2["d2h_ms"]
            return ss
        if world == 1:
            t.build(my_slice.numpy())                       # H2D of the points + LBVH build
            bs = t.stats()
            if args.e2e_shard_api:
                t.search_shard(k, 0, 1, start_radius=args.start_radius, out=out_np)
            else:
                t.search(k, args.start_radius, out=full_np)  # the reference-facing call: rows in file order, search + D2H
            ss = t.stats()
            if record:
                phases["h2d_ms"] += bs["h2d_ms"]
                phases["build_ms"] += bs["build_ms"]
        else:
            per = (n_points + world - 1) // world
            t.build_replicated(my_slice.numpy(), min(n_points, per * rank), n_points)   # H2D slice + ncclAllGather + build
            ds = t.dist_stats()
            t.search_shard(k, rank, world, start_radius=args.start_radius, out=out_np)   # search + D2H
            ss = t.stats()
            if record:
                phases["h2d_ms"] += ds["h2d_ms"]
                phases["allgather_ms"] += ds["allgather_ms"]
                phases["build_ms"] += ds["lbvh_ms"]
        if record:
            phases["search_ms"] += ss["search_ms"]
            phases["d2h_ms"] += ss["d2h_ms"]
        return ss

    if args.output_chunks > 0:
        t.set_option("output_chunks", args.output_chunks)
    if args.file_order_chunks > 0:
        t.set_option("file_order_chunks", args.file_order_chunks)
    e2e_steps = max(1, min(args.steps, args.e2e_steps))
    e2e_step(False)
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    ev0.record(stream)
    for _ in range(e2e_steps):
        es = e2e_step(True)
    ev1.record(stream)
    barrier()
    wall_ms = (time.perf_counter() - t0) * 1e3
    e_ms, wall_ms = max_over_ranks([max(ev0.elapsed_time(ev1), 0.0), wall_ms])
    e_ms /= e2e_steps
    ph = max_over_ranks([phases[p] / e2e_steps for p in ("h2d_ms", "allgather_ms", "build_ms", "search_ms", "d2h_ms")])
    indices_only = None
    if world == 1 and not partition and not args.e2e_shard_api:
        # the same step with dist_out = NULL: only the neighbour indices leave the device (half the D2H bytes)
        def io_step():
            t.build(my_slice.numpy())
            t.search(k, args.start_radius, out=(full_np[0], None))
            return t.stats()
        io_step()
        torch.cuda.synchronize()
        io0, io1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        io0.record(stream)
        for _ in range(e2e_steps):
            ios = io_step()
        io1.record(stream)
        torch.cuda.synchronize()
        io_ms = io0.elapsed_time(io1) / e2e_steps
        indices_only = {"value": total_queries / (io_ms * 1e-3), "unit": "queries/s", "ms_per_step": io_ms,
                        "h2d_bytes_per_step": int(my_slice.shape[0] * 12), "d2h_bytes_per_step": int(ios["d2h_bytes"]),
                        "api": "tknn_build + tknn_search(dist_out = NULL): neighbour indices only, rows in file order",
                        "note": "not the headline: the reference's output is indices AND distances (e2e.value); reported because "
                                "the device->host copy of the rows bounds the step and a distance is recomputable from its index"}
    if partition:
        api = "tknn_partition_build + tknn_partition_search (host arrays)"
    elif world == 1 and not args.e2e_shard_api:
        api = "tknn_build + tknn_search (rows in file order)"
    elif world == 1:
        api = "tknn_build + tknn_search_shard (compact Morton-order rows + query ids)"
    else:
        api = "tknn_build_replicated + tknn_search_shard (compact Morton-order rows + query ids)"
    return {"value": total_queries / (e_ms * 1e-3), "unit": "queries/s", "h2d_bytes_per_step": int(my_slice.shape[0] * 12),
            "d2h_bytes_per_step": int(es["d2h_bytes"]), "ms_per_step": e_ms, "wall_ms_per_step": wall_ms / e2e_steps,
            "phases_ms_max_over_ranks": dict(zip(("h2d_ms", "allgather_ms", "build_ms", "search_ms", "d2h_ms"), ph)),
            "phases_note": "CUDA events inside the library; with host outputs the search is sliced and each slice's D2H overlaps "
                           "the next slice's search, so search_ms includes the overlapped copies and d2h_ms is the exposed tail",
            "h2d_note": ("per rank: its 1/N slice of the points (pinned); one ncclAllGather inside the library replicates the cloud"
                         if world > 1 and not partition else "per rank: its points (pinned)"),
            "steps": e2e_steps, "includes": "H2D points (pinned) + build + search (all rounds) + D2H results (pinned)", "api": api,
            **({"indices_only": indices_only} if indices_only else {})}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="auto", choices=["auto"] + sorted(WORKLOADS))
    ap.add_argument("--points", type=int, default=0, help="override the number of points (debug)")
    ap.add_argument("--start-radius", type=float, default=0.0, help="<= 0: auto")
    ap.add_argument("--cpu-sample", type=int, default=2_000_000, help="queries per CPU step")
    ap.add_argument("--verify-samples", type=int, default=256, help="rows per rank checked against the GPU brute force")
    ap.add_argument("--verify-samples-partition", type=int, default=2048)
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--output-chunks", type=int, default=0, help="e2e: Morton slices whose D2H overlaps the search (0 = library default)")
    ap.add_argument("--file-order-chunks", type=int, default=0, help="e2e through tknn_search: slices by original index (0 = default)")
    ap.add_argument("--e2e-shard-api", action="store_true", help="N=1 e2e through tknn_search_shard (compact Morton rows) instead of tknn_search")
    ap.add_argument("--opt", action="append", default=[], help="library option for experiments, name=value (tknn_set_option)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-single", action="store_true", help="N > 1 strong scaling: skip the single-GPU run of the same workload")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last step's results (a seeded sample, <= 64 MB) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the GPU search's results; it does not apply to --impl reference")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3  # timing rule: at least 3 warm-up steps
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
