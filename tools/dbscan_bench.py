"""DBSCAN benchmark: tknn_dbscan on the flagship clouds, verified against the CPU reference; prints one JSON line.

    python tools/dbscan_bench.py [--steps 5] [--workloads lidar_0.05,lidar_0.3,uniform_0.006] [--sklearn-points 1000000]

Workloads: 10 M `lidar_like` (seed 7) at eps = 0.05 and 0.3, 10 M uniform (seed 42) at eps = 0.006, min_pts = 10.
Per workload: per-phase device times (median of --steps calls after one warm-up call; the cloud and the outputs live
on the device, so no host copy is timed), points/s of the whole call, core fraction and C, node visits and point
tests per query from a separate counters run (summed over the three traversal passes: tknn_stats has one set of
counters per call), a shared-memory roofline fraction computed as bench.py computes it for the search, `verified`
(labels, core flags and C equal the CPU reference), the CPU reference's own time on all host cores, and
scikit-learn (n_jobs=-1) on the first --sklearn-points points.  The GPU's name and power limit are read in the run.
Writes nothing into the tree.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

WORKLOADS = {
    "lidar_0.05": ("lidar_like", 10_000_000, 7, 0.05, 10),
    "lidar_0.3": ("lidar_like", 10_000_000, 7, 0.3, 10),
    "uniform_0.006": ("uniform", 10_000_000, 42, 0.006, 10),
}
PHASES = ("core", "link", "label", "border")


def device_info(torch):
    info = {"name": torch.cuda.get_device_name(0), "power_limit_w": None}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_w"] = float(out.splitlines()[0])
    except Exception as e:  # noqa: BLE001 — reported, not hidden
        info["power_limit_w_error"] = repr(e)
    return info


def cloud(kind, n, seed):
    from owlraytracing_b200 import datasets

    return datasets.lidar_like(n, seed=seed) if kind == "lidar_like" else datasets.uniform(n, seed=seed)


def run_workload(name, x, eps, min_pts, steps, sk_points, smem_peak, torch):
    import dbscan_oracle as DO
    from owlraytracing_b200 import TrueKNN

    n = int(x.shape[0])
    xd = torch.from_numpy(x).cuda()
    res = {"workload": name, "n": n, "eps": eps, "min_pts": min_pts}
    with TrueKNN(0) as t:
        t.build(xd)
        labels, core, c = t.dbscan(eps, min_pts)  # warm-up (module load, scratch allocation)
        phase_ms, call_ms, kern_ms = [], [], []
        for _ in range(steps):
            labels, core, c = t.dbscan(eps, min_pts)
            st = t.stats()
            phase_ms.append(st["round_ms"][:4])
            kern_ms.append(st["kernel_ms"][:4])
            call_ms.append(st["search_ms"])
        labels, core = labels.cpu().numpy(), core.cpu().numpy()
        t.set_option("counters", 1)
        t.dbscan(eps, min_pts)
        cs = t.stats()
    med = float(np.median(call_ms))
    res["phase_ms"] = {p: float(np.median([r[i] for r in phase_ms])) for i, p in enumerate(PHASES)}
    res["kernel_ms"] = {p: float(np.median([r[i] for r in kern_ms])) for i, p in enumerate(PHASES) if p != "label"}
    res["call_ms"] = med
    res["call_ms_all"] = call_ms
    res["points_per_s"] = n / (med * 1e-3)
    res["core_fraction"] = float(core.mean())
    res["clusters"] = int(c)
    res["noise_fraction"] = float((labels < 0).mean())
    res["queries"] = {"core": n, "link": int(core.sum()), "border": int(n - core.sum())}
    res["counters_all_passes"] = {
        "nodes_visited_per_point": cs["nodes_visited"] / n, "points_tested_per_point": cs["points_tested"] / n,
        "warp_node_loads": cs["warp_node_visits"], "warp_point_loads": cs["warp_point_loads"],
        "unions_and_border_hits": cs["heap_inserts"]}
    # shared-memory roofline of the traversal kernels, as bench.py's roofline_block bills the search
    alg_bytes = 64 * cs["nodes_visited"] + 16 * cs["points_tested"]
    kt = sum(res["kernel_ms"].values()) * 1e-3
    res["roofline"] = {"bound": "smem", "achieved_gbs": alg_bytes / kt / 1e9, "peak_gbs": smem_peak,
                       "frac": alg_bytes / kt / 1e9 / smem_peak, "kernel_ms": kt * 1e3,
                       "note": "64 B per node visit + 16 B per point test, every query billed for its own reads, over the "
                               "three traversal kernels' median time; peak = tknn_measure_smem_bandwidth conflict-free LDS.128"}
    t0 = time.perf_counter()
    ref_l, ref_c, ref_n = DO.dbscan(x, eps, min_pts)
    cpu_s = time.perf_counter() - t0
    res["verified"] = bool((ref_l == labels).all() and (ref_c == core).all() and ref_n == c)
    res["cpu_reference"] = {"seconds": cpu_s, "threads": DO.num_threads(), "host_cores": os.cpu_count(),
                            "speedup_of_gpu_call": cpu_s / (med * 1e-3)}
    if sk_points:
        from sklearn.cluster import DBSCAN

        m = min(sk_points, n)
        t0 = time.perf_counter()
        DBSCAN(eps=eps, min_samples=min_pts, n_jobs=-1).fit(x[:m].astype(np.float64))
        res["sklearn"] = {"points": m, "seconds": time.perf_counter() - t0, "n_jobs": -1, "host_cores": os.cpu_count()}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    ap.add_argument("--sklearn-points", type=int, default=1_000_000)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    import torch

    from owlraytracing_b200 import TrueKNN

    if not torch.cuda.is_available():
        raise SystemExit("dbscan_bench: no CUDA device (there is no CPU fallback)")
    with TrueKNN(0) as t:
        smem_peak = t.measure_smem_bandwidth()["smem_conflict_free_gbs"]
    out = {"bench": "tknn_dbscan", "device": device_info(torch), "smem_peak_gbs": smem_peak, "steps": args.steps, "workloads": []}
    clouds = {}
    for name in args.workloads.split(","):
        kind, n, seed, eps, min_pts = WORKLOADS[name]
        if (kind, n, seed) not in clouds:
            clouds.clear()
            clouds[(kind, n, seed)] = cloud(kind, n, seed)
        out["workloads"].append(run_workload(name, clouds[(kind, n, seed)], eps, min_pts, args.steps, args.sklearn_points,
                                             smem_peak, torch))
        print(json.dumps(out["workloads"][-1]), file=sys.stderr, flush=True)  # progress
    out["verified"] = all(w["verified"] for w in out["workloads"])
    print(json.dumps(out))


if __name__ == "__main__":
    main()
