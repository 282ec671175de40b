"""Fixed-radius neighbour-list benchmark: tknn_radius_search on the flagship clouds, verified against the CPU reference;
prints one JSON line.

    python tools/radius_bench.py [--steps 5] [--workloads uniform_16,uniform_100,lidar_0.05,long_rows] [--scipy-points 1000000]

Workloads: 10 M uniform points (seed 42) at radii giving about 16 and 100 neighbours per point, 10 M `lidar_like` points
(seed 7) at r = 0.05, and a cloud whose rows reach the long-row (radix-sort) tier: 1 M uniform points (seed 11), a
coincident cluster of 20 000 points and a Gaussian blob of 100 000 points (sigma 0.02), at r = 0.01.
Per workload: the total entry count (printed before the timed calls), per-phase device times (median of --steps calls
after one warm-up call; cloud and outputs live on the device, so no host copy is timed), entries/s and queries/s of the
whole call, the count phase beside tknn_range_count at the same radius, the host wall time of the two-call protocol
(size call, then fill) against one call with a sufficient `out`, the bytes the fill and order phases move over their
device time against the measured HBM read peak (tknn_measure_bandwidth), `verified` (offsets, indices and d2 bits equal
the CPU reference), the CPU reference's own time on all host cores, and scipy's cKDTree.query_ball_point(workers=-1,
return_sorted=True) on the first --scipy-points points.  The GPU's name and power limit are read in the run.
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

# name: (cloud, n, seed, radius)
WORKLOADS = {
    "uniform_16": ("uniform", 10_000_000, 42, 0.00726),
    "uniform_100": ("uniform", 10_000_000, 42, 0.0134),
    "lidar_0.05": ("lidar_like", 10_000_000, 7, 0.05),
    "long_rows": ("long_rows", 1_120_000, 11, 0.01),
}
PHASES = ("count", "fill", "order")
SHORT_MAX = 1024  # radius.cuh: rows longer than this take the radix-sort tier


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

    if kind == "lidar_like":
        return datasets.lidar_like(n, seed=seed)
    if kind == "uniform":
        return datasets.uniform(n, seed=seed)
    rng = np.random.default_rng(seed)
    x = np.concatenate([rng.random((1_000_000, 3)), np.tile([[0.25, 0.25, 0.25]], (20_000, 1)),
                        rng.normal(0.7, 0.02, (100_000, 3))]).astype(np.float32)
    return x[rng.permutation(len(x))]


def run_workload(name, x, r, steps, scipy_points, hbm_peak, torch):
    import radius_oracle as RO
    from owlraytracing_b200 import TrueKNN

    n = int(x.shape[0])
    xd = torch.from_numpy(x).cuda()
    res = {"workload": name, "n": n, "radius": r}
    with TrueKNN(0) as t:
        t.set_option("squared_dist", 1)
        t.build(xd)
        off, idx, d2 = t.radius_search(r)  # warm-up (module load, scratch allocation)
        total = int(off[-1].item())
        print(json.dumps({"workload": name, "total_entries": total}), file=sys.stderr, flush=True)
        phase_ms, kern_ms, call_ms = [], [], []
        out = (off, idx, d2)
        for _ in range(steps):
            off, idx, d2 = t.radius_search(r, out=out)
            st = t.stats()
            phase_ms.append(st["round_ms"][:3])
            kern_ms.append(st["kernel_ms"][:3])
            call_ms.append(st["search_ms"])
        long_rows = st["round_queries"][2]
        # the host protocol: two calls (size, then fill into fresh tensors) against one call with a sufficient out
        two, one = [], []
        for _ in range(steps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            t.radius_search(r)
            torch.cuda.synchronize()
            two.append((time.perf_counter() - t0) * 1e3)
            t0 = time.perf_counter()
            t.radius_search(r, out=out)
            torch.cuda.synchronize()
            one.append((time.perf_counter() - t0) * 1e3)
        rc_ms = []
        for _ in range(steps + 1):
            t.range_count(r)
            rc_ms.append(t.stats()["search_ms"])
        off, idx, d2 = off.cpu().numpy(), idx.cpu().numpy(), d2.cpu().numpy()
    med = float(np.median(call_ms))
    res["total_entries"] = total
    res["entries_per_query"] = total / n
    res["long_rows"] = int(long_rows)
    res["long_row_entries"] = int(np.diff(off)[np.diff(off) > SHORT_MAX].sum())
    res["phase_ms"] = {p: float(np.median([v[i] for v in phase_ms])) for i, p in enumerate(PHASES)}
    res["kernel_ms"] = {p: float(np.median([v[i] for v in kern_ms])) for i, p in enumerate(PHASES)}
    res["call_ms"] = med
    res["call_ms_all"] = call_ms
    res["entries_per_s"] = total / (med * 1e-3)
    res["queries_per_s"] = n / (med * 1e-3)
    res["count_vs_range_count"] = {"count_traversal_ms": res["kernel_ms"]["count"],
                                   "count_phase_ms": res["phase_ms"]["count"],
                                   "range_count_ms": float(np.median(rc_ms[1:]))}
    res["protocol_host_ms"] = {"two_calls": float(np.median(two)), "one_call_with_out": float(np.median(one))}
    # bytes each phase must move: fill writes one 8 B key per entry (reads of the tree and points are cache traffic);
    # order reads every key and writes a 4 B index and a 4 B distance per entry
    fill_b, order_b = 8 * total, 16 * total
    res["bandwidth"] = {
        "hbm_read_peak_gbs": hbm_peak,
        "fill": {"bytes": fill_b, "gbs": fill_b / (res["phase_ms"]["fill"] * 1e-3) / 1e9},
        "order": {"bytes": order_b, "gbs": order_b / (res["phase_ms"]["order"] * 1e-3) / 1e9}}
    for p in ("fill", "order"):
        res["bandwidth"][p]["frac_of_hbm_peak"] = res["bandwidth"][p]["gbs"] / hbm_peak
    t0 = time.perf_counter()
    ref = RO.radius_lists(x, r)
    cpu_s = time.perf_counter() - t0
    res["verified"] = bool((ref[0] == off).all() and (ref[1] == idx).all() and (ref[2].view(np.uint32) == d2.view(np.uint32)).all())
    del ref
    res["cpu_reference"] = {"seconds": cpu_s, "threads": RO.num_threads(), "host_cores": os.cpu_count(),
                            "speedup_of_gpu_call": cpu_s / (med * 1e-3)}
    if scipy_points:
        from scipy.spatial import cKDTree

        m = min(scipy_points, n)
        xs = x[:m].astype(np.float64)
        t0 = time.perf_counter()
        cKDTree(xs).query_ball_point(xs, r, workers=-1, return_sorted=True)
        res["scipy_ckdtree"] = {"points": m, "seconds": time.perf_counter() - t0, "workers": -1, "host_cores": os.cpu_count()}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    ap.add_argument("--scipy-points", type=int, default=1_000_000)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    import torch

    from owlraytracing_b200 import TrueKNN

    if not torch.cuda.is_available():
        raise SystemExit("radius_bench: no CUDA device (there is no CPU fallback)")
    with TrueKNN(0) as t:
        hbm_peak = t.measure_bandwidth()["hbm_read_gbs"]
    out = {"bench": "tknn_radius_search", "device": device_info(torch), "hbm_read_peak_gbs": hbm_peak, "steps": args.steps,
           "workloads": []}
    clouds = {}
    for name in args.workloads.split(","):
        kind, n, seed, r = WORKLOADS[name]
        if (kind, n, seed) not in clouds:
            clouds.clear()
            clouds[(kind, n, seed)] = cloud(kind, n, seed)
        out["workloads"].append(run_workload(name, clouds[(kind, n, seed)], r, args.steps, args.scipy_points, hbm_peak, torch))
        print(json.dumps(out["workloads"][-1]), file=sys.stderr, flush=True)  # progress
    out["verified"] = all(w["verified"] for w in out["workloads"])
    print(json.dumps(out))


if __name__ == "__main__":
    main()
