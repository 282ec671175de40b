"""Segmented-build benchmark: batches of point clouds through tknn_build_segments + tknn_search (and tknn_radius_search),
verified against the per-segment CPU reference (tests/segment_oracle.py); prints one JSON line.

    python tools/segments_bench.py [--steps 5] [--loop-subset 1024]

Workloads (the batch sizes torch_cluster users run): 1 024 uniform clouds of 4 096 points (k = 16, and radius_graph at
r = 0.123, about 32 neighbours per point), 65 536 uniform clouds of 64 points (k = 16), 16 `lidar_like` sweeps of
120 000 points (k = 16 and k = 64).  Per workload: build ms and search ms (device events of the library, median of
--steps calls after one warm-up call; cloud and outputs on the device), points/s of build + search, and the same clouds
through a per-cloud loop of build + search on one context (host wall time with a device synchronise; the 65 536-cloud
loop times its first --loop-subset clouds and extrapolates).  Reference cost: one unsegmented search of the 4.2 M points
of the first workload at k = 16.  `verified`: indices and distance bits equal the CPU reference.  The GPU's name and
power limit are read in the same run.  Writes nothing into the tree.
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


def device_info(torch):
    info = {"name": torch.cuda.get_device_name(0), "power_limit_w": None}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_w"] = float(out.splitlines()[0])
    except Exception as e:  # noqa: BLE001 — reported, not hidden
        info["power_limit_w_error"] = repr(e)
    return info


def clouds(kind, count, size, seed):
    from owlraytracing_b200 import datasets

    if kind == "uniform":
        return datasets.uniform(count * size, seed=seed)  # consecutive slices: independent unit-cube clouds
    return np.concatenate([datasets.lidar_like(size, seed=seed + s) for s in range(count)])


def median(v):
    return float(np.median(np.asarray(v, np.float64)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--loop-subset", type=int, default=1024)
    args = ap.parse_args()

    import torch

    import segment_oracle as SO
    from owlraytracing_b200 import TrueKNN

    if not torch.cuda.is_available():
        raise SystemExit("segments_bench needs a CUDA device")
    res = {"bench": "segments", "device": device_info(torch), "steps": args.steps, "workloads": []}
    t = TrueKNN(0)
    t.set_option("squared_dist", 1)

    def timed(fn):
        fn()
        torch.cuda.synchronize()
        runs = []
        for _ in range(args.steps):
            fn()
            torch.cuda.synchronize()
            runs.append(t.stats())
        return runs

    work = [("uniform_1024x4096", "uniform", 1024, 4096, 11, [16], 0.123),
            ("uniform_65536x64", "uniform", 65536, 64, 12, [16], None),
            ("lidar_16x120000", "lidar_like", 16, 120_000, 7, [16, 64], None)]
    for name, kind, count, size, seed, ks, radius in work:
        x = clouds(kind, count, size, seed)
        n = len(x)
        off = SO.offsets_of([size] * count)
        xt = torch.from_numpy(x).cuda()
        bt = torch.from_numpy(np.repeat(np.arange(count), size)).cuda()
        builds = timed(lambda: t.build(xt, batch=bt))
        w = {"workload": name, "clouds": count, "points_per_cloud": size, "n": n,
             "build_ms": median([s["build_ms"] for s in builds])}
        for k in ks:
            t.build(xt, batch=bt)
            idx, d2 = t.search(k)
            wi, wd = SO.knn(x, off, k, squared=True)
            ok = bool((idx.cpu().numpy() == wi).all() and (d2.cpu().numpy().view(np.uint32) == wd.view(np.uint32)).all())
            runs = timed(lambda: t.search(k))
            search_ms = median([s["search_ms"] for s in runs])
            # per-cloud loop on one context: build + search of every cloud, host wall time with a device synchronise
            m = min(count, args.loop_subset)
            xs = [xt[c * size:(c + 1) * size] for c in range(m)]
            t.build(xs[0]).search(k)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for c in range(m):
                t.build(xs[c]).search(k)
            torch.cuda.synchronize()
            loop_ms = (time.perf_counter() - t0) * 1e3 * count / m
            w[f"k{k}"] = {"search_ms": search_ms, "rounds": runs[-1]["rounds"],
                          "points_per_s": n / ((w["build_ms"] + search_ms) * 1e-3),
                          "loop_ms": loop_ms, "loop_clouds_timed": m, "loop_extrapolated": m < count,
                          "speedup_vs_loop": loop_ms / (w["build_ms"] + search_ms), "verified": ok}
        if radius is not None:
            t.build(xt, batch=bt)
            o, i, d = t.radius_search(radius)
            wo, wi, wd = SO.radius_lists(x, off, radius)
            ok = bool((o.cpu().numpy() == wo).all() and (i.cpu().numpy() == wi).all() and
                      (d.cpu().numpy().view(np.uint32) == wd.view(np.uint32)).all())
            runs = timed(lambda: t.radius_search(radius))
            w["radius_graph"] = {"r": radius, "mean_neighbours": float(wo[-1]) / n,
                                 "search_ms": median([s["search_ms"] for s in runs]), "verified": ok}
        res["workloads"].append(w)
        if name == "uniform_1024x4096":  # reference: the same 4.2 M points as ONE cloud, unsegmented
            t.build(xt)
            runs = timed(lambda: t.search(16))
            res["reference_unsegmented"] = {"n": n, "k": 16, "build_ms": median([s["build_ms"] for s in timed(lambda: t.build(xt))]),
                                            "search_ms": median([s["search_ms"] for s in runs])}
    t.close()
    res["verified"] = all(w[key]["verified"] for w in res["workloads"] for key in w if key.startswith("k") or key == "radius_graph")
    print(json.dumps(res))


if __name__ == "__main__":
    main()
