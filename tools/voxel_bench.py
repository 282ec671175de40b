"""Voxel-grid benchmark: tknn_voxel_grid + tknn_voxel_pool against the plain-torch route (the grid formula,
torch.unique(return_inverse=True), index_add_ + bincount for the mean, scatter_reduce("amax") for the max) on the same
GPU, verified against the CPU reference (tests/voxel_oracle.py); prints one JSON line.

    python tools/voxel_bench.py [--steps 5] [--out FILE]

Workloads:
  (a) 16 LiDAR-like sweeps x 120 000 points (datasets.lidar_like), at two voxel sizes (about 4 and about 36 points per
      voxel), pooling the positions;
  (b) one LiDAR-like cloud of 10 M points, pooling the positions;
  (c) 1 024 uniform clouds x 4 096 points, pooling F = 64 features;
  (d) 10 M uniform points plus one coincident cluster of 1 M points (the long-voxel tail), pooling the positions.
Per workload: the library's time for voxel_grid (clustering: box, ids, sort, labels) and for each voxel_pool (mean and
max), and the torch route's clustering and pooling times, each the median of --steps calls after one warm-up call,
measured with CUDA events around the call, inputs and outputs on the device; then, from one profiled call each of
voxel_grid and voxel_pool(mean), the device time of every kernel (the radix sort's kernels summed as `sort`).  `verified`: raw ids, dense ids and the
pooled bits equal the CPU reference on every point of (a) and (c) and on 4 096 sampled voxels of (b) and (d).  The GPU's
name and power limit are read in the same run.  Writes nothing into the tree (only --out, when given).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

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


def median_ms(torch, fn, steps):
    fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(steps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    return float(np.median(times))


def torch_route(torch, pos, size, batch):
    p = torch.cat([pos, batch.to(pos.dtype).view(-1, 1)], 1) if batch is not None else pos
    sz = torch.full((p.shape[1],), float(size), device=pos.device)
    if batch is not None:
        sz[-1] = 1.0
    s0, e0 = p.min(0).values, p.max(0).values
    cnt = ((e0 - s0) / sz).long() + 1
    mult = torch.cat([torch.ones(1, dtype=torch.long, device=pos.device), torch.cumprod(cnt, 0)[:-1]])
    raw = (((p - s0) / sz).long() * mult).sum(1)
    _, inv = torch.unique(raw, sorted=True, return_inverse=True)
    return raw, inv


def torch_mean(torch, x, inv, nv):
    s = torch.zeros(nv, x.shape[1], dtype=x.dtype, device=x.device).index_add_(0, inv, x)
    return s / torch.bincount(inv, minlength=nv).to(x.dtype).view(-1, 1)


def torch_max(torch, x, inv, nv):
    out = torch.full((nv, x.shape[1]), -float("inf"), dtype=x.dtype, device=x.device)
    return out.scatter_reduce(0, inv.view(-1, 1).expand(-1, x.shape[1]), x, "amax")


def phases_ms(torch, fn):
    """Device time per kernel group of one call, from torch.profiler (a separate, profiled call after the timed ones):
    the sort kernels (rsort::*) as one group, every other kernel by its own name."""
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        us = getattr(e, "device_time_total", None)
        if us is None:
            us = getattr(e, "cuda_time_total", 0.0)
        if not us or "kernel" not in e.key:
            continue
        name = "sort" if "rsort::" in e.key else e.key.split("(")[0].split("<")[0].split("::")[-1]
        out[name] = round(out.get(name, 0.0) + us / 1000.0, 4)
    return out


def workload(torch, t, name, pos, size, sizes, x, steps, sample):
    import voxel_oracle as V

    dev = torch.device("cuda:0")
    pd = torch.from_numpy(pos).to(dev)
    xd = torch.from_numpy(x).to(dev)
    batch = None if sizes is None else torch.repeat_interleave(torch.arange(len(sizes), device=dev),
                                                               torch.as_tensor(sizes, device=dev))
    grid_ms = median_ms(torch, lambda: t.voxel_grid(pd, size, batch=batch, batch_size=None if sizes is None else len(sizes)), steps)
    raw, cluster, nv = t.voxel_grid(pd, size, batch=batch, batch_size=None if sizes is None else len(sizes))
    mean_ms = median_ms(torch, lambda: t.voxel_pool(xd, "mean"), steps)
    max_ms = median_ms(torch, lambda: t.voxel_pool(xd, "max"), steps)
    mean, mx = t.voxel_pool(xd, "mean"), t.voxel_pool(xd, "max")
    grid_phases = phases_ms(torch, lambda: t.voxel_grid(pd, size, batch=batch, batch_size=None if sizes is None else len(sizes)))
    pool_phases = phases_ms(torch, lambda: t.voxel_pool(xd, "mean"))
    t_grid = median_ms(torch, lambda: torch_route(torch, pd, size, batch), steps)
    traw, inv = torch_route(torch, pd, size, batch)
    tnv = int(inv.max()) + 1
    t_mean = median_ms(torch, lambda: torch_mean(torch, xd, inv, tnv), steps)
    t_max = median_ms(torch, lambda: torch_max(torch, xd, inv, tnv), steps)
    ok = bool(torch.equal(raw, traw)) and bool(torch.equal(cluster.long(), inv)) and nv == tnv
    off = None if sizes is None else np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint64)
    g = V.grid(pos, size, off=off)
    ok = ok and bool((raw.cpu().numpy() == g["raw"]).all()) and bool((cluster.cpu().numpy() == g["cluster"]).all())
    if sample and g["n_voxels"] > sample:  # pooled bits on sampled voxels (always including the largest one)
        rng = np.random.default_rng(0)
        cnt = np.diff(g["offsets"].astype(np.int64))
        vs = np.unique(np.concatenate([rng.choice(g["n_voxels"], sample, replace=False), [int(np.argmax(cnt))]]))
        sub_off = np.concatenate([[0], np.cumsum(cnt[vs])]).astype(np.uint64)
        sub_mem = np.concatenate([g["members"][g["offsets"][v]:g["offsets"][v + 1]] for v in vs]).astype(np.int32)
        sg = dict(offsets=sub_off, members=sub_mem, n_voxels=len(vs))
        rows = vs
    else:
        sg, rows = g, slice(None)
    for got, red in ((mean, "mean"), (mx, "max")):
        want = V.pool(x, sg, red)
        ok = ok and bool((got.cpu().numpy()[rows].view(np.uint32) == want.view(np.uint32)).all())
    return {"workload": name, "n": int(pos.shape[0]), "clouds": 1 if sizes is None else len(sizes), "f": int(x.shape[1]),
            "size": float(size), "n_voxels": int(nv), "points_per_voxel": round(pos.shape[0] / max(nv, 1), 2),
            "largest_voxel": int(np.diff(g["offsets"].astype(np.int64)).max()),
            "voxel_grid_ms": round(grid_ms, 4), "pool_mean_ms": round(mean_ms, 4), "pool_max_ms": round(max_ms, 4),
            "torch_grid_unique_ms": round(t_grid, 4), "torch_mean_ms": round(t_mean, 4), "torch_max_ms": round(t_max, 4),
            "voxel_grid_kernels_ms": grid_phases, "pool_mean_kernels_ms": pool_phases, "verified": ok}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch

    from owlraytracing_b200 import TrueKNN, datasets

    rows = []
    with TrueKNN(0) as t:
        sweeps = np.concatenate([datasets.lidar_like(120_000, seed=s) for s in range(16)])[:, :3].copy()
        for size in (1.0, 5.0):
            rows.append(workload(torch, t, f"a_lidar16x120k_s{size}", sweeps, size, [120_000] * 16, sweeps, a.steps, 0))
        big = np.ascontiguousarray(datasets.lidar_like(10_000_000, seed=3)[:, :3])
        rows.append(workload(torch, t, "b_lidar10M", big, 1.0, None, big, a.steps, 4096))
        rng = np.random.default_rng(1)
        u = rng.random((1024 * 4096, 3), dtype=np.float32)
        feats = rng.normal(size=(u.shape[0], 64)).astype(np.float32)
        rows.append(workload(torch, t, "c_uniform1024x4096_f64", u, 0.1, [4096] * 1024, feats, a.steps, 0))
        del feats
        tail = np.concatenate([rng.random((10_000_000, 3), dtype=np.float32),
                               np.repeat(np.float32([[0.5, 0.5, 0.5]]), 1_000_000, 0)])
        rows.append(workload(torch, t, "d_uniform10M_plus_1M_cluster", tail, 0.01, None, tail, a.steps, 4096))
    line = json.dumps({"bench": "voxel", "device": device_info(torch), "steps": a.steps, "workloads": rows})
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
