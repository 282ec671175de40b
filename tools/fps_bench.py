"""Farthest point sampling benchmark: tknn_fps on batches of clouds and on one large cloud, against the same sampling
written in plain torch on the same GPU, verified against the CPU reference (tests/fps_oracle.py); prints one JSON line.

    python tools/fps_bench.py [--steps 5] [--torch-prefix 2000]

Workloads: (a) 1 024 uniform clouds x 4 096 points, ratio 0.25 (block tier); (b) 65 536 uniform clouds x 64, ratio 0.25
(the block tier's CTA sizing); (c) 16 `lidar_like` sweeps of 120 000 points, ratio 1/16 (grid tier, 16 clouds in
lockstep); (d) one uniform cloud of 10 M points, 100 000 samples (grid tier, one cloud).  Per workload: the library's
device time (search_ms, median of --steps calls after one warm-up call; clouds and outputs on the device) and samples/s;
the torch baseline (a padded [B, n_max] tensor, per iteration one `minimum` update and one `argmax`), timed with CUDA
events on the same inputs, over at most --torch-prefix iterations and extrapolated linearly to all of them (marked
`torch_extrapolated`); for (c) and (d) the leaf box tests and leaf updates per sample from a separate counting run.
`verified`: indices and distance bits equal the CPU reference on all clouds of (a) and (c), every 64th cloud of (b) and
the first 1 024 samples of (d).  The GPU's name and power limit are read in the same run.  Writes nothing into the tree.
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


def torch_fps_ms(torch, x, sizes, counts, prefix):
    """Plain-torch FPS over a padded [B, n_max, 3] tensor (padding rows get D = -inf): ms for all iterations, and whether
    that was extrapolated from the first `prefix` iterations."""
    B, nmax, iters = len(sizes), int(max(sizes)), int(max(counts))
    pad = torch.zeros((B, nmax, 3), device="cuda")
    valid = torch.zeros((B, nmax), dtype=torch.bool, device="cuda")
    off = np.concatenate([[0], np.cumsum(sizes)])
    if len(set(sizes)) == 1:
        pad[:] = x.view(B, nmax, 3)
        valid[:] = True
    else:
        for s in range(B):
            pad[s, : sizes[s]] = x[off[s]: off[s + 1]]
            valid[s, : sizes[s]] = True
    rows = torch.arange(B, device="cuda")
    run = min(iters, prefix)

    def once(n_it):
        D = torch.where(valid, torch.full((B, nmax), float("inf"), device="cuda"),
                        torch.full((B, nmax), float("-inf"), device="cuda"))
        cur = torch.zeros(B, dtype=torch.int64, device="cuda")
        out = torch.empty((B, n_it), dtype=torch.int64, device="cuda")
        out[:, 0] = cur
        for i in range(1, n_it):
            c = pad[rows, cur].unsqueeze(1)
            D = torch.minimum(D, ((pad - c) ** 2).sum(-1))
            cur = torch.argmax(D, dim=1)
            out[:, i] = cur
        return out

    once(min(run, 8))
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    ev0.record()
    once(run)
    ev1.record()
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1)
    return ms * (iters - 1) / max(run - 1, 1), run < iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--torch-prefix", type=int, default=2000)
    args = ap.parse_args()

    import torch

    import fps_oracle as F
    from owlraytracing_b200 import TrueKNN, datasets
    from owlraytracing_b200.trueknn import fps_counts

    result = {"bench": "fps", "device": device_info(torch), "steps": args.steps, "workloads": []}
    work = [
        ("a_uniform_1024x4096", "uniform", 1024, 4096, 0.25, None),
        ("b_uniform_65536x64", "uniform", 65536, 64, 0.25, None),
        ("c_lidar_16x120000", "lidar", 16, 120_000, 1.0 / 16, None),
        ("d_uniform_10M", "uniform", 1, 10_000_000, None, 100_000),
    ]
    for name, kind, count, size, ratio, m in work:
        if kind == "uniform":
            x = datasets.uniform(count * size, seed=5)
            sizes = [size] * count
        else:
            parts = [datasets.lidar_like(size, seed=40 + s) for s in range(count)]
            sizes = [p.shape[0] for p in parts]
            x = np.concatenate(parts)
        counts = fps_counts(sizes, ratio) if m is None else np.array([m], np.int64)
        batch = np.repeat(np.arange(count), sizes)
        xt = torch.from_numpy(x).cuda()
        bt = torch.from_numpy(batch).cuda()
        rec = {"workload": name, "clouds": count, "points": int(x.shape[0]), "samples": int(counts.sum())}
        with TrueKNN(0) as t:
            t.set_option("squared_dist", 1)
            if count == 1:
                t.build(xt)
            else:
                t.build(xt, batch=bt)
            idx, dist = t.fps(num_samples=counts, with_dist=True)
            torch.cuda.synchronize()
            ms, tiers = [], None
            for _ in range(args.steps):
                t.fps(num_samples=counts, out=(idx, dist))
                st = t.stats()
                ms.append(st["search_ms"])
                tiers = {"block_ms": st["round_ms"][0], "grid_ms": st["round_ms"][1],
                         "block_kernel_ms": st["kernel_ms"][0], "grid_kernel_ms": st["kernel_ms"][1],
                         "block_samples": int(st["round_queries"][0]), "grid_samples": int(st["round_queries"][1])}
            rec["search_ms"] = float(np.median(ms))
            rec["search_ms_all"] = [round(v, 4) for v in ms]
            rec["samples_per_s"] = rec["samples"] / (rec["search_ms"] * 1e-3)
            rec.update(tiers)
            if tiers["grid_samples"]:
                t.set_option("counters", 1)
                ci, _ = t.fps(num_samples=counts, with_dist=True)
                st = t.stats()
                t.set_option("counters", 0)
                rec["same_samples_counting"] = bool(torch.equal(ci, idx))
                rec["leaf_box_tests_per_sample"] = st["nodes_visited"] / rec["samples"]
                rec["leaf_updates_per_sample"] = st["warp_leaf_visits"] / rec["samples"]
                rec["point_updates_per_sample"] = st["points_tested"] / rec["samples"]
                rec["leaves"] = int(st["n_leaves"])
            gi, gd = idx.cpu().numpy(), dist.cpu().numpy()
        off = F.offsets_of(sizes)
        so = F.offsets_of(counts).astype(np.int64)
        if name.startswith("b_"):
            ok = True
            for s in range(0, count, 64):
                wi, wd = F.fps(x[off[s]:off[s + 1]], None, [counts[s]])
                ok &= bool((gi[so[s]:so[s + 1]] == wi + int(off[s])).all()
                           and (gd[so[s]:so[s + 1]].view(np.uint32) == wd.view(np.uint32)).all())
            rec["verified"], rec["verified_scope"] = ok, "every 64th cloud"
        else:
            limit = 1024 if name.startswith("d_") else None
            wi, wd = F.fps(x, off, counts, limit=limit)
            mask = np.ones(gi.shape[0], bool) if limit is None else F.prefix_mask(counts, limit)
            rec["verified"] = bool((gi[mask] == wi[mask]).all() and (gd[mask].view(np.uint32) == wd[mask].view(np.uint32)).all())
            rec["verified_scope"] = "all clouds" if limit is None else f"first {limit} samples"
        tms, extrap = torch_fps_ms(torch, xt, sizes, counts, args.torch_prefix)
        rec["torch_ms"] = tms
        rec["torch_extrapolated"] = extrap
        rec["speedup_vs_torch"] = tms / rec["search_ms"]
        result["workloads"].append(rec)
        del xt, bt
        torch.cuda.empty_cache()
        print(json.dumps(rec), file=sys.stderr, flush=True)
    result["all_verified"] = all(r["verified"] for r in result["workloads"])
    print(json.dumps(result))


if __name__ == "__main__":
    main()
