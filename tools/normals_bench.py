"""Surface normals benchmark: the kNN search and tknn_local_frames of estimate_pointcloud_normals' pipeline, beside a
plain-torch body on the same rows (gather, covariance by einsum, torch.linalg.eigh); verified against the CPU reference
(tests/frames_oracle.py); prints one JSON line.

    python tools/normals_bench.py [--steps 5] [--out FILE]

Workloads (neighbourhood = the point itself and its k - 1 nearest others, disambiguated as PyTorch3D does):
  (a) 10 M LiDAR-like points, k = 16;
  (b) 64 clouds x 16 384 uniform points, k = 50 (PyTorch3D's default neighborhood_size);
  (c) 1 M uniform points, k = 50.
Per workload, inputs on the device: the search (build excluded) as the library's search_ms, and the frames kernel's
device time (kernel_ms of tknn_local_frames), each the median of --steps calls after one warm-up call; the bytes the
kernel must move at least (idx once, each row's positions gathered once, the outputs), the bytes its three passes gather
(idx and 12 B per slot and pass), and the first's share of the HBM bandwidth the library measures in the same run;
estimate_pointcloud_normals end to end (CUDA events around the call); the torch body on the same rows (median, events;
in slices of the largest power of two up to 2^20 rows that torch.linalg.eigh accepts: cuSOLVER's batched eigensolver
refuses a batch of 2^20 matrices).
`verified`: 4 096 sampled rows equal the CPU reference bit for bit.  The GPU's name and power limit are read in the same
run.  Writes nothing into the tree (only --out, when given).
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

TORCH_ROWS = 1 << 20  # first try at rows per torch.linalg.eigh call: cuSOLVER's batched eigensolver refuses large batches


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
    """Median device time of fn (CUDA events around the call) over `steps` calls after a warm-up."""
    times = []
    for s in range(steps + 1):
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        if s:
            times.append(a.elapsed_time(b))
    return float(np.median(times))


def workload(name):
    """(points [n, 3] float32 numpy, cloud sizes, k)."""
    from owlraytracing_b200 import datasets

    if name.startswith("a_"):
        return datasets.lidar_like(10_000_000, seed=7), [10_000_000], 16
    if name.startswith("b_"):
        return datasets.uniform(64 * 16_384, seed=11), [16_384] * 64, 50
    return datasets.uniform(1_000_000, seed=12), [1_000_000], 50


def frames_bytes(m, n, k):
    """Least bytes: idx once (4 B per slot), every point's position once (12 B), eigvals and frames (48 B per row).
    Gathered: idx and a 12-byte position per slot, in each of the three passes (L1 / L2 serve the repeats)."""
    least = m * k * 4 + n * 12 + m * 48
    return {"least": least, "gathered": 3 * m * k * 16 + m * 48}


def run(torch, name, steps, hbm_gbs, rng):
    import frames_oracle as F
    from owlraytracing_b200 import TrueKNN, estimate_pointcloud_normals

    xn, sizes, k = workload(name)
    n = len(xn)
    x = torch.from_numpy(xn).cuda()
    batch = torch.repeat_interleave(torch.arange(len(sizes), device="cuda"), torch.tensor(sizes, device="cuda"))
    batch = None if len(sizes) == 1 else batch
    res = {"n": n, "clouds": len(sizes), "k": k}
    with TrueKNN(0) as t:
        t.set_stream(torch.cuda.current_stream().cuda_stream)
        t.build(x, batch=batch)
        search, frames = [], []
        nbr = None

        def do_search():
            nonlocal nbr
            nbr, _ = t.search(k - 1, indices_only=True)
            search.append(t.stats()["search_ms"])

        median_ms(torch, do_search, steps)
        rows = torch.cat([torch.arange(n, device="cuda", dtype=torch.int32)[:, None], nbr], 1).contiguous()
        out = None

        def do_frames():
            nonlocal out
            out = t.local_frames(x, rows, disambiguate=True)
            frames.append(t.stats()["kernel_ms"][0])

        res["local_frames_call_ms"] = median_ms(torch, do_frames, steps)
    res["search_ms"] = float(np.median(search[1:]))
    res["frames_kernel_ms"] = kernel = float(np.median(frames[1:]))
    nb = frames_bytes(n, n, k)
    res["frames_bytes"] = nb
    res["frames_hbm_share"] = nb["least"] / (kernel * 1e-3) / (hbm_gbs * 1e9)
    res["frames_gathered_gbs"] = nb["gathered"] / (kernel * 1e-3) / 1e9
    res["normals_end_to_end_ms"] = median_ms(torch, lambda: estimate_pointcloud_normals(x, k, batch), steps)

    slice_rows = TORCH_ROWS

    def torch_body():  # PyTorch3D's body on the same rows: gather, mean, covariance by einsum, eigh
        for s in range(0, n, slice_rows):
            nbh = x[rows[s:s + slice_rows].long()]
            d = nbh - nbh.mean(1, keepdim=True)
            torch.linalg.eigh(torch.einsum("mki,mkj->mij", d, d) / k)

    while True:  # the largest power-of-two slice cuSOLVER's batched eigensolver accepts
        try:
            torch_body()
            break
        except torch.linalg.LinAlgError:
            slice_rows //= 2
    res["torch_body_ms"] = median_ms(torch, torch_body, steps)
    res["torch_body_rows_per_eigh"] = slice_rows
    torch.cuda.empty_cache()

    sample = np.sort(rng.choice(n, 4096, replace=False))
    srows = rows[torch.from_numpy(sample).cuda()].cpu().numpy()
    reig, rfr = F.local_frames(xn, srows, True)
    eig, fr = out[0][torch.from_numpy(sample).cuda()].cpu().numpy(), out[1][torch.from_numpy(sample).cuda()].cpu().numpy()
    same = lambda a, b: bool((np.asarray(a, np.float32).view(np.uint32) == np.asarray(b, np.float32).view(np.uint32)).all())
    res["verified"] = same(eig, reig) and same(fr, rfr)
    res["verified_rows"] = len(sample)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch

    from oracle import oracle as O
    from owlraytracing_b200 import TrueKNN

    O.build()
    if not torch.cuda.is_available():
        raise SystemExit("normals_bench: no CUDA device (nothing is measured on the CPU)")
    with TrueKNN(0) as t:
        bw = t.measure_bandwidth()
    rng = np.random.default_rng(0)
    names = ["a_lidar_10M_k16", "b_64x16384_k50", "c_uniform_1M_k50"]
    res = {"bench": "normals", "device": device_info(torch), "hbm_read_gbs_measured": bw["hbm_read_gbs"],
           "steps": args.steps, "workloads": {}}
    for name in names:
        res["workloads"][name] = run(torch, name, args.steps, bw["hbm_read_gbs"], rng)
        torch.cuda.empty_cache()
    res["verified"] = all(w["verified"] for w in res["workloads"].values())
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
