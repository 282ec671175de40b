"""Chamfer distance benchmark: chamfer_distance forward (two builds, two k = 1 queries, the reductions) and backward
(autograd through tknn_knn_backward and the reductions' gathers), the knn_backward phases, beside a plain-torch Chamfer
(torch.cdist, min, mean, autograd) and the atomic index_add_ backward on the same idx; verified against the CPU reference
(tests/chamfer_oracle.py); prints one JSON line.

    python tools/chamfer_bench.py [--steps 5] [--out FILE]

Workloads (x -> y, the default reductions: point mean, batch mean):
  (a) 32 clouds x 16 384 / 16 384 points (point-cloud completion scale);
  (b) 256 clouds x 2 048 / 2 048;
  (c) 8 LiDAR-like sweeps x 120 000 / 30 000 (y every fourth point of another sweep);
  (d) one cloud of 2^20 points against one point: every nearest point of direction x -> y is that point, so its
      gradient is one run of 2^20 edges (the long-run chunk path).
Per workload: the device time of the forward and of loss.backward(), each the median of --steps calls after one warm-up
call, measured with CUDA events around the call on torch's stream, inputs on the device; the three phases of
tknn_knn_backward (terms and edge keys, sort, run offsets and chunked sums) from the library's statistics for both
directions on the forward's (idx, grad_d2); the bytes those phases must move (from the shapes) and their share of the HBM
bandwidth the library measures in the same run; the torch body (cdist per cloud, forward + backward) and the atomic
index_add_ backward of both directions on the same idx.  `verified`: per-cloud losses, x.grad and y.grad equal the CPU
reference bit for bit on 4 sampled clouds (every cloud of (d)).  The GPU's name and power limit are read in the same
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


def device_info(torch):
    info = {"name": torch.cuda.get_device_name(0), "power_limit_w": None}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_w"] = float(out.splitlines()[0])
    except Exception as e:  # noqa: BLE001 — reported, not hidden
        info["power_limit_w_error"] = repr(e)
    return info


def timed(torch, fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def median_ms(torch, fn, steps, setup=None):
    """Median device time of fn over `steps` calls after a warm-up; setup (untimed) runs before every call."""
    times = []
    for s in range(steps + 1):
        arg = setup() if setup else None
        torch.cuda.synchronize()
        ms = timed(torch, (lambda: fn(arg)) if setup else fn)
        if s:
            times.append(ms)
    return float(np.median(times))


def workload(name, rng):
    """(x, y, x_sizes, y_sizes) as numpy."""
    from owlraytracing_b200 import datasets

    if name.startswith("a_"):
        xs = ys = [16_384] * 32
    elif name.startswith("b_"):
        xs = ys = [2048] * 256
    elif name.startswith("c_"):
        sweeps = [datasets.lidar_like(120_000, seed=s).astype(np.float32) for s in range(9)]
        return np.concatenate(sweeps[:8]), np.concatenate([s[::4] for s in sweeps[1:]]), [120_000] * 8, [30_000] * 8
    else:
        return rng.random((1 << 20, 3), dtype=np.float32), np.float32([[0.5, 0.5, 0.5]]), [1 << 20], [1]
    return rng.random((sum(xs), 3), dtype=np.float32), rng.random((sum(ys), 3), dtype=np.float32), xs, ys


def knn_backward_bytes(nq, n, k, dim, edges_p):
    """Bytes the three phases must move: terms (q, idx, grad_d2, the gathered p rows, grad_q, term_p) and edge keys
    (idx, keys, values, counts); the sort (about 24 B per edge and pass); offsets (counts, offsets, chunk layout) and
    chunked sums (values, term_p rows, offsets, grad_p)."""
    E = nq * k
    terms = nq * dim * 4 + E * 8 + E * dim * 4 + nq * dim * 4 + E * dim * 4 + E * 16 + n * 4
    passes = (int(n).bit_length() + 7) // 8
    sort = E * 8 + passes * E * 24
    sums = n * 4 + (n + 1) * 8 * 3 + n * 4 + edges_p * 4 + edges_p * dim * 4 + n * dim * 4
    return {"terms_edges": terms, "sort": sort, "offsets_sums": sums, "total": terms + sort + sums}


def run(torch, name, steps, hbm_gbs, rng):
    import chamfer_oracle as R
    from owlraytracing_b200 import TrueKNN, chamfer_distance, knn_points

    xn, yn, xs, ys = workload(name, rng)
    x0, y0 = torch.from_numpy(xn).cuda(), torch.from_numpy(yn).cuda()
    bx = torch.repeat_interleave(torch.arange(len(xs), device="cuda"), torch.tensor(xs, device="cuda"))
    by = torch.repeat_interleave(torch.arange(len(ys), device="cuda"), torch.tensor(ys, device="cuda"))
    res = {"clouds": len(xs), "nx": len(xn), "ny": len(yn)}

    def leaves():
        return x0.clone().requires_grad_(True), y0.clone().requires_grad_(True)

    def forward(xy):
        return chamfer_distance(xy[0], xy[1], bx, by)

    res["forward_ms"] = median_ms(torch, forward, steps, setup=leaves)
    res["backward_ms"] = median_ms(torch, lambda loss: loss.backward(), steps, setup=lambda: forward(leaves()))

    # the knn_backward phases of both directions on the forward's (idx, grad_d2): the gradient of mean-of-means
    phases, nbytes = {}, {}
    B = len(xs)
    for d, (q, p, bq, bp, sizes) in {"x_to_y": (x0, y0, bx, by, xs), "y_to_x": (y0, x0, by, bx, ys)}.items():
        _, idx = knn_points(p, q, 1, bp, bq)
        cnt = torch.tensor(sizes, device="cuda", dtype=torch.float32)
        g = ((torch.ones(B, device="cuda") / B) / cnt).repeat_interleave(torch.tensor(sizes, device="cuda"))
        g = g.reshape(-1, 1).contiguous()
        idx32 = idx.to(torch.int32)
        stats = []
        with TrueKNN(0) as t:
            t.set_stream(torch.cuda.current_stream().cuda_stream)

            def call():
                t.knn_backward(q, p, idx32, g)
                s = t.stats()
                stats.append(s["round_ms"])

            ms = median_ms(torch, call, steps)
        rm = np.median(np.array(stats[1:]), 0)
        nb = knn_backward_bytes(len(q), len(p), 1, 3, len(q))
        phases[d] = {"knn_backward_ms": ms, "terms_edges_ms": float(rm[0]), "sort_ms": float(rm[1]),
                     "offsets_sums_ms": float(rm[2]), "hbm_share": nb["total"] / (ms * 1e-3) / (hbm_gbs * 1e9)}
        nbytes[d] = nb
    res["knn_backward"] = phases
    res["knn_backward_bytes"] = nbytes

    # plain torch: cdist per cloud, min, mean of the per-cloud means; forward + backward (atomics in the scatter)
    xo, yo = np.concatenate([[0], np.cumsum(xs)]), np.concatenate([[0], np.cumsum(ys)])

    def torch_body(xy):
        xr, yr = xy
        for c in range(B):  # one backward per cloud keeps one distance matrix alive at a time
            dd = torch.cdist(xr[xo[c]:xo[c + 1]], yr[yo[c]:yo[c + 1]]) ** 2
            ((dd.min(1).values.mean() + dd.min(0).values.mean()) / B).backward()

    res["torch_cdist_fwd_bwd_ms"] = median_ms(torch, torch_body, steps, setup=leaves)

    # the atomic backward on the same idx: term = 2 g (q - p[j]), index_add_ into both sides
    _, ia = knn_points(y0, x0, 1, by, bx)
    _, ib = knn_points(x0, y0, 1, bx, by)
    ga = ((torch.ones(B, device="cuda") / B) / torch.tensor(xs, device="cuda", dtype=torch.float32)).repeat_interleave(
        torch.tensor(xs, device="cuda"))
    gb = ((torch.ones(B, device="cuda") / B) / torch.tensor(ys, device="cuda", dtype=torch.float32)).repeat_interleave(
        torch.tensor(ys, device="cuda"))

    def atomic_backward():
        gx = torch.zeros_like(x0)
        gy = torch.zeros_like(y0)
        ta = 2 * ga[:, None] * (x0 - y0[ia[:, 0]])
        gx += ta
        gy.index_add_(0, ia[:, 0], -ta)
        tb = 2 * gb[:, None] * (y0 - x0[ib[:, 0]])
        gy += tb
        gx.index_add_(0, ib[:, 0], -tb)

    res["torch_index_add_backward_ms"] = median_ms(torch, atomic_backward, steps)

    # verified: per-cloud losses and gradients against the reference on sampled clouds
    x, y = leaves()
    per = chamfer_distance(x, y, bx, by, batch_reduction=None)
    w = torch.from_numpy(rng.normal(size=B).astype(np.float32)).cuda()
    (per * w).sum().backward()
    clouds = range(B) if B <= 4 else [0, 1, B // 2, B - 1]
    ok = True
    same = lambda a, b: bool((np.asarray(a, np.float32).view(np.uint32) == np.asarray(b, np.float32).view(np.uint32)).all())
    for c in clouds:
        xc, yc = xn[xo[c]:xo[c + 1]], yn[yo[c]:yo[c + 1]]
        loss, gx, gy = R.chamfer(xc, yc, [len(xc)], [len(yc)], "mean", None, grad=w[c:c + 1].cpu().numpy())
        ok &= same(per[c:c + 1].detach().cpu().numpy(), loss)
        ok &= same(x.grad[xo[c]:xo[c + 1]].cpu().numpy(), gx) and same(y.grad[yo[c]:yo[c + 1]].cpu().numpy(), gy)
    res["verified"] = ok
    res["verified_clouds"] = len(list(clouds))
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
        raise SystemExit("chamfer_bench: no CUDA device (nothing is measured on the CPU)")
    with TrueKNN(0) as t:
        bw = t.measure_bandwidth()
    rng = np.random.default_rng(0)
    names = ["a_32x16384_16384", "b_256x2048_2048", "c_lidar_8x120000_30000", "d_one_cloud_2pow20_1"]
    res = {"bench": "chamfer", "device": device_info(torch), "hbm_read_gbs_measured": bw["hbm_read_gbs"],
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
