"""k-NN interpolation benchmark: the kNN query, tknn_interpolate and tknn_interpolate_backward beside PyG's
knn_interpolate body in plain torch (index_select, mul, index_add_, forward + backward) on the same (idx, d2), verified
against the CPU reference (tests/interpolate_oracle.py); prints one JSON line.

    python tools/interpolate_bench.py [--steps 5] [--out FILE]

Workloads (PointNet++ feature propagation, k = 3):
  (a) 1 024 uniform clouds x 1 024 coarse -> 4 096 fine points, F = 128 (the interpolation query of DESIGN.md §3.6, now
      with features);
  (b) 32 clouds x 128 coarse -> 2 048 fine, F = 512 (a ShapeNet-sized FP layer);
  (c) 16 LiDAR-like sweeps x 30 000 coarse -> 120 000 fine, F = 64;
  (d) one coarse point referenced by 2^20 queries, F = 128: the cost of one serial run in the backward pass.
Per workload: the device time of the kNN query, the forward and the backward (with the backward's three phases from the
library's statistics), each the median of --steps calls after one warm-up call, measured with CUDA events around the
call on the stream the context runs on, inputs and outputs on the device; the bytes each pass must move (from the
shapes) and their share of the HBM bandwidth the library measures in the same run; the host wall time of
knn_interpolate forward + backward including context creation; and the torch body's forward + backward.  `verified`:
the kNN rows, out, weight, den and grad_x equal the CPU reference bit for bit on every cloud of (b), (c) and (d) and
on 4 sampled clouds of (a).  The GPU's name and power limit are read in the same run.  Writes nothing into the tree
(only --out, when given).
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


def workload(name, rng):
    """(pos_x, pos_y, x_sizes, y_sizes, f) as numpy."""
    from owlraytracing_b200 import datasets

    if name == "a_1024x1024_to_4096_f128":
        xs, ys, f = [1024] * 1024, [4096] * 1024, 128
        return rng.random((sum(xs), 3), dtype=np.float32), rng.random((sum(ys), 3), dtype=np.float32), xs, ys, f
    if name == "b_32x128_to_2048_f512":
        xs, ys, f = [128] * 32, [2048] * 32, 512
        return rng.random((sum(xs), 3), dtype=np.float32), rng.random((sum(ys), 3), dtype=np.float32), xs, ys, f
    if name == "c_lidar_16x30000_to_120000_f64":
        xs, ys, f = [30_000] * 16, [120_000] * 16, 64
        fine = np.concatenate([datasets.lidar_like(120_000, seed=s) for s in range(16)]).astype(np.float32)
        coarse = np.concatenate([fine[s * 120_000:(s + 1) * 120_000][::4] for s in range(16)])
        return coarse, fine, xs, ys, f
    xs, ys, f = [1], [1 << 20], 128
    return np.float32([[0.5, 0.5, 0.5]]), rng.random((1 << 20, 3), dtype=np.float32), xs, ys, f


def verify(I, idx, d2, x, g, out, w, den, gx, pos_x, pos_y, xs, ys, clouds):
    xo, yo = np.concatenate([[0], np.cumsum(xs)]), np.concatenate([[0], np.cumsum(ys)])
    ok = True
    for c in clouds:
        a, b, q0, q1 = int(xo[c]), int(xo[c + 1]), int(yo[c]), int(yo[c + 1])
        k = idx.shape[1]
        ri, rd = I.knn_rows(pos_x[a:b], pos_y[q0:q1], k)
        li = idx[q0:q1].cpu().numpy()
        li = np.where(li >= 0, li - a, -1).astype(np.int32)
        ld = d2[q0:q1].cpu().numpy()
        ok &= bool((li == ri).all()) and bool((np.where(ri >= 0, ld, 0) == np.where(ri >= 0, rd, 0)).all())
        xc, gc = x[a:b].cpu().numpy(), g[q0:q1].cpu().numpy()
        r_out, r_w, r_den = I.forward(li, ld, xc)
        canon = lambda a: np.where(np.isnan(a), np.float32(np.nan), a).view(np.uint32)  # NaN sign / payload aside
        same = lambda t, r: bool((canon(t.cpu().numpy()) == canon(r)).all())
        ok &= same(out[q0:q1], r_out) and same(w[q0:q1], r_w) and same(den[q0:q1], r_den)
        ok &= same(gx[a:b], I.backward(li, r_w, r_den, gc, b - a))
    return ok


def run(torch, name, steps, hbm_gbs, rng):
    import interpolate_oracle as I
    from owlraytracing_b200 import TrueKNN, knn_interpolate

    pos_x, pos_y, xs, ys, f = workload(name, rng)
    k = min(3, min(s for s in xs if s) if xs else 3)
    n, nq = len(pos_x), len(pos_y)
    px, py = torch.from_numpy(pos_x).cuda(), torch.from_numpy(pos_y).cuda()
    bx = torch.repeat_interleave(torch.arange(len(xs), device="cuda"), torch.tensor(xs, device="cuda"))
    by = torch.repeat_interleave(torch.arange(len(ys), device="cuda"), torch.tensor(ys, device="cuda"))
    x = torch.randn((n, f), device="cuda")
    g = torch.randn((nq, f), device="cuda")
    res = {"n": n, "nq": nq, "f": f, "k": k, "clouds": len(xs)}
    with TrueKNN(0, squared_dist=1) as t:
        t.set_stream(torch.cuda.current_stream().cuda_stream)
        if n > 1:
            t.build(px, batch=bx)
            search = lambda: t.query(py, k, batch=by)
        else:  # one coarse point: knn_interpolate takes its rows from the feature-space search (a build needs two)
            search = lambda: t.feature_knn(px, py, k, batch_x=bx, batch_y=by)
        idx, d2 = search()
        res["query_ms"] = median_ms(torch, search, steps)
        out, w, den = t.interpolate(idx, d2, x)
        res["forward_ms"] = median_ms(torch, lambda: t.interpolate(idx, d2, x), steps)
        gx = t.interpolate_backward(idx, w, den, g, n)
        phases = []

        def bwd():
            t.interpolate_backward(idx, w, den, g, n)
            s = t.stats()
            phases.append((s["round_ms"], s["kernel_ms"]))

        res["backward_ms"] = median_ms(torch, bwd, steps)
        rm = np.median(np.array([p[0] for p in phases]), 0)
        km = np.median(np.array([p[1] for p in phases]), 0)
        res["backward_phase_ms"] = {"edges_counts": float(rm[0]), "sort": float(rm[1]), "offsets_colsums": float(rm[2])}
        res["backward_kernel_ms"] = {"edge_kernel": float(km[0]), "sort": float(km[1]), "colsum_kernel": float(km[2])}
    E = nq * k
    fwd_bytes = E * 8 + E * f * 4 + nq * f * 4 + E * 4 + nq * 4
    passes = (int(n).bit_length() + 7) // 8
    sort_bytes = E * 8 + passes * E * 24
    col_bytes = E * 12 + E * f * 4 + n * f * 4 + (n + 1) * 8
    bwd_bytes = E * 4 + E * 12 + n * 4 + sort_bytes + col_bytes
    res["bytes"] = {"forward": fwd_bytes, "backward": bwd_bytes, "backward_colsum": col_bytes}
    res["hbm_share"] = {"forward": fwd_bytes / (res["forward_ms"] * 1e-3) / (hbm_gbs * 1e9),
                        "backward": bwd_bytes / (res["backward_ms"] * 1e-3) / (hbm_gbs * 1e9)}

    # host wall time of knn_interpolate forward + backward, context creation included
    xr = x.clone().requires_grad_(True)

    def e2e():
        xr.grad = None
        o = knn_interpolate(xr, px, py, bx, by, k=3)
        (o * g).sum().backward()
        torch.cuda.synchronize()

    e2e()
    walls = []
    for _ in range(steps):
        t0 = time.perf_counter()
        e2e()
        walls.append((time.perf_counter() - t0) * 1e3)
    res["knn_interpolate_fwd_bwd_wall_ms"] = float(np.median(walls))

    # PyG's body in torch on the same (idx, d2): index_select, mul, index_add_; forward + backward
    keep = idx.reshape(-1) >= 0
    y_idx = torch.arange(nq, device="cuda").repeat_interleave(k)[keep]
    x_idx = idx.reshape(-1).long()[keep]
    wts = (1.0 / torch.clamp(d2.reshape(-1)[keep], min=1e-16)).view(-1, 1)
    xt = x.clone().requires_grad_(True)

    def body():
        xt.grad = None
        num = torch.zeros((nq, f), device="cuda").index_add_(0, y_idx, xt.index_select(0, x_idx) * wts)
        o = num / torch.zeros((nq, 1), device="cuda").index_add_(0, y_idx, wts)
        (o * g).sum().backward()

    res["torch_body_fwd_bwd_ms"] = median_ms(torch, body, steps)
    res["ours_fwd_bwd_ms"] = res["forward_ms"] + res["backward_ms"]
    body()
    res["torch_grad_max_abs_diff"] = float((xt.grad - gx).abs().max())
    clouds = range(len(xs)) if len(xs) <= 32 else [0, 1, len(xs) // 2, len(xs) - 1]
    res["verified"] = verify(I, idx, d2, x, g, out, w, den, gx, pos_x, pos_y, xs, ys, clouds)
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
        raise SystemExit("interpolate_bench: no CUDA device (nothing is measured on the CPU)")
    with TrueKNN(0) as t:
        bw = t.measure_bandwidth()
    rng = np.random.default_rng(0)
    names = ["a_1024x1024_to_4096_f128", "b_32x128_to_2048_f512", "c_lidar_16x30000_to_120000_f64",
             "d_hot_point_2pow20_f128"]
    res = {"bench": "interpolate", "device": device_info(torch), "hbm_read_gbs_measured": bw["hbm_read_gbs"], "steps": args.steps,
           "workloads": {}}
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
