"""Feature-space kNN benchmark: tknn_feature_knn on DGCNN-sized batches and on one large cloud, against the plain-torch
kNN DGCNN implementations use (a padded batch through torch.cdist + topk) on the same GPU, verified against the CPU
reference (tests/feature_knn_oracle.py); prints one JSON line.

    python tools/feature_knn_bench.py [--steps 5] [--out FILE]

Workloads:
  (a) one DGCNN layer: 32 clouds x 1 024 points, F = 64, k = 20, feature_knn(x, x, ...) (no self exclusion);
  (b) 16 clouds x 2 048 points, F = 128, k = 20, the same form;
  (c) 8 clouds x 4 096 points, F = 3, k = 20, against the LBVH segmented query (build(batch) + query(batch)) on the
      same clouds, whose results must be equal bit for bit;
  (d) one cloud of 65 536 data rows and 4 096 separate queries, F = 32, k = 16: the split + merge path.
(a) and (b) are L2-resident on purpose (8 MB and 16 MB of features): that is the working set of a real DGCNN layer,
which rebuilds its graph from activations that were just written.
Per workload: the library's device time (search_ms: first launch to last result on the device, median of --steps calls
after one warm-up call; inputs and outputs on the device), pair-dims/s (sum_s nq_s * n_s * F over that time), the
torch baseline's time (CUDA events, median of --steps after warm-up) and the fraction of rows where its neighbour list
differs from the exact one (in order, and as a set).  `verified`: indices and distance bits equal the CPU reference on
every row of (a) to (c) and on 256 sampled rows of (d).  The GPU's name and power limit are read in the same run.
Writes nothing into the tree (only --out, when given).
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


def torch_knn(torch, x, y, sizes_x, sizes_y, k):
    """DGCNN-style kNN: pad each cloud to the largest one, torch.cdist (default compute mode) + topk.  Padding data rows
    get +inf distances.  Returns the [nq, k] int64 global indices (unpadded query rows)."""
    B, nx, ny = len(sizes_x), int(max(sizes_x)), int(max(sizes_y))
    F = int(x.shape[1])
    xo = np.concatenate([[0], np.cumsum(sizes_x)])
    yo = np.concatenate([[0], np.cumsum(sizes_y)])
    uniform = len(set(sizes_x)) == 1 and len(set(sizes_y)) == 1
    xp = torch.zeros((B, nx, F), device="cuda")
    yp = torch.zeros((B, ny, F), device="cuda")
    valid = torch.zeros((B, nx), dtype=torch.bool, device="cuda")
    for s in range(B):
        xp[s, : sizes_x[s]] = x[xo[s]: xo[s + 1]]
        yp[s, : sizes_y[s]] = y[yo[s]: yo[s + 1]]
        valid[s, : sizes_x[s]] = True
    base = torch.as_tensor(xo[:-1], device="cuda").view(B, 1, 1)

    def once():
        d = torch.cdist(yp, xp)
        if not uniform:
            d = d.masked_fill(~valid[:, None, :], float("inf"))
        return d.topk(k, dim=-1, largest=False).indices

    def rows():
        i = once() + base
        return torch.cat([i[s, : sizes_y[s]] for s in range(B)]) if not uniform else i.reshape(-1, k)

    return once, rows


def workload(torch, t, name, x_np, y_np, sizes_x, sizes_y, k, steps, verify_rows=None, lbvh=False):
    import feature_knn_oracle as FK

    F = int(x_np.shape[1])
    same = y_np is None
    y_np = x_np if same else y_np
    x = torch.from_numpy(x_np).cuda()
    y = x if same else torch.from_numpy(y_np).cuda()
    bx = torch.from_numpy(np.repeat(np.arange(len(sizes_x)), sizes_x)).cuda()
    by = torch.from_numpy(np.repeat(np.arange(len(sizes_y)), sizes_y)).cuda()
    t.set_option("squared_dist", 1)
    t.feature_knn(x, y, k, batch_x=bx, batch_y=by)  # warm-up
    ms = []
    for _ in range(steps):
        idx, d2 = t.feature_knn(x, y, k, batch_x=bx, batch_y=by)
        ms.append(t.stats()["search_ms"])
    st = t.stats()
    lib_ms = float(np.median(ms))
    pairs = int(sum(a * b for a, b in zip(sizes_x, sizes_y)))
    idx_np, d2_np = idx.cpu().numpy(), d2.cpu().numpy()
    res = {"workload": name, "clouds": len(sizes_x), "n": int(x_np.shape[0]), "nq": int(y_np.shape[0]), "F": F, "k": k,
           "lib_ms": lib_ms, "lib_ms_all": ms, "rounds": int(st["rounds"]), "kernel_ms": list(st["kernel_ms"]),
           "pair_dims": pairs * F, "pair_dims_per_s": pairs * F / (lib_ms * 1e-3)}
    # plain-torch baseline
    once, rows = torch_knn(torch, x, y, sizes_x, sizes_y, k)
    res["torch_ms"] = median_ms(torch, once, steps)
    tb = rows().cpu().numpy()
    res["torch_rows_differ"] = float((tb != idx_np).any(axis=1).mean())
    res["torch_rows_wrong_set"] = float((np.sort(tb, 1) != np.sort(idx_np, 1)).any(axis=1).mean())
    res["speedup_vs_torch"] = res["torch_ms"] / lib_ms
    # exact reference
    xo, yo = FK.offsets_of(sizes_x), FK.offsets_of(sizes_y)
    mask = None
    if verify_rows is not None:
        mask = np.zeros(len(y_np), bool)
        mask[verify_rows] = True
    wi, wd = FK.knn(x_np, y_np, k, xo, yo, rows=mask)
    sel = slice(None) if mask is None else mask
    ok = bool((wi[sel] == idx_np[sel]).all() and (wd[sel].view(np.uint32) == d2_np[sel].view(np.uint32)).all())
    res["verified_rows"] = int(len(y_np) if mask is None else mask.sum())
    if lbvh:  # the LBVH segmented query on the same clouds
        t.build(x, batch=bx, batch_size=len(sizes_x))
        li, ld = t.query(y, k, batch=by)
        lms = []
        for _ in range(steps):
            t.build(x, batch=bx, batch_size=len(sizes_x))
            b_ms = t.stats()["build_ms"]
            t.query(y, k, batch=by)
            lms.append(b_ms + t.stats()["search_ms"])
        res["lbvh_build_plus_query_ms"] = float(np.median(lms))
        eq = bool((li.cpu().numpy() == idx_np).all() and (ld.cpu().numpy().view(np.uint32) == d2_np.view(np.uint32)).all())
        res["lbvh_equal"] = eq
        ok = ok and eq
    res["verified"] = ok
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch

    from owlraytracing_b200 import TrueKNN

    if not torch.cuda.is_available():
        raise SystemExit("feature_knn_bench needs a CUDA device")
    rng = np.random.default_rng(0)
    out = {"bench": "feature_knn", "device": device_info(torch), "steps": a.steps, "workloads": []}
    W = out["workloads"]
    with TrueKNN(0) as t:
        x = rng.standard_normal((32 * 1024, 64)).astype(np.float32)
        W.append(workload(torch, t, "a_dgcnn_32x1024_F64", x, None, [1024] * 32, [1024] * 32, 20, a.steps))
        x = rng.standard_normal((16 * 2048, 128)).astype(np.float32)
        W.append(workload(torch, t, "b_16x2048_F128", x, None, [2048] * 16, [2048] * 16, 20, a.steps))
        x = rng.random((8 * 4096, 3), dtype=np.float32)
        W.append(workload(torch, t, "c_8x4096_F3_vs_lbvh", x, None, [4096] * 8, [4096] * 8, 20, a.steps, lbvh=True))
        x = rng.standard_normal((65536, 32)).astype(np.float32)
        y = rng.standard_normal((4096, 32)).astype(np.float32)
        rows = np.sort(rng.choice(4096, 256, replace=False))
        W.append(workload(torch, t, "d_65536x4096_F32_split", x, y, [65536], [4096], 16, a.steps, verify_rows=rows))
    out["verified"] = all(w["verified"] for w in out["workloads"])
    line = json.dumps(out)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
