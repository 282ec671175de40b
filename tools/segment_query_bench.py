"""Segmented query-set benchmark: batches of point clouds with a separate query set per cloud through
tknn_query_segments / tknn_radius_query_segments, verified against the per-segment CPU reference
(tests/segment_query_oracle.py); prints one JSON line.

    python tools/segment_query_bench.py [--steps 5] [--loop-subset 1024]

Workloads (torch_cluster's knn(x, y, k, batch_x, batch_y) and radius(x, y, r, batch_x, batch_y) as PointNet++ and
knn_interpolate call them):
  set_abstraction_radius   1 024 uniform clouds of 4 096 points, every 4th point a query, r = 0.123
  interpolation_k3         the reverse: data = every 4th point (1 024 per cloud), queries = all 4 096 points, k = 3
  small_clouds_k16         65 536 uniform clouds of 64 points, 16 queries each (every 4th point), k = 16
  self_query_k16           1 024 x 4 096, the built points as queries with self ids and the build's offsets, k = 16,
                           beside tknn_search on the same build (the price of staging a query set)
Per workload: the device time of the call (the library's search_ms, median of --steps calls after one warm-up call;
clouds, queries and outputs on the device; the radius call is the single call with preallocated outputs), the same
clouds through a per-cloud loop of build + query on one context (host wall time ending in a device synchronise; the
65 536-cloud loop times its first --loop-subset clouds and extrapolates), and the same concatenated sets through one
unsegmented tknn_query / tknn_radius_query as a cost reference (its answer is wrong: neighbours leak between clouds; the
radius reference shrinks r by 1024^(1/3) so that its balls hold about as many entries as the segmented ones).
`verified`: indices and distance bits equal the CPU reference (the 65 536-cloud workload checks every 16th cloud).  The
GPU's name and power limit are read in the same run.  Writes nothing into the tree.
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


def median(v):
    return float(np.median(np.asarray(v, np.float64)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--loop-subset", type=int, default=1024)
    args = ap.parse_args()

    import torch

    import segment_query_oracle as SQ
    from owlraytracing_b200 import TrueKNN, datasets

    if not torch.cuda.is_available():
        raise SystemExit("segment_query_bench needs a CUDA device")
    res = {"bench": "segment_query", "device": device_info(torch), "steps": args.steps, "workloads": []}
    t = TrueKNN(0)
    t.set_option("squared_dist", 1)

    def timed_ms(fn):
        """median device time (search_ms) of --steps calls after one warm-up call"""
        fn()
        torch.cuda.synchronize()
        runs = []
        for _ in range(args.steps):
            fn()
            torch.cuda.synchronize()
            runs.append(t.stats()["search_ms"])
        return median(runs)

    def bits(a):
        a = a.cpu().numpy() if hasattr(a, "cpu") else np.asarray(a)
        return a.view(np.uint32) if a.dtype == np.float32 else a.astype(np.int64)

    def same(got, want):
        return all(np.array_equal(bits(g), bits(w)) for g, w in zip(got, want))

    def loop_ms(xc, yc, count, call):
        """build + query of every cloud on one context, host wall time ending in a synchronise (extrapolated)"""
        m = min(count, args.loop_subset)
        call(xc(0), yc(0))
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for c in range(m):
            call(xc(c), yc(c))
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1e3 * count / m, m

    def knn_workload(name, x, xs, y, ys, k, check_segments=None, self_ids=None):
        count = len(xs)
        x_off, y_off = SQ.offsets_of(xs), SQ.offsets_of(ys)
        xt, yt = torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda()
        bx = torch.from_numpy(np.repeat(np.arange(count), xs)).cuda()
        by = torch.from_numpy(np.repeat(np.arange(count), ys)).cuda()
        sid = None if self_ids is None else torch.from_numpy(self_ids).cuda()
        t.build(xt, batch=bx)
        got = t.query(yt, k, self_ids=sid, batch=by)
        want = SQ.knn(x, y, x_off, y_off, k, self_ids=self_ids, squared=True, segments=check_segments)
        rows = slice(None) if check_segments is None else np.concatenate(
            [np.arange(int(y_off[s]), int(y_off[s + 1])) for s in check_segments])
        ok = same((got[0][rows], got[1][rows]), (want[0][rows], want[1][rows]))
        w = {"workload": name, "clouds": count, "data_points": len(x), "queries": len(y), "k": k,
             "call_ms": timed_ms(lambda: t.query(yt, k, self_ids=sid, batch=by)), "rounds": t.stats()["rounds"],
             "verified": ok, "verified_clouds": count if check_segments is None else len(check_segments)}
        xo, yo = x_off.astype(np.int64), y_off.astype(np.int64)
        lm, m = loop_ms(lambda c: xt[xo[c]:xo[c + 1]], lambda c: yt[yo[c]:yo[c + 1]], count,
                        lambda xc, yc: t.build(xc).query(yc, min(k, len(xc))))
        w.update({"loop_ms": lm, "loop_clouds_timed": m, "loop_extrapolated": m < count, "speedup_vs_loop": lm / w["call_ms"]})
        t.build(xt)
        w["unsegmented_query_ms"] = timed_ms(lambda: t.query(yt, k))
        w["ratio_to_unsegmented"] = w["call_ms"] / w["unsegmented_query_ms"]
        return w, t, xt, bx

    # 1 024 x 4 096, every 4th point a query: PointNet++ set abstraction (radius)
    x = datasets.uniform(1024 * 4096, seed=11)
    xs, y, ys = [4096] * 1024, np.ascontiguousarray(x[::4]), [1024] * 1024
    x_off, y_off = SQ.offsets_of(xs), SQ.offsets_of(ys)
    xt, yt = torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda()
    bx = torch.from_numpy(np.repeat(np.arange(1024), 4096)).cuda()
    by = torch.from_numpy(np.repeat(np.arange(1024), 1024)).cuda()
    r = 0.123
    t.build(xt, batch=bx)
    got = t.radius_query(yt, r, batch=by)
    want = SQ.radius_lists(x, y, x_off, y_off, r)
    total = int(want[0][-1])
    out = (torch.empty(len(y) + 1, dtype=torch.int64, device="cuda"), torch.empty(total, dtype=torch.int32, device="cuda"),
           torch.empty(total, dtype=torch.float32, device="cuda"))
    w = {"workload": "set_abstraction_radius", "clouds": 1024, "data_points": len(x), "queries": len(y), "r": r,
         "mean_neighbours": total / len(y), "verified": same(got, want),
         "call_ms": timed_ms(lambda: t.radius_query(yt, r, batch=by, out=out))}
    lm, m = loop_ms(lambda c: xt[c * 4096:(c + 1) * 4096], lambda c: yt[c * 1024:(c + 1) * 1024], 1024,
                    lambda xc, yc: t.build(xc).radius_query(yc, r))
    w.update({"loop_ms": lm, "loop_clouds_timed": m, "loop_extrapolated": m < 1024, "speedup_vs_loop": lm / w["call_ms"]})
    # The 1 024 clouds overlap, so an unsegmented ball of radius r would hold 1 024 times the entries (8.6 G): the
    # reference runs at r / 1024^(1/3), where the concatenated sets give about the same entries per query.
    t.build(xt)
    r_ref = r / 1024 ** (1 / 3)
    _, _, dd = t.radius_query(yt, r_ref)
    uout = (torch.empty(len(y) + 1, dtype=torch.int64, device="cuda"), torch.empty(len(dd), dtype=torch.int32, device="cuda"),
            torch.empty(len(dd), dtype=torch.float32, device="cuda"))
    w["unsegmented_query_ms"] = timed_ms(lambda: t.radius_query(yt, r_ref, out=uout))
    w["unsegmented_r"] = r_ref
    w["unsegmented_mean_neighbours"] = len(dd) / len(y)
    w["ratio_to_unsegmented"] = w["call_ms"] / w["unsegmented_query_ms"]
    res["workloads"].append(w)

    # the reverse at k = 3: knn_interpolate
    w, *_ = knn_workload("interpolation_k3", y, ys, x, xs, 3)
    res["workloads"].append(w)

    # 65 536 clouds of 64 points, 16 queries each
    xsm = datasets.uniform(65536 * 64, seed=12)
    ysm = np.ascontiguousarray(xsm[::4] + np.float32(0.001))
    w, *_ = knn_workload("small_clouds_k16", xsm, [64] * 65536, ysm, [16] * 65536, 16, check_segments=range(0, 65536, 16))
    res["workloads"].append(w)

    # the built points as queries: tknn_query_segments beside tknn_search on the same build
    sid = np.arange(len(x), dtype=np.int32)
    w, t, xt, bx = knn_workload("self_query_k16", x, xs, x, xs, 16, self_ids=sid)
    t.build(xt, batch=bx)
    w["search_ms"] = timed_ms(lambda: t.search(16))
    w["ratio_to_search"] = w["call_ms"] / w["search_ms"]
    sidt = torch.from_numpy(sid).cuda()
    a, b = t.search(16), t.query(xt, 16, self_ids=sidt, batch=bx)
    w["equals_search"] = bool((a[0] == b[0]).all().item() and (a[1].view(torch.int32) == b[1].view(torch.int32)).all().item())
    res["workloads"].append(w)

    t.close()
    res["verified"] = all(w["verified"] for w in res["workloads"]) and res["workloads"][-1]["equals_search"]
    print(json.dumps(res))


if __name__ == "__main__":
    main()
