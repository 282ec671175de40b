"""Round 2 of cfg2 (10 M uniform points, k = 10, all points are queries) on its three kernels, at start radii that leave
between ~100 K and a few K queries to it: one warp per query (traverse_warp_kernel, warp_round_max = n), one thread per
query on the LBVH (traverse_sparse_kernel, grid = 1) and on the cell grid (grid_sparse_kernel), and the default routing
between them (sparse_divisor = 1 in all four: every round after the first is a sparse one).  Per line: the leftover count
and the best round-2 kernel time of 6 searches; all routings of a radius must give the same rows.

    python tools/grid_sparse_sweep.py [factor ...]     (start radius = factor x the estimator's radius; default 1 .. 1.16)
"""
import json
import sys

import torch

sys.path.insert(0, ".")
from owlraytracing_b200 import TrueKNN  # noqa: E402

n, k = 10_000_000, 10
factors = [float(a) for a in sys.argv[1:]] or [1.0, 1.02, 1.05, 1.08, 1.12, 1.16]
x = torch.empty((n, 3), dtype=torch.float32, device="cuda")
with TrueKNN(0) as t:
    t.generate_uniform(42, 0, n, out=x)
    t.build(x)
    t.search_shard(k, 0, 1)
    r0 = t.stats()["start_radius"]
routes = {"default": dict(sparse_divisor=1), "warp": dict(warp_round_max=n, sparse_divisor=1),
          "lbvh_thread": dict(grid=1, warp_round_max=0, sparse_divisor=1), "grid_thread": dict(warp_round_max=0, sparse_divisor=1)}
ctx = {name: TrueKNN(0, **o) for name, o in routes.items()}
for t in ctx.values():
    t.set_stream(torch.cuda.current_stream().cuda_stream)
    t.build(x)
out = (torch.empty((n,), dtype=torch.int32, device="cuda"), torch.empty((n, k), dtype=torch.int32, device="cuda"),
       torch.empty((n, k), dtype=torch.float32, device="cuda"))
for f in factors:
    r = r0 * f
    line, ref = {"factor": f, "start_radius": r}, None
    for name, t in ctx.items():
        best = None
        for _ in range(6):
            t.search_shard(k, 0, 1, start_radius=r, out=out)
            s = t.stats()
            if best is None or s["kernel_ms"][1] < best["kernel_ms"][1]:
                best = s
        chk = (int(out[1].long().sum().item()), float(out[2].double().sum().item()))
        assert ref is None or chk == ref, (name, f)
        ref = chk
        line["round2_queries"] = best["round_queries"][1]
        line[name + "_round2_ms"] = round(best["kernel_ms"][1], 4)
        line[name + "_round1_ms"] = round(best["kernel_ms"][0], 4)
    print(json.dumps(line), flush=True)
for t in ctx.values():
    t.close()
