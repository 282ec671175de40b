"""Where round 1 on the cell grid spends its time: the counting grid_knn_kernel's per-phase clock64() cycles and its
insert-loop figures, for cfg2 (10 M uniform points) and cfg4 (100 M), k = 10, every point a query (tknn_search_shard).

    python tools/grid_phases.py [cfg2|cfg4 ...] [--quantiles 990,900]   (start-radius quantiles in per mille)

Per workload and quantile one JSON line: round 1's share of warp cycles per phase, inserts per query, insert-loop
iterations per warp, and the loop's lane efficiency = inserts / (iterations x 32).  The counting kernel runs at its own
register count and occupancy, so the shares describe where a warp's cycles go, not the production kernel's wall time.
"""
import argparse
import json
import sys

import torch

sys.path.insert(0, ".")
from owlraytracing_b200 import TrueKNN  # noqa: E402

PHASES = ("setup", "walk", "stage", "filter", "insert", "emit")
N = {"cfg2": 10_000_000, "cfg4": 100_000_000}
k = 10

ap = argparse.ArgumentParser()
ap.add_argument("workloads", nargs="*", default=["cfg2", "cfg4"])
ap.add_argument("--quantiles", default="990")
args = ap.parse_args()
print(json.dumps({"gpu": torch.cuda.get_device_name(0)}), flush=True)
for wl in args.workloads:
    n = N[wl]
    x = torch.empty((n, 3), dtype=torch.float32, device="cuda")
    out = (torch.empty((n,), dtype=torch.int32, device="cuda"), torch.empty((n, k), dtype=torch.int32, device="cuda"),
           torch.empty((n, k), dtype=torch.float32, device="cuda"))
    for q in (int(v) for v in args.quantiles.split(",")):
        with TrueKNN(0, counters=1, grid_radius_quantile=q) as t:
            t.set_stream(torch.cuda.current_stream().cuda_stream)
            t.generate_uniform(42, 0, n, out=x)
            t.build(x)
            t.search_shard(k, 0, 1, out=out)
            s = t.stats()
            cyc = s["grid_phase_cycles"]
            tot = sum(cyc) or 1
            it, ins = s["grid_insert_iters"], s["grid_inserts"]
            groups = (n + 31) // 32
            print(json.dumps({
                "workload": wl, "quantile_pm": q, "start_radius": s["start_radius"], "round_queries": s["round_queries"],
                "grid_rounds": s["grid_rounds"],
                "phase_share": {p: round(c / tot, 4) for p, c in zip(PHASES, cyc)},
                "phase_gcycles": {p: round(c / 1e9, 3) for p, c in zip(PHASES, cyc)},
                "round1_inserts_per_query": round(ins / n, 3),
                "insert_iters_per_group": round(it / groups, 2),
                "insert_lane_efficiency": round(ins / (32 * it), 4) if it else None,
                "points_staged_per_group_all_rounds": round(s["warp_point_loads"] / groups, 1),
            }), flush=True)
