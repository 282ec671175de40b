"""Search time against the start-radius quantile (per mille), k = 10, every point a query (tknn_search_shard with device
outputs: the bench's timed call).  By default it sweeps TKNN_OPT_GRID_RADIUS_QUANTILE, the quantile of searches whose
round 1 walks the cell grid; --option radius_quantile sweeps the one of every other search.

    python tools/quantile_sweep.py [cfg2|cfg4] [--option grid_radius_quantile] [q ...]   (default 800 850 900 950 990)

Per quantile one JSON line: the best of 6 searches (search and estimate ms, per-round kernel ms and queries, start radius)
and, from one counting search, inserts per query over all rounds and in round 1.  The rows of every quantile must equal
those of the first.
"""
import argparse
import json
import sys

import torch

sys.path.insert(0, ".")
from owlraytracing_b200 import TrueKNN  # noqa: E402

N = {"cfg2": 10_000_000, "cfg4": 100_000_000}
ap = argparse.ArgumentParser()
ap.add_argument("workload", nargs="?", default="cfg2", choices=sorted(N))
ap.add_argument("quantiles", nargs="*", type=int, default=[800, 850, 900, 950, 990])
ap.add_argument("--option", default="grid_radius_quantile", choices=("grid_radius_quantile", "radius_quantile"))
args = ap.parse_args()
n, k = N[args.workload], 10
x = torch.empty((n, 3), dtype=torch.float32, device="cuda")
out = (torch.empty((n,), dtype=torch.int32, device="cuda"), torch.empty((n, k), dtype=torch.int32, device="cuda"),
       torch.empty((n, k), dtype=torch.float32, device="cuda"))
ref = None
print(json.dumps({"gpu": torch.cuda.get_device_name(0), "workload": args.workload, "option": args.option}), flush=True)
for q in args.quantiles:
    with TrueKNN(0, **{args.option: q}) as t:
        t.set_stream(torch.cuda.current_stream().cuda_stream)
        t.generate_uniform(42, 0, n, out=x)
        t.build(x)
        best = None
        for _ in range(6):
            t.search_shard(k, 0, 1, out=out)
            s = t.stats()
            if best is None or s["search_ms"] < best["search_ms"]:
                best = s
        if ref is None:
            ref = tuple(o.clone() for o in out)
        same = all(torch.equal(a, b) for a, b in zip(ref, out))
        t.set_option("counters", 1)
        t.search_shard(k, 0, 1, out=out)
        c = t.stats()
    print(json.dumps({"quantile_pm": q, "search_ms": round(best["search_ms"], 4), "estimate_ms": round(best["estimate_ms"], 4),
                      "kernel_ms": [round(v, 4) for v in best["kernel_ms"]], "round_queries": best["round_queries"],
                      "grid_rounds": best["grid_rounds"], "start_radius": best["start_radius"],
                      "inserts_per_query": round(c["heap_inserts"] / n, 3),
                      "round1_inserts_per_query": round(c["grid_inserts"] / n, 3), "rows_equal_first": same}), flush=True)
