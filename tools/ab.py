"""A/B of library variants on one GPU: same workload, one subprocess per libtrueknn build (TKNN_LIB_PATH).

    python tools/ab.py cfg2|cfg3|cfg4|cfg1[,k=K] lib1.so lib2.so:curve=1 ...   (paths relative to owlraytracing_b200/lib/;
                                                                             optional tknn_set_option settings after ':')

Per variant: best-of-5 search_ms through tknn_search_shard (compact rows, device outputs: the bench's timed call), the
per-round kernel times, build phases, and a checksum of the result (all variants must agree; the first is compared
with tknn_brute_force on 512 sampled rows).
"""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CFG = {"cfg1": (100_000, 5, "uniform", 42), "cfg2": (10_000_000, 10, "uniform", 42), "cfg3": (10_000_000, 64, "lidar", 7),
       "cfg4": (100_000_000, 10, "uniform", 42)}


def child(which):
    import torch

    sys.path.insert(0, ROOT)
    from owlraytracing_b200 import TrueKNN, datasets

    which, _, kk = which.partition(",k=")  # "cfg2,k=16": the workload's cloud at another k
    n, k, cloud, seed = CFG[which]
    k = int(kk) if kk else k
    opts = {kv.split("=")[0]: int(kv.split("=")[1]) for kv in os.environ.get("TKNN_AB_OPTS", "").split(",") if kv}
    t = TrueKNN(0, **opts)
    t.set_stream(torch.cuda.current_stream().cuda_stream)
    if cloud == "uniform":
        x = torch.empty((n, 3), dtype=torch.float32, device="cuda")
        t.generate_uniform(seed, 0, n, out=x)
    else:
        x = torch.from_numpy(datasets.lidar_like(n, seed)).cuda()
    builds = []
    for _ in range(3):
        t.build(x)
        builds.append(t.stats())
    b = min(builds, key=lambda s: s["build_ms"])
    cap = t.shard_capacity(1)
    out = (torch.empty((cap,), dtype=torch.int32, device="cuda"), torch.empty((cap, k), dtype=torch.int32, device="cuda"),
           torch.empty((cap, k), dtype=torch.float32, device="cuda"))
    best = None
    for _ in range(6):
        qid, idx, dst = t.search_shard(k, 0, 1, out=out)
        s = t.stats()
        if best is None or s["search_ms"] < best["search_ms"]:
            best = s
    order = torch.argsort(qid.long())
    chk = int((idx[order].long() * (torch.arange(k, device="cuda") + 1)).sum().item()) ^ int(dst[order].double().sum().item() * 1e3)
    m = 512
    rows = (torch.arange(m, device="cuda") * qid.shape[0]) // m
    bi, bd = t.brute_force(qid[rows].contiguous(), k)
    ok = bool((bi == idx[rows]).all().item() and (bd == dst[rows]).all().item())
    t.set_option("counters", 1)
    t.search_shard(k, 0, 1, out=out)
    c = t.stats()
    print(json.dumps({"lib": os.path.basename(os.environ.get("TKNN_LIB_PATH", "default")), "opts": opts, "workload": which, "k": k,
                      "search_ms": round(best["search_ms"], 4), "estimate_ms": round(best["estimate_ms"], 4),
                      "kernel_ms": [round(v, 4) for v in best["kernel_ms"]], "round_queries": best["round_queries"],
                      "qps_M": round(n / best["search_ms"] / 1e3, 1), "build_ms": round(b["build_ms"], 4),
                      "build": {p: round(b[p], 4) for p in ("bounds_ms", "morton_ms", "sort_ms", "leaves_ms", "hierarchy_ms", "refit_ms")},
                      "inserts_per_q": round(c["heap_inserts"] / n, 2), "tests_per_q": round(c["points_tested"] / n, 1),
                      "nodes_per_q": round(c["nodes_visited"] / n, 1), "brute_ok": ok, "checksum": chk}), flush=True)


if __name__ == "__main__":
    if len(sys.argv) > 2 and sys.argv[1] == "--child":
        child(sys.argv[2])
    else:
        which, libs = sys.argv[1], sys.argv[2:] or ["libtrueknn.so"]
        for spec in libs:
            lib, _, o = spec.partition(":")     # "lib.so:option=value,option=value"
            env = dict(os.environ, TKNN_LIB_PATH=os.path.join(ROOT, "owlraytracing_b200", "lib", lib), TKNN_AB_OPTS=o)
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", which], env=env, capture_output=True, text=True, timeout=900)
            print(r.stdout.strip().splitlines()[-1] if r.returncode == 0 and r.stdout.strip() else json.dumps({"lib": lib, "rc": r.returncode, "err": r.stderr[-600:]}), flush=True)
