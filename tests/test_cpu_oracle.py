"""CPU suite (no GPU): the oracle against its own ground truth, the committed golden vectors and
the reference-semantics pin; host logic; the C ABI surface."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest

from owlraytracing_b200 import _lib, datasets, read_points

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")


# ---------------------------------------------------------------- oracle vs ground truth
@pytest.mark.parametrize("n,k", [(2, 1), (50, 49), (1000, 1), (1000, 10), (5000, 64)])
def test_kdtree_equals_brute_uniform(oracle, n, k):
    x = datasets.uniform(n, seed=n)
    ib, db = oracle.knn_brute(x, k)
    ik, dk = oracle.knn_kdtree(x, k)
    assert (ib == ik).all() and (db == dk).all()


def test_kdtree_equals_brute_adversarial(oracle):
    rng = np.random.default_rng(0)
    base = rng.random((800, 3), dtype=np.float32)
    clouds = {
        "duplicates": np.concatenate([base, base[:400], np.tile(base[:1], (100, 1))]),
        "line": np.stack([np.linspace(0, 1, 2000, dtype=np.float32)] * 3, 1),
        "plane": np.concatenate([rng.random((2000, 2), dtype=np.float32), np.zeros((2000, 1), np.float32)], 1),
        "lattice": datasets.lattice(9),
        "lidar": datasets.lidar_like(6000, seed=7),
        "identical": np.full((300, 3), 1.5, np.float32),
    }
    for name, x in clouds.items():
        x = np.ascontiguousarray(x, np.float32)
        for k in (1, 6, 27):
            ib, db = oracle.knn_brute(x, k)
            ik, dk = oracle.knn_kdtree(x, k)
            assert (ib == ik).all() and (db == dk).all(), (name, k)


def _numpy_d2(x):
    """The fma-chain d2 of every pair, emulated exactly in float64: differences, products and two-term sums of
    float32 values are exact in float64, so rounding to float32 after each step reproduces fmaf bit for bit."""
    xd = x.astype(np.float64)
    d = (xd[:, None, :] - xd[None, :, :]).astype(np.float32).astype(np.float64)     # dx, dy, dz rounded to fp32
    acc = (d[..., 0] * d[..., 0]).astype(np.float32).astype(np.float64)              # dx * dx
    acc = (d[..., 1] * d[..., 1] + acc).astype(np.float32).astype(np.float64)        # fmaf(dy, dy, .)
    return (d[..., 2] * d[..., 2] + acc).astype(np.float32)                          # fmaf(dz, dz, .)


def test_oracle_properties_hypothesis(oracle):
    """Property test (hypothesis): on small tie-heavy clouds (coordinates on a coarse grid, duplicates, 2-D) the
    brute-force oracle, the kd-tree oracle and an independent numpy restatement agree bit for bit, rows ascend
    in (d2, index), and range_count equals the number of pairs within the radius."""
    from hypothesis import given, settings, strategies as st

    @settings(max_examples=60, deadline=None, derandomize=True)
    @given(st.integers(8, 120), st.integers(1, 7), st.integers(2, 9), st.booleans(), st.integers(0, 2 ** 31 - 1))
    def run(n, k, grid, planar, seed):
        rng = np.random.default_rng(seed)
        x = (rng.integers(0, grid, (n, 3)) / np.float32(grid - 1)).astype(np.float32)
        x += (rng.random((n, 3)) < 0.3) * rng.random((n, 3)).astype(np.float32) * np.float32(1e-3)  # a few off-grid points
        if planar:
            x[:, 2] = 0
        x = np.ascontiguousarray(x, np.float32)
        ib, db = oracle.knn_brute(x, k)
        ik, dk = oracle.knn_kdtree(x, k)
        assert (ib == ik).all() and (db == dk).all()
        # independent restatement: (d2, index) keys, self excluded by index
        d2 = _numpy_d2(x)
        keys = (d2.view(np.uint32).astype(np.uint64) << np.uint64(32)) | np.arange(n, dtype=np.uint64)[None, :]
        keys[np.arange(n), np.arange(n)] = np.uint64(0xFFFFFFFFFFFFFFFF)
        order = np.argsort(keys, axis=1, kind="stable")[:, :k]
        assert (ib == order.astype(np.int32)).all()
        nd2 = np.take_along_axis(d2, order, 1)
        assert (db == np.sqrt(nd2)).all()                              # sqrtf is correctly rounded on both sides
        assert (np.diff(nd2, axis=1) >= 0).all()
        assert (np.diff(ib, axis=1)[np.diff(nd2, axis=1) == 0] > 0).all()   # equal d2 => ascending index
        r = np.float32(db[:, -1].max())
        within = d2 <= r * r
        within[np.arange(n), np.arange(n)] = False
        assert (oracle.range_count(x, float(r)) == within.sum(1)).all()

    run()


def test_lattice_known_answers(oracle):
    """Hand-computable: interior lattice point has 6 neighbours at 1, 12 at sqrt 2, 8 at sqrt 3."""
    m = 7
    x = datasets.lattice(m)
    idx, dist = oracle.knn_brute(x, 26)
    c = 3 * m * m + 3 * m + 3
    assert (dist[c][:6] == 1.0).all()
    assert np.allclose(dist[c][6:18], np.sqrt(np.float32(2)), rtol=0, atol=0)
    assert (dist[c][18:26] == np.sqrt(np.float32(3))).all()
    # lowest-index tie-break inside each shell
    for a, b in ((0, 6), (6, 18), (18, 26)):
        assert (np.diff(idx[c][a:b]) > 0).all()
    expected6 = sorted(c + d for d in (-m * m, -m, -1, 1, m, m * m))
    assert idx[c][:6].tolist() == expected6
    # corner point 0: its three unit neighbours are 1, m, m*m
    assert idx[0][:3].tolist() == [1, m, m * m]


def test_distance_formula_is_the_fma_chain(oracle):
    rng = np.random.default_rng(1)
    a = rng.random((200, 3)).astype(np.float32)
    b = rng.random((200, 3)).astype(np.float32)
    for p, q in zip(a, b):
        d = (p - q).astype(np.float32)
        # fmaf(dz,dz,fmaf(dy,dy,dx*dx)) evaluated exactly in float64 then rounded once per fma
        t0 = np.float32(d[0] * d[0])
        t1 = np.float32(np.float64(d[1]) * np.float64(d[1]) + np.float64(t0))
        t2 = np.float32(np.float64(d[2]) * np.float64(d[2]) + np.float64(t1))
        assert oracle.dist2(p, q) == t2


def test_self_excluded_by_index_not_by_position(oracle):
    x = np.array([[0, 0, 0], [0, 0, 0], [1, 0, 0]], np.float32)
    idx, dist = oracle.knn_brute(x, 2)
    assert idx[0].tolist() == [1, 2] and dist[0].tolist() == [0.0, 1.0]
    assert idx[1].tolist() == [0, 2]


# ---------------------------------------------------------------- reference semantics pin
def test_reference_rounds_equal_exact_when_radius_covers_cloud(oracle):
    """The reference's own rules (deviceCode.cu:62-152, hostCode.cpp:285-340) give the exact answer
    when the first radius already covers every point: the one place its semantics and the exact
    oracle coincide (SURVEY.md F2)."""
    x = datasets.uniform(2500, seed=5)
    ib, db = oracle.knn_brute(x, 7)
    ir, dr, rounds, _, rc = oracle.reference_trueknn(x, 7, 2.0)
    assert rc == 0 and rounds == 1
    assert (ir == ib).all() and (dr == db).all()


def test_reference_rounds_are_inexact_from_a_small_radius(oracle):
    """F2: candidates come from an L-inf cube and a query stops once k were inserted."""
    x = datasets.uniform(4000, seed=6)
    ib, _ = oracle.knn_brute(x, 10)
    ir, dr, rounds, fr, rc = oracle.reference_trueknn(x, 10, 0.01)
    assert rc == 0 and rounds > 1 and fr == pytest.approx(0.01 * 2 ** (rounds - 1))
    wrong = np.mean([set(a) != set(b) for a, b in zip(ir, ib)])
    assert 0.01 < wrong < 0.9
    assert (np.diff(dr, axis=1) >= 0).all()  # still sorted (deviceCode.cu:121-134)


def test_golden_vectors(oracle):
    """Committed fixtures (tests/golden/make_golden.py): the oracle must keep producing them."""
    g = np.load(os.path.join(GOLDEN, "knn_golden.npz"))
    for name in ("uniform", "lidar", "lattice", "dups"):
        x, k = g[f"{name}_x"], int(g[f"{name}_k"])
        idx, dist = oracle.knn_kdtree(x, k)
        assert (idx == g[f"{name}_idx"]).all(), name
        assert (dist == g[f"{name}_dist"]).all(), name
    assert (datasets.uniform(64, seed=42) == g["hash_uniform_seed42_first64"]).all()


# ---------------------------------------------------------------- host logic
def test_point_file_grammar_matches_reference_restatement(oracle, tmp_path):
    text = b"1,2,3\n4 5 6\n 7.5, 8e-1 ,9\n10,11,12,13\n14,15,16\n"
    p = tmp_path / "pts.csv"
    p.write_bytes(text)
    for n, dim in ((1, 3), (3, 3), (2, 2)):
        try:
            want = oracle.parse_points(text, n, dim)
        except ValueError:
            with pytest.raises(ValueError):
                read_points(str(p), n, dim)
            continue
        got = read_points(str(p), n, dim)
        assert got.shape == want.shape and (got == want).all(), (n, dim)
    # a row with more than `dim` columns mis-strides exactly like hostCode.cpp:95-103
    got = read_points(str(p), 5, 2)
    assert got[0].tolist() == [1, 2, 0] and got[1].tolist() == [3, 4, 0]
    # binary fast path
    x = datasets.uniform(100, seed=1)
    b = tmp_path / "pts.f32"
    x.tofile(str(b))
    assert (read_points(str(b), 40, 3) == x[:40]).all()


def test_uniform_generator_is_index_addressable():
    a = datasets.uniform(1000, seed=42)
    b = datasets.uniform(300, seed=42, first=500)
    assert (a[500:800] == b).all()
    assert a.min() >= 0 and a.max() < 1 and a.dtype == np.float32
    assert abs(a.mean() - 0.5) < 0.02


def test_lidar_generator_shape():
    x = datasets.lidar_like(50_000, seed=7)
    assert x.shape == (50_000, 3) and np.isfinite(x).all()
    _, counts = np.unique(x, axis=0, return_counts=True)
    assert (counts > 1).sum() >= 40  # the 0.1 % exact duplicates


# ---------------------------------------------------------------- the C ABI surface (no compute without a GPU)
def test_library_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "trueknn.h")).read()
    declared = sorted(set(re.findall(r"TKNN_API\s+[\w\s\*]+?\b(tknn_\w+)\s*\(", header)))
    assert declared == sorted(_lib.EXPORTS)
    L = _lib.load()
    for name in declared:
        assert hasattr(L, name), name
    out = subprocess.run(["nm", "-D", "--defined-only", _lib.LIB_PATH], capture_output=True, text=True).stdout
    exported = set(re.findall(r" T (\w+)", out))
    assert set(declared) <= exported
    assert not [s for s in exported if not s.startswith("tknn_") and not s.startswith("_")]  # nothing else leaks
    assert L.tknn_version() == 100


def test_option_keys_match_header():
    """Every TKNN_OPT_* key of the header has the same value in the ctypes mirror and a name in TrueKNN._OPTS."""
    from owlraytracing_b200.trueknn import TrueKNN

    header = open(os.path.join(ROOT, "include", "trueknn.h")).read()
    keys = {name: int(val) for name, val in re.findall(r"^\s*,?\s*TKNN_(OPT_\w+)\s*=\s*(\d+)", header, re.M)}
    assert len(keys) >= 15 and len(set(keys.values())) == len(keys)
    for name, val in keys.items():
        assert getattr(_lib, name) == val, name
    assert sorted(TrueKNN._OPTS.values()) == sorted(keys.values())


def test_stats_struct_layout_matches_header(tmp_path):
    src = "#include <stdio.h>\n#include \"trueknn.h\"\nint main(){printf(\"%zu %zu %zu\", sizeof(tknn_stats), " \
          "__builtin_offsetof(tknn_stats, round_ms), __builtin_offsetof(tknn_stats, h2d_bytes));return 0;}"
    exe = str(tmp_path / "tknn_layout")
    subprocess.run(["/usr/bin/gcc", "-x", "c", "-", "-I", os.path.join(ROOT, "include"), "-o", exe], input=src, text=True,
                   check=True)
    size, off_round, off_h2d = (int(v) for v in subprocess.run([exe], capture_output=True, text=True).stdout.split())
    assert size == ctypes.sizeof(_lib.Stats)
    assert off_round == _lib.Stats.round_ms.offset and off_h2d == _lib.Stats.h2d_bytes.offset


def test_dist_stats_struct_layout_matches_header(tmp_path):
    src = "#include <stdio.h>\n#include \"trueknn.h\"\nint main(){printf(\"%zu %zu %zu %zu\", sizeof(tknn_dist_stats), " \
          "__builtin_offsetof(tknn_dist_stats, h2d_ms), __builtin_offsetof(tknn_dist_stats, search_total_ms), " \
          "__builtin_offsetof(tknn_dist_stats, bytes_sent_search));return 0;}"
    exe = str(tmp_path / "tknn_dist_layout")
    subprocess.run(["/usr/bin/gcc", "-x", "c", "-", "-I", os.path.join(ROOT, "include"), "-o", exe], input=src, text=True,
                   check=True)
    size, o1, o2, o3 = (int(v) for v in subprocess.run([exe], capture_output=True, text=True).stdout.split())
    D = _lib.DistStats
    assert size == ctypes.sizeof(D) and o1 == D.h2d_ms.offset and o2 == D.search_total_ms.offset and o3 == D.bytes_sent_search.offset


def test_multi_gpu_calls_fail_cleanly_without_a_device():
    """No GPU: tknn_create_multi reports an error code (no crash, no CPU fallback); comm calls on a null context are EINVAL."""
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    L = _lib.load()
    ids = (ctypes.c_int * 2)(0, 1)
    h = ctypes.c_void_p()
    assert L.tknn_create_multi(ids, 2, _lib.SHARD_QUERIES, ctypes.byref(h)) != _lib.OK and not h.value
    assert L.tknn_create_multi(ids, 0, _lib.SHARD_QUERIES, ctypes.byref(h)) == _lib.EINVAL
    assert L.tknn_create_multi(ids, 2, 7, ctypes.byref(h)) == _lib.EINVAL
    assert L.tknn_comm_init(None, 2, 0, ctypes.c_char_p(b"x" * 128)) == _lib.EINVAL
    assert L.tknn_partition_owned(None) == 0


def test_no_cpu_fallback_without_a_device():
    """Without a usable CUDA device tknn_create fails; nothing silently computes on the host."""
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from owlraytracing_b200 import TrueKNN, TrueKNNError

    with pytest.raises(TrueKNNError) as e:
        TrueKNN(0)
    assert e.value.code == _lib.ECUDA


def test_product_code_never_touches_the_oracle():
    pkg = os.path.join(ROOT, "owlraytracing_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h")):
                text = open(os.path.join(dirpath, f), errors="ignore").read()
                assert "liboracle" not in text and "from oracle" not in text and "import oracle" not in text, f


def test_fast_ingest_matches_grammar_and_writer_round_trips(oracle, tmp_path):
    """tknn_read_points (mmap + parallel parse) against the reference-grammar restatement, and the
    neighbour writer in the format the reference leaves commented out (hostCode.cpp:316)."""
    from owlraytracing_b200 import read_points_fast, write_neighbours

    rng = np.random.default_rng(3)
    x = (rng.random((200_000, 3)) * 200 - 100).astype(np.float32)
    lines = []
    for i, p in enumerate(x):
        sep = ("," if i % 3 == 0 else " " if i % 3 == 1 else ", ")
        lines.append(sep.join(repr(float(v)) for v in p))
    text = ("\n".join(lines) + "\n").encode()
    path = tmp_path / "big.csv"
    path.write_bytes(text)
    for n in (1, 777, 200_000, 300_000):
        got = read_points_fast(str(path), n, 3)
        assert got.shape[0] == min(n, 200_000) and (got == x[: got.shape[0]]).all()
    small = b"1,2,3\n+4 5e0 6\n 7.5, 8e-1 ,9 junk 10\n10,11,12,13\n14,15,16\n"
    sp = tmp_path / "small.csv"
    sp.write_bytes(small)
    for n, dim in ((1, 3), (3, 3), (2, 2), (5, 2), (4, 3)):
        try:
            want = oracle.parse_points(small, n, dim)
        except ValueError:
            with pytest.raises(ValueError):
                read_points_fast(str(sp), n, dim)
            continue
        got = read_points_fast(str(sp), n, dim)
        assert got.shape == want.shape and (got == want).all(), (n, dim)
    b = tmp_path / "pts.f32"
    x[:1000].tofile(str(b))
    assert (read_points_fast(str(b), 400, 3) == x[:400]).all()
    # writer
    idx = rng.integers(0, 1000, (5000, 4)).astype(np.int32)
    dist = rng.random((5000, 4)).astype(np.float32)
    out = tmp_path / "nn.csv"
    write_neighbours(str(out), idx, dist)
    back = np.loadtxt(str(out), delimiter=",")
    assert (back[:, 0] == np.repeat(np.arange(5000), 4)).all()
    assert (back[:, 1].astype(np.int32) == idx.reshape(-1)).all()
    assert (back[:, 2].astype(np.float32) == dist.reshape(-1)).all()
    write_neighbours(str(tmp_path / "nn"), idx, dist, binary=True)
    assert (np.fromfile(str(tmp_path / "nn.idx.i32"), np.int32).reshape(idx.shape) == idx).all()


def test_read_points_reports_the_capacity_it_needs(tmp_path):
    """ADVICE r1: the grammar consumes the LAST line read whole (hostCode.cpp:92), so a file with many floats per line
    yields more than n rows; tknn_read_points then names the capacity a retry needs and the Python / C++ hosts retry."""
    from owlraytracing_b200 import read_points, read_points_fast

    pts = np.arange(300, dtype=np.float32).reshape(100, 3)
    one_line = tmp_path / "one_line.txt"
    one_line.write_text(" ".join(repr(float(v)) for v in pts.reshape(-1)) + "\n")   # all 300 floats on one line
    want = read_points(str(one_line), 10, 3)            # the reference reads the whole line: 100 points, not 10
    assert want.shape == (100, 3)
    got = read_points_fast(str(one_line), 10, 3)
    assert (got == want).all()
    L = _lib.load()
    out = np.empty((18, 3), np.float32)
    m = ctypes.c_uint64(0)
    rc = L.tknn_read_points(str(one_line).encode(), 10, 3, ctypes.c_void_p(out.ctypes.data), 18, ctypes.byref(m))
    assert rc == _lib.EINVAL and m.value == 100       # too small: the row count it needs comes back
    four = tmp_path / "four_per_line.txt"
    four.write_text("\n".join(",".join(repr(float(v)) for v in row) for row in pts.reshape(-1, 12)) + "\n")
    assert (read_points_fast(str(four), 7, 3) == read_points(str(four), 7, 3)).all()


def test_bench_cpu_arm_sampling_is_coherent_and_uses_all_cores(oracle):
    """bench.py's CPU arm: runs of consecutive tree positions (spatially coherent like the GPU's order), answers equal to
    the plain query path, and every core in use even when the launcher exported OMP_NUM_THREADS=1 (torchrun does)."""
    import importlib.util

    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    pos = bench._coherent_positions(1_000_000, 50_000, 3)
    assert pos.shape == (50_000,) and len(np.unique(pos)) == 50_000 and pos.min() >= 0 and pos.max() < 1_000_000
    assert (np.diff(pos.reshape(-1, 4096)[:, :], axis=1) == 1).all() if pos.size % 4096 == 0 else True
    assert (bench._coherent_positions(1000, 5000, 0) < 1000).all()
    x = datasets.uniform(60_000, seed=3)
    t = oracle.KdTree(x, leaf=8)
    ids, idx, dist = t.query_positions(bench._coherent_positions(60_000, 9_000, 1), 7)
    ri, rd = t.query(x[ids], 7, self_ids=ids)
    assert (idx == ri).all() and (dist == rd).all()
    t.close()
    oracle.set_num_threads(os.cpu_count())
    assert oracle.num_threads() == os.cpu_count()


def test_header_is_c99_and_links_from_plain_c(tmp_path):
    """The boundary is a C ABI: include/trueknn.h must compile as C99 (-pedantic) and link from a plain C host — the shape
    of the reference's own API test (tests/t00-c99-compliant-header/hostCode.c:30-46).  No CUDA call is made."""
    src = tmp_path / "host.c"
    src.write_text(
        '#include "trueknn.h"\n#include <stdio.h>\n'
        "int main(void) { tknn_stats s; tknn_dist_stats d; tknn_multi *m = 0; (void)s; (void)d; (void)m;\n"
        '  printf("%d\\n", tknn_version()); return tknn_version() == TKNN_VERSION ? 0 : 1; }\n')
    exe = tmp_path / "host"
    lib_dir = os.path.dirname(_lib.LIB_PATH)
    r = subprocess.run(["/usr/bin/gcc", "-std=c99", "-pedantic", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"),
                        str(src), "-L", lib_dir, "-ltrueknn", f"-Wl,-rpath,{lib_dir}", "-o", str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0 and r.stdout.strip() == "100"


def test_key_layout_policy():
    """tknn_key_layout (host arithmetic, no device): the packed (code << index bits | index) sort key fits 64 bits, keeps
    at least log2(n)/3 + 3 code bits per axis, never needs more than five passes when packed, and falls back to the
    (code, index) pair sort where that is impossible or not asked for."""
    import ctypes as C
    import math

    from owlraytracing_b200 import _lib

    L = _lib.load()

    def layout(n, bits=0, mode=0):
        b, i, p = C.c_int(-1), C.c_int(-1), C.c_int(-1)
        rc = L.tknn_key_layout(n, bits, mode, C.byref(b), C.byref(i), C.byref(p))
        return rc, b.value, i.value, p.value

    assert layout(10_000_000) == (0, 13, 24, 5)        # cfg2: 39 code bits + 24 index bits
    assert layout(100_000_000) == (0, 12, 27, 5)       # cfg4: 36 + 27
    assert layout(100_000) == (0, 13, 17, 5)           # cfg1
    assert layout(250_000_000)[2] == 0                 # a cfg5 rank: log2(n)/3 + 3 bits per axis do not fit beside 28 index bits
    assert layout(10_000_000, mode=1) == (0, 16, 0, 6)  # round 1's pair sort
    assert layout(10_000_000, bits=21) == (0, 21, 0, 8)  # more bits than fit beside the index: pairs
    assert layout(10_000_000, bits=12) == (0, 12, 24, 5)
    for n in [2, 3, 31, 32, 33, 1000, 4097, 2**20 - 1, 2**20, 2**20 + 1, 2**24, 2**24 + 1, 2**27, 2**28, 2**28 + 1, 2**30 - 1]:
        rc, b, i, p = layout(n)
        assert rc == 0 and 4 <= b <= 21 and p == (3 * b + 7) // 8
        lg = max(1, math.ceil(math.log2(n)))
        if i:
            assert i == lg and (n - 1) < (1 << i)        # every index fits below the code
            assert 3 * b + i <= 64 and p <= 5
            assert b >= (lg + 2) // 3 + 3                # cells at least 8x finer per axis than the mean point spacing
        else:
            assert b == min(21, max(10, (lg + 2) // 3 + 8))
    assert layout(1)[0] != 0 and layout(2**30)[0] != 0 and layout(1000, bits=3)[0] != 0 and layout(1000, mode=2)[0] != 0
