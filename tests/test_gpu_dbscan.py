"""tknn_dbscan / TrueKNN.dbscan on the GPU: bit-exact against the CPU reference (tests/dbscan_oracle.c)."""
import ctypes

import numpy as np
import pytest

import dbscan_oracle as DO
from owlraytracing_b200 import MultiTrueKNN, TrueKNNError, datasets
from owlraytracing_b200 import _lib
from test_cpu_dbscan import lattice_roles

pytestmark = pytest.mark.gpu


def assert_same(got, want, what=""):
    gl, gc, gn = got
    wl, wc, wn = want
    gl, gc = np.asarray(gl), np.asarray(gc)
    assert gn == wn, f"{what}: {gn} clusters, want {wn}"
    bad = np.flatnonzero(gc != wc)
    assert bad.size == 0, f"{what}: {bad.size} core flags differ, first at {bad[:10]}"
    bad = np.flatnonzero(gl != wl)
    assert bad.size == 0, f"{what}: {bad.size} labels differ, first at {bad[:10]}: {gl[bad[:10]]} vs {wl[bad[:10]]}"


def check(knn, x, eps, min_pts, what):
    got = knn.build(x).dbscan(eps, min_pts)
    assert got[0].dtype == np.int32 and got[1].dtype == np.uint8
    assert_same(got, DO.dbscan(x, eps, min_pts), what)
    st = knn.stats()
    assert st["rounds"] == 4 and st["k"] == min_pts and st["n_queries"] == len(x)
    n_core = int(got[1].sum())
    assert st["round_queries"] == [len(x), n_core, n_core, len(x) - n_core]
    return got


@pytest.fixture(scope="module")
def uniform200k():
    return datasets.uniform(200_000, seed=42)


@pytest.mark.parametrize("eps", [0.015, 0.025])  # below the percolation point / one giant cluster
def test_uniform_200k(knn, uniform200k, eps):
    labels, core, c = check(knn, uniform200k, eps, 5, f"uniform eps={eps}")
    big = np.bincount(labels[labels >= 0]).max() if c else 0
    if eps == 0.025:
        assert big > len(labels) // 2
    else:
        assert big < len(labels) // 100


@pytest.fixture(scope="module")
def lidar1m():
    return datasets.lidar_like(1_000_000, seed=7)


@pytest.mark.parametrize("eps", [0.05, 0.3])
@pytest.mark.parametrize("min_pts", [5, 20])
def test_lidar_1m(knn, lidar1m, eps, min_pts):
    check(knn, lidar1m, eps, min_pts, f"lidar eps={eps} min_pts={min_pts}")


def duplicate_cloud():
    """The cloud of test_gpu_parity.py::test_duplicates_and_coincident_points."""
    rng = np.random.default_rng(5)
    base = rng.random((3000, 3), dtype=np.float32)
    return np.concatenate([base, base[:1500], base[:700], np.tile(base[:1], (200, 1))]).astype(np.float32)


@pytest.mark.parametrize("eps,min_pts", [(0.0, 2), (0.0, 3), (0.03, 4), (0.06, 12), (0.0, 201)])
def test_duplicates(knn, eps, min_pts):
    check(knn, duplicate_cloud(), eps, min_pts, f"duplicates eps={eps} min_pts={min_pts}")


def test_lattice_closed_ball(knn):
    m = 12
    x = datasets.lattice(m)
    interior, face, edge = lattice_roles(m)
    labels, core, c = check(knn, x, 1.0, 7, "lattice")
    assert c == 1 and (core.astype(bool) == interior).all()
    assert (labels[interior | face] == 0).all() and (labels[edge] == -1).all()
    labels, core, c = check(knn, x, float(np.nextafter(np.float32(1), np.float32(0))), 7, "lattice below 1")
    assert c == 0 and (labels == -1).all()


def test_two_dimensional_input(knn):
    rng = np.random.default_rng(3)
    x2 = np.concatenate([rng.normal(c, 0.02, (5000, 2)) for c in rng.random((8, 2))]).astype(np.float32)
    got = knn.build(x2).dbscan(0.01, 6)
    assert_same(got, DO.dbscan(x2, 0.01, 6), "2-D")
    assert got[2] > 1


def test_special_cases(knn):
    x = datasets.uniform(5000, seed=1)
    labels, core, c = knn.build(x).dbscan(np.inf, 10)
    assert c == 1 and core.all() and (labels == 0).all()
    labels, core, c = knn.dbscan(0.05, 5001)
    assert c == 0 and not core.any() and (labels == -1).all()
    labels, core, c = knn.dbscan(0.02, 1)
    assert_same((labels, core, c), DO.dbscan(x, 0.02, 1), "min_pts 1")
    assert core.all()
    x = np.full((1000, 3), 0.5, np.float32)
    assert_same(knn.build(x).dbscan(0.0, 1000), DO.dbscan(x, 0.0, 1000), "identical")


def test_core_flags_equal_range_count(knn, lidar1m):
    for eps, m in ((0.05, 5), (0.3, 20)):
        _, core, _ = knn.build(lidar1m).dbscan(eps, m)
        cnt = knn.range_count(eps)
        assert (core.astype(bool) == (cnt >= m - 1)).all()


def test_deterministic_and_output_kinds(lidar1m):
    import torch

    from owlraytracing_b200 import TrueKNN

    ref = None
    for bps in (0, 1):
        with TrueKNN(0, blocks_per_sm=bps) as t:
            t.build(lidar1m)
            for _ in range(2):
                got = t.dbscan(0.3, 10)
                if ref is None:
                    ref = got
                assert_same(got, ref, f"repeat blocks_per_sm={bps}")
    # device outputs (torch input) and caller-supplied device arrays give the same result
    with TrueKNN(0) as t:
        xd = torch.from_numpy(lidar1m).cuda()
        labels, core, c = t.build(xd).dbscan(0.3, 10)
        assert labels.is_cuda and labels.dtype == torch.int32 and core.dtype == torch.uint8
        assert_same((labels.cpu().numpy(), core.cpu().numpy(), c), ref, "device outputs")
        t.build(lidar1m)
        lab_d = torch.empty(len(lidar1m), dtype=torch.int32, device="cuda")
        labels, core, c = t.dbscan(0.3, 10, out=(lab_d, None))
        assert core is None and c == ref[2] and (labels.cpu().numpy() == ref[0]).all()
        labels, core, c = t.dbscan(0.3, 10, with_core=False)
        assert core is None and (labels == ref[0]).all()


def test_counters_run_is_identical(knn, lidar1m):
    ref = knn.build(lidar1m).dbscan(0.05, 10)
    knn.set_option("counters", 1)
    got = knn.dbscan(0.05, 10)
    assert_same(got, ref, "counters")
    st = knn.stats()
    assert st["nodes_visited"] > 0 and st["points_tested"] > 0 and st["filter_violations"] == 0


def test_errors(knn):
    labels = np.empty(100, np.int32)

    def rc(t, eps, m, lab=labels):
        return t._L.tknn_dbscan(t._h, ctypes.c_float(eps), m, ctypes.c_void_p(lab.ctypes.data) if lab is not None else None,
                                None, None)

    assert rc(knn, 0.1, 5) == _lib.ESTATE  # before a build
    knn.build(datasets.uniform(100, seed=3))
    assert rc(knn, float("nan"), 5) == _lib.EINVAL
    assert rc(knn, -0.1, 5) == _lib.EINVAL
    assert rc(knn, 0.1, 0) == _lib.EINVAL
    assert rc(knn, 0.1, 5, None) == _lib.EINVAL
    assert rc(knn, 0.1, 5) == _lib.OK
    with pytest.raises(TrueKNNError):
        knn.dbscan(-1.0, 5)
    # a rank of a point-partitioned build holds one Morton range of the cloud under global ids: refused
    with MultiTrueKNN([0, 0], "partition") as m:
        m.build(datasets.uniform(4000, seed=4))
        view = m.rank(0)
        assert rc(view, 0.1, 5, np.empty(4000, np.int32)) == _lib.ESTATE


def test_lidar_10m_fullsize(knn):
    x = datasets.lidar_like(10_000_000, seed=7)
    check(knn, x, 0.05, 10, "lidar 10M")
