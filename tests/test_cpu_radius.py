"""The fixed-radius neighbour-list reference (tests/radius_oracle.c) against the contract and against scipy, and the
neighbour-list writer of libtrueknn, on the CPU.

The contract (include/trueknn.h, tknn_radius_search / tknn_radius_query): the row of q holds every data point p with
index(p) != self(q) and d2(q, p) <= fl(r * r) under d2 = fmaf(dz,dz,fmaf(dy,dy,dx*dx)) in fp32, sorted by (d2, index).
"""
import ctypes
import os

import numpy as np
import pytest
from scipy.spatial import cKDTree

import radius_oracle as RO
from owlraytracing_b200 import _lib, datasets, write_neighbour_lists


def _fmaf(a, b, c):
    # a*b is exact in float64 (24 x 24 bits); the sum then rounds twice (float64, float32), which differs from one
    # rounding only when the float64 result lands exactly on a float32 midpoint (probability ~2^-29 per operation)
    return (a.astype(np.float64) * b.astype(np.float64) + c.astype(np.float64)).astype(np.float32)


def _pad3(x):
    x = np.asarray(x, np.float32)
    return x if x.shape[1] == 3 else np.concatenate([x, np.zeros((x.shape[0], 1), np.float32)], 1)


def lists_brute(x, r, queries=None, self_ids=None):
    """The contract restated on the full query x data d2 matrix (small clouds only)."""
    x = _pad3(x)
    q = x if queries is None else _pad3(queries)
    sid = np.arange(len(x)) if queries is None else (np.full(len(q), -1) if self_ids is None else np.asarray(self_ids))
    d = q[:, None, :] - x[None, :, :]  # fp32 subtraction, round to nearest
    dx, dy, dz = d[..., 0], d[..., 1], d[..., 2]
    d2 = _fmaf(dz, dz, _fmaf(dy, dy, dx * dx))
    r2 = np.float32(np.float32(r) * np.float32(r))
    inball = d2 <= r2
    inball[np.arange(len(q))[sid >= 0], sid[sid >= 0]] = False
    off = [0]
    idx, dd = [], []
    for i in range(len(q)):
        j = np.flatnonzero(inball[i])
        keys = (d2[i, j].view(np.uint32).astype(np.uint64) << np.uint64(32)) | j.astype(np.uint64)
        o = np.argsort(keys, kind="stable")
        idx.append(j[o].astype(np.int32))
        dd.append(d2[i, j][o])
        off.append(off[-1] + len(j))
    return np.asarray(off, np.int64), np.concatenate(idx), np.concatenate(dd).astype(np.float32)


def assert_same(got, want, what=""):
    go, gi, gd = got
    wo, wi, wd = want
    assert (go == wo).all(), f"{what}: offsets differ at rows {np.flatnonzero(go != wo)[:10]}"
    assert (gi == wi).all(), f"{what}: indices differ at {np.flatnonzero(gi != wi)[:10]}"
    assert (np.asarray(gd, np.float32).view(np.uint32) == np.asarray(wd, np.float32).view(np.uint32)).all(), \
        f"{what}: d2 bits differ at {np.flatnonzero(gd != wd)[:10]}"


def _rng(seed):
    return np.random.default_rng(seed)


CASES = {
    "uniform": lambda: (_rng(1).random((900, 3)).astype(np.float32), 0.09),
    # coordinates on a 1/16 grid: many pair distances equal r exactly (closed ball), many equal distances
    "ties": lambda: ((np.round(_rng(4).random((700, 3)) * 16) / 16).astype(np.float32), 0.125),
    "duplicates": lambda: (np.repeat(_rng(5).random((60, 3)).astype(np.float32), 7, axis=0)[_rng(6).permutation(420)], 0.05),
    "collinear": lambda: (np.stack([_rng(7).random(500), np.zeros(500), np.zeros(500)], 1).astype(np.float32), 0.01),
    "planar": lambda: (_rng(10).random((600, 2)).astype(np.float32), 0.05),
    "r_0": lambda: (np.repeat(_rng(8).random((100, 3)).astype(np.float32), 3, axis=0), 0.0),
    "r_inf": lambda: (_rng(9).random((300, 3)).astype(np.float32), np.inf),
    "lattice_r1": lambda: (datasets.lattice(7), 1.0),
    "lattice_below_1": lambda: (datasets.lattice(7), float(np.nextafter(np.float32(1), np.float32(0)))),
}


@pytest.mark.parametrize("case", sorted(CASES))
def test_oracle_matches_brute_force(case):
    x, r = CASES[case]()
    assert_same(RO.radius_lists(x, r), lists_brute(x, r), case)


def test_query_form_matches_brute_force():
    x = _rng(11).random((800, 3)).astype(np.float32)
    q = np.concatenate([x[:100] + np.float32(0.001), _rng(12).random((200, 3)).astype(np.float32) + np.float32(3.0)])
    q = q.astype(np.float32)
    r = 0.08
    # self ids: -1, the data point next to the query (inside the ball) and far points (outside it)
    sid = np.full(len(q), -1, np.int32)
    sid[:50] = np.arange(50)
    sid[50:100] = np.arange(700, 750)
    sid[100:150] = np.arange(150)[:50]
    assert_same(RO.radius_lists(x, r, q, sid), lists_brute(x, r, q, sid), "query form")
    assert_same(RO.radius_lists(x, r, q), lists_brute(x, r, q), "query form, no self ids")
    off, _, _ = RO.radius_lists(x, r, q, sid)
    assert (np.diff(off)[100:] == 0).all(), "far queries have empty rows"


def test_lattice_has_six_neighbours_in_index_order():
    m = 7
    x = datasets.lattice(m)
    g = x.astype(np.int64)
    interior = ((g > 0) & (g < m - 1)).all(1)
    off, idx, d2 = RO.radius_lists(x, 1.0)
    lens = np.diff(off)
    assert (lens[interior] == 6).all()
    for q in np.flatnonzero(interior)[:50]:
        row = idx[off[q]:off[q + 1]]
        assert (np.diff(row) > 0).all() and (d2[off[q]:off[q + 1]] == 1.0).all()
    off, _, _ = RO.radius_lists(x, float(np.nextafter(np.float32(1), np.float32(0))))
    assert off[-1] == 0


def test_r0_keeps_only_duplicates_and_inf_keeps_everything():
    x, _ = CASES["r_0"]()
    off, idx, d2 = RO.radius_lists(x, 0.0)
    assert (np.diff(off) == 2).all() and (d2 == 0).all()
    x, _ = CASES["r_inf"]()
    off, idx, _ = RO.radius_lists(x, np.inf)
    assert (np.diff(off) == len(x) - 1).all()


def clean_radius(x, candidates, rel=2.0 ** -20):
    """The first r of `candidates` such that no pair distance (float64) lies within rel of it."""
    t = cKDTree(np.asarray(x, np.float64))
    for r in candidates:
        if t.count_neighbors(t, r * (1 - rel)) == t.count_neighbors(t, r * (1 + rel)):
            return r
    raise AssertionError("every candidate radius has a pair distance near it")


@pytest.mark.parametrize("cloud", ["uniform", "lidar"])
def test_row_sets_equal_scipy(cloud):
    x = _rng(13).random((20000, 3)).astype(np.float32) if cloud == "uniform" else datasets.lidar_like(20000, seed=7)
    r = clean_radius(x, [0.03, 0.031, 0.029, 0.0305] if cloud == "uniform" else [0.05, 0.051, 0.049])
    off, idx, _ = RO.radius_lists(x, r)
    ref = cKDTree(x.astype(np.float64)).query_ball_point(x.astype(np.float64), r, return_sorted=True)
    for q in range(len(x)):
        want = sorted(set(ref[q]) - {q})
        assert sorted(idx[off[q]:off[q + 1]].tolist()) == want, (cloud, q)


def _lists(seed=14):
    rng = _rng(seed)
    lens = rng.integers(0, 6, 300)
    lens[:3] = 0
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    idx = rng.integers(0, 1 << 30, off[-1]).astype(np.int32)
    dist = rng.random(off[-1]).astype(np.float32)
    return off, idx, dist


def test_writer_text_reads_back(tmp_path):
    off, idx, dist = _lists()
    p = str(tmp_path / "nn.csv")
    write_neighbour_lists(p, off, idx, dist)
    rows = np.loadtxt(p, delimiter=",", dtype=np.float64, ndmin=2)
    assert rows.shape == (off[-1], 3)
    assert (rows[:, 0].astype(np.int64) == np.repeat(np.arange(len(off) - 1), np.diff(off))).all()
    assert (rows[:, 1].astype(np.int64) == idx).all()
    assert (rows[:, 2].astype(np.float32) == dist).all()  # %.9g round-trips every float32
    p2 = str(tmp_path / "nn_idx.csv")
    write_neighbour_lists(p2, off, idx, None)
    rows = np.loadtxt(p2, delimiter=",", dtype=np.int64, ndmin=2)
    assert rows.shape == (off[-1], 2) and (rows[:, 1] == idx).all()


def test_writer_binary_reads_back(tmp_path):
    off, idx, dist = _lists()
    p = str(tmp_path / "nn")
    write_neighbour_lists(p, off, idx, dist, binary=True)
    assert (np.fromfile(p + ".off.u64", np.uint64) == off.astype(np.uint64)).all()
    assert (np.fromfile(p + ".idx.i32", np.int32) == idx).all()
    assert (np.fromfile(p + ".dist.f32", np.float32).view(np.uint32) == dist.view(np.uint32)).all()


def test_writer_empty_and_bad_arguments(tmp_path):
    L = _lib.load()  # loads without a device
    off = np.zeros(5, np.uint64)
    p = str(tmp_path / "empty.csv")
    assert L.tknn_write_neighbour_lists(p.encode(), ctypes.c_void_p(off.ctypes.data), None, None, 4, 0) == _lib.OK
    assert os.path.getsize(p) == 0
    assert L.tknn_write_neighbour_lists(p.encode(), None, None, None, 4, 0) == _lib.EINVAL
    off[-1] = 3
    assert L.tknn_write_neighbour_lists(p.encode(), ctypes.c_void_p(off.ctypes.data), None, None, 4, 0) == _lib.EINVAL
