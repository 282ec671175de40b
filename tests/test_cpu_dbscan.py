"""The DBSCAN reference (tests/dbscan_oracle.c) against the contract and against scikit-learn, on the CPU.

The contract (include/trueknn.h, tknn_dbscan): closed fp32 eps-ball under d2 = fmaf(dz,dz,fmaf(dy,dy,dx*dx)),
core iff the ball holds >= min_pts points (the point itself included), clusters = components of the core points
numbered by smallest core index, border = lowest cluster id among the core points of the ball, noise = -1.
"""
import numpy as np
import pytest
from scipy.sparse import csr_matrix
from scipy.sparse.csgraph import connected_components
from scipy.spatial import cKDTree

import dbscan_oracle as DO
from owlraytracing_b200 import datasets


def _fmaf(a, b, c):
    # a*b is exact in float64 (24 x 24 bits); the sum then rounds twice (float64, float32), which differs from one
    # rounding only when the float64 result lands exactly on a float32 midpoint (probability ~2^-29 per operation)
    return (a.astype(np.float64) * b.astype(np.float64) + c.astype(np.float64)).astype(np.float32)


def d2_matrix(x):
    """All-pairs d2 of the project's distance rule, fp32."""
    x = np.asarray(x, np.float32)
    d = x[:, None, :] - x[None, :, :]  # fp32 subtraction, round to nearest
    dx, dy, dz = d[..., 0], d[..., 1], d[..., 2]
    return _fmaf(dz, dz, _fmaf(dy, dy, dx * dx))


def dbscan_brute(x, eps, min_pts):
    """The contract restated on the full d2 matrix (small clouds only)."""
    n = len(x)
    eps2 = np.float32(eps) * np.float32(eps)
    ball = d2_matrix(x) <= eps2
    core = ball.sum(1) >= min_pts
    ci = np.flatnonzero(core)
    labels = np.full(n, -1, np.int32)
    n_clusters = 0
    if ci.size:
        _, comp = connected_components(csr_matrix(ball[np.ix_(ci, ci)]), directed=False)
        first = {}
        for i, cc in zip(ci, comp):  # ci ascending: the first member seen is the smallest core index
            if cc not in first:
                first[cc] = len(first)
            labels[i] = first[cc]
        n_clusters = len(first)
    for i in np.flatnonzero(~core):
        ids = labels[ball[i] & core]
        if ids.size:
            labels[i] = ids.min()
    return labels, core.astype(np.uint8), n_clusters


def assert_same(got, want, what=""):
    gl, gc, gn = got
    wl, wc, wn = want
    assert gn == wn, f"{what}: {gn} clusters, want {wn}"
    bad = np.flatnonzero(gc != wc)
    assert bad.size == 0, f"{what}: core flags differ at {bad[:10]}"
    bad = np.flatnonzero(gl != wl)
    assert bad.size == 0, f"{what}: labels differ at {bad[:10]}: {gl[bad[:10]]} vs {wl[bad[:10]]}"


def _rng(seed):
    return np.random.default_rng(seed)


CASES = {
    "uniform": lambda: (_rng(1).random((800, 3)).astype(np.float32), 0.08, 5),
    "clustered": lambda: (np.concatenate([_rng(2).normal(c, 0.03, (120, 3)) for c in _rng(3).random((6, 3)) * 0.5])
                          .astype(np.float32), 0.03, 6),
    # coordinates on a 1/16 grid: many pair distances equal eps exactly (closed ball), many equal distances
    "ties": lambda: ((np.round(_rng(4).random((700, 3)) * 16) / 16).astype(np.float32), 0.125, 8),
    "duplicates": lambda: (np.repeat(_rng(5).random((60, 3)).astype(np.float32), 7, axis=0)[_rng(6).permutation(420)],
                           0.05, 9),
    "identical": lambda: (np.full((300, 3), 0.25, np.float32), 0.0, 300),
    "identical_too_few": lambda: (np.full((300, 3), 0.25, np.float32), 0.0, 301),
    "min_pts_1": lambda: (_rng(7).random((500, 3)).astype(np.float32), 0.05, 1),
    "eps_0": lambda: (np.concatenate([_rng(8).random((300, 3)), _rng(8).random((100, 3))]).astype(np.float32), 0.0, 2),
    "eps_inf": lambda: (_rng(9).random((400, 3)).astype(np.float32), np.inf, 10),
    "eps_inf_too_few": lambda: (_rng(9).random((40, 3)).astype(np.float32), np.inf, 41),
    "planar": lambda: (np.concatenate([_rng(10).random((600, 2)), np.zeros((600, 1))], 1).astype(np.float32), 0.04, 4),
}


@pytest.mark.parametrize("case", sorted(CASES))
def test_oracle_matches_brute_force(case):
    x, eps, m = CASES[case]()
    got = DO.dbscan(x, eps, m)
    assert_same(got, dbscan_brute(x, eps, m), case)


def test_special_cases_have_the_expected_shape():
    x, _, _ = CASES["identical"]()
    labels, core, c = DO.dbscan(x, 0.0, 300)
    assert c == 1 and core.all() and (labels == 0).all()
    labels, core, c = DO.dbscan(x, 0.0, 301)
    assert c == 0 and not core.any() and (labels == -1).all()
    x, _, _ = CASES["eps_inf"]()
    labels, core, c = DO.dbscan(x, np.inf, 10)
    assert c == 1 and core.all() and (labels == 0).all()
    x, _, _ = CASES["min_pts_1"]()
    labels, core, c = DO.dbscan(x, 0.05, 1)
    assert core.all() and labels.min() == 0 and labels.max() == c - 1


def clean_eps(x, candidates, rel=2.0 ** -20):
    """The first eps of `candidates` such that no pair distance (float64) lies within rel of it."""
    t = cKDTree(np.asarray(x, np.float64))
    for eps in candidates:
        lo = t.count_neighbors(t, eps * (1 - rel))
        hi = t.count_neighbors(t, eps * (1 + rel))
        if lo == hi:
            return eps
    raise AssertionError("every candidate eps has a pair distance near it")


def overlapping(seed, n_per=250, k=10):
    r = _rng(seed)
    return np.concatenate([r.normal(c, 0.03, (n_per, 3)) for c in r.random((k, 3)) * 0.4]).astype(np.float32)


SK_CASES = {
    "uniform": (lambda: datasets.uniform(4000, seed=42), [0.05, 0.051, 0.052], 5),
    "lidar_like": (lambda: datasets.lidar_like(5000, seed=7), [1.5, 1.51, 1.52], 10),
    "overlapping": (lambda: overlapping(11), [0.03, 0.0301, 0.0302], 8),
    "overlapping_dense": (lambda: overlapping(12, 400, 6), [0.02, 0.0201, 0.0202], 20),
}


@pytest.mark.parametrize("case", sorted(SK_CASES))
def test_oracle_matches_sklearn(case):
    from sklearn.cluster import DBSCAN

    make, candidates, m = SK_CASES[case]
    x = make()
    eps = clean_eps(x, candidates)
    labels, core, c = DO.dbscan(x, eps, m)
    sk = DBSCAN(eps=eps, min_samples=m).fit(x.astype(np.float64))
    sk_core = np.zeros(len(x), np.uint8)
    sk_core[sk.core_sample_indices_] = 1
    assert (core == sk_core).all(), case
    assert (labels == sk.labels_).all(), case
    assert c == sk.labels_.max() + 1
    assert c > 1 and (labels == -1).any() and ((labels >= 0) & (core == 0)).any(), "the case should exercise every kind"


def lattice_roles(m):
    """Interior / face-interior / edge-or-corner masks of the m^3 lattice (datasets.lattice order)."""
    g = datasets.lattice(m).astype(np.int64)
    on_face = ((g == 0) | (g == m - 1)).sum(1)
    return on_face == 0, on_face == 1, on_face >= 2


def test_lattice_closed_ball():
    m = 6
    x = datasets.lattice(m)
    interior, face, edge = lattice_roles(m)
    labels, core, c = DO.dbscan(x, 1.0, 7)  # distance exactly 1 is inside: 6 neighbours + the point itself
    assert c == 1
    assert (core.astype(bool) == interior).all()
    assert (labels[interior] == 0).all() and (labels[face] == 0).all()  # face-interior points are border points
    assert (labels[edge] == -1).all()
    assert_same((labels, core, c), dbscan_brute(x, 1.0, 7), "lattice")
    labels, core, c = DO.dbscan(x, float(np.nextafter(np.float32(1), np.float32(0))), 7)
    assert c == 0 and not core.any() and (labels == -1).all()
