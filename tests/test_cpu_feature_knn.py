"""The CPU reference of tknn_feature_knn (tests/feature_knn_oracle.py) checked without a GPU: bit for bit against the
3-D reference of segmented query sets at f = 3 (and f = 2 with a zero z column), against a float64 ranking on tie-free
data, and on exact ties and overflow, where the (d2, index) key decides.  Also the argument checks of the Python layer
that run before any device is touched."""
import numpy as np
import pytest

import feature_knn_oracle as FK
import segment_query_oracle as SQ


def same(a, b, what):
    (ai, ad), (bi, bd) = a, b
    bad = np.argwhere(ai != bi)
    assert bad.size == 0, f"{what}: {len(bad)} indices differ, first at {tuple(bad[0])}"
    bad = np.argwhere(ad.view(np.uint32) != bd.view(np.uint32))
    assert bad.size == 0, f"{what}: {len(bad)} distances differ, first at {tuple(bad[0])}"


def clouds(kind, rng):
    x_sizes = [300, 0, 1, 7, 250, 40]
    y_sizes = [120, 5, 3, 0, 90, 60]
    if kind == "uniform":
        x = rng.random((sum(x_sizes), 3), dtype=np.float32)
        y = rng.random((sum(y_sizes), 3), dtype=np.float32)
    else:  # duplicate-heavy: few distinct positions on a coarse lattice
        x = (rng.integers(0, 4, (sum(x_sizes), 3)) * 0.25).astype(np.float32)
        y = (rng.integers(0, 4, (sum(y_sizes), 3)) * 0.25).astype(np.float32)
    return x, y, SQ.offsets_of(x_sizes), SQ.offsets_of(y_sizes)


@pytest.mark.parametrize("kind", ["uniform", "duplicates"])
@pytest.mark.parametrize("k", [1, 8, 33])
def test_f3_equals_segment_query_reference(oracle, kind, k):
    rng = np.random.default_rng(7)
    x, y, xo, yo = clouds(kind, rng)
    sid = rng.integers(-1, len(x), size=len(y)).astype(np.int32)
    sid[:50] = np.arange(50)  # rows of segment 0 excluding a point of their own segment
    want = SQ.knn(x, y, xo, yo, k, self_ids=sid, squared=True)
    got = FK.knn(x, y, k, xo, yo, self_ids=sid)
    same(got, want, f"{kind} k={k}")
    # sqrtf form
    same(FK.knn(x, y, k, xo, yo, self_ids=sid, squared=False), SQ.knn(x, y, xo, yo, k, self_ids=sid), f"{kind} sqrt")


def test_f3_all_points_single_segment(oracle):
    rng = np.random.default_rng(8)
    x = rng.random((2000, 3), dtype=np.float32)
    want = SQ.knn(x, x, [0, 2000], [0, 2000], 10, self_ids=np.arange(2000, dtype=np.int32), squared=True)
    same(FK.knn(x, x, 10, self_ids=np.arange(2000)), want, "all points")


def test_f2_equals_zero_z(oracle):
    rng = np.random.default_rng(9)
    x, y, xo, yo = clouds("uniform", rng)
    x2, y2 = np.ascontiguousarray(x[:, :2]), np.ascontiguousarray(y[:, :2])
    want = SQ.knn(x2, y2, xo, yo, 12, squared=True)  # the 2-D path pads z = 0
    same(FK.knn(x2, y2, 12, xo, yo), want, "f = 2")
    same(FK.knn(x, y, 12, xo, yo, f=2), want, "f = 2 through the pitch")


@pytest.mark.parametrize("f", [1, 5, 64, 130])
def test_order_matches_float64_on_tie_free_data(f):
    rng = np.random.default_rng(f)
    x = rng.standard_normal((400, f)).astype(np.float32)
    y = rng.standard_normal((50, f)).astype(np.float32)
    k = 16
    idx, d2 = FK.knn(x, y, k)
    ref = ((y.astype(np.float64)[:, None, :] - x.astype(np.float64)[None, :, :]) ** 2).sum(-1)
    order = np.argsort(ref, axis=1, kind="stable")[:, :k]
    srt = np.sort(ref, axis=1)
    # rows whose k+1 smallest float64 distances are well separated have one right answer
    gaps = np.diff(srt[:, : k + 1], axis=1) / srt[:, 1: k + 1]
    clear = (gaps > 1e-4).all(axis=1)
    assert clear.sum() > 20
    assert (idx[clear] == order[clear]).all()
    assert np.allclose(d2, np.take_along_axis(ref, idx.astype(np.int64), 1), rtol=1e-4)
    assert (np.diff(d2, axis=1) >= 0).all()


def test_integer_features_ties_by_index():
    rng = np.random.default_rng(3)
    x = rng.integers(-2, 3, (600, 8)).astype(np.float32)
    y = rng.integers(-2, 3, (40, 8)).astype(np.float32)
    k = 40
    idx, d2 = FK.knn(x, y, k)
    exact = ((y.astype(np.int64)[:, None, :] - x.astype(np.int64)[None, :, :]) ** 2).sum(-1)  # exact in fp32 too
    for j in range(len(y)):
        want = sorted(range(len(x)), key=lambda p: (exact[j, p], p))[:k]
        assert list(idx[j]) == want
        assert (d2[j] == exact[j, want]).all()


def test_overflow_gives_inf_ordered_by_index():
    rng = np.random.default_rng(4)
    x = (rng.random((64, 6), dtype=np.float32) - 0.5) * np.float32(4e20)
    y = (rng.random((5, 6), dtype=np.float32) - 0.5) * np.float32(4e20)
    idx, d2 = FK.knn(x, y, 10)
    assert np.isinf(d2).all()
    assert (idx == np.arange(10)).all()
    _, dist = FK.knn(x, y, 10, squared=False)
    assert np.isinf(dist).all()


def test_short_rows_padding_and_self():
    x = np.arange(12, dtype=np.float32).reshape(4, 3)
    idx, d2 = FK.knn(x, x, 5, self_ids=np.array([0, -1, 7, 3]))
    assert list(idx[0]) == [1, 2, 3, -1, -1] and d2[0, 3] == FK.FLT_MAX
    assert list(idx[1]) == [1, 0, 2, 3, -1] and d2[1, 0] == 0
    assert list(idx[2]) == [2, 1, 3, 0, -1]
    assert list(idx[3]) == [2, 1, 0, -1, -1]


def test_python_argument_checks():
    from owlraytracing_b200 import TrueKNN, feature_knn, feature_knn_graph

    t = TrueKNN.__new__(TrueKNN)  # argument checks run before any library call
    import torch

    with pytest.raises(TypeError):
        t.feature_knn(torch.zeros((4, 8), dtype=torch.float64), torch.zeros((4, 8), dtype=torch.float64), 2)
    with pytest.raises(TypeError):
        t.feature_knn(torch.zeros((4, 8), dtype=torch.float16), torch.zeros((4, 8), dtype=torch.float16), 2)
    with pytest.raises(ValueError):
        t.feature_knn(np.zeros((4, 8), np.float32), np.zeros((4, 7), np.float32), 2)
    assert feature_knn(np.zeros((0, 8), np.float32), np.zeros((3, 8), np.float32), 4).shape == (2, 0)
    assert feature_knn(np.zeros((3, 8), np.float32), np.zeros((0, 8), np.float32), 4).shape == (2, 0)
    assert feature_knn_graph(np.zeros((0, 8), np.float32), 4).shape == (2, 0)
