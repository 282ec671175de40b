"""Farthest point sampling without a GPU: the CPU reference of tknn_fps (tests/fps_oracle.c) against a direct restatement
of the contract in exact rational arithmetic on tiny tie-heavy clouds, and against a float64 FPS where every argmax has
a clear margin; the ratio count rule, the random start draw and the batch handling of fps()."""
from fractions import Fraction

import numpy as np
import pytest

import fps_oracle as F
from owlraytracing_b200 import trueknn as T


def f32(fr: Fraction) -> np.float32:
    """fr rounded to the nearest float32, ties to even."""
    c = np.float32(float(fr))
    cands = [np.nextafter(c, np.float32(-np.inf)), c, np.nextafter(c, np.float32(np.inf))]
    best = min(cands, key=lambda v: (abs(Fraction(float(v)) - fr), int(np.array(v).view(np.uint32)) & 1))
    return np.float32(best)


def d2_exact(c, p) -> np.float32:
    """fmaf(dz, dz, fmaf(dy, dy, dx * dx)) in fp32, dx = c - p, each operation rounded once."""
    dx, dy, dz = (np.float32(np.float32(a) - np.float32(b)) for a, b in zip(c, p))
    t = f32(Fraction(float(dx)) ** 2)
    t = f32(Fraction(float(dy)) ** 2 + Fraction(float(t)))
    return f32(Fraction(float(dz)) ** 2 + Fraction(float(t)))


def fps_restated(x, sizes, counts, starts=None):
    x = F._xyz(x)
    off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    idx, d2 = [], []
    for s in range(len(sizes)):
        b, e, m = int(off[s]), int(off[s + 1]), int(counts[s])
        if m == 0:
            continue
        D = {p: np.float32(np.inf) for p in range(b, e)}
        cur = b if starts is None else int(starts[s])
        idx.append(cur)
        d2.append(F.FLT_MAX)
        for _ in range(1, m):
            for p in range(b, e):
                D[p] = min(D[p], d2_exact(x[cur], x[p]))
            cur = max(range(b, e), key=lambda p: (D[p], -p))  # largest D, then the lowest index
            idx.append(cur)
            d2.append(D[cur])
    return np.array(idx, np.int32), np.array(d2, np.float32)


def lattice(k):
    g = np.arange(k, dtype=np.float32)
    return np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3)


TINY = {
    "lattice": (lattice(3) * np.float32(0.5), [27], [27]),
    "identical": (np.full((9, 3), 0.25, np.float32), [9], [9]),
    "duplicates": (np.repeat(np.random.default_rng(1).random((6, 3), dtype=np.float32), 3, axis=0), [18], [18]),
    "collinear": (np.stack([np.arange(12, dtype=np.float32) * np.float32(0.1), np.zeros(12, np.float32),
                            np.zeros(12, np.float32)], 1), [12], [12]),
    "2d": (np.random.default_rng(2).integers(0, 4, (20, 2)).astype(np.float32), [20], [15]),
    "batch": (np.concatenate([lattice(2), np.zeros((0, 3), np.float32), np.full((5, 3), 1.0, np.float32),
                              np.random.default_rng(3).random((7, 3), dtype=np.float32)]), [8, 0, 5, 7], [8, 0, 4, 1]),
    "uniform": (np.random.default_rng(4).random((40, 3), dtype=np.float32), [40], [40]),
}


@pytest.mark.parametrize("name", sorted(TINY))
@pytest.mark.parametrize("with_starts", [False, True])
def test_oracle_matches_restatement(name, with_starts):
    x, sizes, counts = TINY[name]
    off = F.offsets_of(sizes)
    starts = None
    if with_starts:
        rng = np.random.default_rng(5)
        starts = np.array([int(off[s]) + int(rng.integers(0, max(n, 1))) for s, n in enumerate(sizes)], np.int32)
    want_i, want_d = fps_restated(x, sizes, counts, starts)
    got_i, got_d = F.fps(x, off, counts, starts)
    np.testing.assert_array_equal(got_i, want_i)
    np.testing.assert_array_equal(got_d.view(np.uint32), want_d.view(np.uint32))


def test_duplicates_repeat_lowest_index():
    x = np.repeat(np.array([[0, 0, 0], [1, 0, 0]], np.float32), 3, axis=0)  # two locations, three copies each
    idx, d = F.fps(x, counts=[6], starts=[4])
    assert list(idx[:2]) == [4, 0]  # the farthest location, lowest index
    assert list(idx[2:]) == [0, 0, 0, 0]  # every D is 0: the lowest index again
    assert (d[2:] == 0).all()


def test_distinct_full_permutation_and_prefix():
    x = np.random.default_rng(6).random((500, 3), dtype=np.float32)
    idx, d = F.fps(x, counts=[500], squared=False)
    assert sorted(idx.tolist()) == list(range(500))
    assert (np.diff(d[1:]) <= 0).all()
    pi, pd = F.fps(x, counts=[500], limit=37, squared=False)
    np.testing.assert_array_equal(pi[:37], idx[:37])
    np.testing.assert_array_equal(pd[:37].view(np.uint32), d[:37].view(np.uint32))
    assert (pi[37:] == -1).all()


def fps64(x, m, start):
    """float64 FPS with the smallest relative gap between the winner and the runner-up of every step"""
    x = x.astype(np.float64)
    D = np.full(x.shape[0], np.inf)
    cur, out, margin = start, [start], np.inf
    for _ in range(1, m):
        D = np.minimum(D, ((x - x[cur]) ** 2).sum(1))
        order = np.argsort(-D, kind="stable")
        margin = min(margin, (D[order[0]] - D[order[1]]) / D[order[0]])
        cur = int(order[0])
        out.append(cur)
    return np.array(out, np.int32), margin


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_oracle_matches_float64_where_margins_are_clear(seed):
    rng = np.random.default_rng(seed)
    x = rng.random((3000, 3), dtype=np.float32) * np.float32(10)
    want, margin = fps64(x, 200, 7)
    assert margin > 2.0 ** -20, "the cloud has a near tie; pick another seed"
    got, d2 = F.fps(x, counts=[200], starts=[7])
    np.testing.assert_array_equal(got, want)
    exact = ((x[got[1:]].astype(np.float64)[:, None] - x.astype(np.float64)[None, got[:-1]]) ** 2).sum(-1)
    ref = np.array([exact[i, : i + 1].min() for i in range(exact.shape[0])])
    np.testing.assert_allclose(d2[1:], ref, rtol=1e-6)


def test_count_rule():
    sizes = np.array([0, 1, 2, 3, 7, 64, 4096, 120000, 16777217], np.int64)
    for ratio in (0.25, 0.5, 1.0 / 16, 0.3, 1.0, 1e-9):
        want = np.ceil(sizes.astype(np.float32) * np.float32(ratio)).astype(np.int64)
        got = T.fps_counts(sizes, ratio)
        np.testing.assert_array_equal(got, np.minimum(want, sizes))
    assert T.fps_counts([0], 0.5)[0] == 0
    assert T.fps_counts([4096], 0.25)[0] == 1024
    for bad in (0.0, -0.1, 1.5, float("nan")):
        with pytest.raises(ValueError):
            T.fps_counts([10], bad)
    with pytest.raises(ValueError):
        T.fps(np.zeros((0, 3), np.float32), ratio=2.0)
    assert T.fps(np.zeros((0, 3), np.float32)).shape == (0,)


def test_count_rule_matches_torch():
    torch = pytest.importorskip("torch")
    sizes = np.array([0, 1, 5, 1000, 4097, 120001], np.int64)
    for ratio in (0.25, 0.1, 1.0 / 3):
        want = torch.ceil(torch.tensor(sizes).float() * ratio).long().numpy()
        np.testing.assert_array_equal(T.fps_counts(sizes, ratio), want)


def test_random_starts_numpy():
    off = np.array([0, 10, 10, 11, 1000], np.int64)
    np.random.seed(0)
    a = T.fps_random_starts(off)
    np.random.seed(0)
    b = T.fps_random_starts(off)
    np.testing.assert_array_equal(a, b)
    assert a.dtype == np.int32 and a.shape == (4,)
    for s in range(4):
        assert off[s] <= a[s] < max(off[s + 1], off[s] + 1)
    draws = np.stack([T.fps_random_starts(off) for _ in range(200)])
    assert len(set(draws[:, 3].tolist())) > 50  # spread over the large cloud


def test_batch_offsets_for_fps():
    batch = np.array([0, 0, 2, 2, 2], np.int64)
    off = T.batch_to_offsets(batch, 5, 4)
    np.testing.assert_array_equal(off, [0, 2, 2, 5, 5])
    np.testing.assert_array_equal(T.fps_counts(np.diff(off.astype(np.int64)), 0.5), [1, 0, 2, 0])
