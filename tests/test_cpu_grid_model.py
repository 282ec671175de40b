"""A numpy model of the cell grid's exactness argument (grid.cuh), checked on the CPU.

This models the kernel; it is not the kernel.  It restates in fp32 the key frame and quantise21 (lbvh.cuh), the frame's
bisected cell boundaries (grid::frame_kernel) and the group's cell range of grid_knn_kernel, and checks the two facts the
grid's exactness rests on:
- every point of cell c lies in [B[c], B[c + 1]];
- for every pair (q, p) with the fp32 dist2(q, p) <= bound, p's cell lies in q's cell range on every axis.
The range formula must be kept in step with grid_knn_kernel by hand.  The kernel itself is compared with the CPU oracle
in test_gpu_grid_oracle.py.
"""
import numpy as np
import pytest
from scipy.spatial import cKDTree

from owlraytracing_b200 import datasets

f32, f64 = np.float32, np.float64
MARGIN = f32(2.0 ** -74)  # the absolute term of the kernel's range: covers the subnormal rounding of dx * dx


def fma32(a, b, c):
    """fmaf(a, b, c) rounded once: a * b is exact in float64, the sum is rounded to odd in float64 (TwoSum), and rounding
    that to float32 gives the correctly rounded result (53 >= 2 * 24 + 2)."""
    p, c = np.asarray(a, f32).astype(f64) * np.asarray(b, f32).astype(f64), np.asarray(c, f32).astype(f64)
    s = p + c
    bb = s - p
    err = (p - (s - bb)) + (c - bb)
    odd = (s.view(np.int64) & 1) == 1
    s = np.where((err != 0) & ~odd, np.nextafter(s, np.where(err > 0, np.inf, -np.inf)), s)
    return s.astype(f32)


def dist2(q, p):
    """common.cuh's dist2: fmaf(dz, dz, fmaf(dy, dy, dx * dx)) in fp32."""
    d = (q - p).astype(f32)
    return fma32(d[..., 2], d[..., 2], fma32(d[..., 1], d[..., 1], d[..., 0] * d[..., 0]))


def key_frame(x):
    lo, hi = x.min(0), x.max(0)
    with np.errstate(over="ignore"):
        ext = max(f32((hi - lo).max()), np.finfo(f32).tiny)
    return lo, hi, f32(f32(2097152.0) / ext)


def cell(v, lo, scale, level):
    """quantise21 >> (21 - level).  fmax / fmin as in CUDA: a frame of scale 0 (an extent that overflows) turns an overflowed
    v - lo into inf * 0 = NaN, which fmaxf maps to cell 0 (np.clip would keep the NaN)."""
    with np.errstate(over="ignore", invalid="ignore"):
        t = ((np.asarray(v, f32) - lo).astype(f32) * scale).astype(f32)
    return np.fmin(np.fmax(t, f32(0)), f32(2097151.0)).astype(np.uint32) >> np.uint32(21 - level)


def _ordered(v):
    b = np.asarray(v, f32).view(np.uint32)
    return np.where(b & 0x80000000, ~b, b | np.uint32(0x80000000)).astype(np.uint32)


def _from_ordered(o):
    o = np.asarray(o, np.uint32)
    return np.where(o & 0x80000000, o & np.uint32(0x7fffffff), ~o).astype(np.uint32).view(f32)


def boundaries(lo, hi, scale, level):
    """frame_kernel along one axis: B[c] = the smallest float in [lo, hi] whose cell is >= c."""
    per = (1 << level) + 1
    c = np.arange(per, dtype=np.uint32)
    top = cell(hi, lo, scale, level)
    olo, ohi = np.full(per, _ordered(lo), np.uint32), np.full(per, _ordered(hi), np.uint32)
    while True:
        live = ohi - olo > 1
        if not live.any():
            break
        mid = olo + (ohi - olo) // 2
        up = cell(_from_ordered(mid), lo, scale, level) >= c
        ohi = np.where(live & up, mid, ohi)
        olo = np.where(live & ~up, mid, olo)
    b = _from_ordered(ohi)
    b = np.where((c == per - 1) | (top < c), hi, b)
    return np.where(c == 0, lo, b).astype(f32), top


def cell_range(qa, bound, lo, scale, level, top, margin=MARGIN):
    """grid_knn_kernel's per-lane range along one axis: s = fma(sqrt(bound), 1.0001, fma(|q|, 2^-18, margin))."""
    s = fma32(np.sqrt(f32(bound)), f32(1.0001), fma32(np.abs(qa), f32(2.0 ** -18), margin))
    return cell((qa - s).astype(f32), lo, scale, level), np.minimum(cell((qa + s).astype(f32), lo, scale, level), top)


def range_misses(x, bound, level, margin=MARGIN):
    """Ordered pairs (q, p), q != p, with dist2(q, p) <= bound whose p lies outside q's cell range on some axis."""
    lo, hi, scale = key_frame(x)
    bound = f32(bound)
    # a superset of the pairs: true distance within sqrt(bound) plus the rounding of dist2, relative and subnormal
    r = np.sqrt((f64(bound) + 2.0 ** -146) * (1 + 2.0 ** -16))
    pairs = cKDTree(x.astype(f64)).query_pairs(r, output_type="ndarray")
    pairs = np.concatenate([pairs, pairs[:, ::-1]])
    q, p = pairs[:, 0], pairs[:, 1]
    within = dist2(x[q], x[p]) <= bound
    q, p = q[within], p[within]
    out = np.zeros(q.shape[0], bool)
    for a in range(3):
        top = cell(hi[a], lo[a], scale, level)
        l, h = cell_range(x[q, a], bound, lo[a], scale, level, top, margin)
        c = cell(x[p, a], lo[a], scale, level)
        out |= (c < l) | (c > h)
    return int(q.shape[0]), int(out.sum())


def quantised(n, seed=1, b=7, dim=3):
    """n distinct points of the 2^-b lattice on [0, 1]^dim with both corners: lo = 0, hi = 1, scale = 2^21 exactly."""
    rng = np.random.default_rng(seed)
    side = 2 ** b + 1
    sites = np.concatenate([[0, side ** dim - 1], 1 + rng.choice(side ** dim - 2, n - 2, replace=False)])
    g = np.stack(np.unravel_index(rng.permutation(sites), (side,) * dim), -1).astype(f32) * f32(2.0 ** -b)
    return np.ascontiguousarray(g)


CLOUDS = {
    "quantised": lambda: (quantised(100_000), 6),
    "quantised_shifted": lambda: ((quantised(100_000) - f32(0.5)).astype(f32), 6),
    "centred_2e-3": lambda: (((datasets.uniform(100_000, seed=5) - f32(0.5)) * f32(2e-3)).astype(f32), 5),
    "lattice": lambda: (datasets.lattice(40), 5),
    "scale_1e-20": lambda: ((datasets.uniform(100_000, seed=3) * f32(1e-20)).astype(f32), 5),
    "scale_1e-21": lambda: ((datasets.uniform(30_000, seed=3) * f32(1e-21)).astype(f32), 5),
    "scale_1e-22": lambda: ((datasets.uniform(2_000, seed=3) * f32(1e-22)).astype(f32), 3),
}


def _bounds(x, k=10):
    """Round-1-like bounds: 0 (a start radius whose square underflows), three times the smallest subnormal, the median k-th
    neighbour d2 (on the lattice exactly a shell's d2: a tie with the bound) and twice that."""
    d = cKDTree(x.astype(f64)).query(x[:2000].astype(f64), k + 1)[0][:, k]
    m = np.median(d) ** 2
    return sorted({f32(0), f32(3 * 2.0 ** -149), f32(m), f32(2 * m)})


@pytest.mark.parametrize("name", list(CLOUDS))
def test_boundaries_bracket_cells(name):
    x, level = CLOUDS[name]()
    lo, hi, scale = key_frame(x)
    for a in range(3):
        B, top = boundaries(lo[a], hi[a], scale, level)
        c = cell(x[:, a], lo[a], scale, level)
        assert (c <= top).all()
        assert (B[c] <= x[:, a]).all() and (x[:, a] <= B[c + 1]).all()
        cs = np.arange(1, top + 1)  # occupied cells above the first: B[c] is the first float of cell >= c
        assert (cell(B[cs], lo[a], scale, level) >= cs).all()
        assert (cell(np.nextafter(B[cs], f32(-np.inf)), lo[a], scale, level) < cs).all()
        assert (B[top + 1:] == hi[a]).all()


@pytest.mark.parametrize("name", list(CLOUDS))
def test_range_covers_every_pair(name):
    x, level = CLOUDS[name]()
    for bound in _bounds(x):
        n_pairs, misses = range_misses(x, bound, level)
        assert misses == 0, (name, bound, n_pairs, misses)


@pytest.mark.parametrize("name", ["scale_1e-21", "scale_1e-22"])
def test_range_without_margin_misses(name):
    """The range without the absolute term (the formula before it was added) misses pairs whose dx * dx underflows: the
    model sees the defect the margin fixes."""
    x, level = CLOUDS[name]()
    n_pairs, misses = range_misses(x, 0.0, level, margin=f32(0))
    assert n_pairs > 0 and misses > 0
