"""A numpy model of the point-partitioned driver's boundary-query routing (dist.cu, brute::reach_mask_of), on the CPU.

This models the kernels; it is not the kernels, and it must be kept in step with them by hand.  It restates in fp32:
- the global frame and scale of lbvh::morton_kernel, and partition_build's cell-aligned split of the Morton order into
  ranks (rank r starts at the first of the 256^3 cells whose exclusive prefix count reaches r * n / ranks);
- the 8 x 8 x 8 summary cells of cell_boxes_kernel and every rank's tight box inside each of them;
- reach_mask_of: rho = fma(sqrt_ru(r2), 1.000001, 2^-74), the outward-rounded cell range [c0, c1] and the box test
  against lim = fma(r2, 1e-5, r2) + 1e-30.  The box sum is taken in two fp32 evaluation orders (plain, and the fma
  chain of dist2) and must pass in both, so the model never flags a rank the kernel would not.
It checks the fact the driver's exactness rests on: for every owned query q with r2 = the k-th d2 over its own rank's
other points, every point p of another rank with the fp32 dist2(q, p) <= r2 lies in a summary cell inside [c0, c1] on
every axis, and the box of p's rank in that cell passes the lim test — so p's rank is asked.  The driver itself is
compared with the CPU oracle in test_gpu_multi_oracle.py, which also checks that this split is the driver's.
"""
import numpy as np
import pytest

import extreme_clouds as E
from owlraytracing_b200 import datasets
from test_cpu_grid_model import dist2, fma32

f32, f64 = np.float32, np.float64
MARGIN = f32(2.0 ** -74)  # the absolute term of rho: covers the subnormal rounding of da * da
SUMMARY_BITS = 3          # dist.cu SUMMARY_AXIS_BITS
SPLIT_BITS = 8            # dist.cu CELL_BITS / 3: splitters fall on the 256^3 grid


def frame(x):
    """(lo [3], hi [3], scale) of morton_kernel on the global box; 2-D clouds get z = 0."""
    x = E.xyz3(x)
    lo, hi = x.min(0), x.max(0)
    with np.errstate(over="ignore"):
        ext = max(f32(np.max((hi - lo).astype(f32))), np.finfo(f32).tiny)
    return lo, hi, f32(f32(2097152.0) / ext)


def quantise(v, lo, scale):
    """quantise21: fminf(fmaxf((v - lo) * scale, 0), 2^21 - 1) -> uint32; fmaxf drops the NaN of inf * 0."""
    with np.errstate(over="ignore", invalid="ignore"):
        t = ((np.asarray(v, f32) - f32(lo)).astype(f32) * scale).astype(f32)
    return np.fmin(np.fmax(t, f32(0)), f32(2097151.0)).astype(np.uint32)


def interleave(c, bits):
    """Morton interleave of per-axis cell coordinates [m, 3], x bit highest at every level."""
    out = np.zeros(c.shape[0], np.int64)
    for b in range(bits):
        for a in range(3):
            out |= ((c[:, a].astype(np.int64) >> b) & 1) << (3 * b + 2 - a)
    return out


def cells(x, fr, bits):
    lo, _, scale = fr
    x = E.xyz3(x)
    return np.stack([quantise(x[:, a], lo[a], scale) >> np.uint32(21 - bits) for a in range(3)], 1)


def split(x, ranks):
    """partition_build's owner of every point, or None when some rank would own fewer than 2 points (TKNN_EINVAL)."""
    fr = frame(x)
    c = np.sort(interleave(cells(x, fr, SPLIT_BITS), SPLIT_BITS))
    n = len(c)
    # rank r starts at the first cell whose exclusive prefix reaches n r / ranks: just past the cell of point target - 1
    sp = np.array([0 if n * r // ranks == 0 else c[n * r // ranks - 1] + 1 for r in range(1, ranks)], np.int64)
    owner = np.searchsorted(sp, interleave(cells(x, fr, SPLIT_BITS), SPLIT_BITS), side="right")
    return None if np.bincount(owner, minlength=ranks).min() < 2 else owner


def summaries(x, owner, ranks, fr):
    """cell_boxes_kernel: [ranks, 512, 6] tight boxes (min xyz, max xyz); an empty cell is (+inf, -inf)."""
    x = E.xyz3(x)
    cell = interleave(cells(x, fr, SUMMARY_BITS), SUMMARY_BITS)
    summ = np.empty((ranks, 1 << (3 * SUMMARY_BITS), 6), f32)
    summ[..., :3], summ[..., 3:] = np.inf, -np.inf
    np.minimum.at(summ[..., :3], (owner, cell), x)
    np.maximum.at(summ[..., 3:], (owner, cell), x)
    return summ, cell


def _round_sum(a, b, up):
    """a + b rounded to fp32 toward +inf (up) or -inf: TwoSum in float64 gives the exact sum as s + e."""
    a, b = np.asarray(a, f32).astype(f64), np.asarray(b, f32).astype(f64)
    s = a + b
    bb = s - a
    e = (a - (s - bb)) + (b - bb)
    y = s.astype(f32)
    yd = y.astype(f64)
    if up:
        low = (yd < s) | ((yd == s) & (e > 0))
        return np.where(low, np.nextafter(y, f32(np.inf)), y).astype(f32)
    high = (yd > s) | ((yd == s) & (e < 0))
    return np.where(high, np.nextafter(y, f32(-np.inf)), y).astype(f32)


def sqrt_ru(r2):
    r2 = np.asarray(r2, f32)
    s = np.sqrt(r2)
    low = np.isfinite(s) & (s.astype(f64) * s.astype(f64) < r2.astype(f64))
    return np.where(low, np.nextafter(s, f32(np.inf)), s).astype(f32)


def reach_range(q, r2, fr, margin=MARGIN):
    """reach_mask_of's cell range [c0, c1] per axis, [m, 3] each; margin 0 is the formula without the absolute term."""
    lo, _, scale = fr
    q = E.xyz3(q)
    rho = fma32(sqrt_ru(r2), f32(1.000001), margin)
    top = (1 << SUMMARY_BITS) - 1
    c0 = np.zeros(q.shape, np.int64)
    c1 = np.full(q.shape, top, np.int64)
    ok = rho < f32(1e30)
    shift = np.uint32(21 - SUMMARY_BITS)
    with np.errstate(over="ignore"):
        for a in range(3):
            c0[ok, a] = quantise(_round_sum(q[ok, a], -rho[ok], False), lo[a], scale) >> shift
            c1[ok, a] = quantise(_round_sum(q[ok, a], rho[ok], True), lo[a], scale) >> shift
    return c0, c1


def box_passes(q, box, r2):
    """The box test `dx * dx + dy * dy + dz * dz <= lim`, true under both fp32 evaluation orders."""
    q = E.xyz3(q)
    with np.errstate(over="ignore", invalid="ignore"):
        lim = (fma32(r2, f32(1e-5), r2) + f32(1e-30)).astype(f32)
        d = np.fmax(np.fmax((box[:, :3] - q).astype(f32), (q - box[:, 3:]).astype(f32)), f32(0))
        sq = (d * d).astype(f32)
        plain = ((sq[:, 0] + sq[:, 1]).astype(f32) + sq[:, 2]).astype(f32)
        chain = fma32(d[:, 2], d[:, 2], fma32(d[:, 1], d[:, 1], sq[:, 0]))
    return (plain <= lim) & (chain <= lim)


def reach_misses(x, ranks_list, ks, margin=MARGIN, block=256):
    """{(ranks, k): (rows that need a remote rank, needed remote pairs, pairs whose rank is not asked, rows with such a
    pair)}; None for a split the driver refuses (a rank with < 2 points, or with <= k points at search)."""
    x3 = E.xyz3(x)
    n = len(x3)
    fr = frame(x)
    setups, out = {}, {}
    for ranks in ranks_list:
        owner = split(x, ranks)
        if owner is not None:
            summ, cell = summaries(x, owner, ranks, fr)
            c9 = cells(x, fr, SUMMARY_BITS).astype(np.int64)
            setups[ranks] = (owner, summ, cell, c9, np.bincount(owner, minlength=ranks).min())
        for k in ks:
            out[(ranks, k)] = None if owner is None or setups[ranks][4] <= k else [0, 0, 0, 0]
    for b0 in range(0, n, block):
        qi = np.arange(b0, min(n, b0 + block))
        with np.errstate(over="ignore", invalid="ignore"):
            d = dist2(x3[qi][:, None, :], x3[None, :, :])
        for ranks, (owner, summ, cell, c9, _) in setups.items():
            same = owner[None, :] == owner[qi][:, None]
            local = np.where(same, d, f32(np.inf))
            local[np.arange(len(qi)), qi] = np.inf  # the query itself
            for k in ks:
                acc = out[(ranks, k)]
                if acc is None:
                    continue
                r2 = np.partition(local, k - 1, axis=1)[:, k - 1]
                bi, pj = np.nonzero(~same & (d <= r2[:, None]))
                if bi.size == 0:
                    continue
                c0, c1 = reach_range(x3[qi], r2, fr, margin)
                inside = ((c9[pj] >= c0[bi]) & (c9[pj] <= c1[bi])).all(1)
                passes = box_passes(x3[qi[bi]], summ[owner[pj], cell[pj]], r2[bi])
                miss = ~(inside & passes)
                acc[0] += np.unique(bi).size
                acc[1] += bi.size
                acc[2] += int(miss.sum())
                acc[3] += np.unique(bi[miss]).size
    return out


MODEL_CLOUDS = dict({name: (lambda name=name: E.cloud(name, 8000 if name == "tiny_1e-21" else 4000)) for name in E.CLOUDS},
                    lattice=lambda: datasets.lattice(16), uniform=lambda: datasets.uniform(4000, seed=21))
REFUSED = {"near_max", "outlier", "outlier_2d", "outlier_1e30"}  # the unit cloud shares one 256^3 cell: a rank owns < 2
RANKS, KS = (2, 3, 4), (1, 4, 10)
pytestmark = [pytest.mark.filterwarnings("ignore:overflow encountered"), pytest.mark.filterwarnings("ignore:invalid value")]


@pytest.mark.parametrize("name", sorted(MODEL_CLOUDS))
def test_reach_asks_every_rank_a_point_needs(name):
    x = MODEL_CLOUDS[name]()
    res = reach_misses(x, RANKS, KS)
    checked = {key: v for key, v in res.items() if v is not None}
    if name in REFUSED:
        assert not checked, f"{name}: the split was expected to be refused: {checked}"
        return
    assert checked, f"{name}: every split refused"
    for key, (rows, pairs, missed, missed_rows) in checked.items():
        assert missed == 0, f"{name} ranks, k = {key}: {missed} of {pairs} needed pairs ({missed_rows} of {rows} rows) unasked"
    assert sum(v[1] for v in checked.values()) > 0, f"{name}: no query needed a remote rank: the check is vacuous"


def test_split_is_cell_aligned_and_balanced():
    """Points of one 256^3 cell share a rank, ranks follow the Morton order, and the counts are near n / ranks."""
    x = datasets.uniform(20_000, seed=5)
    fr = frame(x)
    c = interleave(cells(x, fr, SPLIT_BITS), SPLIT_BITS)
    for ranks in (2, 3, 5, 7):
        owner = split(x, ranks)
        order = np.argsort(c, kind="stable")
        assert (np.diff(owner[order]) >= 0).all()
        assert all(len(np.unique(owner[c == v])) == 1 for v in np.unique(c)[:200])
        counts = np.bincount(owner, minlength=ranks)
        assert np.abs(counts - len(x) / ranks).max() < 0.02 * len(x)


@pytest.mark.parametrize("ranks", [2, 4])
def test_range_without_margin_misses(ranks):
    """rho without the absolute term (the formula before it was added) misses remote points whose d2 underflows to a
    zero or subnormal r2 on the 1e-21 cloud: the model sees the defect the term fixes."""
    x = MODEL_CLOUDS["tiny_1e-21"]()
    old = reach_misses(x, (ranks,), (1,), margin=f32(0))[(ranks, 1)]
    new = reach_misses(x, (ranks,), (1,))[(ranks, 1)]
    assert old[2] > 0 and old[3] > 0, old
    assert new[2] == 0, new
