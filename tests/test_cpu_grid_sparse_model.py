"""A numpy model of grid_sparse_kernel's per-query walk (grid.cuh), checked on the CPU.

This models the kernel; it is not the kernel.  For one query q (a built point) and a bound B it restates in fp32:
- the query's own cell c = cell(q), clamped to the top occupied cell like the range;
- the cell range [lo, hi] (grid_knn_kernel's s) and the ring count max |lo - c|, |hi - c|;
- the deferral: a bound that is not finite or not >= 0, more than MAX_SPAN cells on an axis, more than GRID_CAP cells;
- the early exit: before ring t >= 1, the smallest RN(gap^2) over the axes and sides c -/+ t inside the range; the walk
  stops when it exceeds B;
- the ring's loops: x over [max(lo, c - t), min(hi, c + t)], y likewise, z over the ring's whole z range on its x or y faces
  and, inside them, from c - t in steps of 2t (only its two z faces);
- the box chain of a cell: ax2 = RN(tx * tx), ay2 = fma(ty, ty, ax2), d = fma(tz, tz, ay2), each compared with <= B.
It then checks, for every ordered pair (q, p), p != q, with the fp32 dist2(q, p) <= B and q not deferred, that the walk
reaches p: p's cell is in the range, the three chain terms are <= B, no ring 1 .. ring(p) exits early and the loops visit
p's cell.

A fixed bound is enough.  The kernel's bound starts at the round's r^2 and only shrinks, and it never drops below the
final k-th d2 of the query; every cull above (range, chain terms, early exit) is monotone in the bound, so a point with
d2 <= the final bound that the walk reaches under that bound is reached under every larger one the kernel holds on the
way.  The kernel's visit order decides only how fast the bound shrinks, never which of these points are reached.

The formulas must be kept in step with grid_sparse_kernel by hand; the kernel itself is compared with the CPU oracle in
test_gpu_grid_extreme.py and test_gpu_grid_sparse.py.
"""
import numpy as np
import pytest
from scipy.spatial import cKDTree

import extreme_clouds as E
from test_cpu_grid_model import CLOUDS as MODEL_CLOUDS
from test_cpu_grid_model import MARGIN, boundaries, cell, cell_range, dist2, fma32, key_frame

f32, f64 = np.float32, np.float64
FLT_MAX = f32(np.finfo(f32).max)
MAX_SPAN, GRID_CAP = 31, 1024
QTERM = f32(2.0 ** -18)


def axis_gap(q, lo, hi):
    """grid.cuh's axis_gap: fmaxf(fmaxf(lo - q, q - hi), 0) in fp32."""
    with np.errstate(over="ignore", invalid="ignore"):
        return np.fmax(np.fmax((lo - q).astype(f32), (q - hi).astype(f32)), f32(0))


def sq(g):
    with np.errstate(over="ignore", under="ignore"):
        return (g * g).astype(f32)


def level_for(n, forced=0):
    """grid_level_for with the key's 13 code bits per axis (every n here): floor(log2 n) / 3, or the forced level."""
    return max(1, min(forced if forced > 0 else (int(n).bit_length() - 1) // 3, 13, 8))


class Frame:
    def __init__(self, x, level):
        self.x = E.xyz3(x)
        self.level = level
        self.lo, self.hi, self.scale = key_frame(self.x)
        self.B, self.top = [], []
        for a in range(3):
            b, t = boundaries(self.lo[a], self.hi[a], self.scale, level)
            self.B.append(b)
            self.top.append(int(t))
        self.cells = np.stack([cell(self.x[:, a], self.lo[a], self.scale, level).astype(np.int64) for a in range(3)], 1)


def walk_misses(fr, qs, bound, margin=MARGIN, qterm=QTERM, exit_ge=False, exit_plus_only=False, z_minus_only=False):
    """(pairs with dist2 <= bound from the queries qs, pairs the walk misses, deferred queries).  The keyword arguments
    are deliberate faults of the kernel (the negative tests)."""
    x, lv, bound = fr.x, fr.level, f32(bound)
    m = len(qs)
    q = x[qs]
    c, lo, hi = np.zeros((m, 3), np.int64), np.zeros((m, 3), np.int64), np.zeros((m, 3), np.int64)
    defer = ~((bound >= 0) & (bound <= FLT_MAX)) | np.zeros(m, bool)
    vol = np.ones(m, np.int64)
    for a in range(3):
        if qterm == QTERM:
            l, h = cell_range(q[:, a], bound, fr.lo[a], fr.scale, lv, fr.top[a], margin)
        else:  # the range of a kernel without the |q| 2^-18 term
            with np.errstate(over="ignore", invalid="ignore"):
                s = fma32(np.sqrt(f32(bound)), f32(1.0001), fma32(np.abs(q[:, a]), qterm, margin))
                l = cell((q[:, a] - s).astype(f32), fr.lo[a], fr.scale, lv)
                h = np.minimum(cell((q[:, a] + s).astype(f32), fr.lo[a], fr.scale, lv), fr.top[a])
        lo[:, a], hi[:, a] = l, h
        c[:, a] = np.minimum(fr.cells[qs, a], fr.top[a])
        w = hi[:, a] - lo[:, a] + 1
        defer |= w > MAX_SPAN
        vol *= np.minimum(w, 32)
    defer |= vol > GRID_CAP
    rings = np.max(np.maximum(c - lo, hi - c), 1)

    # the early exit: first ring t >= 1 whose lower bound exceeds the bound (the kernel's `lb > bound`)
    first_exit = np.full(m, 1 << 30, np.int64)
    for t in range(int(rings[~defer].max(initial=0)), 0, -1):
        lb = np.full(m, np.inf, f32)
        for a in range(3):
            B = fr.B[a]
            sides = (+1,) if exit_plus_only else (-1, +1)
            for sgn in sides:
                j = c[:, a] + sgn * t
                ok = (j >= lo[:, a]) & (j <= hi[:, a])
                jj = np.clip(j, 0, len(B) - 2)
                g = axis_gap(q[:, a], B[jj], B[jj + 1])
                lb = np.where(ok, np.fmin(lb, sq(g)), lb)
        stop = (lb >= bound) if exit_ge else (lb > bound)
        first_exit = np.where(stop & (t <= rings), t, first_exit)

    # the pairs: a float64 superset, then the fp32 rule (true distance within sqrt(bound) plus the rounding of dist2)
    live = np.flatnonzero(~defer)
    if live.size == 0 or not np.isfinite(bound):
        return 0, 0, int(defer.sum())
    r = np.sqrt((f64(bound) + 2.0 ** -146) * (1 + 2.0 ** -16))
    tree = cKDTree(x.astype(f64))
    lists = tree.query_ball_point(x[qs[live]].astype(f64), r)
    qi = np.repeat(live, [len(v) for v in lists])
    p = np.concatenate([np.asarray(v, np.int64) for v in lists]) if len(qi) else np.zeros(0, np.int64)
    keep = p != qs[qi]
    qi, p = qi[keep], p[keep]
    with np.errstate(over="ignore", invalid="ignore", under="ignore"):
        within = dist2(q[qi], x[p]) <= bound
    qi, p = qi[within], p[within]
    if qi.size == 0:
        return 0, 0, int(defer.sum())

    pc = fr.cells[p]
    ok = ((pc >= lo[qi]) & (pc <= hi[qi])).all(1)
    pcc = np.clip(pc, 0, None)
    t3 = [axis_gap(q[qi, a], fr.B[a][np.minimum(pcc[:, a], len(fr.B[a]) - 2)],
                   fr.B[a][np.minimum(pcc[:, a], len(fr.B[a]) - 2) + 1]) for a in range(3)]
    with np.errstate(over="ignore", under="ignore"):
        ax2 = sq(t3[0])
        ay2 = fma32(t3[1], t3[1], ax2)
        d = fma32(t3[2], t3[2], ay2)
    ok &= (ax2 <= bound) & (ay2 <= bound) & (d <= bound)
    cq = c[qi]
    t = np.max(np.abs(pc - cq), 1)
    ok &= t < first_exit[qi]
    # ring t's loops: is p's cell one of the cells they visit?
    edge = (pc[:, 0] == cq[:, 0] - t) | (pc[:, 0] == cq[:, 0] + t) | (pc[:, 1] == cq[:, 1] - t) | (pc[:, 1] == cq[:, 1] + t)
    z0 = np.where(edge, np.maximum(lo[qi, 2], cq[:, 2] - t), cq[:, 2] - t)
    zs = np.where(edge, 1, 2 * t)
    z1 = np.minimum(hi[qi, 2], cq[:, 2] + t)
    if z_minus_only:
        z1 = np.where(edge, z1, np.minimum(z1, cq[:, 2] - t))
    z = pc[:, 2]
    ok &= (z >= z0) & (z <= z1) & ((z - z0) % np.maximum(zs, 1) == 0) & (z >= lo[qi, 2])
    return int(qi.size), int((~ok).sum()), int(defer.sum())


def kth_d2(x, k=10, m=2000):
    """fp32 d2 of the k-th neighbour of the first m points (float64 candidates, fp32 rule, ties kept)."""
    x3 = E.xyz3(x)
    tree = cKDTree(x3.astype(f64))
    _, idx = tree.query(x3[:m].astype(f64), k + 8)
    idx = np.where(idx >= len(x3), 0, idx)
    with np.errstate(over="ignore", invalid="ignore", under="ignore"):
        d = dist2(x3[:m, None, :], x3[idx])
    d = np.where(idx == np.arange(m)[:, None], np.inf, d)
    return np.sort(d, 1)[:, k - 1].astype(f32)


def bounds_of(x):
    """0, three subnormal steps, the median k-th d2 and twice it, the k-th d2 most queries share (an exact tie shell where
    the cloud has one), FLT_MAX and +inf."""
    d = kth_d2(x)
    fin = d[np.isfinite(d)]
    out = [f32(0), f32(3 * 2.0 ** -149), FLT_MAX, f32(np.inf)]
    if fin.size:
        med = f32(np.median(fin))
        vals, counts = np.unique(fin, return_counts=True)
        out += [med, f32(min(f64(med) * 2, f64(FLT_MAX))), f32(vals[np.argmax(counts)])]
    return sorted(set(out), key=float)


N_CATALOGUE = 4000
QUERIES = 600


def catalogue(name, level=0):
    x = E.cloud(name, 8000 if name == "tiny_1e-21" else N_CATALOGUE)
    return x, level_for(len(x), level)


def lattice16():
    """The full 1/16 lattice on [0, 1]^3: lo = 0, hi = 1, scale = 2^21, so at level 3 every cell face is a lattice plane and
    every cell holds its face points and, at its centre, the points with three odd coordinates."""
    g = np.stack(np.meshgrid(*[np.arange(17)] * 3, indexing="ij"), -1).reshape(-1, 3)
    return (g / 16.0).astype(f32), 3


CASES = ([(name, lv) for name in E.CLOUDS for lv in (0, 1, 5)] + [(f"model:{name}", 0) for name in MODEL_CLOUDS] +
         [("lattice16", 0)])


def case(name, lv):
    if name.startswith("model:"):
        return MODEL_CLOUDS[name[6:]]()
    if name == "lattice16":
        return lattice16()
    return catalogue(name, lv)


def queries(n, seed=0):
    return np.sort(np.random.default_rng(seed).choice(n, min(n, QUERIES), replace=False))


@pytest.mark.parametrize("name,lv", CASES, ids=[f"{n}-L{lv}" for n, lv in CASES])
def test_walk_reaches_every_pair(name, lv):
    x, level = case(name, lv)
    fr = Frame(x, level)
    qs = queries(len(x))
    for bound in bounds_of(x):
        n_pairs, misses, deferred = walk_misses(fr, qs, bound)
        assert misses == 0, (name, level, bound, n_pairs, misses)
        if not np.isfinite(bound):
            assert deferred == len(qs), "a bound that is not finite tests nothing"


def test_flt_max_bound_is_deferred_on_a_fine_grid():
    """r^2 = FLT_MAX spans the whole scene: on a grid wider than MAX_SPAN cells every query is deferred (on a coarse
    grid, or a frame of scale 0 where every point is in cell 0, the walk runs and test_walk_reaches_every_pair covers it)."""
    x, level = catalogue("offset_1e6", 5)
    fr = Frame(x, level)
    assert max(fr.top) + 1 > MAX_SPAN
    assert walk_misses(fr, queries(len(x)), FLT_MAX)[2] == QUERIES


def test_scale_zero_frame_is_one_cell():
    """near_max: the extent overflows, the scale is 0 and quantise21 sees inf * 0 = NaN; fmaxf maps it to cell 0, so the
    grid is one cell and every range is [0, 0]."""
    x, level = catalogue("near_max")
    fr = Frame(x, level)
    assert fr.scale == 0 and fr.top == [0, 0, 0] and (fr.cells == 0).all()
    assert (fr.B[0][1:] == fr.hi[0]).all()


# ---- negative tests: the model sees each defect of a deliberately wrong kernel ----

def _some_cloud_misses(names, **fault):
    for name, lv in names:
        x, level = case(name, lv)
        fr = Frame(x, level)
        qs = queries(len(x))
        for bound in bounds_of(x):
            if walk_misses(fr, qs, bound, **fault)[1] > 0:
                return True
    return False


def test_early_exit_at_equality_misses():
    """`lb >= bound`: on lattice16 a query at a cell centre has its six nearest neighbours on the faces of the next cells, at
    exactly d2 = 2^-8, the ring-1 lower bound; with the bound on that tie shell (k <= 6) the walk stops one ring short.
    The catalogue clouds' ties do not line up with the cell faces like this, and none of them makes the fault miss."""
    x, level = lattice16()
    fr = Frame(x, level)
    qs = np.arange(len(x))
    assert walk_misses(fr, qs, f32(2.0 ** -8))[1] == 0
    assert walk_misses(fr, qs, f32(2.0 ** -8), exit_ge=True)[1] > 0


def test_early_exit_from_one_side_misses():
    """A lower bound from the c + t side only stops the walk as soon as that side leaves the range or is far."""
    assert _some_cloud_misses([("offset_1e4", 5)], exit_plus_only=True)


def test_interior_z_step_one_face_misses():
    """The interior z step visiting only c - t never reaches the ring's upper z face inside its x and y faces."""
    assert _some_cloud_misses([("offset_1e4", 5)], z_minus_only=True)


@pytest.mark.parametrize("name", ["scale_1e-21", "scale_1e-22"])
def test_range_without_margin_misses(name):
    """Without the 2^-74 term the sparse walk's range misses pairs whose dx * dx underflows (bound 0 or subnormal)."""
    assert _some_cloud_misses([(f"model:{name}", 0)], margin=f32(0))


def test_range_without_q_term_still_covers():
    """The |q| 2^-18 term of s is redundant for these pairs: RN(q - p) differs from q - p by at most u |q - p|, which the
    factor 1.0001 on sqrt(bound) covers, and RN(q -/+ s) is monotone, so p's cell stays in the range.  No cloud here
    makes a kernel without it miss; the term stays as a margin of safety."""
    assert not _some_cloud_misses([(n, 0) for n in E.CLOUDS] + [("model:quantised_shifted", 0)], qterm=f32(0))
