"""Deterministic point clouds at the edges of the fp32 distance rule — TEST INFRASTRUCTURE ONLY.

Every result of the library is defined by d2 = fmaf(dz,dz,fmaf(dy,dy,dx*dx)) in fp32, closed balls d2 <= fl(r*r) and
ties on (d2, index).  These clouds put that rule where it gets awkward: exact ties from coarse ulps, subnormal and zero
d2 between distinct points, d2 that overflows to +inf (some pairs, every pair, or only across clusters), an extent
that overflows (the curve-code scale becomes 0), one normal cloud squeezed into a single curve cell by an outlier, and
signed zeros.  Every cloud is built in float64 and cast, and every coordinate is finite.

CLOUDS maps a name to make(n, seed) -> float32 [n, 3] (or [n, 2] for the 2-D variants, whose z is 0).
"""
import numpy as np

BIG = 3e38           # finite in fp32 (FLT_MAX = 3.4028235e38); any difference of two such values overflows
R_LAST_FINITE = np.float32(1.8446743e19)  # the largest radius whose fp32 square is finite
R_FIRST_INF = np.float32(1.8446744e19)    # the next float: fl(r * r) = +inf admits every pair


def _f32(a):
    a = np.asarray(a, np.float64).astype(np.float32)
    assert np.isfinite(a).all()
    return a


def offset_1e6(n, seed=0):
    """ulp(1e6) = 1/16: about 128 distinct values per axis, exact distance ties everywhere."""
    return _f32(np.random.default_rng(seed).random((n, 3)) * 8 + 1e6)


def offset_1e4(n, seed=0):
    """ulp(1e4) ~ 1e-3: coarse coordinates, few ties."""
    return _f32(np.random.default_rng(seed).random((n, 3)) + 1e4)


def tiny(n, seed=0):
    """Subnormal d2, and d2 == 0 between many distinct points (dx * dx underflows)."""
    return _f32(np.random.default_rng(seed).random((n, 3)) * 1e-21)


def overflow_1e20(n, seed=0):
    """Near pairs have a finite d2, far pairs +inf."""
    return _f32((np.random.default_rng(seed).random((n, 3)) - 0.5) * 1e20)


def far_clusters(n, seed=0):
    """Two clusters of spread 1e18 at -1e20 and +1e20: d2 finite inside a cluster, +inf across."""
    rng = np.random.default_rng(seed)
    side = np.where(rng.random(n) < 0.5, -1e20, 1e20)[:, None]
    return _f32(side + (rng.random((n, 3)) - 0.5) * 1e18)


def near_max(n, seed=0):
    """The extent overflows fp32 (the curve-code scale is 0) and every d2 is +inf."""
    return _f32((np.random.default_rng(seed).random((n, 3)) - 0.5) * 2 * BIG)


def outlier(n, seed=0):
    """A unit cloud plus 4 points at the +-3e38 corners: the unit cloud falls into one curve cell."""
    rng = np.random.default_rng(seed)
    x = rng.random((n, 3))
    at = rng.choice(n, 4, replace=False)
    x[at] = np.array([[BIG, BIG, BIG], [-BIG, -BIG, -BIG], [BIG, -BIG, BIG], [-BIG, BIG, -BIG]])
    return _f32(x)


def outlier_1e30(n, seed=0):
    """A unit cloud plus one point at (1e30, 1e30, 1e30): a finite frame, but the unit cloud still shares one cell."""
    rng = np.random.default_rng(seed)
    x = rng.random((n, 3))
    x[rng.integers(n)] = 1e30
    return _f32(x)


def mixed_scales(n, seed=0):
    """Half the points at 1e-20 scale near the origin, half spread over 1e20: one frame, two scales."""
    rng = np.random.default_rng(seed)
    x = np.where((rng.random(n) < 0.5)[:, None], rng.random((n, 3)) * 1e-20, (rng.random((n, 3)) - 0.5) * 1e20)
    return _f32(x)


def across_zero(n, seed=0):
    """A 1/16 lattice centred on 0 whose zero coordinates are -0.0 or +0.0 at random (n rounded to a cube)."""
    rng = np.random.default_rng(seed)
    s = max(2, int(round(n ** (1 / 3))))
    g = np.stack(np.meshgrid(*[np.arange(s) - s // 2] * 3, indexing="ij"), -1).reshape(-1, 3) / 16.0
    g = g[rng.permutation(len(g))]
    g[(g == 0) & (rng.random(g.shape) < 0.5)] = -0.0
    return _f32(g)


def offset_1e6_2d(n, seed=0):
    return offset_1e6(n, seed)[:, :2].copy()


def outlier_2d(n, seed=0):
    return outlier(n, seed)[:, :2].copy()


CLOUDS = {
    "offset_1e6": offset_1e6,
    "offset_1e4": offset_1e4,
    "tiny_1e-21": tiny,
    "overflow_1e20": overflow_1e20,
    "far_clusters": far_clusters,
    "near_max": near_max,
    "outlier": outlier,
    "outlier_1e30": outlier_1e30,
    "mixed_scales": mixed_scales,
    "across_zero": across_zero,
    "offset_1e6_2d": offset_1e6_2d,
    "outlier_2d": outlier_2d,
}


def cloud(name, n=3000, seed=0):
    return CLOUDS[name](n, seed)


def xyz3(x):
    """[n, 3] float32: 2-D input gets z = 0 (the library's 2-D rule)."""
    x = np.ascontiguousarray(x, np.float32)
    if x.shape[1] == 2:
        x = np.concatenate([x, np.zeros((len(x), 1), np.float32)], 1)
    return x


def next_down(r):
    return np.nextafter(np.float32(r), np.float32(0))
