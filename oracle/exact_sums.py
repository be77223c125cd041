"""When the radius-normal sums do not depend on the order of their additions (test infrastructure).

The default (fast) normals kernel adds a point's neighbours in cell-run order with fused multiply-adds; the oracle adds
them in FLANN's (d2, index) order with separately rounded products.  Everything after the nine sums is the same code in
both.  If every coordinate is a multiple of q = 2^-e (synth.dyadic), every product is a multiple of q^2 and every partial
sum of the x*x .. z*z terms one of q^2 (of q for x, y, z): a float32 holds it exactly while its magnitude stays below
2^24 of those units.  Then every add and fma is exact, the order cannot change a bit, and the fast kernel must equal
the oracle bit for bit.

check() proves that for a cloud and radius before a test compares: with k = |x/q| + ceil(sqrt(r2)/q) per axis (a
neighbour lies within sqrt(r2) of the point, so |its coordinate / q| <= k), every partial sum of the a*b terms of a
point with cnt neighbours is at most cnt * k_a * k_b in units of q^2, and the linear sums are smaller still.
"""
from __future__ import annotations

import numpy as np

LIMIT = 1 << 24


def sum_bound(cloud, cnt, radius, e):
    """-> (worst cnt * k_a * k_b over the points with cnt >= 3 and all axis pairs, int; index of that point or -1).
    Raises AssertionError if a finite coordinate is not a multiple of 2^-e."""
    xyz = np.asarray(cloud, np.float32)[:, :3].astype(np.float64)
    fin = np.isfinite(xyz).all(1)
    m = xyz[fin] * 2.0 ** e
    assert (m == np.round(m)).all(), f"coordinates are not multiples of 2^-{e}"
    sel = fin & (np.asarray(cnt) >= 3)
    if not sel.any():
        return 0, -1
    r2 = np.float64(np.float32(radius * radius))  # the search predicate: d2 < float(radius^2), the square taken in double
    reach = int(np.ceil(np.sqrt(r2) * 2.0 ** e))
    k = np.abs(xyz[sel] * 2.0 ** e).astype(np.int64) + reach
    kmax = k.max(1)  # the largest k_a * k_b of a point is its largest k squared
    b = np.asarray(cnt)[sel].astype(np.int64) * kmax * kmax
    w = int(np.argmax(b))
    return int(b[w]), int(np.flatnonzero(sel)[w])


def check(cloud, cnt, radius, e, n_sample=3000, seed=0):
    """Assert the exactness precondition (see the module docstring) for the cropped cloud `cloud` whose neighbour counts
    are `cnt`; as a second check, take the neighbour sets of up to `n_sample` points from a k-d tree and assert that
    they have `cnt` members and that every prefix sum of their nine terms, in index order and in (d2, index) order, is
    a float32.  -> the worst bound as a fraction of 2^24 (what the test may report as its margin)."""
    from scipy.spatial import cKDTree

    worst, at = sum_bound(cloud, cnt, radius, e)
    assert worst < LIMIT, (f"dyadic scene violates the exact-sum precondition: cnt * k_a * k_b = {worst} >= 2^24 at point {at} "
                           f"(q = 2^-{e}, r = {radius}); choose a coarser q")
    cnt = np.asarray(cnt)
    xyz = np.asarray(cloud, np.float32)[:, :3].astype(np.float64)
    fin = np.flatnonzero(np.isfinite(xyz).all(1))
    cand = np.flatnonzero(np.isfinite(xyz).all(1) & (cnt >= 3))
    if len(cand):
        g = np.random.Generator(np.random.Philox(seed))
        pick = g.choice(cand, min(n_sample, len(cand)), replace=False)
        r2 = np.float64(np.float32(radius * radius))
        tree = cKDTree(xyz[fin])
        for i, nb in zip(pick, tree.query_ball_point(xyz[pick], np.sqrt(r2) * (1.0 + 1e-9))):
            nb = fin[np.asarray(nb, np.int64)]
            d = xyz[nb] - xyz[i]
            d2 = (d * d).sum(1)  # exact: the coordinates are multiples of q and small
            nb, d2 = nb[d2 < r2], d2[d2 < r2]
            assert len(nb) == cnt[i], f"point {i}: {len(nb)} neighbours within r, the oracle counted {cnt[i]}"
            p = xyz[nb]
            terms = np.stack([p[:, 0] * p[:, 0], p[:, 0] * p[:, 1], p[:, 0] * p[:, 2], p[:, 1] * p[:, 1], p[:, 1] * p[:, 2],
                              p[:, 2] * p[:, 2], p[:, 0], p[:, 1], p[:, 2]], 1)
            for order in (np.argsort(nb, kind="stable"), np.lexsort((nb, d2))):
                s = np.cumsum(terms[order], 0)
                assert (s.astype(np.float32).astype(np.float64) == s).all(), f"point {i}: a partial sum is not a float32"
    return worst / LIMIT
