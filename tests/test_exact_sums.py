"""Dyadic scenes (synth.dyadic) and the exact-sum precondition (oracle/exact_sums.py), on the CPU oracle alone.

On a cloud whose coordinates are multiples of q = 2^-e, with every partial sum below 2^24 units, the nine float32
neighbourhood sums of the radius normals do not depend on the order of their additions.  The oracle has two orders
(FLANN's (d2, index) order and index order): on such scenes they must give the same bits, on the raw scans they do
not.  tests/test_gpu_normals_exact.py relies on this to hold the fast normals kernel to the oracle bit for bit.
"""
import numpy as np
import pytest

from geometric_mapping_b200 import synth
from oracle import chain
from oracle import exact_sums as X
from oracle import oracle as O


def test_dyadic_rounds_to_the_lattice_and_keeps_junk():
    pts = np.array([[0.3, -0.01, 5.0, 1.0], [-0.3, 1.0 / 3.0, -5.0, 7.0], [np.nan, np.inf, -np.inf, 1.0],
                    [0.0625, 0.09375, 0.03125, 1.0], [1e30, -1e-30, -0.0, 1.0]], np.float32)
    out = synth.dyadic(pts, 4)
    assert out.dtype == np.float32 and out.shape == pts.shape
    assert np.array_equal(out[0], np.float32([0.3125, 0.0, 5.0, 1.0])) and np.signbit(out[0, 1]) == 0
    assert np.array_equal(out[1], np.float32([-0.3125, 0.3125, -5.0, 7.0]))           # the padding word is kept
    assert np.isnan(out[2, 0]) and out[2, 1] == np.inf and out[2, 2] == -np.inf
    assert np.array_equal(out[3], np.float32([0.0625, 0.125, 0.0, 1.0]))              # ties to even: 1.5 -> 2, 0.5 -> 0
    assert out[4, 0] == np.float32(1e30) and not np.signbit(out[4, 1:3]).any()         # no -0.0 remains
    assert np.array_equal(synth.dyadic(out, 4).view(np.uint32), out.view(np.uint32))   # idempotent


def _junk_scan():
    pts = synth.curved_tunnel(40_000, seed=5, outlier_frac=0.05)
    pts[100] = [np.nan, 0, 0, 1]
    pts[101] = [0, np.inf, 0, 1]
    pts[102] = [9.0, 0, 0, 1]
    pts[200:210] = pts[300:310]
    return pts


@pytest.mark.parametrize("scene,radius,e", [("C0", 0.15, 5), ("C1", 0.05, 6), ("junk", 0.12, 6)])
def test_oracle_summation_orders_agree_bit_for_bit_on_dyadic_scenes(scene, radius, e):
    """The scenes of tests/test_gpu_chain.py rounded to q = 2^-e: the precondition holds with a margin, and the oracle's
    FLANN-order and index-order normals (and curvature) are identical; on the raw scan they differ."""
    raw = {"C0": lambda: synth.straight_cylinder(100_000, seed=1), "C1": lambda: synth.curved_tunnel(1_000_000, seed=2),
           "junk": _junk_scan}[scene]()
    for pts, exact in ((synth.dyadic(raw, e), True), (raw, False)):
        cropped, _ = O.crop(pts, 5.0, True)
        a, ca, _ = O.normals(cropped, radius, order=0)
        b, cb, _ = O.normals(cropped, radius, order=1)
        assert np.array_equal(ca, cb)
        fin = np.isfinite(a[:, 0])
        assert fin.mean() > 0.9
        if exact:
            assert X.check(cropped, ca, radius, e, n_sample=2000) < 0.6
            assert np.array_equal(chain._bits(a), chain._bits(b))
        else:
            same = (chain._bits(a) == chain._bits(b)).all(1)
            assert same[fin].mean() < 0.05        # the order matters on the raw scan: the scene is what makes it exact


def test_precondition_rejects_violating_scenes():
    """Five points near x = 2000 m on the metre lattice, r = 2.5: the middle one has 5 neighbours and k = 2002 + 3, and
    5 * 2005^2 > 2^24 must fail, and say so; the same points near the origin pass; a coordinate off the lattice is
    refused."""
    g = np.arange(5, dtype=np.float32)
    far = np.zeros((5, 4), np.float32)
    far[:, 0] = 2000.0 + g
    far[:, 1] = g % 2
    far[:, 3] = 1.0
    _, cnt, _ = O.normals(far, 2.5)
    assert (cnt >= 3).all()
    worst, at = X.sum_bound(far, cnt, 2.5, 0)
    assert worst >= X.LIMIT and at >= 0
    with pytest.raises(AssertionError, match="violates the exact-sum precondition"):
        X.check(far, cnt, 2.5, 0)
    near = far.copy()
    near[:, 0] -= 2000.0
    _, cnt_near, _ = O.normals(near, 2.5)
    assert np.array_equal(cnt_near, cnt) and X.check(near, cnt_near, 2.5, 0) < 1e-3
    off = near.copy()
    off[2, 2] = 0.5
    with pytest.raises(AssertionError, match="not multiples"):
        X.sum_bound(off, cnt, 2.5, 0)
