"""The deskew restatement (tests/deskew_oracle.py) against scipy's rotation interpolation, its end points, and the swept
scan generator (synth.swept_scan) against it: no device needed."""
import numpy as np
import pytest
from scipy.spatial.transform import Rotation

import deskew_oracle as DK
from geometric_mapping_b200 import synth

PERIOD = 0.1
DELTAS = [synth.pose34((0.0, 0.0, np.radians(1.5)), (0.15, 0.01, 0.0)),
          synth.pose34((0.3, -0.2, 0.5), (-0.4, 0.2, 0.1)),
          synth.pose34((1e-7, 0.0, 0.0), (0.0, 0.0, 0.0)),
          synth.pose34((0.0, 2.5, 0.0), (0.0, 0.0, 1.0))]


@pytest.mark.parametrize("d", range(len(DELTAS)))
def test_rotation_is_scipy_slerp_from_the_identity(d):
    D = DELTAS[d]
    a = np.linspace(-1.5, 1.5, 31)
    ref = Rotation.from_rotvec(a[:, None] * Rotation.from_matrix(D[:, :3]).as_rotvec()[None, :]).as_matrix()
    assert np.abs(DK.rotation(D, a) - ref).max() <= 1e-12


@pytest.mark.parametrize("d", range(len(DELTAS)))
def test_end_points(d):
    D = DELTAS[d]
    p = np.random.default_rng(d).uniform(-5, 5, (100, 3))
    assert np.abs(DK.deskew(p, np.full(100, 1.0, np.float32), D, 0.0, 1.0) - (p @ D[:, :3].T + D[:, 3])).max() <= 1e-12
    assert np.array_equal(DK.deskew(p, np.full(100, 0.25, np.float32), D, 0.25, PERIOD), p)


def test_identity_and_non_finite_points():
    p = np.random.default_rng(1).uniform(-5, 5, (6, 3))
    t = np.linspace(0.0, PERIOD, 6).astype(np.float32)
    assert np.array_equal(DK.deskew(p, t, np.eye(3, 4), 0.0, PERIOD), p)
    p[1, 0], p[2, 2] = np.nan, np.inf
    t[3] = np.nan
    out = DK.deskew(p, t, DELTAS[0], 0.0, PERIOD)
    assert np.isnan(out[1:4]).all() and np.isfinite(out[[0, 4, 5]]).all()


@pytest.mark.parametrize("t_ref", [0.0, 0.05])
def test_swept_scan_deskews_to_the_snapshot(t_ref):
    pose = synth.pose34((0.0, 0.0, np.radians(3.0)), (-0.2, 0.05, 0.0))
    delta = DELTAS[0]
    pts = synth.drift_end_niche(20_000, seed=9)
    q, t = synth.swept_view(pts, pose, delta, PERIOD, t_ref)
    assert t.dtype == np.float32 and t.min() >= 0.0 and t.max() <= PERIOD and np.ptp(t) > 0.9 * PERIOD
    snap = (pts[:, :3].astype(np.float64) - pose[:, 3]) @ pose[:, :3]       # synth.view_from in float64
    assert np.abs(q - snap).max() > 0.05                                    # the sweep moves the points ...
    assert np.abs(DK.deskew(q, t, delta, t_ref, PERIOD) - snap).max() <= 1e-9  # ... and the deskew takes them back
    assert np.abs(synth.view_from(pts, pose)[:, :3] - snap).max() <= 1e-6
    xyzw, t2 = synth.swept_scan(synth.drift_end_niche, pose, delta, PERIOD, seed=9, n=20_000, t_ref=t_ref)
    assert np.array_equal(t2, t) and np.array_equal(xyzw[:, :3], q.astype(np.float32)) and (xyzw[:, 3] == 1).all()
