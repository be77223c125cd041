"""The oracle restatement of sequential multi-primitive extraction on a known answer (CPU only)."""
import numpy as np

from geometric_mapping_b200 import synth
from oracle import primitives as P


def _known_scene(seed=11):
    """Four separated plane patches and a short cylinder (axis x through (0, -5, 0), r = 1), analytic normals, and
    outliers kept 0.3 m away from every surface.  -> cloud, normals8, generator label (0 = outlier, 1..5)."""
    patches = [((0, 0, 1), -3.0), ((1, 0, 0), 4.0), ((0, 1, 0), 4.0), ((0, 0, 1), 3.0)]
    pts, nrm, lab = [], [], []
    for k, (n, off) in enumerate(patches):
        p = synth.plane_patch(3000, seed=seed + k, normal=n, offset=off, half=1.0, noise=0.002)
        pts.append(p)
        nrm.append(np.tile(np.array(n, np.float32), (len(p), 1)))
        lab.append(np.full(len(p), k + 1))
    c = synth.straight_cylinder(4000, seed=seed + 9, radius=1.0, half_length=1.0, noise=0.002)
    c[:, 1] -= 5.0
    radial = c[:, :3].astype(np.float64) - [0.0, -5.0, 0.0]
    radial[:, 0] = 0.0
    pts.append(c)
    nrm.append((radial / np.linalg.norm(radial, axis=1, keepdims=True)).astype(np.float32))
    lab.append(np.full(len(c), 5))
    g = np.random.Generator(np.random.Philox(seed + 20))
    o = g.uniform(-6.0, 6.0, (4000, 3))
    far = (np.abs(np.abs(o[:, 2]) - 3.0) > 0.3) & (np.abs(o[:, 0] - 4.0) > 0.3) & (np.abs(o[:, 1] - 4.0) > 0.3)
    far &= np.abs(np.hypot(o[:, 1] + 5.0, o[:, 2]) - 1.0) > 0.3
    o = o[far][:200]
    pts.append(np.concatenate([o, np.ones((len(o), 1))], 1).astype(np.float32))
    nrm.append(np.tile(np.array([0, 0, 1], np.float32), (len(o), 1)))
    lab.append(np.zeros(len(o), int))
    normals8 = np.zeros((sum(len(p) for p in pts), 8), np.float32)
    normals8[:, :3] = np.concatenate(nrm)
    return np.concatenate(pts), normals8, np.concatenate(lab)


def test_known_answer_five_primitives_then_stop():
    cloud, normals8, lab = _known_scene()
    K = 8
    prims, ids = P.extract(cloud, normals8, synth.sample_draws(K, 256, 3, seed=1), synth.sample_draws(K, 256, 2, seed=2), K,
                           min_inliers=500, rmin=0.5, rmax=3.0)
    assert len(prims) == 5  # the sixth round finds nothing with 500 inliers among the outliers and stops
    assert sorted(p["kind"] for p in prims) == [0, 0, 0, 0, 1]
    assert prims[0]["kind"] == 1  # the largest surface is claimed first
    seen = set()
    for k, p in enumerate(prims):
        members = np.unique(lab[ids == k + 1])
        assert len(members) == 1 and members[0] != 0, (k, members)
        assert np.array_equal(ids == k + 1, lab == members[0])
        assert p["best_count"] == int((ids == k + 1).sum()) == p["refit_count"]
        seen.add(int(members[0]))
    assert seen == {1, 2, 3, 4, 5}
    assert np.all(ids[lab == 0] == 0)
    assert [p["n_remaining"] for p in prims] == [len(cloud) - sum(q["best_count"] for q in prims[:k]) for k in range(len(prims))]


def test_compression_of_the_known_answer():
    cloud, normals8, lab = _known_scene()
    K = 6
    prims, ids = P.extract(cloud, normals8, synth.sample_draws(K, 256, 3, seed=1), synth.sample_draws(K, 256, 2, seed=2), K,
                           min_inliers=500, rmin=0.5, rmax=3.0)
    c = P.compress(cloud, ids, prims, 0.1)
    assert [r["count"] for r in c["records"]] == [p["best_count"] for p in prims]
    assert c["n_residual"] == int((lab == 0).sum())
    for r in c["records"]:
        assert r["rms"] < 0.01
        if r["kind"] == 0:
            assert 1.8 < r["extents"][1] - r["extents"][0] < 2.0 and 1.8 < r["extents"][3] - r["extents"][2] < 2.0
        else:
            assert 1.9 < r["extents"][1] - r["extents"][0] < 2.0


def test_draw_mapping_stays_in_range():
    edge = np.array([0, 1, 0x7FFFFFFF, 0x80000000, 0xFFFFFFFE, 0xFFFFFFFF], np.uint32)
    draws = np.concatenate([edge, synth.sample_draws(1, 1000, 3, seed=5).ravel()])
    assert np.all(P.map_draws(draws, np.empty(0, np.int32)) == -1)
    assert np.all(P.map_draws(draws, np.array([7], np.int32)) == 7)
    two = P.map_draws(draws, np.array([3, 9], np.int32))
    assert set(two.tolist()) == {3, 9}
    n = (1 << 31) - 1
    pos = P.draw_positions(draws, n)
    assert pos.min() == 0 and pos.max() == n - 1 and np.all(pos < n)


def test_trace_records_every_round_and_the_stop():
    cloud, normals8, _ = _known_scene()
    K = 8
    trace = []
    prims, ids = P.extract(cloud, normals8, synth.sample_draws(K, 256, 3, seed=1), synth.sample_draws(K, 256, 2, seed=2), K,
                           min_inliers=500, rmin=0.5, rmax=3.0, trace=trace)
    assert len(trace) == len(prims) + 1
    assert [t[0] for t in trace[:-1]] == [p["n_remaining"] for p in prims]
    assert [max(t[1:]) for t in trace[:-1]] == [p["best_count"] for p in prims]
    assert trace[-1][0] == int((ids == 0).sum()) and max(trace[-1][1:]) < 500


def test_plane_reference_recovers_a_known_plane():
    n = np.array([1.0, 2.0, -2.0]) / 3.0
    p = synth.plane_patch(20_000, seed=31, normal=n, offset=1.25, half=1.5, noise=0.01)
    nr, d, rms = P.plane_fit_d(p)
    s = np.sign(nr @ n)
    assert np.linalg.norm(np.cross(nr, n)) < 1e-3 and abs(s * d + 1.25) < 1e-3 and abs(rms - 0.01) < 5e-4
    # exact points: the eigen-decomposition of the float64 covariance is exact to rounding
    u, v = P.perp_basis_d(n)
    g = np.random.Generator(np.random.Philox(32)).uniform(-1.0, 1.0, (500, 2))
    q = g[:, :1] * u + g[:, 1:] * v - 0.5 * n
    nr, d, rms = P.plane_fit_d(q)
    assert np.linalg.norm(np.cross(nr, n)) < 1e-12 and abs(np.sign(nr @ n) * d - 0.5) < 1e-12 and rms < 1e-7


def test_cylinder_reference_recovers_a_known_cylinder():
    """Points exactly on a tilted cylinder: from a start 0.05 rad and 3 cm off, the fit lands on it to rounding; with
    radial noise, its RMS is the lowest of nearby models."""
    axis = np.array([0.3, -0.2, 1.0]) / np.linalg.norm([0.3, -0.2, 1.0])
    q0, r0 = np.array([0.5, -1.0, 0.2]), 1.7
    u, w = P.perp_basis_d(axis)
    g = np.random.Generator(np.random.Philox(33))
    th, t = g.uniform(0.0, 2.0 * np.pi, 4000), g.uniform(-2.0, 2.0, 4000)
    pts = q0 + t[:, None] * axis + r0 * (np.cos(th)[:, None] * u + np.sin(th)[:, None] * w)
    assert np.abs(P.cylinder_residuals_d(pts, q0, axis, r0)).max() < 1e-12
    start = np.concatenate([q0 + 0.03 * u, axis + 0.05 * w, [r0 + 0.02]])
    assert P.cylinder_rms_d(pts, start) > 1e-3
    q, a, r, rms = P.cylinder_fit_d(pts, start)
    dq = q - q0
    assert np.linalg.norm(np.cross(a, axis)) < 1e-10 and abs(r - r0) < 1e-10 and np.linalg.norm(dq - axis * (dq @ axis)) < 1e-10
    assert rms < 1e-10
    noisy = pts + (g.normal(0.0, 0.01, 4000)[:, None] * (pts - q0 - ((pts - q0) @ axis)[:, None] * axis) / r0)
    q, a, r, rms = P.cylinder_fit_d(noisy, start)
    assert abs(rms - 0.01) < 1e-3 and abs(r - r0) < 1e-3
    best = np.concatenate([q, a, [r]])
    for k in range(7):
        for h in (-1e-4, 1e-4):
            assert P.cylinder_rms_d(noisy, best + h * np.eye(7)[k]) >= rms - 1e-15
