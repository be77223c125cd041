"""CPU checks of the scan-to-map registration oracle (tests/register_map_oracle.py), the reference gm_register_map is
tested against.  None of them reuses the restatement's code: map planes against numpy.linalg.eigh of covariances built
here from a dictionary of cells, a flat sheet and a corner, the search against a k-d tree, and recovery of known
sensor poses against a map of three drift scans at 1M points."""
import numpy as np
import pytest
from scipy.spatial import cKDTree

import register_map_oracle as M
import register_oracle as R
from geometric_mapping_b200 import synth
from oracle import oracle as O

LEAF, DMAX = 0.1, 0.5


def _compacted(pts, radius=0.05):
    crop, _ = O.crop(pts, 5.0, True)
    nrm, _, _ = O.normals(crop, radius)
    return O.compact(crop, nrm)[0]


def _map(scans_and_poses):
    st = None
    for pts, T in scans_and_poses:
        st = O.map_insert(st, pts, LEAF, pose34=None if T is None else np.asarray(T, np.float32))
    return st


@pytest.fixture(scope="module")
def small_map():
    return _map([(_compacted(synth.drift_end_niche(200_000, seed=8), 0.1), None)])


def test_planes_match_numpy_eigh(small_map):
    st = small_map
    pl = M.planes(st["ijk"], st["centroids"], 0.1)
    cells = {tuple(c): i for i, c in enumerate(st["ijk"].tolist())}
    cen = st["centroids"][:, :3].astype(np.float64)
    rng = np.random.default_rng(0)
    checked = 0
    for v in rng.choice(len(cells), 3000, replace=False):
        x, y, z = st["ijk"][v]
        nb = [cells[c] for dz in (-1, 0, 1) for dy in (-1, 0, 1) for dx in (-1, 0, 1) if (c := (x + dx, y + dy, z + dz)) in cells]
        assert pl["count"][v] == len(nb)
        if len(nb) < M.MIN_VOXELS:
            assert not pl["has"][v] and np.isnan(pl["normal"][v]).all()
            continue
        P = cen[nb]
        Cn = (P - P.mean(axis=0)).T @ (P - P.mean(axis=0)) / len(nb)
        C = np.array([[pl["cov"][a, b][v] for b in range(3)] for a in range(3)])
        assert np.abs(C - Cn).max() <= 1e-12 * max(np.abs(Cn).max(), 1e-30)
        w, U = np.linalg.eigh(Cn)
        assert np.abs(pl["vals"][v] - w).max() <= 1e-9 * w[2]
        if w[1] - w[0] > 1e-6 * w[2]:                  # a well separated smallest direction
            n = pl["normal64"][v]
            assert min(np.abs(n - U[:, 0]).max(), np.abs(n + U[:, 0]).max()) <= 1e-9
            checked += 1
        ratio = w[0] / w[1] if w[1] > 0 else np.inf
        if abs(ratio - 0.1) > 1e-6:
            assert pl["has"][v] == (ratio <= 0.1 and w[1] > 0)
    assert checked > 2000 and 0.8 < pl["has"].mean() < 1.0


def _grid(xs, ys, f):
    X, Y = np.meshgrid(xs, ys, indexing="ij")
    return f(X.ravel(), Y.ravel())


def test_flat_sheet_has_a_plane_and_a_corner_does_not():
    s = np.arange(-0.5, 0.5, 0.01) + 0.005
    sheet = _grid(s, s, lambda a, b: np.stack([a, b, np.full_like(a, 0.0123), np.ones_like(a)], axis=1)).astype(np.float32)
    st = _map([(sheet, None)])
    pl = M.planes(st["ijk"], st["centroids"], 0.1)
    inner = (np.abs(st["ijk"][:, :2] + 0.5) < 4).all(axis=1)        # voxels with all 8 sheet neighbours
    assert inner.sum() >= 36 and pl["has"][inner].all()
    assert np.abs(np.abs(pl["normal"][inner][:, 2]) - 1.0).max() <= 1e-6
    # three orthogonal walls meeting at the origin: the corner voxel's neighbourhood spans all three directions
    c = np.arange(0.0, 0.5, 0.01) + 0.005
    walls = [_grid(c, c, lambda a, b: np.stack([a, b, np.full_like(a, 0.005), np.ones_like(a)], axis=1)),
             _grid(c, c, lambda a, b: np.stack([a, np.full_like(a, 0.005), b, np.ones_like(a)], axis=1)),
             _grid(c, c, lambda a, b: np.stack([np.full_like(a, 0.005), a, b, np.ones_like(a)], axis=1))]
    st = _map([(np.concatenate(walls).astype(np.float32), None)])
    pl = M.planes(st["ijk"], st["centroids"], 0.1)
    corner = np.flatnonzero((st["ijk"] == 0).all(axis=1))
    assert len(corner) == 1 and pl["count"][corner[0]] >= M.MIN_VOXELS and not pl["has"][corner[0]]
    assert np.isnan(pl["normal"][corner[0]]).all()


def test_search_equals_kdtree_over_the_candidates(small_map):
    st = small_map
    pm = M.PlaneMap(st["ijk"], st["centroids"], LEAF, 0.1)
    T = synth.pose34(np.radians((1.0, -1.0, 2.0)), (0.12, -0.05, 0.04))
    crop, _ = O.crop(synth.second_scan(synth.drift_end_niche, T, seed=9, n=100_000), 5.0, True)
    src = O.voxel(crop, LEAF)["centroids_fx"]
    far = src[:50].copy()
    far[:, :3] += 20.0
    src = np.concatenate([src, far])
    out = M.icp(src, pm, np.eye(3, 4), max_iterations=1)
    idx = out["index"]
    p = R.transform(src, np.eye(3, 4, dtype=np.float32))
    d, k = cKDTree(pm.cent[:, :3].astype(np.float64)).query(p[:, :3].astype(np.float64))
    acc = idx >= 0
    assert (idx[-50:] == -1).all() and 0.5 * len(idx) < acc.sum() < len(idx)
    assert (d[~acc] >= DMAX * (1 - 1e-6)).all() and (d[acc] < DMAX * (1 + 1e-6)).all()
    e = p[:, :3] - pm.cent[np.where(acc, idx, 0), :3]
    f = pm.cent[k, :3]
    e2 = p[:, :3] - f
    d2_idx = (e[:, 0] * e[:, 0] + e[:, 1] * e[:, 1]) + e[:, 2] * e[:, 2]
    d2_k = (e2[:, 0] * e2[:, 0] + e2[:, 1] * e2[:, 1]) + e2[:, 2] * e2[:, 2]
    other = acc & (k != idx)
    # the k-d tree ranks in float64: where it picks another voxel, both are at the same float distance, the lower key won
    assert np.array_equal(d2_idx[other], d2_k[other]) and (idx[other] < k[other]).all()
    ijk = out["ijk"]
    assert (ijk[~acc] == np.iinfo(np.int32).min).all() and np.array_equal(ijk[acc], pm.ijk[idx[acc]])


# A map of three 1M-point drift scans inserted at their sensor poses (C1: 5 cm normals, 10 cm leaf), planes at ratio 0.1
# (93 % of the 24.7k voxels), and a fourth scan from a known sensor pose registered from the identity.  Measured: 6 .. 8
# iterations, every source centroid matched, rotation errors 3.4e-5 .. 1.7e-4 rad, translation errors 1.15 .. 1.44 mm
# (the voxel centroids of the map sit up to a few mm off curved and edge surfaces, a bias scan-to-scan ICP on the raw
# points does not have).
MAP_POSES = [((0.0, 0.0, 0.0), (0.0, 0.0, 0.0)), ((0.0, 0.0, 2.0), (0.15, 0.03, 0.0)), ((0.0, 0.0, -2.0), (-0.15, -0.03, 0.0))]
RECOVERY_CASES = [((0.0, 0.0, 5.0), (0.3, 0.0, 0.0), 9), ((3.0, -2.0, 2.0), (0.1, -0.2, 0.15), 10),
                  ((-2.0, 4.0, -3.0), (-0.25, 0.1, -0.1), 11)]
MAP_ROT_BAR, MAP_TRANS_BAR = 3e-4, 2e-3


@pytest.fixture(scope="module")
def drift_map():
    scans = [(_compacted(synth.second_scan(synth.drift_end_niche, synth.pose34(np.radians(d), t), seed=40 + k, n=1_000_000)),
              synth.pose34(np.radians(d), t)) for k, (d, t) in enumerate(MAP_POSES)]
    st = _map(scans)
    return M.PlaneMap(st["ijk"], st["centroids"], LEAF, 0.1)


@pytest.mark.parametrize("deg,t,seed", RECOVERY_CASES)
def test_recovers_known_poses_against_a_map(drift_map, deg, t, seed):
    T = synth.pose34(np.radians(deg), t)
    src = O.voxel(_compacted(synth.second_scan(synth.drift_end_niche, T, seed=seed, n=1_000_000)), LEAF)["centroids_fx"]
    out = M.icp(src, drift_map, np.eye(3, 4), d_max=DMAX)
    rot, trans = R.pose_error(out["pose"], T)
    assert out["converged"] == 1 and out["iterations"] < 20 and out["counts"][-1] > 0.9 * len(src)
    assert rot <= MAP_ROT_BAR and trans <= MAP_TRANS_BAR, (rot, trans)
    assert out["n_degenerate"] == 0 and out["eigenvalues"][0] > 1e-2 * out["eigenvalues"][5]


def test_plane_share_on_the_curved_tunnel():
    # the C1 curved tunnel (2 cm noise) at a 10 cm leaf, mapped from its compacted cloud: the share INTEGRATION.md quotes
    st = _map([(_compacted(synth.curved_tunnel(1_000_000, seed=1)), None)])
    assert 0.88 < M.planes(st["ijk"], st["centroids"], 0.1)["has"].mean() < 0.94
    assert M.planes(st["ijk"], st["centroids"], 0.01)["has"].mean() < 0.01
