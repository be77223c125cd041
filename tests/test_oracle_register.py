"""CPU checks of the registration oracle (tests/register_oracle.py), the reference gm_register is tested against:
its search equals brute force and a k-d tree, one iteration's normal equations and step equal an independent numpy
float64 restatement, it recovers known transforms on a scene with all six degrees of freedom observable, and on a
straight bore it finds, reports and leaves alone the two unobservable directions."""
import math

import numpy as np
import pytest
from scipy.spatial import cKDTree

import register_oracle as R
from geometric_mapping_b200 import synth
from oracle import oracle as O

RADIUS, LEAF, DMAX = 0.1, 0.1, 0.5


def _target(pts):
    crop, _ = O.crop(pts, 5.0, True)
    nrm, _, _ = O.normals(crop, RADIUS)
    cc, nc, _ = O.compact(crop, nrm)
    return cc, nc


def _centroids(pts):
    crop, _ = O.crop(pts, 5.0, True)
    return O.voxel(crop, LEAF)["centroids_fx"]


@pytest.fixture(scope="module")
def drift():
    return _target(synth.drift_end_niche(200_000, seed=8))


def _flann_d2(p, q):
    d = p[:, :3].astype(np.float32) - q[:, :3].astype(np.float32)
    return (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]


def test_fmaf_is_correctly_rounded():
    g = np.random.Generator(np.random.Philox(3))
    a, b, c = (g.uniform(-8, 8, 200_000).astype(np.float32) for _ in range(3))
    # exact reference: the product and sum in integer arithmetic via Python fractions on a sample
    from fractions import Fraction
    got = R.fmaf(a, b, c)
    for i in range(0, 200_000, 997):
        exact = Fraction(float(a[i])) * Fraction(float(b[i])) + Fraction(float(c[i]))
        f = np.float32(float(exact))
        cands = [np.nextafter(f, np.float32(-np.inf)), f, np.nextafter(f, np.float32(np.inf))]
        errs = [abs(Fraction(float(x)) - exact) for x in cands]
        best = min(errs)
        assert abs(Fraction(float(got[i])) - exact) == best, i


def test_correspondences_equal_brute_force_and_kdtree(drift):
    cc, _ = drift
    T = synth.pose34((0.02, -0.01, 0.03), (0.1, -0.05, 0.08))
    src = _centroids(synth.second_scan(synth.drift_end_niche, T, seed=9, n=100_000))[:3000]
    far = src[:50].copy()
    far[:, :3] += 20.0                     # far outside the target: no correspondence
    src = np.concatenate([src, far])
    p, idx, _ = R.correspondences(src, cc, DMAX, np.eye(3, 4, dtype=np.float32))
    bi, bd2 = O.nn1(p, cc)
    assert np.array_equal(idx, np.where(bd2 < np.float32(DMAX * DMAX), bi, -1))
    assert (idx[-50:] == -1).all() and 0.5 * len(idx) < (idx >= 0).sum() < len(idx)
    d, k = cKDTree(cc[:, :3].astype(np.float64)).query(p[:, :3].astype(np.float64))
    acc = idx >= 0
    # the k-d tree ranks in float64: where it picks another point, both are at the same float distance
    other = acc & (k != idx)
    assert np.array_equal(_flann_d2(p[other], cc[k[other]]), _flann_d2(p[other], cc[idx[other]]))
    assert (d[~acc] >= DMAX * (1 - 1e-6)).all() and (d[acc] < DMAX * (1 + 1e-6)).all()


def test_one_iteration_matches_numpy_float64(drift):
    cc, nc = drift
    T = synth.pose34((0.03, 0.02, -0.04), (0.2, 0.1, -0.1))
    src = _centroids(synth.second_scan(synth.drift_end_niche, T, seed=10, n=200_000))
    init = np.eye(3, 4)
    out = R.icp(src, cc, nc, init, d_max=DMAX, max_iterations=1)
    p, idx, _ = R.correspondences(src, cc, DMAX, init.astype(np.float32))
    assert np.array_equal(idx, out["index"])
    ok = idx >= 0
    P, Q, N = (a.astype(np.float64) for a in (p[ok, :3], cc[idx[ok], :3], nc[idx[ok], :3]))
    r = np.einsum("ij,ij->i", N, P - Q)
    J = np.hstack([np.cross(P, N), N])
    A, g = J.T @ J, J.T @ r
    assert np.abs(out["A"] - A).max() <= 1e-12 * np.abs(A).max()
    assert np.abs(out["g"] - g).max() <= 1e-12 * np.abs(g).max()
    w, U = np.linalg.eigh(A)
    xi = -(U @ ((U.T @ g) / w))
    assert np.abs(out["xi"] - xi).max() <= 1e-9 * np.abs(xi).max()
    assert np.abs(out["eigenvalues"] - w).max() <= 1e-10 * w[-1]
    V = out["eigenvectors"]
    assert np.abs(V @ np.diag(out["eigenvalues"]) @ V.T - A).max() <= 1e-10 * w[-1]
    assert out["n_degenerate"] == 0 and out["counts"] == [int(ok.sum())]
    np.testing.assert_array_equal(out["residual"][ok], r.astype(np.float32))  # same operation order as the oracle's


# Known transforms (sensor pose of the second scan) up to 5 degrees and 0.3 m, from the identity guess, at the configuration
# of the GPU test: 1M-point scans, C1 (5 cm normals, 10 cm leaf).  Measured: 11 iterations, rotation errors
# 7.2e-5 .. 1.3e-4 rad, translation errors 0.13 .. 0.30 mm.  The smallest eigenvalue, 2.4 .. 3.7 % of the largest, is
# x-translation: only the end face and the niche's x-sides see it.
RECOVERY_CASES = [((0.0, 0.0, 5.0), (0.3, 0.0, 0.0), 9), ((3.0, -2.0, 2.0), (0.1, -0.2, 0.15), 10),
                  ((-2.0, 4.0, -3.0), (-0.25, 0.1, -0.1), 11)]
ROT_BAR, TRANS_BAR = 3e-4, 1e-3


@pytest.fixture(scope="module")
def drift_1m():
    crop, _ = O.crop(synth.drift_end_niche(1_000_000, seed=8), 5.0, True)
    nrm, _, _ = O.normals(crop, 0.05)
    cc, nc, _ = O.compact(crop, nrm)
    return cc, nc


@pytest.mark.parametrize("deg,t,seed", RECOVERY_CASES)
def test_recovers_known_transforms(drift_1m, deg, t, seed):
    cc, nc = drift_1m
    T = synth.pose34(np.radians(deg), t)
    crop, _ = O.crop(synth.second_scan(synth.drift_end_niche, T, seed=seed, n=1_000_000), 5.0, True)
    nrm, _, _ = O.normals(crop, 0.05)
    src = O.voxel(O.compact(crop, nrm)[0], LEAF)["centroids_fx"]
    out = R.icp(src, cc, nc, np.eye(3, 4), d_max=DMAX, max_iterations=30)
    rot, trans = R.pose_error(out["pose"], T)
    assert out["converged"] == 1 and out["iterations"] < 20
    assert rot <= ROT_BAR and trans <= TRANS_BAR, (rot, trans)
    assert out["n_degenerate"] == 0 and out["eigenvalues"][0] > 1e-2 * out["eigenvalues"][5]
    assert abs(out["eigenvectors"][3, 0]) > 0.99                                  # ... and it belongs to vx


# C0: a straight bore along x does not constrain x-translation nor rotation about x.  Measured spectrum / lambda_max:
# 4.2e-4 (vx), 2.3e-3 (wx), then 0.18, 0.18, 1.0, 1.0: ratio 1e-2 separates the two by almost two decades each way.
C0_RATIO = 1e-2


def test_straight_bore_reports_and_keeps_unobservable_directions():
    cc, nc = _target(synth.straight_cylinder(200_000, seed=1, half_length=4.0))
    src = _centroids(synth.second_scan(synth.straight_cylinder, np.eye(3, 4), seed=3, n=200_000, half_length=4.0))
    init = synth.pose34(np.radians((2.0, 1.0, 0.0)), (0.2, 0.05, -0.04))  # x parts unobservable, the rest wrong
    out = R.icp(src, cc, nc, init, d_max=DMAX, max_iterations=30, degeneracy_ratio=C0_RATIO)
    vals, V = out["eigenvalues"], out["eigenvectors"]
    assert vals[1] <= C0_RATIO * vals[5] < vals[2]
    # the two smallest eigenvectors span (wx, vx) within 1e-2
    for k in (0, 1):
        assert V[0, k] ** 2 + V[3, k] ** 2 >= 1.0 - 1e-2
    assert abs(V[3, 0]) > 0.99 and abs(V[0, 1]) > 0.99
    assert out["n_degenerate"] == 2 and out["converged"] == 1
    P = out["pose"]
    dR = P[:, :3] @ init[:, :3].T
    assert abs(P[0, 3] - init[0, 3]) <= 2e-3 and abs(math.asin(dR[2, 1])) <= 5e-4   # measured 0.66 mm, 6.7e-5 rad
    assert abs(P[1, 3]) <= 2e-3 and abs(P[2, 3]) <= 2e-3 and abs(P[0, 2]) <= 5e-4   # the observable ones are corrected
    plain = R.icp(src, cc, nc, init, d_max=DMAX, max_iterations=30)
    assert plain["n_degenerate"] == 0 and abs(plain["pose"][0, 3] - init[0, 3]) > 0.05  # plain Gauss-Newton slides (measured 0.17 m)
