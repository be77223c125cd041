"""The CPU restatement of gm_odometry_step's guess and gate (tests/odometry_oracle.py), checked independently: compositions
against 4x4 homogeneous products and numpy.linalg.inv, constant velocity on a constant screw motion, and gate decisions
at the min_fitness and correspondence-count boundaries."""
import numpy as np

import odometry_oracle as O
from geometric_mapping_b200 import synth


def _random_pose(g):
    return synth.pose34(g.normal(0.0, 1.0, 3), g.uniform(-20.0, 20.0, 3))


def _h(P):
    return np.vstack([np.asarray(P, np.float64), [0.0, 0.0, 0.0, 1.0]])


def test_compose_and_inverse_match_homogeneous_products():
    g = np.random.default_rng(1)
    for _ in range(200):
        A, B = _random_pose(g), _random_pose(g)
        assert np.abs(O.compose(A, B) - (_h(A) @ _h(B))[:3]).max() <= 1e-12
        assert np.abs(O.inverse(A) - np.linalg.inv(_h(A))[:3]).max() <= 1e-12
        assert np.abs(O.compose(O.inverse(A), A) - np.eye(3, 4)).max() <= 1e-12


def test_constant_velocity_reproduces_a_constant_screw_motion():
    M = synth.pose34((0.004, -0.003, 0.02), (0.2, 0.01, -0.005))
    P = [synth.pose34((0.1, 0.2, -0.3), (5.0, -2.0, 1.0))]
    for _ in range(12):
        P.append((_h(P[-1]) @ _h(M))[:3])
    poses = [p.astype(np.float32) for p in P]
    for k in range(2, len(P)):
        G = O.guess(k, None, poses[:k])
        assert G.dtype == np.float32
        # float inputs: the only error is the rounding of P_{k-1}, P_{k-2} and of G (a few float ulps of 10 m)
        assert np.abs(G.astype(np.float64) - P[k]).max() <= 1e-5, k
    assert np.array_equal(O.guess(1, None, poses[:1]), poses[0])  # k = 1: delta = the identity
    assert np.array_equal(O.guess(0, poses[3], []), poses[3])


def test_guess_with_a_motion_prior():
    g = np.random.default_rng(2)
    P0, D = _random_pose(g).astype(np.float32), _random_pose(g).astype(np.float32)
    G = O.guess(1, None, [P0], D)
    ref = (_h(P0.astype(np.float64)) @ _h(D.astype(np.float64)))[:3]
    assert np.abs(G - ref).max() <= 1e-5 and np.array_equal(G, O.compose(P0, D).astype(np.float32))
    assert np.array_equal(O.guess(1, None, [P0], np.eye(3, 4)), P0)  # the identity: constant pose


def test_gate_at_the_fitness_and_correspondence_boundaries():
    fit, _ = O.fitness_rmse(500, 1000, 1.0)
    assert fit == np.float32(0.5) and O.accepted(fit, 500, 0.5)
    fit, _ = O.fitness_rmse(499, 1000, 1.0)
    assert not O.accepted(fit, 499, 0.5)
    # the gate compares the float fitness: a ratio just below 0.5 that rounds to 0.5f is accepted
    fit, _ = O.fitness_rmse(50_000_000 - 1, 100_000_000, 1.0)
    assert fit == np.float32(0.5) and O.accepted(fit, 50_000_000 - 1, 0.5)
    assert not O.accepted(np.float32(1.0), 5, 0.0) and O.accepted(np.float32(1.0), 6, 0.0)
    assert O.accepted(np.float32(1.0), 6, 1.0) and not O.accepted(np.nextafter(np.float32(1.0), np.float32(0.0)), 6, 1.0)
    assert O.accepted(np.float32(0.0), 0, 1.0, registered=False)
    fit, rmse = O.fitness_rmse(0, 0, 0.0)
    assert fit == 0.0 and rmse == 0.0 and not O.accepted(fit, 0, 0.0)
    _, rmse = O.fitness_rmse(4, 10, 4.0)
    assert rmse == np.float32(1.0)
