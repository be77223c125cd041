"""CPU restatement of gm_odometry_step's guess and gate (include/gm_capi.h), TEST INFRASTRUCTURE ONLY.

Poses are 3x4 [R | t].  Compositions take float inputs to double and follow the header's operation order element by
element with unfused numpy float64 arithmetic, so their results are comparable bit for bit with the device's (-fmad=false).
"""
from __future__ import annotations

import numpy as np

MIN_CORRESPONDENCES = 6


def compose(A, B):
    """A o B in double, R[i][j] = (A[i][0]*B[0][j] + A[i][1]*B[1][j]) + A[i][2]*B[2][j], t[i] = (... B[.][3]) + A[i][3]."""
    A, B = np.asarray(A, np.float64), np.asarray(B, np.float64)
    C = np.empty((3, 4))
    for i in range(3):
        for j in range(4):
            C[i, j] = (A[i, 0] * B[0, j] + A[i, 1] * B[1, j]) + A[i, 2] * B[2, j]
        C[i, 3] = C[i, 3] + A[i, 3]
    return C


def inverse(A):
    """[R^T | -(R^T t)], (R^T t)[i] = (R[0][i]*t[0] + R[1][i]*t[1]) + R[2][i]*t[2]."""
    A = np.asarray(A, np.float64)
    C = np.empty((3, 4))
    C[:, :3] = A[:, :3].T
    for i in range(3):
        C[i, 3] = -((A[0, i] * A[0, 3] + A[1, i] * A[1, 3]) + A[2, i] * A[2, 3])
    return C


def f64(P):
    return np.asarray(np.asarray(P, np.float32)[:3, :4], np.float64)


def guess(k, init_pose34, poses, delta34=None):
    """G_k as float32 3x4: poses = the float pose34 of the records 0 .. k-1."""
    if k == 0:
        return np.asarray(init_pose34, np.float32)[:3, :4].copy()
    P1 = f64(poses[k - 1])
    if delta34 is not None:
        D = f64(delta34)
    elif k == 1:
        D = np.eye(3, 4)
    else:
        D = compose(inverse(f64(poses[k - 2])), P1)
    return compose(P1, D).astype(np.float32)


def fitness_rmse(n_correspondences, n_source, sum_r2):
    """The floats gm_get_registration reports."""
    rmse = np.float32(np.sqrt(sum_r2 / n_correspondences)) if n_correspondences > 0 else np.float32(0.0)
    fit = np.float32(n_correspondences / n_source) if n_source > 0 else np.float32(0.0)
    return fit, rmse


def accepted(fitness, n_correspondences, min_fitness, registered=True):
    return (not registered) or (float(np.float32(fitness)) >= min_fitness and n_correspondences >= MIN_CORRESPONDENCES)
