"""CPU restatement of gm_deskew (include/gm_capi.h), TEST INFRASTRUCTURE ONLY.

The constants and the per-point formula in numpy float64.  Pass the delta as the device sees it (float32, taken to double)
to compare with the device; the device's sin / cos / atan2 may differ from libm's in the last double bit.
"""
from __future__ import annotations

import numpy as np


def constants(delta34):
    """-> theta, u (3), td (3) from D = double(delta34), row-major [R | t]."""
    D = np.asarray(delta34, np.float64)[:3, :4]
    v = np.array([D[2, 1] - D[1, 2], D[0, 2] - D[2, 0], D[1, 0] - D[0, 1]])
    nv = np.sqrt((v[0] * v[0] + v[1] * v[1]) + v[2] * v[2])
    if nv == 0.0:
        return 0.0, np.zeros(3), D[:, 3].copy()
    return float(np.arctan2(nv / 2.0, (((D[0, 0] + D[1, 1]) + D[2, 2]) - 1.0) / 2.0)), v / nv, D[:, 3].copy()


def rotation(delta34, a):
    """R(a) = cos(phi) I + sin(phi) [u]x + (1 - cos(phi)) u u^T, phi = a theta, for every a: n x 3 x 3."""
    theta, u, _ = constants(delta34)
    phi = np.atleast_1d(np.asarray(a, np.float64)) * theta
    K = np.array([[0.0, -u[2], u[1]], [u[2], 0.0, -u[0]], [-u[1], u[0], 0.0]])
    c, s = np.cos(phi)[:, None, None], np.sin(phi)[:, None, None]
    return c * np.eye(3) + s * K + (1.0 - c) * np.outer(u, u)


def deskew(points, t, delta34, t_ref, period):
    """p' = R(a) p + a td, a = ((double)t - t_ref) / period, per point (n x 3 float64); a point with a non-finite
    coordinate or time becomes NaN."""
    p = np.asarray(points, np.float64)[:, :3]
    t64 = np.asarray(t, np.float32).astype(np.float64)
    a = (t64 - t_ref) / period
    _, _, td = constants(delta34)
    out = np.einsum("nij,nj->ni", rotation(delta34, a), p) + a[:, None] * td
    bad = ~(np.isfinite(p).all(axis=1) & np.isfinite(t64))
    out[bad] = np.nan
    return out
