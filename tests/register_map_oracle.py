"""CPU restatement of gm_register_map (include/gm_capi.h): scan-to-map point-to-plane ICP, TEST INFRASTRUCTURE ONLY.

Map planes follow k_map_planes' operation order, vectorised over the voxels: the 27 neighbour offsets in ascending
(dz, dy, dx) order, sequential double sums for the mean and the covariance, and a numpy copy of d_jacobi3 whose
element-wise float64 operations round as the device's unfused ones do.  So the planes are comparable bit for bit.  The
search is the oracle's exact grid 1-NN (FLANN distance in float, ties -> lowest index) over the centroids of the voxels
with a plane in key order, so the lowest index is the lowest map key.  The ICP loop reuses register_oracle's transform,
linearisation, Jacobi, step and update.
"""
from __future__ import annotations

import math

import numpy as np

import register_oracle as R

MIN_VOXELS = 5
_OFF = 1 << 20
_M21 = (1 << 21) - 1


def pack(ijk):
    """map_pack of integer cells (n x 3) -> (int64 key, in range)."""
    a = np.asarray(ijk, np.int64)
    ok = ((a >= -_OFF) & (a < _OFF)).all(axis=1)
    k = (a[:, 0] + _OFF) | ((a[:, 1] + _OFF) << 21) | ((a[:, 2] + _OFF) << 42)
    return k, ok


def jacobi3(C):
    """d_jacobi3 vectorised: C = dict (a, b) -> float64 array for a, b in 0..2.  -> vals (n x 3 ascending), vecs (n x 3 x 3,
    vecs[:, r, k] = component r of eigenvector k)."""
    n = C[0, 0].shape[0]
    A = [[C[i, j].astype(np.float64).copy() for j in range(3)] for i in range(3)]
    V = [[np.full(n, 1.0 if i == j else 0.0) for j in range(3)] for i in range(3)]
    active = np.ones(n, bool)
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        for _ in range(64):
            off = A[0][1] * A[0][1] + A[0][2] * A[0][2] + A[1][2] * A[1][2]
            diag = A[0][0] * A[0][0] + A[1][1] * A[1][1] + A[2][2] * A[2][2]
            active &= ~((off <= 1e-300) | (off <= 1e-34 * diag))
            if not active.any():
                break
            for p in range(2):
                for q in range(p + 1, 3):
                    rot = active & (A[p][q] != 0.0)
                    theta = (A[q][q] - A[p][p]) / (2.0 * A[p][q])
                    t = np.where(theta >= 0.0, 1.0, -1.0) / (np.abs(theta) + np.sqrt(theta * theta + 1.0))
                    c = 1.0 / np.sqrt(t * t + 1.0)
                    s = t * c
                    for k in range(3):
                        akp, akq = A[k][p], A[k][q]
                        A[k][p], A[k][q] = np.where(rot, c * akp - s * akq, akp), np.where(rot, s * akp + c * akq, akq)
                    for k in range(3):
                        apk, aqk = A[p][k], A[q][k]
                        A[p][k], A[q][k] = np.where(rot, c * apk - s * aqk, apk), np.where(rot, s * apk + c * aqk, aqk)
                    for k in range(3):
                        vkp, vkq = V[k][p], V[k][q]
                        V[k][p], V[k][q] = np.where(rot, c * vkp - s * vkq, vkp), np.where(rot, s * vkp + c * vkq, vkq)
    d = np.stack([A[0][0], A[1][1], A[2][2]], axis=1)
    order = np.argsort(d, axis=1, kind="stable")            # the device's stable insertion sort
    rows = np.arange(n)
    vals = d[rows[:, None], order]
    vecs = np.empty((n, 3, 3))
    for k in range(3):
        c = order[:, k]
        v = [np.stack([V[r][0], V[r][1], V[r][2]], axis=1)[rows, c] for r in range(3)]
        nrm = np.sqrt(v[0] * v[0] + v[1] * v[1] + v[2] * v[2])
        big = np.zeros(n, np.int64)
        big = np.where(np.abs(v[1]) > np.abs(v[0]), 1, big)
        big = np.where(np.abs(v[2]) > np.abs(np.choose(big, v)), 2, big)
        sgn = np.where(np.choose(big, v) < 0.0, -1.0, 1.0)
        for r in range(3):
            vecs[:, r, k] = sgn * v[r] / nrm
    return vals, vecs


def planes(ijk, centroids, max_planarity):
    """Planes of a map given as gm_map_download / oracle.map_insert arrays (voxels in key order).  -> dict: "has" (bool),
    "normal" (V x 3 float32, NaN without a plane), "normal64", "vals" (V x 3, NaN below MIN_VOXELS), "count" (|N(v)|),
    "cov" (dict (a, b) -> V float64)."""
    ijk = np.asarray(ijk, np.int64)
    cen = np.asarray(centroids, np.float32)[:, :3].astype(np.float64)
    V = ijk.shape[0]
    keys, _ = pack(ijk)
    assert (np.diff(keys) > 0).all(), "voxels must be in key order"
    nb = []                                                  # per offset: (found mask, neighbour index)
    for dz in (-1, 0, 1):
        for dy in (-1, 0, 1):
            for dx in (-1, 0, 1):
                k, ok = pack(ijk + np.array([dx, dy, dz]))
                pos = np.minimum(np.searchsorted(keys, k), max(V - 1, 0))
                found = ok & (V > 0) & (keys[pos] == k) if V else np.zeros(0, bool)
                nb.append((found, pos))
    m = np.zeros(V, np.int64)
    mu = np.zeros((V, 3))
    for found, pos in nb:
        m += found
        mu = np.where(found[:, None], mu + cen[pos], mu)
    with np.errstate(divide="ignore", invalid="ignore"):
        mu = mu / m[:, None].astype(np.float64)
    pairs = [(0, 0), (0, 1), (0, 2), (1, 1), (1, 2), (2, 2)]
    cov = {ab: np.zeros(V) for ab in pairs}
    for found, pos in nb:
        d = cen[pos] - mu
        for a, b in pairs:
            cov[a, b] = np.where(found, cov[a, b] + d[:, a] * d[:, b], cov[a, b])
    for ab in pairs:
        with np.errstate(divide="ignore", invalid="ignore"):
            cov[ab] = cov[ab] / m.astype(np.float64)
    for a, b in pairs:
        cov[b, a] = cov[a, b]
    ok = m >= MIN_VOXELS
    vals = np.full((V, 3), np.nan)
    n64 = np.full((V, 3), np.nan)
    if ok.any():
        va, ve = jacobi3({ab: c[ok] for ab, c in cov.items()})
        vals[ok] = va
        n64[ok] = ve[:, :, 0]
    with np.errstate(invalid="ignore"):
        has = ok & (vals[:, 0] <= max_planarity * vals[:, 1]) & (vals[:, 1] > 0.0)
    normal = np.where(has[:, None], n64, np.nan).astype(np.float32)
    return {"has": has, "normal": normal, "normal64": n64, "vals": vals, "count": m, "cov": cov}


def planes_xyzw(pl):
    """The layout of gm_map_download_planes."""
    out = np.empty((pl["has"].shape[0], 4), np.float32)
    out[:, :3] = pl["normal"]
    out[:, 3] = pl["has"].astype(np.float32)
    return out


class PlaneMap:
    """Search target of the restatement: the voxels with a plane, in key order."""

    def __init__(self, ijk, centroids, leaf, max_planarity=0.1):
        self.pl = planes(ijk, centroids, max_planarity)
        has = self.pl["has"]
        self.leaf = float(leaf)
        self.ijk = np.asarray(ijk, np.int32)[has]
        self.cent = np.ascontiguousarray(np.asarray(centroids, np.float32)[has])
        self.nrm = np.zeros((self.cent.shape[0], 4), np.float32)
        self.nrm[:, :3] = self.pl["normal"][has]


def to_ijk(pm, idx):
    """candidate index or -1 -> the map cell or INT32_MIN x 3 (gm_download_map_correspondences)."""
    out = np.full((idx.shape[0], 3), np.iinfo(np.int32).min, np.int32)
    out[idx >= 0] = pm.ijk[idx[idx >= 0]]
    return out


def icp(src4, pm, init_pose34, d_max=0.5, max_iterations=30, min_rotation_step=1e-5, min_translation_step=1e-5,
        degeneracy_ratio=0.0):
    """gm_register_map on the CPU against a PlaneMap.  -> the dict of register_oracle.icp, with "index" the candidate
    index and "ijk" the matched cells of the last executed iteration."""
    src4 = np.ascontiguousarray(src4, np.float32)
    T = np.asarray(np.asarray(init_pose34, np.float32)[:3, :4], np.float64)
    out = {"poses": [], "counts": [], "converged": 0}
    for _ in range(max_iterations):
        out["poses"].append(T.copy())
        p, idx, _ = R.correspondences(src4, pm.cent, d_max, T.astype(np.float32), pm.leaf)
        r, J = R.linearise(p, pm.cent, pm.nrm, idx)
        A, g, sr2 = R.normal_equations(r, J)
        vals, vecs = R.jacobi6(A)
        xi, ndeg = R.step(vals, vecs, g, degeneracy_ratio)
        res = np.full(src4.shape[0], np.nan, np.float32)
        res[idx >= 0] = r.astype(np.float32)
        m = int(r.shape[0])
        out["counts"].append(m)
        out.update(index=idx, ijk=to_ijk(pm, idx), residual=res, A=A, g=g, sum_r2=sr2, xi=xi, eigenvalues=vals,
                   eigenvectors=vecs, n_degenerate=ndeg)
        if m < 6 or not (vals[5] > 0.0):
            break
        T = R.update(T, xi)
        if math.sqrt((xi[0] * xi[0] + xi[1] * xi[1]) + xi[2] * xi[2]) < min_rotation_step and \
                math.sqrt((xi[3] * xi[3] + xi[4] * xi[4]) + xi[5] * xi[5]) < min_translation_step:
            out["converged"] = 1
            break
    out["pose"] = T
    out["iterations"] = len(out["counts"])
    return out
