"""CPU restatement of gm_register (include/gm_capi.h): point-to-plane ICP, TEST INFRASTRUCTURE ONLY.

The search is the oracle's exact grid 1-NN (oracle.nn1_grid: FLANN distance in float, ties -> lowest index) thresholded
at float(d_max * d_max).  The transform reproduces the device's fmaf chains bit for bit (an exactly rounded float fma
from float64 arithmetic, see fmaf below), and the residuals follow the device's unfused double operation order, so
correspondences and residuals are comparable bit for bit.  The sums run in double in ascending source order (the
device sums in block partials: equal to rounding), and the Jacobi eigen-solver, the step and the Rodrigues update
repeat the device's operation sequence in Python floats.
"""
from __future__ import annotations

import math

import numpy as np

from oracle import oracle as O


def fmaf(a, b, c):
    """float32 fma(a, b, c), correctly rounded, element-wise.  a*b is exact in float64 (24 + 24 bits); s = a*b + c in
    float64 with its exact error e (TwoSum).  Rounding s to float32 is the correctly rounded result unless s lies
    exactly halfway between two floats and e != 0: then e decides the side."""
    a64, b64, c64 = (np.asarray(v, np.float32).astype(np.float64) for v in (a, b, c))
    P = a64 * b64
    s = P + c64
    bb = s - P
    e = (P - (s - bb)) + (c64 - bb)
    f = s.astype(np.float32)
    f64 = f.astype(np.float64)
    up = np.nextafter(f, np.float32(np.inf)).astype(np.float64)
    dn = np.nextafter(f, np.float32(-np.inf)).astype(np.float64)
    tie_up = (s == 0.5 * (f64 + up)) & (e != 0)   # s is the midpoint above f
    tie_dn = (s == 0.5 * (f64 + dn)) & (e != 0)   # s is the midpoint below f
    out = f.copy()
    out[tie_up & (e > 0)] = up[tie_up & (e > 0)].astype(np.float32)
    out[tie_dn & (e < 0)] = dn[tie_dn & (e < 0)].astype(np.float32)
    return out


def transform(pts4, pose34_f32):
    """p = Tf c with the fmaf chains of k_map_insert / k_reg_iter."""
    T = np.asarray(pose34_f32, np.float32).reshape(12)
    c = np.ascontiguousarray(pts4, np.float32)
    x, y, z = c[:, 0], c[:, 1], c[:, 2]
    out = np.empty((c.shape[0], 4), np.float32)
    for r in range(3):
        out[:, r] = fmaf(T[4 * r], x, fmaf(T[4 * r + 1], y, fmaf(T[4 * r + 2], z, T[4 * r + 3])))
    out[:, 3] = 1.0
    return out


def correspondences(src4, tgt4, d_max, pose34_f32, cell=0.1):
    """-> transformed source points, target index or -1, float d^2 of every source point."""
    p = transform(src4, pose34_f32)
    idx = np.full(p.shape[0], -1, np.int32)
    d2 = np.full(p.shape[0], np.inf, np.float32)
    if tgt4.shape[0] == 0:
        return p, idx, d2
    # a query at least d_max (with a margin for the float distance) from the target's bounding box has no correspondence;
    # skipping it only saves time: the grid search's rings would walk out to the whole cloud for it
    lo, hi = tgt4[:, :3].min(axis=0).astype(np.float64), tgt4[:, :3].max(axis=0).astype(np.float64)
    gap = np.maximum(np.maximum(lo - p[:, :3], p[:, :3] - hi), 0.0)
    near = np.sqrt((gap * gap).sum(axis=1)) < d_max * 1.001
    if near.any():
        i, d = O.nn1_grid(p[near], tgt4, cell)
        idx[near], d2[near] = i, d
    r2max = np.float32(d_max * d_max)
    idx = np.where((idx >= 0) & (d2 < r2max), idx, -1).astype(np.int32)
    return p, idx, d2


def linearise(p, tgt4, nrm8, idx):
    """-> r (m,), J (m x 6) in float64 for the accepted points, in ascending source order."""
    ok = idx >= 0
    P = p[ok, :3].astype(np.float64)
    Q = tgt4[idx[ok], :3].astype(np.float64)
    N = nrm8[idx[ok], :3].astype(np.float64)
    d = P - Q
    r = (N[:, 0] * d[:, 0] + N[:, 1] * d[:, 1]) + N[:, 2] * d[:, 2]
    J = np.stack([P[:, 1] * N[:, 2] - P[:, 2] * N[:, 1], P[:, 2] * N[:, 0] - P[:, 0] * N[:, 2],
                  P[:, 0] * N[:, 1] - P[:, 1] * N[:, 0], N[:, 0], N[:, 1], N[:, 2]], axis=1)
    return r, J


def _seqsum(v):
    return float(np.cumsum(v)[-1]) if v.shape[0] else 0.0


def normal_equations(r, J):
    """A (6x6), g (6,), sum r^2 summed sequentially in ascending source order."""
    A = np.zeros((6, 6))
    for a in range(6):
        for b in range(a, 6):
            A[a, b] = A[b, a] = _seqsum(J[:, a] * J[:, b])
    g = np.array([_seqsum(J[:, a] * r) for a in range(6)])
    return A, g, _seqsum(r * r)


def jacobi6(Ain):
    """d_jacobi6: cyclic Jacobi, ascending eigenvalues, unit eigenvector columns with their largest-|component| positive."""
    A = [[float(Ain[i][j]) for j in range(6)] for i in range(6)]
    V = [[1.0 if i == j else 0.0 for j in range(6)] for i in range(6)]
    for _ in range(64):
        off = 0.0
        for p in range(5):
            for q in range(p + 1, 6):
                off += A[p][q] * A[p][q]
        diag = 0.0
        for i in range(6):
            diag += A[i][i] * A[i][i]
        if off <= 1e-300 or off <= 1e-34 * diag:
            break
        for p in range(5):
            for q in range(p + 1, 6):
                if A[p][q] == 0.0:
                    continue
                theta = (A[q][q] - A[p][p]) / (2.0 * A[p][q])
                t = (1.0 if theta >= 0.0 else -1.0) / (abs(theta) + math.sqrt(theta * theta + 1.0))
                c = 1.0 / math.sqrt(t * t + 1.0)
                s = t * c
                for k in range(6):
                    akp, akq = A[k][p], A[k][q]
                    A[k][p], A[k][q] = c * akp - s * akq, s * akp + c * akq
                for k in range(6):
                    apk, aqk = A[p][k], A[q][k]
                    A[p][k], A[q][k] = c * apk - s * aqk, s * apk + c * aqk
                for k in range(6):
                    vkp, vkq = V[k][p], V[k][q]
                    V[k][p], V[k][q] = c * vkp - s * vkq, s * vkp + c * vkq
    d = [A[i][i] for i in range(6)]
    order = [0, 1, 2, 3, 4, 5]
    for i in range(1, 6):
        o, j = order[i], i - 1
        while j >= 0 and d[order[j]] > d[o]:
            order[j + 1] = order[j]
            j -= 1
        order[j + 1] = o
    vals = np.empty(6)
    vecs = np.empty((6, 6))
    for k in range(6):
        c = order[k]
        vals[k] = d[c]
        n2, big = 0.0, 0
        for r in range(6):
            n2 += V[r][c] * V[r][c]
            if abs(V[r][c]) > abs(V[big][c]):
                big = r
        n, sgn = math.sqrt(n2), (-1.0 if V[big][c] < 0.0 else 1.0)
        for r in range(6):
            vecs[r, k] = sgn * V[r][c] / n
    return vals, vecs


def step(vals, vecs, g, ratio):
    """xi = -sum over kept k of (v_k.g / lambda_k) v_k; -> xi, number of dropped directions."""
    xi = [0.0] * 6
    ndeg = 0
    lmax = vals[5]
    for k in range(6):
        if not (vals[k] > ratio * lmax):
            ndeg += 1
            continue
        dot = 0.0
        for i in range(6):
            dot += vecs[i, k] * g[i]
        coef = dot / vals[k]
        for i in range(6):
            xi[i] -= coef * vecs[i, k]
    return np.array(xi), ndeg


def rodrigues(w):
    th2 = (w[0] * w[0] + w[1] * w[1]) + w[2] * w[2]
    th = math.sqrt(th2)
    if th < 1e-6:
        a, b = 1.0 - th2 / 6.0, 0.5 - th2 / 24.0
    else:
        s = math.sin(0.5 * th)
        a, b = math.sin(th) / th, 2.0 * s * s / th2
    K = [0.0, -w[2], w[1], w[2], 0.0, -w[0], -w[1], w[0], 0.0]
    R = np.empty((3, 3))
    for i in range(3):
        for j in range(3):
            R[i, j] = ((1.0 if i == j else 0.0) + a * K[3 * i + j]) + b * (w[i] * w[j] - (th2 if i == j else 0.0))
    return R


def update(T, xi):
    """T_{i+1} = [R(w) | v] o T_i, in the device's operation order."""
    R = rodrigues(xi[:3])
    out = np.empty((3, 4))
    for i in range(3):
        for j in range(3):
            out[i, j] = (R[i, 0] * T[0, j] + R[i, 1] * T[1, j]) + R[i, 2] * T[2, j]
        out[i, 3] = ((R[i, 0] * T[0, 3] + R[i, 1] * T[1, 3]) + R[i, 2] * T[2, 3]) + xi[3 + i]
    return out


def icp(src4, tgt4, nrm8, init_pose34, d_max=0.5, max_iterations=30, min_rotation_step=1e-5, min_translation_step=1e-5,
        degeneracy_ratio=0.0, cell=0.1):
    """gm_register on the CPU.  -> dict: "pose" (3x4 float64 after the last update; float32 of it = the reported pose),
    "poses" (input pose of every executed iteration, float64), "iterations", "converged", "counts" (m per iteration),
    and of the last executed iteration: "index", "residual" (float32, NaN without correspondence), "A", "g", "sum_r2",
    "xi", "eigenvalues", "eigenvectors", "n_degenerate"."""
    src4 = np.ascontiguousarray(src4, np.float32)
    tgt4 = np.ascontiguousarray(tgt4, np.float32)
    nrm8 = np.ascontiguousarray(nrm8, np.float32)
    T = np.asarray(np.asarray(init_pose34, np.float32)[:3, :4], np.float64)
    out = {"poses": [], "counts": [], "converged": 0}
    for _ in range(max_iterations):
        out["poses"].append(T.copy())
        p, idx, _ = correspondences(src4, tgt4, d_max, T.astype(np.float32), cell)
        r, J = linearise(p, tgt4, nrm8, idx)
        A, g, sr2 = normal_equations(r, J)
        vals, vecs = jacobi6(A)
        xi, ndeg = step(vals, vecs, g, degeneracy_ratio)
        res = np.full(src4.shape[0], np.nan, np.float32)
        res[idx >= 0] = r.astype(np.float32)
        m = int(r.shape[0])
        out["counts"].append(m)
        out.update(index=idx, residual=res, A=A, g=g, sum_r2=sr2, xi=xi, eigenvalues=vals, eigenvectors=vecs, n_degenerate=ndeg)
        if m < 6 or not (vals[5] > 0.0):
            break
        T = update(T, xi)
        if math.sqrt((xi[0] * xi[0] + xi[1] * xi[1]) + xi[2] * xi[2]) < min_rotation_step and \
                math.sqrt((xi[3] * xi[3] + xi[4] * xi[4]) + xi[5] * xi[5]) < min_translation_step:
            out["converged"] = 1
            break
    out["pose"] = T
    out["iterations"] = len(out["counts"])
    return out


def pose_error(T_est, T_true):
    """(rotation error in rad, translation error in m) of T_est against T_true (3x4 each)."""
    Te, Tt = np.asarray(T_est, np.float64), np.asarray(T_true, np.float64)
    dR = Te[:, :3] @ Tt[:, :3].T
    # atan2 of the skew and symmetric parts: acos of the trace alone cannot resolve angles below ~3e-4 rad of a float pose
    s = 0.5 * math.sqrt((dR[2, 1] - dR[1, 2]) ** 2 + (dR[0, 2] - dR[2, 0]) ** 2 + (dR[1, 0] - dR[0, 1]) ** 2)
    ang = math.atan2(s, (np.trace(dR) - 1.0) / 2.0)
    return ang, float(np.linalg.norm(Te[:, 3] - Tt[:, 3]))
