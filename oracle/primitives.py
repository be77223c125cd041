"""Sequential multi-primitive extraction and its compression, restated on the CPU oracle (test infrastructure only).

The semantics of gm_extract_primitives (include/gm_capi.h), built from the existing oracle calls: hypotheses from the
ORIGINAL compacted cloud at the mapped sample indices, counts and refits over a copy in which the claimed points are NaN
(the oracle's inlier tests are the same fma forms and reject NaN), claims = the inliers of the winning hypothesis
(gmo_labels applies exactly that fma test).  Extents and RMS of the compression are taken in numpy double.
"""
from __future__ import annotations

import numpy as np

from . import oracle as O


def draw_positions(draws, n):
    """uint32 draws -> positions (u * n) >> 32 in [0, n) of the remaining list (n >= 1)."""
    return ((np.asarray(draws, np.uint32).astype(np.uint64) * np.uint64(n)) >> np.uint64(32)).astype(np.int64)


def map_draws(draws, rem):
    """uint32 draws -> sample indices rem[(u * n) >> 32], or -1 when n = 0 (pure integer rule)."""
    n = len(rem)
    if n == 0:
        return np.full(np.shape(draws), -1, np.int32)
    return np.asarray(rem, np.int32)[draw_positions(draws, n)]


def extract(cloud, normals8, plane_draws, cyl_draws, max_primitives, min_inliers, tau=0.05, rmin=0.5, rmax=10.0, refit_iters=5,
            trace=None):
    """-> (list of primitive dicts, uint8 ids).  plane_draws: K x Hp x 3, cyl_draws: K x Hc x 2 (None = no such kind).
    trace: a list that receives (n_r, best plane count, best cylinder count) of every round run, the stopping one
    included (-1 = no valid hypothesis of that kind)."""
    cloud = np.ascontiguousarray(cloud, np.float32)
    ids = np.zeros(len(cloud), np.uint8)
    work = cloud.copy()
    prims = []
    for r in range(max_primitives):
        rem = np.flatnonzero(ids == 0).astype(np.int32)
        best = [(-1, -1, None), (-1, -1, None)]  # (count, id, tables) per kind
        if plane_draws is not None and plane_draws.shape[1]:
            coef, valid = O.plane_hypotheses(cloud, map_draws(plane_draws[r], rem))
            counts = O.count_plane(work, coef, valid, tau)
            b = O.argmax(counts)
            if b >= 0:
                best[0] = (int(counts[b]), b, coef)
        if cyl_draws is not None and cyl_draws.shape[1]:
            m7, t12, valid = O.cyl_hypotheses(cloud, normals8, map_draws(cyl_draws[r], rem), rmin, rmax, tau)
            counts = O.count_cyl(work, t12, valid)
            b = O.argmax(counts)
            if b >= 0:
                best[1] = (int(counts[b]), b, (m7, t12))
        if trace is not None:
            trace.append((len(rem), best[0][0], best[1][0]))
        kind = 0 if best[0][0] >= best[1][0] else 1
        count, b, tab = best[kind]
        if count < max(min_inliers, 1):
            break
        if kind == 0:
            hyp = tab[b]
            coef_r, refit_count = O.refit_plane(work, hyp, tau)
            claim = O.labels(work, hyp, tau, None) == 1
            rms = None
        else:
            hyp = tab[0][b]
            coef_r, refit_count, rms = O.refit_cylinder(work, hyp, tab[1][b], refit_iters)
            claim = O.labels(work, None, tau, tab[1][b]) == 2
        assert int(claim.sum()) == count
        ids[claim] = r + 1
        work[claim, :3] = np.nan
        prims.append({"kind": kind, "best_id": b, "best_count": count, "refit_count": refit_count, "n_remaining": len(rem),
                      "hyp": np.asarray(hyp, np.float32), "coef": np.asarray(coef_r, np.float32), "rms": rms})
    return prims, ids


def perp_basis_d(d):
    """The canonical perpendicular basis (u, w) of unit `d`, as gm_compress and the cylinder refit build it."""
    d = np.asarray(d, np.float64)
    k = int(np.argmin(np.abs(d)))  # ties -> lowest axis
    c = [np.array([0.0, d[2], -d[1]]), np.array([-d[2], 0.0, d[0]]), np.array([d[1], -d[0], 0.0])][k]
    u = c / np.sqrt(c[0] * c[0] + c[1] * c[1] + c[2] * c[2])
    return u, np.cross(d, u)


def compress(cloud, ids, prims, leaf):
    """Compression of an extraction result: per-primitive count / extents / RMS, residual voxels (O.voxel), totals."""
    p = np.asarray(cloud, np.float64)[:, :3]
    recs, sq = [], 0.0
    for k, pr in enumerate(prims):
        q = p[ids == k + 1]
        c = pr["coef"].astype(np.float64)
        ext = np.zeros(4)
        if pr["kind"] == 0:
            u, v = perp_basis_d(c[:3])
            e = q @ c[:3] + c[3]
            if len(q):
                pu, pv = q @ u, q @ v
                ext = np.array([pu.min(), pu.max(), pv.min(), pv.max()])
        else:
            u, w = perp_basis_d(c[3:6])
            d = q - c[:3]
            e = np.sqrt((d @ u) ** 2 + (d @ w) ** 2) - c[6]
            if len(q):
                t = d @ c[3:6]
                ext = np.array([t.min(), t.max(), 0.0, 0.0])
        sq += float((e * e).sum())
        recs.append({"kind": pr["kind"], "count": len(q), "coef": c[: 4 if pr["kind"] == 0 else 7], "extents": ext,
                     "rms": float(np.sqrt((e * e).mean())) if len(q) else 0.0})
    res = np.ascontiguousarray(np.asarray(cloud, np.float32)[ids == 0])
    vox = O.voxel(res, leaf)
    V = vox["V"]
    rsq = float(((res[:, :3].astype(np.float64) - vox["centroids_fx"][vox["assign"], :3]) ** 2).sum()) if len(res) and V else 0.0
    n = len(p)
    return {"records": recs, "n_points": n, "n_residual": len(res), "n_residual_voxels": V, "residual_centroids": vox["centroids_fx"],
            "residual_rms": float(np.sqrt(rsq / len(res))) if len(res) else 0.0,
            "total_rms": float(np.sqrt((sq + rsq) / n)) if n else 0.0}


# ---- float64 refit references, independent of the oracle's refit code ---------------------------------------------
def plane_fit_d(pts):
    """Total-least-squares plane of `pts` in float64: the normal is the eigenvector of the smallest eigenvalue of the
    (population) covariance, d = -n . mean and rms = sqrt(lambda_min).  -> (n, d, rms)."""
    p = np.asarray(pts, np.float64)[:, :3]
    m = p.mean(0)
    q = p - m
    vals, vecs = np.linalg.eigh(q.T @ q / len(p))
    n = vecs[:, 0]
    return n, float(-n @ m), float(np.sqrt(max(vals[0], 0.0)))


def cylinder_residuals_d(pts, q, axis, r):
    """Orthogonal distances |p - axis line| - r in float64 (axis need not be unit)."""
    p = np.asarray(pts, np.float64)[:, :3]
    a = np.asarray(axis, np.float64)
    a = a / np.linalg.norm(a)
    v = p - np.asarray(q, np.float64)
    return np.linalg.norm(v - np.outer(v @ a, a), axis=1) - float(r)


def cylinder_rms_d(pts, coef7):
    """RMS of the orthogonal residuals of `pts` at the cylinder coef7 = (q, axis, r), evaluated directly in float64."""
    c = np.asarray(coef7, np.float64)
    e = cylinder_residuals_d(pts, c[:3], c[3:6], c[6])
    return float(np.sqrt((e * e).mean()))


def cylinder_fit_d(pts, coef7, tol=1e-15, passes=4):
    """Least-squares cylinder of `pts` in float64 (scipy.optimize.least_squares) from the start coef7 = (q, axis, r).
    The five free parameters are a chart around the current model: q moves in the plane perpendicular to the axis and
    the axis tilts along the same basis; the chart is recentred after every pass.  -> (q, unit axis, r, rms)."""
    from scipy.optimize import least_squares

    p = np.asarray(pts, np.float64)[:, :3]
    c = np.asarray(coef7, np.float64)
    q, a, r = c[:3].copy(), c[3:6] / np.linalg.norm(c[3:6]), float(c[6])
    for _ in range(passes):
        u, w = perp_basis_d(a)

        def model(x, q=q, a=a, u=u, w=w):
            d = a + x[2] * u + x[3] * w
            return q + x[0] * u + x[1] * w, d / np.linalg.norm(d)

        def fun(x):
            qq, dd = model(x)
            return cylinder_residuals_d(p, qq, dd, r + x[4])

        x = least_squares(fun, np.zeros(5), method="lm", xtol=tol, ftol=tol, gtol=tol, x_scale=1.0).x
        q, a = model(x)
        r += x[4]
        if np.abs(x).max() < 1e-13:
            break
    return q, a, r, cylinder_rms_d(p, np.concatenate([q, a, [r]]))
