"""Seeded synthetic tunnel scans and RANSAC sample indices (SURVEY.md section 8(d)).

All generators draw in float64 from numpy's Philox bit generator and return float32 n x 4 arrays
laid out as pcl::PointXYZ (x, y, z, pad=1.0).  Sensor at the origin, frame "/velodyne".
"""
from __future__ import annotations

import numpy as np


def _rng(seed: int) -> np.random.Generator:
    return np.random.Generator(np.random.Philox(seed))


def _xyzw(x, y, z) -> np.ndarray:
    out = np.empty((x.shape[0], 4), np.float32)
    out[:, 0], out[:, 1], out[:, 2], out[:, 3] = x, y, z, 1.0
    return out


def straight_cylinder(n: int = 100_000, seed: int = 1, radius: float = 2.5, half_length: float = 5.0,
                      noise: float = 0.01) -> np.ndarray:
    """C0: straight cylinder, axis = x, x~U[-L,L], theta~U[0,2pi), radial noise N(0, noise)."""
    g = _rng(seed)
    x = g.uniform(-half_length, half_length, n)
    th = g.uniform(0.0, 2.0 * np.pi, n)
    r = radius + g.normal(0.0, noise, n) if noise > 0 else np.full(n, radius)
    return _xyzw(x, r * np.cos(th), r * np.sin(th))


def curved_tunnel(n: int = 1_000_000, seed: int = 2, radius: float = 2.5, arc_radius: float = 50.0,
                  arc_length: float = 10.0, floor_z: float = -1.5, noise: float = 0.02,
                  outlier_frac: float = 0.01, bound: float = 5.0, advance: float = 0.0) -> np.ndarray:
    """C1/C2: curved tunnel.  Centreline = arc of radius `arc_radius` in the xy-plane through the
    origin (tangent +x there), arc length `arc_length` centred on the origin (shifted by
    `advance` metres along the arc for frame sequences).  Circular section of radius `radius`;
    section points below z=floor_z are replaced by samples of the flat floor; radial Gaussian
    noise; `outlier_frac` of the points are uniform in the +-bound box."""
    g = _rng(seed)
    s = g.uniform(-0.5 * arc_length, 0.5 * arc_length, n) + advance
    th = g.uniform(0.0, 2.0 * np.pi, n)
    r = radius + g.normal(0.0, noise, n)
    phi = s / arc_radius
    # centreline point and in-plane normal of the arc
    cx, cy = arc_radius * np.sin(phi), arc_radius * (1.0 - np.cos(phi))
    nx, ny = -np.sin(phi), np.cos(phi)
    lat = r * np.cos(th)  # lateral offset in the section
    x, y, z = cx + lat * nx, cy + lat * ny, r * np.sin(th)
    below = z < floor_z
    # floor: keep the lateral chord position, put the point on the floor plane with vertical noise
    z = np.where(below, floor_z + g.normal(0.0, noise, n), z)
    k = int(round(outlier_frac * n))
    if k > 0:
        idx = g.choice(n, size=k, replace=False)
        x[idx], y[idx], z[idx] = (g.uniform(-bound, bound, k) for _ in range(3))
    return _xyzw(x, y, z)


def tunnel_map(n: int = 10_000_000, seed: int = 4, length: float = 100.0, arc_radius: float = 200.0, bound: float = 60.0,
               **kw) -> np.ndarray:
    """C4: dense aggregated map of `length` metres of gently curved tunnel (same section, floor and noise as
    curved_tunnel), centred on the origin; needs boxFilterBound >= bound."""
    return curved_tunnel(n, seed=seed, arc_radius=arc_radius, arc_length=length, bound=bound, **kw)


def plane_patch(n: int = 10_000, seed: int = 5, normal=(0.0, 0.0, 1.0), offset: float = -1.5, half: float = 2.0,
                noise: float = 0.0) -> np.ndarray:
    g = _rng(seed)
    nrm = np.asarray(normal, np.float64)
    nrm /= np.linalg.norm(nrm)
    a = np.cross(nrm, [1.0, 0.0, 0.0])
    if np.linalg.norm(a) < 1e-6:
        a = np.cross(nrm, [0.0, 1.0, 0.0])
    a /= np.linalg.norm(a)
    b = np.cross(nrm, a)
    u, v = g.uniform(-half, half, n), g.uniform(-half, half, n)
    d = offset + (g.normal(0.0, noise, n) if noise > 0 else 0.0)
    p = u[:, None] * a + v[:, None] * b + d[:, None] * nrm if np.ndim(d) else u[:, None] * a + v[:, None] * b + d * nrm
    return _xyzw(p[:, 0], p[:, 1], p[:, 2])


def dyadic(pts: np.ndarray, e: int) -> np.ndarray:
    """A copy of `pts` with x, y, z rounded to the nearest multiple of q = 2^-e (ties to even) and -0.0 turned into
    +0.0.  NaN and inf stay as they are, and so does every coordinate that already is a multiple of q (the crop
    faces +-bound for dyadic bounds).  On such a cloud every float product and partial sum of coordinates is a
    multiple of q^2 (or q), hence exact while it stays below 2^24 of those units: sums of them do not depend on
    the order of the additions."""
    out = np.array(pts, np.float32, copy=True)
    xyz = out[:, :3].astype(np.float64)
    fin = np.isfinite(xyz)
    s = 2.0 ** e
    xyz[fin] = np.round(xyz[fin] * s) / s + 0.0   # exact in float64; the result is a float32 (|x| < 2^(24-e) or already dyadic)
    out[:, :3] = xyz.astype(np.float32)
    return out


def sample_indices(n_points: int, H: int, per: int, seed: int = 3) -> np.ndarray:
    """H x per int32 sample indices, Philox(seed); injected identically into oracle and GPU."""
    g = _rng(seed)
    return g.integers(0, max(n_points, 1), size=(H, per), dtype=np.int64).astype(np.int32)


def rectangular_drift(n: int = 100_000, seed: int = 6, width: float = 4.0, height: float = 3.0, length: float = 8.0,
                      noise: float = 0.005, outlier_frac: float = 0.01) -> np.ndarray:
    """Multi-surface scene: a rectangular drift along x (floor z = -height/2, walls y = +-width/2, roof z = +height/2),
    each surface sampled in proportion to its area, Gaussian noise along its normal, `outlier_frac` of the points uniform
    inside the section.  One plane per surface: the scene needs four primitives."""
    g = _rng(seed)
    x = g.uniform(-0.5 * length, 0.5 * length, n)
    side = g.choice(4, size=n, p=np.array([width, height, width, height]) / (2.0 * (width + height)))
    a = g.uniform(-0.5, 0.5, n)
    e = g.normal(0.0, noise, n) if noise > 0 else np.zeros(n)
    hw, hh = 0.5 * width, 0.5 * height
    y = np.select([side == 0, side == 1, side == 2], [a * width, hw + e, a * width], -hw + e)
    z = np.select([side == 0, side == 1, side == 2], [-hh + e, a * height, hh + e], a * height)
    k = int(round(outlier_frac * n))
    if k > 0:
        idx = g.choice(n, size=k, replace=False)
        y[idx], z[idx] = g.uniform(-0.8 * hw, 0.8 * hw, k), g.uniform(-0.8 * hh, 0.8 * hh, k)
    return _xyzw(x, y, z)


def drift_end_niche(n: int = 1_000_000, seed: int = 8, width: float = 4.0, height: float = 3.0, length: float = 8.0,
                    niche=(0.5, 1.5, -0.5, 0.5, 0.6), noise: float = 0.005) -> np.ndarray:
    """A scene whose scans constrain all six rigid degrees of freedom, for registration: the rectangular drift of
    `rectangular_drift` (x in [-length/2, length/2]) closed by an end face x = +length/2, with a rectangular niche
    (x0, x1, z0, z1, depth) cut into the wall y = +width/2.  Surfaces are sampled in proportion to their area, Gaussian
    noise along their normals.  Floor, roof and walls fix y, z, roll, pitch and yaw; the end face fixes x."""
    g = _rng(seed)
    L, hw, hh = float(length), 0.5 * width, 0.5 * height
    x0, x1, z0, z1, dep = (float(v) for v in niche)
    xe = 0.5 * L
    # surfaces: floor, roof, wall -y, wall +y (its opening is the niche's back wall, same footprint), end face, the
    # niche's two x-sides and its two z-sides
    areas = np.array([L * width, L * width, L * height, L * height, width * height, 2 * dep * (z1 - z0), 2 * dep * (x1 - x0)])
    side = g.choice(len(areas), size=n, p=areas / areas.sum())
    a, b, c = g.uniform(0.0, 1.0, n), g.uniform(0.0, 1.0, n), g.uniform(0.0, 1.0, n)
    e = g.normal(0.0, noise, n) if noise > 0 else np.zeros(n)
    # every surface takes its two in-surface coordinates from two different uniforms (a and b, or b and c)
    x, y, z = -0.5 * L + a * L, -hw + b * width, -hh + b * height
    wall_y = np.where((x >= x0) & (x < x1) & (z >= z0) & (z < z1), hw + dep, hw)
    ny = hw + a * dep
    cand = [np.stack([x, y, -hh + e], 1), np.stack([x, y, hh + e], 1), np.stack([x, -hw + e, z], 1),
            np.stack([x, wall_y + e, z], 1), np.stack([xe + e, -hw + a * width, z], 1),
            np.stack([np.where(c < 0.5, x0, x1) + e, ny, z0 + b * (z1 - z0)], 1),
            np.stack([x0 + b * (x1 - x0), ny, np.where(c < 0.5, z0, z1) + e], 1)]
    out = np.empty((n, 3))
    for k, v in enumerate(cand):
        out[side == k] = v[side == k]
    return _xyzw(out[:, 0], out[:, 1], out[:, 2])


def pose34(rotvec=(0.0, 0.0, 0.0), t=(0.0, 0.0, 0.0)) -> np.ndarray:
    """3x4 float64 [R|t] with R = exp([rotvec]x) (Rodrigues)."""
    w = np.asarray(rotvec, np.float64)
    th = float(np.linalg.norm(w))
    K = np.array([[0.0, -w[2], w[1]], [w[2], 0.0, -w[0]], [-w[1], w[0], 0.0]])
    R = np.eye(3) if th == 0.0 else np.eye(3) + np.sin(th) / th * K + (1.0 - np.cos(th)) / th ** 2 * (K @ K)
    return np.concatenate([R, np.asarray(t, np.float64).reshape(3, 1)], axis=1)


def view_from(points: np.ndarray, sensor_pose34) -> np.ndarray:
    """The scene points `points` (world frame) as a sensor placed at `sensor_pose34` (sensor -> world, 3x4) sees them:
    p_sensor = R^T (p - t).  Registering such a scan (source) against one taken at the origin (target) recovers
    sensor_pose34."""
    T = np.asarray(sensor_pose34, np.float64)
    p = np.asarray(points, np.float64)[:, :3]
    q = (p - T[:, 3]) @ T[:, :3]
    return _xyzw(q[:, 0], q[:, 1], q[:, 2])


def second_scan(generator, sensor_pose34, seed: int, n: int, **kw) -> np.ndarray:
    """Another scan of the scene of `generator` (new sample draw: `seed`) seen from the sensor pose `sensor_pose34`."""
    return view_from(generator(n, seed=seed, **kw), sensor_pose34)


def sample_draws(K: int, H: int, per: int, seed: int = 7) -> np.ndarray:
    """K x H x per uint32 draws for gm_extract_primitives, Philox(seed): round r maps draw u to the sample index
    R_r[(u * n_r) >> 32] of the points still unclaimed."""
    return _rng(seed).integers(0, 1 << 32, size=(K, H, per), dtype=np.uint64).astype(np.uint32)
