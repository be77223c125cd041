"""Axis polyline (gm_axis_polyline) against a float64 numpy restatement built from the context's own inputs: the
compacted cloud, normals, labels, local frame and sliceLength.  The slice of a point and the slice counts are integer
decisions taken from the same double expressions as the kernels, so `count` must match exactly; the means, circle,
radius, RMS and direction are compared within float32-output tolerances.  Also: a run repeated on one scan and a
replayed CUDA graph give the same bytes as plain launches.
"""
import numpy as np
import pytest

from geometric_mapping_b200 import capi, synth

pytestmark = pytest.mark.gpu

WF = 0.2


def _ctx(n, **kw):
    return capi.Context(capi.default_params(**kw), max_points=n, max_hypotheses=512)


def _scan(ctx, pts, plane=True, cyl=True, H=256):
    ctx.upload_scan(pts)
    ctx.crop()
    ctx.normals()
    nv = ctx.counts().n_valid
    ps = synth.sample_indices(nv, H, 3, seed=3) if plane else None
    cs = synth.sample_indices(nv, H, 2, seed=4) if cyl else None
    ctx.upload_scan(pts)
    ctx.process_scan(ps, cs)
    assert ctx.counts().device_error == 0


def _reference(cloud, normals, labels, axis_f32, L, max_slices):
    """-> (S, count[S], {center, dir, radius, rms, t_mid} for every slice with at least 3 points)."""
    a = axis_f32.astype(np.float64)
    sel = labels == 2
    p = cloud[sel, :3].astype(np.float64)
    if len(p) == 0:
        return 0, np.zeros(0, np.int64), {}
    t = a[0] * p[:, 0] + a[1] * p[:, 1] + a[2] * p[:, 2]
    t0 = np.floor(t.min() / L) * L
    S = min(int(np.floor((t.max() - t0) / L)) + 1, max_slices)
    s = np.floor((t - t0) / L).astype(np.int64)
    keep = (s >= 0) & (s < S)
    count = np.bincount(s[keep], minlength=S)[:S]
    ah = a / np.linalg.norm(a)
    u = np.cross(ah, [1.0, 0.0, 0.0] if abs(ah[0]) < 0.9 else [0.0, 1.0, 0.0])
    u /= np.linalg.norm(u)
    w = np.cross(ah, u)
    curv = normals[sel, 4].astype(np.float64)
    wt = np.exp((curv + 0.001 / WF) ** 2).astype(np.float32).astype(np.float64)
    wn = wt[:, None] * normals[sel, :3].astype(np.float64)
    order = np.argsort(s, kind="stable")
    out = {}
    for k in range(S):
        idx = order[np.searchsorted(s[order], k, "left"):np.searchsorted(s[order], k, "right")]
        if len(idx) < 3:
            continue
        A, B = p[idx] @ u, p[idx] @ w
        ma, mb = A.mean(), B.mean()
        ac, bc = A - ma, B - mb
        z = ac * ac + bc * bc
        M = np.array([[ac @ ac, ac @ bc], [ac @ bc, bc @ bc]])
        ca, cb = 0.5 * np.linalg.solve(M, [ac @ z, bc @ z])
        rad = np.sqrt(z.mean() + ca * ca + cb * cb)
        e = np.sqrt((ac - ca) ** 2 + (bc - cb) ** 2) - rad
        tm = t0 + (k + 0.5) * L
        vals, vecs = np.linalg.eigh(wn[idx].T @ wn[idx])
        d = vecs[:, 0] * (1.0 if vecs[:, 0] @ a >= 0 else -1.0)
        out[k] = {"center": (ma + ca) * u + (mb + cb) * w + tm * a, "dir": d, "radius": rad,
                  "rms": np.sqrt((e * e).mean()), "t_mid": tm}
    return S, count, out


def _check(ctx, min_points=100):
    cloud, normals, labels = ctx.download_cloud(1), ctx.download_normals(1), ctx.download_labels()
    prm = ctx.params
    S, count, ref = _reference(cloud, normals, labels, ctx.frame()["vecs"][:, 0], prm.sliceLength, prm.maxSlices)
    poly = ctx.download_polyline()
    assert len(poly) == S
    assert np.array_equal(poly["count"].astype(np.int64), count)
    checked = 0
    for k, r in ref.items():
        if count[k] < min_points:
            continue
        g = poly[k]
        assert np.abs(g["center"] - r["center"]).max() <= 2e-5, (k, g["center"], r["center"])
        assert abs(g["radius"] - r["radius"]) <= 1e-5 * r["radius"], (k, g["radius"], r["radius"])
        assert abs(g["rms"] - r["rms"]) <= 1e-4 * r["rms"] + 1e-7, (k, g["rms"], r["rms"])
        assert abs(g["t_mid"] - r["t_mid"]) <= 1e-6 * max(abs(r["t_mid"]), 1.0)
        d = g["dir"].astype(np.float64)
        angle = np.arctan2(np.linalg.norm(np.cross(d, r["dir"])), d @ r["dir"])
        assert angle <= 1e-5, (k, g["dir"], r["dir"])
        checked += 1
    return poly, labels, checked


def test_c1_scan_1m_points():
    n = 1_000_000
    with _ctx(n, neighborRadius=0.05, voxelGridLeafSize=0.1) as ctx:
        _scan(ctx, synth.curved_tunnel(n, seed=2))
        poly, labels, checked = _check(ctx)
    assert len(poly) >= 8 and checked >= 8 and (labels == 2).sum() > 50_000


def test_more_slices_than_shared_memory_holds():
    # 0.02 m slices over a 10 m tunnel: ~500 slices, above what both passes keep in shared memory (153 and 256), so
    # every sum goes through the global-memory atomics
    n = 200_000
    with _ctx(n, neighborRadius=0.12, maxSlices=1024, sliceLength=0.02) as ctx:
        _scan(ctx, synth.curved_tunnel(n, seed=5))
        poly, _, checked = _check(ctx, min_points=50)
    assert len(poly) > 256 and checked > 256


def test_no_cylinder_points_gives_no_slices():
    n = 100_000
    with _ctx(n, neighborRadius=0.12) as ctx:
        _scan(ctx, synth.curved_tunnel(n, seed=6), cyl=False)
        poly, labels, _ = _check(ctx)
        assert (labels == 2).sum() == 0 and len(poly) == 0
        ctx.axis_polyline()
        assert len(ctx.download_polyline()) == 0


def test_every_valid_point_on_the_cylinder():
    n = 100_000
    with _ctx(n, neighborRadius=0.15) as ctx:
        _scan(ctx, synth.straight_cylinder(n, seed=7, noise=0.005), plane=False)
        poly, labels, checked = _check(ctx)
    assert len(labels) > 0.99 * n and (labels == 2).all()
    assert int(poly["count"].sum()) == len(labels) and checked >= 9


def test_repeated_runs_and_graph_replay_are_bit_identical():
    n = 200_000
    pts = synth.curved_tunnel(n, seed=8)
    outs = []
    for mode in (0, 1):  # plain launches, then an always-captured graph
        with _ctx(n, neighborRadius=0.12) as ctx:
            ctx.set_graph_mode(mode)
            for _ in range(2):  # graph mode: the second scan replays the captured graph
                _scan(ctx, pts)
                outs.append(ctx.download_polyline().tobytes())
            ctx.axis_polyline()  # once more on the same scan, as a stage call
            outs.append(ctx.download_polyline().tobytes())
            if mode == 1:
                assert ctx.graph_stats()[1] >= 1
    assert len(outs[0]) > 0 and all(o == outs[0] for o in outs)
