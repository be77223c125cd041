"""Sequential multi-primitive extraction (gm_extract_primitives) and its compression against the oracle restatement
(oracle/primitives.py): the whole cascade is an integer function of bit-exact quantities whenever the normals are."""
import ctypes as C
import os

import numpy as np
import pytest

from geometric_mapping_b200 import capi, synth
from oracle import chain
from oracle import primitives as P

pytestmark = pytest.mark.gpu

K, HP, HC = 8, 512, 512
MIN_INLIERS = 300
PRM = dict(boxFilterBound=5.0, neighborRadius=0.1, voxelGridLeafSize=0.1, ransacThreshold=0.05, cylinderRadiusMin=0.3,
           cylinderRadiusMax=10.0, refitIterations=5)


def _scene():
    """~100k points: a rectangular drift (four planes) with a pipe (a cylinder) running along it."""
    d = synth.rectangular_drift(90_000, seed=6)
    c = synth.straight_cylinder(12_000, seed=8, radius=0.5, half_length=3.5, noise=0.005)
    c[:, 1] += 0.9
    c[:, 2] += 0.2
    return np.concatenate([d, c])


def _ctx(n, **kw):
    return capi.Context(capi.default_params(**{**PRM, **kw}), max_points=max(n, 1), max_hypotheses=max(HP, HC))


def _draws(k=K, hp=HP, hc=HC):
    return synth.sample_draws(k, hp, 3, seed=1), synth.sample_draws(k, hc, 2, seed=2)


def _oracle(front, pd, cd, k=K, min_inliers=MIN_INLIERS):
    return P.extract(front["cloud"], front["normals_c"], pd, cd, k, min_inliers, tau=PRM["ransacThreshold"],
                     rmin=PRM["cylinderRadiusMin"], rmax=PRM["cylinderRadiusMax"], refit_iters=PRM["refitIterations"])


def _angle(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.arccos(np.clip(abs(a @ b) / np.linalg.norm(a) / np.linalg.norm(b), -1.0, 1.0)))


def _assert_same(g, gi, o, oi):
    assert len(g) == len(o) >= 4
    for a, b in zip(g, o):
        for f in ("kind", "best_id", "best_count", "n_remaining", "refit_count"):
            assert a[f] == b[f], (f, a[f], b[f])
        assert np.array_equal(a["hyp"].view(np.uint32), b["hyp"].view(np.uint32))
        gc, oc = a["coef"].astype(np.float64), b["coef"].astype(np.float64)
        if a["kind"] == 0:
            assert _angle(gc[:3], oc[:3]) < 1e-4 and abs(gc[3] - oc[3]) < 1e-4
        else:
            assert _angle(gc[3:6], oc[3:6]) < 1e-4 and abs(gc[6] - oc[6]) / oc[6] < 1e-4
            d, ax = gc[:3] - oc[:3], oc[3:6] / np.linalg.norm(oc[3:6])
            assert np.linalg.norm(d - ax * (d @ ax)) / oc[6] < 1e-4
    assert np.array_equal(gi, oi)


@pytest.fixture(scope="module")
def scene():
    return _scene()


@pytest.fixture(scope="module")
def front(scene):
    return chain.front(scene, bound=PRM["boxFilterBound"], radius=PRM["neighborRadius"], leaf=PRM["voxelGridLeafSize"], with_nn=False)


@pytest.fixture(scope="module")
def expected(front):
    pd, cd = _draws()
    return _oracle(front, pd, cd)


def _injected(front, pd, cd, k=K, min_inliers=MIN_INLIERS):
    n = len(front["cloud"])
    with _ctx(n) as ctx:
        ctx.inject_compacted(front["cloud"], front["normals_c"])
        ctx.extract_primitives(pd, cd, k, min_inliers)
        assert ctx.counts().device_error == 0
        return ctx.primitives(), ctx.download_primitive_ids()


def test_injected_cloud_is_bit_exact(front, expected):
    g, gi = _injected(front, *_draws())
    _assert_same(g, gi, *expected)
    assert {p["kind"] for p in g} == {0, 1}


@pytest.mark.parametrize("count_mode", [0, 1])
def test_raw_points_match_the_oracle_chain(scene, front, expected, count_mode):
    """Canonical normals: tile-culled counting over the blanked cell-sorted copy (count_mode 0) and brute force (1)."""
    pd, cd = _draws()
    with _ctx(len(scene)) as ctx:
        ctx.set_normals_mode(1)
        ctx.set_count_mode(count_mode)
        ctx.upload_scan(scene)
        ctx.crop()
        ctx.normals()
        assert np.array_equal(ctx.download_cloud(1).view(np.uint32), front["cloud"].view(np.uint32))
        ctx.extract_primitives(pd, cd, K, MIN_INLIERS)
        assert ctx.counts().device_error == 0
        _assert_same(ctx.primitives(), ctx.download_primitive_ids(), *expected)


def test_stop_rules_and_edges(front, expected):
    pd, cd = _draws()
    n = len(front["cloud"])
    g, ids = _injected(front, pd, cd, min_inliers=n + 1)
    assert g == [] and len(ids) == n and not ids.any()
    g, ids = _injected(front, pd[:2], cd[:2], k=2)
    assert [(p["kind"], p["best_id"], p["best_count"]) for p in g] == [(p["kind"], p["best_id"], p["best_count"]) for p in expected[0][:2]]
    assert np.array_equal(ids, np.where(expected[1] <= 2, expected[1], 0))
    g, _ = _injected(front, None, cd)
    assert g and all(p["kind"] == 1 for p in g)
    g, _ = _injected(front, pd, None)
    assert g and all(p["kind"] == 0 for p in g)
    same = np.zeros_like(pd), np.zeros_like(cd)  # every sample repeats one index: all hypotheses are degenerate
    g, ids = _injected(front, *same)
    assert g == [] and not ids.any()
    with _ctx(16) as ctx:
        ctx.inject_compacted(np.zeros((0, 4), np.float32))
        ctx.extract_primitives(pd, cd, K, 1)
        assert ctx.primitives() == [] and len(ctx.download_primitive_ids()) == 0
    lib = capi._lib()
    with _ctx(16) as ctx:
        p = pd.ctypes.data_as(C.c_void_p)
        c = cd.ctypes.data_as(C.c_void_p)
        assert lib.gm_extract_primitives(ctx._h, 1, 1, p, HP, c, HC) == capi.GM_ERR_STAGE_ORDER
        ctx.inject_compacted(front["cloud"][:16], front["normals_c"][:16])
        assert lib.gm_extract_primitives(ctx._h, 65, 1, p, HP, c, HC) == capi.GM_ERR_INVALID_ARG
        assert lib.gm_extract_primitives(ctx._h, -1, 1, p, HP, c, HC) == capi.GM_ERR_INVALID_ARG
        assert lib.gm_extract_primitives(ctx._h, 1, 1, None, HP, c, HC) == capi.GM_ERR_INVALID_ARG
        assert lib.gm_extract_primitives(ctx._h, 1, 1, p, HP, None, HC) == capi.GM_ERR_INVALID_ARG
        assert lib.gm_extract_primitives(ctx._h, 1, 1, p, -1, c, HC) == capi.GM_ERR_INVALID_ARG
        assert lib.gm_extract_primitives(ctx._h, 1, 1, p, HP + 1, c, HC) == capi.GM_ERR_CAPACITY
        n = C.c_int32(0)
        assert lib.gm_get_primitives(ctx._h, None, 0, C.byref(n)) == capi.GM_ERR_STAGE_ORDER


def test_invariants_at_1m_points():
    pts = synth.curved_tunnel(1_000_000)
    pd, cd = _draws()
    with capi.Context(capi.default_params(), max_points=len(pts), max_hypotheses=512) as ctx:
        ctx.upload_scan(pts)
        ctx.crop()
        ctx.normals()
        nv = ctx.counts().n_valid
        launches, found = [], []
        for run in range(2):
            # run 0 never stops; run 1 stops after round 1: its round 2 is run 0's round 2, one inlier short
            min_inliers = 1 if run == 0 else found[0][1]["best_count"] + 1
            ctx.reset_launch_count()
            ctx.extract_primitives(pd, cd, K, min_inliers)
            launches.append(ctx.launch_count)
            g, ids = ctx.primitives(), ctx.download_primitive_ids()
            found.append(g)
            assert ctx.counts().device_error == 0
            assert sum(p["best_count"] for p in g) + int((ids == 0).sum()) == nv
            assert np.array_equal(np.bincount(ids, minlength=len(g) + 1)[1:], [p["best_count"] for p in g])
        assert len(found[0]) == K and found[0][0]["best_count"] > found[0][1]["best_count"]
        assert len(found[1]) == 1
        assert launches[0] == launches[1]


def _snapshot(ctx):
    s = {}
    for k in (capi.GM_MODEL_PLANE, capi.GM_MODEL_CYLINDER):
        m = ctx.model(k)
        s[f"model{k}"] = (m["best_id"], m["best_count"], m["refit_count"], m["hyp"].tobytes(), m["coef"].tobytes(), m["rms"])
        s[f"hyp{k}"] = tuple(None if a is None else a.tobytes() for a in ctx.download_hypotheses(k, 256))
    s["labels"] = ctx.download_labels().tobytes()
    s["polyline"] = ctx.download_polyline().tobytes()
    s["gmc1"] = ctx.download_compressed()
    return s


def test_existing_outputs_do_not_change_and_compression_ratio(scene):
    ps, cs = synth.sample_indices(len(scene) // 2, 256, 3), synth.sample_indices(len(scene) // 2, 256, 2)
    pd, cd = _draws()
    with _ctx(len(scene)) as ctx:
        ctx.upload_scan(scene)
        ctx.process_scan(ps, cs)
        ctx.compress()
        before = _snapshot(ctx)
        ctx.extract_primitives(pd, cd, K, MIN_INLIERS)
        ctx.compress_primitives()
        assert _snapshot(ctx) == before
        gmc = ctx.compression()
        h = capi.parse_compressed_primitives(ctx.download_compressed_primitives())["header"]
        assert h.n_primitives >= 4
        assert h.ratio > gmc.ratio and h.n_residual_voxels < gmc.n_residual_voxels


def test_stage_rules(scene):
    pd, cd = _draws(k=2)
    n = 20_000
    with _ctx(n) as ctx:
        ctx.upload_scan(scene[:n])
        ctx.crop()
        ctx.normals()
        with pytest.raises(capi.GmError) as e:
            ctx.compress_primitives()
        assert e.value.status == capi.GM_ERR_STAGE_ORDER
        ctx.extract_primitives(pd, cd, 2, 10)
        ctx.set_params(capi.default_params(**PRM))  # identical parameters keep the primitives
        ctx.primitives()
        ctx.compress_primitives()
        ctx.download_compressed_primitives()
        ctx.extract_primitives(pd, cd, 2, 10)  # a new extraction drops the old compression
        with pytest.raises(capi.GmError) as e:
            ctx.download_compressed_primitives()
        assert e.value.status == capi.GM_ERR_STAGE_ORDER
        ctx.set_params(capi.default_params(**{**PRM, "neighborRadius": 0.12}))  # a new neighbour grid
        with pytest.raises(capi.GmError) as e:
            ctx.primitives()
        assert e.value.status == capi.GM_ERR_STAGE_ORDER
        ctx.crop()
        ctx.normals()
        ctx.extract_primitives(pd, cd, 2, 10)
        ctx.upload_scan(scene[:n])  # a new scan
        for fn in (ctx.primitives, ctx.download_primitive_ids, ctx.compress_primitives):
            with pytest.raises(capi.GmError) as e:
                fn()
            assert e.value.status == capi.GM_ERR_STAGE_ORDER


def test_compression_matches_the_oracle_and_round_trips(front, expected, tmp_path):
    pd, cd = _draws()
    n = len(front["cloud"])
    with _ctx(n) as ctx:
        ctx.inject_compacted(front["cloud"], front["normals_c"])
        ctx.extract_primitives(pd, cd, K, MIN_INLIERS)
        ctx.compress_primitives()
        blob = ctx.download_compressed_primitives()
    b = capi.parse_compressed_primitives(blob)
    h, rec = b["header"], b["records"]
    o = P.compress(front["cloud"], expected[1], expected[0], PRM["voxelGridLeafSize"])
    assert (h.n_points, h.n_primitives, h.n_residual, h.n_residual_voxels) == (n, len(o["records"]), o["n_residual"], o["n_residual_voxels"])
    assert h.bytes_out == len(blob) and h.bytes_in == 16 * n and abs(h.ratio - h.bytes_in / h.bytes_out) < 1e-3 * h.ratio
    for g, r in zip(rec, o["records"]):
        assert g["kind"] == r["kind"] and g["count"] == r["count"]
        k = 4 if r["kind"] == 0 else 2
        assert np.abs(g["extents"][:k] - r["extents"][:k]).max() < 1e-4
        assert abs(g["rms"] - r["rms"]) < 1e-4
    assert np.array_equal(b["residual"].view(np.uint32), o["residual_centroids"][:, :3].view(np.uint32))
    assert abs(h.residual_rms - o["residual_rms"]) < 1e-4 and abs(h.total_rms - o["total_rms"]) < 1e-4
    path = os.path.join(str(tmp_path), "prims.gms")
    with capi.PrimitiveStore(path) as st:
        st.append_blob(blob, scan_id=7)
    with capi.PrimitiveStore(path, create=False) as st:
        assert len(st) == 1 and st.read(0) == blob


def test_primitive_struct_matches_header():
    assert C.sizeof(capi.gm_primitive) == C.sizeof(capi.gm_model) + 8 == 96
    assert C.sizeof(capi.gm_primitive_compression) == 48 and capi.PRIMITIVE_RECORD_DTYPE.itemsize == 56
