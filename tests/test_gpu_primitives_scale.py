"""Multi-primitive extraction at full scale: a 1M-point cascade run until the stop rule ends it, a cascade that fills all
64 primitive slots, a cloud whose every point is claimed, the refits against float64 least-squares references that
share no code with the oracle, the compression at the bounds of its fixed-point sums, and the reuse of the extraction's
scratch buffers and streams.

Every tolerance below carries the largest deviation observed on one B200 next to it."""
import numpy as np
import pytest

from geometric_mapping_b200 import capi, synth
from oracle import oracle as O
from oracle import primitives as P

pytestmark = pytest.mark.gpu

K = 64  # GM_MAX_PRIMITIVES
H = 256
TAU, RMIN, RMAX, ITERS = 0.05, 0.5, 10.0, 5  # gm_params_default

# GPU against the oracle restatement (same algorithm, sums in another order).  The coefficients came out bit-identical
# in every case; the tolerances allow about one float32 rounding
TOL_ORACLE_PLANE_ANGLE = 2.0 ** -22  # rad; observed 0
TOL_ORACLE_PLANE_D = 2.0 ** -21  # m, one float32 ulp at 4-8 m; observed 0
TOL_ORACLE_CYL = 2.0 ** -20  # axis angle (rad), relative radius, axis-line distance / radius; observed 0
TOL_ORACLE_CYL_RMS = 2e-7  # relative; observed 4.8e-8
# GPU refits against the float64 references of oracle/primitives.py
TOL_PLANE_ANGLE = 1e-7  # rad; observed 3.2e-8
TOL_PLANE_D = 5e-7  # m; observed 2.3e-7
TOL_PLANE_RMS = 1.5e-7  # relative; observed 4.8e-8
# the Gauss-Newton refit stops once its step is below 1e-4: the cylinder's coefficients stay a few 1e-6 from the
# least-squares optimum, while its RMS is within 1e-8 of the optimum's
TOL_CYL_ANGLE = 1e-5  # rad; observed 4.2e-6
TOL_CYL_RADIUS = 5e-6  # relative; observed 1.5e-6
TOL_CYL_AXIS = 5e-6  # axis-line distance between the q's / radius; observed 1.9e-6
TOL_CYL_RMS_MODEL = 1.5e-7  # relative, the Gauss-Newton model's RMS against the RMS measured at the GPU's float coefficients; observed 4.8e-8
TOL_CYL_RMS_OPT = 2e-8  # relative, RMS at the GPU's coefficients above the float64 optimum; observed 5.0e-9
# compression against P.compress at the GPU's coefficients
TOL_EXTENT = 2.0 ** -20  # m, one float32 ulp at 8-16 m (projections reach 5 * sqrt(3) m); observed 4.0e-7
TOL_RESIDUAL_RMS = 1.0  # float32 ulps; observed 0.37
# per-primitive and total RMS: within _rms_tol, the bound of the fixed-point sums; observed 0.30 and 0.11 of it


def _angle(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.arctan2(np.linalg.norm(np.cross(a, b)), abs(a @ b)))


def _run(pts, prm, pd, cd, k, min_inliers, count_mode=0, knn=0, compress=True):
    """crop + normals (default fast mode, or k-NN) + extraction (+ compression) on one context -> the compacted cloud and
    normals it extracted from, the primitives, the ids and the GMP1 blob."""
    with capi.Context(capi.default_params(**prm), max_points=len(pts), max_hypotheses=H) as ctx:
        ctx.set_count_mode(count_mode)
        if knn:
            ctx.set_knn(knn)
        ctx.upload_scan(pts)
        ctx.crop()
        ctx.normals()
        out = {"cloud": ctx.download_cloud(1), "normals": ctx.download_normals(1)}
        ctx.extract_primitives(pd, cd, k, min_inliers)
        out.update(prims=ctx.primitives(), ids=ctx.download_primitive_ids())
        if compress:
            ctx.compress_primitives()
            out["blob"] = ctx.download_compressed_primitives()
        assert ctx.counts().device_error == 0
    return out


def _oracle(run, pd, cd, k, min_inliers, rmin=RMIN):
    trace = []
    prims, ids = P.extract(run["cloud"], run["normals"], pd, cd, k, min_inliers, tau=TAU, rmin=rmin, rmax=RMAX, refit_iters=ITERS,
                           trace=trace)
    return prims, ids, trace


def _oracle_devs(g, o):
    """Coefficient and RMS deviations of one GPU primitive from the oracle's."""
    gc, oc = g["coef"].astype(np.float64), o["coef"].astype(np.float64)
    if g["kind"] == 0:
        return {"plane_angle": _angle(gc[:3], oc[:3]), "plane_d": abs(gc[3] - oc[3])}
    ax = oc[3:6] / np.linalg.norm(oc[3:6])
    dq = gc[:3] - oc[:3]
    return {"cyl_angle": _angle(gc[3:6], oc[3:6]), "cyl_radius": abs(gc[6] - oc[6]) / oc[6],
            "cyl_axis": np.linalg.norm(dq - ax * (dq @ ax)) / oc[6], "cyl_rms": abs(g["rms"] - o["rms"]) / o["rms"] if o["rms"] else abs(g["rms"])}


def _assert_parity(g, gi, expected, k, min_inliers):
    """Everything the oracle defines, bit for bit where the cascade is integer, and how the cascade ended."""
    o, oi, trace = expected
    assert len(g) == len(o)
    for a, b in zip(g, o):
        for f in ("kind", "best_id", "best_count", "n_remaining", "refit_count"):
            assert a[f] == b[f], (f, a[f], b[f])
        assert np.array_equal(a["hyp"].view(np.uint32), b["hyp"].view(np.uint32))
        d = _oracle_devs(a, b)
        if a["kind"] == 0:
            assert d["plane_angle"] < TOL_ORACLE_PLANE_ANGLE and d["plane_d"] < TOL_ORACLE_PLANE_D, d
        else:
            assert d["cyl_angle"] < TOL_ORACLE_CYL and d["cyl_radius"] < TOL_ORACLE_CYL and d["cyl_axis"] < TOL_ORACLE_CYL, d
            assert d["cyl_rms"] < TOL_ORACLE_CYL_RMS, d
    assert np.array_equal(gi, oi)
    assert [t[0] for t in trace[: len(g)]] == [p["n_remaining"] for p in g]
    if len(g) < k:  # the stop came from the stop rule: round len(g) found no hypothesis with enough inliers
        assert len(trace) == len(g) + 1 and max(trace[-1][1:]) < max(min_inliers, 1)
        assert trace[-1][0] == int((gi == 0).sum())
    np.testing.assert_array_equal(np.bincount(gi, minlength=len(g) + 1)[1:], [p["best_count"] for p in g])


def _reference_devs(cloud, m, inliers):
    """Deviations of one refined model (gm_primitive or gm_model dict) from the float64 reference on its refit set."""
    S = cloud[inliers]
    assert m["refit_count"] == m["best_count"] == len(S)
    c = m["coef"].astype(np.float64)
    if m["kind"] == 0:
        if len(S) <= 3:  # too few points to refit: the hypothesis is kept
            assert np.array_equal(m["coef"], m["hyp"]) and m["rms"] == 0.0
            return {}
        n, d, rms = P.plane_fit_d(S)
        s = 1.0 if n @ c[:3] >= 0 else -1.0
        return {"plane_angle": _angle(c[:3], n), "plane_d": abs(c[3] - s * d), "plane_rms": abs(m["rms"] - rms) / max(rms, 1e-30)}
    if len(S) <= 5:
        assert np.array_equal(m["coef"], m["hyp"]) and m["rms"] == 0.0
        return {}
    q, a, r, rms = P.cylinder_fit_d(S, m["hyp"])
    dq = c[:3] - q
    rms_at = P.cylinder_rms_d(S, c)
    return {"cyl_angle": _angle(c[3:6], a), "cyl_radius": abs(c[6] - r) / r, "cyl_axis": np.linalg.norm(dq - a * (dq @ a)) / r,
            "cyl_rms_model": abs(m["rms"] - rms_at) / rms_at, "cyl_rms_opt": (rms_at - rms) / rms}


def _assert_reference(d):
    if "plane_angle" in d:
        assert d["plane_angle"] < TOL_PLANE_ANGLE and d["plane_d"] < TOL_PLANE_D and d["plane_rms"] < TOL_PLANE_RMS, d
    elif d:
        assert d["cyl_angle"] < TOL_CYL_ANGLE and d["cyl_radius"] < TOL_CYL_RADIUS and d["cyl_axis"] < TOL_CYL_AXIS, d
        assert d["cyl_rms_model"] < TOL_CYL_RMS_MODEL, d
        assert -1e-12 < d["cyl_rms_opt"] < TOL_CYL_RMS_OPT, d  # the reference is the optimum: the GPU's RMS is not below it


def _extraction_reference_devs(run):
    return [_reference_devs(run["cloud"], p, run["ids"] == r + 1) for r, p in enumerate(run["prims"])]


def _rms_tol(o):
    """|rms_gpu - rms| allowed when rms_gpu^2 comes from sums of squares rounded to 2^-32 m^2 per point (n * 2^-33 on a
    sum of n terms, 2^-33 on the mean square), then rounded to float32."""
    return (min(2.0 ** -33 / o, 2.0 ** -16.5) if o > 0 else 2.0 ** -16.5) + float(np.spacing(np.float32(o)))


def _compression_devs(run, leaf):
    """The GMP1 blob against P.compress over the same ids and the GPU's own refined coefficients; integer fields and
    residual centroids are compared exactly (asserted here), float fields return their deviations."""
    b = capi.parse_compressed_primitives(run["blob"])
    h, rec = b["header"], b["records"]
    o = P.compress(run["cloud"], run["ids"], run["prims"], leaf)
    assert (h.n_points, h.n_primitives, h.n_residual, h.n_residual_voxels) == (len(run["cloud"]), len(o["records"]), o["n_residual"],
                                                                                o["n_residual_voxels"])
    assert np.array_equal(b["residual"].view(np.uint32), o["residual_centroids"][:, :3].view(np.uint32))
    ext, rms = 0.0, 0.0
    for g, r, p in zip(rec, o["records"], run["prims"]):
        assert g["kind"] == r["kind"] and g["count"] == r["count"] == p["best_count"]
        assert np.array_equal(g["coef"][: len(p["coef"])].view(np.uint32), p["coef"].view(np.uint32))
        ne = 4 if r["kind"] == 0 else 2
        ext = max(ext, float(np.abs(g["extents"][:ne].astype(np.float64) - r["extents"][:ne]).max()))
        assert not g["extents"][ne:].any()
        rms = max(rms, float(abs(g["rms"] - r["rms"])) / _rms_tol(r["rms"]))
    ulp = float(np.spacing(np.float32(max(o["residual_rms"], 1e-30))))
    return {"extent": ext, "rms_over_bound": rms, "residual_rms_ulps": float(abs(h.residual_rms - o["residual_rms"])) / ulp,
            "total_rms_over_bound": float(abs(h.total_rms - o["total_rms"])) / _rms_tol(o["total_rms"]), "header": h, "oracle": o}


def _assert_compression(d):
    assert d["extent"] <= TOL_EXTENT, d["extent"]
    assert d["rms_over_bound"] <= 1.0 and d["total_rms_over_bound"] <= 1.0, d
    assert d["residual_rms_ulps"] <= TOL_RESIDUAL_RMS, d


# ---- the 1M-point curved tunnel, K = 64, min_inliers = 1: the cascade runs until the points run out -----------------
@pytest.fixture(scope="module")
def tunnel():
    return synth.curved_tunnel(1_000_000)


@pytest.fixture(scope="module")
def tunnel_draws():
    return synth.sample_draws(K, H, 3, seed=11), synth.sample_draws(K, H, 2, seed=12)


@pytest.fixture(scope="module")
def tunnel_run(tunnel, tunnel_draws):
    return _run(tunnel, {}, *tunnel_draws, K, 1, count_mode=0)


@pytest.fixture(scope="module")
def tunnel_expected(tunnel_run, tunnel_draws):
    return _oracle(tunnel_run, *tunnel_draws, K, 1)


def test_1m_cascade_to_exhaustion_tile_culled(tunnel_run, tunnel_expected):
    """Count mode 0: the leaf bounds the claims rewrite cull every later round; a bound that came out too tight would
    undercount some hypothesis and change the cascade."""
    _assert_parity(tunnel_run["prims"], tunnel_run["ids"], tunnel_expected, K, 1)
    assert len(tunnel_run["prims"]) < K
    assert tunnel_run["prims"][-1]["best_count"] < 20  # the last rounds claim a handful of points each


def test_1m_cascade_to_exhaustion_brute_force(tunnel, tunnel_draws, tunnel_run, tunnel_expected):
    run = _run(tunnel, {}, *tunnel_draws, K, 1, count_mode=1, compress=False)
    assert np.array_equal(run["cloud"].view(np.uint32), tunnel_run["cloud"].view(np.uint32))
    assert np.array_equal(run["normals"].view(np.uint32), tunnel_run["normals"].view(np.uint32))
    _assert_parity(run["prims"], run["ids"], tunnel_expected, K, 1)


def test_1m_cascade_with_knn_normals(tunnel, tunnel_draws):
    run = _run(tunnel, {}, *tunnel_draws, K, 1, count_mode=0, knn=32, compress=False)
    expected = _oracle(run, *tunnel_draws, K, 1)
    _assert_parity(run["prims"], run["ids"], expected, K, 1)
    for d in _extraction_reference_devs(run):
        _assert_reference(d)


def test_1m_refits_match_float64_references(tunnel_run):
    devs = _extraction_reference_devs(tunnel_run)
    assert {p["kind"] for p in tunnel_run["prims"]} == {0, 1}
    for d in devs:
        _assert_reference(d)


def test_1m_compression_at_fixed_point_bounds(tunnel_run):
    d = _compression_devs(tunnel_run, 0.1)
    _assert_compression(d)
    assert d["header"].n_primitives == len(tunnel_run["prims"]) and d["header"].n_residual < 20


def test_1m_single_model_refits_match_float64_references(tunnel):
    """gm_ransac_select's refits (process_scan) on the whole compacted cloud: the refit set is the inlier set of the
    winning hypothesis, the same kernels as the extraction's refits."""
    with capi.Context(capi.default_params(), max_points=len(tunnel), max_hypotheses=H) as ctx:
        ctx.upload_scan(tunnel)
        ctx.crop()
        ctx.normals()
        nv = ctx.counts().n_valid
        ctx.upload_scan(tunnel)
        ctx.process_scan(synth.sample_indices(nv, H, 3, seed=13), synth.sample_indices(nv, H, 2, seed=14))
        cloud = ctx.download_cloud(1)
        models = [ctx.model(capi.GM_MODEL_PLANE), ctx.model(capi.GM_MODEL_CYLINDER)]
        test12 = ctx.download_hypotheses(capi.GM_MODEL_CYLINDER, H)[1]
        assert ctx.counts().device_error == 0
    mp, mc = models
    assert mp["best_id"] >= 0 and mc["best_id"] >= 0
    _assert_reference(_reference_devs(cloud, mp, O.labels(cloud, mp["hyp"], TAU, None) == 1))
    _assert_reference(_reference_devs(cloud, mc, O.labels(cloud, None, TAU, test12[mc["best_id"]]) == 2))


def test_scratch_and_stream_reuse(tunnel, tunnel_draws):
    """Repeated extractions, an extraction after a compression (which writes its residual cloud into the extraction's
    working copies) and the one-stream path (profiling on) all give the same bits; gm_ransac's tile-culled counts over
    the context's cell-sorted copy and leaf bounds are the same before and after."""
    pd, cd = tunnel_draws
    with capi.Context(capi.default_params(), max_points=len(tunnel), max_hypotheses=H) as ctx:
        ctx.set_count_mode(0)
        ctx.upload_scan(tunnel)
        ctx.crop()
        ctx.normals()
        nv = ctx.counts().n_valid
        ps, cs = synth.sample_indices(nv, H, 3, seed=15), synth.sample_indices(nv, H, 2, seed=16)

        def ransac_counts():
            ctx.ransac(capi.GM_MODEL_PLANE, ps)
            ctx.ransac(capi.GM_MODEL_CYLINDER, cs)
            return [ctx.download_hypotheses(k, H)[2].copy() for k in (capi.GM_MODEL_PLANE, capi.GM_MODEL_CYLINDER)]

        def extract(compress):
            ctx.extract_primitives(pd, cd, K, 1)
            g = ctx.primitives()
            r = ([(p["kind"], p["best_id"], p["best_count"], p["refit_count"], p["n_remaining"], p["hyp"].tobytes(), p["coef"].tobytes(),
                   p["rms"]) for p in g], ctx.download_primitive_ids().tobytes())
            if compress:
                ctx.compress_primitives()
                r += (ctx.download_compressed_primitives(),)
            return r

        before = ransac_counts()
        first = extract(False)
        second = extract(True)  # extract twice
        third = extract(True)  # after a compression
        ctx.profile_enable(True)
        one_stream = extract(True)
        ctx.profile_enable(False)
        after = ransac_counts()
        assert ctx.counts().device_error == 0
    assert len(first[0]) > 8
    assert second[:2] == first and third == second and one_stream == second
    for a, b in zip(before, after):
        assert np.array_equal(a, b)


# ---- 64 primitives: 90 separated plane patches --------------------------------------------------------------------
CAP_PRM = dict(neighborRadius=0.1, cylinderRadiusMin=0.3)
CAP_HP, CAP_HC, CAP_MIN = 256, 64, 100


def _patches(n_patches=90, seed=40):
    """Plane patches 0.7 m square (800..1690 points, 2 mm noise) of random orientations, one per node of a 2 m lattice in
    the 5 m crop box: a cascade that still finds a patch of 100+ points in round 64."""
    g = np.random.Generator(np.random.Philox(seed))
    nodes = [(x, y, z) for z in (-3.0, -1.0, 1.0, 3.0) for y in (-4.0, -2.0, 0.0, 2.0, 4.0) for x in (-4.0, -2.0, 0.0, 2.0, 4.0)]
    out = []
    for k in range(n_patches):
        p = synth.plane_patch(800 + 10 * k, seed=seed + 1 + k, normal=g.normal(size=3), offset=0.0, half=0.35, noise=0.002)
        p[:, :3] += np.asarray(nodes[k], np.float32)
        out.append(p)
    return np.concatenate(out)


def test_cascade_fills_all_64_slots():
    pd, cd = synth.sample_draws(K, CAP_HP, 3, seed=21), synth.sample_draws(K, CAP_HC, 2, seed=22)
    run = _run(_patches(), CAP_PRM, pd, cd, K, CAP_MIN, count_mode=0)
    expected = _oracle(run, pd, cd, K, CAP_MIN, rmin=CAP_PRM["cylinderRadiusMin"])
    _assert_parity(run["prims"], run["ids"], expected, K, CAP_MIN)
    assert len(run["prims"]) == K and int(run["ids"].max()) == K and len(expected[2]) == K
    for d in _extraction_reference_devs(run):
        _assert_reference(d)
    d = _compression_devs(run, 0.1)
    _assert_compression(d)
    assert d["header"].n_primitives == K and len(capi.parse_compressed_primitives(run["blob"])["records"]) == K


# ---- every point claimed ---------------------------------------------------------------------------------------------
def test_cloud_that_runs_out_of_points():
    """186 compacted points, four planes claim them all: round 5 has n_r = 0, its draws map to -1 and it stops."""
    prm = dict(neighborRadius=0.5)
    pd, cd = synth.sample_draws(8, H, 3, seed=1), synth.sample_draws(8, H, 2, seed=2)
    run = _run(synth.rectangular_drift(300, seed=3), prm, pd, cd, 8, 1)
    expected = _oracle(run, pd, cd, 8, 1)
    _assert_parity(run["prims"], run["ids"], expected, 8, 1)
    assert len(run["prims"]) == 4 and run["ids"].all()
    assert expected[2][-1] == (0, -1, -1)
    for d in _extraction_reference_devs(run):
        _assert_reference(d)
    d = _compression_devs(run, 0.1)
    h, o = d["header"], d["oracle"]
    assert h.n_residual == 0 and h.n_residual_voxels == 0 and h.residual_rms == 0.0
    assert len(capi.parse_compressed_primitives(run["blob"])["residual"]) == 0
    assert abs(h.total_rms - o["total_rms"]) <= _rms_tol(o["total_rms"])
    _assert_compression(d)
