"""gm_register_map on the B200 against the CPU restatement (tests/register_map_oracle.py): bit-exact map planes,
correspondences and residuals, the restatement's trajectory, recovery of known sensor poses at 1M points, an 8-scan
register-then-insert sequence, saved maps, determinism, the launch contract, argument and stage rules, edge inputs and
the ordering of map operations issued from different contexts."""
import ctypes as C
import math

import numpy as np
import pytest

import register_map_oracle as M
import register_oracle as R
from geometric_mapping_b200 import capi, synth

pytestmark = pytest.mark.gpu

N1M = 1_000_000
C1 = dict(neighborRadius=0.05, voxelGridLeafSize=0.1)
LEAF, DMAX, RATIO = 0.1, 0.5, 0.1
# the restatement's map and bars (tests/test_oracle_register_map.py)
MAP_POSES = [((0.0, 0.0, 0.0), (0.0, 0.0, 0.0)), ((0.0, 0.0, 2.0), (0.15, 0.03, 0.0)), ((0.0, 0.0, -2.0), (-0.15, -0.03, 0.0))]
RECOVERY_CASES = [((0.0, 0.0, 5.0), (0.3, 0.0, 0.0), 9), ((3.0, -2.0, 2.0), (0.1, -0.2, 0.15), 10),
                  ((-2.0, 4.0, -3.0), (-0.25, 0.1, -0.1), 11)]
MAP_ROT_BAR, MAP_TRANS_BAR = 3e-4, 2e-3
INT_MIN = np.iinfo(np.int32).min


def _ctx(n, **kw):
    return capi.Context(capi.default_params(**kw), max_points=max(n, 1), max_hypotheses=16)


def _scan(ctx, pts):
    ctx.upload_scan(pts)
    ctx.crop()
    ctx.normals()
    ctx.voxel()


def _centroids(ctx):
    return ctx.download_voxels(with_nn=False)["centroids"]


def _reg_bytes(ctx):
    return bytes(ctx.registration()["_struct"])


def _same_float_bits(a, b):
    return np.array_equal(np.asarray(a, np.float32).view(np.uint32), np.asarray(b, np.float32).view(np.uint32))


def _assert_corr_equal(ijk, res, ref_ijk, ref_res):
    assert np.array_equal(ijk, ref_ijk)
    ok = ijk[:, 0] != INT_MIN
    assert _same_float_bits(res[ok], ref_res[ok]) and np.isnan(res[~ok]).all()


def _plane_map(vmap, ratio=RATIO):
    d = vmap.download()
    return M.PlaneMap(d["ijk"], d["centroids"], vmap.leaf, ratio)


def _pose(deg, t):
    return synth.pose34(np.radians(deg), t)


@pytest.fixture(scope="module")
def world():
    """A map of three 1M-point drift scans inserted at their sensor poses, and the voxel centroids of a fourth scan from a
    known sensor pose as the source."""
    T = _pose((2.0, -1.5, 3.0), (0.2, -0.1, 0.05))
    vmap = capi.VoxelMap(LEAF, 1 << 18)
    ins, src = _ctx(N1M, **C1), _ctx(N1M, **C1)
    for k, (d, t) in enumerate(MAP_POSES):
        P = _pose(d, t)
        _scan(ins, synth.second_scan(synth.drift_end_niche, P, seed=40 + k, n=N1M))
        vmap.insert(ins, P)
    _scan(src, synth.second_scan(synth.drift_end_niche, T, seed=9, n=N1M))
    yield {"map": vmap, "src": src, "ins": ins, "T": T, "pm": _plane_map(vmap), "cen": _centroids(src)}
    src.close()
    ins.close()
    vmap.close()


def test_map_planes_are_bit_identical_to_the_restatement(world):
    vmap = world["map"]
    d = vmap.download()
    for ratio in (0.01, RATIO, 1.0):
        got = vmap.planes(ratio)
        ref = M.planes_xyzw(M.planes(d["ijk"], d["centroids"], ratio))
        assert got.shape == ref.shape == (len(d["ijk"]), 4)
        has = got[:, 3] == 1.0
        assert np.array_equal(got[:, 3], ref[:, 3]) and ((got[:, 3] == 0.0) | has).all()
        assert _same_float_bits(got[has, :3], ref[has, :3]) and np.isnan(got[~has, :3]).all()
        if ratio == RATIO:
            assert 0.85 < has.mean() < 0.99


def test_one_iteration_is_bit_exact_against_the_restatement(world):
    init = _pose((1.0, -1.0, 2.0), (0.15, -0.05, 0.0))
    g = world["src"].register_map(world["map"], init, max_planarity=RATIO, max_iterations=1, max_correspondence_distance=DMAX)
    ijk, res = world["src"].download_map_correspondences()
    ref = M.icp(world["cen"], world["pm"], init, d_max=DMAX, max_iterations=1)
    _assert_corr_equal(ijk, res, ref["ijk"], ref["residual"])
    assert g["n_correspondences"] == ref["counts"][0] > 0.5 * g["n_source"] and g["n_source"] == len(world["cen"])
    assert np.abs(g["eigenvalues"] - ref["eigenvalues"]).max() <= 1e-10 * ref["eigenvalues"][5]
    want = ref["pose"].astype(np.float32)
    assert (np.abs(g["pose"] - want) <= np.spacing(np.abs(want))).all()
    assert g["iterations"] == 1 and g["n_degenerate"] == ref["n_degenerate"] == 0
    assert g["rmse"] == pytest.approx(math.sqrt(ref["sum_r2"] / ref["counts"][0]), rel=1e-6)


def test_full_run_follows_the_restatement(world):
    src, vmap = world["src"], world["map"]
    g = src.register_map(vmap, np.eye(3, 4), max_correspondence_distance=DMAX)
    ref = M.icp(world["cen"], world["pm"], np.eye(3, 4), d_max=DMAX)
    assert g["converged"] == ref["converged"] == 1 and g["iterations"] == ref["iterations"] >= 2
    assert np.abs(g["pose"] - ref["pose"]).max() <= 1e-6
    ijk, res = src.download_map_correspondences()
    # the input pose of the last iteration is the result of a run one iteration shorter (the launches are deterministic)
    T_in = src.register_map(vmap, np.eye(3, 4), max_correspondence_distance=DMAX, max_iterations=g["iterations"] - 1)["pose"]
    last = M.icp(world["cen"], world["pm"], T_in, d_max=DMAX, max_iterations=1)
    _assert_corr_equal(ijk, res, last["ijk"], last["residual"])
    rot, trans = R.pose_error(g["pose"], world["T"])
    assert rot <= MAP_ROT_BAR and trans <= MAP_TRANS_BAR, (rot, trans)


@pytest.mark.parametrize("deg,t,seed", RECOVERY_CASES)
def test_recovers_known_poses_at_1m_points(world, deg, t, seed):
    T = _pose(deg, t)
    with _ctx(N1M, **C1) as src:
        _scan(src, synth.second_scan(synth.drift_end_niche, T, seed=seed, n=N1M))
        g = src.register_map(world["map"], np.eye(3, 4), max_correspondence_distance=DMAX)
    rot, trans = R.pose_error(g["pose"], T)
    assert g["converged"] == 1 and g["fitness"] > 0.9 and rot <= MAP_ROT_BAR and trans <= MAP_TRANS_BAR, (g["iterations"], rot, trans)


# Register each scan to the map of the previous ones (guess: the previous estimate), then insert it at the estimated pose;
# the first scan is inserted at its known pose.  The restatement on this sequence ends 7 registrations later at 3.4e-4 rad
# and 3.0 mm (bars: 2 x the single-registration ones); the scan-to-scan chain of the same scans, at 4.2e-4 rad, 1.9 mm.
SEQ_FACTOR = 2.0


def test_eight_scan_sequence_registered_to_the_growing_map(capsys):
    truth = [_pose((0.0, 0.0, 1.0 * k), (-0.35 + 0.1 * k, 0.02 * k, 0.0)) for k in range(8)]
    ctxs = [_ctx(N1M, **C1), _ctx(N1M, **C1)]
    vmap = capi.VoxelMap(LEAF, 1 << 18)
    rows = []
    try:
        _scan(ctxs[0], synth.second_scan(synth.drift_end_niche, truth[0], seed=50, n=N1M))
        vmap.insert(ctxs[0], truth[0])
        est, chain = truth[0].astype(np.float32), truth[0].astype(np.float64)
        for k in range(1, 8):
            cur, prev = ctxs[k % 2], ctxs[(k - 1) % 2]
            _scan(cur, synth.second_scan(synth.drift_end_niche, truth[k], seed=50 + k, n=N1M))
            g = cur.register_map(vmap, est, max_correspondence_distance=DMAX)
            assert g["converged"] == 1, k
            est = g["pose"]
            vmap.insert(cur, est)
            rel = cur.register(prev, np.eye(3, 4), max_correspondence_distance=DMAX)["pose"].astype(np.float64)
            chain = np.concatenate([chain[:, :3] @ rel[:, :3], (chain[:, :3] @ rel[:, 3] + chain[:, 3])[:, None]], axis=1)
            rows.append((k, *R.pose_error(est, truth[k]), *R.pose_error(chain, truth[k])))
    finally:
        for c in ctxs:
            c.close()
        vmap.close()
    with capsys.disabled():
        for r in rows:
            print("scan %d: to the map %.2e rad %.2f mm | scan-to-scan chain %.2e rad %.2f mm" % (r[0], r[1], 1e3 * r[2], r[3], 1e3 * r[4]))
    k, rot, trans = rows[-1][:3]
    assert rot <= SEQ_FACTOR * MAP_ROT_BAR and trans <= SEQ_FACTOR * MAP_TRANS_BAR, rows[-1]


def test_saved_map_gives_the_same_registration(world, tmp_path):
    src = world["src"]
    init = _pose((1.0, 0.5, -1.0), (0.1, 0.05, 0.0))
    src.register_map(world["map"], init, max_correspondence_distance=DMAX)
    b1, c1 = _reg_bytes(src), src.download_map_correspondences()
    path = str(tmp_path / "drift.gmm")
    world["map"].save(path)
    with capi.VoxelMap.load(path) as loaded:
        src.register_map(loaded, init, max_correspondence_distance=DMAX)
        b2, c2 = _reg_bytes(src), src.download_map_correspondences()
        assert _same_float_bits(loaded.planes(RATIO), world["map"].planes(RATIO))
    assert b1 == b2 and np.array_equal(c1[0], c2[0]) and _same_float_bits(c1[1], c2[1])


def test_deterministic_and_idempotent_after_convergence(world):
    src, vmap = world["src"], world["map"]
    src.register_map(vmap, np.eye(3, 4), max_correspondence_distance=DMAX)
    b1, c1 = _reg_bytes(src), src.download_map_correspondences()
    src.register_map(vmap, np.eye(3, 4), max_correspondence_distance=DMAX)
    b2, c2 = _reg_bytes(src), src.download_map_correspondences()
    assert b1 == b2 and np.array_equal(c1[0], c2[0]) and _same_float_bits(c1[1], c2[1])
    k = src.registration()["iterations"]
    src.register_map(vmap, np.eye(3, 4), max_correspondence_distance=DMAX, max_iterations=k)
    b3 = _reg_bytes(src)
    src.register_map(vmap, np.eye(3, 4), max_correspondence_distance=DMAX, max_iterations=k + 10)
    assert b3 == _reg_bytes(src) == b1


@pytest.mark.parametrize("iters", [1, 5, 30, 64])
def test_launch_count_is_max_iterations_plus_two(world, iters):
    src = world["src"]
    src.synchronize()
    src.reset_launch_count()
    src.register_map_async(world["map"], np.eye(3, 4), max_iterations=iters)
    assert src.launch_count == iters + 2
    src.synchronize()


def test_argument_and_stage_rules(world):
    lib = capi._lib()
    src, vmap = world["src"], world["map"]

    def st(ctx, m, ratio=RATIO, **kw):
        p = capi.icp_params(**kw)
        return lib.gm_register_map(ctx._h, None if m is None else m._h, C.byref(p), C.c_double(ratio))

    for r in (0.0, -0.1, 1.0000001, float("nan"), float("inf")):
        assert st(src, vmap, r) == capi.GM_ERR_INVALID_ARG, r
    assert st(src, vmap, 1.0) == capi.GM_OK
    assert st(src, vmap, max_correspondence_distance=0.0) == capi.GM_ERR_INVALID_ARG
    assert st(src, vmap, max_correspondence_distance=float("nan")) == capi.GM_ERR_INVALID_ARG
    assert st(src, vmap, max_iterations=0) == capi.GM_ERR_INVALID_ARG
    assert st(src, vmap, degeneracy_ratio=1.0) == capi.GM_ERR_INVALID_ARG
    assert st(src, None) == capi.GM_ERR_INVALID_ARG
    bad = capi.icp_params()
    bad.init_pose34[3] = float("inf")
    assert lib.gm_register_map(src._h, vmap._h, C.byref(bad), C.c_double(RATIO)) == capi.GM_ERR_INVALID_ARG
    assert lib.gm_register_map(src._h, vmap._h, None, C.c_double(RATIO)) == capi.GM_ERR_INVALID_ARG
    n = C.c_size_t(0)
    assert lib.gm_map_download_planes(vmap._h, C.c_double(0.0), None, 0, C.byref(n)) == capi.GM_ERR_INVALID_ARG
    pts = synth.drift_end_niche(20_000, seed=13)
    with _ctx(len(pts), **C1) as a, _ctx(len(pts), **C1) as b:
        a.upload_scan(pts)
        a.crop()
        a.normals()
        assert st(a, vmap) == capi.GM_ERR_STAGE_ORDER          # source without voxels
        a.voxel()
        assert st(a, vmap) == capi.GM_OK
        r = capi.gm_registration()
        assert lib.gm_get_registration(a._h, C.byref(r)) == capi.GM_OK and r.n_source > 0
        idx = np.empty(r.n_source, np.int32)
        ijk = np.empty((r.n_source, 3), np.int32)
        assert lib.gm_download_correspondences(a._h, capi._ptr(idx), None, r.n_source) == capi.GM_ERR_STAGE_ORDER
        assert lib.gm_download_map_correspondences(a._h, capi._ptr(ijk), None, r.n_source - 1) == capi.GM_ERR_CAPACITY
        assert lib.gm_download_map_correspondences(a._h, capi._ptr(ijk), None, r.n_source) == capi.GM_OK
        _scan(b, pts)
        a.register(b, np.eye(3, 4))
        assert lib.gm_download_map_correspondences(a._h, capi._ptr(ijk), None, r.n_source) == capi.GM_ERR_STAGE_ORDER
        assert lib.gm_download_correspondences(a._h, capi._ptr(idx), None, r.n_source) == capi.GM_OK
        a.register_map(vmap)
        a.upload_scan(pts)                                      # a new scan on the source drops its registration
        assert lib.gm_get_registration(a._h, C.byref(r)) == capi.GM_ERR_STAGE_ORDER
        assert lib.gm_download_map_correspondences(a._h, capi._ptr(ijk), None, len(ijk)) == capi.GM_ERR_STAGE_ORDER


def _assert_no_match(g, ctx, init):
    ijk, res = ctx.download_map_correspondences()
    assert g["n_correspondences"] == 0 and g["converged"] == 0 and g["iterations"] == 1
    assert (ijk == INT_MIN).all() and np.isnan(res).all() and len(ijk) == g["n_source"] > 0
    assert np.array_equal(g["pose"], init.astype(np.float32))
    assert ctx.counts().device_error == 0


def test_empty_map_map_without_planes_and_source_far_outside(world):
    src = world["src"]
    init = _pose((0.01, 0.0, 0.0), (0.1, 0.2, 0.3))
    with capi.VoxelMap(LEAF, 1000) as empty:
        _assert_no_match(src.register_map(empty, init), src, init)
        assert empty.planes(RATIO).shape == (0, 4)
    # isolated voxels two leaves apart: no voxel has 5 occupied neighbours
    g3 = np.stack(np.meshgrid(*[np.arange(-5, 5) * 0.2 + 0.05] * 3, indexing="ij"), axis=-1).reshape(-1, 3)
    sparse = np.concatenate([g3, np.ones((len(g3), 1))], axis=1).astype(np.float32)
    with _ctx(len(sparse), neighborRadius=0.3, voxelGridLeafSize=LEAF) as c, capi.VoxelMap(LEAF, 4096) as flat:
        _scan(c, sparse)
        flat.insert(c)
        assert flat.stats()[0] > 0 and (flat.planes(RATIO)[:, 3] == 0).all()
        _assert_no_match(src.register_map(flat, init), src, init)
    far = _pose((0.0, 0.0, 0.0), (100.0, -80.0, 60.0))
    _assert_no_match(src.register_map(world["map"], far), src, far)


def test_register_then_insert_from_another_context_without_synchronisation(world, tmp_path):
    path = str(tmp_path / "m.gmm")
    world["map"].save(path)
    other = synth.second_scan(synth.curved_tunnel, np.eye(3, 4), seed=61, n=N1M)
    with _ctx(N1M, **C1) as b, capi.VoxelMap.load(path) as m:
        _scan(b, other)
        b.synchronize()
        src = world["src"]
        ref = src.register_map(m, np.eye(3, 4), max_correspondence_distance=DMAX)
        ref_b, ref_c = bytes(ref["_struct"]), src.download_map_correspondences()
        src.register_map_async(m, np.eye(3, 4), max_correspondence_distance=DMAX)
        m.insert(b, _pose((0.0, 0.0, 0.0), (0.02, 0.01, 0.0)))   # queues behind the registration
        assert _reg_bytes(src) == ref_b
        c = src.download_map_correspondences()
        assert np.array_equal(c[0], ref_c[0]) and _same_float_bits(c[1], ref_c[1])
        assert m.stats()[1] > world["map"].stats()[1]


def test_insert_then_register_from_another_context_without_synchronisation(world, tmp_path):
    path = str(tmp_path / "m.gmm")
    world["map"].save(path)
    P = _pose((0.0, 0.0, 1.0), (0.05, 0.02, 0.0))
    extra = synth.second_scan(synth.drift_end_niche, P, seed=62, n=N1M)
    src = world["src"]
    with _ctx(N1M, **C1) as b:
        _scan(b, extra)
        with capi.VoxelMap.load(path) as m:
            b.synchronize()
            m.insert(b, P)
            b.synchronize()
            ref = src.register_map(m, np.eye(3, 4), max_correspondence_distance=DMAX)
            ref_b, ref_c = bytes(ref["_struct"]), src.download_map_correspondences()
        with capi.VoxelMap.load(path) as m:
            b.synchronize()
            src.synchronize()
            m.insert(b, P)                                      # no synchronisation: the registration waits for it
            got_b = bytes(src.register_map(m, np.eye(3, 4), max_correspondence_distance=DMAX)["_struct"])
            c = src.download_map_correspondences()
    assert got_b == ref_b and np.array_equal(c[0], ref_c[0]) and _same_float_bits(c[1], ref_c[1])


def test_large_d_max_without_reachable_planes_returns_promptly(world):
    # the shell search is bounded by the box of the plane voxels, not by d_max: an empty map, a map without planes and a
    # source far from the map take no search at all, however large d_max is
    import time

    src = world["src"]
    init = _pose((0.0, 0.0, 0.0), (0.05, 0.0, 0.0))
    far = _pose((0.0, 0.0, 0.0), (300.0, -200.0, 100.0))
    g3 = np.stack(np.meshgrid(*[np.arange(-5, 5) * 0.2 + 0.05] * 3, indexing="ij"), axis=-1).reshape(-1, 3)
    sparse = np.concatenate([g3, np.ones((len(g3), 1))], axis=1).astype(np.float32)
    with capi.VoxelMap(LEAF, 1000) as empty, capi.VoxelMap(LEAF, 4096) as flat, \
            _ctx(len(sparse), neighborRadius=0.3, voxelGridLeafSize=LEAF) as c:
        _scan(c, sparse)
        flat.insert(c)
        for m, T, dmax in ((empty, init, 1e4), (flat, init, 1e4), (world["map"], far, 100.0)):
            src.synchronize()
            t0 = time.perf_counter()
            src.register_map_async(m, T, max_correspondence_distance=dmax, max_iterations=64)
            src.synchronize()
            dt = time.perf_counter() - t0
            _assert_no_match(src.registration(), src, T)
            assert dt < 1.0, dt
