"""gm_register on the B200 against the CPU restatement (tests/register_oracle.py): bit-exact correspondences and
residuals, the oracle's trajectory, recovery of known transforms at 1M points, the degenerate bore, determinism, the
launch contract, stage rules and the cross-stream ordering with the target context."""
import ctypes as C
import math

import numpy as np
import pytest

import register_oracle as R
from geometric_mapping_b200 import capi, synth

pytestmark = pytest.mark.gpu

N1M = 1_000_000
C1 = dict(neighborRadius=0.05, voxelGridLeafSize=0.1)   # the C1 configuration: 5 cm neighbour grid
DMAX = 0.5
ROT_BAR, TRANS_BAR = 3e-4, 1e-3                           # the oracle's bars at 1M / C1 (tests/test_oracle_register.py)


def _ctx(n, **kw):
    return capi.Context(capi.default_params(**kw), max_points=max(n, 1), max_hypotheses=16)


def _scan(ctx, pts):
    ctx.upload_scan(pts)
    ctx.crop()
    ctx.normals()
    ctx.voxel()


def _target_arrays(ctx):
    return ctx.download_cloud(1), ctx.download_normals(1)


def _centroids(ctx):
    return ctx.download_voxels(with_nn=False)["centroids"]


def _reg_bytes(ctx):
    return bytes(ctx.registration()["_struct"])


@pytest.fixture(scope="module")
def drift():
    """1M-point target of the six-DoF scene and a 1M-point second scan from a known sensor pose as the source."""
    T = synth.pose34(np.radians((2.0, -1.5, 3.0)), (0.2, -0.1, 0.05))
    tgt, src = _ctx(N1M, **C1), _ctx(N1M, **C1)
    _scan(tgt, synth.drift_end_niche(N1M, seed=8))
    _scan(src, synth.second_scan(synth.drift_end_niche, T, seed=9, n=N1M))
    cc, nc = _target_arrays(tgt)
    yield {"tgt": tgt, "src": src, "T": T, "cc": cc, "nc": nc, "cen": _centroids(src)}
    tgt.close()
    src.close()


def _same_float_bits(a, b):
    return np.array_equal(np.asarray(a, np.float32).view(np.uint32), np.asarray(b, np.float32).view(np.uint32))


def _assert_corr_equal(idx, res, ref_idx, ref_res):
    assert np.array_equal(idx, ref_idx)
    ok = idx >= 0
    assert _same_float_bits(res[ok], ref_res[ok]) and np.isnan(res[~ok]).all()


def test_one_iteration_is_bit_exact_against_the_oracle(drift):
    init = synth.pose34(np.radians((1.0, -1.0, 2.0)), (0.15, -0.05, 0.0))
    g = drift["src"].register(drift["tgt"], init, max_iterations=1, max_correspondence_distance=DMAX)
    idx, res = drift["src"].download_correspondences()
    ref = R.icp(drift["cen"], drift["cc"], drift["nc"], init, d_max=DMAX, max_iterations=1)
    _assert_corr_equal(idx, res, ref["index"], ref["residual"])
    assert g["n_correspondences"] == ref["counts"][0] > 0.5 * g["n_source"] and g["n_source"] == len(drift["cen"])
    lmax = ref["eigenvalues"][5]
    assert np.abs(g["eigenvalues"] - ref["eigenvalues"]).max() <= 1e-10 * lmax
    want = ref["pose"].astype(np.float32)
    assert (np.abs(g["pose"] - want) <= np.spacing(np.abs(want))).all()
    assert g["iterations"] == 1 and g["n_degenerate"] == ref["n_degenerate"] == 0
    assert g["rmse"] == pytest.approx(math.sqrt(ref["sum_r2"] / ref["counts"][0]), rel=1e-6)
    assert g["fitness"] == pytest.approx(ref["counts"][0] / len(drift["cen"]), rel=1e-6)


def test_full_run_follows_the_oracle(drift):
    g = drift["src"].register(drift["tgt"], np.eye(3, 4), max_correspondence_distance=DMAX)
    ref = R.icp(drift["cen"], drift["cc"], drift["nc"], np.eye(3, 4), d_max=DMAX)
    assert g["converged"] == ref["converged"] == 1 and g["iterations"] == ref["iterations"] >= 2
    assert np.abs(g["pose"] - ref["pose"]).max() <= 1e-6
    idx, res = drift["src"].download_correspondences()
    # the input pose of the last iteration is the result of a run one iteration shorter (the launches are deterministic)
    T_in = drift["src"].register(drift["tgt"], np.eye(3, 4), max_correspondence_distance=DMAX, max_iterations=g["iterations"] - 1)["pose"]
    last = R.icp(drift["cen"], drift["cc"], drift["nc"], T_in, d_max=DMAX, max_iterations=1)
    _assert_corr_equal(idx, res, last["index"], last["residual"])
    rot, trans = R.pose_error(g["pose"], drift["T"])
    assert rot <= ROT_BAR and trans <= TRANS_BAR, (rot, trans)


def test_self_registration_search_equals_the_voxel_nn_on_an_ordinary_scan():
    # a noisy scan with outliers, several points per voxel: the centroids sit between points, so both searches walk
    # their shells and break ties; at the identity the transform is exact and the two must agree index for index
    n = 300_000
    with _ctx(n, **C1, nn_index_mode=1) as ctx:
        _scan(ctx, synth.curved_tunnel(n, seed=14))
        vox = ctx.download_voxels()
        g = ctx.register(ctx, np.eye(3, 4), max_iterations=1, max_correspondence_distance=2.0)
        idx, res = ctx.download_correspondences()
        cc, nc = _target_arrays(ctx)
    assert g["n_source"] == len(vox["nn_index"]) and np.array_equal(idx, vox["nn_index"]) and (idx >= 0).all()
    ref = R.icp(vox["centroids"], cc, nc, np.eye(3, 4), d_max=2.0, max_iterations=1)
    _assert_corr_equal(idx, res, ref["index"], ref["residual"])
    assert (res != 0).mean() > 0.9                      # the centroids are not cloud points: real residuals


def test_self_registration_keeps_identity_when_every_centroid_is_a_point():
    # noise-free, dyadic coordinates, one point per voxel: every centroid is a point of the cloud, so r = 0 and g = 0 and
    # the step is exactly zero (the search itself is compared on an ordinary scan above)
    pts = synth.dyadic(synth.drift_end_niche(40_000, seed=12, noise=0.0), 10)
    keys = np.floor(pts[:, :3] * (np.float32(1.0) / np.float32(0.1))).astype(np.int64)   # the VoxelGrid's float cells
    _, first = np.unique(keys, axis=0, return_index=True)
    pts = pts[np.sort(first)]
    with _ctx(len(pts), neighborRadius=0.3, voxelGridLeafSize=0.1, nn_index_mode=1) as ctx:
        _scan(ctx, pts)
        g = ctx.register(ctx, np.eye(3, 4), max_correspondence_distance=2.0)
        idx, res = ctx.download_correspondences()
    assert (idx >= 0).all() and (res == 0).all()
    assert np.abs(g["pose"] - np.eye(3, 4)).max() <= 1e-6 and g["converged"] == 1


@pytest.mark.parametrize("deg,t,seed", [((0.0, 0.0, 5.0), (0.3, 0.0, 0.0), 9), ((3.0, -2.0, 2.0), (0.1, -0.2, 0.15), 10),
                                        ((-2.0, 4.0, -3.0), (-0.25, 0.1, -0.1), 11)])
def test_recovers_known_transforms_at_1m_points(drift, deg, t, seed):
    T = synth.pose34(np.radians(deg), t)
    with _ctx(N1M, **C1) as src:
        _scan(src, synth.second_scan(synth.drift_end_niche, T, seed=seed, n=N1M))
        g = src.register(drift["tgt"], np.eye(3, 4), max_correspondence_distance=DMAX)
    rot, trans = R.pose_error(g["pose"], T)
    assert g["converged"] == 1 and rot <= ROT_BAR and trans <= TRANS_BAR, (g["iterations"], rot, trans)


def test_straight_bore_degeneracy():
    kw = dict(neighborRadius=0.1, voxelGridLeafSize=0.1)
    n = 200_000
    init = synth.pose34(np.radians((2.0, 1.0, 0.0)), (0.2, 0.05, -0.04))
    with _ctx(n, **kw) as tgt, _ctx(n, **kw) as src:
        _scan(tgt, synth.straight_cylinder(n, seed=1, half_length=4.0))
        _scan(src, synth.second_scan(synth.straight_cylinder, np.eye(3, 4), seed=3, n=n, half_length=4.0))
        g = src.register(tgt, init, max_correspondence_distance=DMAX, degeneracy_ratio=1e-2)
        plain = src.register(tgt, init, max_correspondence_distance=DMAX)
    vals, V = g["eigenvalues"], g["eigenvectors"]
    assert vals[1] <= 1e-2 * vals[5] < vals[2]
    for k in (0, 1):
        assert V[0, k] ** 2 + V[3, k] ** 2 >= 1.0 - 1e-2
    assert g["n_degenerate"] == 2 and g["converged"] == 1
    P = g["pose"].astype(np.float64)
    dR = P[:, :3] @ init[:, :3].T
    assert abs(P[0, 3] - init[0, 3]) <= 2e-3 and abs(math.asin(dR[2, 1])) <= 5e-4
    assert abs(P[1, 3]) <= 2e-3 and abs(P[2, 3]) <= 2e-3
    assert plain["n_degenerate"] == 0 and abs(plain["pose"][0, 3] - init[0, 3]) > 0.05


def test_four_scan_sequence_on_two_contexts():
    # sensor poses along the drift; scan k goes to context k % 2 and is registered against scan k - 1
    # the oracle on the same sequence: 0.31, 0.58, 0.87 mm and <= 1.0e-4 rad after 1, 2, 3 registrations (bars k x the single one)
    truth = [synth.pose34(np.radians((0.0, 0.0, 2.0 * k)), (-0.2 + 0.15 * k, 0.03 * k, 0.0)) for k in range(4)]
    ctxs = [_ctx(N1M, **C1), _ctx(N1M, **C1)]
    try:
        world = truth[0]
        _scan(ctxs[0], synth.second_scan(synth.drift_end_niche, truth[0], seed=20, n=N1M))
        for k in range(1, 4):
            cur, prev = ctxs[k % 2], ctxs[(k - 1) % 2]
            _scan(cur, synth.second_scan(synth.drift_end_niche, truth[k], seed=20 + k, n=N1M))
            g = cur.register(prev, np.eye(3, 4), max_correspondence_distance=DMAX)
            rel = g["pose"].astype(np.float64)
            world = np.concatenate([world[:, :3] @ rel[:, :3], (world[:, :3] @ rel[:, 3] + world[:, 3])[:, None]], axis=1)
            rot, trans = R.pose_error(world, truth[k])
            assert g["converged"] == 1 and rot <= k * ROT_BAR and trans <= k * TRANS_BAR, (k, rot, trans)
    finally:
        for c in ctxs:
            c.close()


def test_deterministic_and_idempotent_after_convergence(drift):
    src, tgt = drift["src"], drift["tgt"]
    src.register(tgt, np.eye(3, 4), max_correspondence_distance=DMAX)
    b1, c1 = _reg_bytes(src), src.download_correspondences()
    src.register(tgt, np.eye(3, 4), max_correspondence_distance=DMAX)
    b2, c2 = _reg_bytes(src), src.download_correspondences()
    assert b1 == b2 and np.array_equal(c1[0], c2[0]) and _same_float_bits(c1[1], c2[1])
    k = src.registration()["iterations"]
    src.register(tgt, np.eye(3, 4), max_correspondence_distance=DMAX, max_iterations=k)
    b3 = _reg_bytes(src)
    src.register(tgt, np.eye(3, 4), max_correspondence_distance=DMAX, max_iterations=k + 10)
    assert b3 == _reg_bytes(src) == b1


@pytest.mark.parametrize("iters", [1, 5, 30, 64])
def test_launch_count_is_max_iterations_plus_one(drift, iters):
    src = drift["src"]
    src.synchronize()
    src.reset_launch_count()
    src.register_async(drift["tgt"], np.eye(3, 4), max_iterations=iters)
    assert src.launch_count == iters + 1
    src.synchronize()


def test_stage_rules_and_invalid_arguments(drift):
    lib = capi._lib()
    src, tgt = drift["src"], drift["tgt"]

    def st(a, b, **kw):
        p = capi.icp_params(**kw)
        return lib.gm_register(a._h, b._h, C.byref(p))

    assert st(src, tgt, max_correspondence_distance=0.0) == capi.GM_ERR_INVALID_ARG
    assert st(src, tgt, max_correspondence_distance=float("nan")) == capi.GM_ERR_INVALID_ARG
    assert st(src, tgt, max_iterations=0) == capi.GM_ERR_INVALID_ARG
    assert st(src, tgt, max_iterations=capi.GM_MAX_ICP_ITERATIONS + 1) == capi.GM_ERR_INVALID_ARG
    assert st(src, tgt, degeneracy_ratio=1.0) == capi.GM_ERR_INVALID_ARG
    assert st(src, tgt, degeneracy_ratio=-0.1) == capi.GM_ERR_INVALID_ARG
    assert st(src, tgt, min_rotation_step=-1.0) == capi.GM_ERR_INVALID_ARG
    bad = capi.icp_params()
    bad.init_pose34[3] = float("inf")
    assert lib.gm_register(src._h, tgt._h, C.byref(bad)) == capi.GM_ERR_INVALID_ARG
    assert lib.gm_register(src._h, None, C.byref(bad)) == capi.GM_ERR_INVALID_ARG
    pts = synth.drift_end_niche(20_000, seed=13)
    with _ctx(len(pts), **C1) as a, _ctx(len(pts), **C1) as b:
        r = capi.gm_registration()
        assert lib.gm_get_registration(a._h, C.byref(r)) == capi.GM_ERR_STAGE_ORDER
        a.upload_scan(pts)
        a.crop()
        b.upload_scan(pts)
        b.crop()
        assert st(a, b) == capi.GM_ERR_STAGE_ORDER          # target without normals, source without voxels
        b.normals()
        assert st(a, b) == capi.GM_ERR_STAGE_ORDER          # source without voxels
        a.normals()
        a.voxel()
        assert st(a, b) == capi.GM_OK
        assert lib.gm_get_registration(a._h, C.byref(r)) == capi.GM_OK
        idx = np.empty(r.n_source, np.int32)
        assert lib.gm_download_correspondences(a._h, capi._ptr(idx), None, max(r.n_source - 1, 0)) == capi.GM_ERR_CAPACITY
        b.inject_compacted(b.download_cloud(1), b.download_normals(1))
        assert st(a, b) == capi.GM_ERR_STAGE_ORDER          # an injected cloud has no neighbour grid
        a.upload_scan(pts)                                   # a new scan on the source drops its registration
        assert lib.gm_get_registration(a._h, C.byref(r)) == capi.GM_ERR_STAGE_ORDER


def test_empty_source_and_empty_target(drift):
    init = synth.pose34((0.01, 0.0, 0.0), (0.1, 0.2, 0.3))
    with _ctx(1000, **C1) as e:
        _scan(e, np.zeros((0, 4), np.float32))
        g = e.register(drift["tgt"], init)
        assert g["n_source"] == 0 and g["n_correspondences"] == 0 and g["converged"] == 0 and g["iterations"] == 1
        assert np.array_equal(g["pose"], init.astype(np.float32)) and len(e.download_correspondences()[0]) == 0
        g = drift["src"].register(e, init)
        idx, res = drift["src"].download_correspondences()
        assert g["n_correspondences"] == 0 and (idx == -1).all() and np.isnan(res).all()
        assert np.array_equal(g["pose"], init.astype(np.float32)) and g["converged"] == 0


def test_source_far_outside_the_target_box(drift):
    init = synth.pose34((0.0, 0.0, 0.0), (100.0, -80.0, 60.0))
    g = drift["src"].register(drift["tgt"], init)
    idx, _ = drift["src"].download_correspondences()
    assert g["n_correspondences"] == 0 and (idx == -1).all() and g["converged"] == 0
    assert np.array_equal(g["pose"], init.astype(np.float32))
    assert drift["tgt"].counts().device_error == 0 and drift["src"].counts().device_error == 0
    # partly outside: the points beyond the box find nothing, the others are still searched exactly
    init = synth.pose34((0.0, 0.0, 0.0), (0.0, 0.0, 1.8))   # the roof leaves the cloud, the floor lands inside the drift
    drift["src"].register(drift["tgt"], init, max_iterations=1)
    idx, res = drift["src"].download_correspondences()
    ref = R.icp(drift["cen"], drift["cc"], drift["nc"], init, d_max=DMAX, max_iterations=1)
    _assert_corr_equal(idx, res, ref["index"], ref["residual"])
    assert 0 < (idx >= 0).sum() < len(idx)


def test_target_stream_waits_for_the_registration():
    n = 300_000
    a_pts, b_pts = synth.drift_end_niche(n, seed=30), synth.curved_tunnel(n, seed=31)
    T = synth.pose34(np.radians((1.0, 0.0, -2.0)), (0.1, 0.05, 0.0))
    with _ctx(n, **C1) as tgt, _ctx(n, **C1) as src:
        _scan(src, synth.second_scan(synth.drift_end_niche, T, seed=32, n=n))
        _scan(tgt, a_pts)
        ref = src.register(tgt, np.eye(3, 4))
        ref_b, ref_c = bytes(ref["_struct"]), src.download_correspondences()
        _scan(tgt, a_pts)
        src.register_async(tgt, np.eye(3, 4))
        tgt.upload_scan(b_pts)                   # no synchronisation: the new scan queues behind the search
        tgt.crop()
        tgt.normals()
        assert _reg_bytes(src) == ref_b
        c = src.download_correspondences()
        assert np.array_equal(c[0], ref_c[0]) and _same_float_bits(c[1], ref_c[1])
