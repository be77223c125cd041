"""Per-point times and deskew on the B200: the timed PointCloud2 decode, gm_deskew against the float64 restatement
(tests/deskew_oracle.py) and its exact cases, recovery of the snapshot, the argument and stage rules, gm_odometry_deskew
equal bit for bit to the host loop of public calls, and the accuracy of map odometry on swept scans with and without it."""
import ctypes as C

import numpy as np
import pytest

import deskew_oracle as DK
import odometry_oracle as OD
import register_oracle as R
from geometric_mapping_b200 import capi, synth

pytestmark = pytest.mark.gpu

N1M = 1_000_000
PERIOD = 0.1
WIDE = 1000.0   # a crop bound that keeps every point: gm_crop + download_cloud(0) then read the scan as uploaded
VELODYNE = (32, 0, 4, 8, 24)   # point_step, x, y, z, time: velodyne_pointcloud's PointXYZIRT (intensity @16, ring @20)
PACKED = (19, 1, 5, 9, 14)     # odd point_step, no field 4-byte aligned
C1 = dict(neighborRadius=0.05, voxelGridLeafSize=0.1)
LEAF, DMAX, RATIO, MIN_FIT = 0.1, 0.5, 0.1, 0.5
SEQ = 8


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _h(P):
    return np.vstack([np.asarray(P, np.float64)[:3, :4], [0.0, 0.0, 0.0, 1.0]])


def _records(xyzw, t, layout, fill=0xA5):
    step, ox, oy, oz, ot = layout
    n = len(t)
    raw = np.full((n, step), fill, np.uint8)
    for off, col in ((ox, xyzw[:, 0]), (oy, xyzw[:, 1]), (oz, xyzw[:, 2]), (ot, t)):
        raw[:, off:off + 4] = np.ascontiguousarray(col, np.float32).view(np.uint8).reshape(n, 4)
    return raw


def _upload_timed(ctx, xyzw, t, layout=VELODYNE):
    ctx.upload_pointcloud2_timed(_records(xyzw, t, layout), len(t), *layout)


def _scan_points(ctx):
    ctx.crop()
    return ctx.download_cloud(0)


def _ctx(n, **kw):
    return capi.Context(capi.default_params(**kw), max_points=max(n, 1), max_hypotheses=16)


DELTA = synth.pose34((0.0, 0.0, np.radians(1.5)), (0.15, 0.01, 0.0)).astype(np.float32)


@pytest.fixture(scope="module")
def tunnel():
    """1M-point swept curved tunnel (C1), sensor at the origin at t = 0, delta ~ 0.15 m and 1.5 degrees per period."""
    return synth.swept_scan(synth.curved_tunnel, np.eye(3, 4), DELTA, PERIOD, seed=2, n=N1M)


@pytest.fixture(scope="module")
def wide():
    c = _ctx(1 << 20, boxFilterBound=WIDE)
    yield c
    c.close()


@pytest.mark.parametrize("layout", [VELODYNE, PACKED], ids=["velodyne", "packed"])
def test_timed_decode_is_the_untimed_decode_plus_the_field(wide, tunnel, layout):
    xyzw, t = tunnel
    raw = _records(xyzw, t, layout)
    wide.upload_pointcloud2(raw, N1M, *layout[:4])
    ref = _scan_points(wide)
    wide.upload_pointcloud2_timed(raw, N1M, *layout)
    assert np.array_equal(_bits(wide.point_times()), _bits(t))
    got = _scan_points(wide)
    assert got.shape == (N1M, 4) and np.array_equal(_bits(got), _bits(ref))
    assert np.array_equal(_bits(got[:, :3]), _bits(xyzw[:, :3]))
    # an untimed upload after a timed one: no times, and no deskew
    wide.upload_pointcloud2(raw, N1M, *layout[:4])
    eye = np.eye(3, 4, dtype=np.float32)
    with pytest.raises(capi.GmError) as e:
        wide.deskew(eye, 0.0, PERIOD)
    assert e.value.status == capi.GM_ERR_STAGE_ORDER
    with pytest.raises(capi.GmError) as e:
        wide.point_times()
    assert e.value.status == capi.GM_ERR_STAGE_ORDER


def test_deskew_matches_the_restatement(wide, tunnel):
    xyzw, t = tunnel
    t = t.copy()
    t_ref = float(np.float32(0.05))
    t[::1000] = np.float32(t_ref)                               # points taken at t_ref
    _upload_timed(wide, xyzw, t)
    wide.reset_launch_count()
    wide.deskew(DELTA, t_ref, PERIOD)
    assert wide.launch_count == 1
    got = _scan_points(wide)
    ref = DK.deskew(xyzw, t, DELTA, t_ref, PERIOD)
    assert got.shape == (N1M, 4) and (got[:, 3] == 1.0).all()
    err = np.abs(got[:, :3].astype(np.float64) - ref)
    assert (err <= 2 * np.spacing(np.abs(ref).astype(np.float32))).all(), err.max()
    assert np.array_equal(_bits(got[::1000, :3]), _bits(xyzw[::1000, :3]))    # t == t_ref: unchanged
    assert np.abs(got[:, :3] - xyzw[:, :3]).max() > 0.1                         # the others moved
    _upload_timed(wide, xyzw, t)
    wide.deskew(DELTA, t_ref, PERIOD)
    assert np.array_equal(_bits(_scan_points(wide)), _bits(got))                # run to run


def test_exact_cases(wide, tunnel):
    xyzw, t = (a[:200_000].copy() for a in tunnel)
    _upload_timed(wide, xyzw, t)
    wide.deskew(np.eye(3, 4, dtype=np.float32), 0.03, PERIOD)                   # identity delta
    assert np.array_equal(_bits(_scan_points(wide)), _bits(xyzw))
    nan, inf = np.float32(np.nan), np.float32(np.inf)
    xyzw[1, 0], xyzw[2, 1], xyzw[3, 2], xyzw[4, 0] = nan, inf, -inf, nan
    t[5], t[6], t[7] = nan, inf, -inf
    _upload_timed(wide, xyzw, t)
    wide.deskew(DELTA, 0.0, PERIOD)
    got = _scan_points(wide)
    assert got.shape == xyzw.shape                                              # NaN points stay (is_dense = 1)
    assert np.isnan(got[1:8, :3]).all() and (got[1:8, 3] == 1.0).all()
    assert np.isfinite(got[8:, :3]).all() and np.isfinite(got[0, :3]).all()
    # with is_dense = 0 the crop drops them as it drops NaN input points
    with _ctx(200_000, boxFilterBound=WIDE, is_dense=0) as c:
        _upload_timed(c, xyzw, t)
        c.deskew(DELTA, 0.0, PERIOD)
        assert c.counts().n_input == 200_000 and len(_scan_points(c)) == 200_000 - 7


def test_deskew_recovers_the_snapshot(wide):
    pose = synth.pose34((0.0, 0.0, np.radians(2.0)), (-0.3, 0.05, 0.0))
    pts = synth.drift_end_niche(N1M, seed=31)
    q, t = synth.swept_view(pts, pose, DELTA, PERIOD)
    xyzw = np.concatenate([q.astype(np.float32), np.ones((N1M, 1), np.float32)], axis=1)
    _upload_timed(wide, xyzw, t, PACKED)
    wide.deskew(DELTA, 0.0, PERIOD)
    got = _scan_points(wide)
    snap = synth.view_from(pts, pose)
    assert np.abs(xyzw[:, :3] - snap[:, :3]).max() > 0.1
    assert np.abs(got[:, :3] - snap[:, :3]).max() <= 1e-5


def test_calls_do_not_wait_for_the_device(wide, tunnel):
    import torch

    xyzw, t = tunnel
    stream = torch.cuda.Stream()
    busy = []
    wide.set_stream(stream.cuda_stream)
    try:
        with capi.VoxelMap(LEAF, 1 << 12) as vmap, capi.Odometry(vmap) as odo:
            for call in (lambda: wide.deskew(DELTA, 0.0, PERIOD), lambda: odo.deskew(wide, 0.0, PERIOD)):
                _upload_timed(wide, xyzw, t)
                wide.synchronize()
                with torch.cuda.stream(stream):
                    torch.cuda._sleep(200_000_000)
                call()
                busy.append(not stream.query())
                wide.synchronize()
    finally:
        wide.set_stream(None)
    assert busy == [True, True]


def test_argument_and_stage_rules(wide, tunnel):
    lib = capi._lib()
    xyzw, t = (a[:1000] for a in tunnel)
    raw = _records(xyzw, t, VELODYNE)
    h = wide._h
    eye = np.ascontiguousarray(np.eye(3, 4, dtype=np.float32))
    # the timed upload checks the time offset as the untimed one checks x, y, z
    assert lib.gm_upload_pointcloud2_timed(h, capi._ptr(raw), 1000, 32, 0, 4, 8, 29) == capi.GM_ERR_INVALID_ARG
    assert lib.gm_upload_pointcloud2_timed(h, capi._ptr(raw), 1000, 32, 0, 4, 29, 24) == capi.GM_ERR_INVALID_ARG
    assert lib.gm_upload_pointcloud2_timed(h, capi._ptr(raw), 1000, 32, 0, 4, 8, 28) == capi.GM_OK
    assert lib.gm_download_point_times(h, capi._ptr(np.empty(999, np.float32)), 999) == capi.GM_ERR_CAPACITY
    _upload_timed(wide, xyzw, t)
    wide.synchronize()
    wide.reset_launch_count()
    for bad in (np.nan, np.inf):
        d = eye.copy()
        d[1, 3] = bad
        assert lib.gm_deskew(h, capi._ptr(d), 0.0, PERIOD) == capi.GM_ERR_INVALID_ARG
    assert lib.gm_deskew(h, None, 0.0, PERIOD) == capi.GM_ERR_INVALID_ARG
    assert lib.gm_deskew(None, capi._ptr(eye), 0.0, PERIOD) == capi.GM_ERR_INVALID_ARG
    for t_ref, period in ((np.nan, PERIOD), (np.inf, PERIOD), (0.0, 0.0), (0.0, -PERIOD), (0.0, np.nan), (0.0, np.inf)):
        assert lib.gm_deskew(h, capi._ptr(eye), t_ref, period) == capi.GM_ERR_INVALID_ARG, (t_ref, period)
    assert wide.launch_count == 0
    assert lib.gm_deskew(h, capi._ptr(eye), 0.0, PERIOD) == capi.GM_OK
    assert lib.gm_deskew(h, capi._ptr(eye), 0.0, PERIOD) == capi.GM_ERR_STAGE_ORDER         # a second time
    import torch
    buf = torch.from_numpy(np.ascontiguousarray(xyzw)).cuda()
    for untimed in (lambda: wide.crop(),                                        # after gm_crop of a timed upload
                    lambda: wide.upload_scan(xyzw), lambda: wide.upload_pointcloud2(raw, 1000, *VELODYNE[:4]),
                    lambda: wide.set_scan_device(buf.data_ptr(), 1000)):
        _upload_timed(wide, xyzw, t)
        untimed()
        wide.reset_launch_count()
        assert lib.gm_deskew(h, capi._ptr(eye), 0.0, PERIOD) == capi.GM_ERR_STAGE_ORDER
        assert wide.launch_count == 0
    assert lib.gm_download_point_times(h, capi._ptr(np.empty(1000, np.float32)), 1000) == capi.GM_ERR_STAGE_ORDER
    wide.synchronize()
    # the odometry call: the same rules, capacity and launch count
    with capi.VoxelMap(LEAF, 1 << 12) as vmap, capi.Odometry(vmap, max_steps=1) as odo, _ctx(1000, **C1) as c:
        _upload_timed(c, xyzw, t)
        c.synchronize()
        c.reset_launch_count()
        assert lib.gm_odometry_deskew(None, c._h, 0.0, PERIOD) == capi.GM_ERR_INVALID_ARG
        assert lib.gm_odometry_deskew(odo._h, c._h, 0.0, 0.0) == capi.GM_ERR_INVALID_ARG
        assert lib.gm_odometry_deskew(odo._h, c._h, np.nan, PERIOD) == capi.GM_ERR_INVALID_ARG
        assert c.launch_count == 0
        odo.deskew(c, 0.0, PERIOD)
        assert c.launch_count == 2
        assert lib.gm_odometry_deskew(odo._h, c._h, 0.0, PERIOD) == capi.GM_ERR_STAGE_ORDER
        c.crop()
        c.normals()
        c.voxel()
        odo.step(c)
        _upload_timed(c, xyzw, t)
        c.synchronize()
        c.reset_launch_count()
        assert lib.gm_odometry_deskew(odo._h, c._h, 0.0, PERIOD) == capi.GM_ERR_CAPACITY    # k = max_steps
        assert c.launch_count == 0


# ---- map odometry on swept scans ------------------------------------------------------------------------------------
# The sensor moves at constant velocity, ~0.15 m and 1 degree of yaw per 0.1 s scan, along the drift of
# tests/test_gpu_odometry.py; TRUTH[k] is its pose at the start of sweep k (t_ref = 0).
MOTION = synth.pose34((0.0, 0.0, np.radians(1.0)), (0.15, 0.005, 0.0))
TRUTH = [(_h(synth.pose34((0.0, 0.0, 0.0), (-0.35, 0.0, 0.0))) @ np.linalg.matrix_power(_h(MOTION), k))[:3] for k in range(SEQ)]
MOTION32 = MOTION.astype(np.float32)


@pytest.fixture(scope="module")
def swept():
    return [synth.swept_scan(synth.drift_end_niche, TRUTH[k], MOTION, PERIOD, seed=80 + k, n=N1M) for k in range(SEQ)]


@pytest.fixture(scope="module")
def ctxs():
    cs = [_ctx(N1M, **C1), _ctx(N1M, **C1)]
    yield cs
    for c in cs:
        c.close()


def _process(ctx):
    ctx.crop()
    ctx.normals()
    ctx.voxel()


def _map_state(vmap):
    d = vmap.download()
    return d["ijk"], d["counts"], _bits(d["centroids"]), _bits(vmap.planes(RATIO))


def _run(ctxs, scans, mode):
    """mode: "odo" = gm_odometry_deskew; "host" = gm_deskew with the increment restated from gm_odometry_get."""
    vmap = capi.VoxelMap(LEAF, 1 << 18)
    with capi.Odometry(vmap, TRUTH[0], max_planarity=RATIO, max_correspondence_distance=DMAX, min_fitness=MIN_FIT) as odo:
        for k in range(SEQ):
            ctx = ctxs[k % 2]
            xyzw, t = scans[k]
            _upload_timed(ctx, xyzw, t)
            if mode == "host":
                P = odo.trajectory()["poses"]
                D = np.eye(3, 4) if k < 2 else OD.compose(OD.inverse(OD.f64(P[k - 2])), OD.f64(P[k - 1]))
                ctx.deskew(D.astype(np.float32), 0.0, PERIOD)
            else:
                ctx.reset_launch_count()
                odo.deskew(ctx, 0.0, PERIOD)
                assert ctx.launch_count == 2
            _process(ctx)
            odo.step(ctx)
        traj = odo.trajectory()
    state = _map_state(vmap)
    vmap.close()
    return traj, state


@pytest.fixture(scope="module")
def runs(ctxs, swept):
    return {m: _run(ctxs, swept, m) for m in ("odo", "host")}


def test_odometry_deskew_equals_the_host_loop_bit_for_bit(runs):
    (a, amap), (b, bmap) = runs["odo"], runs["host"]
    assert a["accepted"].all()
    for key in a:
        x, y = a[key], b[key]
        assert np.array_equal(x.view(np.uint32), y.view(np.uint32)) if x.dtype == np.float32 else np.array_equal(x, y), key
    for x, y in zip(amap, bmap):
        assert np.array_equal(x, y)


# Accuracy: 16 swept scans along the drift from x = -1.2 m (2.25 m and 15 degrees in all), constant-velocity guess.
#   "given":    every scan deskewed with the true motion through gm_deskew (what an IMU gives);
#   "odometry": the first two scans as in "given", the rest through gm_odometry_deskew;
#   "none":     the same scans uploaded untimed;  "snapshot": the same draws seen without a sweep (synth.view_from).
# Measured on one NVIDIA B200 (1000 W power limit), largest per-step error over steps 1..15, rotation / translation:
#   given 3.2e-4 rad / 4.4 mm, odometry 8.0e-4 rad / 12.3 mm, none 3.0e-3 rad / 28.5 mm, snapshot 3.2e-4 rad / 3.4 mm.
# The runs are deterministic; the bars below are those numbers with a margin.  Deskewing with the true motion brings the
# swept scans to the accuracy of snapshots and is 6.4x better in translation than no deskew.  The odometry's own
# estimate is only 2.3x better: the increment it deskews with carries the pose errors of the two steps it comes from, and
# those errors feed back (its error grows over the last steps, 7.8 and 12.3 mm).  Neither run meets the per-step bars of
# snapshot registration in tests/test_gpu_register_map.py (3e-4 rad, 2e-3 m); over 16 scans the snapshot run does not
# either (3.4 mm): they bound one registration, this is 2.25 m of odometry.  Under constant velocity every skewed scan is
# distorted alike in its own frame, so the skew reaches the trajectory only as the scene moves relative to the sensor:
# over the 8 scans of SEQ (0.15 m, 1 degree a scan from x = -0.35 m) "odometry" and "none" measured 2.9 mm / 2.8e-4 rad
# and 3.0 mm / 4.6e-4 rad, which does not separate them.
ACC = 16
ACC_START = synth.pose34((0.0, 0.0, 0.0), (-1.2, 0.0, 0.0))
ACC_TRUTH = [(_h(ACC_START) @ np.linalg.matrix_power(_h(MOTION), k))[:3] for k in range(ACC)]


def _accuracy_run(ctxs, mode):
    with capi.VoxelMap(LEAF, 1 << 18) as vmap, capi.Odometry(vmap, ACC_TRUTH[0], max_planarity=RATIO,
                                                             max_correspondence_distance=DMAX, min_fitness=MIN_FIT) as odo:
        for k in range(ACC):
            ctx = ctxs[k % 2]
            pts = synth.drift_end_niche(N1M, seed=100 + k)
            if mode == "snapshot":
                ctx.upload_scan(synth.view_from(pts, ACC_TRUTH[k]))
            else:
                q, t = synth.swept_view(pts, ACC_TRUTH[k], MOTION, PERIOD)
                xyzw = np.concatenate([q.astype(np.float32), np.ones((N1M, 1), np.float32)], axis=1)
                if mode == "none":
                    ctx.upload_scan(xyzw)
                else:
                    _upload_timed(ctx, xyzw, t)
                    if mode == "given" or k < 2:
                        ctx.deskew(MOTION32, 0.0, PERIOD)
                    else:
                        odo.deskew(ctx, 0.0, PERIOD)
            _process(ctx)
            odo.step(ctx)
        traj = odo.trajectory()
    assert traj["accepted"].all(), mode
    return np.array([R.pose_error(traj["poses"][k], ACC_TRUTH[k]) for k in range(1, ACC)])


def test_deskewed_odometry_is_accurate_and_the_skewed_one_is_not(ctxs):
    e = {m: _accuracy_run(ctxs, m) for m in ("given", "odometry", "none", "snapshot")}
    for m, v in e.items():
        print("\n%s: max rot %.3e rad, max trans %.3e m; per step %s" % (m, v[:, 0].max(), v[:, 1].max(), v.round(6).tolist()))
    rot, trans = {m: v[:, 0].max() for m, v in e.items()}, {m: v[:, 1].max() for m, v in e.items()}
    assert rot["given"] <= 4e-4 and trans["given"] <= 5e-3, e["given"]
    assert rot["odometry"] <= 1e-3 and trans["odometry"] <= 1.5e-2, e["odometry"]
    assert trans["given"] <= 1.5 * trans["snapshot"]
    assert trans["none"] >= 5 * trans["given"] and rot["none"] >= 5 * rot["given"], (trans, rot)
    assert trans["none"] >= 2 * trans["odometry"] and rot["none"] >= 3 * rot["odometry"], (trans, rot)
