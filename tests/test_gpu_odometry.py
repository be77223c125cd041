"""gm_odometry_* on the B200: every step equal bit for bit to the host loop of public calls it replaces (register_map from
the restated guess, the gate, insert at the returned pose), accuracy on the 8-scan drift sequence, the gate, a motion
prior on a straight bore, a reloaded map, no host synchronisation and the launch contract, determinism and the argument,
stage and capacity rules."""
import ctypes as C

import numpy as np
import pytest

import odometry_oracle as OD
import register_oracle as R
from geometric_mapping_b200 import capi, synth

pytestmark = pytest.mark.gpu

N1M = 1_000_000
C1 = dict(neighborRadius=0.05, voxelGridLeafSize=0.1)
LEAF, DMAX, RATIO, MIN_FIT = 0.1, 0.5, 0.1, 0.5
MAP_ROT_BAR, MAP_TRANS_BAR = 3e-4, 2e-3  # tests/test_gpu_register_map.py
SEQ = 8


def _ctx(n, **kw):
    return capi.Context(capi.default_params(**kw), max_points=max(n, 1), max_hypotheses=16)


def _scan(ctx, pts):
    ctx.upload_scan(pts)
    ctx.crop()
    ctx.normals()
    ctx.voxel()


def _pose(deg, t):
    return synth.pose34(np.radians(deg), t)


def _h(P):
    return np.vstack([np.asarray(P, np.float64)[:3, :4], [0.0, 0.0, 0.0, 1.0]])


def _increment(A, B):
    """A^-1 o B as float32: the motion from A to B in A's frame."""
    return np.linalg.solve(_h(A), _h(B))[:3].astype(np.float32)


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _map_state(vmap):
    d = vmap.download()
    return d["ijk"], d["counts"], _bits(d["centroids"]), _bits(vmap.planes(RATIO))


def _assert_same_map(a, b):
    for x, y in zip(a, b):
        assert np.array_equal(x, y)


# the sensor poses of tests/test_gpu_register_map.py::test_eight_scan_sequence_registered_to_the_growing_map
TRUTH = [_pose((0.0, 0.0, 1.0 * k), (-0.35 + 0.1 * k, 0.02 * k, 0.0)) for k in range(SEQ)]
DELTAS = [None] + [_increment(TRUTH[k - 1], TRUTH[k]) for k in range(1, SEQ)]


@pytest.fixture(scope="module")
def scans():
    return [synth.second_scan(synth.drift_end_niche, TRUTH[k], seed=50 + k, n=N1M) for k in range(SEQ)]


@pytest.fixture(scope="module")
def ctxs():
    cs = [_ctx(N1M, **C1), _ctx(N1M, **C1)]
    yield cs
    for c in cs:
        c.close()


def _host_loop(ctxs, scans, use_delta):
    """The loop gm_odometry_step replaces, written with public calls and the restated guess and gate."""
    vmap = capi.VoxelMap(LEAF, 1 << 18)
    poses, rows = [], []
    for k in range(SEQ):
        ctx = ctxs[k % 2]
        _scan(ctx, scans[k])
        G = OD.guess(k, TRUTH[0], poses, DELTAS[k] if use_delta and k > 0 else None)
        if k == 0:
            vmap.insert(ctx, G)
            poses.append(G)
            rows.append((G, G, 1, 0, 0))
            continue
        g = ctx.register_map(vmap, G, max_planarity=RATIO, max_correspondence_distance=DMAX)
        ok = OD.accepted(g["fitness"], g["n_correspondences"], MIN_FIT)
        P = g["pose"] if ok else G
        if ok:
            vmap.insert(ctx, P)
        poses.append(P)
        rows.append((P, G, int(ok), g["iterations"], g["n_correspondences"], g["converged"]))
    state = _map_state(vmap)
    vmap.close()
    return rows, state


def _odometry(ctxs, scans, use_delta, before_step=None):
    vmap = capi.VoxelMap(LEAF, 1 << 18)
    with capi.Odometry(vmap, TRUTH[0], max_planarity=RATIO, max_correspondence_distance=DMAX, min_fitness=MIN_FIT) as odo:
        for k in range(SEQ):
            ctx = ctxs[k % 2]
            _scan(ctx, scans[k])
            if before_step:
                before_step(ctx, k)
            odo.step(ctx, DELTAS[k] if use_delta and k > 0 else None)
            if before_step:
                before_step(ctx, None)
        assert odo.steps == SEQ
        traj = odo.trajectory()
    state = _map_state(vmap)
    vmap.close()
    return traj, state


@pytest.fixture(scope="module")
def runs(ctxs, scans):
    out = {}
    for use_delta in (False, True):
        out["host", use_delta] = _host_loop(ctxs, scans, use_delta)
        out["odo", use_delta] = _odometry(ctxs, scans, use_delta)
    return out


@pytest.mark.parametrize("use_delta", [False, True], ids=["constant_velocity", "delta"])
def test_steps_equal_the_host_loop_bit_for_bit(runs, use_delta):
    rows, host_map = runs["host", use_delta]
    traj, odo_map = runs["odo", use_delta]
    assert traj["registered"].tolist() == [0] + [1] * (SEQ - 1) and traj["accepted"].all()
    for k, row in enumerate(rows):
        assert np.array_equal(_bits(traj["poses"][k]), _bits(row[0])), k
        assert np.array_equal(_bits(traj["guesses"][k]), _bits(row[1])), k
        if k:
            assert (traj["iterations"][k], traj["n_correspondences"][k], traj["converged"][k]) == row[3:], k
    _assert_same_map(odo_map, host_map)


# The constant-velocity run ends within the bars of the 8-scan sequence of tests/test_gpu_register_map.py.
def test_constant_velocity_run_is_accurate(runs):
    traj, _ = runs["odo", False]
    rot, trans = R.pose_error(traj["poses"][-1], TRUTH[-1])
    assert rot <= 2 * MAP_ROT_BAR and trans <= 2 * MAP_TRANS_BAR, (rot, trans)
    assert (traj["fitness"][1:] > 0.9).all() and (traj["converged"][1:] == 1).all()


def test_deterministic(runs, ctxs, scans):
    traj, state = _odometry(ctxs, scans, False)
    ref, ref_state = runs["odo", False]
    for key in ref:
        a, b = traj[key], ref[key]
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32)) if a.dtype == np.float32 else np.array_equal(a, b), key
    _assert_same_map(state, ref_state)


def test_a_scan_that_cannot_match_is_rejected(ctxs, scans):
    with capi.VoxelMap(LEAF, 1 << 18) as vmap:
        with capi.Odometry(vmap, TRUTH[0], max_correspondence_distance=DMAX) as odo:
            for k in range(3):
                _scan(ctxs[k % 2], scans[k])
                odo.step(ctxs[k % 2], DELTAS[k] if k else None)
            before = _map_state(vmap)
            _scan(ctxs[1], scans[3])
            far = DELTAS[3].copy()
            far[:, 3] += (100.0, 0.0, 0.0)                      # the guess 100 m down the drift, away from the map
            odo.step(ctxs[1], far)
            _assert_same_map(_map_state(vmap), before)
            t = odo.trajectory()
            assert t["accepted"][3] == 0 and t["registered"][3] == 1 and t["n_correspondences"][3] == 0 and t["fitness"][3] == 0
            assert np.array_equal(_bits(t["poses"][3]), _bits(t["guesses"][3]))
            g = ctxs[1].registration()                          # the rejected ICP result stays readable
            assert g["n_correspondences"] == 0 and g["n_source"] == t["n_source"][3] > 0
            # the next guess dead-reckons across the rejected step: a prior that brings it back is accepted
            _scan(ctxs[0], scans[4])
            back = np.linalg.solve(_h(t["poses"][3]), _h(TRUTH[4]))[:3].astype(np.float32)
            odo.step(ctxs[0], back)
            t = odo.trajectory()
            assert t["accepted"][4] == 1 and t["fitness"][4] > 0.9
            assert R.pose_error(t["poses"][4], TRUTH[4])[1] <= 2 * MAP_TRANS_BAR
        assert vmap.stats()[1] > 0


def test_min_fitness_one_inserts_nothing_after_step_zero(ctxs, scans):
    # step 0 sees only the half x < 0 of the drift (world frame): the later scans see the other half too, so their
    # fitness stays below 1 (full drift scans can reach exactly 1.0)
    world = (scans[0][:, :3].astype(np.float64) @ TRUTH[0][:, :3].T) + TRUTH[0][:, 3]
    half = np.ascontiguousarray(scans[0][world[:, 0] < 0.0])
    with capi.VoxelMap(LEAF, 1 << 18) as vmap, capi.Odometry(vmap, TRUTH[0], min_fitness=1.0, max_correspondence_distance=DMAX) as odo:
        _scan(ctxs[0], half)
        odo.step(ctxs[0])
        first = _map_state(vmap)
        for k in range(1, 4):
            _scan(ctxs[k % 2], scans[k])
            odo.step(ctxs[k % 2], DELTAS[k])
        t = odo.trajectory()
        _assert_same_map(_map_state(vmap), first)
    assert t["accepted"].tolist() == [1, 0, 0, 0]
    assert (t["fitness"][1:] < 1.0).all() and (t["n_correspondences"][1:] >= 6).all()
    assert all(np.array_equal(_bits(t["poses"][k]), _bits(t["guesses"][k])) for k in range(4))


# Straight bore (C0 at the settings of tests/test_oracle_register.py::test_straight_bore_reports_and_keeps_unobservable_
# directions, degeneracy_ratio 1e-2): translation along the axis and the roll about it are unobservable and keep the guess.
# The sensor advances 0.2 m per step with small lateral and yaw offsets.  The restatement (register_map_oracle.icp over
# oracle.map_insert, 400k points, bore 16 m long) measured, after 5 steps: with the truth increments as delta34 an
# along-axis error below 0.1 mm; without a prior 1.0004 m (the 1.0 m travelled); lateral errors <= 0.64 mm and yaw
# <= 2.2e-4 rad in both runs.
BORE_N, BORE_HL, BORE_RATIO, BORE_STEPS = 400_000, 8.0, 1e-2, 6


def _bore_truth(k):
    return synth.pose34((0.0, 0.0, 0.004 * np.sin(1.3 * k)), (0.2 * k, 0.03 * np.cos(0.9 * k) - 0.03, 0.0))


def test_unobservable_directions_take_the_motion_prior():
    truth = [_bore_truth(k) for k in range(BORE_STEPS)]
    pts = [synth.second_scan(synth.straight_cylinder, truth[k], seed=70 + k, n=BORE_N, half_length=BORE_HL) for k in range(BORE_STEPS)]
    ctx = _ctx(BORE_N, neighborRadius=0.1, voxelGridLeafSize=LEAF)
    err = {}
    try:
        for prior in (True, False):
            with capi.VoxelMap(LEAF, 1 << 18) as vmap, capi.Odometry(vmap, truth[0], max_correspondence_distance=DMAX,
                                                                     degeneracy_ratio=BORE_RATIO) as odo:
                for k in range(BORE_STEPS):
                    _scan(ctx, pts[k])
                    odo.step(ctx, _increment(truth[k - 1], truth[k]) if prior and k else None)
                t = odo.trajectory()
            assert t["accepted"].all() and (t["n_degenerate"][1:] == 2).all() and (t["converged"][1:] == 1).all()
            err[prior] = [(t["poses"][k].astype(np.float64) - truth[k], t["poses"][k][:, :3].astype(np.float64) @ truth[k][:, :3].T)
                          for k in range(BORE_STEPS)]
    finally:
        ctx.close()
    travelled = truth[-1][0, 3] - truth[0][0, 3]
    assert abs(err[True][-1][0][0, 3]) <= 5e-3                               # along the axis: the prior
    assert abs(abs(err[False][-1][0][0, 3]) - travelled) <= 0.05 * travelled  # no prior: the guess, i.e. standing still
    for prior in (True, False):
        for e, dR in err[prior][1:]:
            assert abs(e[1, 3]) <= 3e-3 and abs(e[2, 3]) <= 3e-3 and abs(dR[1, 0]) <= 1e-3   # observable: corrected


def test_register_first_on_a_reloaded_map(ctxs, scans, tmp_path):
    path = str(tmp_path / "four.gmm")
    with capi.VoxelMap(LEAF, 1 << 18) as vmap:
        for k in range(4):
            _scan(ctxs[0], scans[k])
            vmap.insert(ctxs[0], TRUTH[k])
        vmap.save(path)
    init = (_h(TRUTH[4]) @ _h(_pose((0.5, -0.5, 1.0), (0.05, -0.03, 0.02))))[:3]
    ctx = ctxs[1]
    _scan(ctx, scans[4])
    with capi.VoxelMap.load(path) as ref_map:
        ref = ctx.register_map(ref_map, init, max_planarity=RATIO, max_correspondence_distance=DMAX)
        ref_corr = ctx.download_map_correspondences()
    with capi.VoxelMap.load(path) as vmap, capi.Odometry(vmap, init, register_first=1, max_correspondence_distance=DMAX) as odo:
        odo.step(ctx)
        t = odo.trajectory()
        got = ctx.registration()
        corr = ctx.download_map_correspondences()
    assert bytes(got["_struct"]) == bytes(ref["_struct"])
    assert np.array_equal(corr[0], ref_corr[0]) and np.array_equal(_bits(corr[1]), _bits(ref_corr[1]))
    assert t["registered"][0] == 1 and t["accepted"][0] == 1
    assert np.array_equal(_bits(t["poses"][0]), _bits(ref["pose"])) and np.array_equal(_bits(t["guesses"][0]), _bits(np.float32(init)))
    assert (t["iterations"][0], t["n_correspondences"][0], t["converged"][0]) == (ref["iterations"], ref["n_correspondences"], ref["converged"])
    assert t["fitness"][0] == np.float32(ref["fitness"]) and t["rmse"][0] == np.float32(ref["rmse"])


def test_steps_do_not_wait_for_the_device(runs, ctxs, scans):
    import torch

    stream = torch.cuda.Stream()
    with capi.VoxelMap(LEAF, 1000) as empty:   # first registrations allocate the contexts' buffers
        for c in ctxs:
            _scan(c, scans[0])
            c.register_map(empty)
    pending = []

    def before_step(ctx, k):
        if k is None:
            pending.append(stream.query())
            return
        with torch.cuda.stream(stream):
            torch.cuda._sleep(200_000_000)

    for c in ctxs:
        c.set_stream(stream.cuda_stream)
    try:
        traj, state = _odometry(ctxs, scans, False, before_step)
    finally:
        for c in ctxs:
            c.set_stream(None)
    assert not any(pending), pending
    ref, ref_state = runs["odo", False]
    assert np.array_equal(_bits(traj["poses"]), _bits(ref["poses"])) and np.array_equal(_bits(traj["guesses"]), _bits(ref["guesses"]))
    _assert_same_map(state, ref_state)


@pytest.mark.parametrize("iters", [1, 30])
def test_launch_count(ctxs, scans, iters):
    ctx = ctxs[0]
    _scan(ctx, scans[0])
    with capi.VoxelMap(LEAF, 1 << 18) as vmap:
        for register_first, expect in ((0, 3), (1, iters + 4)):
            with capi.Odometry(vmap, TRUTH[0], register_first=register_first, max_iterations=iters) as odo:
                ctx.synchronize()
                ctx.reset_launch_count()
                odo.step(ctx)
                assert ctx.launch_count == expect, register_first
                ctx.reset_launch_count()
                odo.step(ctx)
                assert ctx.launch_count == iters + 4
        with capi.Odometry(vmap, TRUTH[0]) as odo, _ctx(1000, **C1) as empty:
            _scan(empty, np.zeros((0, 4), np.float32))
            odo.step(ctx)
            empty.reset_launch_count()
            odo.step(empty)                                     # an empty scan still launches its insert
            assert empty.launch_count == 30 + 4 and odo.trajectory()["accepted"][1] == 0
        ctx.synchronize()


def test_argument_stage_and_capacity_rules(ctxs, scans):
    lib = capi._lib()
    assert C.sizeof(capi.gm_odometry_params) == 112 and capi.gm_odometry_params.max_steps.offset == 108
    assert capi.gm_odometry_params.max_planarity.offset == 88 and capi.gm_odometry_params.register_first.offset == 104
    assert C.sizeof(capi.gm_odometry_record) == 136 and capi.gm_odometry_record.accepted.offset == 96
    assert capi.gm_odometry_record.rmse.offset == 124 and capi.gm_odometry_record.pad_.offset == 132
    p = capi.odometry_params()
    assert (p.max_planarity, p.min_fitness, p.register_first, p.max_steps) == (0.1, 0.5, 0, 4096)
    with capi.VoxelMap(LEAF, 1 << 18) as vmap:
        h = C.c_void_p()
        for bad in (dict(min_fitness=-0.1), dict(min_fitness=1.01), dict(min_fitness=float("nan")), dict(register_first=2),
                    dict(max_steps=0), dict(max_planarity=0.0), dict(max_iterations=0), dict(max_correspondence_distance=0.0),
                    dict(degeneracy_ratio=1.0)):
            q = capi.odometry_params(**bad)
            assert lib.gm_odometry_create(vmap._h, C.byref(q), C.byref(h)) == capi.GM_ERR_INVALID_ARG, bad
        q = capi.odometry_params()
        q.icp.init_pose34[3] = float("nan")
        assert lib.gm_odometry_create(vmap._h, C.byref(q), C.byref(h)) == capi.GM_ERR_INVALID_ARG
        assert lib.gm_odometry_create(None, C.byref(capi.odometry_params()), C.byref(h)) == capi.GM_ERR_INVALID_ARG
        with capi.Odometry(vmap, TRUTH[0], max_steps=2) as odo, _ctx(20_000, **C1) as c:
            eye = np.ascontiguousarray(np.eye(3, 4, dtype=np.float32))
            c.upload_scan(scans[0][:20_000])
            c.crop()
            c.normals()
            c.reset_launch_count()
            assert lib.gm_odometry_step(odo._h, c._h, None) == capi.GM_ERR_STAGE_ORDER    # no voxels
            c.voxel()
            c.reset_launch_count()
            assert lib.gm_odometry_step(odo._h, c._h, capi._ptr(eye)) == capi.GM_ERR_INVALID_ARG  # delta34 at step 0
            assert odo.steps == 0 and c.launch_count == 0
            odo.step(c)
            bad = eye.copy()
            bad[0] = np.inf
            assert lib.gm_odometry_step(odo._h, c._h, capi._ptr(bad)) == capi.GM_ERR_INVALID_ARG
            odo.step(c, eye)
            c.reset_launch_count()
            assert lib.gm_odometry_step(odo._h, c._h, None) == capi.GM_ERR_CAPACITY
            assert odo.steps == 2 and c.launch_count == 0
            n = C.c_int32(0)
            recs = (capi.gm_odometry_record * 1)()
            assert lib.gm_odometry_get(odo._h, recs, 1, C.byref(n)) == capi.GM_ERR_CAPACITY and n.value == 2
            assert lib.gm_odometry_get(odo._h, None, 0, C.byref(n)) == capi.GM_OK and n.value == 2
            assert len(odo.records()) == 2
