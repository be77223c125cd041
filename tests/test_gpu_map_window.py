"""gm_map_evict, gm_map_merge and the odometry window on the B200.

Map part: a map built from a real scan is split by the window exactly as tests/map_window_oracle.py restates it (local =
the kept voxels, archive = the rest, statistics), merging back gives the original file byte for byte, a pre-filled
archive receives the oracle's file merge, planes of the kept voxels are those of tests/register_map_oracle.py, the edge
cases, fifty evictions, a small map that only fits with a window, the argument rules, the launch count and no host wait.
Odometry part: a 60-scan run along a curved tunnel, every step equal to the host loop of public calls it replaces, a
window at twice the sizing rule leaving the trajectory bit for bit and the merged map byte for byte as without it, a
local map too small for the run, the launch contract and determinism."""
import ctypes as C
import math

import numpy as np
import pytest

import map_window_oracle as W
import odometry_oracle as OD
import register_map_oracle as RM
from geometric_mapping_b200 import capi, synth

pytestmark = pytest.mark.gpu

LEAF, RATIO, DMAX = 0.1, 0.1, 0.5
E = 3                                     # GM_MAP_EVICT_LAUNCHES
N_MAP = 400_000
C1 = dict(neighborRadius=0.05, voxelGridLeafSize=LEAF)
P0 = synth.pose34((0.0, 0.0, 0.0), (0.0, 0.0, 0.0))
P1 = synth.pose34((0.0, 0.0, 0.12), (1.3, 0.4, -0.1))
P2 = synth.pose34((0.0, 0.05, -0.2), (-2.2, -0.3, 0.2))
FAR = synth.pose34((0.0, 0.0, 0.0), (5.0e5, 0.0, 0.0))   # every point's cell outside the key range: out_of_range


def _ctx(n, **kw):
    return capi.Context(capi.default_params(**kw), max_points=max(n, 1), max_hypotheses=16)


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _file(vmap, tmp_path, name):
    p = str(tmp_path / name)
    vmap.save(p)
    return open(p, "rb").read()


def _read(vmap, tmp_path, name):
    return W.read_gmm1(_file(vmap, tmp_path, name))


def _assert_download(vmap, m):
    d = vmap.download()
    assert np.array_equal(d["ijk"], W.unpack(m["keys"]).astype(np.int32))
    assert np.array_equal(d["counts"], m["counts"])
    assert np.array_equal(_bits(d["centroids"][:, :3]), _bits(W.centroids(m)))


@pytest.fixture(scope="module")
def mctx():
    c = _ctx(N_MAP, **C1)
    c.upload_scan(synth.curved_tunnel(N_MAP, seed=2))
    c.crop()
    c.normals()
    yield c
    c.close()


def _build(ctx, capacity=1 << 18, poses=(P0, P1)):
    m = capi.VoxelMap(LEAF, capacity)
    for P in poses:
        m.insert(ctx, P)
    m.insert(ctx, FAR)
    return m


@pytest.fixture(scope="module")
def ref(mctx, tmp_path_factory):
    with _build(mctx) as m:
        d = tmp_path_factory.mktemp("ref")
        b = _file(m, d, "ref.gmm")
        st = m.stats()
    assert st[2] > 0 and not st[3]
    return {"bytes": b, "map": W.read_gmm1(b), "stats": st}


CASES = [((0.37, -0.05, 0.2), 30), ((-2.0, 1.0, -1.0), 25), ((3.04, -0.05, -1.45), 31)]


@pytest.mark.parametrize("center,half", CASES)
def test_evict_keeps_the_window_and_archives_the_rest(mctx, ref, tmp_path, center, half):
    kept, gone = W.evict(ref["map"], center, half)
    assert kept["keys"].size and gone["keys"].size
    with _build(mctx) as local, capi.VoxelMap(LEAF, 1 << 18) as arch:
        local.evict(mctx, center, half, arch)
        _assert_download(local, kept)
        _assert_download(arch, gone)
        nv, npts, oor, full = local.stats()
        assert nv == kept["keys"].size and npts == int(kept["counts"].sum())
        assert ref["stats"][0] - nv == gone["keys"].size and ref["stats"][1] - npts == int(gone["counts"].sum())
        assert oor == ref["stats"][2] and not full                 # out_of_range and overflow stay as they were
        assert arch.stats() == (gone["keys"].size, int(gone["counts"].sum()), 0, False)
        assert W.write_gmm1(kept) == _file(local, tmp_path, "local.gmm")
        # merge back: byte for byte the map that was never evicted
        assert arch.merge(local) is False
        assert _file(arch, tmp_path, "whole.gmm") == ref["bytes"]
        assert _file(local, tmp_path, "local2.gmm") == W.write_gmm1(kept)   # src unchanged


def test_prefilled_archive_receives_the_file_merge(mctx, ref, tmp_path):
    center, half = CASES[0]
    kept, gone = W.evict(ref["map"], center, half)
    with _build(mctx) as local, capi.VoxelMap(LEAF, 1 << 18) as arch:
        arch.insert(mctx, P2)
        before = _read(arch, tmp_path, "before.gmm")
        shared = np.intersect1d(before["keys"], gone["keys"]).size
        assert 0 < shared < gone["keys"].size
        local.evict(mctx, center, half, arch)
        assert _file(arch, tmp_path, "after.gmm") == W.write_gmm1(W.merge(before, gone))
        assert _file(local, tmp_path, "local.gmm") == W.write_gmm1(kept)


def test_planes_after_eviction_are_the_kept_voxels_planes(mctx, ref):
    center, half = CASES[1]
    kept, _ = W.evict(ref["map"], center, half)
    with _build(mctx) as local:
        local.planes(RATIO)                                        # plane tables of the full map first
        local.evict(mctx, center, half)
        got = local.planes(RATIO)
    want = RM.planes_xyzw(RM.planes(W.unpack(kept["keys"]), W.centroids(kept), RATIO))
    has = got[:, 3] == 1.0
    assert has.sum() > 100 and np.array_equal(got[:, 3], want[:, 3])
    assert np.array_equal(_bits(got[has, :3]), _bits(want[has, :3])) and np.isnan(got[~has, :3]).all()


def test_edge_cases(mctx, ref, tmp_path):
    m = ref["map"]
    with _build(mctx) as local, capi.VoxelMap(LEAF, 1 << 18) as arch:
        local.evict(mctx, (0.0, 0.0, 0.0), 2**31 - 1, arch)          # a window larger than the key range
        assert _file(local, tmp_path, "a.gmm") == ref["bytes"] and arch.stats()[:2] == (0, 0)
        assert local.stats() == ref["stats"]
        i = len(m["keys"]) // 3
        cell = W.unpack(m["keys"][i:i + 1])[0]
        c = ((cell + 0.5) * LEAF).astype(np.float32)
        assert W.center_cell(c, LEAF).tolist() == cell.tolist()
        local.evict(mctx, c, 0, arch)                                # half_cells 0: the centre cell alone
        d = local.download()
        assert d["ijk"].tolist() == [cell.tolist()]
        arch.merge(local)
        assert _file(arch, tmp_path, "b.gmm") == ref["bytes"]
    kept, _ = W.evict(m, CASES[2][0], CASES[2][1])
    with _build(mctx) as local:                                      # archive NULL: dropped
        local.evict(mctx, *CASES[2])
        assert _file(local, tmp_path, "c.gmm") == W.write_gmm1(kept)
    # inserting after an eviction re-creates voxels: local + archive = the map given every insert
    with _build(mctx) as local, capi.VoxelMap(LEAF, 1 << 18) as arch, _build(mctx, poses=(P0, P1, P2)) as whole:
        local.evict(mctx, *CASES[0], arch)
        local.insert(mctx, P2)
        local.evict(mctx, *CASES[1], arch)
        local.insert(mctx, P0)
        whole.insert(mctx, P0)
        arch.merge(local)
        assert _file(arch, tmp_path, "d.gmm") == _file(whole, tmp_path, "e.gmm")


def test_many_evictions_leave_no_residue(mctx, ref, tmp_path):
    with _build(mctx) as local, capi.VoxelMap(LEAF, 1 << 18) as arch:
        for i in range(50):
            local.evict(mctx, (-4.0 + 0.17 * i, 0.3 * math.sin(i), 0.1 * math.cos(i)), 12 + i % 7, arch)
        nv, npts, _, full = local.stats()
        d = local.download()
        assert nv == d["ijk"].shape[0] and npts == int(d["counts"].sum()) and not full
        arch.merge(local)
        assert _file(arch, tmp_path, "a.gmm") == ref["bytes"]
        local.insert(mctx, P2)                                        # the rebuilt table takes new voxels
        nv, _, _, full = local.stats()
        assert nv == local.download()["ijk"].shape[0] and not full


def test_a_small_map_fits_with_a_window(mctx):
    poses = [synth.pose34((0.0, 0.0, 0.0), (3.0 * k, 0.0, 0.0)) for k in range(12)]
    half = 30

    def run(vmap, window):
        peak = 0
        for P in poses:
            vmap.insert(mctx, P)
            peak = max(peak, vmap.stats()[0])
            if window:
                vmap.evict(mctx, P[:, 3], half)
        return peak, vmap.stats()

    with capi.VoxelMap(LEAF, 1 << 19) as big:
        total = run(big, False)[1][0]
    with capi.VoxelMap(LEAF, 1 << 19) as big:
        peak, _ = run(big, True)
    slots = 1 << (int(total - 1).bit_length() - 1)                  # a power of two below the run's voxel count
    assert peak < 0.8 * slots, (peak, slots, total)
    with capi.VoxelMap(LEAF, slots // 2) as small:
        assert run(small, False)[1][3]                               # full without a window
    with capi.VoxelMap(LEAF, slots // 2) as small:
        p, st = run(small, True)
        assert not st[3] and p == peak


def test_argument_rules_launches_and_no_host_wait(mctx, ref, tmp_path):
    import torch

    lib = capi._lib()
    with _build(mctx) as local, capi.VoxelMap(LEAF, 1 << 10) as arch, capi.VoxelMap(0.1000001, 1 << 10) as other:
        ok = np.zeros(3, np.float32)

        def ev(c, half, a=arch, m=local, ctx=mctx):
            c = np.ascontiguousarray(np.asarray(c, np.float32))
            return lib.gm_map_evict(m._h if m else None, ctx._h if ctx else None, a._h if a else None, capi._ptr(c), half)

        mctx.synchronize()
        mctx.reset_launch_count()
        for c, half, a in ((ok, -1, arch), ((np.nan, 0, 0), 5, arch), ((0, np.inf, 0), 5, arch), ((0, 0, -np.inf), 5, None),
                           ((2.0e5, 0, 0), 5, arch), ((0, -104857.7, 0), 5, arch), (ok, 5, local), (ok, 5, other)):
            assert ev(c, half, a) == capi.GM_ERR_INVALID_ARG, (c, half)
        assert ev(ok, 5, ctx=None) == capi.GM_ERR_INVALID_ARG and ev(ok, 5, m=None) == capi.GM_ERR_INVALID_ARG
        assert lib.gm_map_evict(local._h, mctx._h, None, None, 5) == capi.GM_ERR_INVALID_ARG
        assert mctx.launch_count == 0
        assert local.stats() == ref["stats"]
        assert lib.gm_map_merge(local._h, local._h) == capi.GM_ERR_INVALID_ARG
        assert lib.gm_map_merge(local._h, other._h) == capi.GM_ERR_INVALID_ARG
        assert lib.gm_map_merge(None, local._h) == capi.GM_ERR_INVALID_ARG
        # E launches whether or not anything is evicted
        local.evict(mctx, ok, 2**31 - 1)
        assert mctx.launch_count == E
        local.evict(mctx, ok, 20, arch)                               # a small archive overflows: GM_ERR_CAPACITY
        assert mctx.launch_count == 2 * E
        assert arch.stats()[3] and lib.gm_map_stats(arch._h, None, None, None) == capi.GM_ERR_CAPACITY
        assert not local.stats()[3]
        if torch.cuda.device_count() > 1:                             # a context on another device
            with torch.cuda.device(1):
                c2 = _ctx(1000, **C1)
            with c2:
                assert ev(ok, 5, ctx=c2) == capi.GM_ERR_INVALID_ARG
        with capi.VoxelMap(LEAF, 1 << 10) as a2, capi.Odometry(arch) as odo:
            for half, a in ((-1, None), (5, arch), (5, other)):
                assert lib.gm_odometry_set_window(odo._h, half, a._h if a else None) == capi.GM_ERR_INVALID_ARG
            assert lib.gm_odometry_set_window(None, 5, None) == capi.GM_ERR_INVALID_ARG
            odo.set_window(5, a2)
            odo.set_window(0)
    # the call returns while the stream is still busy
    stream = torch.cuda.Stream()
    center, half = CASES[0]
    kept, gone = W.evict(ref["map"], center, half)
    with _build(mctx) as local, capi.VoxelMap(LEAF, 1 << 18) as arch:
        local.evict(mctx, center, 2**31 - 1, arch)                   # the first eviction allocates the map's scratch
        mctx.synchronize()
        mctx.set_stream(stream.cuda_stream)
        try:
            with torch.cuda.stream(stream):
                torch.cuda._sleep(200_000_000)
            local.evict(mctx, center, half, arch)
            pending = stream.query()
        finally:
            mctx.set_stream(None)
        assert not pending
        assert _file(local, tmp_path, "l.gmm") == W.write_gmm1(kept) and _file(arch, tmp_path, "a.gmm") == W.write_gmm1(gone)


# ---- odometry with a window, along a curved tunnel ------------------------------------------------------------------
# 60 scans 1 m apart along the arc of synth.curved_tunnel (arc radius 50 m: the run turns by 1.2 rad and stays within
# 60 m of the origin), each a 14 m section seen from its pose with small lateral and yaw offsets.  The along-axis direction is
# weak, so the steps take the truth increments as delta34 and degeneracy_ratio as the straight-bore test of
# tests/test_gpu_odometry.py.  Sizing rule with B = 5 (boxFilterBound), s = 1.5 m, d_max = 0.5 m, leaf 0.1 m.
SEQ, N_SCAN, ARC_R, STEP = 60, 240_000, 50.0, 1.0
ODO = dict(neighborRadius=0.1, voxelGridLeafSize=LEAF)
BORE_RATIO, MIN_FIT = 1e-2, 0.5
RULE = math.floor((math.sqrt(3.0) * 5.0 + 1.5 + DMAX) / LEAF) + 2


def _truth(k):
    s = STEP * k
    phi = s / ARC_R
    return synth.pose34((0.0, 0.0, phi + 0.004 * math.sin(1.3 * k)),
                        (ARC_R * math.sin(phi) - 0.03 * math.sin(phi) * math.cos(0.9 * k),
                         ARC_R * (1.0 - math.cos(phi)) + 0.03 * math.cos(phi) * math.cos(0.9 * k), 0.0))


TRUTH = [_truth(k) for k in range(SEQ)]


def _h(P):
    return np.vstack([np.asarray(P, np.float64)[:3, :4], [0.0, 0.0, 0.0, 1.0]])


DELTAS = [None] + [np.linalg.solve(_h(TRUTH[k - 1]), _h(TRUTH[k]))[:3].astype(np.float32) for k in range(1, SEQ)]
ICP = dict(max_planarity=RATIO, max_correspondence_distance=DMAX, degeneracy_ratio=BORE_RATIO, min_fitness=MIN_FIT)


@pytest.fixture(scope="module")
def tunnel():
    scans = [synth.view_from(synth.curved_tunnel(N_SCAN, seed=300 + k, arc_length=14.0, advance=STEP * k, outlier_frac=0.0),
                             TRUTH[k]) for k in range(SEQ)]
    cs = [_ctx(N_SCAN, **ODO), _ctx(N_SCAN, **ODO)]
    yield scans, cs
    for c in cs:
        c.close()


def _scan(ctx, pts):
    ctx.upload_scan(pts)
    ctx.crop()
    ctx.normals()
    ctx.voxel()


def _odometry(tunnel, tmp_path, name, half=0, local_capacity=1 << 18):
    scans, cs = tunnel
    out = {}
    with capi.VoxelMap(LEAF, local_capacity) as vmap, capi.VoxelMap(LEAF, 1 << 18) as arch:
        with capi.Odometry(vmap, TRUTH[0], **ICP) as odo:
            for k in range(SEQ):
                if half and k == 0:
                    odo.set_window(half, arch)
                _scan(cs[k % 2], scans[k])
                odo.step(cs[k % 2], DELTAS[k])
            out["traj"] = odo.trajectory()
        out["local_stats"], out["archive_stats"] = vmap.stats(), arch.stats()
        out["local"] = _file(vmap, tmp_path, name + "_local.gmm")
        out["archive"] = _file(arch, tmp_path, name + "_archive.gmm")
        if not out["local_stats"][3]:
            arch.merge(vmap)
            out["merged"] = _file(arch, tmp_path, name + "_merged.gmm")
    return out


@pytest.fixture(scope="module")
def runs(tunnel, tmp_path_factory):
    d = tmp_path_factory.mktemp("odo")
    r = {"none": _odometry(tunnel, d, "none"), "wide": _odometry(tunnel, d, "wide", 2 * RULE)}
    # a local map of fewer slots than the run's voxels.  Without a window it fills up; that is shown by inserting the scans
    # at the run's poses (registering against a full table would probe all of it for every absent cell)
    r["small_slots"] = 1 << (int(r["none"]["local_stats"][0] - 1).bit_length() - 1)
    scans, cs = tunnel
    with capi.VoxelMap(LEAF, r["small_slots"] // 2) as small:
        for k in range(SEQ):
            _scan(cs[0], scans[k])
            small.insert(cs[0], r["none"]["traj"]["poses"][k])
        r["small_none_full"] = small.stats()[3]
    r["small_wide"] = _odometry(tunnel, d, "small_wide", 2 * RULE, r["small_slots"] // 2)
    return r


def _same_traj(a, b):
    for key in a:
        x, y = a[key], b[key]
        assert np.array_equal(x.view(np.uint32), y.view(np.uint32)) if x.dtype == np.float32 else np.array_equal(x, y), key


def test_the_tunnel_run_is_accurate_and_accepted(runs):
    t = runs["none"]["traj"]
    assert t["accepted"].all() and (t["fitness"][1:] > 0.7).all()
    for k in (SEQ // 2, SEQ - 1):                                          # within 0.5 % of the distance travelled
        err = np.linalg.norm(t["poses"][k][:, 3].astype(np.float64) - TRUTH[k][:, 3])
        assert err < 0.005 * STEP * k, (k, err)
    assert np.linalg.norm(TRUTH[-1][:, 3]) < 100.0


def test_host_loop_equals_the_windowed_odometry(tunnel, tmp_path):
    """Every step bit for bit: register_map from the restated guess, the gate, insert, evict at the recorded pose."""
    scans, cs = tunnel
    half = RULE
    got = _odometry(tunnel, tmp_path, "rule", half)
    poses, rows = [], []
    with capi.VoxelMap(LEAF, 1 << 18) as vmap, capi.VoxelMap(LEAF, 1 << 18) as arch:
        for k in range(SEQ):
            ctx = cs[k % 2]
            _scan(ctx, scans[k])
            G = OD.guess(k, TRUTH[0], poses, DELTAS[k])
            if k == 0:
                P, ok, g = G, True, None
            else:
                g = ctx.register_map(vmap, G, max_planarity=RATIO, max_correspondence_distance=DMAX, degeneracy_ratio=BORE_RATIO)
                ok = OD.accepted(g["fitness"], g["n_correspondences"], MIN_FIT)
                P = np.asarray(g["pose"], np.float32) if ok else G
            if ok:
                vmap.insert(ctx, P)
            vmap.evict(ctx, np.asarray(P, np.float32)[:, 3], half, arch)
            poses.append(np.asarray(P, np.float32))
            rows.append((P, G, int(ok), g))
        local, archive = _file(vmap, tmp_path, "host_local.gmm"), _file(arch, tmp_path, "host_archive.gmm")
    t = got["traj"]
    for k, (P, G, ok, g) in enumerate(rows):
        assert np.array_equal(_bits(t["poses"][k]), _bits(P)) and np.array_equal(_bits(t["guesses"][k]), _bits(G)), k
        assert t["accepted"][k] == ok, k
        if g is not None:
            assert (t["iterations"][k], t["n_correspondences"][k], t["converged"][k]) == (g["iterations"], g["n_correspondences"], g["converged"]), k
    assert got["local"] == local and got["archive"] == archive
    assert got["archive_stats"][0] > 0                                     # it evicted


def test_a_wide_window_changes_nothing(runs):
    none, wide = runs["none"], runs["wide"]
    _same_traj(wide["traj"], none["traj"])
    assert wide["archive_stats"][0] > 0 and wide["local_stats"][0] < none["local_stats"][0]
    assert wide["merged"] == none["local"]


def test_a_small_local_map_runs_with_the_window(runs):
    assert runs["small_none_full"]                                          # without a window: GM_ERR_CAPACITY
    sw = runs["small_wide"]
    assert sw["local_stats"][0] < 0.85 * runs["small_slots"]
    assert not sw["local_stats"][3] and not sw["archive_stats"][3]
    _same_traj(sw["traj"], runs["wide"]["traj"])
    assert sw["merged"] == runs["none"]["local"]


def test_window_launches_and_determinism(runs, tunnel, tmp_path):
    again = _odometry(tunnel, tmp_path, "again", 2 * RULE)
    _same_traj(again["traj"], runs["wide"]["traj"])
    assert again["local"] == runs["wide"]["local"] and again["archive"] == runs["wide"]["archive"]
    scans, cs = tunnel
    ctx = cs[0]
    iters = 30
    with capi.VoxelMap(LEAF, 1 << 18) as vmap, capi.VoxelMap(LEAF, 1 << 18) as arch, \
            capi.Odometry(vmap, TRUTH[0], max_iterations=iters, **ICP) as odo:
        odo.set_window(RULE, arch)
        for k, expect in ((0, 3 + E), (1, iters + 4 + E)):
            _scan(ctx, scans[k])
            ctx.synchronize()
            ctx.reset_launch_count()
            odo.step(ctx, DELTAS[k])
            assert ctx.launch_count == expect, k
        odo.set_window(0)
        _scan(ctx, scans[2])
        ctx.synchronize()
        ctx.reset_launch_count()
        odo.step(ctx, DELTAS[2])
        assert ctx.launch_count == iters + 4
