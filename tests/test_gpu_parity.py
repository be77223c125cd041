"""GPU parity: the CUDA path (through the C-ABI, via ctypes) against the CPU oracle on the same
seeded inputs.  Integer / index outputs are compared bit-exactly; floating-point outputs within
the tolerance written next to each check (north_star: coefficients within 1e-4 relative).
"""
import numpy as np
import pytest

from geometric_mapping_b200 import capi, synth
from oracle import oracle as O

pytestmark = pytest.mark.gpu

TAU = 0.05


def _angle(a, b):
    a = a / np.linalg.norm(a, axis=-1, keepdims=True)
    b = b / np.linalg.norm(b, axis=-1, keepdims=True)
    return np.arccos(np.clip(np.abs((a * b).sum(-1)), -1.0, 1.0))


def _ctx(n, **kw):
    return capi.Context(capi.default_params(**kw), max_points=max(n, 1), max_hypotheses=4096)


def _centroids_match(got, ref):
    """VoxelGrid centroids: bit-exact against the order-independent fixed-point restatement (what the CUDA path
    defines: sums of llrint(coord * 2^20), exact to 1e-6 m), and as close to pcl::VoxelGrid's float accumulation
    as that accumulation is to the true mean: a sequential float32 sum of n values carries up to n * 2^-24 relative
    error (and PCL's summation order is itself unspecified: unstable std::sort)."""
    assert np.array_equal(got.view(np.uint32), ref["centroids_fx"].view(np.uint32))
    n = ref["voxel_counts"].astype(np.float64)[:, None]
    tol = 1e-6 + n * 2.0 ** -24 * np.maximum(np.abs(ref["centroids"][:, :3]), 1.0)
    assert (np.abs(got[:, :3].astype(np.float64) - ref["centroids"][:, :3]) <= tol).all()


def _scan_with_junk(n=60_000, seed=11):
    pts = synth.curved_tunnel(n, seed=seed, outlier_frac=0.02)
    g = np.random.Generator(np.random.Philox(seed + 1))
    # points outside the crop box, exactly on its faces, and NaN / inf coordinates
    pts[g.choice(n, 500, replace=False), 0] += 20.0
    pts[7] = [5.0, -5.0, 5.0, 1.0]
    pts[8] = [np.nextafter(np.float32(5.0), np.float32(6.0)), 0.0, 0.0, 1.0]
    pts[9] = [np.nan, 0.0, 0.0, 1.0]
    pts[10] = [0.0, np.inf, 0.0, 1.0]
    pts[11] = [0.0, 0.0, -np.inf, 1.0]
    return pts


# ---- a1 crop -------------------------------------------------------------------------------
@pytest.mark.parametrize("is_dense", [1, 0])
def test_crop_bit_exact(is_dense):
    pts = _scan_with_junk()
    ref, _ = O.crop(pts, 5.0, bool(is_dense))
    with _ctx(len(pts), is_dense=is_dense) as ctx:
        ctx.upload_scan(pts)
        ctx.crop()
        out = ctx.download_cloud(0)
    assert out.shape == ref.shape
    assert np.array_equal(out.view(np.uint32), ref.view(np.uint32))  # order and bits, NaN included


def test_crop_empty_and_tiny():
    with _ctx(16) as ctx:
        ctx.upload_scan(np.zeros((0, 4), np.float32))
        ctx.crop()
        assert ctx.counts().n_cropped == 0
        one = np.array([[1, 2, 3, 1]], np.float32)
        ctx.upload_scan(one)
        ctx.crop()
        assert np.array_equal(ctx.download_cloud(0), one)
        far = np.array([[100, 0, 0, 1]], np.float32)
        ctx.upload_scan(far)
        ctx.crop()
        assert ctx.counts().n_cropped == 0


# ---- a2/a3 normals + compaction ------------------------------------------------------------
@pytest.mark.parametrize("radius", [0.15, 0.3])
def test_normals_parity(radius):
    pts = _scan_with_junk(40_000)
    cropped, _ = O.crop(pts, 5.0, True)
    ref, ref_cnt, truth = O.normals(cropped, radius, mode=0, order=0, truth=True)
    with _ctx(len(pts), neighborRadius=radius) as ctx:
        ctx.upload_scan(pts)
        ctx.crop()
        ctx.normals()
        got = ctx.download_normals(0)
        cnt = ctx.download_neighbor_counts()
        vmap = ctx.download_valid_map()
        cloud_c = ctx.download_cloud(1)
        normals_c = ctx.download_normals(1)
        assert ctx.counts().device_error == 0
    # neighbour sets: exact (same strict d2 < r2 predicate in unfused float)
    assert np.array_equal(cnt, ref_cnt)
    # NaN pattern and compaction: exact
    ref_nan = ~np.isfinite(ref[:, :3]).all(1)
    assert np.array_equal(~np.isfinite(got[:, :3]).all(1), ref_nan)
    rc, rn, rmap = O.compact(cropped, got)
    assert np.array_equal(vmap, rmap)
    assert np.array_equal(cloud_c.view(np.uint32), rc.view(np.uint32))
    assert np.array_equal(normals_c.view(np.uint32), rn.view(np.uint32))
    # normals / curvature: float, accumulation order differs (PCL sums in distance order) and the
    # single-pass covariance is ill-conditioned, so compare against the double-precision truth:
    # the GPU may not be further from it than the float oracle is, up to a small slack.
    ok = ~ref_nan & (ref_cnt >= 8)
    ang_gpu = _angle(got[ok, :3].astype(np.float64), truth[ok, :3])
    ang_ref = _angle(ref[ok, :3].astype(np.float64), truth[ok, :3])
    # well-conditioned neighbourhoods (curvature not tiny relative to float noise)
    assert np.median(ang_gpu) <= 2.0 * np.median(ang_ref) + 1e-4
    assert np.quantile(ang_gpu, 0.99) <= 2.0 * np.quantile(ang_ref, 0.99) + 2e-3
    ang = _angle(got[ok, :3].astype(np.float64), ref[ok, :3].astype(np.float64))
    assert np.quantile(ang, 0.99) < 2e-2  # rad, GPU vs float oracle
    dc = np.abs(got[ok, 4] - ref[ok, 4])
    assert np.quantile(dc, 0.99) < 5e-3
    # orientation: flipped towards the viewpoint (origin)
    dots = -(cropped[ok, :3] * got[ok, :3]).sum(1)
    assert (dots >= -1e-6).all()
    # pcl::Normal padding
    assert (got[~ref_nan][:, [3, 5, 6, 7]] == 0).all()


def test_normals_small_exact_brute_force():
    pts = synth.straight_cylinder(3000, seed=3, noise=0.005)
    ref, ref_cnt, _ = O.normals(pts, 0.4, mode=1, order=0)
    with _ctx(len(pts), neighborRadius=0.4) as ctx:
        ctx.upload_scan(pts)
        ctx.crop()
        ctx.normals()
        cnt = ctx.download_neighbor_counts()
        got = ctx.download_normals(0)
    assert np.array_equal(cnt, ref_cnt)
    ok = ref_cnt >= 3
    assert np.quantile(_angle(got[ok, :3].astype(np.float64), ref[ok, :3].astype(np.float64)), 0.99) < 1e-2


@pytest.mark.parametrize("bound,radius,box", [
    (5.0, 0.5, None),                         # the launch-file radius: a 20-cell grid, 3 block bits per axis
    (2.6, 2.5, None),                         # radius ~ the whole cloud: 2-3 cells per axis
    (50.0, 0.03, None),                       # crop cube too large for 4-cell blocks of r: the cell grows, still exact
    (5.0, 0.11, ((-5.0, -3.0, -1.7), (5.0, 3.0, 0.2))),    # flat grid box: unequal block bits (Morton + stacked high bits)
    (5.0, 0.11, ((-0.5, -0.5, -0.5), (0.5, 0.5, 0.5))),    # box much smaller than the data: border cells take the rest
    (40.0, 0.2, ((-30.0, -2.0, -2.0), (30.0, 2.0, 2.0))),  # long thin box
])
def test_neighbour_grid_shapes_keep_exact_neighbour_sets(bound, radius, box):
    """Whatever the neighbour grid looks like (cube, flat, tiny, enlarged cells, clamped outliers), the radius
    search returns the exact FLANN neighbour sets: counts bit-exact, 1-NN of the voxel centroids exact, voxel
    grid and compaction unchanged."""
    pts = _scan_with_junk(25_000, seed=88)
    if bound > 10:
        pts = pts.copy()
        pts[::7, 0] *= 5.0                    # stretch part of the cloud along x so that the larger boxes hold data
    cropped, _ = O.crop(pts, bound, True)
    ref, ref_cnt, _ = O.normals(cropped, radius, mode=0, order=0)
    cloud_c_ref, nrm_ref, _ = O.compact(cropped, ref)
    with _ctx(len(pts), boxFilterBound=bound, neighborRadius=radius, voxelGridLeafSize=0.2, nn_index_mode=1) as ctx:
        if box is not None:
            ctx.set_grid_box(box[0], box[1])
        ctx.upload_scan(pts)
        ctx.crop()
        ctx.normals()
        ctx.voxel()
        cnt = ctx.download_neighbor_counts()
        cloud_c = ctx.download_cloud(1)
        vox = ctx.download_voxels()
        cand, nbr = ctx.search_stats()
        assert ctx.counts().device_error == 0
    assert np.array_equal(cnt, ref_cnt)                                        # neighbour counts: bit-exact
    assert np.array_equal(cloud_c.view(np.uint32), cloud_c_ref.view(np.uint32))
    assert nbr == int(ref_cnt.astype(np.int64).sum()) and cand >= nbr
    refv = O.voxel(cloud_c, 0.2)
    assert np.array_equal(vox["keys"], refv["voxel_keys"])
    _centroids_match(vox["centroids"], refv)
    ref_idx, _ = O.nn1(vox["centroids"], cloud_c)
    assert np.array_equal(vox["nn_index"], ref_idx)                            # exact nearest neighbour, ties -> lowest index


def test_normals_isolated_points_become_nan_and_are_dropped():
    pts = np.array([[0, 0, 0, 1], [0.01, 0, 0, 1], [3, 3, 3, 1], [0, 0.01, 0, 1], [0.01, 0.01, 0.002, 1]], np.float32)
    with _ctx(8, neighborRadius=0.05) as ctx:
        ctx.upload_scan(pts)
        ctx.crop()
        ctx.normals()
        cnt = ctx.download_neighbor_counts()
        vmap = ctx.download_valid_map()
        c = ctx.counts()
    assert list(cnt) == [4, 4, 1, 4, 4]
    assert list(vmap) == [0, 1, -1, 2, 3]
    assert c.n_valid == 4


# ---- a4 voxel grid + 1-NN --------------------------------------------------------------------
@pytest.mark.parametrize("leaf,radius", [(0.1, 0.15), (0.5, 0.3), (0.07, 0.25)])
def test_voxel_bit_exact(leaf, radius):
    pts = _scan_with_junk(50_000, seed=21)
    cropped, _ = O.crop(pts, 5.0, True)
    with _ctx(len(pts), neighborRadius=radius, voxelGridLeafSize=leaf) as ctx:
        ctx.upload_scan(pts)
        ctx.crop()
        ctx.normals()
        ctx.voxel()
        cloud_c = ctx.download_cloud(1)
        normals_c = ctx.download_normals(1)
        vmap = ctx.download_valid_map()
        keys, assign, st = ctx.download_voxel_assignment()
        vox = ctx.download_voxels()
        grid6 = ctx.voxel_grid()
        c = ctx.counts()
    ref = O.voxel(cloud_c, leaf)
    assert c.n_voxels == ref["V"] and st == capi.GM_OK
    assert np.array_equal(grid6, ref["grid6"])
    assert np.array_equal(keys, ref["keys"])          # voxel keys: bit-exact
    assert np.array_equal(assign, ref["assign"])      # point -> voxel rank: bit-exact
    assert np.array_equal(vox["keys"], ref["voxel_keys"])
    assert np.array_equal(vox["counts"], ref["voxel_counts"])
    _centroids_match(vox["centroids"], ref)
    # 1-NN over the PRE-compaction cloud (quirk B.3), exact, ties -> lowest index
    finite = np.isfinite(cropped[:, :3]).all(1)
    search = cropped.copy()
    search[~finite, :3] = 1e30  # never the nearest
    ref_idx, _ = O.nn1(vox["centroids"], search)
    assert np.array_equal(vox["nn_index"], ref_idx)
    inr = ref_idx < c.n_valid
    assert np.array_equal(vox["nn_normal"][inr].view(np.uint32), normals_c[ref_idx[inr]].view(np.uint32))
    assert c.nn_out_of_range == int((~inr).sum())


@pytest.mark.parametrize("leaf,bound", [(0.1, 5.0), (0.37, 5.0), (0.05, 3.0)])
def test_voxel_dense_tables_equal_sort_path(leaf, bound):
    """gm_voxel without a sort (dense tables, default when the lattice of the crop box fits) and with the
    radix sort (mode 1) give identical keys, assignments, voxel order, counts and centroids; twice in a row on
    the same context (the tables clean themselves), and through the compression stage."""
    pts = _scan_with_junk(50_000, seed=23)
    out = {}
    with _ctx(len(pts), neighborRadius=0.15, voxelGridLeafSize=leaf, boxFilterBound=bound) as ctx:
        for mode in (0, 1, 0):
            ctx.set_voxel_mode(mode)
            ctx.upload_scan(pts)
            ctx.crop()
            ctx.normals()
            nv = ctx.counts().n_valid
            ctx.upload_scan(pts)
            ctx.process_scan(synth.sample_indices(nv, 128, 3, seed=3), synth.sample_indices(nv, 128, 2, seed=4))
            ctx.compress()
            keys, assign, st = ctx.download_voxel_assignment()
            got = (keys, assign, ctx.download_voxels(), ctx.voxel_grid(), ctx.download_compressed(), ctx.counts())
            assert st == capi.GM_OK and got[5].device_error == 0
            if mode in out:
                prev = out[mode]
                assert np.array_equal(prev[0], got[0]) and prev[4] == got[4]          # second dense run == first
            out[mode] = got
        cloud_c = ctx.download_cloud(1)
    a, b = out[0], out[1]
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and np.array_equal(a[3], b[3])
    for k in ("keys", "counts", "nn_index"):
        assert np.array_equal(a[2][k], b[2][k]), k
    assert np.array_equal(a[2]["centroids"].view(np.uint32), b[2]["centroids"].view(np.uint32))
    assert a[4] == b[4]                                                                   # compressed blob byte-identical
    ref = O.voxel(cloud_c, leaf)
    assert np.array_equal(a[0], ref["keys"]) and np.array_equal(a[1], ref["assign"])
    _centroids_match(a[2]["centroids"], ref)


def test_voxel_dense_tables_grow_on_demand():
    """The dense VoxelGrid tables are (re)allocated when a parameter change needs a larger lattice; the very first
    call after that must already be right (a legacy-stream memset once raced with the ctx's non-blocking stream and
    left zero centroids: found by tools/fuzz_more.py)."""
    pts = synth.curved_tunnel(3000, seed=3, outlier_frac=0.0)
    with _ctx(len(pts), neighborRadius=1.1, voxelGridLeafSize=0.3, boxFilterBound=0.75) as ctx:
        for leaf, bound in ((0.3, 0.75), (0.125, 5.0), (0.05, 5.0), (0.3, 0.75), (0.05, 5.0)):
            ctx.set_params(capi.default_params(neighborRadius=1.1, voxelGridLeafSize=leaf, boxFilterBound=bound))
            for rep in range(2):
                ctx.upload_scan(pts)
                ctx.crop()
                ctx.normals()
                ctx.voxel()
                keys, assign, st = ctx.download_voxel_assignment()
                vox = ctx.download_voxels()
                ref = O.voxel(ctx.download_cloud(1), leaf)
                assert np.array_equal(keys, ref["keys"]) and np.array_equal(assign, ref["assign"]), (leaf, bound, rep)
                assert np.array_equal(vox["counts"], ref["voxel_counts"])
                _centroids_match(vox["centroids"], ref)
        assert ctx.counts().device_error == 0


def test_voxel_fixed_nn_mode_indexes_compacted_cloud():
    pts = _scan_with_junk(30_000, seed=5)
    with _ctx(len(pts), neighborRadius=0.12, voxelGridLeafSize=0.2, nn_index_mode=1) as ctx:
        ctx.upload_scan(pts)
        ctx.crop()
        ctx.normals()
        ctx.voxel()
        cloud_c = ctx.download_cloud(1)
        normals_c = ctx.download_normals(1)
        vox = ctx.download_voxels()
        c = ctx.counts()
    assert c.n_valid < c.n_cropped  # some normals were NaN, so the two modes differ
    ref_idx, _ = O.nn1(vox["centroids"], cloud_c)
    assert np.array_equal(vox["nn_index"], ref_idx)
    assert np.array_equal(vox["nn_normal"].view(np.uint32), normals_c[ref_idx].view(np.uint32))
    assert vox["status"] == capi.GM_OK


def test_voxel_lattice_known_keys_and_overflow_rule():
    # points on a lattice: known keys
    g = np.arange(-2, 3, dtype=np.float32) * 0.25 + 0.01
    xx, yy, zz = np.meshgrid(g, g, g, indexing="ij")
    pts = np.stack([xx.ravel(), yy.ravel(), zz.ravel(), np.ones(xx.size)], 1).astype(np.float32)
    with _ctx(len(pts), voxelGridLeafSize=0.25) as ctx:
        ctx.inject_compacted(pts)
        ctx.voxel()
        keys, assign, st = ctx.download_voxel_assignment()
        vox = ctx.download_voxels(with_nn=False)
    ref = O.voxel(pts, 0.25)
    assert np.array_equal(keys, ref["keys"]) and np.array_equal(assign, ref["assign"])
    assert len(np.unique(keys)) == 125 and ref["V"] == 125
    _centroids_match(vox["centroids"], ref)
    # overflow rule: leaf so small that dx*dy*dz > INT32_MAX -> cloud returned unchanged
    big = synth.straight_cylinder(5000, seed=9)
    with _ctx(len(big), voxelGridLeafSize=0.001) as ctx:
        ctx.inject_compacted(big)
        ctx.voxel()
        vox = ctx.download_voxels(with_nn=False)
        c = ctx.counts()
    ref = O.voxel(big, 0.001)
    assert ref["status"] == 1 and c.voxel_overflow == 1 and vox["status"] == capi.GM_WARN_VOXEL_OVERFLOW
    assert c.n_voxels == len(big)
    assert np.array_equal(vox["centroids"][:, :3], big[:, :3])


# ---- a5 local frame + a6 markers -----------------------------------------------------------------
def _frame_close(fr, ref):
    scale = np.abs(ref["vals"]).max()
    assert np.abs(fr["scatter"] - ref["scatter"]).max() <= 1e-4 * scale          # 1e-4 relative to ||S||
    assert np.abs(fr["scatter"].astype(np.float64) - ref["scatter_truth"]).max() <= 2e-6 * scale
    assert np.abs(fr["vals"] - ref["vals"]).max() <= 1e-4 * scale
    # axis (eigenvector 0) up to sign; the other two only as a subspace (near-degenerate pair)
    assert _angle(fr["vecs"][:, 0].astype(np.float64), ref["vecs"][:, 0].astype(np.float64)) < 1e-3
    assert abs(np.dot(fr["vecs"][:, 0], ref["vecs"][:, 1])) < 2e-3 and abs(np.dot(fr["vecs"][:, 0], ref["vecs"][:, 2])) < 2e-3


def test_local_frame_parity_and_known_answer():
    pts = synth.straight_cylinder(50_000, seed=1, noise=0.01)
    with _ctx(len(pts), neighborRadius=0.2) as ctx:
        ctx.upload_scan(pts)
        ctx.crop()
        ctx.normals()
        ctx.local_frame()
        normals_c = ctx.download_normals(1)
        fr = ctx.frame()
    ref = O.local_frame(normals_c, 0.2)
    _frame_close(fr, ref)
    # known answer (src/tunnel_processing.cpp:91): min eigenvector = cylinder axis (x)
    assert abs(abs(fr["vecs"][0, 0]) - 1.0) < 1e-3
    assert fr["vals"][0] < 1e-2 * fr["vals"][2]
    # a6: arrow payload of rvizEigens
    arrows = capi.markers_eigen(fr["_struct"])
    refm = O.eigen_markers(fr["vals"], fr["vecs"])
    for i in range(3):
        assert np.array_equal(arrows[i]["start"], refm[i, 0:3])
        assert np.array_equal(arrows[i]["end"], refm[i, 3:6])
        assert np.array_equal(arrows[i]["scale"], refm[i, 6:9])
    assert arrows["color_argb"].tolist() == [[1, 1, 0, 0], [1, 0, 1, 0], [1, 0, 0, 1]]


def test_local_frame_injected_normals():
    g = np.random.Generator(np.random.Philox(4))
    n = 200_000
    nr = np.zeros((n, 8), np.float32)
    v = g.normal(size=(n, 3))
    v[:, 2] *= 0.05
    nr[:, :3] = v / np.linalg.norm(v, axis=1, keepdims=True)
    nr[:, 4] = g.uniform(0, 0.3, n)
    pts = np.ones((n, 4), np.float32)
    with _ctx(n, weightingFactor=0.13) as ctx:
        ctx.inject_compacted(pts, nr)
        ctx.local_frame()
        fr = ctx.frame()
    _frame_close(fr, O.local_frame(nr, 0.13))


def test_quirk_switches_weight_law_and_arrow_end():
    """SURVEY 8f.2: the reference's quirks stay the default; mode 1 of each switch is checked against the oracle's
    restatement (weights) and by construction (arrows)."""
    pts = synth.curved_tunnel(40_000, seed=12)
    out = {}
    for wm in (0, 1):
        with _ctx(len(pts), neighborRadius=0.15, weightingFactor=0.13, weight_mode=wm, arrow_mode=wm) as ctx:
            ctx.upload_scan(pts)
            ctx.crop()
            ctx.normals()
            ctx.voxel()
            ctx.local_frame()
            nrm = ctx.download_normals(1)
            fr = ctx.frame()
            vox = ctx.download_voxels()
            arrows = capi.markers_normals(vox["centroids"], vox["nn_normal"], ctx.params.arrow_mode)
        _frame_close(fr, O.local_frame(nrm, 0.13, weight_mode=wm))
        out[wm] = (fr, arrows, vox)
    assert not np.allclose(out[0][0]["scatter"], out[1][0]["scatter"], rtol=1e-3)          # the two laws differ
    a0, a1, vox = out[0][1], out[1][1], out[0][2]
    ok = np.isfinite(vox["nn_normal"][:, 0])
    assert np.array_equal(a0["end"][ok], vox["nn_normal"][ok, :3])                           # quirk B.4: end = the normal itself
    assert np.array_equal(a1["end"][ok], vox["centroids"][ok, :3] + vox["nn_normal"][ok, :3])  # fixed: start + normal
    assert np.array_equal(a0["start"], a1["start"])


# ---- a8 RANSAC (builder-defined; oracle = builder restatement of the PCL semantics) --------------
def _compacted_scan(n=80_000, seed=31, radius=0.15):
    pts = synth.curved_tunnel(n, seed=seed)
    cropped, _ = O.crop(pts, 5.0, True)
    nr, _, _ = O.normals(cropped, radius)
    return O.compact(cropped, nr)[:2]


def test_ransac_plane_counts_bit_exact_and_refit():
    cloud, nrm = _compacted_scan()
    H = 700
    samples = synth.sample_indices(len(cloud), H, 3, seed=3)
    samples[5] = [1, 1, 2]            # duplicate index -> degenerate
    samples[6] = [0, 1, len(cloud)]   # out of range -> degenerate
    coef, valid = O.plane_hypotheses(cloud, samples)
    counts = O.count_plane(cloud, coef, valid, TAU)
    with _ctx(len(cloud), ransacThreshold=TAU) as ctx:
        ctx.inject_compacted(cloud, nrm)
        ctx.ransac(capi.GM_MODEL_PLANE, samples)
        gcoef, _, gcounts = ctx.download_hypotheses(capi.GM_MODEL_PLANE, H)
        ctx.ransac_select(capi.GM_MODEL_PLANE)
        m = ctx.model(capi.GM_MODEL_PLANE)
    assert np.array_equal(gcoef.view(np.uint32), coef.view(np.uint32))  # hypothesis generation: bit-exact
    assert np.array_equal(gcounts, counts)                                # inlier counts: bit-exact
    assert counts[5] == -1 and counts[6] == -1
    best = O.argmax(counts)
    assert m["best_id"] == best and m["best_count"] == counts[best]
    ref_coef, ref_cnt = O.refit_plane(cloud, coef[best], TAU)
    assert m["refit_count"] == ref_cnt
    assert np.abs(m["coef"] - ref_coef).max() <= 1e-4 * max(1.0, np.abs(ref_coef).max())
    # the floor of the synthetic tunnel is z = -1.5
    assert abs(abs(m["coef"][2]) - 1.0) < 1e-3 and abs(abs(m["coef"][3]) - 1.5) < 5e-3


def test_ransac_cylinder_counts_bit_exact_and_refit():
    cloud, nrm = _compacted_scan()
    H = 600
    samples = synth.sample_indices(len(cloud), H, 2, seed=4)
    samples[3] = [9, 9]
    m7, t12, valid = O.cyl_hypotheses(cloud, nrm, samples, 0.5, 10.0, TAU)
    counts = O.count_cyl(cloud, t12, valid)
    with _ctx(len(cloud), ransacThreshold=TAU) as ctx:
        ctx.inject_compacted(cloud, nrm)
        ctx.ransac(capi.GM_MODEL_CYLINDER, samples)
        gm7, gt12, gcounts = ctx.download_hypotheses(capi.GM_MODEL_CYLINDER, H)
        ctx.ransac_select(capi.GM_MODEL_CYLINDER)
        m = ctx.model(capi.GM_MODEL_CYLINDER)
    assert np.array_equal(gm7.view(np.uint32), m7.view(np.uint32))
    assert np.array_equal(gt12.view(np.uint32), t12.view(np.uint32))
    assert np.array_equal(gcounts, counts)
    assert counts[3] == -1 and (counts >= 0).sum() > H // 4
    best = O.argmax(counts)
    assert m["best_id"] == best and m["best_count"] == counts[best]
    ref_m, ref_cnt, ref_rms = O.refit_cylinder(cloud, m7[best], t12[best], 5)
    assert m["refit_count"] == ref_cnt
    # axis direction and radius within 1e-4 relative; the axis point q is only defined up to a
    # shift along the axis, so compare its distance from the reference axis line
    assert _angle(m["coef"][3:6].astype(np.float64), ref_m[3:6].astype(np.float64)) < 1e-4
    assert abs(m["coef"][6] - ref_m[6]) <= 1e-4 * ref_m[6]
    dq = (m["coef"][:3] - ref_m[:3]).astype(np.float64)
    d = ref_m[3:6].astype(np.float64)
    assert np.linalg.norm(dq - d * dq.dot(d)) <= 1e-4 * ref_m[6]
    assert abs(m["rms"] - ref_rms) <= 1e-4 * max(ref_rms, 1e-3)
    assert abs(m["coef"][6] - 2.5) < 0.05  # the synthetic tunnel radius


def test_ransac_hypothesis_sharding_matches_single_range():
    """Multi-GPU contract emulated on one device: two half-ranges, max of the packed keys."""
    cloud, nrm = _compacted_scan(40_000, seed=41)
    H = 512
    samples = synth.sample_indices(len(cloud), H, 3, seed=8)
    with _ctx(len(cloud)) as ctx:
        ctx.inject_compacted(cloud, nrm)
        ctx.ransac(capi.GM_MODEL_PLANE, samples)
        _, _, full = ctx.download_hypotheses(capi.GM_MODEL_PLANE, H)
        parts = []
        for lo, hi in ((0, 256), (256, 512)):
            ctx.ransac(capi.GM_MODEL_PLANE, samples, lo, hi)
            _, _, c = ctx.download_hypotheses(capi.GM_MODEL_PLANE, H)
            assert (c[:lo] == -1).all() and (c[hi:] == -1).all()
            parts.append(c[lo:hi])
    assert np.array_equal(np.concatenate(parts), full)


def test_ransac_all_degenerate_reports_no_model():
    cloud, nrm = _compacted_scan(20_000, seed=43)
    samples = np.zeros((64, 3), np.int32)
    with _ctx(len(cloud)) as ctx:
        ctx.inject_compacted(cloud, nrm)
        ctx.ransac(capi.GM_MODEL_PLANE, samples)
        ctx.ransac_select(capi.GM_MODEL_PLANE)
        m = ctx.model(capi.GM_MODEL_PLANE)
    assert m["status"] == capi.GM_ERR_NO_MODEL and m["best_id"] == -1


# ---- fused path -----------------------------------------------------------------------------------
def test_process_scan_end_to_end_against_oracle_chain():
    n = 120_000
    radius, leaf = 0.12, 0.1
    pts = synth.curved_tunnel(n, seed=2)
    with _ctx(n, neighborRadius=radius, voxelGridLeafSize=leaf, sliceLength=1.0) as ctx:
        ctx.upload_scan(pts)
        ctx.crop()
        ctx.normals()
        c0 = ctx.counts()
        ps = synth.sample_indices(c0.n_valid, 512, 3, seed=3)
        cs = synth.sample_indices(c0.n_valid, 512, 2, seed=4)
        ctx.upload_scan(pts)
        ctx.process_scan(ps, cs)
        c = ctx.counts()
        cloud_c, normals_c = ctx.download_cloud(1), ctx.download_normals(1)
        fr = ctx.frame()
        mp, mc = ctx.model(capi.GM_MODEL_PLANE), ctx.model(capi.GM_MODEL_CYLINDER)
        labels = ctx.download_labels()
        poly = ctx.download_polyline()
        _, _, pc = ctx.download_hypotheses(capi.GM_MODEL_PLANE, 512)
        _, _, cc = ctx.download_hypotheses(capi.GM_MODEL_CYLINDER, 512)
    assert c.device_error == 0 and c.n_valid == c0.n_valid
    # oracle chain on the GPU's own compacted cloud/normals (stage inputs identical)
    coef, valid = O.plane_hypotheses(cloud_c, ps)
    assert np.array_equal(pc, O.count_plane(cloud_c, coef, valid, TAU))
    m7, t12, cvalid = O.cyl_hypotheses(cloud_c, normals_c, cs, 0.5, 10.0, TAU)
    assert np.array_equal(cc, O.count_cyl(cloud_c, t12, cvalid))
    # labels from the GPU's refined models, evaluated by the oracle: bit-exact
    ref_labels = O.labels(cloud_c, mp["coef"], TAU, O.cyl_test_params(mc["coef"], TAU)[0])
    assert np.array_equal(labels, ref_labels)
    assert (labels == 1).mean() > 0.1 and (labels == 2).mean() > 0.2
    # polyline vs oracle
    ref_poly, _ = O.polyline(cloud_c, normals_c, labels, 2, fr["vecs"][:, 0], 0.2, 1.0, 256)
    assert len(poly) == len(ref_poly) and len(poly) >= 8
    for s in range(len(poly)):
        assert poly["count"][s] == int(ref_poly[s, 7])
        if ref_poly[s, 7] < 50:
            continue
        assert np.abs(poly["center"][s] - ref_poly[s, 0:3]).max() <= 1e-4 * 5.0
        assert abs(poly["radius"][s] - ref_poly[s, 6]) <= 1e-4 * ref_poly[s, 6]
        assert abs(poly["rms"][s] - ref_poly[s, 8]) <= 1e-4 * max(ref_poly[s, 8], 1e-2)
        assert _angle(poly["dir"][s].astype(np.float64), ref_poly[s, 3:6]) < 1e-3
    # cross-section radius ~ tunnel radius in well-populated slices
    good = poly["count"] > 2000
    assert np.abs(poly["radius"][good] - 2.5).max() < 0.1


# ---- the reference's own call sequence through the mirrored host API --------------------------------
def test_cloud_cb_sequence_through_the_mirror_api():
    """src/geometric_mapping.cpp:48-125 with the four L1 calls swapped for the mirror functions."""
    from geometric_mapping_b200 import tunnel_processing as tp
    from geometric_mapping_b200.params import LAUNCH_FILE_VALUES, Parameters

    params = Parameters({**LAUNCH_FILE_VALUES, "neighborRadius": 0.3, "voxelGridLeafSize": 0.5})
    assert params.getBoxFilterBound() == 5.0 and params.displayNormals() is False
    cloud = _scan_with_junk(30_000, seed=13)
    with capi.Context(params.to_gm_params(), max_points=len(cloud)) as ctx:
        cloudChopped = tp.chopCloud(params.getBoxFilterBound(), cloud, ctx)                    # :57
        cloudNormals, cloudChopped = tp.getNormals(params.getNeighborRadius(), cloudChopped, ctx)   # :63
        normalsDisp = tp.rvizNormals(params.getLeafSize(), cloudChopped, ctx, cloudNormals)    # :70
        eigenVals, eigenVecs = tp.getLocalFrame(len(cloudChopped), params.getWeightingFactor(), cloudNormals, ctx)  # :82
        centerAxis = eigenVecs[:, 0]                                                           # :91-92
        eigenBasis = tp.rvizEigens(eigenVals, eigenVecs)                                       # :96
    ref_crop, _ = O.crop(cloud, 5.0, True)
    ref_n, _, _ = O.normals(ref_crop, 0.3)
    ref_cloud, ref_nc, _ = O.compact(ref_crop, ref_n)
    assert np.array_equal(cloudChopped.view(np.uint32), ref_cloud.view(np.uint32))
    assert cloudNormals.shape == ref_nc.shape
    ref_f = O.local_frame(cloudNormals, 0.2)
    assert np.abs(eigenVals - ref_f["vals"]).max() <= 1e-4 * ref_f["vals"].max()
    assert _angle(centerAxis.astype(np.float64), ref_f["vecs"][:, 0].astype(np.float64)) < 1e-3
    ref_v = O.voxel(cloudChopped, 0.5)
    assert len(normalsDisp) == ref_v["V"]
    m0 = normalsDisp[0]
    assert m0["ns"] == "normals" and m0["header"]["frame_id"] == "/velodyne" and m0["type"] == "ARROW"
    assert m0["color"] == {"a": 1.0, "r": 0.0, "g": 0.0, "b": 1.0}                  # quirk B.5: (1,0,0,1) pushed as a,r,g,b
    assert np.allclose(m0["points"][0], ref_v["centroids"][0, :3])
    assert m0["scale"] == tuple(float(np.float32(v)) for v in (0.025, 0.075, 0.0625))        # :230 stored as floats
    assert [m["ns"] for m in eigenBasis] == ["eigenBasis"] * 3 and [m["id"] for m in eigenBasis] == [0, 1, 2]
    assert eigenBasis[0]["points"][0] == (0.0, 0.0, 0.0) and np.allclose(eigenBasis[0]["points"][1], centerAxis)
    assert eigenBasis[1]["color"] == {"a": 1.0, "r": 0.0, "g": 1.0, "b": 0.0}


def test_stage_order_and_capacity_errors():
    with _ctx(100) as ctx:
        with pytest.raises(capi.GmError) as e:
            ctx.crop()
        assert e.value.status == capi.GM_ERR_STAGE_ORDER
        with pytest.raises(capi.GmError) as e:
            ctx.upload_scan(np.zeros((101, 4), np.float32))
        assert e.value.status == capi.GM_ERR_CAPACITY
        ctx.upload_scan(np.zeros((10, 4), np.float32))
        with pytest.raises(capi.GmError) as e:
            ctx.normals()
        assert e.value.status == capi.GM_ERR_STAGE_ORDER
        ctx.crop()
        ctx.normals()
        with pytest.raises(capi.GmError) as e:
            ctx.axis_polyline()
        assert e.value.status == capi.GM_ERR_STAGE_ORDER


def test_strided_upload_and_results_are_reproducible():
    """PointCloud2-like point_step of 32 bytes (x,y,z,+intensity,ring...) and run-to-run determinism."""
    pts = synth.curved_tunnel(40_000, seed=3)
    wide = np.zeros((len(pts), 8), np.float32)
    wide[:, :3] = pts[:, :3]
    wide[:, 3:] = 123.0
    outs = []
    with _ctx(len(pts), neighborRadius=0.15) as ctx:
        for rep in range(2):
            if rep == 0:
                ctx.upload_scan_raw(wide.ctypes.data, len(wide), 32)
            else:
                ctx.upload_scan(pts)
            ps = synth.sample_indices(30_000, 256, 3, seed=3)
            cs = synth.sample_indices(30_000, 256, 2, seed=4)
            ctx.process_scan(ps, cs)
            outs.append((ctx.download_normals(1), ctx.frame()["scatter"], ctx.model(0)["coef"], ctx.model(1)["coef"],
                         ctx.download_polyline(), ctx.download_labels()))
    a, b = outs
    assert np.array_equal(a[0].view(np.uint32), b[0].view(np.uint32))     # normals bitwise reproducible
    assert np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2]) and np.array_equal(a[3], b[3])
    assert a[4].tobytes() == b[4].tobytes() and np.array_equal(a[5], b[5])


def test_cpp_host_shim_node_harness_runs_cloud_cb(tmp_path):
    """The compiled C++ mirror of the node (geometric_mapping_b200/host) through the C-ABI."""
    import subprocess

    from geometric_mapping_b200 import build as gm_build

    exe = gm_build.build_host()
    pts = synth.straight_cylinder(50_000, seed=1, noise=0.01)
    path = str(tmp_path / "scan.f32x4")
    pts.tofile(path)
    res = subprocess.run([exe, "--set", "neighborRadius=0.2", "--set", "voxelGridLeafSize=0.5", "--set", "displayNormals=true",
                          "--scan", path], capture_output=True, text=True, timeout=120)
    assert res.returncode == 0, res.stderr
    lines = res.stdout.splitlines()
    axis = np.array([float(v) for v in lines[lines.index("Center Axis is:") + 1].split()])
    vals = np.array([float(v) for v in lines[lines.index("Eigenvalues are:") + 1].split()])
    assert abs(abs(axis[0]) - 1.0) < 1e-3 and vals[0] < 1e-2 * vals[2]
    with _ctx(len(pts), neighborRadius=0.2, voxelGridLeafSize=0.5) as ctx:
        ctx.upload_scan(pts)
        ctx.process_scan(None, None)
        fr = ctx.frame()
        c = ctx.counts()
    assert np.allclose(vals, fr["vals"], rtol=1e-5) and np.allclose(axis, fr["vecs"][:, 0], atol=1e-5)
    assert f"publish cloudOutput: {c.n_valid} points" in res.stdout
    assert f"publish normalsOutput: {c.n_voxels} markers" in res.stdout


# ---- compression (builder-defined, SURVEY A.10) ----------------------------------------------------
def test_compression_parity_and_blob_layout():
    import ctypes as C
    import struct

    n = 150_000
    pts = synth.curved_tunnel(n, seed=6, outlier_frac=0.02)
    with _ctx(n, neighborRadius=0.1, voxelGridLeafSize=0.2) as ctx:
        ctx.upload_scan(pts)
        ctx.crop()
        ctx.normals()
        nv = ctx.counts().n_valid
        ps, cs = synth.sample_indices(nv, 512, 3, seed=3), synth.sample_indices(nv, 512, 2, seed=4)
        ctx.upload_scan(pts)
        ctx.process_scan(ps, cs)
        ctx.compress()
        c = ctx.compression()
        blob = ctx.download_compressed()
        cloud_c, labels = ctx.download_cloud(1), ctx.download_labels()
        mp, mc = ctx.model(0), ctx.model(1)
        poly = ctx.download_polyline()
        assert ctx.counts().device_error == 0
    ref = O.compress(cloud_c, labels, mp["coef"], mc["coef"], TAU, 0.2)
    # counts: exact
    assert (c.n_points, c.n_plane, c.n_cylinder, c.n_residual, c.n_residual_voxels) == \
        (ref["n_points"], ref["n_plane"], ref["n_cylinder"], ref["n_residual"], ref["n_residual_voxels"])
    assert c.n_plane == int((labels == 1).sum()) and c.n_cylinder == int((labels == 2).sum()) and c.n_slices == len(poly)
    # primitives: 1e-4 relative (bounds relative to the 10 m box)
    assert np.allclose(np.array(c.plane_u), ref["plane_u"], atol=1e-6) and np.allclose(np.array(c.plane_v), ref["plane_v"], atol=1e-6)
    assert np.abs(np.array(c.plane_bounds) - ref["plane_bounds"]).max() <= 1e-4 * 10
    assert np.abs(np.array(c.cyl_t_range) - ref["cyl_t_range"]).max() <= 1e-4 * 10
    for k in ("plane_rms", "cyl_rms", "residual_rms", "total_rms"):
        assert abs(getattr(c, k) - ref[k]) <= 1e-4 * max(ref[k], 1e-3), k
    assert np.array_equal(np.array(c.plane_coef), mp["coef"]) and np.array_equal(np.array(c.cyl_coef), mc["coef"])
    # it actually compresses, and the error is bounded by the leaf / inlier threshold
    assert c.bytes_in == 16 * c.n_points and c.bytes_out == len(blob) and c.ratio > 4.0
    assert c.total_rms < 0.2 and c.plane_rms < TAU and c.cyl_rms < TAU
    # blob: 'GMC1' | version | gm_compression | slices | residual centroids (bit-exact vs the oracle voxel grid)
    magic, version = struct.unpack_from("<II", blob, 0)
    assert magic == 0x31434D47 and version == 1
    hdr = capi.gm_compression.from_buffer_copy(blob[8:8 + C.sizeof(capi.gm_compression)])
    assert hdr.n_residual_voxels == c.n_residual_voxels and hdr.bytes_out == c.bytes_out
    off = 8 + C.sizeof(capi.gm_compression)
    sl = np.frombuffer(blob, capi.SLICE_DTYPE, count=c.n_slices, offset=off)
    assert sl.tobytes() == poly.tobytes()
    cen = np.frombuffer(blob, np.float32, count=3 * c.n_residual_voxels, offset=off + 40 * c.n_slices).reshape(-1, 3)
    assert np.array_equal(cen.view(np.uint32), ref["residual_centroids"][:, :3].copy().view(np.uint32))


def test_compression_without_models_keeps_everything_as_residual():
    pts = synth.straight_cylinder(20_000, seed=2)
    with _ctx(len(pts), neighborRadius=0.2, voxelGridLeafSize=0.25) as ctx:
        ctx.upload_scan(pts)
        ctx.process_scan(None, None)
        ctx.compress()
        c = ctx.compression()
        cloud_c = ctx.download_cloud(1)
    ref = O.voxel(cloud_c, 0.25)
    assert c.n_plane == 0 and c.n_cylinder == 0 and c.n_residual == c.n_points == len(cloud_c)
    assert c.n_residual_voxels == ref["V"] and c.n_slices == 0


# ---- BASELINE.json full size (1M points): size-independent properties -------------------------------
def test_full_size_properties_1m_points():
    n = 1_000_000
    pts = synth.curved_tunnel(n, seed=2)
    H = 1024
    with capi.Context(capi.default_params(neighborRadius=0.05, voxelGridLeafSize=0.1), max_points=n, max_hypotheses=4096) as ctx:
        ctx.upload_scan(pts)
        ctx.crop()
        cropped = ctx.download_cloud(0)
        ctx.normals()
        nv = ctx.counts().n_valid
        ps, cs = synth.sample_indices(nv, H // 2, 3, seed=3), synth.sample_indices(nv, H // 2, 2, seed=4)
        ctx.upload_scan(pts)
        ctx.process_scan(ps, cs)
        c = ctx.counts()
        cloud_c, normals_c = ctx.download_cloud(1), ctx.download_normals(1)
        keys, assign, _ = ctx.download_voxel_assignment()
        vox = ctx.download_voxels()
        pcoef, _, pcounts = ctx.download_hypotheses(capi.GM_MODEL_PLANE, H // 2)
        _, ct12, ccounts = ctx.download_hypotheses(capi.GM_MODEL_CYLINDER, H // 2)
        mp, mc = ctx.model(0), ctx.model(1)
        labels = ctx.download_labels()
        # crop is idempotent: cropping the cropped cloud changes nothing
        ctx.upload_scan(cropped)
        ctx.crop()
        assert np.array_equal(ctx.download_cloud(0).view(np.uint32), cropped.view(np.uint32))
    assert c.device_error == 0 and c.n_cropped == len(cropped) and c.n_valid == len(cloud_c) == nv
    # crop: every kept point is inside the box, order preserved (a subsequence of the input)
    assert (np.abs(cropped[:, :3]) <= 5.0).all()
    inside = (np.abs(pts[:, :3]) <= 5.0).all(1)
    assert np.array_equal(cropped.view(np.uint32), pts[inside].view(np.uint32))
    # normals: unit length, flipped towards the sensor, curvature in [0, 1/3]
    assert np.abs(np.linalg.norm(normals_c[:, :3], axis=1) - 1.0).max() < 1e-4
    assert (-(cloud_c[:, :3] * normals_c[:, :3]).sum(1) >= -1e-5).all()
    assert (normals_c[:, 4] >= 0).all() and (normals_c[:, 4] <= 1 / 3 + 1e-4).all()
    # voxel grid: voxel keys strictly ascending, assignment consistent with the per-point keys, counts conserve points
    assert (np.diff(vox["keys"].astype(np.int64)) > 0).all() and c.n_voxels == len(vox["keys"])
    assert np.array_equal(vox["keys"][assign], keys)
    assert vox["counts"].sum() == len(cloud_c) and np.array_equal(np.bincount(assign, minlength=c.n_voxels), vox["counts"])
    # centroid of a voxel lies inside that voxel's cell of the lattice (leaf 0.1)
    inv = np.float32(1.0) / np.float32(0.1)
    assert np.array_equal(np.floor(vox["centroids"][:, :3] * inv).astype(np.int64), np.floor(cloud_c[np.unique(assign, return_index=True)[1], :3] * inv).astype(np.int64))
    # the 1-NN of a centroid is at most one voxel diagonal away
    nn = vox["nn_index"]
    ok = (nn >= 0) & (nn < len(cropped))
    assert ok.all()
    assert (np.linalg.norm(cropped[nn, :3] - vox["centroids"][:, :3], axis=1) <= 0.1 * np.sqrt(3) + 1e-5).all()
    # RANSAC: counts bounded by the cloud size, argmax/tie rule, labels consistent with the refined models
    assert pcounts.max() <= len(cloud_c) and ccounts.max() <= len(cloud_c) and pcounts.min() >= -1
    assert mp["best_count"] == pcounts.max() and mp["best_id"] == int(np.argmax(pcounts))
    assert mc["best_count"] == ccounts.max() and mc["best_id"] == int(np.argmax(ccounts))
    d = (cloud_c[:, :3].astype(np.float64) @ mp["coef"][:3].astype(np.float64)) + float(mp["coef"][3])
    assert (np.abs(d[labels == 1]) < TAU + 1e-5).all() and (np.abs(d[labels != 1]) > TAU - 1e-5).all()
    # exact linearity with numpy: the winning plane's count equals the number of points passing the canonical test
    best = pcoef[mp["best_id"]]
    dd = np.abs((cloud_c[:, :3].astype(np.float64) @ best[:3].astype(np.float64)) + float(best[3]))
    assert abs(int((dd < TAU).sum()) - mp["best_count"]) <= 4          # float vs double only at the boundary
    assert abs(abs(mp["coef"][3]) - 1.5) < 5e-3 and abs(mc["coef"][6] - 2.5) < 0.7   # a straight cylinder on a curved tunnel with a floor: a weak model (~15 % inliers)


@pytest.mark.parametrize("n,radius,tau", [(90_000, 0.1, 0.05), (30_000, 0.3, 0.2), (700, 0.5, 0.05), (20, 1.0, 0.05)])
def test_tile_culled_counts_equal_brute_force_and_oracle(n, radius, tau):
    """gm_ransac counts over the cell-sorted cloud with tile culling (mode 0, the default after
    gm_normals) == the brute-force kernels (mode 1) == the oracle, bit for bit: junk points (NaN, inf,
    outliers), more hypotheses than one chunk, a sharded hypothesis range, tiny clouds."""
    pts = _scan_with_junk(n, seed=77) if n >= 1000 else synth.curved_tunnel(n, seed=78, outlier_frac=0.1)
    Hp, Hc = 1300, 1100
    with _ctx(n, neighborRadius=radius, ransacThreshold=tau) as ctx:
        ctx.upload_scan(pts)
        ctx.crop()
        ctx.normals()
        nv = ctx.counts().n_valid
        cloud_c, normals_c = ctx.download_cloud(1), ctx.download_normals(1)
        ps = synth.sample_indices(nv, Hp, 3, seed=13)
        cs = synth.sample_indices(nv, Hc, 2, seed=14)
        ps[3] = [0, 0, 1]
        got = {}
        for mode in (0, 1):
            ctx.set_count_mode(mode)
            ctx.ransac(capi.GM_MODEL_PLANE, ps)
            ctx.ransac(capi.GM_MODEL_CYLINDER, cs)
            got[mode] = (ctx.download_hypotheses(0, Hp)[2], ctx.download_hypotheses(1, Hc)[2])
            ctx.ransac_select(0)
            ctx.ransac_select(1)
            got[mode] += (ctx.model(0)["best_id"], ctx.model(1)["best_id"])
        ctx.set_count_mode(0)
        ctx.ransac(capi.GM_MODEL_PLANE, ps, 517, 1203)   # a rank's shard: ids outside score -1
        shard = ctx.download_hypotheses(0, Hp)[2]
        assert ctx.counts().device_error == 0
    coef, valid = O.plane_hypotheses(cloud_c, ps)
    ref_p = O.count_plane(cloud_c, coef, valid, tau)
    m7, t12, cvalid = O.cyl_hypotheses(cloud_c, normals_c, cs, 0.5, 10.0, tau)
    ref_c = O.count_cyl(cloud_c, t12, cvalid)
    for mode in (0, 1):
        assert np.array_equal(got[mode][0], ref_p), f"plane counts, mode {mode}"
        assert np.array_equal(got[mode][1], ref_c), f"cylinder counts, mode {mode}"
    assert got[0][2:] == got[1][2:]
    assert np.array_equal(shard[517:1203], ref_p[517:1203]) and (shard[:517] == -1).all() and (shard[1203:] == -1).all()
    if n >= 30_000:
        assert ref_p.max() > 0.1 * nv and ref_c.max() > 0.1 * nv   # the test is not vacuous


def test_ransac_pair_equals_separate_calls_and_sharded_keys_compose():
    """gm_ransac_pair / gm_ransac_select_pair (plane and cylinder side by side on two streams) == the four separate
    calls; and the max of the per-shard keys, imported as 16 bytes, selects the single-range winners."""
    import torch

    n = 60_000
    pts = synth.curved_tunnel(n, seed=41)
    with _ctx(n, neighborRadius=0.12) as ctx:
        ctx.upload_scan(pts); ctx.crop(); ctx.normals()
        nv = ctx.counts().n_valid
        ps, cs = synth.sample_indices(nv, 640, 3, seed=3), synth.sample_indices(nv, 600, 2, seed=4)
        ctx.ransac(0, ps); ctx.ransac(1, cs)
        ref_counts = (ctx.download_hypotheses(0, 640)[2], ctx.download_hypotheses(1, 600)[2])
        ctx.ransac_select(0); ctx.ransac_select(1)
        ref_models = (ctx.model(0), ctx.model(1))
        ctx.ransac_pair(ps, cs)
        got_counts = (ctx.download_hypotheses(0, 640)[2], ctx.download_hypotheses(1, 600)[2])
        ctx.ransac_select_pair()
        got_models = (ctx.model(0), ctx.model(1))
        # three "ranks" on one GPU: shard, export 16 bytes, max, import, select
        keys = torch.zeros(2, dtype=torch.int64, device="cuda")
        best = torch.zeros(2, dtype=torch.int64, device="cuda")
        from geometric_mapping_b200 import distributed as D
        for r in range(3):
            ctx.ransac_pair(ps, cs, D.shard_range(640, r, 3), D.shard_range(600, r, 3))
            ctx.ransac_export_keys(keys.data_ptr())
            ctx.synchronize()
            best = torch.maximum(best, keys)
        ctx.ransac_import_keys(best.data_ptr())
        ctx.ransac_select_pair()
        shard_models = (ctx.model(0), ctx.model(1))
        assert ctx.counts().device_error == 0
    for k in (0, 1):
        assert np.array_equal(got_counts[k], ref_counts[k])
        for m in (got_models[k], shard_models[k]):
            assert m["best_id"] == ref_models[k]["best_id"] and m["best_count"] == ref_models[k]["best_count"]
            assert m["refit_count"] == ref_models[k]["refit_count"]
            assert np.array_equal(m["coef"].view(np.uint32), ref_models[k]["coef"].view(np.uint32))   # same kernels, same bits


def test_count_linearity_over_a_split_cloud():
    """counts(cloud) == counts(first half) + counts(second half) for fixed hypotheses: exact."""
    cloud, nrm = _compacted_scan(60_000, seed=51)
    H = 256
    g = np.random.Generator(np.random.Philox(5))
    half = len(cloud) // 2
    # samples drawn from the first half only, so both runs build the same hypotheses
    ps = g.integers(0, half, size=(H, 3)).astype(np.int32)
    cs = g.integers(0, half, size=(H, 2)).astype(np.int32)
    out = {}
    with _ctx(len(cloud)) as ctx:
        for name, sl in (("all", slice(None)), ("a", slice(0, half))):
            ctx.inject_compacted(cloud[sl], nrm[sl])
            ctx.ransac(capi.GM_MODEL_PLANE, ps)
            ctx.ransac(capi.GM_MODEL_CYLINDER, cs)
            out[name] = (ctx.download_hypotheses(0, H), ctx.download_hypotheses(1, H))
    (pc_all, _, pn_all), (cm_all, ct_all, cn_all) = out["all"]
    (pc_a, _, pn_a), (cm_a, ct_a, cn_a) = out["a"]
    assert np.array_equal(pc_all.view(np.uint32), pc_a.view(np.uint32)) and np.array_equal(ct_all.view(np.uint32), ct_a.view(np.uint32))
    # second half evaluated by the oracle with the same coefficients
    pn_b = O.count_plane(cloud[half:], pc_all, (pn_all >= 0).astype(np.int32), TAU)
    cn_b = O.count_cyl(cloud[half:], ct_all, (cn_all >= 0).astype(np.int32))
    v = pn_all >= 0
    assert np.array_equal(pn_all[v], pn_a[v] + pn_b[v])
    v = cn_all >= 0
    assert np.array_equal(cn_all[v], cn_a[v] + cn_b[v])


def test_frame_sequence_polyline_per_frame():
    """Config C3 in miniature: consecutive frames of the same tunnel through one context."""
    n, frames = 60_000, 4
    with _ctx(n, neighborRadius=0.15, voxelGridLeafSize=0.2) as ctx:
        for f in range(frames):
            pts = synth.curved_tunnel(n, seed=100 + f, advance=1.0 * f)
            ctx.upload_scan(pts)
            ctx.crop()
            ctx.normals()
            nv = ctx.counts().n_valid
            ps, cs = synth.sample_indices(nv, 256, 3, seed=3 + f), synth.sample_indices(nv, 256, 2, seed=4 + f)
            ctx.upload_scan(pts)
            ctx.process_scan(ps, cs)
            cloud_c, normals_c, labels = ctx.download_cloud(1), ctx.download_normals(1), ctx.download_labels()
            fr, poly = ctx.frame(), ctx.download_polyline()
            ref_poly, _ = O.polyline(cloud_c, normals_c, labels, 2, fr["vecs"][:, 0], 0.2, 1.0, 256)
            assert len(poly) == len(ref_poly) and len(poly) >= 5
            assert np.array_equal(poly["count"], ref_poly[:, 7].astype(np.int32))
            big = ref_poly[:, 7] > 200
            assert np.abs(poly["center"][big] - ref_poly[big, 0:3]).max() <= 5e-4
            assert np.abs(poly["radius"][big] - ref_poly[big, 6]).max() <= 1e-4 * 2.5
            assert ctx.counts().device_error == 0


# ---- randomised small cases --------------------------------------------------------------------------------
def _fuzz_cloud(g, n):
    kind = int(g.integers(0, 6))
    if n == 0:
        return np.zeros((0, 4), np.float32)
    if kind == 0:      # tunnel piece with junk
        pts = synth.curved_tunnel(n, seed=int(g.integers(1, 1 << 30)), outlier_frac=0.05)
    elif kind == 1:    # uniform blob
        pts = np.ones((n, 4), np.float32); pts[:, :3] = g.uniform(-1.5, 1.5, (n, 3))
    elif kind == 2:    # all points identical
        pts = np.ones((n, 4), np.float32); pts[:, :3] = g.uniform(-1, 1, 3).astype(np.float32)
    elif kind == 3:    # collinear
        t = g.uniform(-2, 2, n); pts = np.ones((n, 4), np.float32); pts[:, 0] = t; pts[:, 1] = 0.5 * t; pts[:, 2] = -0.25 * t
    elif kind == 4:    # on a lattice (points exactly on cell / voxel faces)
        q = g.integers(-20, 21, (n, 3)).astype(np.float32) * np.float32(0.125)
        pts = np.ones((n, 4), np.float32); pts[:, :3] = q
    else:              # thin plane patch
        pts = synth.plane_patch(n, seed=int(g.integers(1, 1 << 30)), noise=0.003)
    pts = np.ascontiguousarray(pts, np.float32)
    k = min(n, int(g.integers(0, 4)))
    if k:
        idx = g.choice(n, k, replace=False)
        pts[idx, int(g.integers(0, 3))] = [np.nan, np.inf, -np.inf, 7.5][int(g.integers(0, 4))]
    return pts


@pytest.mark.parametrize("seed", [1, 2, 3, 4])
def test_fuzz_small_clouds_every_exact_output(seed):
    """Many small random clouds (degenerate shapes, NaN/inf, points on cell faces) and random parameters through
    the whole chain; every integer / index output against the oracle, bit for bit."""
    g = np.random.Generator(np.random.Philox(1000 + seed))
    with _ctx(4096) as ctx:
        for case in range(12):
            n = int(g.choice([0, 1, 2, 3, 7, 33, 200, 1000, 4000]))
            pts = _fuzz_cloud(g, n)
            bound = float(g.choice([0.75, 2.0, 5.0]))
            radius = float(g.choice([0.05, 0.13, 0.4, 1.1]))
            leaf = float(g.choice([0.05, 0.125, 0.3]))
            tau = float(g.choice([0.02, 0.1]))
            dense = int(g.integers(0, 2))
            p = capi.default_params(boxFilterBound=bound, neighborRadius=radius, voxelGridLeafSize=leaf, ransacThreshold=tau,
                                    is_dense=dense, nn_index_mode=1)
            ctx.set_params(p)
            ctx.upload_scan(pts)
            ctx.crop()
            ctx.normals()
            c0 = ctx.counts()
            tag = f"seed {seed} case {case} n {n} bound {bound} r {radius} leaf {leaf}"
            cropped, _ = O.crop(pts, bound, bool(dense))
            assert c0.n_cropped == len(cropped), tag
            ref_n, ref_cnt, _ = O.normals(cropped, radius, mode=0, order=0)
            assert np.array_equal(ctx.download_neighbor_counts(), ref_cnt), tag
            cloud_c = ctx.download_cloud(1)
            nrm_c = ctx.download_normals(1)
            # the GPU's own validity decides the compaction (a NaN from a degenerate eigen solve is data dependent in the
            # last bit); the oracle must agree wherever its normal is safely finite or safely missing
            vmap = ctx.download_valid_map()
            assert ((ref_cnt < 3) <= (vmap < 0)).all(), tag
            assert np.array_equal(cloud_c.view(np.uint32), cropped[vmap >= 0].view(np.uint32)), tag
            nv = c0.n_valid
            ctx.voxel()
            keys, assign, st = ctx.download_voxel_assignment()
            vox = ctx.download_voxels()
            refv = O.voxel(cloud_c, leaf)
            if refv["status"] == 0:
                assert np.array_equal(keys, refv["keys"]) and np.array_equal(assign, refv["assign"]), tag
                assert np.array_equal(vox["counts"], refv["voxel_counts"]), tag
                if nv:
                    _centroids_match(vox["centroids"], refv)
                    ref_idx, _ = O.nn1(vox["centroids"], cloud_c)
                    assert np.array_equal(vox["nn_index"], ref_idx), tag
            H = 96
            ps, cs = synth.sample_indices(max(nv, 1), H, 3, seed=case), synth.sample_indices(max(nv, 1), H, 2, seed=case + 50)
            coef, valid = O.plane_hypotheses(cloud_c, ps)
            ref_p = O.count_plane(cloud_c, coef, valid, tau)
            m7, t12, cvalid = O.cyl_hypotheses(cloud_c, nrm_c, cs, 0.5, 10.0, tau)
            ref_c = O.count_cyl(cloud_c, t12, cvalid)
            for mode in (0, 1):
                ctx.set_count_mode(mode)
                ctx.ransac(0, ps); ctx.ransac(1, cs)
                assert np.array_equal(ctx.download_hypotheses(0, H)[2], ref_p), tag + f" plane mode {mode}"
                assert np.array_equal(ctx.download_hypotheses(1, H)[2], ref_c), tag + f" cyl mode {mode}"
            ctx.set_count_mode(0)
            ctx.ransac_select(0); ctx.ransac_select(1)
            ctx.label()
            mp, mc = ctx.model(0), ctx.model(1)
            ref_lab = O.labels(cloud_c, mp["coef"] if mp["best_id"] >= 0 else None, tau,
                               O.cyl_test_params(mc["coef"], tau)[0] if mc["best_id"] >= 0 else None)
            assert np.array_equal(ctx.download_labels(), ref_lab), tag
            assert ctx.counts().device_error == 0, tag


# ---- scans in flight: the way bench.py measures throughput ------------------------------------------------------
def test_three_contexts_in_flight_give_the_single_context_results():
    """Three contexts fed round robin without waiting (their kernels overlap on the GPU, as in bench.py's throughput
    measurement): every scan's results are bit-identical to the same scan processed alone."""
    n, rounds = 70_000, 4
    scans = [synth.curved_tunnel(n, seed=300 + k) for k in range(3)]

    def snapshot(ctx):
        keys, assign, _ = ctx.download_voxel_assignment()
        vox = ctx.download_voxels()
        return (ctx.download_cloud(1), ctx.download_normals(1), keys, vox["centroids"], vox["nn_index"],
                ctx.download_hypotheses(0, 256)[2], ctx.download_hypotheses(1, 256)[2], ctx.download_labels(),
                ctx.model(0)["coef"], ctx.model(1)["coef"], ctx.download_polyline())

    params = dict(neighborRadius=0.12, voxelGridLeafSize=0.1)
    alone, samples = [], []
    with _ctx(n, **params) as ctx:
        for k in range(3):
            ctx.upload_scan(scans[k]); ctx.crop(); ctx.normals()
            nv = ctx.counts().n_valid
            samples.append((synth.sample_indices(nv, 256, 3, seed=3 + k), synth.sample_indices(nv, 256, 2, seed=4 + k)))
            ctx.upload_scan(scans[k])
            ctx.process_scan(*samples[k])
            alone.append(snapshot(ctx))
    ctxs = [_ctx(n, **params) for _ in range(3)]
    try:
        for r in range(rounds):
            for k in range(3):                       # enqueue on all three without synchronising
                c = ctxs[(k + r) % 3]
                c.upload_scan(scans[k])
                c.process_scan(*samples[k])
            for k in range(3):
                got = snapshot(ctxs[(k + r) % 3])
                for a, b in zip(got, alone[k]):
                    assert np.array_equal(np.asarray(a).view(np.uint8), np.asarray(b).view(np.uint8)), (r, k)
        assert all(c.counts().device_error == 0 for c in ctxs)
    finally:
        for c in ctxs:
            c.close()


# ---- map slabs (SURVEY 8e / config C4) ---------------------------------------------------------------
def test_map_slabs_reproduce_the_whole_map():
    """A map cut into 3 slabs at voxel faces, each processed with a halo on its own context, gives for
    its owned points exactly the compacted cloud, normals, voxel keys and centroids of the whole map."""
    from geometric_mapping_b200 import distributed as D

    n, bound, radius, leaf = 150_000, 20.0, 0.2, 0.25
    pts = synth.curved_tunnel(n, seed=5, arc_length=30.0, arc_radius=100.0, bound=bound, outlier_frac=0.02)
    pts[11] = [np.nan, 0.0, 0.0, 1.0]
    kw = dict(boxFilterBound=bound, neighborRadius=radius, voxelGridLeafSize=leaf)
    with _ctx(n, **kw) as ctx:
        ctx.upload_scan(pts)
        ctx.crop()
        ctx.normals()
        ctx.voxel()
        ctx.local_frame()
        w_cloud, w_nrm = ctx.download_cloud(1), ctx.download_normals(1)
        w_vox = ctx.download_voxels()
        w_bbox = ctx.voxel_bbox()
        w_scatter = ctx.frame()["scatter"].astype(np.float64).reshape(-1)
    cuts = D.slab_cuts(pts[:, 0], 3, leaf)
    assert cuts[0][1] < cuts[1][1] < cuts[2][1]
    got_keys, got_cen, got_cnt, scatter, n_owned = [], [], [], np.zeros((3, 3)), 0
    boxes = []
    with _ctx(n, **kw) as ctx:
        for variant in ("cube", "box"):
            for lo, hi in cuts:
                sl = D.slab_select(pts, 0, lo, hi, halo=1.01 * radius)
                assert len(sl) < 0.5 * n
                ctx.set_owned_range(0, lo, hi)
                if variant == "box":   # the grid a production rank would use: its own region only
                    fin = np.isfinite(sl[:, :3]).all(1)
                    ctx.set_grid_box(sl[fin, :3].min(0), sl[fin, :3].max(0))
                ctx.upload_scan(sl)
                ctx.crop()
                ctx.normals()
                cloud, nrm = ctx.download_cloud(1), ctx.download_normals(1)
                own = (w_cloud[:, 0] >= np.float32(lo)) & (w_cloud[:, 0] < np.float32(hi))
                assert np.array_equal(cloud.view(np.uint32), w_cloud[own].view(np.uint32))       # same points, same order
                if variant == "cube":
                    assert np.array_equal(nrm.view(np.uint32), w_nrm[own].view(np.uint32))       # bit-identical normals
                    boxes.append(ctx.voxel_bbox())
                    ctx.set_voxel_bbox(*w_bbox)     # what the MIN/MAX all-reduce delivers (checked below)
                    ctx.voxel()
                    ctx.local_frame()
                    v = ctx.download_voxels()
                    got_keys.append(v["keys"]); got_cen.append(v["centroids"]); got_cnt.append(v["counts"])
                    scatter += ctx.frame()["scatter"].astype(np.float64).reshape(3, 3)
                    n_owned += len(cloud)
                else:
                    ang = _angle(nrm[:, :3].astype(np.float64), w_nrm[own][:, :3].astype(np.float64))
                    assert np.percentile(ang, 99) < 2e-2   # other cell boundaries -> other summation order only
                assert ctx.counts().device_error == 0
            ctx.set_voxel_bbox(None)
        ctx.set_owned_range(-1)
        ctx.set_grid_box(None)
    assert n_owned == len(w_cloud)
    mn = np.min([b[0] for b in boxes if np.isfinite(b[0]).all()], axis=0)
    mx = np.max([b[1] for b in boxes if np.isfinite(b[1]).all()], axis=0)
    assert np.array_equal(mn, w_bbox[0]) and np.array_equal(mx, w_bbox[1])                       # the all-reduced box
    keys, cen, cnt = np.concatenate(got_keys), np.concatenate(got_cen), np.concatenate(got_cnt)
    o = np.argsort(keys, kind="stable")
    assert np.array_equal(keys[o], w_vox["keys"]) and len(np.unique(keys)) == len(keys)           # disjoint, complete
    assert np.array_equal(cnt[o], w_vox["counts"])
    assert np.array_equal(cen[o].view(np.uint32), w_vox["centroids"].view(np.uint32))             # bit-identical centroids
    assert np.abs(scatter.reshape(-1) - w_scatter).max() <= 1e-5 * np.abs(w_scatter).max()        # sum of the partial scatters


# ---- aggregated voxel map across scans (SURVEY 8f.3) ----------------------------------------------------
def _pose(yaw, t):
    c, s_ = np.cos(yaw), np.sin(yaw)
    return np.array([[c, -s_, 0, t[0]], [s_, c, 0, t[1]], [0, 0, 1, t[2]]], np.float32)


def test_voxel_map_matches_oracle_and_is_order_independent(tmp_path):
    n, frames, leaf = 40_000, 4, 0.1
    poses = [_pose(0.02 * f, (1.0 * f, 0.05 * f, 0.0)) for f in range(frames)]
    clouds, labels = [], []
    with _ctx(n, neighborRadius=0.15) as ctx, capi.VoxelMap(leaf, 1 << 18) as vm, capi.VoxelMap(leaf, 1 << 18) as vm_rev, \
            capi.VoxelMap(leaf, 1 << 18) as vm_cyl:
        for f in range(frames):
            pts = _scan_with_junk(n, seed=200 + f)
            ctx.upload_scan(pts)
            ctx.crop()
            ctx.normals()
            nv = ctx.counts().n_valid
            ctx.upload_scan(pts)
            ctx.process_scan(synth.sample_indices(nv, 128, 3, seed=3), synth.sample_indices(nv, 128, 2, seed=4))
            clouds.append(ctx.download_cloud(1)); labels.append(ctx.download_labels())
            vm.insert(ctx, poses[f])
            vm_cyl.insert(ctx, None, label_filter=2)
        for f in reversed(range(frames)):                      # same scans, other order, through injection
            ctx.inject_compacted(clouds[f], None)
            vm_rev.insert(ctx, poses[f])
        got, got_rev, got_cyl = vm.download(), vm_rev.download(), vm_cyl.download()
        stats = vm.stats()
        path = str(tmp_path / "map.gmm")
        vm.save(path)
        with capi.VoxelMap.load(path) as vm2:
            again = vm2.download()
            assert abs(vm2.leaf - leaf) < 1e-12 and vm2.stats()[:2] == stats[:2]
            ctx.inject_compacted(clouds[0], None)              # a loaded map keeps aggregating
            vm2.insert(ctx, poses[1])
            more = vm2.download()
    ref, ref_cyl = None, None
    for f in range(frames):
        ref = O.map_insert(ref, clouds[f], leaf, pose34=poses[f])
        ref_cyl = O.map_insert(ref_cyl, clouds[f], leaf, labels=labels[f], label_filter=2)
    assert stats[0] == len(ref["ijk"]) and stats[1] == sum(len(c) for c in clouds) - ref["out_of_range"] and not stats[3]
    for g in (got, got_rev, again):
        assert np.array_equal(g["ijk"], ref["ijk"]) and np.array_equal(g["counts"], ref["counts"])       # cells, counts: exact
        assert np.array_equal(g["centroids"].view(np.uint32), ref["centroids"].view(np.uint32))         # fixed-point sums: exact
    assert np.array_equal(got_cyl["ijk"], ref_cyl["ijk"]) and np.array_equal(got_cyl["counts"], ref_cyl["counts"])
    assert np.array_equal(got_cyl["centroids"].view(np.uint32), ref_cyl["centroids"].view(np.uint32))
    ref_more = O.map_insert(ref, clouds[0], leaf, pose34=poses[1])
    assert np.array_equal(more["ijk"], ref_more["ijk"]) and np.array_equal(more["counts"], ref_more["counts"])
    # one identity-pose frame: same cells and counts as pcl::VoxelGrid of that frame, centroids within the fixed-point step
    vg = O.voxel(clouds[0], leaf)
    one = O.map_insert(None, clouds[0], leaf)
    lin = (one["ijk"] - vg["grid6"][:3]) @ np.array([1, vg["grid6"][3], vg["grid6"][3] * vg["grid6"][4]])
    assert np.array_equal(lin, vg["voxel_keys"]) and np.array_equal(one["counts"], vg["voxel_counts"])
    assert np.abs(one["centroids"][:, :3] - vg["centroids"][:, :3]).max() < 1e-5


def test_voxel_map_capacity_and_range_are_reported():
    n = 20_000
    pts = synth.curved_tunnel(n, seed=9)
    with _ctx(n, neighborRadius=0.2) as ctx, capi.VoxelMap(0.1, 64) as small, capi.VoxelMap(1e-6, 1 << 16) as fine:
        ctx.upload_scan(pts); ctx.crop(); ctx.normals()
        small.insert(ctx)
        v, p, oor, full = small.stats()
        assert full and v == 128 and p < n                     # 128 slots, every slot taken, the rest dropped and flagged
        fine.insert(ctx)                                       # 1 um voxels: indices beyond +-2^20 are counted, not wrapped
        v, p, oor, full = fine.stats()
        assert oor > 0 and p + oor == ctx.counts().n_valid and not full
        fine.clear()
        assert fine.stats()[:3] == (0, 0, 0)


# ---- the C++ mirror of the reference seam (host/): the ROS-free node on one synthetic scan ---------------------
def test_cpp_host_node_runs_the_reference_callback_flow():
    """geometric_mapping_node (C++ shim: chopCloud / getNormals / rvizNormals / getLocalFrame / rvizEigens on top of
    the C-ABI, control flow of cloud_cb) on a straight cylinder along x: the printed center axis is the cylinder
    axis (the analytic known answer of src/tunnel_processing.cpp:91,139-143) and the publish lines are gated by
    the display parameters of the launch file."""
    import os
    import subprocess

    from geometric_mapping_b200 import build as gm_build

    exe = gm_build.build_host()
    assert os.path.exists(exe)
    res = subprocess.run([exe, "--synthetic", "60000", "--set", "neighborRadius=0.15", "--set", "displayNormals=false"],
                         capture_output=True, text=True, timeout=120)
    assert res.returncode == 0, res.stderr
    out = res.stdout.splitlines()
    i = out.index("Center Axis is:")
    axis = np.array([float(v) for v in out[i + 1].split()])
    assert abs(abs(axis[0]) - 1.0) < 1e-3 and np.abs(axis[1:]).max() < 3e-2
    j = out.index("Eigenvalues are:")
    vals = np.array([float(v) for v in out[j + 1].split()])
    assert vals[0] < 0.02 * vals[1] and vals[1] <= vals[2]                      # ascending, smallest ~ 0 for a cylinder
    assert any(l.startswith("publish cloudOutput:") for l in out) and any(l.startswith("publish eigenBasisOutput: 3 markers") for l in out)
    assert not any(l.startswith("publish normalsOutput") for l in out)


# ---- I/O seams ---------------------------------------------------------------------------------------
def test_pointcloud2_decode_velodyne_layout():
    """sensor_msgs/PointCloud2 as the Velodyne driver publishes it: point_step 22 (x,y,z,intensity f32 +
    ring u16 + time f32 would be 22 bytes, unaligned records) and a padded 32-byte layout."""
    pts = _scan_with_junk(20_000, seed=61)
    n = len(pts)
    for step, (ox, oy, oz) in ((22, (0, 4, 8)), (32, (4, 12, 20)), (12, (0, 4, 8))):
        raw = np.full((n, step), 0xAB, np.uint8)
        for k, o in enumerate((ox, oy, oz)):
            raw[:, o:o + 4] = pts[:, k].copy().view(np.uint8).reshape(n, 4)
        with _ctx(n, neighborRadius=0.2) as ctx:
            ctx.upload_pointcloud2(raw, n, step, ox, oy, oz)
            ctx.crop()
            got = ctx.download_cloud(0)
        ref, _ = O.crop(pts, 5.0, True)
        assert np.array_equal(got[:, :3].view(np.uint32), ref[:, :3].view(np.uint32)) and (got[:, 3] == 1.0).all()


def test_fetch_async_matches_synchronous_downloads():
    import ctypes as C

    n = 80_000
    pts = synth.curved_tunnel(n, seed=9)
    with _ctx(n, neighborRadius=0.12, voxelGridLeafSize=0.2) as ctx:
        ctx.upload_scan(pts)
        ctx.crop()
        ctx.normals()
        nv = ctx.counts().n_valid
        ps, cs = synth.sample_indices(nv, 256, 3, seed=3), synth.sample_indices(nv, 256, 2, seed=4)
        ctx.upload_scan(pts)
        ctx.process_scan(ps, cs)
        summ = capi.gm_scan_summary()
        cloud = np.zeros((n, 4), np.float32)
        normals = np.zeros((n, 8), np.float32)
        labels = np.zeros(n, np.uint8)
        slices = np.zeros(256, capi.SLICE_DTYPE)
        cen = np.zeros((n, 4), np.float32)
        nnn = np.zeros((n, 8), np.float32)
        o = capi.gm_host_outputs()
        o.summary = C.addressof(summ)
        o.cloud_xyzw, o.cloud_capacity = cloud.ctypes.data, n
        o.normals8, o.normals_capacity = normals.ctypes.data, n
        o.labels, o.labels_capacity = labels.ctypes.data, n
        o.slices, o.slices_capacity = slices.ctypes.data, 256
        o.centroids_xyzw, o.nn_normal8, o.voxel_capacity = cen.ctypes.data, nnn.ctypes.data, n
        ctx.fetch_async(o)
        ctx.synchronize()
        c = ctx.counts()
        assert (summ.counts.n_input, summ.counts.n_cropped, summ.counts.n_valid, summ.counts.n_voxels) == (c.n_input, c.n_cropped, c.n_valid, c.n_voxels)
        assert np.array_equal(cloud[:c.n_valid], ctx.download_cloud(1)) and np.array_equal(labels[:c.n_valid], ctx.download_labels())
        assert np.array_equal(normals[:c.n_valid].view(np.uint32), ctx.download_normals(1).view(np.uint32))
        vox = ctx.download_voxels()
        assert np.array_equal(cen[:c.n_voxels], vox["centroids"]) and np.array_equal(nnn[:c.n_voxels].view(np.uint32), vox["nn_normal"].view(np.uint32))
        fr, mp, mc, poly = ctx.frame(), ctx.model(0), ctx.model(1), ctx.download_polyline()
        assert np.array_equal(np.array(summ.frame.vals), fr["vals"]) and np.array_equal(np.array(summ.frame.vecs).reshape(3, 3), fr["vecs"])
        assert (summ.plane.best_id, summ.plane.best_count, summ.plane.refit_count) == (mp["best_id"], mp["best_count"], mp["refit_count"])
        assert np.array_equal(np.array(summ.plane.coef[:4]), mp["coef"]) and np.array_equal(np.array(summ.cylinder.coef[:7]), mc["coef"])
        assert summ.n_slices == len(poly) and slices[:len(poly)].tobytes() == poly.tobytes()


# ---- CUDA-graph replay of gm_process_scan ------------------------------------------------------------------
def _scan_outputs(ctx):
    keys, assign, _ = ctx.download_voxel_assignment()
    vox = ctx.download_voxels()
    fr = ctx.frame()
    _, _, pc = ctx.download_hypotheses(capi.GM_MODEL_PLANE, 256)
    _, _, cc = ctx.download_hypotheses(capi.GM_MODEL_CYLINDER, 256)
    return [ctx.download_cloud(1), ctx.download_normals(1), keys, assign, vox["centroids"], vox["nn_index"], fr["scatter"], fr["vals"],
            pc, cc, ctx.model(0)["coef"], ctx.model(1)["coef"], ctx.download_labels(), ctx.download_polyline()]


def test_graph_replay_reproduces_stream_launches_bit_for_bit():
    """Scans of different sizes inside one 32768-point bucket share ONE captured graph; every output of a replayed scan
    is bit-identical to the same scan processed with plain stream launches."""
    sizes = [60_000, 58_123, 61_440, 57_001, 60_000]
    scans = [synth.curved_tunnel(n, seed=40 + i) for i, n in enumerate(sizes)]
    ps = synth.sample_indices(50_000, 256, 3, seed=3)
    cs = synth.sample_indices(50_000, 256, 2, seed=4)
    ref = []
    with _ctx(65_536, neighborRadius=0.12) as ctx:
        ctx.set_graph_mode(0)
        for pts in scans:
            ctx.upload_scan(pts)
            ctx.process_scan(ps, cs)
            ref.append(_scan_outputs(ctx))
        assert ctx.graph_stats() == (0, 0)
    with _ctx(65_536, neighborRadius=0.12) as ctx:   # default graph mode = auto: these scans are below the size threshold
        for i, pts in enumerate(scans):
            ctx.upload_scan(pts)
            ctx.process_scan(ps, cs)
            got = _scan_outputs(ctx)
            assert ctx.counts().device_error == 0
            for a, b in zip(got, ref[i]):
                assert a.tobytes() == b.tobytes(), f"scan {i}"
        captures, replays = ctx.graph_stats()
        assert captures == 1 and replays == len(scans) - 1   # scan 0: plain launches; scan 1: captured + launched; 2..: replays
        # a parameter change starts a new generation: first scan eager again, same results as a fresh context
        p = ctx.params
        p.ransacThreshold = 0.08
        ctx.set_params(p)
        for _ in range(3):
            ctx.upload_scan(scans[0])
            ctx.process_scan(ps, cs)
        changed = _scan_outputs(ctx)
        assert ctx.graph_stats()[0] == 2
    with _ctx(65_536, neighborRadius=0.12, ransacThreshold=0.08) as ctx:
        ctx.set_graph_mode(0)
        ctx.upload_scan(scans[0])
        ctx.process_scan(ps, cs)
        for a, b in zip(changed, _scan_outputs(ctx)):
            assert a.tobytes() == b.tobytes()


# ---- peer-memory collectives with one rank (the multi-rank path needs one GPU per rank: tools/peer_check.py) -------
def test_sharded_round_and_map_collectives_with_a_single_rank():
    cloud, normals = _compacted_scan(60_000, seed=33)
    pts = synth.curved_tunnel(60_000, seed=33)
    ps = synth.sample_indices(50_000, 300, 3, seed=3)
    cs = synth.sample_indices(50_000, 200, 2, seed=4)
    with _ctx(len(pts), neighborRadius=0.15) as ctx, _ctx(len(pts), neighborRadius=0.15) as ref:
        comm = capi.PeerComm(0, 1)
        ctx.set_comm(comm)
        for c in (ctx, ref):
            c.upload_scan(pts)
            c.crop()
            c.normals()
        ref.ransac_pair(ps, cs)
        ref.ransac_select_pair()
        for _ in range(3):  # sequence numbers advance; slots are reused after 4 rounds
            ctx.ransac_sharded(ps, cs)
        for kind in (0, 1):
            a, b = ctx.model(kind), ref.model(kind)
            assert a["best_id"] == b["best_id"] and a["best_count"] == b["best_count"] and a["refit_count"] == b["refit_count"]
            assert np.array_equal(a["coef"].view(np.uint32), b["coef"].view(np.uint32))
        bb = ctx.voxel_bbox()
        ctx.allreduce_voxel_bbox()
        assert np.array_equal(np.concatenate(ctx.voxel_bbox()), np.concatenate(bb))
        for c in (ctx, ref):
            c.voxel()
            c.local_frame()
        ctx.allreduce_frame()
        fa, fb = ctx.frame(), ref.frame()
        assert np.array_equal(fa["scatter"], fb["scatter"]) and np.array_equal(fa["vals"], fb["vals"]) and np.array_equal(fa["vecs"], fb["vecs"])
        assert ctx.counts().device_error == 0
        ctx.set_comm(None)
        comm.close()


def test_cpp_host_shim_keeps_the_quirk_switches_of_the_parameters(tmp_path):
    """The per-call parameters of the seam (bound, radius, leaf, wf) are written into the context read-modify-write: the
    quirk switches installed with useParameters() survive them (a thread-local all-defaults cache used to reset them)."""
    import subprocess

    from geometric_mapping_b200 import build as gm_build

    exe = gm_build.build_host()
    pts = synth.straight_cylinder(40_000, seed=3, noise=0.01)
    path = str(tmp_path / "scan.f32x4")
    pts.tofile(path)
    args = [exe, "--set", "neighborRadius=0.2", "--set", "voxelGridLeafSize=0.5", "--set", "weightingFactor=0.25", "--scan", path]
    vals = {}
    for wm in (0, 1):
        res = subprocess.run(args + ["--set", f"weightMode={wm}", "--set", "arrowMode=1"], capture_output=True, text=True, timeout=120)
        assert res.returncode == 0, res.stderr
        assert f"context weight_mode {wm} arrow_mode 1" in res.stdout
        lines = res.stdout.splitlines()
        vals[wm] = np.array([float(v) for v in lines[lines.index("Eigenvalues are:") + 1].split()])
        with _ctx(len(pts), neighborRadius=0.2, voxelGridLeafSize=0.5, weightingFactor=0.25, weight_mode=wm) as ctx:
            ctx.upload_scan(pts)
            ctx.process_scan(None, None)
            assert np.allclose(vals[wm], ctx.frame()["vals"], rtol=1e-5)
    assert not np.allclose(vals[0], vals[1], rtol=1e-3)   # the two weight laws really differ


def test_primitive_store_persists_the_compressed_scans(tmp_path):
    """SURVEY 8f.3: the per-scan GMC1 blobs go to an append-only file and come back byte for byte after a reopen."""
    path = str(tmp_path / "run.gms")
    blobs = []
    with _ctx(60_000, neighborRadius=0.12) as ctx, capi.PrimitiveStore(path) as st:
        for f in range(3):
            pts = synth.curved_tunnel(60_000, seed=80 + f, advance=1.0 * f)
            ctx.upload_scan(pts)
            ctx.crop()
            ctx.normals()
            nv = ctx.counts().n_valid
            ctx.upload_scan(pts)
            ctx.process_scan(synth.sample_indices(nv, 128, 3, seed=3), synth.sample_indices(nv, 128, 2, seed=4))
            ctx.compress()
            blobs.append(ctx.download_compressed())
            st.append(ctx, scan_id=f, stamp_ns=100 * f, pose34=_pose(0.1 * f, [1.0 * f, 0, 0]))
    with capi.PrimitiveStore(path, create=False) as st:
        assert len(st) == 3
        for f in range(3):
            assert st.read(f) == blobs[f] and st.info(f)["scan_id"] == f
            assert np.allclose(st.info(f)["pose"], np.asarray(_pose(0.1 * f, [1.0 * f, 0, 0]), np.float32).reshape(3, 4))
