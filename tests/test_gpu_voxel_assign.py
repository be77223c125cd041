"""Per-point voxel keys and ids (gm_download_voxel_assignment) against the oracle on every path that produces them: the
dense VoxelGrid computes them only when they are downloaded, the sort-based one (voxel mode 1, injected or overflowing
clouds) writes them as it goes.  And the voxel 1-NN where the centroid's own cell does not settle it: sparse clouds
whose centroids lie in empty cells or several cells away from every point."""
import numpy as np
import pytest

from geometric_mapping_b200 import capi, synth
from oracle import oracle as O

pytestmark = pytest.mark.gpu

LEAF = 0.1


def _ctx(n, **kw):
    return capi.Context(capi.default_params(**kw), max_points=max(n, 1), max_hypotheses=512)


def _assert_assignment(ctx):
    keys, assign, st = ctx.download_voxel_assignment()
    ref = O.voxel(ctx.download_cloud(1), LEAF)
    assert st == capi.GM_OK and ctx.counts().device_error == 0
    assert np.array_equal(keys, ref["keys"]) and np.array_equal(assign, ref["assign"])


def _samples(nv):
    return synth.sample_indices(nv, 128, 3, seed=3), synth.sample_indices(nv, 128, 2, seed=4)


def test_after_voxel_and_again_after_compress():
    """Dense path: computed on download, right after voxel(), and still right after compress() has run its own dense
    VoxelGrid over the residual cloud (which rewrites the per-key id table the scan's voxels came from)."""
    pts = synth.curved_tunnel(60_000, seed=5)
    with _ctx(len(pts), neighborRadius=0.12, voxelGridLeafSize=LEAF) as ctx:
        ctx.upload_scan(pts)
        ctx.crop()
        ctx.normals()
        ctx.voxel()
        _assert_assignment(ctx)
        ps, cs = _samples(ctx.counts().n_valid)
        ctx.process_scan(ps, cs)
        ctx.compress()
        assert ctx.compression() is not None
        _assert_assignment(ctx)
        _assert_assignment(ctx)  # a second download computes the same arrays


def test_after_graph_replayed_scans():
    """process_scan replayed from a captured graph leaves the assignment to the download as well; a sort-path
    VoxelGrid of an injected cloud in between (which does write the per-point arrays) must not be taken for it."""
    scans = [synth.curved_tunnel(n, seed=50 + i) for i, n in enumerate((60_000, 58_000, 61_000, 59_500))]
    ps, cs = _samples(50_000)
    with _ctx(65_536, neighborRadius=0.12, voxelGridLeafSize=LEAF) as ctx:
        for i, pts in enumerate(scans):
            ctx.upload_scan(pts)
            ctx.process_scan(ps, cs)
            _assert_assignment(ctx)
            if i == 2:
                ctx.inject_compacted(synth.straight_cylinder(20_000, seed=8))
                ctx.voxel()
                _assert_assignment(ctx)
        captures, replays = ctx.graph_stats()
        assert captures == 1 and replays == len(scans) - 1


def test_voxel_mode_1_and_back():
    pts = synth.curved_tunnel(50_000, seed=6)
    with _ctx(len(pts), neighborRadius=0.12, voxelGridLeafSize=LEAF) as ctx:
        for mode in (1, 0, 1):
            ctx.set_voxel_mode(mode)
            ctx.upload_scan(pts)
            ctx.crop()
            ctx.normals()
            ctx.voxel()
            _assert_assignment(ctx)


def test_overflowing_lattice():
    """dx*dy*dz > INT32_MAX: pcl::VoxelGrid returns the cloud unchanged (the oracle then defines no keys), here every
    point is its own voxel: key = voxel id = point index."""
    big = synth.straight_cylinder(5000, seed=9)
    with _ctx(len(big), voxelGridLeafSize=0.001) as ctx:
        ctx.inject_compacted(big)
        ctx.voxel()
        keys, assign, st = ctx.download_voxel_assignment()
        c = ctx.counts()
    assert O.voxel(big, 0.001)["status"] == 1
    assert st == capi.GM_WARN_VOXEL_OVERFLOW and c.voxel_overflow == 1 and c.n_voxels == len(big) and c.device_error == 0
    assert np.array_equal(keys, np.arange(len(big), dtype=np.int32)) and np.array_equal(assign, keys)


def _sparse_clusters(seed):
    """Small planar clusters (valid normals) scattered through 1 m voxels, two or three per voxel so that centroids fall
    between them, plus lone points whose normals are NaN (candidates of nn_index_mode 0 only)."""
    g = np.random.Generator(np.random.Philox(seed))
    out = []
    for v in g.choice(8 ** 3, 120, replace=False):
        base = np.array([v % 8, (v // 8) % 8, v // 64], np.float64) - 4.0
        for _ in range(g.integers(2, 4)):
            centre = base + g.uniform(0.05, 0.95, 3)
            patch = g.uniform(-0.01, 0.01, (5, 3))
            patch[:, 2] = 0.0
            out.append(centre + patch)
    out.append(g.uniform(-4.0, 4.0, (400, 3)))
    pts = np.concatenate(out)
    return np.concatenate([pts, np.ones((len(pts), 1))], 1).astype(np.float32)


@pytest.mark.parametrize("nn_index_mode", [0, 1])
def test_nn_beyond_the_centroid_cell(nn_index_mode):
    pts = _sparse_clusters(17)
    radius = 0.05
    with _ctx(len(pts), neighborRadius=radius, voxelGridLeafSize=1.0, nn_index_mode=nn_index_mode) as ctx:
        ctx.upload_scan(pts)
        ctx.crop()
        ctx.normals()
        ctx.voxel()
        cropped = ctx.download_cloud(0)
        cloud_c = ctx.download_cloud(1)
        normals_c = ctx.download_normals(1)
        vox = ctx.download_voxels()
        c = ctx.counts()
    assert c.device_error == 0 and 0 < c.n_valid < c.n_cropped
    if nn_index_mode == 0:
        search = cropped.copy()
        search[~np.isfinite(cropped[:, :3]).all(1), :3] = 1e30
    else:
        search = cloud_c
    ref_idx, ref_d2 = O.nn1(vox["centroids"], search)
    cell = radius * (1 + 1 / 256)
    assert (ref_d2 > (2 * cell) ** 2).sum() > 10 and (ref_d2 < cell ** 2).any()  # many need ring 2 or more
    assert np.array_equal(vox["nn_index"], ref_idx)
    inr = ref_idx < c.n_valid
    assert np.array_equal(vox["nn_normal"][inr].view(np.uint32), normals_c[ref_idx[inr]].view(np.uint32))
    assert c.nn_out_of_range == int((~inr).sum())
    if nn_index_mode == 1:
        assert inr.all()
