"""Which results a context holds after each call: the stage-validity rules of gm_capi.cu, asserted through the
Python binding.  A getter of a stage that was never run, or whose input has since changed, fails with
GM_ERR_STAGE_ORDER; a getter of a stage that is still valid succeeds.
"""
import numpy as np
import pytest

from geometric_mapping_b200 import capi, synth

pytestmark = pytest.mark.gpu

N = 20_000
H = 128
PARAMS = dict(neighborRadius=0.15, voxelGridLeafSize=0.1)


def _ctx(**kw):
    return capi.Context(capi.default_params(**{**PARAMS, **kw}), max_points=N, max_hypotheses=H)


@pytest.fixture(scope="module")
def scan():
    return synth.curved_tunnel(N, seed=21)


@pytest.fixture(scope="module")
def samples(scan):
    with _ctx() as ctx:
        ctx.upload_scan(scan)
        ctx.crop()
        ctx.normals()
        nv = ctx.counts().n_valid
    return synth.sample_indices(nv, H, 3, seed=3), synth.sample_indices(nv, H, 2, seed=4)


def _status(fn):
    try:
        fn()
    except capi.GmError as e:
        return e.status
    return capi.GM_OK


def _raises_stage_order(fn):
    return _status(fn) == capi.GM_ERR_STAGE_ORDER


GETTERS = {
    "cloud0": lambda c: c.download_cloud(0),
    "cloud1": lambda c: c.download_cloud(1),
    "normals0": lambda c: c.download_normals(0),
    "normals1": lambda c: c.download_normals(1),
    "neighbor_counts": lambda c: c.download_neighbor_counts(),
    "valid_map": lambda c: c.download_valid_map(),
    "search_stats": lambda c: c.search_stats(),
    "voxel_bbox": lambda c: c.voxel_bbox(),
    "voxel_assignment": lambda c: c.download_voxel_assignment(),
    "voxels": lambda c: c.download_voxels(),
    "voxel_grid": lambda c: c.voxel_grid(),
    "frame": lambda c: c.frame(),
    "hyp_plane": lambda c: c.download_hypotheses(capi.GM_MODEL_PLANE, H),
    "hyp_cyl": lambda c: c.download_hypotheses(capi.GM_MODEL_CYLINDER, H),
    "model_plane": lambda c: c.model(capi.GM_MODEL_PLANE),
    "model_cyl": lambda c: c.model(capi.GM_MODEL_CYLINDER),
    "labels": lambda c: c.download_labels(),
    "polyline": lambda c: c.download_polyline(),
    "compression": lambda c: c.compression(),
}


def _getter_status(ctx):
    return {name: _status(lambda: fn(ctx)) for name, fn in GETTERS.items()}


def _counts(ctx):
    c = ctx.counts()
    return tuple(getattr(c, f) for f, _ in capi.gm_counts._fields_)


def test_new_crop_bound_invalidates_the_crop(scan):
    with _ctx() as ctx:
        ctx.upload_scan(scan)
        ctx.crop()
        ctx.normals()
        ctx.set_params(capi.default_params(**{**PARAMS, "boxFilterBound": 4.0}))
        assert _raises_stage_order(ctx.normals)
        assert _raises_stage_order(lambda: ctx.download_cloud(0))
        ctx.crop()
        ctx.normals()
        ctx.voxel()


def test_is_dense_change_invalidates_the_crop(scan):
    with _ctx() as ctx:
        ctx.upload_scan(scan)
        ctx.crop()
        ctx.set_params(capi.default_params(**{**PARAMS, "is_dense": 0}))
        assert _raises_stage_order(ctx.normals)
        ctx.crop()
        ctx.normals()


def test_grid_change_keeps_the_crop_and_drops_what_follows(scan, samples):
    ps, cs = samples
    with _ctx() as ctx:
        ctx.upload_scan(scan)
        ctx.process_scan(ps, cs)
        ctx.set_params(capi.default_params(**{**PARAMS, "neighborRadius": 0.2}))  # only the neighbour grid changes
        st = _getter_status(ctx)
        assert st["cloud0"] == capi.GM_OK
        assert all(s == capi.GM_ERR_STAGE_ORDER for k, s in st.items() if k != "cloud0"), st
        assert _raises_stage_order(ctx.voxel)
        assert _raises_stage_order(ctx.local_frame)
        c = ctx.counts()
        assert c.n_cropped >= 0 and c.n_valid == -1 and c.n_voxels == -1 and c.n_cells == -1
        ctx.normals()
        ctx.voxel()
        # gm_set_grid_box moves the grid the same way
        ctx.set_grid_box([-1.0, -1.0, -1.0], [1.0, 1.0, 1.0])
        assert _status(lambda: ctx.download_cloud(0)) == capi.GM_OK
        assert _raises_stage_order(ctx.voxel)


def test_identical_params_invalidate_nothing(scan, samples):
    ps, cs = samples
    with _ctx() as ctx:
        ctx.upload_scan(scan)
        ctx.process_scan(ps, cs)
        ctx.compress()
        before, counts = _getter_status(ctx), _counts(ctx)
        assert all(s != capi.GM_ERR_STAGE_ORDER for s in before.values()), before
        ctx.set_params(capi.default_params(**PARAMS))
        assert _getter_status(ctx) == before
        assert _counts(ctx) == counts


def test_rerunning_an_earlier_stage_keeps_later_ones(scan, samples):
    ps, cs = samples
    with _ctx() as ctx:
        ctx.upload_scan(scan)
        ctx.process_scan(ps, cs)
        before = _getter_status(ctx)
        ctx.crop()
        ctx.normals()
        assert _getter_status(ctx) == before


def test_injected_cloud_has_no_crop_or_search_results(scan):
    with _ctx() as ctx:
        ctx.upload_scan(scan)
        ctx.crop()
        ctx.normals()
        cloud, normals = ctx.download_cloud(1), ctx.download_normals(1)
    ps = synth.sample_indices(len(cloud), H, 3, seed=5)
    with _ctx() as ctx:
        ctx.inject_compacted(cloud, normals)
        ctx.voxel()
        ctx.local_frame()
        ctx.ransac(capi.GM_MODEL_PLANE, ps)
        ctx.ransac_select(capi.GM_MODEL_PLANE)
        assert _raises_stage_order(lambda: ctx.download_normals(0))
        assert _raises_stage_order(ctx.download_neighbor_counts)
        assert _raises_stage_order(lambda: ctx.download_cloud(0))
        assert _raises_stage_order(ctx.normals)
        c = ctx.counts()
        assert c.n_cropped == -1 and c.n_cells == -1 and c.n_valid == len(cloud) and c.n_voxels > 0
        # a grid change drops the injected cloud too
        ctx.set_params(capi.default_params(**{**PARAMS, "neighborRadius": 0.2}))
        assert _raises_stage_order(ctx.voxel)


@pytest.mark.parametrize("kind", [capi.GM_MODEL_PLANE, capi.GM_MODEL_CYLINDER])
def test_a_new_ransac_round_drops_its_model_until_selected(scan, samples, kind):
    ps, cs = samples
    with _ctx() as ctx:
        ctx.upload_scan(scan)
        ctx.process_scan(ps, cs)
        ctx.model(kind)
        ctx.ransac(kind, ps if kind == capi.GM_MODEL_PLANE else cs)
        assert _raises_stage_order(lambda: ctx.model(kind))
        ctx.model(1 - kind)  # the other primitive keeps its model
        ctx.download_hypotheses(kind, H)
        ctx.ransac_select(kind)
        ctx.model(kind)


def test_a_new_scan_drops_every_result(scan, samples):
    ps, cs = samples
    with _ctx() as ctx:
        ctx.upload_scan(scan)
        ctx.process_scan(ps, cs)
        ctx.compress()
        ctx.upload_scan(scan)
        assert _raises_stage_order(ctx.download_labels)
        assert all(s == capi.GM_ERR_STAGE_ORDER for s in _getter_status(ctx).values())
        c = ctx.counts()
        assert c.n_input == N and c.n_cropped == -1 and c.n_valid == -1 and c.n_voxels == -1 and c.n_cells == -1


def _process_three_times(mode, scan, ps, cs):
    with _ctx() as ctx:
        ctx.set_graph_mode(mode)
        for _ in range(3):
            ctx.upload_scan(scan)
            ctx.process_scan(ps, cs)
        after_scan = (_getter_status(ctx), _counts(ctx))
        # the compression result of the same scan survives another process_scan without a new upload
        ctx.compress()
        ctx.process_scan(ps, cs)
        after_compress = (_getter_status(ctx), _counts(ctx))
        for _ in range(3):  # no cylinder hypotheses: the cylinder round is not run
            ctx.upload_scan(scan)
            ctx.process_scan(ps, None)
        no_cyl = (_getter_status(ctx), _counts(ctx))
        return after_scan, after_compress, no_cyl, ctx.graph_stats()


def test_graph_replay_leaves_the_same_results_as_plain_launches(scan, samples):
    ps, cs = samples
    plain = _process_three_times(0, scan, ps, cs)
    graphed = _process_three_times(1, scan, ps, cs)
    assert plain[3] == (0, 0)
    captures, replays = graphed[3]
    assert captures >= 1 and replays >= 2
    for p, g in zip(plain[:3], graphed[:3]):
        assert p == g
    after_scan, after_compress, no_cyl = plain[:3]
    assert after_scan[0]["compression"] == capi.GM_ERR_STAGE_ORDER
    assert all(s != capi.GM_ERR_STAGE_ORDER for k, s in after_scan[0].items() if k != "compression"), after_scan[0]
    assert after_compress[0]["compression"] == capi.GM_OK
    assert no_cyl[0]["model_cyl"] == capi.GM_ERR_STAGE_ORDER and no_cyl[0]["hyp_cyl"] == capi.GM_ERR_STAGE_ORDER
    assert no_cyl[0]["model_plane"] == capi.GM_OK
