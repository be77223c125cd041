"""The map calls that take no context run on the map's device whatever device is current.

A map made and filled with device 0 current is read, saved, merged into a second device-0 map, cleared and closed, once
with device 0 current and once with device 1 current: the results are the same, the saved files are byte-identical,
and every call leaves device 1 current."""
import numpy as np
import pytest

from geometric_mapping_b200 import capi, synth

pytestmark = pytest.mark.gpu

LEAF, RATIO, N = 0.1, 0.1, 200_000
POSES = [synth.pose34((0.0, 0.0, 0.0), (0.0, 0.0, 0.0)), synth.pose34((0.0, 0.0, 0.12), (1.3, 0.4, -0.1)),
         synth.pose34((0.0, 0.05, -0.2), (-2.2, -0.3, 0.2))]


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _calls(ctx, current, path):
    import torch

    with torch.cuda.device(0):                       # the maps and the inserts on device 0
        a, b = capi.VoxelMap(LEAF, 1 << 18), capi.VoxelMap(LEAF, 1 << 18)
        a.insert(ctx, POSES[0])
        a.insert(ctx, POSES[1])
        b.insert(ctx, POSES[2])
    out = {}
    with torch.cuda.device(current):
        for name, fn in (("stats", a.stats), ("download", a.download), ("planes", lambda: a.planes(RATIO)),
                         ("save", lambda: a.save(str(path / "a.gmm"))), ("merge", lambda: b.merge(a)),
                         ("merged_stats", b.stats), ("merged_save", lambda: b.save(str(path / "b.gmm"))),
                         ("clear", a.clear), ("cleared_stats", a.stats), ("close", a.close), ("close_merged", b.close)):
            out[name] = fn()
            assert torch.cuda.current_device() == current, name
    out["files"] = [(path / n).read_bytes() for n in ("a.gmm", "b.gmm")]
    return out


def test_map_calls_run_on_the_maps_device(tmp_path):
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    with torch.cuda.device(0):
        ctx = capi.Context(capi.default_params(neighborRadius=0.05, voxelGridLeafSize=LEAF), max_points=N, max_hypotheses=16)
    with ctx:
        with torch.cuda.device(0):
            ctx.upload_scan(synth.curved_tunnel(N, seed=2))
            ctx.crop()
            ctx.normals()
        (tmp_path / "d0").mkdir()
        (tmp_path / "d1").mkdir()
        ref = _calls(ctx, 0, tmp_path / "d0")
        got = _calls(ctx, 1, tmp_path / "d1")
    assert ref["stats"][0] > 0 and (ref["planes"][:, 3] == 1.0).sum() > 0 and ref["cleared_stats"] == (0, 0, 0, False)
    assert ref["merged_stats"][0] > ref["stats"][0]
    for key in ("stats", "merge", "merged_stats", "cleared_stats", "files"):
        assert got[key] == ref[key], key
    for key in ("ijk", "counts"):
        assert np.array_equal(got["download"][key], ref["download"][key]), key
    assert np.array_equal(_bits(got["download"]["centroids"]), _bits(ref["download"]["centroids"]))
    assert np.array_equal(_bits(got["planes"]), _bits(ref["planes"]))
