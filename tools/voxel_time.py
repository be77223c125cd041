"""Time the VoxelGrid stage (gm_voxel: dense accumulation + table scan + voxel 1-NN) and the on-demand per-point voxel
assignment (gm_download_voxel_assignment) on one processed scan.

    python tools/voxel_time.py [--points N] [--calls K] [--out FILE]

The scan goes through gm_process_scan once; then each call runs K more times on it, back to back:
  * voxel_ms        CUDA events around K gm_voxel calls on the context's stream, per call (launch gaps included)
  * segments_ms     the library's voxel_keys / voxel_reduce / voxel_nn profile segments of those calls, per call
  * assignment_ms   host clock around K gm_download_voxel_assignment calls (the key / id kernel, then a synchronous copy
                    of 8 B per point to pageable host memory), per call
  * kernels_us      per-kernel mean device time from torch.profiler, in a separate run of K calls of each
The inputs (the compacted and cell-sorted clouds, ~50 MB at 1M points) stay in L2 between calls.  Prints one JSON line.
"""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from geometric_mapping_b200 import capi, synth  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--points", type=int, default=1_000_000)
ap.add_argument("--radius", type=float, default=0.05)
ap.add_argument("--leaf", type=float, default=0.1)
ap.add_argument("--hyp", type=int, default=1024)
ap.add_argument("--calls", type=int, default=300)
ap.add_argument("--out", default=None)
a = ap.parse_args()

dev = torch.device("cuda", 0)
stream = torch.cuda.Stream(device=dev)
pts = synth.curved_tunnel(a.points, seed=2)
prm = capi.default_params(neighborRadius=a.radius, voxelGridLeafSize=a.leaf)
with capi.Context(prm, max_points=a.points, max_hypotheses=a.hyp) as ctx:
    ctx.set_stream(stream.cuda_stream)
    ctx.upload_scan(pts)
    ctx.crop()
    ctx.normals()
    nv = ctx.counts().n_valid
    ctx.upload_scan(pts)
    ctx.process_scan(synth.sample_indices(nv, a.hyp // 2, 3, seed=3), synth.sample_indices(nv, a.hyp - a.hyp // 2, 2, seed=4))
    for _ in range(20):
        ctx.voxel()
        ctx.download_voxel_assignment()
    ctx.synchronize()
    V = ctx.counts().n_voxels

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(a.calls):
        ctx.voxel()
    e1.record(stream)
    e1.synchronize()
    voxel_ms = e0.elapsed_time(e1) / a.calls

    t0 = time.perf_counter()
    for _ in range(a.calls):
        ctx.download_voxel_assignment()
    assignment_ms = (time.perf_counter() - t0) * 1e3 / a.calls

    ctx.profile_enable(True)
    ctx.profile_read()
    for _ in range(a.calls):
        ctx.voxel()
    ctx.synchronize()
    prof_seg = ctx.profile_read()
    ctx.profile_enable(False)
    segments = {k: prof_seg[k][0] / max(prof_seg[k][1], 1) for k in ("voxel_keys", "voxel_reduce", "voxel_nn") if k in prof_seg}

    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(a.calls):
            ctx.voxel()
        for _ in range(a.calls):
            ctx.download_voxel_assignment()
        ctx.synchronize()
    kernels = {}
    for ev in prof.key_averages():
        for name in ("k_voxel_accumulate_sorted", "k_voxel_dense_scan", "k_voxel_assign", "k_voxel_lookup", "k_voxel_nn"):
            if name + "(" in ev.key:  # demangled: "gm::k_voxel_nn(float4 const*, ...)"
                t = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0.0)
                kernels[name] = {"mean_us": t / max(ev.count, 1), "count": ev.count}
                break
    assert ctx.counts().device_error == 0

line = {"gpu": torch.cuda.get_device_name(0), "points": a.points, "n_valid": nv, "voxels": V, "calls": a.calls,
        "voxel_ms": voxel_ms, "segments_ms": segments, "assignment_ms": assignment_ms, "kernels_us": kernels}
print(json.dumps(line))
if a.out:
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(json.dumps(line) + "\n")
