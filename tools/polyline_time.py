"""Time the axis polyline (gm_axis_polyline: k_poly_range, k_poly_pass<0>, k_poly_pass<2>) on one processed scan.

    python tools/polyline_time.py [--points N] [--calls K] [--slice-length L] [--max-slices S] [--out FILE]

The scan goes through gm_process_scan once; then the polyline stage runs K more times on it, back to back:
  * stage_ms   CUDA events around the K calls on the context's stream, per call (launch gaps included)
  * segment_ms the library's own `polyline` profile segment, per call
  * kernels_us per-kernel mean device time from torch.profiler, in a separate run of K calls
The inputs of the stage (48 MB at 1M points) stay in L2 between calls.  Prints one JSON line.
"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from geometric_mapping_b200 import capi, synth  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--points", type=int, default=1_000_000)
ap.add_argument("--radius", type=float, default=0.05)
ap.add_argument("--hyp", type=int, default=1024)
ap.add_argument("--calls", type=int, default=500)
ap.add_argument("--slice-length", type=float, default=1.0)
ap.add_argument("--max-slices", type=int, default=256)
ap.add_argument("--out", default=None)
a = ap.parse_args()

dev = torch.device("cuda", 0)
stream = torch.cuda.Stream(device=dev)
pts = synth.curved_tunnel(a.points, seed=2)
prm = capi.default_params(neighborRadius=a.radius, voxelGridLeafSize=0.1, sliceLength=a.slice_length, maxSlices=a.max_slices)
with capi.Context(prm, max_points=a.points, max_hypotheses=a.hyp) as ctx:
    ctx.set_stream(stream.cuda_stream)
    ctx.upload_scan(pts)
    ctx.crop()
    ctx.normals()
    nv = ctx.counts().n_valid
    ctx.upload_scan(pts)
    ctx.process_scan(synth.sample_indices(nv, a.hyp // 2, 3, seed=3), synth.sample_indices(nv, a.hyp - a.hyp // 2, 2, seed=4))
    n_cyl = int((ctx.download_labels() == 2).sum())
    for _ in range(20):
        ctx.axis_polyline()
    ctx.synchronize()

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(a.calls):
        ctx.axis_polyline()
    e1.record(stream)
    e1.synchronize()
    stage_ms = e0.elapsed_time(e1) / a.calls

    ctx.profile_enable(True)
    ctx.profile_read()
    for _ in range(a.calls):
        ctx.axis_polyline()
    ctx.synchronize()
    seg_ms, seg_calls = ctx.profile_read()["polyline"]
    ctx.profile_enable(False)

    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(a.calls):
            ctx.axis_polyline()
        ctx.synchronize()
    kernels = {}
    for ev in prof.key_averages():
        if "k_poly" in ev.key:
            name = "k_poly_range" if "k_poly_range" in ev.key else ("k_poly_pass<0>" if "ILi0E" in ev.key or "<0>" in ev.key else "k_poly_pass<2>")
            t = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0.0)
            kernels[name] = {"mean_us": t / max(ev.count, 1), "count": ev.count}
    poly = ctx.download_polyline()
    assert ctx.counts().device_error == 0

line = {"gpu": torch.cuda.get_device_name(0), "points": a.points, "n_valid": nv, "n_cylinder": n_cyl, "slices": len(poly),
        "calls": a.calls, "stage_ms": stage_ms, "segment_ms": seg_ms / max(seg_calls, 1), "kernels_us": kernels}
print(json.dumps(line))
if a.out:
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(json.dumps(line) + "\n")
