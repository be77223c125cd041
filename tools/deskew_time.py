"""Time the deskew path on the device and record the card it ran on.

  k_deskew alone (gm_deskew on a fresh timed upload, CUDA events around the call) at 1M and 10M points, --reps launches
    each: 36 bytes a point (16 read, 4 read, 16 written) over the median time, against the 7.7 TB/s of HBM.  A 1M-point
    scan (36 MB) has just been written by the upload and runs from the 126 MB L2; 10M points (360 MB) do not fit.  The
    same launches with every time non-finite move the same bytes without the double-precision arithmetic: the gap
    between the two is what the arithmetic costs.
  The timed against the untimed PointCloud2 upload (H2D copy of 32-byte records + decode) at 1M points, alternating.
  Map odometry on 16 swept 1M-point drift scans (synth.swept_scan of synth.drift_end_niche, C1: neighbour radius 5 cm,
    leaf 10 cm; 0.15 m and 1 degree of yaw per 0.1 s sweep), two contexts taking turns, constant-velocity guess:
      none:      timed upload, no deskew;
      given:     gm_deskew with the true motion (what an IMU gives; keeps the overlap of two contexts);
      odometry:  gm_odometry_deskew (waits for the previous step), after the first two scans deskewed as in "given"
                 (the trajectory has no velocity before step 2).
    ms per scan = host clock over the 16 scans ending in a synchronise, median of --repeats after a warm-up, the modes
    alternating; the largest per-step pose errors of each mode.

    python tools/deskew_time.py --out profiles/r10_deskew.json
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from geometric_mapping_b200 import capi, synth  # noqa: E402

C1 = dict(neighborRadius=0.05, voxelGridLeafSize=0.1)
LEAF, DMAX, PERIOD, SCANS = 0.1, 0.5, 0.1, 16
VELODYNE = (32, 0, 4, 8, 24)
HBM_TBS = 7.7
MOTION = synth.pose34((0.0, 0.0, np.radians(1.0)), (0.15, 0.005, 0.0))


def _card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        name, power, clock = (s.strip() for s in q.stdout.strip().splitlines()[0].split(","))
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # the timing itself needs no nvidia-smi
        return {"error": repr(e)}


def _records(xyzw, t):
    step, ox, oy, oz, ot = VELODYNE
    raw = np.zeros((len(t), step), np.uint8)
    for off, col in ((ox, xyzw[:, 0]), (oy, xyzw[:, 1]), (oz, xyzw[:, 2]), (ot, t)):
        raw[:, off:off + 4] = np.ascontiguousarray(col, np.float32).view(np.uint8).reshape(len(t), 4)
    return raw


def _h(P):
    return np.vstack([np.asarray(P, np.float64)[:3, :4], [0.0, 0.0, 0.0, 1.0]])


def _pose_error(P, T):
    dR = np.asarray(P, np.float64)[:, :3] @ T[:, :3].T
    s = 0.5 * np.linalg.norm([dR[2, 1] - dR[1, 2], dR[0, 2] - dR[2, 0], dR[1, 0] - dR[0, 1]])
    return float(np.arctan2(s, (np.trace(dR) - 1.0) / 2.0)), float(np.linalg.norm(np.asarray(P, np.float64)[:, 3] - T[:, 3]))


def _kernel(torch, n, reps, nan_times):
    xyzw, t = synth.swept_scan(synth.curved_tunnel, np.eye(3, 4), MOTION, PERIOD, seed=2, n=1_000_000)
    k = -(-n // len(t))
    xyzw, t = np.tile(xyzw, (k, 1))[:n], np.tile(t, k)[:n]
    if nan_times:
        t = np.full(n, np.nan, np.float32)
    raw = _records(xyzw, t)
    stream = torch.cuda.Stream()
    ms = []
    with capi.Context(capi.default_params(**C1), max_points=n, max_hypotheses=16) as ctx:
        ctx.set_stream(stream.cuda_stream)
        d = MOTION.astype(np.float32)
        for i in range(reps + 5):
            ctx.upload_pointcloud2_timed(raw, n, *VELODYNE)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            ctx.deskew(d, 0.0, PERIOD)
            e1.record(stream)
            e1.synchronize()
            if i >= 5:
                ms.append(e0.elapsed_time(e1))
        ctx.set_stream(None)
    med = float(np.median(ms))
    return {"points": n, "launches": reps, "median_ms": med, "min_ms": float(np.min(ms)), "mean_ms": float(np.mean(ms)),
            "bytes": 36 * n, "achieved_TBps": 36 * n / (med * 1e-3) / 1e12, "share_of_hbm": 36 * n / (med * 1e-3) / 1e12 / HBM_TBS}


def _upload(torch, reps):
    n = 1_000_000
    xyzw, t = synth.swept_scan(synth.curved_tunnel, np.eye(3, 4), MOTION, PERIOD, seed=2, n=n)
    raw = _records(xyzw, t)
    stream = torch.cuda.Stream()
    out = {"timed": [], "untimed": []}
    with capi.Context(capi.default_params(**C1), max_points=n, max_hypotheses=16) as ctx:
        ctx.set_stream(stream.cuda_stream)
        for i in range(reps + 5):
            for kind in ("untimed", "timed"):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                if kind == "timed":
                    ctx.upload_pointcloud2_timed(raw, n, *VELODYNE)
                else:
                    ctx.upload_pointcloud2(raw, n, *VELODYNE[:4])
                e1.record(stream)
                e1.synchronize()
                if i >= 5:
                    out[kind].append(e0.elapsed_time(e1))
        ctx.set_stream(None)
    return {"points": n, "point_step": VELODYNE[0], "reps": reps,
            **{k + "_median_ms": float(np.median(v)) for k, v in out.items()}}


def _odometry_run(ctxs, raws, truth, mode):
    vmap = capi.VoxelMap(LEAF, 1 << 18)
    d = MOTION.astype(np.float32)
    with capi.Odometry(vmap, truth[0], max_correspondence_distance=DMAX) as odo:
        for c in ctxs:
            c.synchronize()
        t0 = time.perf_counter()
        for k in range(SCANS):
            ctx = ctxs[k % 2]
            ctx.upload_pointcloud2_timed(raws[k], len(raws[k]), *VELODYNE)
            if mode == "given" or (mode == "odometry" and k < 2):
                ctx.deskew(d, 0.0, PERIOD)
            elif mode == "odometry":
                odo.deskew(ctx, 0.0, PERIOD)
            ctx.crop()
            ctx.normals()
            ctx.voxel()
            odo.step(ctx)
        for c in ctxs:
            c.synchronize()
        ms = (time.perf_counter() - t0) * 1e3 / SCANS
        traj = odo.trajectory()
    vmap.close()
    err = np.array([_pose_error(traj["poses"][k], truth[k]) for k in range(1, SCANS)])
    return ms, {"max_rot_rad": float(err[:, 0].max()), "max_trans_m": float(err[:, 1].max()),
                "accepted": int(traj["accepted"].sum())}


def _odometry(repeats):
    start = _h(synth.pose34((0.0, 0.0, 0.0), (-1.2, 0.0, 0.0)))
    truth = [(start @ np.linalg.matrix_power(_h(MOTION), k))[:3] for k in range(SCANS)]
    raws = [_records(*synth.swept_scan(synth.drift_end_niche, truth[k], MOTION, PERIOD, seed=100 + k, n=1_000_000))
            for k in range(SCANS)]
    modes = ("none", "given", "odometry")
    ctxs = [capi.Context(capi.default_params(**C1), max_points=1 << 20, max_hypotheses=16) for _ in range(2)]
    times, errors = {m: [] for m in modes}, {}
    try:
        for m in modes:                                          # warm-up: buffers, first registrations
            _odometry_run(ctxs, raws, truth, m)
        for _ in range(repeats):
            for m in modes:
                ms, errors[m] = _odometry_run(ctxs, raws, truth, m)
                times[m].append(ms)
    finally:
        for c in ctxs:
            c.close()
    return {"scans": SCANS, "points": 1_000_000, "contexts": 2, "repeats": repeats,
            **{m: {"ms_per_scan_median": float(np.median(times[m])), "ms_per_scan": times[m], **errors[m]} for m in modes}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="JSON file to write (default: print only)")
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--repeats", type=int, default=5)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: nothing to measure")
    res = {"card": _card(), "torch_device": torch.cuda.get_device_name(0), "hbm_TBps": HBM_TBS}
    res["k_deskew"] = [_kernel(torch, n, a.reps, False) for n in (1_000_000, 10_000_000)]
    res["k_deskew_nonfinite_times"] = [_kernel(torch, n, a.reps, True) for n in (1_000_000, 10_000_000)]
    res["upload_1m"] = _upload(torch, a.reps)
    res["odometry"] = _odometry(a.repeats)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
