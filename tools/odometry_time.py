"""Time map odometry on the device (gm_odometry_step) against the host loop it replaces, and record the card it ran on.

Sequence: 16 scans of the drift (synth.drift_end_niche, 1M points, C1: neighbour radius 5 cm, leaf 10 cm), the sensor
advancing 0.1 m and turning 0.5 degrees per scan along the drift.  Two contexts take turns.  Both loops process every
scan (upload, crop, normals, voxel) and start from a new map:
  host loop:  gm_register_map from the last pose, gm_get_registration (a host synchronisation), gm_map_insert at the result;
  odometry:   gm_odometry_step with delta34 = the identity (the same guess, so the same ICP work as the host loop: the two
              trajectories are bit-identical); the host goes on to the next scan while the step runs;
  and gm_odometry_step with the constant-velocity guess (delta34 = NULL), timed the same way.
Reported: ms per scan (host clock over the 16 scans ending in a synchronise, median of --repeats after --warmup, the
loops alternating), whether the host loop and the identity-delta odometry agree bit for bit, the final pose errors and
iteration counts; then, from torch.profiler in a
separate pass, the device time per launch of k_odom_begin, k_odom_gate, k_map_insert_gated (and of the host loop's
k_map_insert for comparison).  The card's name and power limit are read in the same run.

    python tools/odometry_time.py --out profiles/r07_odometry_time.json
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
LEAF, DMAX, SCANS = 0.1, 0.5, 16
KERNELS = ("k_odom_begin", "k_odom_gate", "k_map_insert_gated", "k_map_insert", "k_map_planes", "k_regmap_iter")


def _card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        name, power, clock = (s.strip() for s in q.stdout.strip().splitlines()[0].split(","))
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # the timing itself needs no nvidia-smi
        return {"error": repr(e)}


def _pose_error(P, T):
    dR = np.asarray(P, np.float64)[:, :3] @ T[:, :3].T
    s = 0.5 * np.linalg.norm([dR[2, 1] - dR[1, 2], dR[0, 2] - dR[2, 0], dR[1, 0] - dR[0, 1]])
    ang = float(np.arctan2(s, (np.trace(dR) - 1.0) / 2.0))
    return ang, float(np.linalg.norm(np.asarray(P, np.float64)[:, 3] - T[:, 3]))


def _scan(ctx, pts):
    ctx.upload_scan(pts)
    ctx.crop()
    ctx.normals()
    ctx.voxel()


def host_loop(ctxs, scans, truth):
    with capi.VoxelMap(LEAF, 1 << 20) as vmap:
        t0 = time.perf_counter()
        _scan(ctxs[0], scans[0])
        pose = truth[0].astype(np.float32)
        vmap.insert(ctxs[0], pose)
        poses = [pose]
        for k in range(1, len(scans)):
            ctx = ctxs[k % 2]
            _scan(ctx, scans[k])
            pose = ctx.register_map(vmap, pose, max_correspondence_distance=DMAX)["pose"]   # synchronises
            vmap.insert(ctx, pose)
            poses.append(pose)
        for c in ctxs:
            c.synchronize()
        dt = time.perf_counter() - t0
    return dt, np.array(poses, np.float32)


def odometry(ctxs, scans, truth, velocity=False):
    eye = np.eye(3, 4, dtype=np.float32)
    with capi.VoxelMap(LEAF, 1 << 20) as vmap:
        with capi.Odometry(vmap, truth[0], max_correspondence_distance=DMAX) as odo:
            t0 = time.perf_counter()
            for k in range(len(scans)):
                ctx = ctxs[k % 2]
                _scan(ctx, scans[k])
                odo.step(ctx, None if velocity or k == 0 else eye)
            traj = odo.trajectory()                              # synchronises
            for c in ctxs:
                c.synchronize()
            dt = time.perf_counter() - t0
    return dt, traj


def _kernel_ms(fn):
    import torch
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        for k in KERNELS:
            name = e.key.split("(")[0].split("::")[-1].split("<")[0].strip()
            if name == k:
                dev_us = getattr(e, "device_time_total", None)
                if dev_us is None:
                    dev_us = e.cuda_time_total
                out[k] = {"launches": e.count, "ms_mean": dev_us / 1e3 / max(e.count, 1)}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--repeats", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("odometry_time: no CUDA device (the library has no CPU path)")
    truth = [synth.pose34(np.radians((0.0, 0.0, 0.5 * k)), (-0.75 + 0.1 * k, 0.01 * k, 0.0)) for k in range(SCANS)]
    scans = [synth.second_scan(synth.drift_end_niche, truth[k], seed=100 + k, n=a.n) for k in range(SCANS)]
    res = {"card": _card(), "scene": "drift_end_niche", "n_points": a.n, "scans": SCANS, "contexts": 2,
           "motion_per_scan": {"advance_m": 0.1, "yaw_deg": 0.5, "lateral_m": 0.01},
           "icp": {"max_correspondence_distance": DMAX, "max_iterations": 30, "max_planarity": 0.1},
           "method": "host clock over the whole sequence (scan processing included) ending in a synchronise, per scan; "
                     "median of repeats after warm-up, the two loops alternating; kernel times: torch.profiler device "
                     "time per launch over one odometry sequence and one host-loop sequence in a separate pass"}
    with capi.Context(capi.default_params(**C1), max_points=a.n, max_hypotheses=16) as c0, \
            capi.Context(capi.default_params(**C1), max_points=a.n, max_hypotheses=16) as c1:
        ctxs = [c0, c1]
        for _ in range(a.warmup):
            host_loop(ctxs, scans, truth)
            odometry(ctxs, scans, truth)
        times = {"host_loop": [], "odometry_step": [], "odometry_step_constant_velocity": []}
        for _ in range(a.repeats):
            dt, host_poses = host_loop(ctxs, scans, truth)
            times["host_loop"].append(dt * 1e3 / SCANS)
            dt, traj = odometry(ctxs, scans, truth)
            times["odometry_step"].append(dt * 1e3 / SCANS)
            dt, vel = odometry(ctxs, scans, truth, velocity=True)
            times["odometry_step_constant_velocity"].append(dt * 1e3 / SCANS)
        for key, t in times.items():
            res[key] = {"ms_per_scan_median": float(np.median(t)), "ms_min": float(np.min(t)), "ms_max": float(np.max(t))}
        res["host_minus_odometry_ms_per_scan"] = res["host_loop"]["ms_per_scan_median"] - res["odometry_step"]["ms_per_scan_median"]
        res["host_loop_and_odometry_bit_identical"] = bool(np.array_equal(host_poses.view(np.uint32), traj["poses"].view(np.uint32)))
        for key, t in (("odometry_step", traj), ("odometry_step_constant_velocity", vel)):
            rot, trans = _pose_error(t["poses"][-1], truth[-1])
            res[key].update(final_rotation_error_rad=rot, final_translation_error_m=trans, accepted=t["accepted"].tolist(),
                            iterations=t["iterations"].tolist(), fitness=[float(f) for f in t["fitness"]])
        res["kernels_odometry"] = _kernel_ms(lambda: odometry(ctxs, scans, truth))
        res["kernels_host_loop"] = _kernel_ms(lambda: host_loop(ctxs, scans, truth))
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
