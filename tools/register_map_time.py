"""Time gm_register_map on the device and record the card it ran on.

Drift: a map of four 1M-point drift scans (synth.drift_end_niche, C1: neighbour radius 5 cm, leaf 10 cm) inserted at
their sensor poses, and the voxel centroids of a fifth 1M-point scan from a known sensor pose as the source, registered
from the identity at max_planarity 0.1.  Reported: ms per gm_register_map at max_iterations 10 and 30 (host clock around
the call and a synchronise of the source stream, median of --repeats after --warmup), iterations taken, V, the map's
voxels and planes, correspondences and the pose error; then, from torch.profiler in a separate pass, the mean device time
of k_map_planes, k_reg_begin and k_regmap_iter.
C4: a map of the 10M-point, 100 m tunnel (synth.tunnel_map, box 60 m) inserted in one go, and the device time of
k_map_planes at its voxel count (gm_register_map of an empty source, one iteration, under torch.profiler).
The card's name and power limit are read in the same run.

    python tools/register_map_time.py --out profiles/r06_register_map_time.json
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
KERNELS = ("k_map_planes", "k_reg_begin", "k_regmap_iter")


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


def _kernel_ms(fn, calls):
    """mean device time per launch (ms) and launches of the kernels in KERNELS over `calls` calls of fn, torch.profiler"""
    import torch
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            fn()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        for k in KERNELS:
            if k in e.key:
                dev_us = getattr(e, "device_time_total", None)
                if dev_us is None:
                    dev_us = e.cuda_time_total
                out[k] = {"launches": e.count, "ms_mean": dev_us / 1e3 / max(e.count, 1)}
    return out


def drift(n, repeats, warmup):
    T = synth.pose34(np.radians((2.0, -1.5, 3.0)), (0.2, -0.1, 0.05))
    poses = [synth.pose34(np.radians((0.0, 0.0, d)), (x, y, 0.0)) for d, x, y in
             ((0.0, 0.0, 0.0), (2.0, 0.15, 0.03), (-2.0, -0.15, -0.03), (1.0, 0.3, -0.02))]
    out = {"scene": "drift_end_niche", "n_points": n, "map_scans": len(poses), "true_t": T[:, 3].tolist(), "max_planarity": 0.1}
    with capi.Context(capi.default_params(**C1), max_points=n, max_hypotheses=16) as ins, \
            capi.Context(capi.default_params(**C1), max_points=n, max_hypotheses=16) as src, capi.VoxelMap(0.1, 1 << 20) as vmap:
        for k, P in enumerate(poses):
            _scan(ins, synth.second_scan(synth.drift_end_niche, P, seed=40 + k, n=n))
            vmap.insert(ins, P)
        _scan(src, synth.second_scan(synth.drift_end_niche, T, seed=9, n=n))
        pl = vmap.planes(0.1)
        out["map_voxels"], out["map_planes"] = int(len(pl)), int((pl[:, 3] == 1).sum())
        for iters in (10, 30):
            for _ in range(warmup):
                src.register_map(vmap, np.eye(3, 4), max_iterations=iters)
            times = []
            for _ in range(repeats):
                src.synchronize()
                t0 = time.perf_counter()
                src.register_map_async(vmap, np.eye(3, 4), max_iterations=iters)
                src.synchronize()
                times.append((time.perf_counter() - t0) * 1e3)
            g = src.registration()
            rot, trans = _pose_error(g["pose"], T)
            ms = float(np.median(times))
            out[f"max_iterations_{iters}"] = {
                "ms_per_register_median": ms, "ms_min": float(np.min(times)), "ms_max": float(np.max(times)),
                "iterations": g["iterations"], "converged": g["converged"], "ms_per_executed_iteration": ms / max(g["iterations"], 1),
                "V": g["n_source"], "correspondences": g["n_correspondences"], "rmse": g["rmse"], "fitness": g["fitness"],
                "rotation_error_rad": rot, "translation_error_m": trans}
        out["kernels_max_iterations_30"] = _kernel_ms(lambda: src.register_map_async(vmap, np.eye(3, 4), max_iterations=30), repeats)
    return out


def c4(n, repeats):
    p = capi.default_params(boxFilterBound=60.0, **C1)
    out = {"scene": "tunnel_map_C4", "n_points": n}
    with capi.Context(p, max_points=n, max_hypotheses=16) as ins, capi.VoxelMap(0.1, 1 << 23) as vmap, \
            capi.Context(capi.default_params(**C1), max_points=1000, max_hypotheses=16) as empty:
        ins.upload_scan(synth.tunnel_map(n, seed=4, bound=60.0))
        ins.crop()
        ins.normals()
        vmap.insert(ins)
        _scan(empty, np.zeros((0, 4), np.float32))
        pl = vmap.planes(0.1)
        out["map_voxels"], out["map_planes_at_0.1"] = int(len(pl)), int((pl[:, 3] == 1).sum())
        empty.register_map(vmap, np.eye(3, 4), max_iterations=1)
        out["kernels"] = _kernel_ms(lambda: empty.register_map_async(vmap, np.eye(3, 4), max_iterations=1), repeats)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--c4-n", type=int, default=10_000_000)
    ap.add_argument("--repeats", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("register_map_time: no CUDA device (the library has no CPU path)")
    res = {"card": _card(), "true_rotvec_deg": [2.0, -1.5, 3.0],
           "method": "host clock around gm_register_map + gm_synchronize, median of repeats after warm-up; kernel times: "
                     "torch.profiler device time per launch in a separate pass",
           "scenes": [drift(a.n, a.repeats, a.warmup), c4(a.c4_n, a.repeats)]}
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
