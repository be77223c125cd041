"""Time gm_register on 1M-point targets and record the card it ran on.

For each scene -- the six-DoF drift with an end face and a niche (synth.drift_end_niche) and the C1 curved tunnel --
the target is a 1M-point scan at the origin (crop, normals, voxel at C1: neighbour radius 5 cm, leaf 10 cm).  The source
is the voxel centroids of a second 1M-point scan of the same scene (another seed) taken from a known sensor pose.  The
registration starts from the identity.  Reported per scene: ms per gm_register at max_iterations 10 and 30 (host clock
around the call and a synchronise of the source stream, median of --repeats after --warmup; the target is untouched), ms
per executed iteration, iterations taken, V, correspondences, and the pose error against the known offset.  The card's
name and power limit are read in the same run.

    python tools/register_time.py --out profiles/r05_register_time.json
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


def run_scene(name, gen, T, n, repeats, warmup, d_max):
    kw = dict(neighborRadius=0.05, voxelGridLeafSize=0.1)
    out = {"scene": name, "n_points": n, "true_t": T[:, 3].tolist(), "d_max": d_max}
    with capi.Context(capi.default_params(**kw), max_points=n, max_hypotheses=16) as tgt, \
            capi.Context(capi.default_params(**kw), max_points=n, max_hypotheses=16) as src:
        _scan(tgt, gen(n, seed=8))
        _scan(src, synth.second_scan(gen, T, seed=9, n=n))
        for iters in (10, 30):
            for _ in range(warmup):
                src.register(tgt, np.eye(3, 4), max_iterations=iters, max_correspondence_distance=d_max)
            times = []
            for _ in range(repeats):
                src.synchronize()
                tgt.synchronize()
                t0 = time.perf_counter()
                src.register_async(tgt, np.eye(3, 4), max_iterations=iters, max_correspondence_distance=d_max)
                src.synchronize()
                times.append((time.perf_counter() - t0) * 1e3)
            g = src.registration()
            rot, trans = _pose_error(g["pose"], T)
            ms = float(np.median(times))
            out[f"max_iterations_{iters}"] = {
                "ms_per_register_median": ms, "ms_min": float(np.min(times)), "ms_max": float(np.max(times)),
                "iterations": g["iterations"], "converged": g["converged"], "ms_per_executed_iteration": ms / max(g["iterations"], 1),
                "V": g["n_source"], "correspondences": g["n_correspondences"], "rmse": g["rmse"], "fitness": g["fitness"],
                "rotation_error_rad": rot, "translation_error_m": trans,
                "eigenvalues": [float(v) for v in g["eigenvalues"]]}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--repeats", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--d-max", type=float, default=0.5)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("register_time: no CUDA device (the library has no CPU path)")
    T = synth.pose34(np.radians((2.0, -1.5, 3.0)), (0.2, -0.1, 0.05))
    res = {"card": _card(), "true_rotvec_deg": [2.0, -1.5, 3.0],
           "method": "host clock around gm_register + gm_synchronize, median of repeats after warm-up",
           "scenes": [run_scene("drift_end_niche", synth.drift_end_niche, T, a.n, a.repeats, a.warmup, a.d_max),
                      run_scene("curved_tunnel_C1", synth.curved_tunnel, T, a.n, a.repeats, a.warmup, a.d_max)]}
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
