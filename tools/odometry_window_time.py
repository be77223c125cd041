"""Time map odometry with and without a window (gm_odometry_set_window) on one long sequence, and record the card it ran on.

Sequence: 64 scans 0.8 m apart along about 50 m of the curved tunnel of synth.curved_tunnel (arc radius 50 m), each a
14 m section (240k points before the crop, no outliers) seen from its pose with small lateral and yaw offsets; radius
normals at 0.1 m, leaf 0.1 m, d_max 0.5 m, degeneracy_ratio 1e-2, the truth increments as delta34.  One context on one
stream.  Run five ways, each from a new map:
  none:           no window, a local map with capacity for the whole run (2^18 voxels, 2^19 slots);
  window:         a window at the sizing rule of include/gm_capi.h (B = 5 m, s = 1.3 m), an archive, and a local map
                  sized to the window (2^16 voxels, 2^17 slots: the window holds about 57k voxels of this tunnel);
  window_drop:    the same window with archive = NULL;
  window_big:     the same window and archive with the whole-run local map (what eviction costs at 2^19 slots);
  window_tight:   the same window and archive with a local map of 2^15 voxels (2^16 slots), too small for the window:
                  it fills to a load of about 0.9 and every hash probe sequence grows.
Reported per step index: the step's device time (CUDA events on the context's stream around gm_odometry_step: the
launches of one step, scan processing excluded), and, from torch.profiler in a separate pass, the device time of
k_map_planes and of the eviction kernels (k_map_evict_split, k_map_evict_clear, k_map_restore).  Also whether each
windowed trajectory is bit-identical to the unwindowed one, and the final voxel counts.  The card's name and power
limit are read in the same run.

    python tools/odometry_window_time.py --out profiles/r09_odometry_window.json
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from geometric_mapping_b200 import capi, synth  # noqa: E402

LEAF, DMAX, RATIO, BORE_RATIO = 0.1, 0.5, 0.1, 1e-2
SCANS, STEP, ARC_R, N = 64, 0.8, 50.0, 240_000
B, S = 5.0, 1.3
RULE = math.floor((math.sqrt(3.0) * B + S + DMAX) / LEAF) + 2
EVICT = ("k_map_evict_split", "k_map_evict_clear", "k_map_restore")
KERNELS = ("k_map_planes",) + EVICT
CONFIGS = {"none": (0, 1 << 18, False), "window": (RULE, 1 << 16, True), "window_drop": (RULE, 1 << 16, False),
           "window_big": (RULE, 1 << 18, True), "window_tight": (RULE, 1 << 15, True)}


def _card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        name, power, clock = (s.strip() for s in q.stdout.strip().splitlines()[0].split(","))
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # the timing itself needs no nvidia-smi
        return {"error": repr(e)}


def _truth(k):
    phi = STEP * k / ARC_R
    return synth.pose34((0.0, 0.0, phi + 0.004 * math.sin(1.3 * k)),
                        (ARC_R * math.sin(phi) - 0.03 * math.sin(phi) * math.cos(0.9 * k),
                         ARC_R * (1.0 - math.cos(phi)) + 0.03 * math.cos(phi) * math.cos(0.9 * k), 0.0))


def _h(P):
    return np.vstack([np.asarray(P, np.float64)[:3, :4], [0.0, 0.0, 0.0, 1.0]])


def run(ctx, scans, truth, deltas, config, events=None):
    """One sequence; events = (torch module, list to fill with per-step ms) or None.  -> trajectory, stats"""
    half, capacity, archive = CONFIGS[config]
    out = {}
    with capi.VoxelMap(LEAF, capacity) as vmap, capi.VoxelMap(LEAF, 1 << 18) as arch:
        with capi.Odometry(vmap, truth[0], max_planarity=RATIO, max_correspondence_distance=DMAX, degeneracy_ratio=BORE_RATIO) as odo:
            if half:
                odo.set_window(half, arch if archive else None)
            marks = []
            for k in range(len(scans)):
                ctx.upload_scan(scans[k])
                ctx.crop()
                ctx.normals()
                ctx.voxel()
                if events:
                    torch = events[0]
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                odo.step(ctx, deltas[k])
                if events:
                    e1.record()
                    marks.append((e0, e1))
            out["traj"] = odo.trajectory()
        if events:
            events[0].cuda.synchronize()
            events[1].extend(a.elapsed_time(b) for a, b in marks)
        out["local"] = vmap.stats()
        out["archive"] = arch.stats()
    return out


def _kernels(fn):
    import torch
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    per = {k: [] for k in KERNELS}
    try:
        evs = [e for e in prof.events() if str(getattr(e, "device_type", "")).endswith("CUDA")]
        evs.sort(key=lambda e: e.time_range.start)
        for e in evs:
            name = e.name.split("(")[0].split("::")[-1].split("<")[0].strip()
            if name in per:
                per[name].append(e.time_range.elapsed_us() / 1e3)
    except Exception as ex:  # the means below do not need the event list
        per["error"] = repr(ex)
    means = {}
    for e in prof.key_averages():
        name = e.key.split("(")[0].split("::")[-1].split("<")[0].strip()
        if name in KERNELS:
            dev_us = getattr(e, "device_time_total", None)
            if dev_us is None:
                dev_us = e.cuda_time_total
            means[name] = {"launches": e.count, "ms_mean": dev_us / 1e3 / max(e.count, 1)}
    return per, means


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scans", type=int, default=SCANS)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("odometry_window_time: no CUDA device (the library has no CPU path)")
    truth = [_truth(k) for k in range(a.scans)]
    deltas = [None] + [np.linalg.solve(_h(truth[k - 1]), _h(truth[k]))[:3].astype(np.float32) for k in range(1, a.scans)]
    scans = [synth.view_from(synth.curved_tunnel(N, seed=500 + k, arc_length=14.0, advance=STEP * k, outlier_frac=0.0), truth[k])
             for k in range(a.scans)]
    res = {"card": _card(), "scene": "curved_tunnel arc radius 50 m, 14 m sections", "n_points": N, "scans": a.scans,
           "step_m": STEP, "run_length_m": STEP * (a.scans - 1), "leaf": LEAF,
           "icp": {"max_correspondence_distance": DMAX, "max_iterations": 30, "max_planarity": RATIO, "degeneracy_ratio": BORE_RATIO},
           "window": {"half_cells": RULE, "rule": "floor((sqrt(3)*B + s + d_max) / leaf) + 2", "B": B, "s": S},
           "configs": {k: {"half_cells": v[0], "local_capacity_voxels": v[1], "archive": v[2]} for k, v in CONFIGS.items()},
           "method": "step_ms: CUDA events on the context's stream around each gm_odometry_step (its launches only), one "
                     "sequence after one warm-up sequence per config; kernel times: torch.profiler device time per launch "
                     "in a separate pass, in launch order (one k_map_planes per registered step)"}
    stream = torch.cuda.Stream()
    with capi.Context(capi.default_params(neighborRadius=0.1, voxelGridLeafSize=LEAF), max_points=N, max_hypotheses=16) as ctx:
        ctx.set_stream(stream.cuda_stream)
        with torch.cuda.stream(stream):
            results = {}
            for cfg in CONFIGS:
                run(ctx, scans, truth, deltas, cfg)                      # warm-up
                ms = []
                r = run(ctx, scans, truth, deltas, cfg, (torch, ms))
                per, means = _kernels(lambda: run(ctx, scans, truth, deltas, cfg))
                results[cfg] = r
                t = r["traj"]
                res[cfg] = {"step_ms": [round(x, 4) for x in ms], "step_ms_first8_median": float(np.median(ms[1:9])),
                            "step_ms_last8_median": float(np.median(ms[-8:])),
                            "k_map_planes_ms": [round(x, 4) for x in per.get("k_map_planes", [])],
                            "evict_ms_per_step": [round(sum(x), 4) for x in zip(*(per.get(k, []) for k in EVICT))] if per.get(EVICT[0]) else [],
                            "kernel_means": means, "accepted": int(t["accepted"].sum()),
                            "local_voxels": r["local"][0], "local_full": r["local"][3],
                            "archive_voxels": r["archive"][0], "archive_full": r["archive"][3]}
                if "error" in per:
                    res[cfg]["profiler_events_error"] = per["error"]
            ref = results["none"]["traj"]["poses"].view(np.uint32)
            for cfg in CONFIGS:
                res[cfg]["trajectory_bit_identical_to_none"] = bool(np.array_equal(results[cfg]["traj"]["poses"].view(np.uint32), ref))
            P = results["none"]["traj"]["poses"][-1].astype(np.float64)
            res["none"]["final_translation_error_m"] = float(np.linalg.norm(P[:, 3] - truth[-1][:, 3]))
        ctx.set_stream(None)
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
