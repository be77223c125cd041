"""Time gm_extract_primitives with CUDA events and compare gm_compress_primitives with gm_compress on the same cloud.
    python tools/primitives_time.py [out.json]
Two workloads: a 1M-point C1 scan (K = 8) and the 10M-point C4 map (synth.tunnel_map, K = 32), 512 plane + 512 cylinder
draws per round.  Reports ms per extraction and per round, launches, primitives found, and ratio / total_rms of both
compressions, next to the GPU's name and power limit."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

H = 512
REPS = 5


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()[0]
        name, power = (s.strip() for s in out.split(","))
        return {"gpu": name, "power_limit": power}
    except Exception as e:  # the numbers still stand; say what is missing
        return {"gpu": "unknown", "power_limit": f"unknown ({e})"}


def leg(name, pts, params, K, grid_box=None):
    import torch

    from geometric_mapping_b200 import capi, synth

    stream = torch.cuda.Stream()
    with capi.Context(params, max_points=len(pts), max_hypotheses=H) as ctx:
        ctx.set_stream(stream.cuda_stream)
        if grid_box is not None:
            ctx.set_grid_box(*grid_box)
        ctx.upload_scan(pts)
        ctx.crop()
        ctx.normals()
        nv = ctx.counts().n_valid
        ps, cs = synth.sample_indices(nv, H, 3, seed=3), synth.sample_indices(nv, H, 2, seed=4)
        ctx.upload_scan(pts)
        ctx.process_scan(ps, cs)
        ctx.compress()
        gmc = ctx.compression()
        pd, cd = synth.sample_draws(K, H, 3, seed=1), synth.sample_draws(K, H, 2, seed=2)
        ctx.extract_primitives(pd, cd, K, 1000)  # warm-up: first-call allocations, module loads
        ts = []
        for _ in range(REPS):
            ctx.reset_launch_count()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            ctx.extract_primitives(pd, cd, K, 1000)
            e1.record(stream)
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        launches = ctx.launch_count
        prims = ctx.primitives()
        ctx.compress_primitives()
        h = capi.parse_compressed_primitives(ctx.download_compressed_primitives())["header"]
        assert ctx.counts().device_error == 0
    ms = float(np.median(ts))
    return {"name": name, "points": len(pts), "n_valid": nv, "K": K, "Hp": H, "Hc": H, "min_inliers": 1000,
            "ms_per_extraction_median": ms, "ms_per_extraction_all": [round(t, 3) for t in ts], "ms_per_round": ms / K,
            "launches": launches, "primitives": len(prims), "kinds": [p["kind"] for p in prims],
            "claimed": int(sum(p["best_count"] for p in prims)),
            "compress": {"ratio": float(gmc.ratio), "total_rms": float(gmc.total_rms), "residual_voxels": int(gmc.n_residual_voxels)},
            "compress_primitives": {"ratio": float(h.ratio), "total_rms": float(h.total_rms), "residual_voxels": int(h.n_residual_voxels)}}


def main():
    from geometric_mapping_b200 import capi, distributed, synth

    out = {**gpu_info(), "timing": "CUDA events around gm_extract_primitives, median of %d after one warm-up call" % REPS, "legs": []}
    c1 = synth.curved_tunnel(1_000_000, seed=2)
    out["legs"].append(leg("C1 1M scan", c1, capi.default_params(neighborRadius=0.05, voxelGridLeafSize=0.1), 8))
    del c1
    c4 = synth.tunnel_map(10_000_000, seed=4, bound=60.0)
    box = distributed.robust_box(c4[:, :3])
    out["legs"].append(leg("C4 10M map", c4, capi.default_params(boxFilterBound=60.0, neighborRadius=0.05, voxelGridLeafSize=0.1), 32,
                           grid_box=box))
    text = json.dumps(out, indent=1)
    print(text)
    if len(sys.argv) > 1:
        with open(sys.argv[1], "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
