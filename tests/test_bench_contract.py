"""bench.py contract on CPU: the reference arm prints ONE JSON line with the agreed keys (the CUDA arm needs a
GPU and is exercised by the driver), non-zero ranks of the reference arm stay silent, and the CUDA arm refuses to run
without a device instead of falling back."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, env=e, timeout=600)


def test_reference_arm_json_line():
    res = _run(["--impl", "reference", "--steps", "1", "--warmup", "1", "--points", "100000", "--hyp", "64"])
    assert res.returncode == 0, res.stderr
    lines = [l for l in res.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "points/s" and d["higher_is_better"] is True and d["value"] > 0
    for k in ("metric", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data", "config"):
        assert k in d
    assert d["config"]["workload"].startswith("C1 synthetic curved tunnel") and d["vs_baseline"] is None
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "parity unpinned" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "points/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_thread_count_ignores_omp_num_threads():
    """torchrun exports OMP_NUM_THREADS=1; the CPU arm must still use (and report) every usable core."""
    res = _run(["--impl", "reference", "--steps", "1", "--warmup", "1", "--points", "60000", "--hyp", "64"], env={"OMP_NUM_THREADS": "1"})
    assert res.returncode == 0, res.stderr
    d = json.loads(res.stdout.strip())
    assert d["cpu_baseline"]["cores"] == len(os.sched_getaffinity(0))
    assert d["config"]["points_per_scan"] == 60000 and d["config"]["plane_hypotheses"] == 32


def test_reference_arm_other_ranks_print_nothing():
    res = _run(["--impl", "reference", "--steps", "1", "--warmup", "1", "--points", "50000"], env={"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert res.returncode == 0 and res.stdout.strip() == ""


@pytest.mark.gpu
def test_dump_outputs_are_reproducible_and_bounded(tmp_path):
    """--dump-outputs: two runs with the same arguments write the same finite arrays (float32 / float64, at most 64 MB in all;
    2M points per scan is over that, so the per-point arrays are sampled)."""
    import numpy as np

    dumps = []
    for run in ("a", "b"):
        d = tmp_path / run
        res = _run(["--steps", "3", "--warmup", "1", "--points", "2000000", "--map-points", "0", "--shard-hyp-large", "0",
                    "--no-cpu-baseline", "--dump-outputs", str(d)])
        assert res.returncode == 0, res.stderr[-3000:]
        assert json.loads(res.stdout.strip())["steps"] == 3
        files = sorted(os.listdir(d))
        assert {"cloud.npy", "normals.npy", "labels.npy", "plane_coef.npy", "cylinder_coef.npy", "frame_vecs.npy"} <= set(files)
        assert sum(os.path.getsize(d / f) for f in files) <= 64 << 20
        dumps.append({f: np.load(d / f) for f in files})
    a, b = dumps
    assert a.keys() == b.keys()
    for f in a:
        assert a[f].dtype in (np.float32, np.float64) and np.isfinite(a[f]).all(), f
        assert a[f].tobytes() == b[f].tobytes(), f
    assert len(a["voxel_nn_index.npy"]) == len(a["voxel_nn_normals.npy"])
    n_valid = int(a["counts.npy"][2])
    assert 0 < len(a["cloud.npy"]) < n_valid and len(a["normals.npy"]) == len(a["cloud.npy"])


def test_cuda_arm_fails_loudly_without_a_device():
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    res = _run(["--steps", "1", "--warmup", "1"])
    assert res.returncode != 0 and "no CUDA device" in (res.stderr + res.stdout)
