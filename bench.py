#!/usr/bin/env python
"""bench.py — points/s of the per-scan hot path (crop -> normals -> voxel -> local frame -> RANSAC
plane+cylinder -> refit -> labels -> polyline) on synthetic 1M-point curved-tunnel scans.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...   # the CPU oracle (reference arm)

Contract (see the task statement): one JSON line on stdout from rank 0.
  value     whole-job input points/s, scans already resident in HBM, CUDA-event timed, max over ranks
  e2e       same metric through the C-ABI with HOST (pinned) buffers: H2D of the scan and D2H of the
            published results inside the timed region (3 contexts pipelined on 3 streams)
  roofline  the dominant kernel family, CUDA-event timed per segment inside this run
  cpu_baseline  the CPU oracle on this box's host cores (rank 0, N=1)
N>1: frame-parallel (each rank processes its own scans, no data-path collective; weak scaling) plus
a hypothesis-sharded RANSAC leg (4096 hypotheses split across ranks, NCCL max-allreduce of the
packed (count,id) key) reported under "ransac".
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark leaves the tree it runs from untouched (it may be read-only)

TAU = 0.05
KNN_CAP = 0.25  # radius cap of the k-NN mode (gm_set_knn_max_radius): isolated outliers do not drag the search across the grid
RING = 12  # distinct resident scans cycled through: 12 x 16 MB = 192 MB > 126 MB L2


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--points", type=int, default=1_000_000)
    ap.add_argument("--hyp", type=int, default=1024, help="total RANSAC hypotheses (half plane, half cylinder)")
    ap.add_argument("--shard-hyp", type=int, default=4096, help="hypotheses of the sharded RANSAC leg (N>1)")
    ap.add_argument("--shard-hyp-large", type=int, default=65536, help="second sharded RANSAC leg, large enough to amortise the "
                    "fixed cost of a round (0 = skip)")
    ap.add_argument("--radius", type=float, default=0.05)
    ap.add_argument("--leaf", type=float, default=0.1)
    ap.add_argument("--refit-iters", type=int, default=5)
    ap.add_argument("--map-points", type=int, default=10_000_000, help="points of the aggregated-map leg (configs[4]); 0 = skip")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-points", type=int, default=0, help="points of the CPU baseline sample (0 = full scan)")
    ap.add_argument("--knn", type=int, default=0, help="k-nearest-neighbour normals with this k instead of the radius search (0 = radius)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step of the headline leg computed to DIR/<name>.npy (rank 0)")
    return ap.parse_args()


def workload_name(a):
    return (f"C1 synthetic curved tunnel + floor + noise, {a.points} pts/scan, {a.hyp // 2} plane + {a.hyp - a.hyp // 2} "
            f"cylinder hypotheses, r={a.radius} leaf={a.leaf} tau={TAU}")


def workload_config(a):
    """The `config` object: identical in both arms (b200 and --impl reference), it names the workload only."""
    return {"workload": workload_name(a), "points_per_scan": a.points, "plane_hypotheses": a.hyp // 2,
            "cylinder_hypotheses": a.hyp - a.hyp // 2, "radius_m": a.radius, "leaf_m": a.leaf, "tau_m": TAU,
            "refit_iterations": a.refit_iters, "scans": f"ring of {RING} distinct seeded scans (seeds 2..{1 + RING}) cycled",
            "l2": f"inputs larger than L2: the ring holds {RING * a.points * 16 / 1e6:.0f} MB of scans, one step = the next scan of the ring"}


def host_threads() -> int:
    """Threads the CPU arm uses: every core this process may run on (torchrun forces OMP_NUM_THREADS=1, which must not
    decide it: the count is passed to the oracle explicitly)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


# ---------------------------------------------------------------------------------------------
# CPU arm: the oracle's restatement of the reference path, the oracle ALONE from raw points (oracle/chain.py;
# used by cpu_baseline and --impl reference, never by the product)
def cpu_process_scan(pts, a, ps, cs, nthreads):
    from oracle import chain

    f = chain.front(pts, bound=5.0, radius=a.radius, leaf=a.leaf, wf=0.2, nthreads=nthreads, knn=a.knn, knn_max_radius=KNN_CAP if a.knn else 0.0)
    nv = f["n_valid"]
    ps = None if ps is None else (ps % max(nv, 1)).astype(np.int32)   # same rule as the GPU arm (ring_samples)
    cs = None if cs is None else (cs % max(nv, 1)).astype(np.int32)
    b = chain.back(f, ps, cs, tau=TAU, refit_iters=a.refit_iters, nthreads=nthreads)
    return f, b


def ring_scan(a, s, rank=0):
    from geometric_mapping_b200 import synth

    return synth.curved_tunnel(a.points, seed=2 + s + 1000 * rank, advance=0.0)


def ring_samples(a, s, n_valid=None, hyp=None):
    """Injected RANSAC sample indices of ring scan s: Philox(seed) draws over the INPUT size, reduced modulo the compacted
    size of the scan once that is known (n_valid): both arms apply the same rule, so they test the same hypotheses."""
    from geometric_mapping_b200 import synth

    hyp = a.hyp if hyp is None else hyp
    ps, cs = synth.sample_indices(a.points, hyp // 2, 3, seed=3 + s), synth.sample_indices(a.points, hyp - hyp // 2, 2, seed=4 + s)
    if n_valid is not None:
        ps, cs = (ps % max(n_valid, 1)).astype(np.int32), (cs % max(n_valid, 1)).astype(np.int32)
    return ps, cs


def run_reference(a, rank):
    """CPU arm: the oracle on all host threads, on the SAME workload as the GPU arm: the same ring of full scans, the
    same hypothesis counts (sample indices drawn with the same seeds from each scan's own compacted size).  A step is
    one whole scan; when a step takes so long that K steps would not end within a few minutes the run is cut short and
    `steps` reports what was timed."""
    if rank != 0:
        return
    from oracle import oracle as O

    threads = host_threads()
    budget_s = float(os.environ.get("GM_REF_BUDGET_S", "150"))
    scans, smp = {}, {}

    def get(i):
        s = i % RING
        if s not in scans:
            scans[s] = ring_scan(a, s)
            smp[s] = ring_samples(a, s)  # reduced modulo n_valid inside cpu_process_scan
        return scans[s], smp[s]

    nwarm = min(max(a.warmup, 1), 2)
    for i in range(nwarm):
        pts, (ps, cs) = get(i)
        cpu_process_scan(pts, a, ps, cs, threads)
    for i in range(a.steps):  # generate the ring outside the timed region
        if i < RING:
            get(i)
    done, dt = 0, 0.0
    for i in range(a.steps):
        pts, (ps, cs) = get(i)
        t0 = time.perf_counter()
        cpu_process_scan(pts, a, ps, cs, threads)
        dt += time.perf_counter() - t0
        done += 1
        if dt > budget_s:
            break
    v = a.points * done / dt
    line = {
        "impl": "reference", "metric": "input points/s, per-scan segmentation+fit", "value": v, "unit": "points/s",
        "n_gpus": a.gpus, "steps": done, "warmup": nwarm, "ms_per_step": 1e3 * dt / done,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(a),
        "cpu_baseline": {"value": v, "unit": "points/s", "cores": threads, "kind": "port",
                         "sample": f"{done} full scans of {a.points} points (the GPU arm's ring, same seeds and hypothesis counts), whole path "
                                   f"from raw points on the oracle alone; OpenMP with {threads} threads over points (normals, 1-NN) and "
                                   f"hypotheses (counting), serial elsewhere; steps requested {a.steps}, time budget {budget_s:.0f} s; "
                                   f"parity unpinned (the reference cannot be built here: PCL/Eigen/ROS absent)"},
        "e2e": {"value": v, "unit": "points/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ---------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons of one GPU with NVML while the timed region runs."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz, self._stop_evt = index, [], set(), None, threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception:
            self.nv = None

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40, "sw_power_cap": 0x4,
                 "hw_power_brake": 0x80}
        while not self._stop_evt.is_set():
            try:
                self.samples.append(int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                r = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            self._stop_evt.wait(0.002)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


def physical_gpu_index(local_rank: int) -> int:
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_rank])
        except Exception:
            return local_rank
    return local_rank


def bind_to_gpu_numa_node(index: int):
    """Pin this rank (and therefore its pinned host buffers, first touch) to the CPUs of the NUMA node its GPU
    hangs off: with 8 ranks streaming 33 MB per scan each way, cross-socket traffic caps the end-to-end rate."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()
        if len(bus.split(":")[0]) == 8:      # nvml: 00000000:1B:00.0 -> sysfs: 0000:1b:00.0
            bus = bus[4:]
        with open(f"/sys/bus/pci/devices/{bus}/numa_node") as f:
            node = int(f.read().strip())
        if node < 0:
            return None
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            cpus = set()
            for part in f.read().strip().split(","):
                a, _, b = part.partition("-")
                cpus.update(range(int(a), int(b or a) + 1))
        allowed = os.sched_getaffinity(0) & cpus
        if allowed:
            os.sched_setaffinity(0, allowed)
            return node
    except Exception:
        return None
    return None


def load_traffic(points: int):
    """Per-launch DRAM traffic (dram__bytes_read.sum + dram__bytes_write.sum) of the main kernels from the committed
    `ncu --set full` captures (profiles/r02_traffic.json: {"1M": {kernel: bytes}, "10M": {...}, "_source": ...}).
    Only the capture of the same workload size is used; none -> {} (traffic fields are then null)."""
    p = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if not os.path.exists(p):
        return {}
    with open(p) as f:
        d = json.load(f)
    if 0.7e6 <= points <= 1.5e6:
        return d.get("1M", {})
    if 0.7e7 <= points <= 1.5e7:
        return d.get("10M", {})
    return {}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


DUMP_LIMIT = 64 << 20


def scan_outputs(cx):
    """What a caller of process_scan receives for one scan, as float32 / float64 arrays (integers are exact in float64)."""
    from geometric_mapping_b200 import capi

    c = cx.counts()
    fr = cx.frame()
    out = {"counts": np.array([getattr(c, f) for f, _ in c._fields_], np.float64),
           "frame_vals": fr["vals"], "frame_vecs": fr["vecs"]}
    for kind, name in ((capi.GM_MODEL_PLANE, "plane"), (capi.GM_MODEL_CYLINDER, "cylinder")):
        m = cx.model(kind)
        out[f"{name}_coef"] = m["coef"]
        out[f"{name}_fit"] = np.array([m["best_id"], m["best_count"], m["refit_count"], m["rms"]], np.float64)
    out["cloud"] = cx.download_cloud(1)
    out["normals"] = cx.download_normals(1)
    out["labels"] = cx.download_labels().astype(np.float32)
    v = cx.download_voxels(with_nn=True)
    # a 1-NN index outside the compacted cloud (nn_index_mode 0, counted in nn_out_of_range) has no normal: the library
    # returns NaN there, the dump zeros; voxel_nn_index tells those rows apart
    has_normal = (v["nn_index"] >= 0) & (v["nn_index"] < c.n_valid)
    out["voxel_centroids"] = v["centroids"]
    out["voxel_nn_index"] = v["nn_index"].astype(np.float64)
    out["voxel_nn_normals"] = np.where(has_normal[:, None], v["nn_normal"], np.float32(0))
    pl = cx.download_polyline()
    out["polyline"] = np.concatenate([pl["center"], pl["dir"]] + [pl[k][:, None] for k in ("radius", "rms", "t_mid", "count")],
                                     axis=1).astype(np.float64)
    return out


def dump_outputs(outs: dict, path: str):
    """DIR/<name>.npy for every array, DUMP_LIMIT bytes in all: when the arrays are larger, every array of more than 4096
    rows keeps the same share of its rows, a fixed seeded sample in row order, so two runs keep the same rows."""
    bad = [name for name, a in outs.items() if not np.isfinite(a).all()]
    if bad:
        raise SystemExit(f"bench.py: non-finite values in the outputs {bad}")
    limit = DUMP_LIMIT - 256 * len(outs)   # room for the .npy headers
    total = sum(a.nbytes for a in outs.values())
    big = sum(a.nbytes for a in outs.values() if len(a) > 4096)
    keep = 1.0 if total <= limit else max(0.0, (limit - (total - big)) / big)
    os.makedirs(path, exist_ok=True)
    for name, a in outs.items():
        if keep < 1.0 and len(a) > 4096:
            rows = np.random.default_rng(0).choice(len(a), int(len(a) * keep), replace=False)
            a = a[np.sort(rows)]
        np.save(os.path.join(path, name + ".npy"), a)


_REAL_STDOUT = None


def guard_stdout():
    """stdout carries exactly ONE line, the JSON record: libraries that print there (NCCL's version banner at
    NCCL_DEBUG=VERSION, torch warnings) are sent to stderr for the whole run; emit() writes the record to the real stdout."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line: dict):
    data = (json.dumps(line) + "\n").encode()
    sys.stdout.flush()
    if _REAL_STDOUT is None:
        os.write(1, data)
    else:
        os.write(_REAL_STDOUT, data)


def main():
    a = parse_args()
    guard_stdout()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if a.impl == "reference":
        run_reference(a, rank)
        return

    import torch
    import torch.distributed as dist

    from geometric_mapping_b200 import capi, synth

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; this framework has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa_node = bind_to_gpu_numa_node(physical_gpu_index(local_rank)) if world > 1 else None
    if world > 1:
        # keep stdout to the single JSON line: NCCL prints its version banner there at NCCL_DEBUG=VERSION
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)

    n, Hp, Hc = a.points, a.hyp // 2, a.hyp - a.hyp // 2
    params = capi.default_params(neighborRadius=a.radius, voxelGridLeafSize=a.leaf, ransacThreshold=TAU, refitIterations=a.refit_iters)
    # an explicit non-default stream for everything (context work, copies, CUDA events, NCCL): the
    # default stream's handle is 0, which would not order the context's work with torch's
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)

    # ---- synthetic ring of scans: distinct per slot and per rank (frame-parallel = weak scaling)
    host_scans, dev_scans = [], []
    for s in range(RING):
        pts = ring_scan(a, s, rank)
        hp = torch.from_numpy(pts).pin_memory()
        host_scans.append(hp)
        dev_scans.append(hp.to(dev, non_blocking=False))
    def new_ctx(max_h):
        cx = capi.Context(params, max_points=n, max_hypotheses=max_h)
        if a.knn:
            cx.set_knn(a.knn, max_radius=KNN_CAP)
        return cx

    ctx = new_ctx(max(4096, a.shard_hyp, a.shard_hyp_large))
    ctx.set_stream(stream.cuda_stream)

    # sample indices need the compacted size of each scan: learn it once (untimed)
    samples = []
    n_valid = []
    nbr_sum = []
    for s in range(RING):
        ctx.set_scan_device(dev_scans[s].data_ptr(), n)
        ctx.crop()
        ctx.normals()
        nv = ctx.counts().n_valid
        n_valid.append(nv)
        if s < 2:
            nbr_sum.append(ctx.search_stats())
        samples.append(ring_samples(a, s, nv))

    def step(i):
        s = i % RING
        ctx.set_scan_device(dev_scans[s].data_ptr(), n)
        ctx.process_scan(samples[s][0], samples[s][1])

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident throughput ------------------------------------------------------------
    # (a) one scan at a time on one context: per-scan latency
    for i in range(max(a.warmup, 3)):
        step(i)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for i in range(a.steps):
        step(i)
    e1.record(stream)
    barrier()
    latency_ms = max_over_ranks(e0.elapsed_time(e1)) / a.steps

    # (b) throughput: NFLIGHT scans in flight, one context (and CUDA stream) each, round robin, the way
    # a stream of scans is processed.  Timed with CUDA events: e0 on the first context's stream before
    # the first step, e1 on a stream that has waited for every context's last step.
    NFLIGHT = max(1, int(os.environ.get("GM_BENCH_NFLIGHT", "3")))
    tctx = [ctx] + [new_ctx(max(4096, a.shard_hyp)) for _ in range(NFLIGHT - 1)]
    tstreams = [stream] + [torch.cuda.Stream(device=dev) for _ in range(NFLIGHT - 1)]
    for cx, st_ in zip(tctx[1:], tstreams[1:]):
        cx.set_stream(st_.cuda_stream)

    def tstep(i):
        s, cx = i % RING, tctx[i % NFLIGHT]
        cx.set_scan_device(dev_scans[s].data_ptr(), n)
        cx.process_scan(samples[s][0], samples[s][1])

    for i in range(max(a.warmup, 3) * NFLIGHT):
        tstep(i)   # (>= 3 scans per context: plain launches, graph capture, first replay)
    barrier()
    sampler = ClockSampler(physical_gpu_index(local_rank))
    sampler.start()
    for cx in tctx:
        cx.reset_launch_count()
    for st_ in tstreams[1:]:
        st_.wait_stream(stream)
    e0.record(stream)
    for st_ in tstreams[1:]:
        st_.wait_event(e0)
    for i in range(a.steps):
        tstep(i)
    for st_ in tstreams[1:]:
        stream.wait_stream(st_)
    e1.record(stream)
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1))
    launches = sum(cx.launch_count for cx in tctx)
    graph_stats = ctx.graph_stats()
    clocks = sampler.stop()
    for cx in tctx:
        if cx.counts().device_error:
            raise SystemExit("device-side error flag set")
    if a.dump_outputs and rank == 0:
        dump_outputs(scan_outputs(tctx[(a.steps - 1) % NFLIGHT]), a.dump_outputs)   # the legs below reuse these contexts
    c = ctx.counts()
    value = world * n * a.steps / (ms * 1e-3)
    # the same throughput measurement at the north-star's hypothesis count (2048 plane + 2048 cylinder)
    H4 = 4096
    samples4 = [ring_samples(a, s, n_valid[s], hyp=H4) for s in range(RING)]

    def tstep4(i):
        s, cx = i % RING, tctx[i % NFLIGHT]
        cx.set_scan_device(dev_scans[s].data_ptr(), n)
        cx.process_scan(samples4[s][0], samples4[s][1])

    steps4 = max(12, a.steps)  # as many as the headline: a pipelined measurement of a handful of scans is mostly fill and drain
    for i in range(3 * NFLIGHT):
        tstep4(i)
    barrier()
    for st_ in tstreams[1:]:
        st_.wait_stream(stream)
    e0.record(stream)
    for st_ in tstreams[1:]:
        st_.wait_event(e0)
    for i in range(steps4):
        tstep4(i)
    for st_ in tstreams[1:]:
        stream.wait_stream(st_)
    e1.record(stream)
    barrier()
    ms4 = max_over_ranks(e0.elapsed_time(e1)) / steps4
    h4096 = {"hypotheses": H4, "ms_per_step": ms4, "points_per_s": world * n / (ms4 * 1e-3), "steps": steps4,
             "note": "same workload with 2048 plane + 2048 cylinder hypotheses per scan (north-star target count)"}
    # ---- configs[3]: a batch of 64 frames x 200k points split by frame over the ranks (no collective) ----
    from geometric_mapping_b200 import distributed as gmd_
    F_TOTAL, F_PTS = 64, 200_000
    my_frames = gmd_.frames_of_rank(F_TOTAL, rank, world)
    fr_dev, fr_smp = [], []
    for f in my_frames:
        fp = torch.from_numpy(synth.curved_tunnel(F_PTS, seed=100 + f, advance=1.0 * f)).to(dev)
        ctx.set_scan_device(fp.data_ptr(), F_PTS)
        ctx.crop()
        ctx.normals()
        nvf = ctx.counts().n_valid
        fr_dev.append(fp)
        fr_smp.append((synth.sample_indices(nvf, Hp, 3, seed=300 + f), synth.sample_indices(nvf, Hc, 2, seed=400 + f)))

    def frames_pass():
        for j in range(len(my_frames)):
            cx = tctx[j % NFLIGHT]
            cx.set_scan_device(fr_dev[j].data_ptr(), F_PTS)
            cx.process_scan(fr_smp[j][0], fr_smp[j][1])

    for _ in range(3):
        frames_pass()
    barrier()
    for st_ in tstreams[1:]:
        st_.wait_stream(stream)
    e0.record(stream)
    for st_ in tstreams[1:]:
        st_.wait_event(e0)
    FREPS = 3
    for _ in range(FREPS):
        frames_pass()
    for st_ in tstreams[1:]:
        stream.wait_stream(st_)
    e1.record(stream)
    barrier()
    fms = max_over_ranks(e0.elapsed_time(e1)) / FREPS
    frames_c3 = {"frames": F_TOTAL, "points_per_frame": F_PTS, "ms_per_batch": fms, "frames_per_s": F_TOTAL / (fms * 1e-3),
                 "points_per_s": F_TOTAL * F_PTS / (fms * 1e-3),
                 "mode": f"frame f -> rank f mod {world}, {NFLIGHT} frames in flight per rank, full per-frame output incl. the polyline; "
                         f"{Hp}+{Hc} hypotheses per frame"}
    del fr_dev
    for cx in tctx[1:]:
        cx.close()

    # ---- per-segment timing of the same steps (roofline) ------------------------------------------
    # CUDA-event pairs inside the library around every stage (gm_profile_*: plain stream launches on one stream, so the
    # segments add up; the timed legs above replay the graph on three streams).
    def profile_steps(count, knn=0, voxel_mode=0, count_mode=0, cx=None):
        cx = cx or ctx
        cx.set_voxel_mode(voxel_mode)
        cx.set_count_mode(count_mode)
        cx.set_knn(knn, max_radius=KNN_CAP if knn else 0.0)

        def one(i):
            s = i % RING
            cx.set_scan_device(dev_scans[s].data_ptr(), n)
            cx.process_scan(samples[s][0], samples[s][1])

        for i in range(2):
            one(i)
        cx.profile_enable(True)
        for i in range(count):
            one(i)
        pr = cx.profile_read()
        cx.profile_enable(False)
        cx.set_voxel_mode(0)
        cx.set_count_mode(0)
        cx.set_knn(a.knn, max_radius=KNN_CAP if a.knn else 0.0)
        return {k: (v[0] / max(count, 1)) for k, v in pr.items()}

    nb = max(4, min(a.steps, 20))
    seg_ms = profile_steps(a.steps, knn=a.knn)
    seg_brute = profile_steps(nb, knn=a.knn, count_mode=1)       # every point x hypothesis test executed: the FP32-pipe figure
    seg_sortvox = profile_steps(nb, knn=a.knn, voxel_mode=1)     # sort-based VoxelGrid (keys -> radix sort -> heads -> centroids)
    seg_knn = None
    KNN_CELL = 0.07   # grid cell of the k-NN leg: near the distance of the 32nd neighbour on this scan (the search is exact for any cell)
    if not a.knn:      # k-NN normals (k = 32, SURVEY 8d) on the same scans
        kparams = capi.default_params(neighborRadius=KNN_CELL, voxelGridLeafSize=a.leaf, ransacThreshold=TAU, refitIterations=a.refit_iters)
        with capi.Context(kparams, max_points=n, max_hypotheses=4096) as kctx:
            kctx.set_stream(stream.cuda_stream)
            seg_knn = profile_steps(nb, knn=32, cx=kctx)
    brute_ms = seg_brute["plane_count"] + seg_brute["cyl_count"]
    M = float(np.mean(n_valid))
    Mc = float(c.n_cropped)
    V = float(c.n_voxels)
    hbm_peak, peak_src = load_peaks()
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    clk = clocks["sm_mhz"] or clocks["sm_max_mhz"] or 1965.0
    fp32_peak_tflops = sms * 128 * 2 * clk * 1e6 / 1e12
    count_ms = seg_ms["plane_count"] + seg_ms["cyl_count"]
    count_flops = M * (Hp * 6.0 + Hc * 16.0)
    count_tflops = count_flops / (count_ms * 1e-3) / 1e12 if count_ms > 0 else 0.0
    traffic = load_traffic(n)
    fp32_src = f"{sms} SMs x 128 lanes x 2 x {clk:.0f} MHz observed ({clocks['samples']} NVML samples during the timed region)"
    cand_per_scan = float(np.mean([c_ for c_, _ in nbr_sum])) if nbr_sum else 150.0 * M
    nbr_per_scan = float(np.mean([n_ for _, n_ in nbr_sum])) if nbr_sum else 40.0 * M
    nrm_ms = seg_ms["normals"]
    # k_normals, grid-hashed radius search (cell = radius, 27-cell stencil): every point of the stencil takes the
    # exact FLANN distance test (8 flop), every neighbour the 9-accumulator update (15 flop), every point ~150 flop of
    # eigen33.  The counts are measured by the kernel itself (gm_get_search_stats).
    nrm_flops = 8.0 * cand_per_scan + 15.0 * nbr_per_scan + 150.0 * M
    nrm_tflops = nrm_flops / (nrm_ms * 1e-3) / 1e12 if nrm_ms > 0 else 0.0
    brute_tflops = count_flops / (brute_ms * 1e-3) / 1e12 if brute_ms > 0 else 0.0

    def gbs(nbytes, ms_):
        return nbytes / (ms_ * 1e-3) / 1e9 if (ms_ and nbytes) else None

    def tsum(*names):
        vals = [traffic.get(k) for k in names]
        return None if any(v is None for v in vals) else float(sum(vals))

    # ---- HBM-bound families.  Two byte counts each: SURVEY 8(d)'s ALGORITHMIC bytes (what `achieved` / `frac` use) and the
    # dram__bytes the same kernels move under `ncu --set full` on this workload size (`traffic`, with `achieved_on_traffic`):
    # at 1M points the working set sits in the 126 MB L2, so the DRAM traffic is far below the algorithmic bytes and neither
    # figure is an HBM-pipe utilisation -- the 10M-point line (bench.py --points 10000000 --radius 0.02) is the HBM-bound one.
    key_bits_grid = 24 if n <= 2_000_000 else 32   # neighbour-grid cell key: 18 block bits + 6 at C1 (3 passes of 8 bits)
    P_grid = (key_bits_grid + 7) // 8
    sort_bytes = 20.0 * P_grid * Mc                 # per pass: histogram read 4 + (key,index) read 8 + write 8
    sort_ms = seg_ms["grid_sort"]
    down_keys = [k for k in traffic if k.startswith("k_rs2_down")]
    sort_traffic = None if (traffic.get("k_rs2_hist") is None or not down_keys) else P_grid * (traffic["k_rs2_hist"] + traffic[down_keys[0]])
    P_vox = 3
    vox8d_bytes = 16.0 * n + (68.0 + 16.0 * P_vox) * M + 20.0 * V     # SURVEY 8(d): crop + keys + P-pass sort + heads + centroids
    voxdense_ms = seg_ms["crop"] + seg_ms["voxel_keys"] + seg_ms["voxel_sort"] + seg_ms["voxel_reduce"]
    voxsort_ms = seg_sortvox["crop"] + seg_sortvox["voxel_keys"] + seg_sortvox["voxel_sort"] + seg_sortvox["voxel_reduce"]
    voxdense_traffic = tsum("k_crop", "k_voxel_accumulate_sorted", "k_voxel_dense_scan", "k_voxel_assign")
    families = {
        "normals": {"bound": "fp32", "achieved": nrm_tflops, "peak": fp32_peak_tflops, "unit": "TFLOP/s",
                    "frac": nrm_tflops / fp32_peak_tflops, "traffic": traffic.get("k_normals<0>"), "ms_per_step": nrm_ms,
                    "kernels": "k_normals<0>",
                    "algorithmic": f"8 flop x {cand_per_scan:.0f} stencil candidates + 15 flop x {nbr_per_scan:.0f} neighbours + 150 flop x "
                                   f"{M:.0f} points; the kernel is instruction-issue bound (ncu: ~77 % of issue slots active, ~26 "
                                   f"instructions per candidate slot of which 8 are these flops)",
                    "points_per_s": M / (nrm_ms * 1e-3) if nrm_ms > 0 else 0.0, "peak_source": fp32_src},
        "inlier_count": {"bound": "fp32", "achieved": count_tflops, "peak": fp32_peak_tflops, "unit": "TFLOP/s",
                         "frac": count_tflops / fp32_peak_tflops, "traffic": tsum("k_count_tiles<0>", "k_count_tiles<1>"), "ms_per_step": count_ms,
                         "kernels": "k_count_tiles<plane> + k_count_tiles<cylinder> (tile-culled: ~10 % of the point x hypothesis tests "
                                    "are executed, the rest are proven non-inliers per 32-point tile; identical counts) -- an equivalent "
                                    "rate, NOT a pipe utilisation: see inlier_count_brute",
                         "algorithmic": f"{M:.0f} pts x ({Hp} x 6 + {Hc} x 16) flop", "peak_source": fp32_src},
        "inlier_count_brute": {"bound": "fp32", "achieved": brute_tflops, "peak": fp32_peak_tflops, "unit": "TFLOP/s",
                               "frac": brute_tflops / fp32_peak_tflops, "traffic": None, "ms_per_step": brute_ms,
                               "kernels": "k_count_plane<8> + k_count_cyl<4> (gm_set_count_mode(1): every test executed)",
                               "algorithmic": f"{M:.0f} pts x ({Hp} x 6 + {Hc} x 16) flop", "peak_source": fp32_src},
        "radix_sort": {"bound": "hbm", "achieved": gbs(sort_bytes, sort_ms), "peak": hbm_peak, "unit": "GB/s",
                       "frac": (gbs(sort_bytes, sort_ms) or 0.0) / hbm_peak, "traffic": sort_traffic,
                       "achieved_on_traffic": gbs(sort_traffic, sort_ms), "ms_per_step": sort_ms,
                       "kernels": f"{P_grid} x (k_rs2_hist + k_rs2_down): the neighbour-grid sort of the cropped cloud (segment form, "
                                  f"csrc/gm_sort.cuh)",
                       "algorithmic": f"20 B x {P_grid} passes x {Mc:.0f} keys (SURVEY 8(d): histogram read 4 + pair read 8 + pair write 8 per pass)",
                       "peak_source": peak_src},
        "voxel_dense": {"bound": "hbm", "achieved": gbs(vox8d_bytes, voxdense_ms), "peak": hbm_peak, "unit": "GB/s",
                        "frac": (gbs(vox8d_bytes, voxdense_ms) or 0.0) / hbm_peak, "traffic": voxdense_traffic,
                        "achieved_on_traffic": gbs(voxdense_traffic, voxdense_ms),
                        "frac_on_traffic": None if voxdense_traffic is None else gbs(voxdense_traffic, voxdense_ms) / hbm_peak,
                        "ms_per_step": voxdense_ms,
                        "kernels": "k_crop + k_voxel_accumulate_sorted + k_voxel_dense_scan + k_voxel_assign (default: sort-free dense tables)",
                        "algorithmic": f"SURVEY 8(d) sort-based count 16N + (68+16P)M + 20V = {vox8d_bytes / 1e6:.1f} MB with P={P_vox}: the work the "
                                       f"stage REPLACES; this path itself moves far less, so `frac` is an equivalent rate and "
                                       f"`frac_on_traffic` is the bandwidth actually drawn",
                        "peak_source": peak_src},
        "voxel_sort": {"bound": "hbm", "achieved": gbs(vox8d_bytes, voxsort_ms), "peak": hbm_peak, "unit": "GB/s",
                       "frac": (gbs(vox8d_bytes, voxsort_ms) or 0.0) / hbm_peak, "traffic": None, "ms_per_step": voxsort_ms,
                       "kernels": "k_crop + k_voxel_keys + radix sort + k_voxel_heads + k_voxel_centroids (gm_set_voxel_mode(1): the path the "
                                  "SURVEY 8(d) byte count describes)",
                       "algorithmic": f"16N + (68+16P)M + 20V = {vox8d_bytes / 1e6:.1f} MB, P={P_vox}", "peak_source": peak_src},
    }
    dominant = max(("inlier_count", "voxel_dense", "normals", "radix_sort"), key=lambda k: families[k]["ms_per_step"])
    roofline = dict(families[dominant])
    roofline["dominant_segment"] = dominant
    knn_leg = None
    if seg_knn is not None:
        knn_leg = {"k": 32, "normals_ms": seg_knn["normals"], "points_per_s": M / (seg_knn["normals"] * 1e-3) if seg_knn["normals"] > 0 else 0.0,
                   "scan_ms_single_stream": float(sum(seg_knn.values())),
                   "grid_cell_m": KNN_CELL, "max_radius_m": KNN_CAP,
                   "note": "gm_set_knn(32): pcl::NormalEstimation::setKSearch(32) instead of setRadiusSearch; exact k-NN, neighbours summed in "
                           "FLANN's order (normals bit-identical to the oracle's: tests/test_gpu_chain.py); the grid cell only sizes the search"}

    # ---- end to end through the C-ABI with host buffers (NCTX contexts pipelined) --------------------
    # Per step: H2D of the scan from pinned memory as 12-byte xyz records (what a PointCloud2 of x,y,z float32 carries;
    # gathered to PointXYZ on the device), the whole per-scan path, and D2H of everything cloud_cb publishes
    # (src/geometric_mapping.cpp:100-117): the cropped + compacted cloud (cloudOutput), the voxel centroids and their
    # 1-NN normals (normalsOutput markers), the frame (eigenBasisOutput), plus the builder-defined results
    # (models, labels, polyline) -- all through gm_fetch_async into pinned buffers.
    NCTX = int(os.environ.get("GM_E2E_CONTEXTS", "4"))
    host_xyz = [torch.from_numpy(np.ascontiguousarray(h.numpy()[:, :3])).pin_memory() for h in host_scans]
    VCAP = 49152   # voxels fetched per scan (a 10 m scan at leaf 0.1 has ~30k)
    ectx, outs, keep = [], [], []
    for k in range(NCTX):
        cx = new_ctx(4096)
        ectx.append(cx)
        summ = torch.empty(C.sizeof(capi.gm_scan_summary), dtype=torch.uint8).pin_memory()
        cloud = torch.empty((n, 4), dtype=torch.float32).pin_memory()
        labels = torch.empty(n, dtype=torch.uint8).pin_memory()
        slices = torch.empty(256 * C.sizeof(capi.gm_slice), dtype=torch.uint8).pin_memory()
        cen = torch.empty((VCAP, 4), dtype=torch.float32).pin_memory()
        nnn = torch.empty((VCAP, 8), dtype=torch.float32).pin_memory()
        keep.append((summ, cloud, labels, slices, cen, nnn))
        o = capi.gm_host_outputs()
        o.summary = summ.data_ptr()
        o.cloud_xyzw, o.cloud_capacity = cloud.data_ptr(), n
        o.labels, o.labels_capacity = labels.data_ptr(), n
        o.slices, o.slices_capacity = slices.data_ptr(), 256
        o.centroids_xyzw, o.nn_normal8, o.voxel_capacity = cen.data_ptr(), nnn.data_ptr(), VCAP
        outs.append(o)
    vfetch = min(n, VCAP)
    h2d = n * 12
    d2h = C.sizeof(capi.gm_scan_summary) + n * 16 + n + 256 * C.sizeof(capi.gm_slice) + vfetch * 48

    # the same with displayCloud = displayNormals = false (launch/mapping.launch:12-13 are parameters of the node): only the
    # frame, the models and the polyline come back -- the per-scan traffic of a mapper that keeps the primitives, not the cloud
    outs_small = []
    for k in range(NCTX):
        o = capi.gm_host_outputs()
        o.summary = keep[k][0].data_ptr()
        o.slices, o.slices_capacity = keep[k][3].data_ptr(), 256
        outs_small.append(o)
    d2h_small = C.sizeof(capi.gm_scan_summary) + 256 * C.sizeof(capi.gm_slice)

    def run_e2e(smp, steps, fetch=None):
        fetch = outs if fetch is None else fetch

        def e2e_step(i):
            k, s = i % NCTX, i % RING
            cx = ectx[k]
            cx.synchronize()  # results of the scan this context processed NCTX steps ago are now on the host
            cx.upload_pointcloud2_raw(host_xyz[s].data_ptr(), n, 12, 0, 4, 8)
            cx.process_scan(smp[s][0], smp[s][1])
            cx.fetch_async(fetch[k])

        for i in range(max(a.warmup, 3 * NCTX)):   # every context: plain launches, graph capture, first replay
            e2e_step(i)
        for cx in ectx:
            cx.synchronize()
        barrier()
        t0 = time.perf_counter()
        for i in range(steps):
            e2e_step(i)
        for cx in ectx:
            cx.synchronize()
        torch.cuda.synchronize()
        secs = max_over_ranks(time.perf_counter() - t0)
        if world > 1:
            dist.barrier()
        last = capi.gm_scan_summary.from_buffer_copy(bytes(keep[(steps - 1) % NCTX][0].numpy()))
        assert last.counts.n_input == n and last.counts.device_error == 0 and last.counts.n_voxels <= VCAP
        return secs

    # the host side of this leg (pinned-memory traffic of a shared box) is the noisy part of the whole bench: K steps are timed
    # three times and the MEDIAN is reported (all three are kept in e2e.repeats_ms_per_step)
    e2e_runs = sorted(run_e2e(samples, a.steps) for _ in range(3))
    e2e_s = e2e_runs[1]
    e2e_value = world * n * a.steps / e2e_s
    e2e4_s = run_e2e(samples4, steps4)
    e2es_s = run_e2e(samples, a.steps, outs_small)
    e2e_small = {"value": world * n * a.steps / e2es_s, "unit": "points/s", "ms_per_step": 1e3 * e2es_s / a.steps,
                 "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h_small,
                 "note": "displayCloud = displayNormals = false: up 12-byte xyz records, down the scan summary (frame, models, counts) and the polyline"}
    h4096["e2e_points_per_s"] = world * n * steps4 / e2e4_s
    h4096["e2e_ms_per_step"] = 1e3 * e2e4_s / steps4

    # ---- hypothesis-sharded RANSAC leg (configs[2]) ----------------------------------------------
    # Every rank holds the same scan; rank r evaluates its share of the H hypotheses.  "peer" = the library's own
    # collective (csrc/gm_comm.cuh): the counting kernel's last block stores (key, winner coefficients) into every peer's
    # mailbox over NVLink, a one-warp kernel picks the winner, the refit follows -- no host code in between.
    # "nccl" = the same round with torch.distributed's all_reduce(MAX) of the two keys (the portable path / cross-check).
    from geometric_mapping_b200 import distributed as gmd
    comm = gmd.connect_peers()
    ctx.set_comm(comm)
    shared = synth.curved_tunnel(n, seed=2)  # the same scan on every rank
    d_shared = torch.from_numpy(shared).to(dev)
    ctx.set_scan_device(d_shared.data_ptr(), n)
    ctx.crop()
    ctx.normals()
    nv = ctx.counts().n_valid
    key_t = torch.zeros(2, dtype=torch.int64, device=dev)  # torch-owned buffer for the 16-byte collective (both keys)

    def ransac_leg(Hs, reps, seed):
        sp, sc = synth.sample_indices(nv, Hs // 2, 3, seed=seed), synth.sample_indices(nv, Hs - Hs // 2, 2, seed=seed + 1)
        res = {"H": Hs, "points": nv}
        for name, fn in (("peer", lambda: ctx.ransac_sharded(sp, sc)), ("nccl", lambda: gmd.sharded_ransac_pair(ctx, sp, sc, rank, world, key_t))):
            for _ in range(3):
                fn()
            barrier()
            e0.record(stream)
            for _ in range(reps):
                fn()
            e1.record(stream)
            barrier()
            rms = max_over_ranks(e0.elapsed_time(e1)) / reps
            mp, mc = ctx.model(0), ctx.model(1)
            res[name] = {"ms_per_round": rms, "hyp_pts_per_sec": Hs * nv / (rms * 1e-3),
                         "plane_best": [mp["best_id"], mp["best_count"]], "cyl_best": [mc["best_id"], mc["best_count"]]}
        res["winners_equal"] = res["peer"]["plane_best"] == res["nccl"]["plane_best"] and res["peer"]["cyl_best"] == res["nccl"]["cyl_best"]
        res.update(ms_per_round=res["peer"]["ms_per_round"], hyp_pts_per_sec=res["peer"]["hyp_pts_per_sec"],
                   plane_best=res["peer"]["plane_best"], cyl_best=res["peer"]["cyl_best"])
        return res

    ransac = ransac_leg(a.shard_hyp, a.steps, 3)
    ransac["mode"] = ("hypotheses sharded across ranks, plane and cylinder side by side; headline = peer-memory exchange of (key, winner "
                      "coefficients) issued by the counting kernel itself, refit on every rank; 'nccl' = torch.distributed all_reduce(MAX)")
    if a.shard_hyp_large > 0:
        ransac["large"] = ransac_leg(a.shard_hyp_large, max(3, min(a.steps, 10)), 5)
    ctx.set_comm(None)

    # ---- compression of the segmented cloud (extra stage, reported separately) -------------------------
    for i in range(3):
        step(i)
        ctx.compress()
    barrier()
    e0.record(stream)
    for i in range(a.steps):
        step(i)
        ctx.compress()
    e1.record(stream)
    barrier()
    cms = max_over_ranks(e0.elapsed_time(e1)) / a.steps
    cc = ctx.compression()
    compress = {"ms_per_scan_with_compression": cms, "added_ms": cms - ms / a.steps, "ratio": float(cc.ratio),
                "bytes_in": int(cc.bytes_in), "bytes_out": int(cc.bytes_out), "total_rms_m": float(cc.total_rms),
                "n_plane": cc.n_plane, "n_cylinder": cc.n_cylinder, "n_residual": cc.n_residual,
                "n_residual_voxels": cc.n_residual_voxels}

    # ---- aggregated map cut into slabs, one per rank (configs[4]; strong scaling of ONE map) -------------
    map_leg = None
    if a.map_points > 0:
        for cx in ectx:
            cx.close()
        ctx.close()
        del dev_scans, d_shared
        torch.cuda.empty_cache()
        mbound, mleaf, mrad = 60.0, a.leaf, a.radius
        mp_all = synth.tunnel_map(a.map_points, seed=4, bound=mbound)
        lo, hi = gmd.slab_cuts(mp_all[:, 0], world, mleaf)[rank]
        slab = gmd.slab_select(mp_all, 0, lo, hi, halo=1.01 * mrad)
        del mp_all
        ns = len(slab)
        fin = np.isfinite(slab[:, :3]).all(1)
        # grid box = where the slab's points actually are (1 % of them are outliers spread over the whole crop
        # cube: those fall outside the box and are clamped into its border cells, which is correct, only slower)
        box = gmd.robust_box(slab[fin, :3]) if fin.any() else (np.zeros(3, np.float32), np.ones(3, np.float32))
        mparams = capi.default_params(boxFilterBound=mbound, neighborRadius=mrad, voxelGridLeafSize=mleaf, ransacThreshold=TAU,
                                      refitIterations=a.refit_iters)
        mctx = capi.Context(mparams, max_points=max(ns, 1), max_hypotheses=4096)
        mctx.set_stream(stream.cuda_stream)
        mctx.set_grid_box(box[0], box[1])
        mctx.set_owned_range(0, lo, hi)
        d_slab = torch.from_numpy(slab).to(dev)

        mctx.set_comm(comm)
        # where the whole map lies (known once, at set-up): only sizes the VoxelGrid tables; the box itself is computed and
        # all-reduced on the device in every pass
        mctx.set_scan_device(d_slab.data_ptr(), ns)
        mctx.crop()
        mctx.normals()
        hint = gmd.allreduce_bbox(*mctx.voxel_bbox())   # set-up only (torch.distributed); + 0.25 m of slack
        mctx.set_voxel_bbox_hint(np.maximum(np.asarray(hint[0]) - 0.25, -mbound), np.minimum(np.asarray(hint[1]) + 0.25, mbound))

        def map_pass(sp_, sc_):
            mctx.set_scan_device(d_slab.data_ptr(), ns)
            mctx.crop()
            mctx.normals()
            mctx.allreduce_voxel_bbox()   # 6 floats over peer memory, one kernel, no host round trip
            mctx.voxel()
            mctx.local_frame()
            mctx.allreduce_frame()        # the frame of the WHOLE map: sum of the slabs' scatter matrices
            for kind, smp in ((0, sp_), (1, sc_)):
                if smp is not None:
                    mctx.ransac(kind, smp)
                    mctx.ransac_select(kind)
            mctx.label()
            mctx.axis_polyline()
            mctx.compress()

        map_pass(None, None)
        mnv = mctx.counts().n_valid
        msp = synth.sample_indices(mnv, Hp, 3, seed=3 + rank) if mnv >= 3 else None
        msc = synth.sample_indices(mnv, Hc, 2, seed=4 + rank) if mnv >= 3 else None
        map_pass(msp, msc)
        barrier()
        reps = 3
        e0.record(stream)
        for _ in range(reps):
            map_pass(msp, msc)
        e1.record(stream)
        barrier()
        mms = max_over_ranks(e0.elapsed_time(e1)) / reps
        mc, mcc = mctx.counts(), mctx.compression()
        if mc.device_error:
            raise SystemExit("device-side error flag set (map leg)")
        tot_valid = mnv
        if world > 1:
            t = torch.tensor([mnv], device=dev, dtype=torch.int64)
            dist.all_reduce(t)
            tot_valid = int(t.item())
        map_leg = {"points": a.map_points, "ms_per_map": mms, "points_per_s": a.map_points / (mms * 1e-3),
                   "valid_points_all_ranks": tot_valid, "slab_points_rank0": ns, "owned_valid_rank0": mnv, "halo_m": 1.01 * mrad,
                   "voxels_rank0": mc.n_voxels, "compression_ratio_rank0": float(mcc.ratio), "rms_m_rank0": float(mcc.total_rms),
                   "mode": f"100 m tunnel map cut into {world} slab(s) at voxel faces, halo = neighbour radius, one plane + one "
                           f"cylinder per slab ({Hp}+{Hc} hypotheses each), VoxelGrid on the all-reduced global lattice; strong scaling"}
        mctx.close()
    comm.close()

    # ---- CPU baseline + parity of the same scan (rank 0, N=1 only) --------------------------------------
    cpu, parity = None, None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        from oracle import chain
        ncpu = a.cpu_points or n
        cp = np.ascontiguousarray(host_scans[0].numpy()[:ncpu])
        raw_ps, raw_cs = ring_samples(a, 0)
        t0 = time.perf_counter()
        of, ob = cpu_process_scan(cp, a, raw_ps, raw_cs, 1)
        dt = time.perf_counter() - t0
        cpu = {"value": ncpu / dt, "unit": "points/s", "cores": 1, "kind": "port",
               "sample": f"1 scan of {ncpu} points (ring scan 0), whole path from raw points on the oracle alone, single thread as the "
                         f"reference is (serial pcl::NormalEstimation + ros::spin); host has {host_threads()} usable cores; "
                         f"parity unpinned",
               "seconds": dt}
        # the CUDA path on the same raw points and sample indices, against that oracle run (never timed)
        parity = {}
        ps0, cs0 = ring_samples(a, 0, of["n_valid"])
        for canonical, name in ((True, "canonical"), (False, "fast")):
            try:
                g_ = chain.gpu_chain(cp, ps0, cs0, canonical, a.radius, a.leaf, tau=TAU, refit_iters=a.refit_iters, knn=a.knn, knn_max_radius=KNN_CAP if a.knn else 0.0)
                m_ = chain.compare(g_, of, ob, exact_normals=canonical)
                m_["exact_outputs_equal"] = True   # compare() asserts every integer / bit-pattern output
                m_["plane_best"] = [g_["plane"]["best_id"], g_["plane"]["best_count"]]
                m_["cyl_best"] = [g_["cyl"]["best_id"], g_["cyl"]["best_count"]]
            except AssertionError as e:
                m_ = {"exact_outputs_equal": False, "first_violation": str(e)}
            parity[name] = m_
        parity["oracle"] = {"n_cropped": of["n_cropped"], "n_valid": of["n_valid"], "V": of["vox"]["V"],
                            "plane_best": [int(ob["plane_best"]), int(ob["plane_counts"][ob["plane_best"]])],
                            "cyl_best": [int(ob["cyl_best"]), int(ob["cyl_counts"][ob["cyl_best"]])]}
        parity["note"] = ("CUDA path vs the oracle ALONE from the same raw points and sample indices; canonical = "
                          "gm_set_normals_mode(1) (FLANN summation order, every integer output must be equal), fast = the timed default "
                          "(neighbour sets equal, float sums differ by rounding, so cylinder counts may move)")

    if rank == 0:
        line = {
            "metric": "input points/s, per-scan segmentation+fit", "value": value, "unit": "points/s", "n_gpus": world,
            "steps": a.steps, "warmup": max(a.warmup, 3), "ms_per_step": ms / a.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(a),
            "run": {"parallelism": f"frame-parallel x{world} (each rank cycles its own ring of scans)" if world > 1 else "1 GPU",
                    "in_flight": f"{NFLIGHT} scans in flight (one context + CUDA stream each); single-scan latency in latency_ms_per_scan",
                    "mean_valid_points": M, "voxels": int(V)},
            "latency_ms_per_scan": latency_ms,
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "points/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": 1e3 * e2e_s / a.steps, "repeats_ms_per_step": [1e3 * t / a.steps for t in e2e_runs],
                    "pipeline": f"{NCTX} contexts / streams, pinned host buffers; up: 12-byte xyz records (gm_upload_pointcloud2); down: "
                                f"summary, compacted cloud (16 B/pt), labels, polyline, voxel centroids + 1-NN normals",
                    "numa_node_rank0": numa_node},
            "e2e_frame_only": e2e_small,
            "gpu_launches": int(launches),
            "roofline": roofline,
            "roofline_families": families,
            "segments_ms_per_step": seg_ms,
            "knn32": knn_leg,
            "graph": {"captures_ctx0": graph_stats[0], "replays_ctx0": graph_stats[1],
                      "note": "graph mode auto: scans of up to 524288 points (the 200k-point frames of frames_c3) replay a captured CUDA graph, "
                              "1M-point scans use plain launches (same device throughput, better overlap with the host copies of e2e)"},
            "h4096": h4096,
            "frames_c3": frames_c3,
            "ransac": ransac,
            "compress": compress,
            "map_slabs": map_leg,
            "cpu_baseline": cpu,
            "parity": parity,
        }
        emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
