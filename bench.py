#!/usr/bin/env python
"""Benchmark of the per-frame detection hot path (BASELINE.json metric: fused frames/s and points/s
through ST-DBSCAN; HBM GB/s of the spoke-to-point kernel vs peak).

    python bench.py --gpus N --steps K --warmup W            # our CUDA path
    python bench.py --impl reference --steps K --warmup W    # the reference's CPU path (oracle port)
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's result as DIR/*.npy

A step = one pass of the whole hot path (spoke-to-point + gain concat -> land persistence filter ->
ST-DBSCAN) over one block of synthetic frames (2048 spokes x 1024 echoes x gains 40/50/75, the
BASELINE.json config-3 shape: "gain-fused tracker with land persistence filter", reference defaults
thr 10 / stride 4 / eps 8,2,15). With N ranks every rank owns a contiguous time block of
`--frames-per-step` frames of one long recording (weak scaling) and exchanges an eps_time halo.
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

REPO = Path(__file__).resolve().parent
sys.path.insert(0, str(REPO))

METRIC = "fused_frames_per_s_through_stdbscan"
UNIT = "frames/s"

# BASELINE.json configs 2-5 as bench workloads (config 1 is the reference's CPU-runnable case: a parity test, not a bench
# line). `cfg` = what differs from the reference defaults (thr 10 / stride 4 / eps 8, 2, 15, land filter on);
# `frames` / `e2e_frames` = default block lengths; `cpu_*` = the bounded sample of the reference arm: frames per worker
# and the divisor of the angular sector it takes (1 = whole sweeps; config 4's neighbour lists do not fit a host at full
# density: SURVEY 8(d) "a documented subset ... and/or an angular sector").
WORKLOADS = {
    "config3": dict(desc="config3-shard: gain-fused 40/50/75, 2048x1024 sweeps, land filter, ST-DBSCAN eps 8/2/15 (thr 10, stride 4)",
                    gains=(40, 50, 75), cfg={}, frames=1024, e2e_frames=128, cpu_frames=64, cpu_sector=1, streams=4),
    "config2": dict(desc="config2: single-gain (50) stacked cloud of 500 sweeps, 3-D ST-DBSCAN on (x, y, intensity) with time = frame "
                         "index, eps 5/1/10, no land filter (3_stdbscan_point_clouds.py:177-182), thr 10 / stride 4",
                    gains=(50,), cfg=dict(land_filter=False, eps_space=5.0, eps_time=1.0, min_samples=10, cluster_3d=True),
                    frames=500, e2e_frames=250, cpu_frames=32, cpu_sector=1, streams=3),
    "config4": dict(desc="config4: dense clutter stress, gain-fused 40/50/75, thr 2 / stride 2 / eps 12 (~2.2 M points per frame), "
                         "land filter, ST-DBSCAN eps 12/2/15",
                    gains=(40, 50, 75), cfg=dict(intensity_threshold=2.0, point_stride=2, eps_space=12.0),
                    frames=64, e2e_frames=32, cpu_frames=11, cpu_sector=1024, streams=2, shard_in_flight=2),
    "config5": dict(desc="config5: long horizon, gain-fused 40/50/75, land filter, ST-DBSCAN eps 8/5/15 (eps_time 5: an 11-frame window, "
                         "5-frame halo between time shards), thr 10 / stride 4",
                    gains=(40, 50, 75), cfg=dict(eps_time=5.0), frames=1024, e2e_frames=128, cpu_frames=64, cpu_sector=1, streams=4),
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=32)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--shard-in-flight", type=int, default=0, help="N>1: blocks interleaved per rank (one host thread, one communicator)")
    ap.add_argument("--workload", default="config3", choices=sorted(WORKLOADS), help="BASELINE.json configuration (default: config 3, the "
                    "one the metric is quoted on)")
    ap.add_argument("--frames-per-step", type=int, default=0, help="frames per rank and step (device-resident `value`); 0 = the workload's default")
    ap.add_argument("--e2e-frames", type=int, default=0, help="frames per rank and step of the end-to-end measurement (bounds the "
                    "pinned host buffers: 3.2 GB float32 per rank at 128); 0 = the workload's default")
    ap.add_argument("--e2e-in-flight", type=int, default=2, help="blocks in flight of the end-to-end measurement")
    ap.add_argument("--spokes", type=int, default=2048)
    ap.add_argument("--bins", type=int, default=1024)
    ap.add_argument("--seed", type=int, default=2025)
    ap.add_argument("--clutter-p", type=float, default=0.003)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--streams", type=int, default=0, help="N=1: blocks in flight (host threads x CUDA streams x library contexts) "
                    "for `value`; 0 = the workload's default")
    ap.add_argument("--cpu-frames", type=int, default=0, help="frames per CPU worker in the reference/cpu_baseline sample; 0 = the workload's default")
    ap.add_argument("--shard-profile", action="store_true", help="N>1: print per-stage wall-clock of the sharded driver to stderr")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="write the result of the last timed step (what "
                    "DetectionResult.to_host() hands a caller) as float32/float64 .npy files under DIR, at most 64 MB in all")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    w = WORKLOADS[args.workload]
    args.frames_per_step = args.frames_per_step or w["frames"]
    args.e2e_frames = args.e2e_frames or w["e2e_frames"]
    args.cpu_frames = args.cpu_frames or w["cpu_frames"]
    args.shard_in_flight = args.shard_in_flight or w.get("shard_in_flight", 6)
    args.streams = args.streams or w["streams"]          # blocks in flight: 4 where the HBM-bound mask kernel dominates, 2 for the dense stress
    return args


def workload_config(args) -> dict:
    """The `config` object of the JSON line: identical keys and values in both arms (ours / reference)."""
    w = WORKLOADS[args.workload]
    p = dict(intensity_threshold=10.0, point_stride=4, land_filter=True, eps_space=8.0, eps_time=2.0, min_samples=15, cluster_3d=False)
    p.update(w["cfg"])
    return {"workload": w["desc"], "name": args.workload, "spokes": args.spokes, "bins": args.bins, "gains": list(w["gains"]),
            "seed": args.seed, "clutter_p": args.clutter_p, "params": p}


def load_traffic(frames_per_launch: int):
    """DRAM bytes (read + write) of the mask kernel per launch, from the committed ncu --set full capture,
    scaled from the captured launch size to this run's (the kernel's traffic is proportional to its input)."""
    cands = [REPO / "profiles" / n for n in ("r02_ncu_spoke_traffic.json", "r01_ncu_spoke_final_traffic.json")]
    p = next((c for c in cands if c.exists()), None)
    if p is None:
        return None, None
    d = json.loads(p.read_text())
    per_frame = (d["dram_bytes_read"] + d["dram_bytes_write"]) / d["frames_per_launch"]
    return int(per_frame * frames_per_launch), f"{d['capture']}: {d['dram_bytes_read']} B read + {d['dram_bytes_write']} B written per {d['frames_per_launch']}-frame launch, scaled to {frames_per_launch} frames"


def load_peaks():
    p = REPO / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


DUMP_BYTES = 64 << 20


def dump_outputs(host: dict, n_clusters: int, out_dir: str, suffix: str = "", budget: int = DUMP_BYTES) -> None:
    """Write one block's result as a caller receives it (``to_host()``: points, gains, labels, frame offsets and ids, plus
    the cluster count) to ``out_dir/<name><suffix>.npy`` in float32 / float64, so two builds can be compared output for
    output. Per-point arrays that would exceed ``budget`` bytes are cut to a fixed, seeded sample of points, sorted, whose
    indices are written as ``point_index``; the per-frame arrays and the cluster count are always whole."""
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    n = len(host["labels"])
    per_frame = {"frame_off": np.asarray(host["frame_off"]).astype(np.float64),
                 "frame_ids": np.asarray(host["frame_ids"]).astype(np.float64),
                 "n_clusters": np.array([n_clusters], dtype=np.float64)}
    point_bytes = 3 * 4 + 4 + 8 + 8                       # points, gains, labels, point_index
    headers = 7 * 4096                                    # room for the .npy headers
    keep = max(0, (budget - headers - sum(a.nbytes for a in per_frame.values())) // point_bytes)
    idx = np.arange(n) if n <= keep else np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
    out = {"points": np.asarray(host["points"])[idx].astype(np.float32),
           "gains": np.asarray(host["gains"])[idx].astype(np.float32),
           "labels": np.asarray(host["labels"])[idx].astype(np.float64),
           "point_index": idx.astype(np.float64), **per_frame}
    for name, a in out.items():
        np.save(d / f"{name}{suffix}.npy", a)


# ------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region: NVML through nvidia_ml_py (a query takes
    well under a millisecond, so even a 10 ms timed region gets several samples); nvidia-smi as fallback."""
    QUERY = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
    REASONS = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}

    def __init__(self, index: int, period_s: float = 0.01):
        self.index = index
        self.period = period_s
        self.rows = []            # (sm_mhz, max_mhz, power_w, reason bits)
        self._stop = threading.Event()
        self._t = threading.Thread(target=self._run, daemon=True)
        self.source = "nvml"

    def _run_nvml(self):
        import pynvml
        pynvml.nvmlInit()
        visible = os.environ.get("CUDA_VISIBLE_DEVICES")
        idx = self.index
        if visible:
            try:
                idx = int(visible.split(",")[self.index])
            except (ValueError, IndexError):
                pass
        h = pynvml.nvmlDeviceGetHandleByIndex(idx)
        mx = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
        get_reasons = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or pynvml.nvmlDeviceGetCurrentClocksThrottleReasons
        while not self._stop.is_set():
            sm = pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
            try:
                pw = pynvml.nvmlDeviceGetPowerUsage(h) / 1000.0
            except Exception:
                pw = 0.0
            self.rows.append((float(sm), float(mx), pw, int(get_reasons(h))))
            self._stop.wait(self.period)

    def _run_smi(self):
        self.source = "nvidia-smi"
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                                      "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    c = [v.strip() for v in out.splitlines()[0].split(",")]
                    bits = sum(bit for (name, bit), v in zip(self.REASONS.items(), c[3:7]) if v.lower().startswith("active"))
                    self.rows.append((float(c[0]), float(c[1]), float(c[2]) if c[2].replace(".", "").isdigit() else 0.0, bits))
            except Exception:
                pass
            self._stop.wait(0.2)

    def _run(self):
        try:
            self._run_nvml()
        except Exception:
            self._run_smi()

    def __enter__(self):
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def mark(self):
        """Index of the next sample: call at the start of the timed region."""
        return len(self.rows)

    def summary(self, first: int = 0, last=None):
        rows = self.rows[first:last] or self.rows
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        reasons = [n for n, bit in self.REASONS.items() if any(r[3] & bit for r in rows)]
        return {"sm_mhz": statistics.median(r[0] for r in rows), "sm_max_mhz": max(r[1] for r in rows),
                "power_w_max": max(r[2] for r in rows), "reasons": reasons, "samples": len(rows), "source": self.source}


# ------------------------------------------------------------------------------------ CPU (oracle port)
_CPU_CACHE = {}
_REF_T4 = []


def reference_t4():
    """The UNMODIFIED reference script ``4_temporal_object_tracker.py`` as a module, if a copy of it has been placed
    under ``baseline/_ref/PointCloudWork/`` (git-ignored: it is not part of this repository), else ``None``."""
    if not _REF_T4:
        import importlib.util
        path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "baseline", "_ref", "PointCloudWork", "4_temporal_object_tracker.py")
        mod = None
        if os.path.exists(path):
            try:
                os.environ.setdefault("MPLBACKEND", "Agg")
                spec = importlib.util.spec_from_file_location("reference_t4_unmodified", path)
                mod = importlib.util.module_from_spec(spec)
                sys.modules["reference_t4_unmodified"] = mod
                spec.loader.exec_module(mod)
                if not getattr(mod, "HAS_SKLEARN", False):
                    mod = None
            except Exception as e:                                       # a missing plotting dependency, say: the port takes over
                sys.stderr.write(f"reference T4 not importable ({e!r}); timing the oracle port instead\n")
                mod = None
        _REF_T4.append(mod)
    return _REF_T4[0]



def cpu_block_sample(args_tuple):
    """One bounded sample of the reference path on the CPU oracle: `frames` FULL-SIZE frames (all spokes, all
    gains) of the same synthetic recording, starting at `first_frame`, through spoke-to-point, gain concat,
    land filter and the reference's sequential ST-DBSCAN (numpy + scikit-learn BallTree + the reference's
    Python expansion loop). Input generation and imports are outside the timed region.
    Returns (seconds per stage, points, clusters)."""
    seed, first_frame, frames, total_frames, spokes, bins, clutter_p, gains, sector, prm = args_tuple
    prm = dict(prm)
    from oracle import numpy_oracle as O
    from radar_point_cloud_tracking_b200 import synthetic as syn

    spec = syn.SweepSpec(seed=seed, frames=max(total_frames, first_frame + frames), spokes=spokes, bins=bins, clutter_p=clutter_p,
                         gains=tuple(gains))
    key = args_tuple
    keep_spokes = max(1, spokes // max(sector, 1))                         # the angular sector of the sample (all spokes when 1)
    if key not in _CPU_CACHE:
        _CPU_CACHE.clear()
        rects = syn.build_rects(spec)
        _CPU_CACHE[key] = [[np.ascontiguousarray(syn.synth_sweep(spec, first_frame + f, g, rects)[:keep_spokes])
                            for g in range(len(spec.gains))] for f in range(frames)]
        O._query_radius(np.zeros((4, 2), np.float32), 1.0)               # import scikit-learn before the clock starts
    echo = _CPU_CACHE[key]
    T4 = None if prm["cluster_3d"] else reference_t4()                     # imported before the clock starts
    ang, scale = spec.angle_units()[:keep_spokes], spec.scale()[:keep_spokes]
    t0 = time.perf_counter()
    pts = []
    for f in range(frames):
        per_gain = {gain: O.sweep_to_points(echo[f][gi], ang, scale, prm["intensity_threshold"], prm["point_stride"])
                    for gi, gain in enumerate(spec.gains)}
        fused = O.fuse_concat(per_gain)
        pts.append(fused[0] if fused is not None else np.zeros((0, 3), np.float32))
    t1 = time.perf_counter()
    if T4 is not None:
        # land filter and ST-DBSCAN (incl. its per-frame Cluster records) by the reference's OWN functions, called the way
        # its run_pipeline does (T4:936-975) with its own land-filter constants (the workloads do not change those)
        import contextlib
        import datetime
        import io
        t_stamp = datetime.datetime(2025, 1, 1)
        with contextlib.redirect_stdout(io.StringIO()):
            frs = [T4.RadarFrame(timestamp=t_stamp, timestamp_ms=f, frame_id=f, points=p, gains=np.zeros(len(p), np.int32))
                   for f, p in enumerate(pts) if len(p)]
            if prm["land_filter"] and len(frs) > 10:
                count, isum, edges = T4.build_occupancy_grid(frs, T4.LAND_GRID_RESOLUTION)
                land = T4.identify_land_cells(count, isum, len(frs))
                frs = [T4.filter_land_from_frame(fr, land, edges) for fr in frs]
            t2 = time.perf_counter()
            by_frame = T4.st_dbscan(frs, prm["eps_space"], prm["eps_time"], prm["min_samples"])
        t3 = time.perf_counter()
        ids = {c.cluster_id for cl in by_frame.values() for c in cl}
        return (t1 - t0, t2 - t1, t3 - t2, int(sum(fr.num_points for fr in frs)), len(ids), True)
    built = [p for p in pts if len(p)]
    if prm["land_filter"] and len(built) > 10:
        count, isum, edges = O.occupancy_grid(built)
        land = O.land_cells(count, isum, len(built))
        pts = [p[O.land_keep_mask(p, land, edges)] if len(p) else p for p in pts]
    t2 = time.perf_counter()
    if prm["cluster_3d"]:                                                 # T3:177-182: coords = (x, y, z), flat labels
        coords = np.concatenate(pts) if pts else np.zeros((0, 3), np.float32)
        times = np.concatenate([np.full(len(p), f, np.float32) for f, p in enumerate(pts)]) if pts else np.zeros(0, np.float32)
        labels = O.st_dbscan_sequential(coords, times, prm["eps_space"], prm["eps_time"], prm["min_samples"])
    else:
        labels, _ = O.st_dbscan_frames(list(enumerate(pts)), prm["eps_space"], prm["eps_time"], prm["min_samples"], sequential=True)
    t3 = time.perf_counter()
    return (t1 - t0, t2 - t1, t3 - t2, int(sum(len(p) for p in pts)), int(labels.max() + 1 if len(labels) else 0), False)


def run_cpu_reference(args, steps: int, warmup: int, workers: int, frames: int = 64):
    """Times the oracle port with `workers` processes, each on its own block of `frames` consecutive full-size
    frames (the reference is single-threaded; independent time blocks are the only way to use more cores).
    A step = every worker finishing one block; value = frames of all workers / slowest worker's time."""
    import multiprocessing as mp

    workers = max(1, workers)
    ctx = mp.get_context("spawn")
    times, detail = [], None
    total = frames * workers
    w = WORKLOADS[args.workload]
    sector = int(w["cpu_sector"])
    prm = tuple(sorted(workload_config(args)["params"].items()))
    with ctx.Pool(workers) as pool:
        jobs = [(args.seed, i * frames, frames, total, args.spokes, args.bins, args.clutter_p, tuple(w["gains"]), sector, prm)
                for i in range(workers)]
        for it in range(warmup + steps):
            res = pool.map(cpu_block_sample, jobs, chunksize=1)
            dt = max(r[0] + r[1] + r[2] for r in res)
            if it >= warmup:
                times.append(dt)
                detail = res
    mean_t = sum(times) / len(times)
    what = (f"consecutive full-size frames ({args.spokes}x{args.bins} x {len(w['gains'])} gain(s))" if sector == 1 else
            f"consecutive frames cut to an angular sector of 1/{sector} of the spokes ({max(1, args.spokes // sector)}x{args.bins} x "
            f"{len(w['gains'])} gains, at the recording's true density; value = frames x 1/{sector} per second, which FAVOURS the CPU: "
            f"its cost grows faster than the sector)")
    real = all(r[5] for r in detail)
    how = ("land filter, ST-DBSCAN and Cluster records by the functions of the UNMODIFIED reference script (baseline/_ref/PointCloudWork/"
           "4_temporal_object_tracker.py: build_occupancy_grid, identify_land_cells, filter_land_from_frame, st_dbscan), spoke-to-point "
           "(T4:200-232, which the reference only has inside its CSV reader) by the numpy port pinned to it"
           if real else
           "numpy/scikit-learn oracle port of the reference incl. its sequential ST-DBSCAN expansion")
    return {"value": frames * workers / sector / mean_t, "ms_per_step": mean_t * 1e3, "cores": workers,
            "kind": "reference" if real else "port",
            "sample": f"{workers} worker(s) x {frames} {what} of the same "
                      f"synthetic recording; {how}; input generation untimed; the reference's cost per frame grows with the "
                      f"block length (spatial-only BallTree over all frames, T4:474-475)",
            "stage_seconds": [float(sum(r[i] for r in detail) / len(detail)) for i in range(3)],
            "points_per_sample": int(sum(r[3] for r in detail) / len(detail)),
            "clusters_per_sample": int(sum(r[4] for r in detail) / len(detail))}


# ------------------------------------------------------------------------------------ ours
def check_sharded_labels(args, cfg, wl, rank, world, device):
    """Before anything is timed at N > 1: a small recording (same workload parameters, 12 frames x 512 spokes per rank)
    through the time-sharded path on all ranks AND, on rank 0, through the single-GPU path as one block; labels and
    points must be identical id for id. The JSON line carries the outcome (`sharded_labels_identical`)."""
    import torch
    import torch.distributed as dist

    from radar_point_cloud_tracking_b200 import device as dev
    from radar_point_cloud_tracking_b200 import synthetic as syn
    from radar_point_cloud_tracking_b200.pipeline import DetectionPipeline
    from radar_point_cloud_tracking_b200.sharded import ShardedDetection

    Bc = 12
    spec = syn.SweepSpec(seed=args.seed + 1, frames=Bc * world, spokes=512, bins=args.bins, clutter_p=max(args.clutter_p, 0.004),
                         gains=tuple(wl["gains"]))
    sd = ShardedDetection(cfg, rank, world, device.index)
    first = rank * Bc
    echo = dev.synth_echo(spec, first_frame=first, n_frames=Bc, device=device)
    tabs = [torch.from_numpy(t).to(device) for t in sd.base.spoke_tables(spec.angle_units(), spec.scale(), Bc, spec.bins)]
    res = sd.run_device(echo, *tabs, np.arange(first, first + Bc))
    host = res.to_host()
    gathered = [None] * world
    dist.gather_object({"labels": host["labels"], "points": host["points"], "ncl": res.n_clusters}, gathered if rank == 0 else None, dst=0)
    out = None
    if rank == 0:
        pipe = DetectionPipeline(cfg, device.index)
        full = dev.synth_echo(spec, device=device)
        tabs = [torch.from_numpy(t).to(device) for t in pipe.spoke_tables(spec.angle_units(), spec.scale(), spec.frames, spec.bins)]
        want = pipe.run_device(full, *tabs)
        wh = want.to_host()
        got_l = np.concatenate([g["labels"] for g in gathered])
        got_p = np.concatenate([g["points"] for g in gathered])
        same = bool(np.array_equal(got_p, wh["points"]) and np.array_equal(got_l, wh["labels"]) and
                    all(g["ncl"] == want.n_clusters for g in gathered))
        out = {"identical": same, "points": int(len(got_l)), "clusters": int(want.n_clusters), "frames": int(spec.frames),
               "what": f"{Bc} frames x 512 spokes per rank, workload parameters, sharded x{world} vs one block on rank 0"}
    flag = torch.tensor([1 if (out is None or out["identical"]) else 0], device=device)
    dist.broadcast(flag, src=0)
    torch.cuda.synchronize()
    return out


def run_ours(args):
    import torch
    import torch.distributed as dist

    from radar_point_cloud_tracking_b200 import _lib, device as dev
    from radar_point_cloud_tracking_b200 import synthetic as syn
    from radar_point_cloud_tracking_b200.pipeline import DetectionConfig, DetectionPipeline

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    numa_cpus = _lib.bind_to_gpu_numa(local_rank)        # before any pinned allocation: host buffers next to the GPU
    if world > 1:
        dist.init_process_group("nccl", device_id=device)

    B = args.frames_per_step
    wl = WORKLOADS[args.workload]
    G = len(wl["gains"])
    spec = syn.SweepSpec(seed=args.seed, frames=B * world, spokes=args.spokes, bins=args.bins, clutter_p=args.clutter_p,
                         gains=tuple(wl["gains"]))
    cfg = DetectionConfig(gains=tuple(wl["gains"]), **wl["cfg"])
    sharded_check = None
    if world > 1:
        if cfg.cluster_3d:
            raise SystemExit("bench.py: config2 (3-D single-gain clustering) is a single-GPU workload (BASELINE.json: '1 B200')")
        from radar_point_cloud_tracking_b200.sharded import ShardedDetection
        pipe = ShardedDetection(cfg, rank, world, device.index)
        sharded_check = check_sharded_labels(args, cfg, wl, rank, world, device)
    else:
        pipe = DetectionPipeline(cfg, device.index)
    first = rank * B
    frame_ids = np.arange(first, first + B)

    # inputs resident in HBM before the timed region (device generator == numpy generator, tested)
    echo = dev.synth_echo(spec, first_frame=first, n_frames=B, device=device)
    base = pipe.base if hasattr(pipe, "base") else pipe
    c, s, r = base.spoke_tables(spec.angle_units(), spec.scale(), B, args.bins)
    d_c, d_s, d_r = (torch.from_numpy(t).to(device) for t in (c, s, r))
    torch.cuda.synchronize()

    ctx = base.ctx
    hbm_peak, peak_src = load_peaks()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(fn, steps, warmup, collect=None):
        for _ in range(warmup):
            fn()
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = ctx.launch_count()
        ev0.record()
        for _ in range(steps):
            out = fn()
            if collect is not None:
                collect(out)
        ev1.record()
        barrier()
        ms = ev0.elapsed_time(ev1)
        if world > 1:
            t = torch.tensor([ms], device=device, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, ctx.launch_count() - l0

    # ---- device-resident throughput -----------------------------------------------------------------
    results = []
    overlapped = None
    with ClockSampler(device.index) as clocks:
        if world == 1 and args.streams > 1:
            # throughput path: `streams` host threads, each with its own CUDA stream and library context, run whole
            # blocks concurrently; timed from an event recorded before the first block is submitted to an event the
            # current stream records after waiting for every block
            from radar_point_cloud_tracking_b200.pipeline import OverlappedPipeline
            overlapped = OverlappedPipeline(cfg, device.index, workers=args.streams)
            block = ((echo, d_c, d_s, d_r, frame_ids), {})
            overlapped.map([block] * max(args.warmup, 2 * args.streams), keep=False)
            barrier()
            l0 = overlapped.launch_count()
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c0 = clocks.mark()
            ev0.record()
            results = overlapped.map([block] * args.steps, start_event=ev0, keep=False)
            ev1.record()
            barrier()
            c1 = clocks.mark()
            ms, launches = ev0.elapsed_time(ev1), overlapped.launch_count() - l0
        else:
            if world > 1:                                   # warm every block slot (stream, library context, allocator pool)
                pipe.run_blocks([(echo, d_c, d_s, d_r, frame_ids)] * max(args.warmup, 2 * args.shard_in_flight), keep=False, in_flight=args.shard_in_flight)
            else:
                for _ in range(args.warmup):
                    pipe.run_device(echo, d_c, d_s, d_r, frame_ids)
            keep_last = lambda r: results.__setitem__(slice(None), [r])        # earlier results are released: their buffers get recycled
            if world > 1:
                # time-sharded: `streams` blocks are interleaved inside every rank (generators that yield at every host
                # read-back, each on its own CUDA stream and library context); one communicator, one host thread
                blk = (echo, d_c, d_s, d_r, frame_ids)
                barrier()
                l0 = _lib.launch_count_all()
                ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                c0 = clocks.mark()
                ev0.record()
                results = pipe.run_blocks([blk] * args.steps, keep=False, in_flight=args.shard_in_flight)
                ev1.record()
                barrier()
                c1 = clocks.mark()
                tmax = torch.tensor([ev0.elapsed_time(ev1)], device=device, dtype=torch.float64)
                dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
                ms, launches = float(tmax.item()), _lib.launch_count_all() - l0
            else:
                c0 = clocks.mark()
                ms, launches = timed(lambda: pipe.run_device(echo, d_c, d_s, d_r, frame_ids), args.steps, 0, collect=keep_last)
                c1 = clocks.mark()
    res = results[-1]
    if args.dump_outputs:
        dump_outputs(res.to_host(), res.n_clusters, args.dump_outputs, f"_rank{rank}" if world > 1 else "", DUMP_BYTES // world)
    n_raw, n_pts = res.raw.n, res.points.n
    echo_bytes = B * G * args.spokes * args.bins * 4
    spoke_bytes = echo_bytes + B * G * args.spokes * 12 + 16 * n_raw          # SURVEY.md 8(d), whole stage
    # per-kernel split of the stage: a few extra (untimed) steps with events recorded inside the library,
    # on the launch stream, around each of the three kernels
    ctx.set_option("spoke_profile", 1)
    split = []
    for _ in range(3):
        pipe.run_device(echo, d_c, d_s, d_r, frame_ids)
        split.append([ctx.info(k) * 1e-6 for k in ("spoke_mask_ns", "spoke_offsets_ns", "spoke_emit_ns")])
    ctx.set_option("spoke_profile", 0)
    st = dev.stdbscan_stats(device.index)              # counters of a device-resident block of the timed size (not of the e2e runs)
    mask_ms, offs_ms, emit_ms = (sum(r[i] for r in split) / len(split) for i in range(3))
    achieved = echo_bytes / (mask_ms * 1e-3) / 1e9 if mask_ms > 0 else 0.0
    spoke_ms_mean = mask_ms + offs_ms + emit_ms                               # first event to last event of the stage
    stage_gbs = spoke_bytes / (spoke_ms_mean * 1e-3) / 1e9 if spoke_ms_mean > 0 else 0.0
    traffic, traffic_src = load_traffic(B)
    frames_total = B * world * args.steps
    value = frames_total / (ms * 1e-3)
    pts_t = torch.tensor([n_raw, n_pts, res.n_clusters], device=device, dtype=torch.int64)
    if world > 1:
        dist.all_reduce(pts_t)
    n_raw_all, n_pts_all = int(pts_t[0]), int(pts_t[1])

    # ---- end to end through the host API -------------------------------------------------------------
    # Host buffers in (pinned), host buffers out, every step: the echo block crosses PCIe, the points / labels come back.
    # Two blocks are in flight (N = 1: two worker streams; N > 1: two interleaved block slots per rank), so the upload
    # of one block runs under the kernels and the read-back of the other. Timed by the wall clock between device
    # synchronisations (the host's share - spoke tables, unpacking the result - belongs to an end-to-end number).
    e2e = e2e_u8 = None
    if not args.no_e2e:
        Be = max(1, min(args.e2e_frames, B))
        e_ids = frame_ids[:Be]
        e_steps = args.steps
        ov2 = None
        if world == 1:
            from radar_point_cloud_tracking_b200.pipeline import OverlappedPipeline
            ov2 = OverlappedPipeline(cfg, device.index, workers=args.e2e_in_flight)

        def e2e_run(host_t):
            if world == 1:
                run = lambda k: ov2.map_host([((None, spec.angle_units(), spec.scale(), e_ids), {"pinned": host_t})] * k)
            else:
                run = lambda k: pipe.run_host_blocks([(host_t, spec.angle_units(), spec.scale(), e_ids)] * k, in_flight=args.e2e_in_flight)
            run(args.e2e_in_flight)                                          # warm-up: every slot, its buffers and context
            barrier()
            t0 = time.perf_counter()
            outs = run(e_steps)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            if world > 1:
                t = torch.tensor([dt], device=device, dtype=torch.float64)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                dt = float(t.item())
            barrier()
            return dt * 1e3, outs[-1]

        host_echo = torch.empty(echo[:Be].shape, dtype=torch.float32, pin_memory=True)
        host_echo.copy_(echo[:Be])
        torch.cuda.synchronize()
        # what the platform gives: the same pinned buffer copied to the device and nothing else, all ranks at once
        d_tmp = torch.empty_like(echo[:Be])
        d_tmp.copy_(host_echo, non_blocking=True)
        barrier()
        t0 = time.perf_counter()
        for _ in range(3):
            d_tmp.copy_(host_echo, non_blocking=True)
        torch.cuda.synchronize()
        copy_s = (time.perf_counter() - t0) / 3
        if world > 1:
            t = torch.tensor([copy_s], device=device, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            copy_s = float(t.item())
        del d_tmp
        ms_e, out_f = e2e_run(host_echo)
        e2e = {"value": Be * world * e_steps / (ms_e * 1e-3), "unit": UNIT, "frames_per_step_per_gpu": Be, "steps": e_steps,
               "h2d_bytes_per_step": int(out_f["h2d_bytes"]), "d2h_bytes_per_step": int(out_f["d2h_bytes"]),
               "ms_per_step": ms_e / e_steps, "host_buffers": "float32 echoes (the reference's in-memory type), pinned",
               "blocks_in_flight": args.e2e_in_flight, "timing": "wall clock between device synchronisations, max over ranks",
               "h2d_copy_only": {"ms_per_step": copy_s * 1e3, "gb_per_s_per_gpu": host_echo.numel() * 4 / copy_s / 1e9,
                                 "frames_per_s": Be * world / copy_s,
                                 "note": "the pinned echo buffer copied to the device and nothing else, all ranks at once: the "
                                         "ceiling the platform's host-to-device path sets for this end-to-end number"}}
        del host_echo
        # the same with the radar's native uint8 echoes in the pinned host buffer (identical results, a quarter of the
        # bytes over PCIe) - the transport the drop-in uses when it parses sweeps itself; reported next to the float32
        # number, which stays the headline
        host_u8 = torch.empty(echo[:Be].shape, dtype=torch.uint8, pin_memory=True)
        host_u8.copy_(echo[:Be].to(torch.uint8))
        torch.cuda.synchronize()
        ms_u, out_u = e2e_run(host_u8)
        e2e_u8 = {"value": Be * world * e_steps / (ms_u * 1e-3), "unit": UNIT, "frames_per_step_per_gpu": Be, "steps": e_steps,
                  "h2d_bytes_per_step": int(out_u["h2d_bytes"]), "d2h_bytes_per_step": int(out_u["d2h_bytes"]), "ms_per_step": ms_u / e_steps,
                  "labels_equal_float32_run": bool(np.array_equal(out_u["labels"], out_f["labels"]))}
        del host_u8
        if ov2 is not None:
            ov2.close()

    if args.shard_profile and world > 1:
        pipe.profile, pipe.timings = True, {}
        for _ in range(3):
            pipe.run_device(echo, d_c, d_s, d_r, frame_ids)
        pipe.profile = False
        sys.stderr.write("rank %d shard stages (ms/step): %s\n" % (rank, {k: round(v / 3 * 1e3, 3) for k, v in pipe.timings.items()}))
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32 (points) / f64 (neighbour test) / i32 (labels)", "data": "synthetic",
        "config": workload_config(args),
        "run": {"frames_per_step_per_gpu": B, "numa_bound_cpus": len(numa_cpus) if numa_cpus else None,
                "parallelism": f"time-sharded x{world}, {args.shard_in_flight} blocks interleaved per rank (one communicator)" if world > 1 else f"single GPU, {args.streams if overlapped else 1} block(s) in flight",
                "l2_policy": "inputs larger than L2 (echo block %.2f GB per step)" % (echo.numel() * 4 / 1e9)},
        "points_per_s": n_raw_all * args.steps / (ms * 1e-3),
        "points_per_step": {"after_stride": n_raw_all, "after_land_filter": n_pts_all, "clusters": int(pts_t[2])},
        "roofline": {"bound": "hbm", "kernel": "spoke_mask_tma_kernel", "achieved": achieved, "peak": hbm_peak,
                     "unit": "GB/s", "frac": achieved / hbm_peak, "frac_of_nominal_8TBs": achieved / 8000.0,
                     "peak_source": peak_src, "traffic": traffic, "traffic_source": traffic_src,
                     "algorithmic_bytes_per_launch": echo_bytes,
                     "kernel_ms": mask_ms, "share_of_step": mask_ms / (ms / args.steps),
                     "note": "dominant kernel of the spoke-to-point stage: reads every echo byte once (algorithmic "
                             "bytes = echo tensor only; its 1-bit/cell mask output is overhead, not counted)",
                     "stage": {"kernels_ms": {"spoke_mask_kernel": mask_ms, "spoke_offsets_kernel": offs_ms,
                                              "spoke_emit_kernel": emit_ms},
                               "stage_ms": spoke_ms_mean, "algorithmic_bytes": spoke_bytes,
                               "achieved": stage_gbs, "frac": stage_gbs / hbm_peak,
                               "note": "whole rb_spoke_to_points call (3 launches), first to last CUDA event recorded inside the "
                                       "library on the launch stream; bytes = echo + spoke tables + 16 B per kept point"}},
        "stdbscan": {"pair_tests_per_step": st["pair_tests_count"] + st["pair_tests_union"] + st["pair_tests_border"],
                     "pair_tests": [st["pair_tests_count"], st["pair_tests_union"], st["pair_tests_border"]], "tight": st["tight"],
                     "cells": st["n_cells"], "dims": st["dims"], "time_radius": st["time_radius"],
                     "pair_tests_per_s": (st["pair_tests_count"] + st["pair_tests_union"] + st["pair_tests_border"]) * (value / B),
                     "note": "counters of one device-resident block on rank 0 (neighbour-count / union / border kernels); per second = "
                             "per block x blocks per second of the whole job"},
        "gpu_launches": launches,
        "clocks": clocks.summary(c0, c1),
    }
    if sharded_check is not None:
        line["sharded_labels_identical"] = sharded_check["identical"]
        line["sharded_check"] = sharded_check
    if e2e:
        line["e2e"] = e2e
        line["e2e_uint8_echoes"] = e2e_u8
    if not args.no_cpu_baseline:
        cb = run_cpu_reference(args, steps=1, warmup=0, workers=1, frames=args.cpu_frames)
        line["cpu_baseline"] = {"value": cb["value"], "unit": UNIT, "cores": cb["cores"], "kind": cb["kind"],
                                "sample": cb["sample"], "stage_seconds": cb["stage_seconds"],
                                "host_cpus": os.cpu_count()}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    workers = max(1, min(os.cpu_count() or 1, 32))
    # every worker keeps its block of float32 sweeps in memory (input generation stays outside the timed region): leave
    # at least half of the available RAM alone
    try:
        import psutil
        w = WORKLOADS[args.workload]
        per_worker = args.cpu_frames * len(w["gains"]) * max(1, args.spokes // int(w["cpu_sector"])) * args.bins * 4 * 1.5 + 1.5e9
        workers = max(1, min(workers, int(psutil.virtual_memory().available * 0.5 / per_worker)))
    except Exception:
        pass
    steps = max(1, min(args.steps, 2))
    warm = min(args.warmup, 1)
    cb = run_cpu_reference(args, steps=steps, warmup=warm, workers=workers, frames=args.cpu_frames)
    line = {
        "impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": steps, "warmup": warm, "ms_per_step": cb["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32/f64 (numpy, scikit-learn)", "data": "synthetic",
        "config": workload_config(args),
        "cpu_baseline": {"value": cb["value"], "unit": UNIT, "cores": cb["cores"], "kind": cb["kind"], "sample": cb["sample"],
                         "stage_seconds": cb["stage_seconds"], "host_cpus": os.cpu_count()},
        "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def main():
    args = parse_args()
    # exactly ONE line on stdout: libraries under us (NCCL's version banner, for one) write to fd 1, so fd 1
    # points at stderr while the benchmark runs and is restored for the JSON line
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    buf = []
    try:
        import builtins
        real_print = builtins.print
        builtins.print = lambda *a, **k: buf.append(" ".join(str(x) for x in a)) if k.get("file") in (None, sys.stdout) else real_print(*a, **k)
        try:
            if args.impl == "reference":
                run_reference(args)
            else:
                run_ours(args)
        finally:
            builtins.print = real_print
    finally:
        sys.stdout.flush()
        os.dup2(saved, 1)
        os.close(saved)
    for line in buf:
        print(line)
    sys.stdout.flush()


if __name__ == "__main__":
    main()
