"""Whole-recording detection on one GPU (RecordingDetection): one JSON line per run under --out.

    python tools/run_recording.py --out DIR --run config5 --frames 20000 --islands
    python tools/run_recording.py --out DIR --run config3 --frames 2000
    python tools/run_recording.py --out DIR --run config4 --frames 320 --block-frames 16   # several windows by default
    python tools/run_recording.py --out DIR --run scratch

The recording is synthesized block by block on the device (device.synth_echo), so it never exists at once. A line
holds frames/s over the whole recording (the synthesis of the input excluded), wall time per phase (spoke over all blocks, land,
clustering, cluster records), raw / filtered points, windows, clusters, peak device memory, and the card's name and
power limit read in the same run. --islands also runs DetectionPipeline.run_device per 1024-frame block on the same
frames (each block its own land grid and numbering) and reports its rate and how its result differs. "scratch" measures
the device memory one rb_stdbscan call takes per point (free memory before / after, fresh context) at config-3 and
config-4 density.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))

from radar_point_cloud_tracking_b200 import _lib  # noqa: E402
from radar_point_cloud_tracking_b200 import device as dev  # noqa: E402
from radar_point_cloud_tracking_b200 import synthetic as syn  # noqa: E402
from radar_point_cloud_tracking_b200.pipeline import DetectionConfig, DetectionPipeline  # noqa: E402
from radar_point_cloud_tracking_b200.recording import RecordingDetection  # noqa: E402

RUNS = {   # bench.py's workloads of the same names
    "config3": dict(cfg={}, block=512),
    "config5": dict(cfg=dict(eps_time=5.0), block=512),
    "config4": dict(cfg=dict(intensity_threshold=2.0, point_stride=2, eps_space=12.0), block=16),
}


def card() -> dict:
    out = dict(name=torch.cuda.get_device_name(0))
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                           text=True, timeout=30)
        out["power_limit"] = q.stdout.strip()
    except Exception as e:                                # noqa: BLE001
        out["power_limit"] = f"unknown ({e})"
    return out


class MemWatch:
    """Device memory the recording takes: free memory when it starts (the synthetic input buffer already allocated)
    minus the lowest free memory seen after every block and after finish (library scratch is not in torch's counts).
    Work of other processes on the same card during the run would be counted too."""

    def __init__(self):
        torch.cuda.synchronize()
        self.base = torch.cuda.mem_get_info(0)[0]
        self.min_free = self.base

    def mark(self):
        torch.cuda.synchronize()
        self.min_free = min(self.min_free, torch.cuda.mem_get_info(0)[0])

    def peak_used(self) -> int:
        return int(self.base - self.min_free)


def spec_for(frames: int, seed: int) -> syn.SweepSpec:
    return syn.SweepSpec(seed=seed, frames=frames, spokes=2048, bins=1024)


def run_recording(args, name: str) -> dict:
    r = RUNS[name]
    cfg = DetectionConfig(**r["cfg"])
    if name == "config4":
        spec = syn.SweepSpec(seed=args.seed, frames=args.frames, spokes=2048, bins=1024)
    else:
        spec = spec_for(args.frames, args.seed)
    bf = args.block_frames or r["block"]
    d = torch.device("cuda", 0)
    buf = torch.empty((bf, len(spec.gains), spec.spokes, spec.bins), dtype=torch.float32, device=d)
    mw = MemWatch()
    rec = RecordingDetection(cfg, 0, max_window_points=args.max_window_points)
    c, s, rr = rec.pipe.spoke_tables(spec.angle_units(), spec.scale(), bf, spec.bins)
    tabs = [torch.from_numpy(t).to(d) for t in (c, s, rr)]
    G = len(spec.gains)
    t_synth = 0.0
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for a in range(0, spec.frames, bf):
        nb = min(bf, spec.frames - a)
        ts = time.perf_counter()
        echo = dev.synth_echo(spec, a, nb, out=buf[:nb])
        torch.cuda.synchronize()
        t_synth += time.perf_counter() - ts
        rec.add_block(echo, *(t[:nb * G] for t in tabs), np.arange(a, a + nb))
        mw.mark()
    t_spoke = time.perf_counter() - t0 - t_synth
    del buf, echo
    res = rec.finish()
    mw.mark()
    t_finish = time.perf_counter()
    rec_t = time.perf_counter()
    recs = dev.cluster_records(res.points, res.labels, res.n_clusters) if res.labels.numel() else {}
    t_records = time.perf_counter() - rec_t
    total = t_finish - t0 - t_synth                      # the synthetic input is not part of the path
    n_win = len(res.cuts) - 1 if res.cuts is not None else 0
    line = dict(run=name, frames=spec.frames, block_frames=bf, spokes=spec.spokes, bins=spec.bins, gains=list(spec.gains),
                params=dict(eps_space=cfg.eps_space, eps_time=cfg.eps_time, min_samples=cfg.min_samples,
                            threshold=cfg.intensity_threshold, stride=cfg.point_stride),
                frames_per_s=spec.frames / total, seconds=total,
                phases_s=dict(synth_excluded=t_synth, spoke=t_spoke, land=res.timings.get("land"), cluster=res.timings.get("cluster"),
                              records=t_records),
                raw_points=int(res.raw.n), filtered_points=int(res.points.n), frames_built=res.frames_built,
                land_applied=res.land is not None, windows=n_win, plans=1 if n_win == 1 else 3 * n_win, clusters=int(res.n_clusters),
                segments=int(len(recs.get("frame", []))), recording_device_bytes_peak=mw.peak_used(),
                max_window_points=args.max_window_points, card=card())
    if args.islands:
        line["islands"] = run_islands(spec, cfg, res)
    return line


def run_islands(spec, cfg, res) -> dict:
    """run_device per 1024-frame block on the same frames: the old behaviour, each block a recording of its own."""
    pipe = DetectionPipeline(cfg, 0)
    bf = 1024
    d = torch.device("cuda", 0)
    c, s, rr = pipe.spoke_tables(spec.angle_units(), spec.scale(), bf, spec.bins)
    tabs = [torch.from_numpy(t).to(d) for t in (c, s, rr)]
    buf = torch.empty((bf, len(spec.gains), spec.spokes, spec.bins), dtype=torch.float32, device=d)
    rec_off = res.points.frame_off.cpu().numpy()
    rec_lab = res.labels.cpu().numpy()
    rec_x = res.points.x[:res.points.n].cpu().numpy()
    G = len(spec.gains)
    n_pts = n_cl = frames_same = lab_diff = pts_cmp = 0
    t_total = 0.0
    for a in range(0, spec.frames, bf):
        nb = min(bf, spec.frames - a)
        echo = dev.synth_echo(spec, a, nb, out=buf[:nb])
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = pipe.run_device(echo, *(t[:nb * G] for t in tabs), frame_ids=np.arange(a, a + nb))
        torch.cuda.synchronize()
        t_total += time.perf_counter() - t0
        n_pts += r.points.n
        n_cl += r.n_clusters
        off = r.points.frame_off.cpu().numpy()
        lab = r.labels.cpu().numpy()
        x = r.points.x[:r.points.n].cpu().numpy()
        for f in range(nb):
            g = a + f
            xa, xb = x[off[f]:off[f + 1]], rec_x[rec_off[g]:rec_off[g + 1]]
            if np.array_equal(xa, xb):                    # same filtered points: compare the labels point for point
                frames_same += 1
                pts_cmp += len(xa)
                lab_diff += int(np.count_nonzero(lab[off[f]:off[f + 1]] != rec_lab[rec_off[g]:rec_off[g + 1]]))
    return dict(block_frames=bf, seconds_excl_synth=t_total, frames_per_s=spec.frames / t_total, filtered_points=int(n_pts),
                clusters_summed_over_blocks=int(n_cl), frames_with_the_same_filtered_points=frames_same,
                labels_compared=pts_cmp, labels_differ=lab_diff)


def run_scratch(args) -> list:
    """Device memory one rb_stdbscan call takes per point, measured with a fresh context (its scratch starts empty)."""
    out = []
    for name, frames in (("config3", 64), ("config4", 4)):
        r = RUNS[name]
        cfg = DetectionConfig(**r["cfg"])
        spec = (syn.SweepSpec(seed=args.seed, frames=frames, spokes=2048, bins=1024) if name == "config4"
                else spec_for(frames, args.seed))
        rec = RecordingDetection(cfg, 0)
        d = torch.device("cuda", 0)
        c, s, rr = rec.pipe.spoke_tables(spec.angle_units(), spec.scale(), frames, spec.bins)
        rec.add_block(dev.synth_echo(spec), *(torch.from_numpy(t).to(d) for t in (c, s, rr)), np.arange(frames))
        res = rec.finish(cluster=False)
        p = res.points
        times = dev.expand_frame_times(p.frame_off, torch.arange(frames, dtype=torch.float32, device=d), p.n)
        labels = torch.empty(p.n, dtype=torch.int32, device=d)
        torch.cuda.synchronize()
        ctx = _lib.Context(0)
        free0 = torch.cuda.mem_get_info(0)[0]
        ncl = C.c_int64(0)
        _lib.check(ctx.lib.rb_stdbscan(ctx.handle, _lib.ptr(p.x), _lib.ptr(p.y), None, 1, _lib.ptr(times), p.n, float(cfg.eps_space),
                                       float(np.float32(cfg.eps_time)), int(cfg.min_samples), _lib.ptr(labels), None, C.byref(ncl),
                                       _lib.stream_ptr()), "rb_stdbscan")
        torch.cuda.synchronize()
        free1 = torch.cuda.mem_get_info(0)[0]
        ctx.close()
        out.append(dict(run="scratch", density=name, frames=frames, points=int(p.n), scratch_bytes=int(free0 - free1),
                        bytes_per_point=(free0 - free1) / max(p.n, 1), card=card()))
        del rec, res, p, times, labels
        torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--run", required=True, choices=sorted(RUNS) + ["scratch"])
    ap.add_argument("--frames", type=int, default=2000)
    ap.add_argument("--block-frames", type=int, default=0)
    ap.add_argument("--max-window-points", type=int, default=None)
    ap.add_argument("--islands", action="store_true")
    ap.add_argument("--seed", type=int, default=2025)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("run_recording.py needs a CUDA device")
    torch.cuda.set_device(0)
    lines = run_scratch(args) if args.run == "scratch" else [run_recording(args, args.run)]
    out = Path(args.out)
    out.mkdir(parents=True, exist_ok=True)
    with open(out / "recording.jsonl", "a") as fh:
        for ln in lines:
            s = json.dumps(ln)
            print(s)
            fh.write(s + "\n")


if __name__ == "__main__":
    main()
