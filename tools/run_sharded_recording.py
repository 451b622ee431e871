"""The multi-GPU recording's protocol on one GPU next to RecordingDetection: one JSON line per run under --out.

    python tools/run_sharded_recording.py --out DIR --frames 20000                 # config 5 (eps_time 5)
    python tools/run_sharded_recording.py --out DIR --frames 2000 --max-window-points 4000000

The same recording (synthesized block by block on the device, 512-frame blocks, never all at once) goes once through
RecordingDetection.finish and once through ShardedRecording's protocol at world 1 (ShardedRecording._finish_protocol:
every collective is the identity there, so what remains is the protocol's own cost - gathers of host vectors, the halo
bookkeeping, the three windowed pass entries called one by one and the stitch in Python). A line holds the wall time of
each finish, the protocol's per-stage times (stats, land, layout and halos, each pass, stitch), whether the two results
are identical, peak device memory of each run, and the card's name and power limit read in the same run. Times of
several ranks are not measured by this script: it needs one GPU per rank and NCCL (tools/check_sharded_recording.py).
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))

from radar_point_cloud_tracking_b200 import device as dev  # noqa: E402
from radar_point_cloud_tracking_b200 import synthetic as syn  # noqa: E402
from radar_point_cloud_tracking_b200.pipeline import DetectionConfig  # noqa: E402
from radar_point_cloud_tracking_b200.recording import RecordingDetection  # noqa: E402
from radar_point_cloud_tracking_b200.sharded import ShardedRecording  # noqa: E402


def card() -> dict:
    out = dict(name=torch.cuda.get_device_name(0))
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                           text=True, timeout=30)
        out["power_limit"] = q.stdout.strip()
    except Exception as e:                                # noqa: BLE001
        out["power_limit"] = f"unknown ({e})"
    return out


def feed(rec, spec, bf: int) -> float:
    """All frames in blocks of ``bf``; returns the seconds spent synthesizing the input (not part of the path)."""
    d = torch.device("cuda", 0)
    buf = torch.empty((bf, len(spec.gains), spec.spokes, spec.bins), dtype=torch.float32, device=d)
    c, s, rr = rec.pipe.spoke_tables(spec.angle_units(), spec.scale(), bf, spec.bins)
    tabs = [torch.from_numpy(t).to(d) for t in (c, s, rr)]
    G = len(spec.gains)
    t_synth = 0.0
    for a in range(0, spec.frames, bf):
        nb = min(bf, spec.frames - a)
        ts = time.perf_counter()
        echo = dev.synth_echo(spec, a, nb, out=buf[:nb])
        torch.cuda.synchronize()
        t_synth += time.perf_counter() - ts
        rec.add_block(echo, *(t[:nb * G] for t in tabs), np.arange(a, a + nb))
    return t_synth


def run(args, kind: str) -> tuple:
    spec = syn.SweepSpec(seed=args.seed, frames=args.frames, spokes=2048, bins=1024)
    cfg = DetectionConfig(eps_time=args.eps_time, min_frames=args.min_frames)
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats(0)
    free0 = torch.cuda.mem_get_info(0)[0]
    if kind == "recording":
        rec = RecordingDetection(cfg, 0, max_window_points=args.max_window_points)
        feed(rec, spec, args.block_frames)
        t0 = time.perf_counter()
        res = rec.finish()
    else:
        rec = ShardedRecording(cfg, rank=0, world=1, max_window_points=args.max_window_points)
        feed(rec, spec, args.block_frames)
        t0 = time.perf_counter()
        res = rec._finish_protocol()
    torch.cuda.synchronize()
    t_finish = time.perf_counter() - t0
    free1 = torch.cuda.mem_get_info(0)[0]
    host = dict(x=res.points.x[:res.points.n].cpu().numpy(), labels=res.labels.cpu().numpy(),
                core=res.core.cpu().numpy() if res.core is not None else None, ncl=res.n_clusters)
    line = dict(kind=kind, frames=spec.frames, eps_time=cfg.eps_time, min_frames=cfg.min_frames, finish_s=t_finish,
                timings_s={k: float(v) for k, v in res.timings.items()}, raw_points=int(res.raw.n), filtered_points=int(res.points.n),
                windows=len(res.cuts) - 1 if res.cuts is not None else 0, clusters=int(res.n_clusters),
                torch_peak_bytes=int(torch.cuda.max_memory_allocated(0)), device_bytes_after_finish=int(free0 - free1),
                max_window_points=args.max_window_points)
    del rec, res
    return line, host


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--frames", type=int, default=20000)
    ap.add_argument("--eps-time", type=float, default=5.0)
    ap.add_argument("--min-frames", type=int, default=None)
    ap.add_argument("--block-frames", type=int, default=512)
    ap.add_argument("--max-window-points", type=int, default=None)
    ap.add_argument("--seed", type=int, default=2025)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("run_sharded_recording.py needs a CUDA device")
    torch.cuda.set_device(0)
    lines, hosts = [], []
    for kind in ("recording", "protocol_world1"):
        ln, h = run(args, kind)
        lines.append(ln)
        hosts.append(h)
    a, b = hosts
    same = (np.array_equal(a["x"], b["x"]) and np.array_equal(a["labels"], b["labels"]) and a["ncl"] == b["ncl"]
            and ((a["core"] is None and b["core"] is None) or np.array_equal(a["core"], b["core"])))
    c = card()
    for ln in lines:
        ln["identical"] = bool(same)
        ln["card"] = c
    lines[1]["overhead_s"] = lines[1]["finish_s"] - lines[0]["finish_s"]
    out = Path(args.out)
    out.mkdir(parents=True, exist_ok=True)
    with open(out / "sharded_recording.jsonl", "a") as fh:
        for ln in lines:
            s = json.dumps(ln)
            print(s)
            fh.write(s + "\n")


if __name__ == "__main__":
    main()
