"""The PointCloudWorkF clustering (DetectionConfig.min_frames) of a whole recording on one GPU: one JSON line per run.

    python tools/run_recording_wf.py [--out profiles/r05_recording_wf.jsonl] [--frames 2048] [--repeats 5]

A config-5 recording (2048 x 1024 x 3 gains, eps_time 5) is synthesized block by block on the device and detected by
RecordingDetection without clustering; its filtered points are then labelled twice:
  one_window  rb_stdbscan_windowed_wf in one window (= rb_stdbscan_wf, min_frames 3) next to the T4 clustering
              (rb_stdbscan_windowed) of the same points, also in one window
  windows     rb_stdbscan_windowed_wf with at most an eighth of the points per window (>= 8 windows), checked against
              the one-window labels, core flags and cluster count
Times are the host clock around each call (every call ends in a stream sync), after one warm-up call, as the median and
minimum of --repeats calls. Each line carries the card's name and power limit, read in the same run.
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
from radar_point_cloud_tracking_b200.recording import RecordingDetection, plan_windows, stdbscan_windowed  # noqa: E402


def card() -> dict:
    out = dict(name=torch.cuda.get_device_name(0))
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                           text=True, timeout=30)
        out["power_limit"] = q.stdout.strip()
    except Exception as e:                                # noqa: BLE001
        out["power_limit"] = f"unknown ({e})"
    return out


def timed(fn, repeats: int):
    """(result of the last call, median seconds, min seconds) over `repeats` calls after one warm-up call."""
    out = fn()
    ts = []
    for _ in range(repeats):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    return out, float(np.median(ts)), float(np.min(ts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(Path(__file__).resolve().parents[1] / "profiles" / "r05_recording_wf.jsonl"))
    ap.add_argument("--frames", type=int, default=2048)
    ap.add_argument("--block-frames", type=int, default=512)
    ap.add_argument("--min-frames", type=int, default=3)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--seed", type=int, default=2025)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("run_recording_wf.py needs a CUDA device")
    torch.cuda.set_device(0)
    d = torch.device("cuda", 0)
    spec = syn.SweepSpec(seed=args.seed, frames=args.frames, spokes=2048, bins=1024)
    cfg = DetectionConfig(eps_time=5.0, min_frames=args.min_frames)
    rec = RecordingDetection(cfg, 0)
    bf = args.block_frames
    c, s, r = rec.pipe.spoke_tables(spec.angle_units(), spec.scale(), bf, spec.bins)
    tabs = [torch.from_numpy(t).to(d) for t in (c, s, r)]
    G = len(spec.gains)
    for a in range(0, spec.frames, bf):
        nb = min(bf, spec.frames - a)
        echo = dev.synth_echo(spec, a, nb)
        rec.add_block(echo, *(t[:nb * G] for t in tabs), np.arange(a, a + nb))
        del echo
    res = rec.finish(cluster=False)
    p = res.points
    off = p.frame_off.cpu().numpy()
    ids = res.frame_ids
    h = int(np.floor(np.float32(cfg.eps_time)))
    one = np.array([0, spec.frames], np.int64)
    many = plan_windows(off, h, p.n // 8)
    common = dict(frames=spec.frames, spokes=spec.spokes, bins=spec.bins, gains=list(spec.gains),
                  params=dict(eps_space=cfg.eps_space, eps_time=cfg.eps_time, min_samples=cfg.min_samples, min_frames=cfg.min_frames),
                  filtered_points=int(p.n), land_applied=res.land is not None, repeats=args.repeats, card=card())

    def wf(cuts):
        return stdbscan_windowed(p.x, p.y, None, off, ids, cuts, cfg.eps_space, cfg.eps_time, cfg.min_samples, bounds4=rec._b4,
                                 min_frames=cfg.min_frames)

    def t4(cuts):
        return stdbscan_windowed(p.x, p.y, None, off, ids, cuts, cfg.eps_space, cfg.eps_time, cfg.min_samples, bounds4=rec._b4)

    (lab1, core1, ncl1), wf_med, wf_min = timed(lambda: wf(one), args.repeats)
    (lab_t4, _, ncl_t4), t4_med, t4_min = timed(lambda: t4(one), args.repeats)
    lines = [dict(run="one_window", windows=1, **common, wf_seconds_median=wf_med, wf_seconds_min=wf_min, wf_clusters=int(ncl1),
                  wf_core_points=int(core1.sum().item()), wf_labelled_points=int((lab1 >= 0).sum().item()),
                  t4_seconds_median=t4_med, t4_seconds_min=t4_min, t4_clusters=int(ncl_t4),
                  t4_labelled_points=int((lab_t4 >= 0).sum().item()))]
    del lab_t4
    (labk, corek, nclk), k_med, k_min = timed(lambda: wf(many), args.repeats)
    same = bool(torch.equal(labk, lab1) and torch.equal(corek, core1) and nclk == ncl1)
    lines.append(dict(run="windows", windows=len(many) - 1, plans=3 * (len(many) - 1), **common, wf_seconds_median=k_med,
                      wf_seconds_min=k_min, wf_clusters=int(nclk), equal_to_one_window=same))
    out = Path(args.out)
    out.parent.mkdir(parents=True, exist_ok=True)
    with open(out, "a") as fh:
        for ln in lines:
            s = json.dumps(ln)
            print(s)
            fh.write(s + "\n")
    if not same:
        raise SystemExit("the windowed labels differ from the one-window labels")


if __name__ == "__main__":
    main()
