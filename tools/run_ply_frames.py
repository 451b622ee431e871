"""PLY output of whole fused recordings (T5's output stage): one JSON line per run.

    python tools/run_ply_frames.py [--frames 64] [--repeats 3] [--dir DIR] [--out profiles/r07_ply_frames.jsonl]

Input: ``fusion.fuse_frames_max`` of --frames full-size synthetic frames at T5's settings (2048 spokes x 1024 bins x 3
gains, threshold 5, stride 8, resolution 1.0), as in r06, kept on the device. Two paths write one ASCII PLY per frame
(x, y, max intensity, ``intensity_to_rgb(max intensity)``), alternating, --repeats times each, into a temporary directory
under --dir (default: tmpfs when there is one, as r06):
(host)   r06's loop (c): ``FusedFrames.frames()`` (one read-back), then per frame ``plyio.intensity_to_rgb`` in numpy and
         ``plyio.write_ply_fast``;
(device) ``plyio.intensity_rgb`` + ``plyio.write_ply_frames``: colours and text made on the device, finished bytes copied.
Every file of both paths must be byte-identical. Stages of the device path: colours and formatting (CUDA events), the
device-to-host copies, and the file writes (time the main thread waits for the writer threads after its own work). The
ceiling: the same bytes written from memory to the same filesystem, one file after the other and with as many threads as
the writer pool. The filesystem type, the card's name and its power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import contextlib
import io
import json
import os
import shutil
import sys
import tempfile
import time
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
sys.path.insert(0, str(Path(__file__).resolve().parent))

from radar_point_cloud_tracking_b200 import fusion, plyio  # noqa: E402
from radar_point_cloud_tracking_b200 import synthetic as syn  # noqa: E402
from run_csv_recording import card  # noqa: E402
from run_fuse_frames import RES, device_block  # noqa: E402


def fs_type(path: Path) -> str:
    """Type of the filesystem holding ``path``: the longest mount point of /proc/mounts that contains it."""
    best, kind = "", "?"
    p = str(path.resolve())
    with open("/proc/mounts") as fh:
        for line in fh:
            parts = line.split()
            mnt = parts[1]
            if (p == mnt or p.startswith(mnt.rstrip("/") + "/")) and len(mnt) >= len(best):
                best, kind = mnt, parts[2]
    return kind


def host_path(fused, paths):
    for f, (x, y, m) in enumerate(fused.frames()):
        plyio.write_ply_fast(paths[f], x, y, m, plyio.intensity_to_rgb(m))


def device_path(fused, paths, stages):
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    rgb = plyio.intensity_rgb(fused.cell_max)
    ev[1].record()
    plyio.write_ply_frames(paths, fused.cell_x, fused.cell_y, fused.cell_max, rgb, fused.cell_off, timings=stages)
    stages["colours"] = stages.get("colours", 0.0) + ev[0].elapsed_time(ev[1]) * 1e-3


def fresh(root: Path, tag: str, F: int):
    d = root / tag
    shutil.rmtree(d, ignore_errors=True)
    d.mkdir(parents=True)
    return [d / f"frame_{f:05d}.ply" for f in range(F)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=64)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--dir", type=str, default=None)
    ap.add_argument("--out", type=str, default="profiles/r07_ply_frames.jsonl")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("needs a CUDA device")
    torch.cuda.set_device(0)
    base = args.dir or ("/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else None)
    root = Path(tempfile.mkdtemp(prefix="rb_ply_frames_", dir=base))
    try:
        spec = syn.SweepSpec(seed=2026, frames=args.frames)
        batch, _ = device_block(spec)
        fused = fusion.fuse_frames_max(batch, RES)
        del batch
        F = args.frames
        quiet = contextlib.redirect_stdout
        with quiet(io.StringIO()):                                    # warm-up of both paths (modules, pinned buffers)
            host_path(fused, fresh(root, "host", F))
            device_path(fused, fresh(root, "dev", F), {})
        t_host, t_dev, stages = [], [], []
        identical = True
        for _ in range(args.repeats):
            hp, dp = fresh(root, "host", F), fresh(root, "dev", F)
            out_h, out_d = io.StringIO(), io.StringIO()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            with quiet(out_h):
                host_path(fused, hp)
            t_host.append(time.perf_counter() - t0)
            st = {}
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            with quiet(out_d):
                device_path(fused, dp, st)
            t_dev.append(time.perf_counter() - t0)
            stages.append(st)
            identical &= out_h.getvalue() == out_d.getvalue()
            identical &= all(a.read_bytes() == b.read_bytes() for a, b in zip(hp, dp))
        assert identical, "the two paths wrote different bytes"
        shutil.rmtree(root / "dev")
        blobs = [p.read_bytes() for p in sorted((root / "host").iterdir())]
        ply_bytes = sum(len(b) for b in blobs)

        # ceiling: the same bytes from memory to the same filesystem
        def write_all(paths, workers):
            def one(k):
                with open(paths[k], "wb") as fh:
                    fh.write(blobs[k])
            if workers == 1:
                for k in range(len(paths)):
                    one(k)
            else:
                with ThreadPoolExecutor(workers) as pool:
                    list(pool.map(one, range(len(paths))))
        workers = min(16, os.cpu_count() or 1)
        ceil = {}
        for w in (1, workers):
            ts = []
            for _ in range(args.repeats):
                ps = fresh(root, "plain", len(blobs))
                t0 = time.perf_counter()
                write_all(ps, w)
                ts.append(time.perf_counter() - t0)
            ceil[f"threads_{w}"] = {"seconds_median": float(np.median(ts)), "GB_per_s": ply_bytes / float(np.median(ts)) / 1e9}

        med = lambda v: float(np.median(v))
        st_med = {k: med([s[k] for s in stages]) for k in ("colours", "format", "d2h", "write")}
        out = {
            "run": "ply_frames", "resolution": RES, "threshold": 5.0, "stride": 8,
            "frames": F, "spokes": spec.spokes, "bins": spec.bins, "gains": list(spec.gains), "vertices": fused.n, "ply_bytes": ply_bytes,
            "dir": {"fs_type": fs_type(root), "on": "tmpfs" if base == "/dev/shm" else str(root)},
            "repeats": args.repeats, "bytes_identical": bool(identical),
            "host_write_ply_fast": {"seconds_median": med(t_host), "seconds_all": t_host, "frames_per_s": F / med(t_host)},
            "device_write_ply_frames": {"seconds_median": med(t_dev), "seconds_all": t_dev, "frames_per_s": F / med(t_dev),
                                        "stages_s_median": st_med, "chunk_bytes": plyio.DEFAULT_CHUNK_BYTES, "writers": workers,
                                        "stage_notes": "colours, format: CUDA events; d2h: host clock around the copies and their "
                                                       "syncs; write: main-thread wait for the writer threads"},
            "speedup_device_over_host": med(t_host) / med(t_dev),
            "ceiling_plain_write": ceil,
            "card": card(),
        }
        line = json.dumps(out)
        print(line)
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        with open(args.out, "a") as fh:
            fh.write(line + "\n")
    finally:
        shutil.rmtree(root, ignore_errors=True)


if __name__ == "__main__":
    main()
