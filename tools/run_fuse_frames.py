"""Max fusion (T5's fuse_gains_max) of whole recordings: one JSON line per run.

    python tools/run_fuse_frames.py [--frames 64] [--subset 16] [--block 1024] [--repeats 20] [--out profiles/r06_fuse_frames.jsonl]

In one run, with T5's settings (threshold 5, stride 8, resolution 1.0):
(a) a synthetic 2048x1024x3-gain tree of --frames frames is written to tmpfs (when there is one) and read once, so every
    timed read comes from the page cache. The per-frame drop-in ``fusion.fuse_gains_max`` runs on the first --subset
    frames, ``fusion.fuse_csv_frames_max`` on all of them (with its stage timings); both must agree on the subset;
(b) ``fusion.fuse_frames_max`` alone on the points of a device-resident --block-frame block (spoke stage on device-made
    echoes), timed with CUDA events over --repeats calls after a warm-up: time per call and per frame, and the bytes the
    kernels move per point (points read twice, grids written once and read twice, cells written);
(c) ``plyio.write_ply_fast`` of every fused frame of (a) (x, y, max intensity, intensity_to_rgb colours) into a
    temporary directory: the next stage of a T5 run.
The card's name and power limit are read in the same run.
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
from concurrent.futures import ProcessPoolExecutor
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
sys.path.insert(0, str(Path(__file__).resolve().parent))

from radar_point_cloud_tracking_b200 import device as dev  # noqa: E402
from radar_point_cloud_tracking_b200 import fusion, plyio  # noqa: E402
from radar_point_cloud_tracking_b200 import synthetic as syn  # noqa: E402
from radar_point_cloud_tracking_b200.tracker import sweep_tables  # noqa: E402
from run_csv_recording import _write_frame, card  # noqa: E402

RES = 1.0


def same(a, b):
    return all(x.dtype == y.dtype and np.array_equal(x, y) for x, y in zip(a, b))


def device_block(spec, chunk=64):
    """Points of every frame of ``spec`` through the spoke stage, concatenated on the device."""
    d = torch.device("cuda", 0)
    G, S, E = len(spec.gains), spec.spokes, spec.bins
    xs, ys, zs, offs = [], [], [], [np.zeros(1, np.int64)]
    for f0 in range(0, spec.frames, chunk):
        F = min(chunk, spec.frames - f0)
        echo = dev.synth_echo(spec, first_frame=f0, n_frames=F, device=d).reshape(F * G, S, E)
        c, s, r = sweep_tables(np.tile(spec.angle_units(), (F * G, 1)), np.tile(spec.scale(), (F * G, 1)), E)
        gains = torch.tensor(list(spec.gains) * F, dtype=torch.int32, device=d)
        b = dev.spoke_to_points(echo, *(torch.from_numpy(np.ascontiguousarray(t)).to(d) for t in (c, s, r)), gains, 5.0, 8,
                                gains_per_frame=G)
        del echo
        xs.append(b.x[:b.n].clone()), ys.append(b.y[:b.n].clone()), zs.append(b.inten[:b.n].clone())
        offs.append(b.frame_off.cpu().numpy()[1:] + offs[-1][-1])
    off = np.concatenate(offs)
    x, y, z = torch.cat(xs), torch.cat(ys), torch.cat(zs)
    return dev.PointBatch(x, y, z, None, torch.from_numpy(off).to(d), int(off[-1])), off


def grid_cells(batch, off, res):
    """Grid cells of every frame as numpy computes them (T5:251-256)."""
    x, y = batch.x[:batch.n].cpu().numpy(), batch.y[:batch.n].cpu().numpy()
    total = 0
    for a, b in zip(off[:-1], off[1:]):
        if b > a:
            nx = int(np.ceil((x[a:b].max() - x[a:b].min()) / res)) + 1
            ny = int(np.ceil((y[a:b].max() - y[a:b].min()) / res)) + 1
            total += nx * ny
    return total


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=64)
    ap.add_argument("--subset", type=int, default=16)
    ap.add_argument("--block", type=int, default=1024)
    ap.add_argument("--repeats", type=int, default=20)
    ap.add_argument("--out", type=str, default="profiles/r06_fuse_frames.jsonl")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("needs a CUDA device")
    torch.cuda.set_device(0)
    spec = syn.SweepSpec(seed=2026, frames=args.frames)
    base = "/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else None
    tmp = tempfile.mkdtemp(prefix="rb_fuse_tree_", dir=base)
    root = Path(tmp)
    try:
        with ProcessPoolExecutor(max_workers=min(32, os.cpu_count() or 1)) as pool:
            frames = [{g: Path(p) for g, p in fr.items()} for fr in pool.map(_write_frame, [(spec, str(root / "tree"), f) for f in range(spec.frames)])]
        files = [p for fr in frames for p in fr.values()]
        text_bytes = sum(p.stat().st_size for p in files)
        for p in files:
            p.read_bytes()
        fusion.fuse_gains_max(frames[0], RES)                      # warm-up of both paths
        fusion.fuse_csv_frames_max(frames[:1], RES)

        # (a) the per-frame drop-in on the subset, fuse_csv_frames_max on the whole tree
        sub = frames[:args.subset]
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        drop = [fusion.fuse_gains_max(ff, RES) for ff in sub]
        t_a = time.perf_counter() - t0
        timings = {}
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fused = fusion.fuse_csv_frames_max(frames, RES, timings=timings)
        t_b = time.perf_counter() - t0
        equal = all(same(a, b) for a, b in zip(drop, fused[:len(sub)]))
        cells_out = sum(len(f[0]) for f in fused)

        # (c) PLY output of every fused frame
        ply_dir = root / "ply"
        ply_dir.mkdir()
        t0 = time.perf_counter()
        with contextlib.redirect_stdout(io.StringIO()):
            for f, (x, y, m) in enumerate(fused):
                plyio.write_ply_fast(ply_dir / f"frame_{f:05d}.ply", x, y, m, plyio.intensity_to_rgb(m))
        t_ply = time.perf_counter() - t0
        ply_bytes = sum(p.stat().st_size for p in ply_dir.iterdir())

        # (b) fuse_frames_max alone on a device-resident block
        bspec = syn.SweepSpec(seed=2026, frames=args.block)
        batch, off = device_block(bspec)
        cells = grid_cells(batch, off, RES)
        r = fusion.fuse_frames_max(batch, RES)                     # warm-up (scratch, modules)
        n_out = r.n
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        ms = []
        for _ in range(args.repeats):
            ev[0].record()
            fusion.fuse_frames_max(batch, RES)
            ev[1].record()
            ev[1].synchronize()
            ms.append(ev[0].elapsed_time(ev[1]))
        med = float(np.median(ms))
        n = batch.n
        # points: x, y read by the bounds pass, x, y, intensity by the pooling pass, one 4-byte atomic each; grids: zeroed,
        # read to count, read to emit (4 bytes per cell each); output cells: 8 + 8 + 4 bytes
        moved = n * (8 + 12 + 4) + cells * 12 + n_out * 20
        out = {
            "run": "fuse_frames", "resolution": RES, "threshold": 5.0, "stride": 8,
            "tree": {"frames": spec.frames, "spokes": spec.spokes, "bins": spec.bins, "gains": list(spec.gains), "text_bytes": text_bytes,
                     "on": "tmpfs" if base else str(root), "page_cache_warmed": True},
            "a_dropin_fuse_gains_max": {"frames": len(sub), "seconds": t_a, "frames_per_s": len(sub) / t_a},
            "b_fuse_csv_frames_max": {"frames": spec.frames, "seconds": t_b, "frames_per_s": spec.frames / t_b,
                                      "stages_s": {k: timings.get(k, 0.0) for k in ("pin", "read", "h2d", "parse", "lead", "spoke", "fuse")},
                                      "cells_out": cells_out},
            "subset_equal_to_dropin": equal,
            "speedup_b_over_a_frames_per_s": (spec.frames / t_b) / (len(sub) / t_a),
            "device_block": {"frames": args.block, "points": n, "grid_cells": cells, "cells_out": n_out, "repeats": args.repeats,
                             "ms_per_call_median": med, "ms_per_call_min": float(np.min(ms)), "us_per_frame": med * 1e3 / args.block,
                             "bytes_moved_per_point": moved / max(n, 1), "GB_per_s": moved / (med * 1e-3) / 1e9,
                             "timing": "CUDA events around each call, after one warm-up call; points and grids exceed L2"},
            "ply_write_fast": {"frames": len(fused), "seconds": t_ply, "frames_per_s": len(fused) / t_ply, "bytes": ply_bytes},
            "card": card(),
        }
        line = json.dumps(out)
        print(line)
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        with open(args.out, "a") as fh:
            fh.write(line + "\n")
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    main()
