"""A recording from its sweep CSV files: the drop-in's per-file path against RecordingDetection.add_csv_frames.

    python tools/run_csv_recording.py [--frames 64] [--subset 16] [--root DIR] [--out profiles/r04_csv_recording.jsonl]

Writes (or, with --root, reuses) a synthetic 2048x1024x3-gain tree (``synthetic``'s CSV layout) on tmpfs when there is
one, and reads it once so that every timed read comes from the page cache. Times in one run:
(a) the drop-in on the first --subset frames: ``build_frame`` per frame, then land and ``st_dbscan`` as run_pipeline does;
(b) ``add_csv_frames`` + ``finish`` + ``clusters_by_frame`` on the whole tree, twice: "cold", with torch's cache of
    pinned host blocks emptied first, so the slots are page-locked inside the timed window as in the first recording of a
    process (stage "pin"); then "warm", a second recording whose slots come from that cache;
and checks that (a) and ``add_csv_frames`` on the same subset give identical clusters. Prints one JSON line and appends it
to --out.
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time
from concurrent.futures import ProcessPoolExecutor
from datetime import datetime, timedelta
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import numpy as np
import torch

from radar_point_cloud_tracking_b200 import synthetic as syn
from radar_point_cloud_tracking_b200 import tracker as trk
from radar_point_cloud_tracking_b200.pipeline import DetectionConfig
from radar_point_cloud_tracking_b200.recording import RecordingDetection

START = "20250813_142602"
PERIOD_MS = 2500


def _write_frame(args):
    """The files of frame f, as synthetic.write_csv_tree writes them."""
    spec, root, f = args
    rects = [r for r in syn.build_rects(spec) if r.frame == f]
    header = "Status,Scale,Range,Gain,Angle," + ",".join(f"Echo_{i}" for i in range(spec.bins))
    ang, scale = spec.angle_units(), spec.scale()
    t0 = datetime.strptime(START, "%Y%m%d_%H%M%S")
    out = {}
    for gi, gain in enumerate(spec.gains):
        e = syn.synth_sweep(spec, f, gi, rects).astype(np.int64)
        ts = t0 + timedelta(milliseconds=f * PERIOD_MS + gi * 100)
        d = Path(root) / f"gain_{gain}"
        d.mkdir(parents=True, exist_ok=True)
        p = d / (ts.strftime("%Y%m%d_%H%M%S") + f"_{ts.microsecond // 1000:03d}.csv")
        rows = [header] + [f"1,{scale[s]:g},3,{gain},{int(ang[s])}," + ",".join(map(str, e[s].tolist())) for s in range(spec.spokes)]
        p.write_text("\n".join(rows) + "\n")
        out[gain] = str(p)
    return out


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (q.stdout.strip().splitlines() or ["?, ?"])[0].split(", ")
    return {"name": name, "power_limit": power}


def rows(clusters):
    return sorted((int(fid), c.cluster_id, c.num_points, float(c.centroid[0]), float(c.centroid[1]), c.mean_intensity)
                  for fid, cl in clusters.items() for c in cl)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=64)
    ap.add_argument("--subset", type=int, default=16)
    ap.add_argument("--root", type=str, default=None)
    ap.add_argument("--out", type=str, default="profiles/r04_csv_recording.jsonl")
    ap.add_argument("--batch-mb", type=int, default=None, help="batch_bytes of (b) in MiB (default: add_csv_frames' own)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("needs a CUDA device")
    torch.cuda.set_device(0)
    spec = syn.SweepSpec(seed=2026, frames=args.frames)
    tmp = None
    if args.root:
        root = Path(args.root)
    else:
        base = "/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else None
        tmp = tempfile.mkdtemp(prefix="rb_csv_tree_", dir=base)
        root = Path(tmp)
    try:
        t0 = time.perf_counter()
        with ProcessPoolExecutor(max_workers=min(32, os.cpu_count() or 1)) as pool:
            frames = [{g: Path(p) for g, p in fr.items()} for fr in pool.map(_write_frame, [(spec, str(root), f) for f in range(spec.frames)])]
        t_write = time.perf_counter() - t0
        files = [p for fr in frames for p in fr.values()]
        text_bytes = sum(p.stat().st_size for p in files)
        for p in files:                                    # warm the page cache: every timed read below comes from memory
            p.read_bytes()
        cfg = DetectionConfig()
        # warm-up of both paths (contexts, kernels, pandas import) on one frame
        trk.build_frame(frames[0], 0)
        w = RecordingDetection(cfg, 0)
        w.add_csv_frames(frames[:1])
        w.finish()
        del w

        # (a) the drop-in per-file path on the subset
        sub = frames[:args.subset]
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        built = [f for f in (trk.build_frame(ff, i) for i, ff in enumerate(sub)) if f is not None]
        if len(built) > 10:
            count, isum, edges = trk.build_occupancy_grid(built, cfg.land_resolution)
            land = trk.identify_land_cells(count, isum, len(built))
            built = [trk.filter_land_from_frame(f, land, edges) for f in built]
        drop_clusters = trk.st_dbscan(built, cfg.eps_space, cfg.eps_time, cfg.min_samples)
        t_a = time.perf_counter() - t0

        # the same subset through add_csv_frames: clusters must be identical
        r = RecordingDetection(cfg, 0)
        r.add_csv_frames(sub)
        same = rows(r.finish().clusters_by_frame()) == rows(drop_clusters)
        del r

        # (b) the whole tree, twice. Cold: no pinned block left in torch's host cache, so the slots are page-locked inside
        # the window (the first recording of a process). Warm: a second recording, whose slots come from that cache.
        kw = {} if args.batch_mb is None else {"batch_bytes": args.batch_mb << 20}
        arms = {}
        for arm in ("cold", "warm"):
            if arm == "cold":
                torch._C._host_emptyCache()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            rec = RecordingDetection(cfg, 0)
            rec.add_csv_frames(frames, **kw)
            t1 = time.perf_counter()
            res = rec.finish()
            t2 = time.perf_counter()
            clusters = res.clusters_by_frame()
            t3 = time.perf_counter()
            t_b = t3 - t0
            st = res.timings
            stages = {"pin": st.get("pin", 0.0), "read_wait": st.get("read", 0.0), "h2d": st.get("h2d", 0.0), "parse": st.get("parse", 0.0),
                      "lead_fields_and_trig": st.get("lead", 0.0), "spoke": st.get("spoke", 0.0), "finish": t2 - t1, "records": t3 - t2}
            arms[arm] = {"frames": spec.frames, "seconds": t_b, "frames_per_s": spec.frames / t_b, "text_GB_per_s": text_bytes / t_b / 1e9,
                         "slots_page_locked_in_window": arm == "cold", "slot_bytes": rec._reader.slot_bytes, "files": rec.csv_files,
                         "stages_s": dict(stages, add_csv_frames=t1 - t0), "largest_stage": max(stages, key=stages.get),
                         "speedup_over_a": (spec.frames / t_b) / (len(sub) / t_a),
                         "raw_points": res.raw.n, "filtered_points": res.points.n, "clusters": res.n_clusters,
                         "cluster_records": sum(len(v) for v in clusters.values())}
            del rec, res, clusters
        out = {
            "run": "csv_recording", "frames": spec.frames, "spokes": spec.spokes, "bins": spec.bins, "gains": list(spec.gains),
            "text_bytes": text_bytes, "tree_on": "tmpfs" if str(root).startswith("/dev/shm") else str(root),
            "page_cache_warmed": True, "tree_write_s": t_write, "batch_bytes": kw.get("batch_bytes", "default (64 MiB)"),
            "a_dropin": {"frames": len(sub), "seconds": t_a, "frames_per_s": len(sub) / t_a,
                         "text_GB_per_s": sum(p.stat().st_size for fr in sub for p in fr.values()) / t_a / 1e9},
            "b_add_csv_frames_cold": arms["cold"], "b_add_csv_frames_warm": arms["warm"],
            "subset_clusters_identical": same,
            "card": card(),
        }
        line = json.dumps(out)
        print(line)
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        with open(args.out, "a") as fh:
            fh.write(line + "\n")
    finally:
        if tmp:
            shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    main()
