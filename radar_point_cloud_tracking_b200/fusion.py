"""Multi-gain fusion modes of ``5_gain_fusion_ply_builder.py`` on the GPU.

``fuse_gains_absolute`` (T5:193-219) is the concatenation the tracker uses (see ``tracker.build_frame``);
``fuse_gains_max`` (T5:222-273) pools all gains on a grid and keeps the maximum intensity per cell.
``fuse_points_*`` take already-converted per-gain points so they can be fed from files or from device batches;
``fuse_gains_*`` are the reference's file-level functions (same names and arguments), and :func:`install` swaps them
- with the loader, the colour helpers and the PLY writers - into an imported ``5_gain_fusion_ply_builder`` module.
Whole recordings: :func:`fuse_frames_max` fuses every frame of a device point batch in one call, and
:func:`fuse_csv_frames_max` does ``fuse_gains_max`` for a tree of sweep CSV files, batch by batch as they are parsed."""
from __future__ import annotations

import os
import time
from dataclasses import dataclass
from pathlib import Path
from typing import Dict, List, Mapping, Optional, Sequence, Tuple

import numpy as np
import torch

from . import device as dev
from ._lib import RadarB200Error

Points = Tuple[np.ndarray, np.ndarray, np.ndarray]


def fuse_points_absolute(per_gain: Dict[int, Points]):
    """Concatenate in ascending gain order with an int32 gain label per point (T5:202-219)."""
    xs, ys, zs, gs = [], [], [], []
    for gain in sorted(per_gain):
        x, y, z = per_gain[gain]
        if len(x) == 0:
            continue
        xs.append(x), ys.append(y), zs.append(z), gs.append(np.full(len(x), gain, dtype=np.int32))
    if not xs:
        return np.array([]), np.array([]), np.array([]), np.array([])
    return np.concatenate(xs), np.concatenate(ys), np.concatenate(zs), np.concatenate(gs)


def fuse_points_max(per_gain: Dict[int, Points], grid_resolution: float = 1.0) -> Points:
    """Grid max-pooling of all gains (T5:222-273): returns ``(x, y, max_intensity)`` — cell centres
    (float64) of the occupied cells in y-major order and their float32 maximum intensity. One frame of
    :func:`fuse_frames_max`."""
    res = dev.check_resolution(grid_resolution)
    if not torch.cuda.is_available():
        raise RadarB200Error("no CUDA device: fuse_points_max is GPU only (no CPU fallback)")
    parts = [per_gain[g] for g in sorted(per_gain) if len(per_gain[g][0])]
    if not parts:
        return np.array([]), np.array([]), np.array([])
    d = torch.device("cuda", torch.cuda.current_device())
    x, y, z = (torch.from_numpy(np.concatenate([p[k] for p in parts]).astype(np.float32, copy=False)).to(d) for k in range(3))
    n = x.numel()
    batch = dev.PointBatch(x, y, z, None, torch.tensor([0, n], dtype=torch.int64, device=d), n)
    return fuse_frames_max(batch, res).frames()[0]


@dataclass
class FusedFrames:
    """Max fusion of a batch of frames, on the device: frame f's cells are ``[cell_off[f], cell_off[f+1])`` of
    ``cell_x`` / ``cell_y`` (float64 centres) and ``cell_max`` (float32), y-major within the frame. ``frame_off`` = the
    batch's point offsets (a frame without points fuses to three float64 empty arrays, as in the reference)."""
    cell_x: torch.Tensor
    cell_y: torch.Tensor
    cell_max: torch.Tensor
    cell_off: torch.Tensor
    frame_off: torch.Tensor

    @property
    def n(self) -> int:
        return int(self.cell_x.numel())

    def frames(self) -> List[Points]:
        """Per frame ``(x, y, max_intensity)`` host arrays, exactly what ``fuse_gains_max`` returns for the frame's points,
        from ONE read-back (the arrays of a call are views of the same host buffers)."""
        cx, cy, cm, co, fo = dev.to_pinned_host(self.cell_x, self.cell_y, self.cell_max, self.cell_off, self.frame_off)
        out = []
        for f in range(len(co) - 1):
            if fo[f + 1] == fo[f]:                         # no points at all (T5:245-248)
                out.append((np.array([]), np.array([]), np.array([])))
            else:
                a, b = int(co[f]), int(co[f + 1])
                out.append((cx[a:b], cy[a:b], cm[a:b]))
        return out


def fuse_frames_max(batch: dev.PointBatch, grid_resolution: float = 1.0) -> FusedFrames:
    """``fuse_gains_max`` (T5:222-273) for every frame of a device point batch (``RecordingResult.raw``, a
    ``DetectionResult``'s points, ...) in one library call (``rb_fuse_max_frames``: two syncs whatever the number of
    frames). Frame f's result is what ``fuse_gains_max`` returns for the points ``[frame_off[f], frame_off[f+1])``."""
    res = dev.check_resolution(grid_resolution)
    cx, cy, cm, co = dev.fuse_max_frames(batch, res)
    return FusedFrames(cx, cy, cm, co, batch.frame_off)


# ---- the reference's file-level surface (T5) -------------------------------------------------------------------
# T5's own configuration globals (T5:52-63); a module passed to :func:`install` keeps using ITS values, read at call time
NUM_ECHO_COLUMNS = 1024
INTENSITY_THRESHOLD = 5.0
POINT_STRIDE = 8
_CFG_NAMES = ("NUM_ECHO_COLUMNS", "INTENSITY_THRESHOLD", "POINT_STRIDE")


def _config(module=None):
    import sys
    from types import SimpleNamespace

    m = module or sys.modules[__name__]
    return SimpleNamespace(**{k: getattr(m, k) for k in _CFG_NAMES})


def load_radar_csv(path, _cfg=None):
    """``(x, y, intensity, gain)`` of one sweep file (T5:84-121 - the tracker's loader with T5's threshold / stride)."""
    from . import tracker

    return tracker.load_radar_csv(path, _cfg=_cfg or _config())


def _load_all(frame_files, cfg) -> Dict[int, Points]:
    per_gain = {}
    for gain, path in sorted(frame_files.items()):
        x, y, z, _ = load_radar_csv(path, _cfg=cfg)
        per_gain[gain] = (x, y, z)                    # labelled with the directory's gain, not the file's (T5:202,209)
    return per_gain


def fuse_gains_absolute(frame_files, _cfg=None):
    """``(x, y, intensity, gain_labels)`` of all gains of a frame, ascending gain order (T5:193-219)."""
    return fuse_points_absolute(_load_all(frame_files, _cfg or _config()))


def fuse_gains_max(frame_files, grid_resolution: float = 1.0, _cfg=None) -> Points:
    """``(x, y, max_intensity)``: all gains pooled on a grid, maximum per occupied cell (T5:222-273)."""
    return fuse_points_max(_load_all(frame_files, _cfg or _config()), grid_resolution)


class _BatchPoints:
    """Device points of one CSV batch, appended launch by launch (``csvbatch.spoke_batch``'s ``append``) at the worst-case
    size of each launch, so no launch is ever repeated. The buffers are kept from batch to batch and only grow."""

    def __init__(self, device: torch.device, threshold: float, stride: int):
        self.device, self.threshold, self.stride = device, float(threshold), int(stride)
        self.store: Optional[Tuple[torch.Tensor, ...]] = None
        self.n = 0

    def reset(self) -> None:
        self.n = 0

    def append(self, echo, cos_tab, sin_tab, range_res, sweep_gain) -> np.ndarray:
        W, S, E = echo.shape
        need = self.n + W * -(-S * E // max(self.stride, 1))
        cap = 0 if self.store is None else self.store[0].numel()
        if need > cap:
            new = max(need, 2 * cap, 1 << 16)
            store = tuple(torch.empty(new, dtype=dt, device=self.device) for dt in (torch.float32,) * 3 + (torch.int32,))
            if self.n:
                for s, o in zip(store, self.store):
                    s[:self.n].copy_(o[:self.n])
            self.store = store
        out = (*(t[self.n:need] for t in self.store), torch.empty(W + 1, dtype=torch.int64, device=self.device))
        dev.spoke_to_points_raw(echo, cos_tab, sin_tab, range_res, sweep_gain, self.threshold, self.stride, need - self.n, out=out)
        (sweep_base,) = dev.to_pinned_host(out[4])
        self.n += int(sweep_base[-1])
        return sweep_base

    def batch(self, frame_off: np.ndarray) -> dev.PointBatch:
        if self.store is None:                              # no sweep so far: every frame of the batch is empty
            self.store = tuple(torch.empty(1, dtype=dt, device=self.device) for dt in (torch.float32,) * 3 + (torch.int32,))
        x, y, z, g = self.store
        return dev.PointBatch(x, y, z, g, torch.from_numpy(np.ascontiguousarray(frame_off, np.int64)).to(self.device), self.n)


def fuse_csv_frames_max(frame_files: Sequence[Mapping[int, "os.PathLike"]], grid_resolution: float = 1.0, batch_bytes: int = 64 << 20,
                        readers: Optional[int] = None, _cfg=None, timings: Optional[Dict[str, float]] = None,
                        ply_paths: Optional[Sequence["os.PathLike"]] = None) -> List[Points]:
    """``fuse_gains_max(frame_files[f], grid_resolution)`` for every frame of a recording: one ``(x, y, max_intensity)`` per
    frame, equal to the reference's with the configuration globals ``NUM_ECHO_COLUMNS``, ``INTENSITY_THRESHOLD`` and
    ``POINT_STRIDE`` (``_cfg`` = :func:`_config` of a T5 module; default this module's). File handling is that of
    ``RecordingDetection.add_csv_frames``: files are read by ``readers`` threads into pinned slots and parsed a batch of
    whole frames (at most ``batch_bytes``) per ``rb_csv_parse_sweeps`` launch; unreadable files print the reference's
    message and add no points, as do empty and header-only ones; files outside the device grammar or larger than a batch
    take the per-file readers. Each batch is fused as it arrives (spoke stage, then :func:`fuse_frames_max`), so device
    memory follows one batch, not the recording. ``timings`` (optional) accumulates the seconds of each stage.
    ``ply_paths`` (optional, one path per frame): each batch's fused frames are also written from the device as the batch
    arrives, file f with the bytes of ``write_ply_fast(ply_paths[f], x, y, max_intensity, intensity_to_rgb(max_intensity))``
    and its ``Wrote`` line (``plyio.intensity_rgb`` and ``plyio.write_ply_frames``, stage "ply")."""
    from . import csvbatch

    res = dev.check_resolution(grid_resolution)
    cfg = _cfg or _config()
    E = int(cfg.NUM_ECHO_COLUMNS)
    if E < 1:
        raise RadarB200Error("NUM_ECHO_COLUMNS must be >= 1")
    if not (csvbatch.CSV_CHUNK <= int(batch_bytes) <= csvbatch.MAX_BATCH_BYTES):
        raise RadarB200Error(f"batch_bytes must be in [{csvbatch.CSV_CHUNK}, {csvbatch.MAX_BATCH_BYTES}]")
    frames = [sorted((g, Path(p)) for g, p in ff.items()) for ff in frame_files]
    if ply_paths is not None:
        ply_paths = [Path(p) for p in ply_paths]
        if len(ply_paths) != len(frames):
            raise RadarB200Error(f"{len(ply_paths)} PLY paths for {len(frames)} frames")
    if not frames:
        return []
    if not torch.cuda.is_available():
        raise RadarB200Error("no CUDA device: fuse_csv_frames_max is GPU only (no CPU fallback)")
    from .tracker import ANGLE_SCALE

    d = torch.device("cuda", torch.cuda.current_device())
    timings = {} if timings is None else timings
    for k in ("read", "h2d", "parse", "lead", "spoke", "fuse") + (("ply",) if ply_paths is not None else ()):
        timings.setdefault(k, 0.0)
    pts = _BatchPoints(d, cfg.INTENSITY_THRESHOLD, cfg.POINT_STRIDE)
    out: List[Points] = []

    def consume(fa, fb, results):
        pts.reset()
        off = csvbatch.spoke_batch(results, E, ANGLE_SCALE, d, pts.append, timings)
        t0 = time.perf_counter()
        fused = fuse_frames_max(pts.batch(off), res)
        out.extend(fused.frames())
        timings["fuse"] += time.perf_counter() - t0
        if ply_paths is not None:
            from . import plyio

            t0 = time.perf_counter()
            plyio.write_ply_frames(ply_paths[fa:fb], fused.cell_x, fused.cell_y, fused.cell_max, plyio.intensity_rgb(fused.cell_max),
                                   fused.cell_off)
            timings["ply"] += time.perf_counter() - t0

    csvbatch.SweepReader().run(frames, E, d, readers or min(8, os.cpu_count() or 1), consume, timings, batch_bytes)
    return out


def install(ref_module) -> None:
    """Replace the hot and the output functions of an imported ``5_gain_fusion_ply_builder`` module: the loader and
    both fusion modes (GPU), the colour helpers and the PLY writers (byte-identical, native formatter). File
    discovery, grouping, plots and the CLI stay the module's own; its configuration globals are read at call time."""
    from . import plyio

    cfg = lambda: _config(ref_module)
    ref_module.load_radar_csv = lambda path: load_radar_csv(path, _cfg=cfg())
    ref_module.fuse_gains_absolute = lambda frame_files: fuse_gains_absolute(frame_files, _cfg=cfg())
    ref_module.fuse_gains_max = lambda frame_files, grid_resolution=1.0: fuse_gains_max(frame_files, grid_resolution, _cfg=cfg())
    for name in ("normalize_intensity", "intensity_to_rgb", "gain_to_rgb", "write_ply", "write_ply_fast"):
        setattr(ref_module, name, getattr(plyio, name))
