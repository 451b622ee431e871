"""Host-side mirror of the hot functions of ``PointCloudWork/4_temporal_object_tracker.py`` ("T4").

Same names, arguments, return types and error behaviour as the reference functions they replace,
so ``run_pipeline``, ``ObjectTracker`` and ``save_tracking_results`` of the reference consume the
output unchanged (see :func:`install`). Every numeric stage runs in the CUDA library; what stays on
the host is what the reference's own host would do anyway: CSV parsing, per-spoke trig tables
(numpy, so they are bit-identical to the reference's), ``np.arange`` grid edges and the per-frame
``Cluster`` records (``np.mean`` centroids).

    load_radar_csv            T4:184-232      build_frame              T4:312-352
    build_occupancy_grid      T4:359-391      identify_land_cells      T4:394-410
    filter_land_from_frame    T4:413-436      st_dbscan                T4:443-536
"""
from __future__ import annotations

import re
from collections import defaultdict
from dataclasses import dataclass
from datetime import datetime
from pathlib import Path
from types import SimpleNamespace
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import device as dev
from ._lib import RadarB200Error

# ---- configuration: same names and defaults as T4:55-90 ---------------------------------------
SUPPORTED_GAINS = {40, 50, 70, 75}
ANGLE_SCALE = 360.0 / 8196.0
NUM_ECHO_COLUMNS = 1024
INTENSITY_THRESHOLD = 10.0
POINT_STRIDE = 4
MAX_TIME_DIFF_MS = 2000
EPS_SPACE = 8.0
EPS_TIME = 2.0
MIN_SAMPLES = 15
LAND_PERSISTENCE_THRESHOLD = 0.8
LAND_GRID_RESOLUTION = 5.0
LAND_MIN_INTENSITY = 100


@dataclass
class RadarFrame:
    """Same fields as the reference's ``RadarFrame`` (T4:97-108)."""
    timestamp: datetime
    timestamp_ms: int
    frame_id: int
    points: np.ndarray      # (N, 3) float32: x, y, intensity
    gains: np.ndarray       # (N,) int32

    @property
    def num_points(self) -> int:
        return self.points.shape[0]


@dataclass
class Cluster:
    """Same fields as the reference's ``Cluster`` (T4:143-158)."""
    cluster_id: int
    frame_id: int
    points: np.ndarray
    intensities: np.ndarray
    centroid: np.ndarray

    @property
    def num_points(self) -> int:
        return self.points.shape[0]

    @property
    def mean_intensity(self) -> float:
        return float(np.mean(self.intensities))


def _cuda() -> torch.device:
    if not torch.cuda.is_available():
        raise RadarB200Error("no CUDA device: the radar-b200 detection path is GPU only (no CPU fallback)")
    return torch.device("cuda", torch.cuda.current_device())


# ---- host-side pieces ---------------------------------------------------------------------------
def parse_timestamp(filename: str) -> Tuple[datetime, int]:
    """``YYYYMMDD_HHMMSS_mmm.csv`` -> (datetime, epoch milliseconds) as T4:165-181."""
    m = re.match(r"(\d{8})_(\d{6})_(\d{3})\.csv", filename)
    if not m:
        raise ValueError(f"Cannot parse timestamp from {filename}")
    day, clock, ms = m.groups()
    dt = datetime.strptime(f"{day}_{clock}", "%Y%m%d_%H%M%S")
    return dt, int(dt.timestamp() * 1000) + int(ms)


def read_sweep_csv(path: Path, num_echo_columns: int = NUM_ECHO_COLUMNS):
    """Host CSV parse of one sweep (T4:189-209): returns ``(angle_units f32[S], scale f32[S],
    echo f32[S,E], gain)`` or ``None`` for an unreadable / empty file (T4:193-198)."""
    import pandas as pd

    names = ["Status", "Scale", "Range", "Gain", "Angle"] + [f"Echo_{i}" for i in range(num_echo_columns)]
    try:
        df = pd.read_csv(path, header=None, names=names, skiprows=1, engine="c")
    except Exception as e:  # same message as the reference
        print(f"Error loading {path}: {e}")
        return None
    if df.empty:
        return None
    gain = int(df["Gain"].iloc[0])
    angle = df["Angle"].to_numpy(np.float32)
    echo = df.iloc[:, 5:].fillna(0).to_numpy(np.float32)
    scale = df["Scale"].to_numpy(np.float32)
    return angle, scale, np.ascontiguousarray(echo), gain


def read_sweep_csv_device(path: Path, num_echo_columns: int = NUM_ECHO_COLUMNS):
    """:func:`read_sweep_csv` with the echo columns parsed on the GPU (``rb_csv_parse_sweep``): same return value
    except that ``echo`` is a uint8 DEVICE tensor ``[S, E]`` - it goes straight into the uint8 spoke-to-point kernel
    and never exists as float32 on the host. The five leading fields of every row (a few bytes) are parsed by pandas,
    the reference's parser, from the offsets the device returns. A file outside the device grammar (non-integer or
    > 255 echoes, ragged rows, blank lines, quotes) is handed to :func:`read_sweep_csv` whole, so it behaves exactly
    as in the reference."""
    path = Path(path)
    try:
        raw = path.read_bytes()
    except Exception as e:  # same message as the reference (T4:194)
        print(f"Error loading {path}: {e}")
        return None
    echo, row_start, prefix_end, status = dev.csv_parse_sweep(raw, num_echo_columns, _cuda())
    if status:
        return read_sweep_csv(path, num_echo_columns)
    if echo.shape[0] == 0:
        return None                                               # header only / empty: df.empty (T4:197-198)
    lead = lead_fields_pandas(raw, row_start, prefix_end, echo.shape[0])
    if lead is None:
        return read_sweep_csv(path, num_echo_columns)              # let the reference's parser decide (and report)
    angle, scale, gain = lead
    return angle, scale, echo, gain


def lead_fields_pandas(raw, row_start: np.ndarray, prefix_end: np.ndarray, n_rows: int):
    """The five leading fields of a file's rows, ``raw[row_start[r]:prefix_end[r]]``, through pandas (the reference's
    parser): ``(angle f32, scale f32, gain)``, or ``None`` when pandas fails or finds another number of rows - the file
    then goes to :func:`read_sweep_csv` whole."""
    import io

    import pandas as pd

    lead = b"\n".join(bytes(raw[a:b]) for a, b in zip(row_start.tolist(), prefix_end.tolist()))
    try:
        df = pd.read_csv(io.BytesIO(lead), header=None, names=["Status", "Scale", "Range", "Gain", "Angle"], engine="c")
        gain = int(df["Gain"].iloc[0])
        angle = df["Angle"].to_numpy(np.float32)
        scale = df["Scale"].to_numpy(np.float32)
    except Exception:
        return None
    if len(df) != n_rows:
        return None
    return angle, scale, gain


def sweep_tables(angle_units: np.ndarray, scale: np.ndarray, num_bins: int, angle_scale: float = ANGLE_SCALE
                 ) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """Per-spoke ``cos``, ``sin`` and range resolution with the reference's own numpy expressions
    (T4:203, T4:213, T4:217-218) so the trig is bit-identical to the reference on this host.
    Works on any leading shape (``[S]`` or ``[W, S]``)."""
    rad = np.deg2rad(np.asarray(angle_units).astype(np.float32) * angle_scale)
    res = np.asarray(scale).astype(np.float32) / num_bins
    return np.cos(rad), np.sin(rad), res.astype(np.float32)


def _points_from_sweeps(sweeps: Sequence[Tuple[np.ndarray, np.ndarray, np.ndarray, int]], threshold: float,
                        stride: int) -> List[Tuple[np.ndarray, np.ndarray, np.ndarray]]:
    """GPU spoke-to-point for a list of parsed sweeps ``(angle, scale, echo, gain_label)``; one
    launch when they share a shape. Returns per-sweep ``(x, y, intensity)`` numpy arrays."""
    d = _cuda()
    out: List[Tuple[np.ndarray, np.ndarray, np.ndarray]] = [None] * len(sweeps)      # type: ignore
    by_shape: Dict[Tuple[int, int], List[int]] = defaultdict(list)
    for i, (_, _, echo, _) in enumerate(sweeps):
        by_shape[tuple(echo.shape)].append(i)
    for (S, E), idxs in by_shape.items():
        if S == 0 or E == 0:
            for i in idxs:
                out[i] = (np.array([], np.float32), np.array([], np.float32), np.array([], np.float32))
            continue
        if all(isinstance(sweeps[i][2], torch.Tensor) for i in idxs):
            echo = torch.stack([sweeps[i][2] for i in idxs])                  # parsed on the device (uint8), already there
        else:
            stacked = np.stack([sweeps[i][2].cpu().numpy() if isinstance(sweeps[i][2], torch.Tensor) else sweeps[i][2] for i in idxs])
            # real echoes are 8-bit (PIPELINE_DOCUMENTATION.txt:47): when the parsed values are exactly 0..255 integers
            # they travel as uint8 - a quarter of the PCIe bytes, identical points (rb_spoke_to_points_u8)
            as_u8 = stacked.astype(np.uint8)
            echo = torch.from_numpy(as_u8 if np.array_equal(as_u8, stacked) else stacked).to(d)
        cs, sn, rs = sweep_tables(np.stack([sweeps[i][0] for i in idxs]), np.stack([sweeps[i][1] for i in idxs]), E)
        gains = torch.tensor([sweeps[i][3] for i in idxs], dtype=torch.int32, device=d)
        batch = dev.spoke_to_points(echo, torch.from_numpy(cs).to(d), torch.from_numpy(sn).to(d),
                                    torch.from_numpy(rs).to(d), gains, threshold, stride, gains_per_frame=1)
        off = batch.frame_off.cpu().numpy()
        x, y, z = batch.x[:batch.n].cpu().numpy(), batch.y[:batch.n].cpu().numpy(), batch.inten[:batch.n].cpu().numpy()
        for k, i in enumerate(idxs):
            out[i] = (x[off[k]:off[k + 1]], y[off[k]:off[k + 1]], z[off[k]:off[k + 1]])
    return out


# ---- a1 ------------------------------------------------------------------------------------------
def load_radar_csv(path: Path, _cfg=None) -> Tuple[np.ndarray, np.ndarray, np.ndarray, int]:
    """Load a radar CSV and convert to Cartesian. Returns ``(x, y, intensity, gain)`` (T4:184-232).
    Threshold and stride are the module globals, exactly as in the reference."""
    cfg = _cfg or _module_config()
    sweep = read_sweep_csv_device(Path(path), cfg.NUM_ECHO_COLUMNS)
    if sweep is None:
        return np.array([]), np.array([]), np.array([]), 0
    angle, scale, echo, gain = sweep
    (x, y, z), = _points_from_sweeps([(angle, scale, echo, gain)], cfg.INTENSITY_THRESHOLD, cfg.POINT_STRIDE)
    return x, y, z, gain


# ---- a2 ------------------------------------------------------------------------------------------
def build_frame(frame_files: Dict[int, Path], frame_id: int, _cfg=None, _frame_cls=None) -> Optional[RadarFrame]:
    """Fuse the gains of one frame by concatenation in ascending gain order (T4:312-352).
    All gains of the frame go through the spoke-to-point kernel in one launch."""
    cfg = _cfg or _module_config()
    frame_cls = _frame_cls or RadarFrame
    first_ts = first_ts_ms = None
    sweeps, labels = [], []
    for gain, path in sorted(frame_files.items()):
        path = Path(path)
        if first_ts is None:
            first_ts, first_ts_ms = parse_timestamp(path.name)
        sweep = read_sweep_csv_device(path, cfg.NUM_ECHO_COLUMNS)
        if sweep is None:
            continue
        angle, scale, echo, _ = sweep
        sweeps.append((angle, scale, echo, gain))     # label = the directory's gain (T4:333)
        labels.append(gain)
    parts = _points_from_sweeps(sweeps, cfg.INTENSITY_THRESHOLD, cfg.POINT_STRIDE) if sweeps else []
    xs, ys, zs, gs = [], [], [], []
    for gain, (x, y, z) in zip(labels, parts):
        if len(x) == 0:
            continue
        xs.append(x), ys.append(y), zs.append(z)
        gs.append(np.full(len(x), gain, dtype=np.int32))
    if not xs:
        return None
    points = np.column_stack([np.concatenate(xs), np.concatenate(ys), np.concatenate(zs)])
    return frame_cls(timestamp=first_ts, timestamp_ms=first_ts_ms, frame_id=frame_id, points=points,
                     gains=np.concatenate(gs))


# ---- a4 - a6 ---------------------------------------------------------------------------------------
def _to_device_points(frames) -> Tuple[dev.PointBatch, np.ndarray]:
    d = _cuda()
    counts = np.array([f.points.shape[0] for f in frames], dtype=np.int64)
    offs = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    n = int(offs[-1])
    if n:
        pts = np.concatenate([np.asarray(f.points, dtype=np.float32).reshape(-1, 3) for f in frames])
        gains = np.concatenate([np.asarray(f.gains, dtype=np.int32) for f in frames])
    else:
        pts, gains = np.zeros((0, 3), np.float32), np.zeros(0, np.int32)
    t = torch.from_numpy(np.ascontiguousarray(pts.T)).to(d)           # SoA on the device
    batch = dev.PointBatch(t[0].contiguous(), t[1].contiguous(), t[2].contiguous(),
                           torch.from_numpy(gains).to(d), torch.from_numpy(offs).to(d), n)
    return batch, offs


def grid_edges_from_bounds(b4: np.ndarray, resolution: float) -> Tuple[np.ndarray, np.ndarray]:
    """``np.arange(min, max + res, res)`` with float32 scalar bounds (T4:368-373) -> float64 edges."""
    x_min, x_max, y_min, y_max = (np.float32(v) for v in b4)
    return (np.arange(x_min, x_max + resolution, resolution), np.arange(y_min, y_max + resolution, resolution))


def build_occupancy_grid(frames: List[RadarFrame], resolution: float
                         ) -> Tuple[np.ndarray, np.ndarray, Tuple[np.ndarray, np.ndarray]]:
    """Occupancy grid over all frames: per-cell POINT counts (int32) and float64 intensity sums
    (T4:359-391). Returns ``(count_grid, intensity_sum_grid, (x_edges, y_edges))``."""
    batch, _ = _to_device_points(frames)
    if batch.n == 0:
        raise ValueError("zero-size array to reduction operation minimum which has no identity")   # as numpy
    b4 = dev.bounds(batch.x, batch.y).cpu().numpy()
    xe, ye = grid_edges_from_bounds(b4, resolution)
    d = batch.x.device
    count, isum = dev.land_accumulate(batch.x, batch.y, batch.inten, torch.from_numpy(xe).to(d),
                                      torch.from_numpy(ye).to(d))
    return count.cpu().numpy(), isum.cpu().numpy(), (xe, ye)


def identify_land_cells(count_grid: np.ndarray, intensity_grid: np.ndarray, num_frames: int, _cfg=None) -> np.ndarray:
    """Boolean land mask: high persistence AND high mean intensity (T4:394-410)."""
    cfg = _cfg or _module_config()
    d = _cuda()
    count = torch.from_numpy(np.ascontiguousarray(count_grid, dtype=np.int32)).to(d)
    isum = torch.from_numpy(np.ascontiguousarray(intensity_grid, dtype=np.float64)).to(d)
    land = dev.land_cells(count, isum, num_frames, cfg.LAND_PERSISTENCE_THRESHOLD, cfg.LAND_MIN_INTENSITY)
    return land.cpu().numpy().astype(bool)


def filter_land_from_frame(frame: RadarFrame, land_mask: np.ndarray, edges: Tuple[np.ndarray, np.ndarray],
                           _frame_cls=None) -> RadarFrame:
    """Remove land points from a frame, keeping order (T4:413-436)."""
    frame_cls = _frame_cls or type(frame)
    (out,) = filter_land_from_frames([frame], land_mask, edges, frame_cls)
    return out


def filter_land_from_frames(frames: Sequence[RadarFrame], land_mask: np.ndarray,
                            edges: Tuple[np.ndarray, np.ndarray], frame_cls=None) -> List[RadarFrame]:
    """All frames in one launch (same result as calling :func:`filter_land_from_frame` per frame)."""
    xe, ye = edges
    batch, _ = _to_device_points(frames)
    d = batch.x.device
    land = torch.from_numpy(np.ascontiguousarray(land_mask).astype(np.uint8)).to(d)
    if land.shape[0] != len(xe) - 1 or land.shape[1] != len(ye) - 1:
        # the reference clips to land_mask.shape - 1 (T4:424-425); same thing when shapes agree
        raise RadarB200Error("land_mask shape must match the edges")
    out = dev.land_filter(batch, torch.from_numpy(np.asarray(xe, np.float64)).to(d),
                          torch.from_numpy(np.asarray(ye, np.float64)).to(d), land)
    n = out.n
    pts = torch.stack([out.x[:n], out.y[:n], out.inten[:n]], dim=1).cpu().numpy()
    gains = out.gain[:n].cpu().numpy()
    off = out.frame_off.cpu().numpy()
    res = []
    for i, f in enumerate(frames):
        cls = frame_cls or type(f)
        res.append(cls(timestamp=f.timestamp, timestamp_ms=f.timestamp_ms, frame_id=f.frame_id,
                       points=pts[off[i]:off[i + 1]], gains=gains[off[i]:off[i + 1]]))
    return res


# ---- a7 + a8 ---------------------------------------------------------------------------------------
def st_dbscan_labels(frames: Sequence[RadarFrame], eps_space: float, eps_time: float, min_samples: int
                     ) -> Tuple[np.ndarray, np.ndarray]:
    """Flat labels of all frames' points (stacked in frame order) + per-frame offsets."""
    offs = np.concatenate([[0], np.cumsum([f.points.shape[0] for f in frames])]).astype(np.int64)
    n = int(offs[-1])
    if n == 0:
        return np.zeros(0, np.int32), offs
    d = _cuda()
    coords = np.vstack([f.points[:, :2] for f in frames]).astype(np.float32, copy=False)      # T4:466
    fid = np.concatenate([np.full(f.points.shape[0], f.frame_id) for f in frames]).astype(np.float32)   # T4:467
    xy = torch.from_numpy(np.ascontiguousarray(coords)).to(d)
    t = torch.from_numpy(fid).to(d)
    flat = xy.view(-1)
    labels, _ = dev.stdbscan(flat, flat[1:], None, t, eps_space, eps_time, min_samples, stride=2, n=n)
    return labels.cpu().numpy(), offs


def clusters_host(frames: Sequence[RadarFrame], labels: np.ndarray, offs: np.ndarray, cluster_cls=None) -> Dict[int, List[Cluster]]:
    """The reference's own loop (T4:511-534) in host numpy: boolean masks and ``np.mean`` per cluster. Kept as the
    cross-check of :func:`device.cluster_records` (the tests compare the two record for record); the product path below
    does not call it."""
    cluster_cls = cluster_cls or Cluster
    by_frame: Dict[int, List[Cluster]] = defaultdict(list)
    for i, frame in enumerate(frames):
        lab = labels[offs[i]:offs[i + 1]]
        xy = frame.points[:, :2]
        inten = frame.points[:, 2]
        ids = set(lab)
        ids.discard(-1)
        for c in ids:
            m = lab == c
            pts = xy[m]
            by_frame[frame.frame_id].append(cluster_cls(cluster_id=int(c), frame_id=frame.frame_id, points=pts,
                                                        intensities=inten[m], centroid=np.mean(pts, axis=0)))
    return dict(by_frame)


def st_dbscan(frames: List[RadarFrame], eps_space: float, eps_time: float, min_samples: int,
              _cluster_cls=None) -> Dict[int, List[Cluster]]:
    """ST-DBSCAN across all frames; returns ``{frame_id: [Cluster]}`` (T4:443-536). Labels AND the per-frame cluster
    records (T4:511-534: member points, ``np.mean`` centroid) are computed on the device; the host only wraps the
    records into ``Cluster`` objects, in the reference's order."""
    cluster_cls = _cluster_cls or Cluster
    if not frames:                                            # T4:463-464
        return {}
    batch, offs = _to_device_points(frames)
    if batch.n == 0:
        return {}
    d = batch.x.device
    ids = np.array([f.frame_id for f in frames])
    times = dev.expand_frame_times(batch.frame_off, torch.from_numpy(ids.astype(np.float32)).to(d), batch.n)      # T4:460,467
    labels, n_clusters = dev.stdbscan(batch.x, batch.y, None, times, eps_space, eps_time, min_samples, stride=1, n=batch.n)
    rec = dev.cluster_records(batch, labels, n_clusters)
    return dev.clusters_from_records(rec, [f.frame_id for f in frames], cluster_cls, frame_id_type=lambda v: v)


# ---- whole recordings from CSV files ----------------------------------------------------------------------
def detect_csv_frames(frame_files: Sequence[Dict[int, Path]], skip_land_filter: bool, eps_space: float, eps_time: float,
                      min_samples: int, _cfg=None, _cluster_cls=None) -> Dict[int, List[Cluster]]:
    """What T4:941-977 of ``run_pipeline`` computes from the grouped files - ``build_frame`` per frame (frame id = index),
    the land filter when more than 10 frames were built, one ``st_dbscan`` - as one :class:`recording.RecordingDetection`
    fed by :meth:`~recording.RecordingDetection.add_csv_frames`. Configuration globals as ``install`` reads them
    (``_cfg`` = a T4 module's :func:`_module_config`). Returns ``{frame_id: [Cluster]}``."""
    from .pipeline import DetectionConfig
    from .recording import RecordingDetection

    cfg = _cfg or _module_config()
    if not frame_files:
        return {}
    dc = DetectionConfig(intensity_threshold=cfg.INTENSITY_THRESHOLD, point_stride=cfg.POINT_STRIDE, land_filter=not skip_land_filter,
                         land_resolution=cfg.LAND_GRID_RESOLUTION, land_persistence=cfg.LAND_PERSISTENCE_THRESHOLD,
                         land_min_intensity=cfg.LAND_MIN_INTENSITY, eps_space=eps_space, eps_time=eps_time, min_samples=min_samples)
    rec = RecordingDetection(dc, _cuda().index)
    rec.add_csv_frames(frame_files, num_echo_columns=cfg.NUM_ECHO_COLUMNS)
    res = rec.finish()
    if res.points.n == 0:
        return {}
    return res.clusters_by_frame(cluster_cls=_cluster_cls or Cluster)


# ---- drop-in installation ----------------------------------------------------------------------------
_CFG_NAMES = ("NUM_ECHO_COLUMNS", "INTENSITY_THRESHOLD", "POINT_STRIDE", "LAND_PERSISTENCE_THRESHOLD",
              "LAND_GRID_RESOLUTION", "LAND_MIN_INTENSITY")


def _module_config(module=None):
    """Live view of the configuration globals of ``module`` (default: this module)."""
    import sys

    m = module or sys.modules[__name__]
    return SimpleNamespace(**{k: getattr(m, k) for k in _CFG_NAMES})


def install(ref_module) -> None:
    """Replace the hot functions of an imported reference ``4_temporal_object_tracker`` module with
    the CUDA path. The module's own ``RadarFrame`` / ``Cluster`` classes and its configuration
    globals (``INTENSITY_THRESHOLD``, ``POINT_STRIDE``, ``LAND_*`` — read at call time, so the
    ``--intensity-threshold`` flag stays the no-op it is in the reference, T4:896 vs T4:221) are
    used, and everything else (``run_pipeline``, ``ObjectTracker``, writers, plots) is untouched."""
    frame_cls, cluster_cls = ref_module.RadarFrame, ref_module.Cluster

    def _load_radar_csv(path):
        return load_radar_csv(path, _cfg=_module_config(ref_module))

    def _build_frame(frame_files, frame_id):
        return build_frame(frame_files, frame_id, _cfg=_module_config(ref_module), _frame_cls=frame_cls)

    def _identify_land_cells(count_grid, intensity_grid, num_frames):
        return identify_land_cells(count_grid, intensity_grid, num_frames, _cfg=_module_config(ref_module))

    def _filter_land_from_frame(frame, land_mask, edges):
        return filter_land_from_frame(frame, land_mask, edges, _frame_cls=frame_cls)

    def _st_dbscan(frames, eps_space, eps_time, min_samples):
        return st_dbscan(frames, eps_space, eps_time, min_samples, _cluster_cls=cluster_cls)

    ref_module.load_radar_csv = _load_radar_csv
    ref_module.build_frame = _build_frame
    ref_module.build_occupancy_grid = build_occupancy_grid
    ref_module.identify_land_cells = _identify_land_cells
    ref_module.filter_land_from_frame = _filter_land_from_frame
    ref_module.st_dbscan = _st_dbscan
