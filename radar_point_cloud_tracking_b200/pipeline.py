"""Batch detection pipeline on one GPU: the whole hot path for a block of frames, device resident.

    echo[F,G,S,E] -> spoke-to-point (+ gain concat) -> land persistence filter -> ST-DBSCAN labels

This is the throughput path (what ``bench.py`` times). It computes exactly what the reference's
``run_pipeline`` computes between "CSV parsed" and "labels known" (T4:941-977), frame for frame, and
hands back the same per-point arrays the reference keeps in its ``RadarFrame`` objects, so the
per-frame ``Cluster`` records, the Hungarian tracker and the CSV writers can consume them unchanged
(:meth:`DetectionResult.to_frames` / :meth:`DetectionResult.clusters_by_frame`).
"""
from __future__ import annotations

from collections import defaultdict
from dataclasses import dataclass
from datetime import datetime
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import device as dev
from . import tracker as trk
from ._lib import RadarB200Error, context


@dataclass
class DetectionConfig:
    """Parameters of the path; defaults are the reference's (T4:70-82)."""
    gains: Tuple[int, ...] = (40, 50, 75)
    intensity_threshold: float = trk.INTENSITY_THRESHOLD
    point_stride: int = trk.POINT_STRIDE
    land_filter: bool = True
    land_min_frames: int = 10                    # run_pipeline filters only when len(frames) > 10 (T4:954)
    land_resolution: float = trk.LAND_GRID_RESOLUTION
    land_persistence: float = trk.LAND_PERSISTENCE_THRESHOLD
    land_min_intensity: float = trk.LAND_MIN_INTENSITY
    eps_space: float = trk.EPS_SPACE
    eps_time: float = trk.EPS_TIME
    min_samples: int = trk.MIN_SAMPLES
    angle_scale: float = trk.ANGLE_SCALE
    cluster_3d: bool = False                     # cluster on (x, y, z = intensity) like 3_stdbscan_point_clouds.py (T3:177)
    #: None: the T4 clustering. k >= 1: the PointCloudWorkF variant (stdbscan_denoising_pipeline.py:264-369, rb_stdbscan_wf):
    #: a core point's neighbours must also cover at least k distinct frames, and its order-dependent border rule
    min_frames: Optional[int] = None

    def __post_init__(self):
        self.validate()

    def validate(self) -> None:
        """Raises :class:`RadarB200Error` when ``min_frames`` is set but not an int >= 1, or ``eps_time`` exceeds 30 with it
        (the variant keeps a neighbourhood's frames in a 64-bit mask)."""
        mf = self.min_frames
        if mf is None:
            return
        if isinstance(mf, bool) or not isinstance(mf, (int, np.integer)) or mf < 1:
            raise RadarB200Error(f"min_frames must be None or an int >= 1, not {mf!r}")
        if not float(np.float32(self.eps_time)) <= 30.0:
            raise RadarB200Error("min_frames needs eps_time <= 30")


@dataclass
class DetectionResult:
    """Device-resident result of one block of frames."""
    frame_ids: np.ndarray                 # [F] ids of the block's frames (host)
    raw: dev.PointBatch                   # points after spoke-to-point (before the land filter)
    points: dev.PointBatch                # points that went into ST-DBSCAN
    labels: torch.Tensor                  # int32 [points.n]
    n_clusters: int
    land: Optional[torch.Tensor] = None   # uint8 [nx, ny]
    edges: Optional[Tuple[np.ndarray, np.ndarray]] = None
    count: Optional[torch.Tensor] = None
    isum: Optional[torch.Tensor] = None

    def tensors(self):
        """Every device tensor the result holds (for stream bookkeeping)."""
        for b in (self.raw, self.points):
            yield from (b.x, b.y, b.inten, b.gain, b.frame_off)
        yield self.labels
        yield from (t for t in (self.land, self.count, self.isum) if t is not None)

    def to_host(self) -> dict:
        """One device->host read of everything the consumers need."""
        n = self.points.n
        p = self.points
        packed = torch.stack([p.x[:n], p.y[:n], p.inten[:n]], dim=1)
        points, gains, frame_off, labels = dev.to_pinned_host(packed, p.gain[:n], p.frame_off, self.labels[:n])
        return dict(points=points, gains=gains, frame_off=frame_off, labels=labels, frame_ids=self.frame_ids)

    def to_frames(self, host: Optional[dict] = None, frame_cls=None) -> list:
        """``RadarFrame`` objects as the reference's ``build_frame`` + land filter would hold them.
        Frames with no points are dropped, like ``build_frame`` returning ``None`` (T4:335-336,943)."""
        h = host or self.to_host()
        cls = frame_cls or trk.RadarFrame
        off = h["frame_off"]
        raw_off = self.raw.frame_off.cpu().numpy()
        out = []
        for i, fid in enumerate(h["frame_ids"]):
            if raw_off[i + 1] == raw_off[i]:
                continue
            out.append(cls(timestamp=datetime.fromtimestamp(0), timestamp_ms=0, frame_id=int(fid),
                           points=h["points"][off[i]:off[i + 1]], gains=h["gains"][off[i]:off[i + 1]]))
        return out

    def clusters_by_frame(self, host: Optional[dict] = None, cluster_cls=None) -> Dict[int, list]:
        """``{frame_id: [Cluster]}`` exactly as T4:511-534 builds it. The records (member points grouped per cluster,
        ``np.mean`` centroids bit for bit) come from the device (``rb_cluster_records``) in one packed read-back; the host
        wraps them into ``Cluster`` objects in the reference's order."""
        rec = dev.cluster_records(self.points, self.labels, self.n_clusters)
        return dev.clusters_from_records(rec, self.frame_ids, cluster_cls or trk.Cluster)

    def clusters_by_frame_host(self, host: Optional[dict] = None, cluster_cls=None) -> Dict[int, list]:
        """The same through the reference's own host loop (boolean masks + ``np.mean`` per cluster): the cross-check of the
        device records and the "before" of their timing (DESIGN.md)."""
        h = host or self.to_host()
        cls = cluster_cls or trk.Cluster
        off, labels, pts = h["frame_off"], h["labels"], h["points"]
        out: Dict[int, list] = defaultdict(list)
        for i, fid in enumerate(h["frame_ids"]):
            lab = labels[off[i]:off[i + 1]]
            xy = pts[off[i]:off[i + 1], :2]
            inten = pts[off[i]:off[i + 1], 2]
            ids = set(lab)
            ids.discard(-1)
            for c in ids:
                m = lab == c
                sel = xy[m]
                out[int(fid)].append(cls(cluster_id=int(c), frame_id=int(fid), points=sel, intensities=inten[m],
                                         centroid=np.mean(sel, axis=0)))
        return dict(out)


class DetectionPipeline:
    """Runs the hot path for blocks of frames on the current CUDA device."""

    def __init__(self, config: Optional[DetectionConfig] = None, device: Optional[int] = None):
        if not torch.cuda.is_available():
            raise RadarB200Error("no CUDA device: the radar-b200 detection path is GPU only (no CPU fallback)")
        self.cfg = config or DetectionConfig()
        self.cfg.validate()
        self.device = torch.device("cuda", torch.cuda.current_device() if device is None else device)
        self.ctx = context(self.device.index)
        self._cap_hint = 0
        self._grid_hint = (256, 32768)                 # land grid capacity: edges per axis, cells
        self._gain_cache = None

    # ---- host-side tables ---------------------------------------------------------------------
    def spoke_tables(self, angle_units: np.ndarray, scale: np.ndarray, n_frames: int, n_bins: int):
        """cos/sin/range-resolution tables ``[F*G, S]`` (numpy, the reference's own expressions).
        ``angle_units`` / ``scale`` may be ``[S]`` (shared by all sweeps) or ``[F, G, S]``."""
        G = len(self.cfg.gains)
        a = np.asarray(angle_units)
        sc = np.asarray(scale)
        c, s, r = trk.sweep_tables(a, sc, n_bins, self.cfg.angle_scale)
        if a.ndim == 1:
            W = n_frames * G
            c, s, r = (np.broadcast_to(t, (W, t.shape[0])) for t in (c, s, r))
        else:
            c, s, r = (t.reshape(n_frames * G, -1) for t in (c, s, r))
        return (np.ascontiguousarray(c, dtype=np.float32), np.ascontiguousarray(s, dtype=np.float32),
                np.ascontiguousarray(r, dtype=np.float32))

    # ---- device path ----------------------------------------------------------------------------
    def run_device(self, echo: torch.Tensor, cos_tab: torch.Tensor, sin_tab: torch.Tensor, range_res: torch.Tensor,
                   frame_ids: Optional[Sequence[int]] = None, cluster: bool = True) -> DetectionResult:
        """``echo[F,G,S,E]`` float32 (or uint8: the radar's native 0..255 echoes, identical results, a quarter of
        the bytes) already on the device; tables ``[F*G,S]`` on the device.
        One library call (``rb_detect_block``): every launch and the small read-backs in between happen in the
        native driver, not in Python. With ``config.min_frames`` set the block is detected without clustering and the
        filtered points are then labelled by ``rb_stdbscan_wf`` (times = frame ids)."""
        from . import _lib

        cfg = self.cfg
        F, G, S, E = echo.shape
        if G != len(cfg.gains):
            raise RadarB200Error("echo gain dimension does not match config.gains")
        d = echo.device
        ids = np.arange(F, dtype=np.int64) if frame_ids is None else np.asarray(frame_ids, dtype=np.int64)
        if self._gain_cache is None or self._gain_cache.numel() != F * G or self._gain_cache.device != d:
            self._gain_cache = torch.tensor(list(cfg.gains) * F, dtype=torch.int32, device=d)
        prm = _lib.DetectParams(n_frames=F, gains_per_frame=G, n_spokes=S, n_bins=E,
                                intensity_threshold=float(cfg.intensity_threshold), point_stride=int(cfg.point_stride),
                                land_filter=int(bool(cfg.land_filter)), land_min_frames=int(cfg.land_min_frames),
                                land_resolution=float(cfg.land_resolution), land_persistence=float(cfg.land_persistence),
                                land_min_intensity=float(cfg.land_min_intensity), eps_space=float(cfg.eps_space),
                                eps_time=float(np.float32(cfg.eps_time)), min_samples=int(cfg.min_samples),
                                cluster=int(bool(cluster) and cfg.min_frames is None),
                                cluster_3d=int(bool(cfg.cluster_3d)))
        cap = self._cap_hint or dev.default_capacity(F * G, S, E, cfg.point_stride)
        echo3 = echo.view(F * G, S, E)
        for _ in range(4):
            max_edges, max_cells = self._grid_hint
            rc, res, t = dev.detect_block(echo3, cos_tab, sin_tab, range_res, self._gain_cache, ids, prm, cap, max_edges, max_cells)
            if rc == 0:
                break
            if res.n_raw > cap:                                    # too many points for the capacity guess
                cap = int(res.n_raw * 1.1) + 1024
            else:                                                  # the land grid is larger than the guess
                ne = max(res.n_x_edges, res.n_y_edges) + 8
                self._grid_hint = (max(ne, max_edges), max(int(res.n_x_edges) * int(res.n_y_edges) + 64, max_cells))
        else:
            raise RadarB200Error("rb_detect_block: capacity negotiation did not converge")
        self._cap_hint = max(self._cap_hint, int(res.n_raw * 1.25) + 1024)
        n_raw, n_pts = int(res.n_raw), int(res.n_points)
        raw = dev.PointBatch(t["x"], t["y"], t["inten"], t["gain"], t["frame_off"], n_raw)
        pts = raw if res.filtered_is_raw else dev.PointBatch(t["fx"], t["fy"], t["finten"], t["fgain"], t["f_frame_off"], n_pts)
        land = edges = count = isum = None
        if res.land_applied:
            nx, ny = res.n_x_edges - 1, res.n_y_edges - 1
            edges = (t["x_edges"][:res.n_x_edges].copy(), t["y_edges"][:res.n_y_edges].copy())
            count, isum, land = (t[k][:nx * ny].view(nx, ny) for k in ("count", "isum", "land"))
        labels = t["labels"][:n_pts] if (cluster and n_pts > 0) else torch.empty(0, dtype=torch.int32, device=d)
        n_clusters = int(res.n_clusters)
        if cluster and n_pts > 0 and cfg.min_frames is not None:
            labels, n_clusters = self._cluster_wf(pts, ids)
        return DetectionResult(ids, raw, pts, labels, n_clusters, land, edges, count, isum)

    def _cluster_wf(self, pts: dev.PointBatch, ids: np.ndarray):
        """``rb_stdbscan_wf`` (``config.min_frames``) on a block's filtered points, times = their frame ids."""
        cfg = self.cfg
        times = dev.expand_frame_times(pts.frame_off, torch.from_numpy(ids.astype(np.float32)).to(pts.x.device), pts.n)
        return dev.stdbscan(pts.x, pts.y, pts.inten if cfg.cluster_3d else None, times, cfg.eps_space, cfg.eps_time,
                            cfg.min_samples, stride=1, n=pts.n, min_frames=cfg.min_frames)

    def run_device_staged(self, echo: torch.Tensor, cos_tab: torch.Tensor, sin_tab: torch.Tensor, range_res: torch.Tensor,
                          frame_ids: Optional[Sequence[int]] = None, cluster: bool = True) -> DetectionResult:
        """The same path driven stage by stage from Python through the per-function entry points (the calls the
        drop-in shims of :mod:`tracker` make). Kept for cross-checking the native driver."""
        cfg = self.cfg
        F, G, S, E = echo.shape
        if G != len(cfg.gains):
            raise RadarB200Error("echo gain dimension does not match config.gains")
        d = echo.device
        ids = np.arange(F, dtype=np.int64) if frame_ids is None else np.asarray(frame_ids, dtype=np.int64)
        sweep_gain = torch.tensor(list(cfg.gains) * F, dtype=torch.int32, device=d)
        cap = self._cap_hint or dev.default_capacity(F * G, S, E, cfg.point_stride)
        raw = dev.spoke_to_points(echo.view(F * G, S, E), cos_tab, sin_tab, range_res, sweep_gain,
                                  cfg.intensity_threshold, cfg.point_stride, gains_per_frame=G, cap=cap)
        self._cap_hint = max(self._cap_hint, int(raw.n * 1.25) + 1024)
        pts = raw
        land = edges = count = isum = None
        if cfg.land_filter and raw.n > 0:
            raw_off = raw.frame_off.cpu().numpy()
            built = int(np.count_nonzero(np.diff(raw_off)))           # frames build_frame would return
            if built > cfg.land_min_frames:
                b4 = dev.bounds(raw.x[:raw.n], raw.y[:raw.n]).cpu().numpy()
                xe, ye = trk.grid_edges_from_bounds(b4, cfg.land_resolution)
                d_xe, d_ye = torch.from_numpy(xe).to(d), torch.from_numpy(ye).to(d)
                count, isum = dev.land_accumulate(raw.x[:raw.n], raw.y[:raw.n], raw.inten[:raw.n], d_xe, d_ye)
                land = dev.land_cells(count, isum, built, cfg.land_persistence, cfg.land_min_intensity)
                pts = dev.land_filter(raw, d_xe, d_ye, land)
                edges = (xe, ye)
        labels = torch.empty(0, dtype=torch.int32, device=d)
        n_clusters = 0
        if cluster and pts.n > 0:
            times = dev.expand_frame_times(pts.frame_off, torch.from_numpy(ids.astype(np.float32)).to(d), pts.n)
            labels, n_clusters = dev.stdbscan(pts.x, pts.y, pts.inten if cfg.cluster_3d else None, times, cfg.eps_space,
                                              cfg.eps_time, cfg.min_samples, stride=1, n=pts.n, min_frames=cfg.min_frames)
        return DetectionResult(ids, raw, pts, labels, n_clusters, land, edges, count, isum)

    # ---- host entry (the call a user of the reference makes with parsed sweeps) -----------------
    def run_host(self, echo: np.ndarray, angle_units: np.ndarray, scale: np.ndarray,
                 frame_ids: Optional[Sequence[int]] = None, pinned: Optional[torch.Tensor] = None) -> dict:
        """Host buffers in, host buffers out: uploads ``echo[F,G,S,E]`` (numpy or pinned torch tensor),
        computes the spoke tables with numpy, runs the device path and reads the result back."""
        if pinned is not None:
            t_echo = pinned
        else:
            a = np.asarray(echo)
            t_echo = torch.from_numpy(np.ascontiguousarray(a, dtype=np.uint8 if a.dtype == np.uint8 else np.float32))
        F, G, S, E = t_echo.shape
        c, s, r = self.spoke_tables(angle_units, scale, F, E)
        d = self.device
        d_echo = t_echo.to(d, non_blocking=True)
        res = self.run_device(d_echo, torch.from_numpy(c).to(d), torch.from_numpy(s).to(d),
                              torch.from_numpy(r).to(d), frame_ids)
        out = res.to_host()
        out["n_clusters"] = res.n_clusters
        out["h2d_bytes"] = t_echo.numel() * t_echo.element_size() + 3 * c.nbytes
        out["d2h_bytes"] = out["points"].nbytes + out["gains"].nbytes + out["labels"].nbytes + out["frame_off"].nbytes
        return out


class OverlappedPipeline:
    """Throughput driver: ``workers`` host threads, each with its own CUDA stream and its own library context
    (scratch), run whole blocks concurrently, so the host-side gaps of one block (its read-backs, launch
    latency of the many small ST-DBSCAN kernels) are filled by another block's kernels - the HBM-bound mask
    kernel of block k+1 runs next to the latency-bound clustering of block k. Results are exactly those of
    :meth:`DetectionPipeline.run_device` per block."""

    def __init__(self, config: Optional[DetectionConfig] = None, device: Optional[int] = None, workers: int = 2):
        from concurrent.futures import ThreadPoolExecutor

        self.base = DetectionPipeline(config, device)
        self.device = self.base.device
        self.workers = max(1, int(workers))
        self._pool = ThreadPoolExecutor(max_workers=self.workers, thread_name_prefix="radarb200")
        import threading
        self._tls = threading.local()
        self._ctxs = []

    def _worker_state(self):
        st = getattr(self._tls, "state", None)
        if st is None:
            torch.cuda.set_device(self.device)
            st = self._tls.state = (DetectionPipeline(self.base.cfg, self.device.index), torch.cuda.Stream(self.device))
            self._ctxs.append(st[0].ctx)
        return st

    def _run(self, start_event, consumer, args, kwargs):
        pipe, stream = self._worker_state()
        with torch.cuda.stream(stream):
            stream.wait_event(start_event)                  # inputs still being written on the caller's stream
            res = pipe.run_device(*args, **kwargs)          # ends with the block's final read-back (stream sync)
            done = torch.cuda.Event()
            done.record(stream)
        # the outputs were allocated in the worker stream's pool but are consumed (and freed) on the caller's stream:
        # tell the caching allocator, or a later block could get their memory while the consumer still reads it
        for t in res.tensors():
            t.record_stream(consumer)
        return res, done, pipe.ctx.launch_count()

    def map(self, blocks, start_event=None, keep: bool = True) -> List[DetectionResult]:
        """``blocks``: iterable of ``(args, kwargs)`` for :meth:`DetectionPipeline.run_device`. Every block starts after
        ``start_event`` (default: everything queued on the current stream at the time of the call). Returns the results
        in order (``keep=False``: only the last one - earlier results are released as soon as they are complete,
        so their buffers are recycled by the following blocks instead of growing the pool); the current stream
        waits for all of them."""
        cur = torch.cuda.current_stream(self.device)
        if start_event is None:                             # order every block after what the caller has queued so far
            start_event = torch.cuda.Event()
            start_event.record(cur)
        futs = [self._pool.submit(self._run, start_event, cur, a, k) for a, k in blocks]
        out = []
        for i in range(len(futs)):
            res, done, _ = futs[i].result()
            futs[i] = None
            cur.wait_event(done)
            if keep or i == len(futs) - 1:
                out.append(res)
            del res
        return out

    def _run_host(self, args, kwargs):
        pipe, stream = self._worker_state()
        with torch.cuda.stream(stream):
            return pipe.run_host(*args, **kwargs)           # upload, device path and read-back, all on this worker's stream

    def map_host(self, blocks) -> List[dict]:
        """End-to-end blocks ``(args, kwargs)`` of :meth:`DetectionPipeline.run_host` on the worker streams: the
        host-to-device copy of one block runs under the kernels and the read-back of another (copy engines and SMs work
        side by side). Host dictionaries in order."""
        futs = [self._pool.submit(self._run_host, a, k) for a, k in blocks]
        return [f.result() for f in futs]

    def launch_count(self) -> int:
        """Kernels launched so far by all worker contexts (each worker registers its ctx on first use)."""
        return sum(c.launch_count() for c in self._ctxs)

    def close(self):
        self._pool.shutdown(wait=True)
