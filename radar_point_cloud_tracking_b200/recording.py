"""A whole recording on one GPU: frame blocks in, one land grid and one ST-DBSCAN labelling out.

The reference's ``run_pipeline`` treats a recording as one problem (T4:941-977): one occupancy grid over all frames,
land filtering only when more than ``land_min_frames`` frames were built, and one ``st_dbscan`` whose cluster ids are
ranks over the whole recording. :class:`RecordingDetection` computes exactly that for a recording fed block by block:

    add_block(echo block) ...  ->  spoke-to-point per block into one device point store (echo blocks are not kept)
    add_csv_frames(files) ...  ->  the same from sweep CSV files, parsed in batches on the device (csvbatch)
    finish()                   ->  land grid from the recording's bounds, land filter, rb_stdbscan_windowed

Frame for frame and bit for bit the result equals :meth:`pipeline.DetectionPipeline.run_device` on the concatenation
of all blocks as one block. Clustering runs in time windows (DESIGN.md section 3.8) when the filtered points do not fit
one ST-DBSCAN call; ``max_window_points`` forces smaller windows.
"""
from __future__ import annotations

import ctypes as C
import math
import os
import time
from dataclasses import dataclass, field
from pathlib import Path
from typing import Dict, Mapping, Optional, Sequence

import numpy as np
import torch

from . import _lib
from . import device as dev
from ._lib import RadarB200Error, check, context, ptr, stream_ptr
from .pipeline import DetectionConfig, DetectionPipeline, DetectionResult

#: one ST-DBSCAN call takes fewer than 2^31 - 1 points (rb_stdbscan)
MAX_CALL_POINTS = (1 << 31) - 2
#: device scratch per point of one window: rb_stdbscan's, measured on a B200 (321 B at config-3, 100 B at config-4 density;
#: DESIGN.md section 7), plus the windowed driver's 29 B; the default budget keeps it within 80 % of the free memory
SCRATCH_BYTES_PER_POINT = 360
_ID_LIMIT = 1 << 24


def check_frame_ids(ids: np.ndarray, after: Optional[int] = None) -> np.ndarray:
    """``ids`` as int64 if they are integers, strictly increasing, above ``after`` and of magnitude below 2^24 (so their
    float32 times stay distinct); raises :class:`RadarB200Error` otherwise."""
    a = np.asarray(ids)
    if a.ndim != 1 or a.size == 0:
        raise RadarB200Error("frame ids must be a non-empty 1-D sequence")
    f = a.astype(np.float64)
    if not np.all(np.isfinite(f)) or not np.array_equal(f, np.rint(f)):
        raise RadarB200Error("frame ids must be integers")
    if np.any(np.abs(f) >= _ID_LIMIT):
        raise RadarB200Error("frame ids must be of magnitude below 2^24")
    out = f.astype(np.int64)
    if np.any(np.diff(out) <= 0) or (after is not None and out[0] <= after):
        raise RadarB200Error("frame ids must increase strictly across the recording")
    return out


def plan_windows(frame_off: np.ndarray, h: int, max_window_points: int) -> np.ndarray:
    """Window cuts (frame indices ``0 = c_0 < ... < c_K = F``) for the frame-ordered points delimited by ``frame_off``
    (int64 [F+1]): one window when all points fit ``max_window_points``; otherwise windows of at least ``max(h, 1)``
    frames, each as long as its local problem (the window plus ``h`` frames on each side) stays within the budget. A
    window whose minimum length already exceeds the budget is kept at that minimum."""
    off = np.asarray(frame_off, dtype=np.int64)
    F = len(off) - 1
    if F <= 0:
        raise RadarB200Error("a recording needs at least one frame")
    if off[-1] <= max_window_points:
        return np.array([0, F], dtype=np.int64)
    hmin = max(int(h), 1)
    cuts = [0]
    a = 0
    while a < F:
        base = off[max(a - h, 0)]
        # largest b in [a + hmin, F] with off[min(b + h, F)] - base <= budget (monotone in b)
        lo, hi = min(a + hmin, F), F
        if off[min(lo + h, F)] - base <= max_window_points:
            while lo < hi:
                mid = (lo + hi + 1) // 2
                if off[min(mid + h, F)] - base <= max_window_points:
                    lo = mid
                else:
                    hi = mid - 1
        b = lo
        if 0 < F - b < hmin:                              # the rest would be too short: end this window earlier
            b = F - hmin if F - hmin >= a + hmin else F
        cuts.append(b)
        a = b
    return np.array(cuts, dtype=np.int64)


def stdbscan_windowed(x: torch.Tensor, y: Optional[torch.Tensor], z: Optional[torch.Tensor], frame_off: np.ndarray,
                      frame_ids: np.ndarray, cuts: np.ndarray, eps_space: float, eps_time: float, min_samples: int,
                      bounds4: Optional[np.ndarray] = None):
    """``rb_stdbscan_windowed`` on SoA device tensors: returns ``(labels int32, core uint8, n_clusters)``. ``bounds4`` =
    a box ``[x_min, x_max, y_min, y_max]`` containing every 2-D point: the plans then do not sync."""
    ctx = context(x.device.index)
    off = np.ascontiguousarray(frame_off, dtype=np.int64)
    ids = np.ascontiguousarray(frame_ids, dtype=np.float32)
    cu = np.ascontiguousarray(cuts, dtype=np.int64)
    n = int(off[-1]) if len(off) else 0
    labels = torch.empty(max(n, 1), dtype=torch.int32, device=x.device)
    core = torch.empty(max(n, 1), dtype=torch.uint8, device=x.device)
    hint = None
    if bounds4 is not None and z is None:
        hint = _lib.StdbscanHint()
        hint.lo[0], hint.hi[0], hint.lo[1], hint.hi[1] = (float(v) for v in bounds4)
        hint.times_integer = 1
    ncl = C.c_int64(0)
    check(ctx.lib.rb_stdbscan_windowed(ctx.handle, ptr(x), ptr(y), ptr(z), 1, off.ctypes.data, ids.ctypes.data, len(ids), cu.ctypes.data,
                                       len(cu) - 1, float(eps_space), float(np.float32(eps_time)), int(min_samples),
                                       C.byref(hint) if hint is not None else None, ptr(labels), ptr(core), C.byref(ncl), stream_ptr()),
          "rb_stdbscan_windowed")
    return labels[:n], core[:n], int(ncl.value)


def _available_bytes(device: torch.device) -> int:
    free, _ = torch.cuda.mem_get_info(device)
    return int(free) + int(torch.cuda.memory_reserved(device)) - int(torch.cuda.memory_allocated(device))


@dataclass
class RecordingResult(DetectionResult):
    """Device-resident result of a whole recording: the fields of :class:`DetectionResult` (its ``to_host``,
    ``to_frames``, ``clusters_by_frame`` and ``clusters_by_frame_host`` apply unchanged - the cluster records are built
    over frame chunks small enough for the records' slot table), plus the clustering's window cuts and what ran."""
    core: Optional[torch.Tensor] = None                 # uint8 [points.n]: core flags of the clustered points
    cuts: Optional[np.ndarray] = None                   # window cuts (frame indices) of the clustering
    frames_built: int = 0
    land_ordered: bool = False                          # non-integer intensities: the ordered accumulation ran
    timings: Dict[str, float] = field(default_factory=dict)
    frame_times: Optional[list] = None                  # per frame (timestamp, timestamp_ms) when CSV frames were added
                                                        # (build_frame's, T4:319-323); (None, None) for block frames


class RecordingDetection:
    """Detection over one recording fed as any number of frame blocks (see the module docstring)."""

    def __init__(self, config: Optional[DetectionConfig] = None, device: Optional[int] = None,
                 max_window_points: Optional[int] = None):
        self.pipe = DetectionPipeline(config, device)
        self.cfg, self.device, self.ctx = self.pipe.cfg, self.pipe.device, self.pipe.ctx
        self.max_window_points = None if max_window_points is None else int(max_window_points)
        if self.max_window_points is not None and self.max_window_points < 1:
            raise RadarB200Error("max_window_points must be >= 1")
        self._store = None                              # raw points (x, y, inten, gain), capacity = len
        self._n = 0
        self._offs = [np.zeros(1, np.int64)]            # per block: frame offsets inside the block (from 0)
        self._bases = []                                # per block: first point of the block in the store
        self._ids = []
        self._b4 = None
        self._gain_cache = None
        self._finished = False
        self._times = []                                # per frame: (timestamp, timestamp_ms)
        self._csv_frames = False
        self._reader = None                             # csvbatch.SweepReader: pinned slots, allocated on first use
        #: CSV files parsed in a batch by rb_csv_parse_sweeps / read by the drop-in's per-file reader (unreadable, or
        #: larger than batch_bytes)
        self.csv_files: Dict[str, int] = {"batched": 0, "per_file": 0}
        self.timings: Dict[str, float] = {"spoke": 0.0}

    # ---- blocks -------------------------------------------------------------------------------------------------------
    def _grow(self, need: int) -> None:
        cap = 0 if self._store is None else self._store[0].numel()
        if need <= cap:
            return
        new = max(need, 2 * cap, 1 << 16)
        nbytes = 16 * new
        avail = _available_bytes(self.device)
        if nbytes > avail:
            raise RadarB200Error(f"the recording's point store needs {nbytes} bytes of device memory ({new} points); "
                                 f"{avail} are free")
        d = self.device
        store = (torch.empty(new, dtype=torch.float32, device=d), torch.empty(new, dtype=torch.float32, device=d),
                 torch.empty(new, dtype=torch.float32, device=d), torch.empty(new, dtype=torch.int32, device=d))
        if self._n:
            for s, o in zip(store, self._store):
                s[:self._n].copy_(o[:self._n])
        self._store = store

    def add_block(self, echo: torch.Tensor, cos_tab: torch.Tensor, sin_tab: torch.Tensor, range_res: torch.Tensor,
                  frame_ids: Sequence[int]) -> None:
        """Spoke-to-point for ``echo[F,G,S,E]`` (float32 or uint8, on the device; tables ``[F*G,S]``) with the frame ids
        of its frames, which must continue the recording's strictly increasing integer ids. Only the points are kept."""
        if self._finished:
            raise RadarB200Error("add_block after finish(): start a new RecordingDetection")
        if echo.dim() != 4:
            raise RadarB200Error("echo must be [frames, gains, spokes, bins]")
        F, G, S, E = echo.shape
        if G != len(self.cfg.gains):
            raise RadarB200Error("echo gain dimension does not match config.gains")
        ids = check_frame_ids(frame_ids, self._ids[-1][-1] if self._ids else None)
        if len(ids) != F:
            raise RadarB200Error(f"{len(ids)} frame ids for {F} frames")
        t0 = time.perf_counter()
        cfg, d = self.cfg, echo.device
        W = F * G
        if self._gain_cache is None or self._gain_cache.numel() < W:
            self._gain_cache = torch.tensor(list(cfg.gains) * F, dtype=torch.int32, device=d)
        base = self._n
        off = self._spoke_append(echo.reshape(W, S, E), cos_tab, sin_tab, range_res, self._gain_cache[:W],
                                 lambda sweep_base: dev.frame_offsets(sweep_base, F, G))
        self._add_frames(base, off, ids, [(None, None)] * F)
        self.timings["spoke"] += time.perf_counter() - t0

    def _spoke_append(self, echo3: torch.Tensor, cos_tab, sin_tab, range_res, sweep_gain: torch.Tensor, offsets_of) -> np.ndarray:
        """One spoke launch over ``echo3[W,S,E]`` writing straight behind the store's points, with the capacity negotiation
        of ``run_device_staged``; folds the bounds and advances the store. Returns the host copy of
        ``offsets_of(sweep_base)`` (point offsets from the launch's first point; its last entry = the points written)."""
        W, S, E = echo3.shape
        cfg = self.cfg
        cap = self.pipe._cap_hint or dev.default_capacity(W, S, E, cfg.point_stride)
        while True:
            self._grow(self._n + cap)
            out = (*(t[self._n:] for t in self._store), torch.empty(W + 1, dtype=torch.int64, device=echo3.device))
            x, y, inten, gain, sweep_base = dev.spoke_to_points_raw(echo3, cos_tab, sin_tab, range_res, sweep_gain,
                                                                    cfg.intensity_threshold, cfg.point_stride, cap, out=out)
            cap = out[0].numel()
            off_d = offsets_of(sweep_base)
            b4_d = dev.bounds_counted(x, y, sweep_base[W:])
            off, b4 = dev.to_pinned_host(off_d, b4_d)    # the launch's one read-back
            n = int(off[-1])
            if n <= cap:
                break
            cap = int(n * 1.1) + 1024
        self.pipe._cap_hint = max(self.pipe._cap_hint, int(n * 1.25) + 1024)
        if n:
            self._b4 = b4.copy() if self._b4 is None else np.array(
                [min(self._b4[0], b4[0]), max(self._b4[1], b4[1]), min(self._b4[2], b4[2]), max(self._b4[3], b4[3])], np.float32)
        self._n += n
        return off

    def _add_frames(self, base: int, off: np.ndarray, ids: np.ndarray, times: list) -> None:
        """Book frames whose points start at store index ``base`` (``off`` = their offsets from there)."""
        self._bases.append(base)
        self._offs.append(np.asarray(off, dtype=np.int64))
        self._ids.append(ids)
        self._times.extend(times)

    def add_host_block(self, echo, angle_units, scale, frame_ids: Sequence[int]) -> None:
        """Host echoes (numpy, or a pinned torch tensor) ``[F,G,S,E]``: spoke tables from ``angle_units`` / ``scale`` as
        :meth:`DetectionPipeline.spoke_tables` computes them, upload, then :meth:`add_block`."""
        t = echo if isinstance(echo, torch.Tensor) else torch.from_numpy(
            np.ascontiguousarray(echo, dtype=np.uint8 if np.asarray(echo).dtype == np.uint8 else np.float32))
        F, G, S, E = t.shape
        c, s, r = self.pipe.spoke_tables(angle_units, scale, F, E)
        d = self.device
        self.add_block(t.to(d, non_blocking=True), torch.from_numpy(c).to(d), torch.from_numpy(s).to(d),
                       torch.from_numpy(r).to(d), frame_ids)

    def add_csv_frames(self, frame_files: Sequence[Mapping[int, "os.PathLike"]], frame_ids: Optional[Sequence[int]] = None,
                       num_echo_columns: int = 1024, batch_bytes: int = 64 << 20, readers: Optional[int] = None) -> None:
        """Frames from sweep CSV files, with ``build_frame``'s semantics (T4:312-352) for every frame: ``frame_files[f]``
        maps a gain to its file; sweeps are taken in ascending gain order and their points are labelled with that key (not
        the file's Gain column); unreadable files print the reference's message and are skipped, as are empty and
        header-only ones; a frame left without points keeps its id with zero points. ``frame_ids`` default to the index,
        continuing the recording's ids (from 0). ``config.gains`` is not used: frames may carry any set of gains.

        Files are read by ``readers`` threads into two pinned slots kept by the recording and parsed by
        ``rb_csv_parse_sweeps`` a batch of whole frames (at most ``batch_bytes``) at a time. The slots are allocated when a
        call first needs them and grow, never shrink, when a later call's files need more, up to that call's
        ``batch_bytes``: only a file larger than ``batch_bytes``, or one that cannot be read, takes the drop-in's per-file
        reader (``csv_files`` counts both kinds). What a file outside the device grammar gets instead is decided per file
        (``csvbatch``). Spoke-to-point runs over runs of consecutive sweeps of the same spoke count and echo type,
        appended behind the store in sweep order."""
        from . import csvbatch
        from .tracker import parse_timestamp

        if self._finished:
            raise RadarB200Error("add_csv_frames after finish(): start a new RecordingDetection")
        E = int(num_echo_columns)
        if E < 1:
            raise RadarB200Error("num_echo_columns must be >= 1")
        if not (csvbatch.CSV_CHUNK <= int(batch_bytes) <= csvbatch.MAX_BATCH_BYTES):
            raise RadarB200Error(f"batch_bytes must be in [{csvbatch.CSV_CHUNK}, {csvbatch.MAX_BATCH_BYTES}]")
        frames = [sorted((g, Path(p)) for g, p in ff.items()) for ff in frame_files]
        if not frames:
            if frame_ids is not None and len(frame_ids):
                raise RadarB200Error(f"{len(frame_ids)} frame ids for 0 frames")
            return
        after = self._ids[-1][-1] if self._ids else None
        if frame_ids is None:
            frame_ids = np.arange(len(frames)) + (0 if after is None else after + 1)
        ids = check_frame_ids(frame_ids, after)
        if len(ids) != len(frames):
            raise RadarB200Error(f"{len(ids)} frame ids for {len(frames)} frames")
        times = [parse_timestamp(fr[0][1].name) if fr else (None, None) for fr in frames]        # T4:319-323
        if self._reader is None:
            self._reader = csvbatch.SweepReader()
        for k in ("read", "h2d", "parse", "lead"):
            self.timings.setdefault(k, 0.0)

        def consume(fa, fb, results):
            self._add_csv_batch(results, ids[fa:fb], times[fa:fb], E)

        self._reader.run(frames, E, self.device, readers or min(8, os.cpu_count() or 1), consume, self.timings, batch_bytes)
        self._csv_frames = True

    def _add_csv_batch(self, results, ids: np.ndarray, times: list, E: int) -> None:
        """Spoke stage of one batch of parsed frames (see :meth:`add_csv_frames`), booked as one block."""
        from . import csvbatch
        from .tracker import sweep_tables

        t0 = time.perf_counter()
        d, cfg = self.device, self.cfg
        sweeps, per_frame = [], []                       # sweeps: (gain label, angle, scale, echo device tensor, batch rows)
        for frame in results:
            for _, r in frame:
                self.csv_files["per_file" if r.status is None else "batched"] += 1
            got = [(g, r.sweep, r.rows) for g, r in frame if r.sweep is not None and r.sweep[2].shape[0] > 0]
            host = [isinstance(sw[2], np.ndarray) for _, sw, _ in got]
            as_u8 = [sw[2].astype(np.uint8) if h else None for (_, sw, _), h in zip(got, host)]
            exact = all(np.array_equal(u, sw[2]) for (_, sw, _), u, h in zip(got, as_u8, host) if h)
            for (g, sw, rows), u, h in zip(got, as_u8, host):
                if exact:                                # 0..255 integers travel as uint8 (rb_spoke_to_points_u8)
                    echo = torch.from_numpy(u).to(d) if h else sw[2]
                else:                                    # the frame goes through the float32 kernel
                    echo = torch.from_numpy(np.ascontiguousarray(sw[2], np.float32)).to(d) if h else sw[2].float()
                    rows = None
                sweeps.append((g, sw[0], sw[1], echo, None if h else rows))
            per_frame.append(len(got))
        tl = time.perf_counter()
        self.timings["lead"] += tl - t0
        base = self._n
        sweep_off = [np.zeros(1, np.int64)]
        for a, b in csvbatch.sweep_runs([(sw[3].shape[0], sw[3].dtype) for sw in sweeps]):
            run = sweeps[a:b]
            S = run[0][3].shape[0]
            rows = [sw[4] for sw in run]
            if all(r is not None for r in rows) and all(rows[i][1] == rows[i + 1][0] for i in range(len(rows) - 1)):
                # consecutive rows of the batch's echo (same storage): a view, no copy
                echo = run[0][3].as_strided((b - a, S, E), (S * E, E, 1))
            else:
                echo = torch.stack([sw[3] for sw in run])
            t1 = time.perf_counter()
            c, s_, r = sweep_tables(np.stack([sw[1] for sw in run]), np.stack([sw[2] for sw in run]), E, cfg.angle_scale)
            self.timings["lead"] += time.perf_counter() - t1
            gains = torch.tensor([sw[0] for sw in run], dtype=torch.int32, device=d)
            off = self._spoke_append(echo, *(torch.from_numpy(np.ascontiguousarray(t)).to(d) for t in (c, s_, r)), gains,
                                     lambda sweep_base: sweep_base)
            sweep_off.append(off[1:] + sweep_off[-1][-1])
        self._add_frames(base, csvbatch.frame_offsets(np.concatenate(sweep_off), per_frame), ids, times)
        self.timings["spoke"] += time.perf_counter() - tl

    # ---- the recording ------------------------------------------------------------------------------------------------
    def window_budget(self, n_points: int) -> int:
        """Points per window: ``max_window_points`` if set, else what one ST-DBSCAN call takes (under 2^31 points and
        within the free device memory at ``SCRATCH_BYTES_PER_POINT``)."""
        if self.max_window_points is not None:
            return self.max_window_points
        return max(1, min(MAX_CALL_POINTS, int(0.8 * _available_bytes(self.device)) // SCRATCH_BYTES_PER_POINT))

    def finish(self, cluster: bool = True) -> RecordingResult:
        if self._finished:
            raise RadarB200Error("finish() was already called")
        if not self._ids:
            raise RadarB200Error("finish() without any block")
        self._finished = True
        cfg, d = self.cfg, self.device
        timings = dict(self.timings)
        ids = np.concatenate(self._ids)
        F = len(ids)
        raw_off = np.concatenate([[0]] + [o[1:] + b for o, b in zip(self._offs[1:], self._bases)]).astype(np.int64)
        n_raw = self._n
        if self._store is None:
            self._grow(1)
        xs, ys, iss, gs = self._store
        raw = dev.PointBatch(xs, ys, iss, gs, torch.from_numpy(raw_off).to(d), n_raw)
        built = int(np.count_nonzero(np.diff(raw_off)))
        pts, land, edges, count, isum, land_ordered = raw, None, None, None, None, False

        # ---- land: one grid over the recording, filled chunk by chunk (each chunk < 2^31 points) ---------------------
        t0 = time.perf_counter()
        if cfg.land_filter and n_raw > 0 and built > cfg.land_min_frames:
            b4 = self._b4
            xe, ye = dev.arange_edges(b4[0], b4[1], cfg.land_resolution), dev.arange_edges(b4[2], b4[3], cfg.land_resolution)
            if len(xe) < 2 or len(ye) < 2:
                raise RadarB200Error("degenerate land grid")
            nx, ny = len(xe) - 1, len(ye) - 1
            d_xe, d_ye = torch.from_numpy(xe).to(d), torch.from_numpy(ye).to(d)
            chunks = self._chunks(raw_off)
            count = torch.zeros((nx, ny), dtype=torch.int32, device=d)
            isum = torch.zeros((nx, ny), dtype=torch.float64, device=d)
            lib, h = self.ctx.lib, self.ctx.handle
            for ordered in (False, True):
                entry = lib.rb_land_accumulate_ordered if ordered else lib.rb_land_accumulate
                for fa, fb in chunks:                    # in block order: the ordered kernel continues from the stored sums
                    a, b = int(raw_off[fa]), int(raw_off[fb])
                    check(entry(h, ptr(xs[a:]), ptr(ys[a:]), ptr(iss[a:]), b - a, ptr(d_xe), nx + 1, ptr(d_ye), ny + 1, ptr(count),
                                ptr(isum), stream_ptr()), "rb_land_accumulate")
                if ordered:
                    break
                flag = C.c_int32(0)
                check(lib.rb_land_accumulate_status(h, C.byref(flag), stream_ptr()), "rb_land_accumulate_status")
                if not flag.value:
                    break
                land_ordered = True
                count.zero_(), isum.zero_()
            land = dev.land_cells(count, isum, built, cfg.land_persistence, cfg.land_min_intensity)
            fx, fy, fi = (torch.empty(max(n_raw, 1), dtype=torch.float32, device=d) for _ in range(3))
            fg = torch.empty(max(n_raw, 1), dtype=torch.int32, device=d)
            f_off = np.zeros(F + 1, np.int64)
            at = 0
            for fa, fb in chunks:
                a, b = int(raw_off[fa]), int(raw_off[fb])
                loc_off = torch.from_numpy(raw_off[fa:fb + 1] - a).to(d)
                out_off = torch.empty(fb - fa + 1, dtype=torch.int64, device=d)
                check(lib.rb_land_filter(h, ptr(xs[a:]), ptr(ys[a:]), ptr(iss[a:]), ptr(gs[a:]), b - a, ptr(loc_off), fb - fa,
                                         ptr(d_xe), nx + 1, ptr(d_ye), ny + 1, ptr(land), ptr(fx[at:]), ptr(fy[at:]), ptr(fi[at:]),
                                         ptr(fg[at:]), ptr(out_off), None, stream_ptr()), "rb_land_filter")
                o = out_off.cpu().numpy()
                f_off[fa + 1:fb + 1] = o[1:] + at
                at += int(o[-1])
            pts = dev.PointBatch(fx, fy, fi, fg, torch.from_numpy(f_off).to(d), at)
            edges = (xe, ye)
        torch.cuda.current_stream(d).synchronize()
        timings["land"] = time.perf_counter() - t0

        # ---- one ST-DBSCAN labelling of the recording ----------------------------------------------------------------
        t0 = time.perf_counter()
        labels = torch.empty(0, dtype=torch.int32, device=d)
        core, cuts, n_clusters = None, None, 0
        if cluster and pts.n > 0:
            p_off = raw_off if pts is raw else pts.frame_off.cpu().numpy()
            h_t = int(math.floor(np.float32(cfg.eps_time))) if cfg.eps_time >= 0 else 0
            cuts = plan_windows(p_off, h_t, self.window_budget(pts.n))
            z = pts.inten if cfg.cluster_3d else None
            labels, core, n_clusters = stdbscan_windowed(pts.x, pts.y, z, p_off, ids, cuts, cfg.eps_space, cfg.eps_time,
                                                         cfg.min_samples, bounds4=self._b4)
        timings["cluster"] = time.perf_counter() - t0
        return RecordingResult(ids, raw, pts, labels, n_clusters, land, edges, count, isum, core=core, cuts=cuts,
                               frames_built=built, land_ordered=land_ordered, timings=timings,
                               frame_times=list(self._times) if self._csv_frames else None)

    def _chunks(self, raw_off: np.ndarray):
        """Consecutive blocks grouped into frame ranges of fewer than 2^31 points (the land kernels' per-call limit)."""
        out, fa, f = [], 0, 0
        for o in self._offs[1:]:
            fb = f + len(o) - 1
            if raw_off[fb] - raw_off[fa] > MAX_CALL_POINTS and f > fa:
                out.append((fa, f))
                fa = f
            f = fb
        out.append((fa, f))
        return out
