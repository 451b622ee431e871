"""Device-resident stages of the detection path: thin, typed wrappers over the C ABI.

Everything here takes and returns CUDA ``torch`` tensors (torch = allocator + stream only) and
launches the hand-written kernels of ``libradarb200.so`` on torch's current stream. No stage has a
CPU implementation; calling one without a GPU raises :class:`RadarB200Error`.
"""
from __future__ import annotations

import ctypes as C
import os
import threading
from dataclasses import dataclass
from typing import Optional, Tuple

import numpy as np
import torch

from . import _lib
from ._lib import RadarB200Error, check, context, ptr, stream_ptr

check_rc = check


def _dev(t: torch.Tensor, dtype: torch.dtype, name: str) -> torch.Tensor:
    if not t.is_cuda:
        raise RadarB200Error(f"{name} must be a CUDA tensor")
    if t.dtype != dtype:
        raise RadarB200Error(f"{name} must be {dtype}, got {t.dtype}")
    return t.contiguous()


@dataclass
class PointBatch:
    """Points of a batch of frames, SoA on the device, frames concatenated in order.

    ``frame_off`` (int64[F+1], device) delimits the frames; ``n`` is the number of valid points
    (host int). The tensors may be longer than ``n`` (capacity)."""
    x: torch.Tensor
    y: torch.Tensor
    inten: torch.Tensor
    gain: torch.Tensor
    frame_off: torch.Tensor
    n: int

    def trimmed(self) -> "PointBatch":
        n = self.n
        return PointBatch(self.x[:n], self.y[:n], self.inten[:n], self.gain[:n], self.frame_off, n)


_staging = threading.local()
# how results travel device -> host: "staging" (default), "pinned" (a fresh pinned tensor per array, handed out without
# a host copy) or "pageable" (plain .cpu()); the environment variable is for measurements only
HOST_READBACK_MODE = os.environ.get("RB_HOST_READBACK", "staging")


def _staging_views(buf: torch.Tensor, tensors) -> list:
    """Views into the byte buffer ``buf``, one per tensor (same dtype and shape), at 256-byte aligned offsets."""
    views, off = [], 0
    for t in tensors:
        nb = t.numel() * t.element_size()
        views.append(buf[off:off + nb].view(t.dtype).view(t.shape))
        off += (nb + 255) & ~255
    return views


def _staging_buffer(nbytes: int, pinned: bool) -> torch.Tensor:
    """This thread's reusable host staging buffer, grown geometrically: after the first blocks of a run no call
    allocates page-locked memory any more."""
    buf = getattr(_staging, "buf", None)
    if buf is None or buf.numel() < nbytes or buf.is_pinned() != pinned:
        _staging.buf = buf = None                                   # give the old block back before asking for a bigger one
        _staging.buf = buf = torch.empty(max(nbytes + nbytes // 2, 1 << 20), dtype=torch.uint8, pin_memory=pinned)
    return buf


def to_pinned_host(*tensors):
    """Device tensors -> numpy arrays through PINNED host memory: all copies in flight together and ONE stream sync.
    A plain ``.cpu()`` goes through pageable memory at a fraction of the PCIe rate, which is what a dense block's
    read-back (config 4: 1.4 GB of points and labels per 32 frames) is made of. The pinned memory is a per-thread
    staging buffer that is reused from call to call and the arrays handed out are ordinary numpy copies of it: allocating
    page-locked memory is an implicit device-wide synchronisation point, and a caller that keeps its results (so that
    torch's host cache can never recycle the blocks) would pay for it on every block - seen once on one box, two blocks in flight:
    152 ms per 128-frame block instead of 62 (profiles/r02_e2e_readback_modes.txt)."""
    if not tensors:
        return []
    if not tensors[0].is_cuda:
        return [t.detach().clone().numpy() for t in tensors]
    if HOST_READBACK_MODE == "pageable":
        return [t.cpu().numpy() for t in tensors]
    stream = torch.cuda.current_stream(tensors[0].device)
    if HOST_READBACK_MODE == "pinned":
        host = [torch.empty(t.shape, dtype=t.dtype, pin_memory=True) for t in tensors]
        for h, t in zip(host, tensors):
            h.copy_(t, non_blocking=True)
        stream.synchronize()
        return [h.numpy() for h in host]
    total = sum((t.numel() * t.element_size() + 255) & ~255 for t in tensors)
    views = _staging_views(_staging_buffer(total, True), tensors)
    for v, t in zip(views, tensors):
        if t.numel():
            v.copy_(t, non_blocking=True)
    stream.synchronize()
    return [np.array(v.numpy()) for v in views]                     # np.array copies: the staging buffer is free again


# --------------------------------------------------------------------------------------- a1 + a2
def spoke_to_points_raw(echo: torch.Tensor, cos_tab: torch.Tensor, sin_tab: torch.Tensor,
                        range_res: Optional[torch.Tensor], sweep_gain: torch.Tensor, threshold: float, stride: int,
                        cap: int, out: Optional[Tuple[torch.Tensor, ...]] = None,
                        ranges: Optional[torch.Tensor] = None):
    """One launch over ``echo[W,S,E]``; returns ``(x, y, inten, gain, sweep_base)`` without syncing.
    ``sweep_base[W]`` (device) is the true total, which may exceed ``cap`` (then points were dropped)."""
    ctx = context(echo.device.index)
    if echo.dtype not in (torch.float32, torch.uint8):
        raise RadarB200Error(f"echo must be float32 or uint8, got {echo.dtype}")
    echo = _dev(echo, echo.dtype, "echo")
    if echo.dim() != 3:
        raise RadarB200Error("echo must be [sweeps, spokes, bins]")
    W, S, E = echo.shape
    cos_tab = _dev(cos_tab, torch.float32, "cos_tab")
    sin_tab = _dev(sin_tab, torch.float32, "sin_tab")
    if range_res is not None:
        range_res = _dev(range_res, torch.float32, "range_res")
    if ranges is not None:
        ranges = _dev(ranges, torch.float32, "ranges")
        if ranges.numel() != W * S * E:
            raise RadarB200Error("ranges must be [sweeps, spokes, bins]")
    elif range_res is None:
        raise RadarB200Error("need range_res or ranges")
    sweep_gain = _dev(sweep_gain, torch.int32, "sweep_gain")
    if cos_tab.numel() != W * S or sin_tab.numel() != W * S or (range_res is not None and range_res.numel() != W * S):
        raise RadarB200Error("spoke tables must be [sweeps, spokes]")
    if sweep_gain.numel() != W:
        raise RadarB200Error("sweep_gain must be [sweeps]")
    dev = echo.device
    if out is None:
        x = torch.empty(cap, dtype=torch.float32, device=dev)
        y = torch.empty(cap, dtype=torch.float32, device=dev)
        inten = torch.empty(cap, dtype=torch.float32, device=dev)
        gain = torch.empty(cap, dtype=torch.int32, device=dev)
        sweep_base = torch.empty(W + 1, dtype=torch.int64, device=dev)
    else:
        x, y, inten, gain, sweep_base = out
        cap = min(x.numel(), y.numel(), inten.numel(), gain.numel())
    entry = ctx.lib.rb_spoke_to_points_u8 if echo.dtype == torch.uint8 else ctx.lib.rb_spoke_to_points
    check(entry(ctx.handle, ptr(echo), ptr(cos_tab), ptr(sin_tab), ptr(range_res),
                ptr(ranges), ptr(sweep_gain), W, S, E, float(threshold), int(stride),
                ptr(x), ptr(y), ptr(inten), ptr(gain), cap, ptr(sweep_base), stream_ptr()),
          "rb_spoke_to_points")
    return x, y, inten, gain, sweep_base


def default_capacity(W: int, S: int, E: int, stride: int) -> int:
    worst = W * ((S * E + max(stride, 1) - 1) // max(stride, 1))
    if worst * 16 <= (1 << 30):
        return max(worst, 1)
    return max(worst // 8, 1 << 22)


def spoke_to_points(echo: torch.Tensor, cos_tab: torch.Tensor, sin_tab: torch.Tensor,
                    range_res: Optional[torch.Tensor], sweep_gain: torch.Tensor, threshold: float, stride: int,
                    gains_per_frame: int = 1, cap: Optional[int] = None,
                    ranges: Optional[torch.Tensor] = None) -> PointBatch:
    """Spoke-to-point for ``echo[W,S,E]`` (W = frames x gains, frame major). Syncs once to learn the
    point count; re-runs with a larger buffer if the capacity guess was too small."""
    W, S, E = echo.shape
    if W % gains_per_frame:
        raise RadarB200Error("sweeps must be a multiple of gains_per_frame")
    if cap is None:
        cap = default_capacity(W, S, E, stride)
    ctx = context(echo.device.index)
    while True:
        x, y, inten, gain, sweep_base = spoke_to_points_raw(echo, cos_tab, sin_tab, range_res, sweep_gain,
                                                            threshold, stride, cap, ranges=ranges)
        n = int(sweep_base[-1].item())
        if n <= cap:
            break
        cap = n
    F = W // gains_per_frame
    frame_off = torch.empty(F + 1, dtype=torch.int64, device=echo.device)
    check(ctx.lib.rb_frame_offsets(ctx.handle, ptr(sweep_base), F, gains_per_frame, ptr(frame_off), stream_ptr()),
          "rb_frame_offsets")
    return PointBatch(x, y, inten, gain, frame_off, n)


def polar_to_cartesian(ranges: torch.Tensor, cos_tab: torch.Tensor, sin_tab: torch.Tensor):
    """Full-grid ``x = ranges*cos[:,None]``, ``y = ranges*sin[:,None]`` (PKG transforms.py:13-34)."""
    ctx = context(ranges.device.index)
    ranges = _dev(ranges, torch.float32, "ranges")
    n, m = ranges.shape
    x = torch.empty_like(ranges)
    y = torch.empty_like(ranges)
    check(ctx.lib.rb_polar_to_cartesian(ctx.handle, ptr(ranges), ptr(_dev(cos_tab, torch.float32, "cos_tab")),
                                        ptr(_dev(sin_tab, torch.float32, "sin_tab")), n, m, ptr(x), ptr(y),
                                        stream_ptr()), "rb_polar_to_cartesian")
    return x, y


def frame_offsets(sweep_base: torch.Tensor, n_frames: int, gains_per_frame: int) -> torch.Tensor:
    ctx = context(sweep_base.device.index)
    frame_off = torch.empty(n_frames + 1, dtype=torch.int64, device=sweep_base.device)
    check(ctx.lib.rb_frame_offsets(ctx.handle, ptr(sweep_base), n_frames, gains_per_frame, ptr(frame_off),
                                   stream_ptr()), "rb_frame_offsets")
    return frame_off


def expand_frame_times(frame_off: torch.Tensor, frame_ids: torch.Tensor, n_points: int) -> torch.Tensor:
    """float32 frame id per point (reference T4:460,467)."""
    ctx = context(frame_off.device.index)
    frame_ids = _dev(frame_ids, torch.float32, "frame_ids")
    frame_off = _dev(frame_off, torch.int64, "frame_off")
    times = torch.empty(max(n_points, 1), dtype=torch.float32, device=frame_off.device)[:n_points]
    check(ctx.lib.rb_expand_frame_times(ctx.handle, ptr(frame_off), ptr(frame_ids), frame_ids.numel(), n_points,
                                        ptr(times), stream_ptr()), "rb_expand_frame_times")
    return times


# --------------------------------------------------------------------------------------- a3
def fuse_max_cells(x: torch.Tensor, y: torch.Tensor, inten: torch.Tensor, x_min: float, y_min: float,
                   resolution: float, nx: int, ny: int):
    """Occupied cells of the max-pooling grid in y-major order: ``(ix, iy, max_intensity)``."""
    ctx = context(x.device.index)
    n = x.numel()
    cap = min(n, nx * ny)
    ix = torch.empty(max(cap, 1), dtype=torch.int32, device=x.device)
    iy = torch.empty(max(cap, 1), dtype=torch.int32, device=x.device)
    mx = torch.empty(max(cap, 1), dtype=torch.float32, device=x.device)
    n_cells = C.c_int64(0)
    check(ctx.lib.rb_fuse_max(ctx.handle, ptr(_dev(x, torch.float32, "x")), ptr(_dev(y, torch.float32, "y")),
                              ptr(_dev(inten, torch.float32, "inten")), n, float(x_min), float(y_min),
                              float(resolution), int(nx), int(ny), ptr(ix), ptr(iy), ptr(mx), cap,
                              C.byref(n_cells), stream_ptr()), "rb_fuse_max")
    k = n_cells.value
    return ix[:k], iy[:k], mx[:k]


# --------------------------------------------------------------------------------------- a4-a6
def bounds(x: torch.Tensor, y: torch.Tensor) -> torch.Tensor:
    """Device float32 ``[x_min, x_max, y_min, y_max]`` (no sync)."""
    ctx = context(x.device.index)
    out = torch.empty(4, dtype=torch.float32, device=x.device)
    check(ctx.lib.rb_bounds(ctx.handle, ptr(_dev(x, torch.float32, "x")), ptr(_dev(y, torch.float32, "y")),
                            x.numel(), ptr(out), stream_ptr()), "rb_bounds")
    return out


def bounds_counted(x: torch.Tensor, y: torch.Tensor, n_dev: torch.Tensor) -> torch.Tensor:
    """:func:`bounds` over the first ``min(n_dev[0], len(x))`` points, the count being a device int64 (no sync)."""
    ctx = context(x.device.index)
    out = torch.empty(4, dtype=torch.float32, device=x.device)
    check(ctx.lib.rb_bounds_counted(ctx.handle, ptr(_dev(x, torch.float32, "x")), ptr(_dev(y, torch.float32, "y")),
                                    ptr(_dev(n_dev, torch.int64, "n_dev")), x.numel(), ptr(out), stream_ptr()), "rb_bounds_counted")
    return out


def land_accumulate(x, y, inten, x_edges: torch.Tensor, y_edges: torch.Tensor,
                    count: Optional[torch.Tensor] = None, isum: Optional[torch.Tensor] = None, check: bool = True):
    """Accumulate per-cell point counts (int32) and intensity sums (float64) — T4:378-389.

    The fast kernel is exact for integer-valued intensities (radar echoes) and checks that on the device. With
    ``check=True`` (one stream sync) a batch with other intensities is accumulated again by the ordered kernel, which adds
    in ``np.add.at``'s order; ``check=False`` leaves the flag to the caller (``land_accumulate_flag``)."""
    ctx = context(x.device.index)
    x_edges = _dev(x_edges, torch.float64, "x_edges")
    y_edges = _dev(y_edges, torch.float64, "y_edges")
    nx, ny = x_edges.numel() - 1, y_edges.numel() - 1
    fresh = count is None
    if fresh:
        count = torch.zeros((nx, ny), dtype=torch.int32, device=x.device)
        isum = torch.zeros((nx, ny), dtype=torch.float64, device=x.device)
    elif check:
        count0, isum0 = count.clone(), isum.clone()
    args = (ctx.handle, ptr(_dev(x, torch.float32, "x")), ptr(_dev(y, torch.float32, "y")), ptr(_dev(inten, torch.float32, "inten")),
            x.numel(), ptr(x_edges), nx + 1, ptr(y_edges), ny + 1, ptr(count), ptr(isum), stream_ptr())
    check_rc(ctx.lib.rb_land_accumulate(*args), "rb_land_accumulate")
    if check:
        flag = C.c_int32(0)
        check_rc(ctx.lib.rb_land_accumulate_status(ctx.handle, C.byref(flag), stream_ptr()), "rb_land_accumulate_status")
        if flag.value:
            if fresh:
                count.zero_(), isum.zero_()
            else:
                count.copy_(count0), isum.copy_(isum0)
            check_rc(ctx.lib.rb_land_accumulate_ordered(*args), "rb_land_accumulate_ordered")
    return count, isum


def land_accumulate_flag(device_index: Optional[int] = None) -> torch.Tensor:
    """Device int32[1]: 1 if a ``land_accumulate(check=False)`` call since the last query saw a non-integer intensity
    (copy enqueued on the current stream, no sync; the library's flag is cleared)."""
    ctx = context(device_index)
    out = torch.zeros(1, dtype=torch.int32, device=torch.device("cuda", ctx.device))
    check_rc(ctx.lib.rb_land_accumulate_status_async(ctx.handle, ptr(out), stream_ptr()), "rb_land_accumulate_status_async")
    return out


def land_cells(count: torch.Tensor, isum: torch.Tensor, num_frames: int, persistence: float,
               min_intensity: float) -> torch.Tensor:
    ctx = context(count.device.index)
    land = torch.empty(count.shape, dtype=torch.uint8, device=count.device)
    check(ctx.lib.rb_land_cells(ctx.handle, ptr(_dev(count, torch.int32, "count")),
                                ptr(_dev(isum, torch.float64, "isum")), count.numel(), int(num_frames),
                                float(persistence), float(min_intensity), ptr(land), stream_ptr()), "rb_land_cells")
    return land


def land_filter(batch: PointBatch, x_edges: torch.Tensor, y_edges: torch.Tensor, land: torch.Tensor,
                want_mask: bool = False, sync: bool = True):
    """Order-preserving removal of land points for all frames at once — T4:413-436.
    Returns a new :class:`PointBatch` (and the uint8 keep mask if asked)."""
    ctx = context(batch.x.device.index)
    n = batch.n
    dev = batch.x.device
    F = batch.frame_off.numel() - 1
    xo = torch.empty(max(n, 1), dtype=torch.float32, device=dev)
    yo = torch.empty(max(n, 1), dtype=torch.float32, device=dev)
    io = torch.empty(max(n, 1), dtype=torch.float32, device=dev)
    go = torch.empty(max(n, 1), dtype=torch.int32, device=dev)
    fo = torch.empty(F + 1, dtype=torch.int64, device=dev)
    mask = torch.empty(max(n, 1), dtype=torch.uint8, device=dev) if want_mask else None
    x_edges = _dev(x_edges, torch.float64, "x_edges")
    y_edges = _dev(y_edges, torch.float64, "y_edges")
    land = _dev(land, torch.uint8, "land")
    check(ctx.lib.rb_land_filter(ctx.handle, ptr(batch.x), ptr(batch.y), ptr(batch.inten), ptr(batch.gain), n,
                                 ptr(batch.frame_off), F, ptr(x_edges), x_edges.numel(), ptr(y_edges),
                                 y_edges.numel(), ptr(land), ptr(xo), ptr(yo), ptr(io), ptr(go), ptr(fo),
                                 ptr(mask), stream_ptr()), "rb_land_filter")
    n_out = int(fo[-1].item()) if sync else -1
    out = PointBatch(xo, yo, io, go, fo, n_out)
    return (out, mask[:n]) if want_mask else out


# --------------------------------------------------------------------------------------- a7
def stdbscan(x: torch.Tensor, y: Optional[torch.Tensor], z: Optional[torch.Tensor], times: torch.Tensor,
             eps_space: float, eps_time: float, min_samples: int, stride: int = 1, n: Optional[int] = None,
             want_core: bool = False, min_frames: Optional[int] = None):
    """ST-DBSCAN labels (int32, the reference's own numbering). ``x/y/z`` may be SoA tensors
    (stride 1) or views into one row-major ``[N,D]`` tensor (stride D)."""
    ctx = context(x.device.index)
    if n is None:
        n = times.numel()
    dev = x.device
    labels = torch.empty(max(n, 1), dtype=torch.int32, device=dev)[:n]
    core = torch.empty(max(n, 1), dtype=torch.uint8, device=dev)[:n] if want_core else None
    ncl = C.c_int64(0)
    for name, t in (("x", x), ("y", y), ("z", z), ("times", times)):
        if t is not None and (not t.is_cuda or t.dtype != torch.float32):
            raise RadarB200Error(f"{name} must be a float32 CUDA tensor")
    if min_frames is None:
        check(ctx.lib.rb_stdbscan(ctx.handle, ptr(x), ptr(y), ptr(z), int(stride), ptr(times), int(n),
                                  float(eps_space), float(np.float32(eps_time)), int(min_samples), ptr(labels), ptr(core),
                                  C.byref(ncl), stream_ptr()), "rb_stdbscan")
    else:                                                         # PointCloudWorkF variant (WF:264-369)
        check(ctx.lib.rb_stdbscan_wf(ctx.handle, ptr(x), ptr(y), ptr(z), int(stride), ptr(times), int(n),
                                     float(eps_space), float(np.float32(eps_time)), int(min_samples), int(min_frames),
                                     ptr(labels), ptr(core), C.byref(ncl), stream_ptr()), "rb_stdbscan_wf")
    if want_core:
        return labels, core, ncl.value
    return labels, ncl.value


class StDbscanPhases:
    """ST-DBSCAN in phases (``rb_stdbscan_plan`` / ``_cores`` / ``_set_cores`` / ``_components`` /
    ``_assign``) for callers that exchange data in between — the time-sharded multi-GPU driver.
    Points are SoA tensors (stride 1) or views into one row-major ``[N,D]`` tensor (stride D)."""

    def __init__(self, x: torch.Tensor, y: Optional[torch.Tensor], z: Optional[torch.Tensor], times: torch.Tensor,
                 eps_space: float, eps_time: float, min_samples: int, stride: int = 1, n: Optional[int] = None,
                 hint: Optional[Tuple[float, ...]] = None):
        """``hint`` = ``(x_min, x_max, y_min, y_max, t_min, t_max)`` of a box that contains every point, with integer
        times: the plan then needs no bounds pass and does not sync (``rb_stdbscan_plan_hinted``)."""
        self.ctx = context(x.device.index)
        self.n = times.numel() if n is None else int(n)
        self.device = x.device
        for name, t in (("x", x), ("y", y), ("z", z), ("times", times)):
            if t is not None and (not t.is_cuda or t.dtype != torch.float32):
                raise RadarB200Error(f"{name} must be a float32 CUDA tensor")
        if self.n > 0:
            h = None
            if hint is not None and z is None and y is not None:
                h = _lib.StdbscanHint()
                h.lo[0], h.hi[0], h.lo[1], h.hi[1], h.lo[3], h.hi[3] = (float(v) for v in hint)
                h.lo[2] = h.hi[2] = 0.0
                h.times_integer = 1
            check(self.ctx.lib.rb_stdbscan_plan_hinted(self.ctx.handle, ptr(x), ptr(y), ptr(z), int(stride), ptr(times), self.n,
                                                       float(eps_space), float(np.float32(eps_time)), int(min_samples),
                                                       C.byref(h) if h is not None else None, stream_ptr()), "rb_stdbscan_plan")

    def check(self) -> None:
        """Sync and fail if the ``hint`` box did not contain every point and time (``rb_stdbscan_check``)."""
        if self.n > 0:
            check(self.ctx.lib.rb_stdbscan_check(self.ctx.handle, stream_ptr()), "rb_stdbscan_check")

    def cores(self) -> torch.Tensor:
        core = torch.empty(max(self.n, 1), dtype=torch.uint8, device=self.device)[:self.n]
        if self.n > 0:
            check(self.ctx.lib.rb_stdbscan_cores(self.ctx.handle, ptr(core), stream_ptr()), "rb_stdbscan_cores")
        return core

    def set_cores(self, core: torch.Tensor) -> None:
        if self.n > 0:
            check(self.ctx.lib.rb_stdbscan_set_cores(self.ctx.handle, ptr(_dev(core, torch.uint8, "core")), stream_ptr()),
                  "rb_stdbscan_set_cores")

    def components(self, global_index: Optional[torch.Tensor] = None) -> torch.Tensor:
        key = torch.empty(max(self.n, 1), dtype=torch.int64, device=self.device)[:self.n]
        if self.n > 0:
            gi = None if global_index is None else _dev(global_index, torch.int64, "global_index")
            check(self.ctx.lib.rb_stdbscan_components(self.ctx.handle, ptr(gi), ptr(key), stream_ptr()),
                  "rb_stdbscan_components")
        return key

    def assign(self, core_label: torch.Tensor) -> torch.Tensor:
        labels = torch.empty(max(self.n, 1), dtype=torch.int32, device=self.device)[:self.n]
        if self.n > 0:
            check(self.ctx.lib.rb_stdbscan_assign(self.ctx.handle, ptr(_dev(core_label, torch.int32, "core_label")),
                                                  ptr(labels), stream_ptr()), "rb_stdbscan_assign")
        return labels


def relabel(keys: torch.Tensor, table_keys: torch.Tensor, table_ids: torch.Tensor) -> torch.Tensor:
    """``out[i] = table_ids[j]`` where ``table_keys[j] == keys[i]`` (sorted int64 table); -1 otherwise."""
    ctx = context(keys.device.index)
    keys = _dev(keys, torch.int64, "keys")
    out = torch.empty(max(keys.numel(), 1), dtype=torch.int32, device=keys.device)[:keys.numel()]
    if keys.numel():
        tk = _dev(table_keys, torch.int64, "table_keys")
        ti = _dev(table_ids, torch.int32, "table_ids")
        check(ctx.lib.rb_relabel(ctx.handle, ptr(keys), keys.numel(), ptr(tk), ptr(ti), tk.numel(), ptr(out), stream_ptr()),
              "rb_relabel")
    return out


def stdbscan_stats(device: Optional[int] = None) -> dict:
    ctx = context(device)
    st = _lib.DbscanStats()
    check(ctx.lib.rb_stdbscan_last_stats(ctx.handle, C.byref(st)), "rb_stdbscan_last_stats")
    d = {k: getattr(st, k) for k, _ in st._fields_ if k != "dims"}
    d["dims"] = list(st.dims)
    return d


# --------------------------------------------------------------------------------------- a8: cluster records
def cluster_records(batch: PointBatch, labels: torch.Tensor, n_clusters: int) -> dict:
    """Per-frame cluster records of a labelled batch computed on the device (``rb_cluster_records``; T4:511-534) and
    read back with ONE packed device->host copy into pinned memory. Returns host arrays: the segment table
    ``frame, label, first, count, start, cx, cy, mean_intensity`` (segments ordered by frame, then label; label -1 = the
    frame's noise entry) and the grouped points ``gx, gy, gi`` (each cluster's points contiguous, original order)."""
    ctx = context(batch.x.device.index)
    d = batch.x.device
    n = int(batch.n)
    F = batch.frame_off.numel() - 1
    empty = dict(frame=np.zeros(0, np.int32), label=np.zeros(0, np.int32), first=np.zeros(0, np.int32), count=np.zeros(0, np.int32),
                 start=np.zeros(0, np.int64), cx=np.zeros(0, np.float32), cy=np.zeros(0, np.float32),
                 mean_intensity=np.zeros(0, np.float32), gx=np.zeros(0, np.float32), gy=np.zeros(0, np.float32), gi=np.zeros(0, np.float32))
    if n == 0 or F == 0:
        return empty
    width = int(n_clusters) + 1
    if F * width > (1 << 27):                         # frames are independent: split the call
        half = F // 2
        if half == 0:
            raise RadarB200Error("cluster_records: too many clusters for the slot table")
        off = batch.frame_off
        cut = int(off[half].item())
        a = cluster_records(PointBatch(batch.x[:cut], batch.y[:cut], batch.inten[:cut], batch.gain[:cut], off[:half + 1], cut),
                            labels[:cut], n_clusters)
        b = cluster_records(PointBatch(batch.x[cut:n], batch.y[cut:n], batch.inten[cut:n], batch.gain[cut:n], off[half:] - cut, n - cut),
                            labels[cut:n], n_clusters)
        b["frame"] = b["frame"] + half
        b["start"] = np.where(b["start"] >= 0, b["start"] + len(a["gx"]), -1)
        return {k: np.concatenate([a[k], b[k]]) for k in a}
    labels = _dev(labels, torch.int32, "labels")
    cap = min(n + F, F * width)
    guess = getattr(cluster_records, "_cap_hint", 0) or min(cap, max(4096, 64 * F))
    while True:
        cap_s = min(cap, guess)
        # one packed buffer: 4 int32 columns | start (int64) | 3 float32 columns | 3 grouped float32 arrays
        i32 = torch.empty(4 * cap_s, dtype=torch.int32, device=d)
        i64 = torch.empty(cap_s, dtype=torch.int64, device=d)
        f32 = torch.empty(3 * cap_s + 3 * n, dtype=torch.float32, device=d)
        tab = _lib.ClusterTable(*(ptr(i32[k * cap_s:]) for k in range(4)), ptr(i64), *(ptr(f32[k * cap_s:]) for k in range(3)))
        g = f32[3 * cap_s:]
        n_seg, n_grp = C.c_int64(0), C.c_int64(0)
        rc = ctx.lib.rb_cluster_records(ctx.handle, ptr(batch.x), ptr(batch.y), ptr(batch.inten), ptr(labels), n, ptr(batch.frame_off), F,
                                        int(n_clusters), C.byref(tab), cap_s, ptr(g), ptr(g[n:]), ptr(g[2 * n:]), C.byref(n_seg),
                                        C.byref(n_grp), stream_ptr())
        if rc == RB_ERR_CAPACITY and n_seg.value > cap_s:
            guess = int(n_seg.value * 1.25) + 64
            continue
        check(rc, "rb_cluster_records")
        break
    cluster_records._cap_hint = max(getattr(cluster_records, "_cap_hint", 0), int(n_seg.value * 1.25) + 64)
    S, M = int(n_seg.value), int(n_grp.value)
    hi32, hi64, hf32 = i32.cpu().numpy(), i64[:S].cpu().numpy(), f32.cpu().numpy()
    out = {k: hi32[j * cap_s:j * cap_s + S] for j, k in enumerate(("frame", "label", "first", "count"))}
    out["start"] = hi64
    out.update({k: hf32[j * cap_s:j * cap_s + S] for j, k in enumerate(("cx", "cy", "mean_intensity"))})
    base = 3 * cap_s
    out.update(gx=hf32[base:base + M], gy=hf32[base + n:base + n + M], gi=hf32[base + 2 * n:base + 2 * n + M])
    return out


def clusters_from_records(rec: dict, frame_ids, cluster_cls, frame_id_type=int) -> dict:
    """``{frame_id: [Cluster]}`` from the device-computed records, in the reference's order: per frame the clusters come
    out in the iteration order of ``set(frame_labels)`` (T4:518-521), which depends on the order in which the labels
    FIRST OCCUR in the frame (hash collisions, table growth) - replayed here with a real Python set fed in that order.
    ``points`` / ``intensities`` of a cluster are views of the grouped arrays; ``centroid`` rows of one ``[S, 2]`` array."""
    out = {}
    S = len(rec["frame"])
    if S == 0:
        return out
    gxy = np.stack([rec["gx"], rec["gy"]], axis=1)
    gi = rec["gi"]
    cent = np.stack([rec["cx"], rec["cy"]], axis=1)
    frame, label, first = rec["frame"], rec["label"], rec["first"]
    start, count = rec["start"].tolist(), rec["count"].tolist()
    order = np.lexsort((first, frame))                                    # per frame: segments by first occurrence
    lab_l, fr_l = label.tolist(), frame.tolist()
    bounds = np.flatnonzero(np.diff(frame[order], prepend=-1, append=-2))  # starts of the frames' runs in `order`
    order_l = order.tolist()
    ids = [frame_id_type(v) for v in np.asarray(frame_ids).tolist()]
    for a, b in zip(bounds[:-1].tolist(), bounds[1:].tolist()):
        segs = order_l[a:b]
        seg_of = {lab_l[k]: k for k in segs}
        seen = set(lab_l[k] for k in segs)                                 # same insertion order as set(frame_labels)
        seen.discard(-1)
        if not seen:
            continue
        fid = ids[fr_l[segs[0]]]
        lst = []
        for c in seen:
            k = seg_of[c]
            s0 = start[k]
            lst.append(cluster_cls(cluster_id=c, frame_id=fid, points=gxy[s0:s0 + count[k]], intensities=gi[s0:s0 + count[k]],
                                   centroid=cent[k]))
        out[fid] = lst
    return out


# --------------------------------------------------------------------------------------- whole block, one call
RB_ERR_CAPACITY = -3


def arange_edges(lo: float, hi: float, step: float) -> np.ndarray:
    """The library's host-side restatement of ``np.arange(lo32, lo32.dtype.type(hi32 + step), step)`` (T4:372-373)."""
    lib = _lib.load()
    n = int(lib.rb_arange_edges(float(np.float32(lo)), float(np.float32(hi)), float(step), None, 0))
    out = np.empty(max(n, 0), dtype=np.float64)
    if n > 0:
        lib.rb_arange_edges(float(np.float32(lo)), float(np.float32(hi)), float(step), out.ctypes.data, n)
    return out


def detect_block(echo: torch.Tensor, cos_tab: torch.Tensor, sin_tab: torch.Tensor, range_res: torch.Tensor,
                 sweep_gain: torch.Tensor, frame_ids: np.ndarray, params: "_lib.DetectParams", cap: int,
                 max_edges: int, max_cells: int):
    """``rb_detect_block``: the whole hot path for ``echo[F*G,S,E]`` in one library call.
    Returns ``(rc, result struct, buffers dict)``; rc is 0 or ``RB_ERR_CAPACITY`` (the struct then holds the
    sizes that are needed); anything else raises."""
    ctx = context(echo.device.index)
    dev = echo.device
    F = int(params.n_frames)
    f32 = lambda n: torch.empty(max(n, 1), dtype=torch.float32, device=dev)
    i32 = lambda n: torch.empty(max(n, 1), dtype=torch.int32, device=dev)
    t = dict(x=f32(cap), y=f32(cap), inten=f32(cap), gain=i32(cap), frame_off=torch.empty(F + 1, dtype=torch.int64, device=dev),
             fx=f32(cap), fy=f32(cap), finten=f32(cap), fgain=i32(cap), f_frame_off=torch.empty(F + 1, dtype=torch.int64, device=dev),
             labels=i32(cap), count=i32(max_cells), isum=torch.empty(max(max_cells, 1), dtype=torch.float64, device=dev),
             land=torch.empty(max(max_cells, 1), dtype=torch.uint8, device=dev))
    xe = np.empty(max(max_edges, 1), dtype=np.float64)
    ye = np.empty(max(max_edges, 1), dtype=np.float64)
    buf = _lib.DetectBuffers(**{k: ptr(v) for k, v in t.items()}, cap=int(cap), max_cells=int(max_cells),
                             x_edges=xe.ctypes.data, y_edges=ye.ctypes.data, max_edges=int(max_edges))
    res = _lib.DetectResult()
    ids = np.ascontiguousarray(frame_ids, dtype=np.float32)
    if echo.dtype not in (torch.float32, torch.uint8):
        raise RadarB200Error(f"echo must be float32 or uint8, got {echo.dtype}")
    params.echo_u8 = int(echo.dtype == torch.uint8)
    rc = ctx.lib.rb_detect_block(ctx.handle, ptr(_dev(echo, echo.dtype, "echo")), ptr(_dev(cos_tab, torch.float32, "cos_tab")),
                                 ptr(_dev(sin_tab, torch.float32, "sin_tab")), ptr(_dev(range_res, torch.float32, "range_res")),
                                 ptr(_dev(sweep_gain, torch.int32, "sweep_gain")), ids.ctypes.data, C.byref(params), C.byref(buf),
                                 C.byref(res), stream_ptr())
    if rc not in (0, RB_ERR_CAPACITY):
        check(rc, "rb_detect_block")
    t["x_edges"], t["y_edges"] = xe, ye
    return rc, res, t


# --------------------------------------------------------------------------------------- ingest
CSV_STATUS_BITS = {1: "an echo field is not a plain 0..255 integer", 2: "an echo value above 255", 4: "a row without exactly E + 5 fields",
                   8: "a blank line among the rows", 16: "more rows than expected"}


def csv_parse_sweep(raw, n_echo_columns: int, device=None):
    """Parse the echo columns of one sweep CSV on the device (``rb_csv_parse_sweep``; T4:189-206).

    ``raw``: the file's bytes (``bytes`` / ``bytearray`` / uint8 array). Returns ``(echo_u8[S, E] device tensor,
    row_start int32[S], prefix_end int32[S], status)``: rows ``r`` of the file start at byte ``row_start[r]`` and their
    five leading fields end at ``prefix_end[r]`` (host arrays - the caller parses those few bytes itself);
    ``status == 0`` means the file fitted the device grammar, otherwise (see ``CSV_STATUS_BITS``) the caller must parse
    the file with the reference's parser and the other outputs are meaningless."""
    buf = np.frombuffer(raw, dtype=np.uint8) if not isinstance(raw, np.ndarray) else raw
    dev_ = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    ctx = context(dev_.index)
    n = int(buf.size)
    E = int(n_echo_columns)
    if n >= 2 ** 31 - 1:                              # offsets are int32: leave such a file to the reference's parser
        return torch.empty((0, E), dtype=torch.uint8, device=dev_), np.zeros(0, np.int32), np.zeros(0, np.int32), 16
    max_rows = n // (E + 5) + 1                       # a row has at least E + 4 commas and a newline
    staged = torch.empty(max(n, 1), dtype=torch.uint8, pin_memory=True)
    staged[:n].copy_(torch.from_numpy(buf if buf.flags.writeable else buf.copy()))
    text = staged.to(dev_, non_blocking=True)
    echo = torch.empty((max_rows, E), dtype=torch.uint8, device=dev_)
    offs = torch.empty((2, max_rows), dtype=torch.int32, device=dev_)
    info = torch.empty(2, dtype=torch.int32, device=dev_)
    check(ctx.lib.rb_csv_parse_sweep(ctx.handle, ptr(text), n, E, max_rows, ptr(echo), ptr(offs[0]), ptr(offs[1]), ptr(info),
                                     stream_ptr()), "rb_csv_parse_sweep")
    n_lines, status = (int(v) for v in info.cpu().numpy())         # the one sync of the call
    rows = max(n_lines - 1, 0)
    if status or rows == 0:
        return echo[:0], np.zeros(0, np.int32), np.zeros(0, np.int32), status
    host_offs = offs[:, :rows].cpu().numpy()
    return echo[:rows], host_offs[0], host_offs[1], 0


CSV_CHUNK = 4096                                      # files of a batch start at multiples of this (csv.cu)
CSV_LEAD_FIELDS = 32                                  # RB_CSV_LEAD_FIELDS: leading fields outside the device grammar


@dataclass
class CsvBatch:
    """What ``rb_csv_parse_sweeps`` made of a batch of W files. Host arrays except ``echo``: ``status[W]`` (RB_CSV_* bits),
    ``rows[W]`` (rows parsed; 0 for a file with a line-level status), ``row_base[W+1]``, and per parsed row
    ``angle`` / ``scale`` (float32) and file-relative ``row_start`` / ``prefix_end``; ``gain[W]`` = Gain of row 0.
    ``echo`` = uint8 device ``[row_base[W], E]``: file w's sweep is ``echo[row_base[w]:row_base[w + 1]]``."""
    status: np.ndarray
    rows: np.ndarray
    row_base: np.ndarray
    echo: torch.Tensor
    angle: np.ndarray
    scale: np.ndarray
    gain: np.ndarray
    row_start: np.ndarray
    prefix_end: np.ndarray


def csv_parse_sweeps(text: torch.Tensor, file_off: np.ndarray, file_len: np.ndarray, n_echo_columns: int) -> CsvBatch:
    """Parse the W files held by the uint8 device tensor ``text`` (file w = ``text[file_off[w]:file_off[w] + file_len[w]]``,
    offsets ascending multiples of ``CSV_CHUNK``, total under 2^31 bytes): ``rb_csv_sweeps_lines``, one read-back of the
    row counts, exact allocation, ``rb_csv_parse_sweeps``, one read-back of the statuses and leading fields."""
    E = int(n_echo_columns)
    fo = np.ascontiguousarray(file_off, dtype=np.int64)
    fl = np.ascontiguousarray(file_len, dtype=np.int64)
    W, n = len(fo), int(text.numel())
    if len(fl) != W or E < 1 or n >= (1 << 31):
        raise RadarB200Error("csv batch: one length per file, num_echo_columns >= 1 and under 2^31 bytes of text")
    # every kernel attributes a chunk to the last file starting at or before it: files must not overlap
    if W and (np.any(fo % CSV_CHUNK) or np.any(fl < 0) or fo[0] < 0 or np.any(fo[:-1] + fl[:-1] > fo[1:]) or int(fo[-1] + fl[-1]) > n):
        raise RadarB200Error("csv batch: files must lie in the text at ascending, non-overlapping 4096-byte aligned offsets")
    d = text.device
    ctx = context(d.index)
    text = _dev(text, torch.uint8, "text")
    d_off = torch.from_numpy(fo).to(d)
    d_len = torch.from_numpy(fl).to(d)
    chunks = (n + CSV_CHUNK - 1) // CSV_CHUNK
    chunk_base = torch.empty(chunks + 1, dtype=torch.int32, device=d)
    rows_d = torch.empty(max(W, 1), dtype=torch.int32, device=d)
    status_d = torch.empty(max(W, 1), dtype=torch.int32, device=d)
    check(ctx.lib.rb_csv_sweeps_lines(ctx.handle, ptr(text), n, ptr(d_off), ptr(d_len), W, E, ptr(chunk_base), ptr(rows_d), ptr(status_d),
                                      stream_ptr()), "rb_csv_sweeps_lines")
    rows, status, n_nl = to_pinned_host(rows_d[:W], status_d[:W], chunk_base[chunks:])
    rows = np.where(status == 0, rows, 0).astype(np.int64)        # a file with a line-level status is not parsed
    row_base = np.concatenate([[0], np.cumsum(rows)]).astype(np.int64)
    R = int(row_base[-1])
    echo = torch.empty((max(R, 1), E), dtype=torch.uint8, device=d)
    offs = torch.empty((2, max(R, 1)), dtype=torch.int32, device=d)
    lead = torch.empty((2, max(R, 1)), dtype=torch.float32, device=d)
    gain = torch.zeros(max(W, 1), dtype=torch.int32, device=d)
    if R:
        d_base = torch.from_numpy(row_base).to(d)
        check(ctx.lib.rb_csv_parse_sweeps(ctx.handle, ptr(text), n, ptr(d_off), ptr(d_len), W, E, ptr(chunk_base), int(n_nl[0]), ptr(d_base), R,
                                          ptr(echo), ptr(offs[0]), ptr(offs[1]), ptr(lead[0]), ptr(lead[1]), ptr(gain), ptr(status_d),
                                          stream_ptr()), "rb_csv_parse_sweeps")
        status, gain_h, offs_h, lead_h = to_pinned_host(status_d[:W], gain[:W], offs[:, :R], lead[:, :R])
    else:
        gain_h, offs_h, lead_h = np.zeros(W, np.int32), np.zeros((2, 0), np.int32), np.zeros((2, 0), np.float32)
    return CsvBatch(status, rows, row_base, echo[:R], lead_h[0], lead_h[1], gain_h, offs_h[0], offs_h[1])


# --------------------------------------------------------------------------------------- synthetic input
def synth_echo(spec, first_frame: int = 0, n_frames: Optional[int] = None, device=None,
               out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Device twin of :func:`synthetic.synth_echo` for frames ``first_frame .. first_frame+n_frames-1``
    of the data set described by ``spec``: ``[F, G, S, E]`` float32 on the device."""
    from . import synthetic as syn

    if n_frames is None:
        n_frames = spec.frames - first_frame
    device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    ctx = context(device.index)
    G = len(spec.gains)
    W = n_frames * G
    keys = np.array([spec.sweep_key(first_frame + w // G, w % G) for w in range(W)], dtype=np.uint32)
    thr = np.array([spec.clutter_threshold(spec.gains[w % G]) for w in range(W)], dtype=np.uint32)
    rects, offs = syn.rects_to_array(spec, syn.build_rects(spec))
    if len(rects) == 0:
        rects = np.zeros((1, syn.RECT_COLS), dtype=np.int32)
    d_keys = torch.from_numpy(keys.view(np.int32)).to(device)
    d_thr = torch.from_numpy(thr.view(np.int32)).to(device)
    d_rects = torch.from_numpy(rects).to(device)
    d_offs = torch.from_numpy(offs).to(device)
    if out is None:
        out = torch.empty((n_frames, G, spec.spokes, spec.bins), dtype=torch.float32, device=device)
    check(ctx.lib.rb_synth_echo(ctx.handle, ptr(out), W, spec.spokes, spec.bins, G, first_frame, ptr(d_keys),
                                ptr(d_thr), ptr(d_rects), ptr(d_offs), stream_ptr()), "rb_synth_echo")
    return out
