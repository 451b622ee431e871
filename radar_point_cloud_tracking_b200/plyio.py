"""PLY output (SURVEY.md section 8 f, rank 4): the reference's writers and colour helpers with the same names,
arguments and bytes on disk.

* :func:`write_ply_fast` / :func:`write_ply` — ``5_gain_fusion_ply_builder.py:370-403`` / ``:345-367`` (ASCII);
  the body is written by the library's host function ``rb_ply_append_ascii`` (exact ``%.4f``, see ``csrc/plyfmt.cu``)
  instead of a float64 table formatted row by row in Python;
* :func:`write_ply_binary` — the binary branch of ``PointCloudWorkF/stdbscan_denoising_pipeline.py:797-827``;
* :func:`normalize_intensity`, :func:`intensity_to_rgb`, :func:`gain_to_rgb` — ``T5:276-342``;
* whole recordings from the device: :func:`intensity_rgb` / :func:`gain_rgb` colour device tensors on the device, and
  :func:`write_ply_frames` writes one file per frame with the bytes of :func:`write_ply_fast` (or
  :func:`write_ply_binary`), formatted on the device many frames per launch.

Coordinates / colours may be numpy arrays or torch tensors (device tensors are brought back once).
"""
from __future__ import annotations

import ctypes as C
import os
import threading
from pathlib import Path
from typing import Dict, Optional, Sequence, Tuple

import numpy as np

from . import _lib

GAIN_COLORS: Dict[int, Tuple[int, int, int]] = {40: (0, 114, 255), 50: (0, 200, 83), 70: (255, 165, 0), 75: (255, 87, 34)}   # T5:45-50
INTENSITY_PERCENTILE = 99                                                                                   # T5:63

_HEADER = ("ply\nformat {fmt} 1.0\nelement vertex {n}\nproperty float x\nproperty float y\nproperty float z\n"
           "property uchar red\nproperty uchar green\nproperty uchar blue\nend_header\n")


def _host(a) -> np.ndarray:
    if hasattr(a, "detach"):                      # torch tensor, any device
        a = a.detach().cpu().numpy()
    return np.asarray(a)


# ---- colours ------------------------------------------------------------------------------------------
def normalize_intensity(intensity) -> np.ndarray:
    """Intensities scaled to 0..255 between their minimum and their 99th percentile, clipped (T5:276-289)."""
    v = _host(intensity)
    if len(v) == 0:
        return v
    top, low = np.percentile(v, INTENSITY_PERCENTILE), np.min(v)
    if top <= low:
        return np.zeros_like(v)
    return np.clip((v - low) / (top - low) * 255.0, 0, 255)


def intensity_to_rgb(intensity) -> np.ndarray:
    """Blue -> cyan -> green -> yellow -> red over four quarters of 0..255 (T5:292-327): in every quarter one channel
    ramps with ``t = 4 * (v/255 - quarter start)``, the others sit at 0 or 255; ramps are truncated to uint8."""
    u = _host(intensity) / 255.0
    rgb = np.zeros((len(u), 3), dtype=np.uint8)
    quarter = [u < 0.25, (u >= 0.25) & (u < 0.5), (u >= 0.5) & (u < 0.75), u >= 0.75]
    ramp = lambda sel, start: (u[sel] - start) * 4 if start else u[sel] * 4
    q = quarter[0]
    rgb[q, 1] = (ramp(q, 0) * 255).astype(np.uint8); rgb[q, 2] = 255
    q = quarter[1]
    rgb[q, 1] = 255; rgb[q, 2] = ((1 - ramp(q, 0.25)) * 255).astype(np.uint8)
    q = quarter[2]
    rgb[q, 0] = (ramp(q, 0.5) * 255).astype(np.uint8); rgb[q, 1] = 255
    q = quarter[3]
    rgb[q, 0] = 255; rgb[q, 1] = ((1 - ramp(q, 0.75)) * 255).astype(np.uint8)
    return rgb


def gain_to_rgb(gains) -> np.ndarray:
    """One fixed colour per gain label, black for anything else (T5:330-342)."""
    g = _host(gains)
    rgb = np.zeros((len(g), 3), dtype=np.uint8)
    for gain, colour in GAIN_COLORS.items():
        rgb[g == gain] = colour
    return rgb


# ---- writers ------------------------------------------------------------------------------------------
def _append_ascii(path: Path, x: np.ndarray, y: np.ndarray, z: np.ndarray, colors: np.ndarray) -> None:
    """Vertex lines ``%.4f %.4f %.4f %d %d %d``: native for float32 coordinates + uint8 colours, numpy otherwise."""
    if all(a.dtype == np.float32 for a in (x, y, z)) and colors.dtype == np.uint8 and colors.ndim == 2 and colors.shape[1] == 3:
        lib = _lib.load()
        arrs = [np.ascontiguousarray(a) for a in (x, y, z, colors)]
        ptr = lambda a: a.ctypes.data_as(C.c_void_p)
        rc = lib.rb_ply_append_ascii(str(path).encode(), ptr(arrs[0]), ptr(arrs[1]), ptr(arrs[2]), ptr(arrs[3]), len(x))
        if rc != 0:
            raise _lib.RadarB200Error(f"rb_ply_append_ascii: {lib.rb_last_error().decode()}")
        return
    data = np.column_stack([x, y, z, colors[:, 0].astype(int), colors[:, 1].astype(int), colors[:, 2].astype(int)])
    with path.open("a", encoding="utf-8") as fh:
        np.savetxt(fh, data, fmt="%.4f %.4f %.4f %d %d %d")


def write_ply_fast(path: Path, x, y, z, colors) -> None:
    """ASCII PLY, coordinates cast to float32 first (T5:370-403)."""
    path = Path(path)
    x, y, z = (_host(a).astype(np.float32) for a in (x, y, z))
    colors = _host(colors)
    with path.open("w", encoding="utf-8") as fh:
        fh.write(_HEADER.format(fmt="ascii", n=len(x)))
    _append_ascii(path, x, y, z, colors)
    print(f"  Wrote {len(x):,} points to {path.name}")


def write_ply(path: Path, x, y, z, colors) -> None:
    """ASCII PLY, every value formatted as it is (T5:345-367: ``f"{xp:.4f}"`` formats the value's own precision, so
    float64 input is NOT rounded to float32 first - only float32 input takes the native writer)."""
    path = Path(path)
    x, y, z, colors = _host(x), _host(y), _host(z), _host(colors)
    with path.open("w", encoding="utf-8") as fh:
        fh.write(_HEADER.format(fmt="ascii", n=len(x)))
    if all(a.dtype == np.float32 for a in (x, y, z)) and colors.dtype == np.uint8:
        _append_ascii(path, x, y, z, colors)
    else:
        with path.open("a", encoding="utf-8") as fh:
            for xp, yp, zp, (r, g, b) in zip(x, y, z, colors):
                fh.write(f"{xp:.4f} {yp:.4f} {zp:.4f} {r} {g} {b}\n")
    print(f"  Wrote {len(x):,} points to {path.name}")


def write_ply_binary(path: Path, x, y, z, colors) -> None:
    """Binary little-endian PLY: 15-byte records ``<f4 x, y, z; u1 r, g, b`` (WF:797-827). Colours are the caller's
    (the reference derives them from cluster labels / intensities with matplotlib colour maps)."""
    path = Path(path)
    x, y, z, colors = _host(x), _host(y), _host(z), _host(colors)
    rec = np.empty(len(x), dtype=np.dtype([("x", "<f4"), ("y", "<f4"), ("z", "<f4"), ("r", "u1"), ("g", "u1"), ("b", "u1")]))
    rec["x"], rec["y"], rec["z"] = x.astype(np.float32), y.astype(np.float32), z.astype(np.float32)
    rec["r"], rec["g"], rec["b"] = colors[:, 0], colors[:, 1], colors[:, 2]
    with path.open("wb") as fh:
        fh.write(_HEADER.format(fmt="binary_little_endian", n=len(x)).encode("ascii"))
        rec.tofile(fh)


# ---- whole recordings from the device -------------------------------------------------------------------------
#: bytes of the longest vertex line "%.4f %.4f %.4f %d %d %d\n" (three 45-character floats); a chunk of text holds
#: chunk_bytes // PLY_LINE_MAX lines, so it never overflows, whatever the values
PLY_LINE_MAX = 150
PLY_RECORD_BYTES = 15
DEFAULT_CHUNK_BYTES = 256 << 20


def _cuda(t, name: str):
    import torch

    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise _lib.RadarB200Error(f"{name} must be a CUDA tensor")
    return t


def _frame_offsets(frame_off, n: int, name: str = "frame_off") -> np.ndarray:
    """Host copy of a device int64[F+1] offset tensor, checked: non-decreasing, within [0, n]."""
    import torch

    _cuda(frame_off, name)
    if frame_off.dtype != torch.int64 or frame_off.dim() != 1 or frame_off.numel() < 1:
        raise _lib.RadarB200Error(f"{name} must be a 1-D int64 tensor of F + 1 offsets")
    off = frame_off.cpu().numpy()
    if off[0] < 0 or off[-1] > n or np.any(np.diff(off) < 0):
        raise _lib.RadarB200Error(f"{name} must be non-decreasing within [0, {n}]")
    return off


def intensity_rgb(values, frame_off=None, normalize: bool = False):
    """``intensity_to_rgb`` of a float32 / float64 device tensor, on the device (uint8 ``[N, 3]`` CUDA tensor): each frame
    ``[frame_off[f], frame_off[f+1])`` gets ``intensity_to_rgb(normalize_intensity(v))`` with ``normalize``, else
    ``intensity_to_rgb(v)`` (without ``frame_off`` the whole tensor is one frame). Raises :class:`RadarB200Error` for a NaN
    or a value outside [0, 255] after the optional normalisation: the reference's ``astype(np.uint8)`` has no defined
    result there."""
    import torch

    _cuda(values, "values")
    if values.dtype not in (torch.float32, torch.float64) or values.dim() != 1:
        raise _lib.RadarB200Error("values must be a 1-D float32 or float64 tensor")
    n = values.numel()
    if frame_off is None:
        frame_off = torch.tensor([0, n], dtype=torch.int64, device=values.device)
    elif frame_off.device != values.device:
        raise _lib.RadarB200Error("frame_off must be on the device of values")
    off = _frame_offsets(frame_off, n)
    ctx = _lib.context(values.device.index)
    v = values.contiguous()
    rgb = torch.zeros((n, 3), dtype=torch.uint8, device=values.device)
    status = torch.empty(1, dtype=torch.int32, device=values.device)
    with torch.cuda.device(values.device):
        _lib.check(ctx.lib.rb_ply_colors_intensity(ctx.handle, _lib.ptr(v), int(v.dtype == torch.float64), n, _lib.ptr(frame_off),
                                                   len(off) - 1, int(bool(normalize)), _lib.ptr(rgb), _lib.ptr(status),
                                                   _lib.stream_ptr()), "rb_ply_colors_intensity")
        if int(status.item()):
            raise _lib.RadarB200Error("intensity_rgb: a value is NaN or outside [0, 255]" + (" after normalisation" if normalize else "")
                                      + "; intensity_to_rgb has no defined colour for it")
    return rgb


def gain_rgb(gains):
    """``gain_to_rgb`` of an int32 device tensor, on the device (uint8 ``[N, 3]`` CUDA tensor)."""
    import torch

    _cuda(gains, "gains")
    if gains.dtype != torch.int32 or gains.dim() != 1:
        raise _lib.RadarB200Error("gains must be a 1-D int32 tensor")
    ctx = _lib.context(gains.device.index)
    g = gains.contiguous()
    rgb = torch.empty((g.numel(), 3), dtype=torch.uint8, device=g.device)
    with torch.cuda.device(g.device):
        _lib.check(ctx.lib.rb_ply_colors_gain(ctx.handle, _lib.ptr(g), g.numel(), _lib.ptr(rgb), _lib.stream_ptr()),
                   "rb_ply_colors_gain")
    return rgb


def plan_chunks(off: np.ndarray, lines_per_chunk: int):
    """Cut the vertices ``[off[0], off[-1])`` into chunks of at most ``lines_per_chunk`` lines. Returns a list of
    ``(v0, v1, pieces)``: ``pieces`` = ``(frame, a, b)`` vertex ranges of the chunk in frame order. A frame spanning chunks
    has a piece in each; a frame without vertices has one empty piece, in the chunk that holds its position (the last
    chunk for the end), so every frame's last piece comes no earlier than the previous frame's."""
    if lines_per_chunk < 1:
        raise _lib.RadarB200Error("a chunk must hold at least one line")
    start, end = int(off[0]), int(off[-1])
    n_chunks = max(1, -(-(end - start) // lines_per_chunk))
    bounds = [(start + k * lines_per_chunk, min(end, start + (k + 1) * lines_per_chunk)) for k in range(n_chunks)]
    pieces = [[] for _ in range(n_chunks)]
    for f in range(len(off) - 1):
        a, b = int(off[f]), int(off[f + 1])
        if a == b:
            pieces[min((a - start) // lines_per_chunk, n_chunks - 1)].append((f, a, a))
            continue
        for k in range((a - start) // lines_per_chunk, (b - 1 - start) // lines_per_chunk + 1):
            v0, v1 = bounds[k]
            pieces[k].append((f, max(a, v0), min(b, v1)))
    return [(v0, v1, p) for (v0, v1), p in zip(bounds, pieces)]


_ply_staging = threading.local()


def _pinned_pair(nbytes: int):
    """This thread's two pinned staging buffers of at least ``nbytes`` each, kept from call to call."""
    import torch

    bufs = getattr(_ply_staging, "bufs", None)
    if bufs is None or bufs[0].numel() < nbytes:
        _ply_staging.bufs = None
        _ply_staging.bufs = bufs = [torch.empty(nbytes, dtype=torch.uint8, pin_memory=True) for _ in range(2)]
    return bufs


def _write_piece(path: Path, header: Optional[bytes], body) -> None:
    try:
        with path.open("wb" if header is not None else "ab") as fh:
            if header is not None:
                fh.write(header)
            fh.write(body)
    except OSError as e:
        raise _lib.RadarB200Error(f"write_ply_frames: cannot write {path}: {e}") from None


def write_ply_frames(paths: Sequence, x, y, z, colors, frame_off, binary: bool = False,
                     chunk_bytes: int = DEFAULT_CHUNK_BYTES, writers: Optional[int] = None,
                     timings: Optional[Dict[str, float]] = None) -> None:
    """One PLY file per frame from device tensors: file k gets exactly the bytes of
    ``write_ply_fast(paths[k], x[a:b], y[a:b], z[a:b], colors[a:b])`` (``write_ply_binary``'s with ``binary``) for
    ``a, b = frame_off[k], frame_off[k+1]``, and in ASCII the same ``Wrote`` line is printed per file, in order.

    ``x, y, z``: floating CUDA tensors (cast to float32 first), ``colors``: uint8 ``[N, 3]``, ``frame_off``: int64 ``[F+1]``
    (``PointBatch.frame_off`` or ``FusedFrames.cell_off``), all on one device; ``len(paths) == F``. The text is formatted
    on the device (``rb_ply_format_ascii`` / ``rb_ply_pack_binary``) in chunks of at most ``chunk_bytes``, never splitting a
    line (a frame may span chunks: its file is appended in order), and copied into two pinned buffers that are kept from
    call to call. While ``writers`` threads write one chunk's files, the next chunk is formatted and copied. A chunk costs
    two syncs (one with ``binary``), whatever the number of frames in it. Every argument is checked before any device work
    or file creation. ``timings`` (optional) accumulates the seconds of "format" (CUDA events), "d2h" and "write"."""
    import time
    from concurrent.futures import ThreadPoolExecutor

    import torch

    paths = [Path(p) for p in paths]
    for name, t in (("x", x), ("y", y), ("z", z)):
        _cuda(t, name)
        if not t.is_floating_point() or t.dim() != 1:
            raise _lib.RadarB200Error(f"{name} must be a 1-D floating tensor")
    _cuda(colors, "colors")
    if colors.dtype != torch.uint8 or colors.dim() != 2 or colors.shape[1] != 3:
        raise _lib.RadarB200Error("colors must be a uint8 [N, 3] tensor")
    _cuda(frame_off, "frame_off")
    device = x.device
    if any(t.device != device for t in (y, z, colors, frame_off)):
        raise _lib.RadarB200Error("x, y, z, colors and frame_off must be on one device")
    unit = PLY_RECORD_BYTES if binary else PLY_LINE_MAX
    if int(chunk_bytes) < unit:
        raise _lib.RadarB200Error(f"chunk_bytes must be at least {unit}")
    n = min(x.numel(), y.numel(), z.numel(), colors.shape[0])
    off = _frame_offsets(frame_off, n)
    if len(paths) != len(off) - 1:
        raise _lib.RadarB200Error(f"{len(paths)} paths for {len(off) - 1} frames")

    timings = {} if timings is None else timings
    for k in ("format", "d2h", "write"):
        timings.setdefault(k, 0.0)
    L = int(chunk_bytes) // unit
    chunks = plan_chunks(off, L)
    lines = max(v1 - v0 for v0, v1, _ in chunks)
    ctx = _lib.context(device.index)
    fmt = "binary_little_endian" if binary else "ascii"
    last_piece = {f: (k, a, b) for k, (_, _, ps) in enumerate(chunks) for f, a, b in ps}
    with torch.cuda.device(device):
        xf, yf, zf = (t.to(torch.float32).contiguous() for t in (x, y, z))
        rgb = colors.contiguous()
        cap = max(lines * unit, 1)
        text = torch.empty(cap, dtype=torch.uint8, device=device)
        ends = torch.empty(max(lines, 1), dtype=torch.int64, device=device)
        total = torch.empty(1, dtype=torch.int64, device=device)
        ends_at = (cap + 7) & ~7
        hosts = _pinned_pair(ends_at + 8 * max(lines, 1))
        stream = torch.cuda.current_stream(device)
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        pool = ThreadPoolExecutor(max_workers=writers or min(16, os.cpu_count() or 1))
        pending: list = []
        done: list = []

        def finish_pending():
            t0 = time.perf_counter()
            for fut in pending:
                fut.result()
            timings["write"] += time.perf_counter() - t0
            for f in done if not binary else ():               # write_ply_binary prints nothing
                print(f"  Wrote {int(off[f + 1] - off[f]):,} points to {paths[f].name}")
            pending.clear(), done.clear()

        try:
            for k, (v0, v1, pieces) in enumerate(chunks):
                m = v1 - v0
                host = hosts[k % 2]
                ev[0].record(stream)
                if binary:
                    _lib.check(ctx.lib.rb_ply_pack_binary(ctx.handle, _lib.ptr(xf) + 4 * v0, _lib.ptr(yf) + 4 * v0, _lib.ptr(zf) + 4 * v0,
                                                          _lib.ptr(rgb) + 3 * v0, m, _lib.ptr(text), _lib.stream_ptr()), "rb_ply_pack_binary")
                else:
                    _lib.check(ctx.lib.rb_ply_format_ascii(ctx.handle, _lib.ptr(xf) + 4 * v0, _lib.ptr(yf) + 4 * v0, _lib.ptr(zf) + 4 * v0,
                                                           _lib.ptr(rgb) + 3 * v0, m, _lib.ptr(text), cap, _lib.ptr(ends),
                                                           _lib.ptr(total), _lib.stream_ptr()), "rb_ply_format_ascii")
                ev[1].record(stream)
                t0 = time.perf_counter()
                if binary:
                    line_end = None
                    nbytes = unit * m
                else:
                    line_end = host[ends_at:ends_at + 8 * max(m, 1)].view(torch.int64)
                    if m:
                        line_end[:m].copy_(ends[:m], non_blocking=True)
                    stream.synchronize()
                    nbytes = int(line_end[m - 1]) if m else 0
                    line_end = line_end.numpy()
                if nbytes:
                    host[:nbytes].copy_(text[:nbytes], non_blocking=True)
                stream.synchronize()
                timings["d2h"] += time.perf_counter() - t0
                timings["format"] += ev[0].elapsed_time(ev[1]) * 1e-3
                finish_pending()                                  # the previous chunk's files, before this chunk appends
                body = host.numpy()
                for f, a, b in pieces:
                    if binary:
                        lo, hi = unit * (a - v0), unit * (b - v0)
                    else:
                        lo = int(line_end[a - v0 - 1]) if a > v0 else 0
                        hi = int(line_end[b - v0 - 1]) if b > v0 else lo
                    header = _HEADER.format(fmt=fmt, n=int(off[f + 1] - off[f])).encode("ascii") if a == off[f] else None
                    pending.append(pool.submit(_write_piece, paths[f], header, memoryview(body[lo:hi])))
                    if last_piece[f] == (k, a, b):
                        done.append(f)
            finish_pending()
        finally:
            pool.shutdown(wait=True, cancel_futures=True)
