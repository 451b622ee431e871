"""Sweep CSV files in batches: reader threads fill pinned slots, ``rb_csv_parse_sweeps`` parses a whole batch per launch.

A batch is a run of whole frames whose files, each at a 4096-byte aligned offset, fit one pinned slot (and stay under
2^31 bytes). While one batch is copied to the device and parsed, the reader threads fill the other slot with the next.
Every file ends in one of three ways, decided for that file alone:

* parsed on the device: uint8 echoes stay on the device, Angle / Scale come back as float32 (a few bytes per row);
* ``RB_CSV_LEAD_FIELDS``: echoes from the device, leading fields through pandas from the row offsets, exactly as
  ``tracker.read_sweep_csv_device`` does;
* anything else outside the device grammar, a file that cannot be read, or one larger than a slot: the drop-in's own
  per-file readers (``tracker.read_sweep_csv`` / ``read_sweep_csv_device``), which print the reference's message.
"""
from __future__ import annotations

import os
import time
from concurrent.futures import ThreadPoolExecutor
from dataclasses import dataclass
from pathlib import Path
from typing import Callable, Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import device as dev
from . import tracker as trk

CSV_CHUNK = dev.CSV_CHUNK
MAX_BATCH_BYTES = (1 << 31) - CSV_CHUNK         # the parser's offsets are int32
MIN_SLOTS = 2


def aligned(n: int) -> int:
    return (int(n) + CSV_CHUNK - 1) // CSV_CHUNK * CSV_CHUNK


# ---- host-side planning (pure functions) -----------------------------------------------------------------------------
def pack_batches(frame_sizes: Sequence[Sequence[Optional[int]]], slot_bytes: int):
    """Plan batches of whole frames for slots of ``slot_bytes``. ``frame_sizes[f][k]`` = byte size of file k of frame f
    (``None``: it cannot be read). Returns ``(batches, offsets)``: ``batches`` = list of ``(frame_a, frame_b, bytes)``
    covering every frame in order; ``offsets[f][k]`` = the file's aligned offset in its batch's slot, or -1 when the
    file takes the per-file path (unreadable, or the frame's files do not all fit one slot: those that do not are
    taken out, in order)."""
    cap = min(int(slot_bytes), MAX_BATCH_BYTES)
    batches, offsets = [], []
    fa, used = 0, 0
    for f, sizes in enumerate(frame_sizes):
        need = sum(aligned(s) for s in sizes if s is not None)
        if used and used + need > cap:                  # the frame starts a new batch
            batches.append((fa, f, used))
            fa, used = f, 0
        offs = []
        for s in sizes:
            if s is None or used + aligned(s) > cap:
                offs.append(-1)
            else:
                offs.append(used)
                used += aligned(s)
        offsets.append(offs)
    if len(frame_sizes):
        batches.append((fa, len(frame_sizes), used))
    return batches, offsets


def sweep_runs(keys: Sequence) -> List[Tuple[int, int]]:
    """``[a, b)`` ranges of consecutive equal keys (one spoke launch per ``(spokes, dtype)`` run, in sweep order)."""
    runs, a = [], 0
    for i in range(1, len(keys) + 1):
        if i == len(keys) or keys[i] != keys[a]:
            runs.append((a, i))
            a = i
    return runs


def frame_offsets(sweep_off: np.ndarray, sweeps_per_frame: Sequence[int]) -> np.ndarray:
    """Frame point offsets ``[F+1]`` from the point offsets of the sweeps in order (``sweep_off[W+1]``) and the number
    of sweeps of each frame (0 for a frame with none: it gets no points)."""
    idx = np.concatenate([[0], np.cumsum(np.asarray(sweeps_per_frame, dtype=np.int64))]).astype(np.int64)
    off = np.asarray(sweep_off, dtype=np.int64)
    if idx[-1] != len(off) - 1:
        raise ValueError("sweep counts do not add up to the sweeps")
    return off[idx]


def lead_field_value(token: str, integer_only: bool = False) -> Optional[np.float32]:
    """The device's leading-field rule in Python: ``-?D+`` or ``-?D+.D+`` (``integer_only``: ``-?D+``) with at most 15
    digits and not a negative zero; value = the digits as an exact float divided once by ``10**fraction_digits``, rounded
    to float32. ``None`` for a token outside the grammar (pandas then decides)."""
    t = token[1:] if token.startswith("-") else token
    whole, dot, frac = t.partition(".")
    if not whole.isdigit() or not whole.isascii() or (dot and (integer_only or not frac.isdigit() or not frac.isascii())):
        return None
    digits = whole + frac
    if len(digits) > 15 or (token.startswith("-") and int(digits) == 0):
        return None
    v = float(int(digits)) / float(10 ** len(frac))
    return np.float32(-v if token.startswith("-") else v)


# ---- one parsed batch ----------------------------------------------------------------------------------------------
@dataclass
class FileResult:
    """How one file ended: ``sweep`` = ``(angle f32[S], scale f32[S], echo, gain)`` as ``tracker.read_sweep_csv_device``
    returns it, or ``None`` (unreadable, empty or header only); ``status`` = the file's RB_CSV_* bits (``None``: not in a
    batch); ``rows`` = ``(a, b)`` rows of the batch's echo when the echo is a slice of it."""
    sweep: Optional[tuple]
    status: Optional[int]
    rows: Optional[Tuple[int, int]] = None


def resolve_batch(parsed: dev.CsvBatch, raw: np.ndarray, files: Sequence[Tuple[Path, int, int]], E: int) -> List[FileResult]:
    """The outcome of each file ``(path, offset, size)`` of a parsed batch; ``raw`` = the batch's host bytes."""
    out = []
    for w, (path, off, size) in enumerate(files):
        st = int(parsed.status[w])
        if st & ~dev.CSV_LEAD_FIELDS:                                # outside the echo grammar: the reference's parser
            out.append(FileResult(trk.read_sweep_csv(path, E), st))
            continue
        a, b = int(parsed.row_base[w]), int(parsed.row_base[w + 1])
        if a == b:                                                   # empty / header only: df.empty (T4:197-198)
            out.append(FileResult(None, st))
            continue
        echo = parsed.echo[a:b]
        if st & dev.CSV_LEAD_FIELDS:
            lead = trk.lead_fields_pandas(raw[off:off + size], parsed.row_start[a:b], parsed.prefix_end[a:b], b - a)
            if lead is None:
                out.append(FileResult(trk.read_sweep_csv(path, E), st))
                continue
            angle, scale, gain = lead
        else:
            angle, scale, gain = parsed.angle[a:b], parsed.scale[a:b], int(parsed.gain[w])
        out.append(FileResult((angle, scale, echo, gain), st, (a, b)))
    return out


def parse_files(paths: Sequence[Path], num_echo_columns: int, device=None) -> List[FileResult]:
    """Every file of ``paths`` in ONE batch (no slots, no threads): what a batch of :class:`SweepReader` makes of them."""
    d = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    raws = [Path(p).read_bytes() for p in paths]
    offs = np.cumsum([0] + [aligned(len(r)) for r in raws]).astype(np.int64)
    host = torch.zeros(max(int(offs[-1]), 1), dtype=torch.uint8, pin_memory=True)
    hn = host.numpy()
    for r, o in zip(raws, offs):
        hn[o:o + len(r)] = np.frombuffer(r, dtype=np.uint8)
    text = host.to(d)
    parsed = dev.csv_parse_sweeps(text[:int(offs[-1])], offs[:-1], [len(r) for r in raws], num_echo_columns)
    return resolve_batch(parsed, hn, [(Path(p), int(o), len(r)) for p, o, r in zip(paths, offs, raws)], num_echo_columns)


# ---- the reader ------------------------------------------------------------------------------------------------------
def _read_into(buf: np.ndarray, path: Path, size: int) -> bool:
    """``size`` bytes of ``path`` into ``buf``; False when the file cannot be read or no longer has that size."""
    try:
        with open(path, "rb", buffering=0) as fh:
            mv = memoryview(buf)
            n = 0
            while n < size:
                k = fh.readinto(mv[n:size])
                if not k:
                    break
                n += k
            return n == size and not fh.read(1)
    except OSError:
        return False


class SweepReader:
    """Pinned slots, reused by every call, and the batch loop of :meth:`run`. The slots are allocated by the first call
    that needs them and only ever grow: a call whose files need more than the slots hold (up to its ``batch_bytes``)
    replaces them once by slots at least twice as large, so the size a recording ends with is reached in a few steps."""

    def __init__(self, n_slots: int = MIN_SLOTS):
        self.n_slots = max(int(n_slots), MIN_SLOTS)
        self.slots: List[torch.Tensor] = []
        self.views: List[np.ndarray] = []
        self.events: List[Optional[torch.cuda.Event]] = []
        self.slot_bytes = 0

    def reserve(self, need: int, limit: int, timings: Dict[str, float]) -> None:
        """Slots of at least ``need`` bytes (``need <= limit``), grown geometrically up to ``limit``."""
        if need <= self.slot_bytes:
            return
        t0 = time.perf_counter()
        for ev in self.events:                                   # no copy may still read an old slot
            if ev is not None:
                ev.synchronize()
        new = min(limit, max(need, 2 * self.slot_bytes, 1 << 20))
        self.slots = self.views = []
        self.slots = [torch.empty(new, dtype=torch.uint8, pin_memory=True) for _ in range(self.n_slots)]
        self.views = [t.numpy() for t in self.slots]
        self.events = [None] * self.n_slots
        self.slot_bytes = new
        timings["pin"] = timings.get("pin", 0.0) + time.perf_counter() - t0

    def run(self, frames: Sequence[Sequence[Tuple[int, Path]]], E: int, device: torch.device, readers: int,
            consume: Callable[[int, int, List[List[Tuple[int, FileResult]]]], None], timings: Dict[str, float],
            batch_bytes: int) -> None:
        """Parse ``frames`` (per frame: ``(gain, path)`` in sweep order) in batches of at most ``batch_bytes``;
        ``consume(fa, fb, results)`` gets the results of frames ``[fa, fb)`` (per frame: ``(gain, FileResult)``) while
        the next batch is being read."""
        sizes = []
        for fr in frames:
            row = []
            for _, p in fr:
                try:
                    row.append(os.stat(p).st_size)
                except OSError:
                    row.append(None)
            sizes.append(row)
        limit = max(min(aligned(batch_bytes), MAX_BATCH_BYTES), CSV_CHUNK)
        total = sum(aligned(v) for row in sizes for v in row if v is not None)
        self.reserve(max(min(total, limit), CSV_CHUNK), limit, timings)
        cap = min(self.slot_bytes, limit)
        batches, offsets = pack_batches(sizes, cap)
        pool = ThreadPoolExecutor(max_workers=max(1, int(readers)), thread_name_prefix="radarb200-csv")
        try:
            def submit(k):
                s = k % len(self.slots)
                if self.events[s] is not None:
                    self.events[s].synchronize()                 # the slot's previous batch has reached the device
                fa, fb, _ = batches[k]
                return [(f, j, pool.submit(_read_into, self.views[s][offsets[f][j]:], frames[f][j][1], sizes[f][j]))
                        for f in range(fa, fb) for j in range(len(frames[f])) if offsets[f][j] >= 0]

            pending = submit(0)
            for k, (fa, fb, nbytes) in enumerate(batches):
                t0 = time.perf_counter()
                ok = {(f, j): fut.result() for f, j, fut in pending}
                t1 = time.perf_counter()
                timings["read"] = timings.get("read", 0.0) + t1 - t0
                pending = submit(k + 1) if k + 1 < len(batches) else []
                s = k % len(self.slots)
                files = [(f, j) for f in range(fa, fb) for j in range(len(frames[f])) if offsets[f][j] >= 0 and ok[(f, j)]]
                results: Dict[Tuple[int, int], FileResult] = {}
                if files:
                    t1 = time.perf_counter()
                    text = torch.empty(nbytes, dtype=torch.uint8, device=device)
                    text.copy_(self.slots[s][:nbytes], non_blocking=True)
                    ev = self.events[s] = torch.cuda.Event()
                    ev.record(torch.cuda.current_stream(device))
                    ev.synchronize()
                    t2 = time.perf_counter()
                    parsed = dev.csv_parse_sweeps(text, [offsets[f][j] for f, j in files], [sizes[f][j] for f, j in files], E)
                    t3 = time.perf_counter()
                    res = resolve_batch(parsed, self.views[s], [(frames[f][j][1], offsets[f][j], sizes[f][j]) for f, j in files], E)
                    results = dict(zip(files, res))
                    t4 = time.perf_counter()
                    timings["h2d"] = timings.get("h2d", 0.0) + t2 - t1
                    timings["parse"] = timings.get("parse", 0.0) + t3 - t2
                    timings["lead"] = timings.get("lead", 0.0) + t4 - t3
                out = []
                for f in range(fa, fb):
                    per = []
                    for j, (gain, path) in enumerate(frames[f]):
                        r = results.get((f, j))
                        if r is None:                             # unreadable or too large for a slot: the drop-in's reader
                            r = FileResult(trk.read_sweep_csv_device(path, E), None)
                        per.append((gain, r))
                    out.append(per)
                consume(fa, fb, out)
        finally:
            pool.shutdown(wait=True, cancel_futures=True)
