"""Time-sharded multi-GPU driver of the detection path (SURVEY.md section 8 e): one process per GPU, a few small
exchanges per block over NCCL (NVLink/NVSwitch) issued by ``libradarb200.so`` itself; gloo through ``torch.distributed``
in the CPU tests.

Rank r owns a contiguous block of frames. Spoke-to-point is embarrassingly parallel; the land filter
needs two tiny reductions; ST-DBSCAN couples frame f only to frames within ``eps_time``, so every rank
clusters its own frames plus a ``floor(eps_time)``-frame halo from each neighbour and the cluster ids are
stitched from the ranks' component keys. Per block (details and measurements: DESIGN.md section 6):

1. ``all_gather`` of ``[frames built, points, x/y bounds, capacity]``   -> identical ``np.arange`` edges everywhere
2. ``all_reduce(SUM)`` of the per-cell point counts / intensity sums    -> identical land mask everywhere
3. ``all_gather`` of the ranks' halo layouts (points owned, ids and per-frame counts of the boundary frames)
4. neighbour send/recv of the boundary frames' filtered points (x, y)   -> exact core flags of OWNED points
5. neighbour send/recv of those points' core flags (1 B/point)          -> exact core flags of HALO points
6. components over owned + halo cores, keyed by GLOBAL point index; ``all_gather`` of the local component keys of the
   boundary zones (run-length encoded over the zones' points: a dense zone of one component is a single entry) and of
   every rank's distinct keys; EVERY rank merges the neighbours' encodings of the same points by position
   (:func:`pair_zone_runs`), unions the keys that share a point and numbers the components by their smallest core index
   - exactly the reference's numbering (``rb_stitch_components``)
7. ``rb_relabel`` + border assignment (all neighbours of an owned point are present locally)

What the collectives carry is assembled on the device; a block reads back to the host three times, asynchronously into
pinned memory. A block is a generator that yields before each read-back, so one host thread keeps several blocks going,
each in its own block slot - CUDA stream, library context and communicator - and steps whichever block's read-back has
arrived (:meth:`ShardedDetection.run_blocks`).

The result equals the single-GPU labels of the concatenated recording, id for id.

The protocol (what is exchanged when, the halo layout, the stitching) is host logic in this file; everything that
touches data goes through an *engine*. :class:`CudaEngine` is the product: every numeric stage, the packing of what the
collectives carry AND the collectives themselves (NCCL, ``rb_comm_*``) are calls into ``libradarb200.so`` on the block's
own stream - no tensor arithmetic happens in Python. :class:`TorchEngineBase` implements the same bookkeeping and
collectives with plain torch ops over ``torch.distributed``; the CPU tests derive an oracle-backed engine from it and
drive this file's protocol over gloo.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Optional, Sequence, Tuple

import numpy as np
import torch
import torch.distributed as dist

from . import tracker as trk
from ._lib import RadarB200Error
from .device import PointBatch


# ------------------------------------------------------------------------------------------ stitching (host)
def stitch_components(seg_keys: Sequence[Sequence[np.ndarray]], keys: Sequence[np.ndarray]
                      ) -> Tuple[np.ndarray, np.ndarray, int]:
    """Global cluster numbering from the ranks' local components.

    ``keys[r]``: the distinct local component keys of rank r (key = smallest global core index the rank
    saw in that component). ``seg_keys[r]`` = four arrays with the local key of every CORE point of rank r's
    boundary zones, each in point order: ``[left halo, own first frames, own last frames, right halo]``.
    Rank r's "own last frames" and rank r+1's "left halo" are the same points with the same core flags, in
    the same order (likewise "right halo" / "own first frames"), so the two key arrays pair up position by
    position: each pair ties two local components together. Returns ``(table_keys sorted, table_ids,
    n_clusters)`` where the id of a component is the rank of its smallest global core index among all
    components — the reference's numbering (SURVEY.md N4)."""
    import ctypes as C

    from . import _lib

    lib = _lib.load()
    i64 = lambda parts: np.ascontiguousarray(np.concatenate([np.asarray(k, dtype=np.int64).ravel() for k in parts] + [np.zeros(0, np.int64)]))
    all_keys = i64(keys)
    pa, pb = [], []
    for r in range(len(seg_keys) - 1):
        for mine, theirs in ((seg_keys[r][2], seg_keys[r + 1][0]), (seg_keys[r][3], seg_keys[r + 1][1])):
            if len(mine) != len(theirs):
                raise RadarB200Error("stitch: boundary zones of neighbouring ranks do not match")
            pa.append(mine); pb.append(theirs)
    pa, pb = i64(pa), i64(pb)
    table_keys = np.empty(max(len(all_keys), 1), dtype=np.int64)
    table_ids = np.empty(max(len(all_keys), 1), dtype=np.int32)
    ncl = C.c_int64(0)
    ptr = lambda a: a.ctypes.data_as(C.c_void_p)
    m = lib.rb_stitch_components(ptr(all_keys), len(all_keys), ptr(pa), ptr(pb), len(pa), ptr(table_keys), ptr(table_ids),
                                 len(table_keys), C.byref(ncl))
    if m < 0:
        raise RadarB200Error(f"rb_stitch_components: {lib.rb_last_error().decode()}")
    return table_keys[:m], table_ids[:m], int(ncl.value)


def pair_zone_runs(keys_a: np.ndarray, starts_a: np.ndarray, keys_b: np.ndarray, starts_b: np.ndarray
                   ) -> Tuple[np.ndarray, np.ndarray]:
    """Two ranks hold the SAME boundary points (rank r's own last frames = rank r+1's left halo, ...) with the same core
    flags, each under its own component keys, and ship them run-length encoded: ``keys[j]`` holds from position
    ``starts[j]`` of the zone to the next start (-1 = not a core point). Returns the distinct ``(key_a, key_b)`` pairs under
    which one core point is known to the two ranks - what ties their local components together. The cost follows the
    number of RUNS, not of points: a dense boundary zone of millions of core points of one component is a single run."""
    e = np.zeros(0, np.int64)
    if len(keys_a) == 0 or len(keys_b) == 0:
        if len(keys_a) != len(keys_b):
            raise RadarB200Error("stitch: boundary zones of neighbouring ranks do not match")
        return e, e
    cuts = np.union1d(starts_a, starts_b)
    ka = keys_a[np.searchsorted(starts_a, cuts, side="right") - 1]
    kb = keys_b[np.searchsorted(starts_b, cuts, side="right") - 1]
    core = ka >= 0
    if not np.array_equal(core, kb >= 0):
        raise RadarB200Error("stitch: neighbouring ranks disagree on the core points of a boundary zone")
    if not core.any():
        return e, e
    pairs = np.unique(np.stack([ka[core], kb[core]], axis=1), axis=0)
    return np.ascontiguousarray(pairs[:, 0]), np.ascontiguousarray(pairs[:, 1])


# ------------------------------------------------------------------------------------------ engines
class TorchEngineBase:
    """Bookkeeping and collectives of the protocol with torch ops over ``torch.distributed`` (any backend, any device).
    The CPU test engine derives from this (numeric stages from the oracle, gloo underneath); :class:`CudaEngine`
    overrides every method with library calls."""

    #: collectives of all blocks share the backend's one stream: issue them only after the block's GPU work is done
    wait_before_collective = True
    rank, world, group = 0, 1, None

    def attach(self, rank: int, world: int, group) -> None:
        self.rank, self.world, self.group = rank, world, group

    def prepare_slots(self, n_slots: int, slot_ctx) -> None:
        """Called (collectively) before blocks run in ``n_slots`` block slots."""

    def upload(self, arr, dtype=None) -> torch.Tensor:
        t = torch.from_numpy(np.ascontiguousarray(arr))
        if dtype is not None and t.dtype != dtype:
            t = t.to(dtype)
        return t.to(self.device)

    # -- what the collectives carry
    def pack_stats(self, raw_off_d, b4_d, cap: int) -> torch.Tensor:
        f64 = torch.float64
        return torch.cat([torch.count_nonzero(torch.diff(raw_off_d))[None].to(f64), raw_off_d[-1:].to(f64), b4_d.to(f64),
                          self.upload(np.array([cap], dtype=np.float64))])

    def pack_layout(self, off_d, ids: np.ndarray, F: int, hh: int) -> torch.Tensor:
        ids_d, per = self.upload(ids), torch.diff(off_d)
        return torch.cat([off_d[F:F + 1], off_d[F - hh:F - hh + 1], ids_d[:hh], per[:hh], ids_d[F - hh:], per[F - hh:]])

    def pack_keys(self, key, gidx, zones, n_loc: int, cap_k: int) -> torch.Tensor:
        """``[5 running entry counts | 4 zone lengths | keys[cap_k] | starts[cap_k]]`` (int64): the component keys of the
        four boundary zones RUN-LENGTH ENCODED over all their points (an entry = a key and the position in the zone where
        it starts to hold; -1 = not a core point), then the rank's distinct component keys (the points that are their
        component's smallest core). Entries beyond ``cap_k`` are dropped; the counts stay true."""
        buf = torch.zeros(9 + 2 * cap_k, dtype=torch.int64, device=self.device)
        if n_loc == 0:
            return buf
        ent_k, ent_s = [], []
        for a, b in zones:
            k = key[a:b]
            if b > a:
                flag = torch.ones(b - a, dtype=torch.bool, device=self.device)
                flag[1:] = k[1:] != k[:-1]
                idx = torch.nonzero(flag)[:, 0]
            else:
                idx = torch.zeros(0, dtype=torch.int64, device=self.device)
            ent_k.append(k[idx]); ent_s.append(idx)
        roots = key[key == gidx]
        ent_k.append(roots); ent_s.append(torch.zeros_like(roots))
        lens = np.array([len(t) for t in ent_k], dtype=np.int64)
        buf[:5] = self.upload(np.cumsum(lens))
        buf[5:9] = self.upload(np.array([b - a for a, b in zones], dtype=np.int64))
        allk, alls = torch.cat(ent_k)[:cap_k], torch.cat(ent_s)[:cap_k]
        buf[9:9 + len(allk)] = allk
        buf[9 + cap_k:9 + cap_k + len(alls)] = alls
        return buf

    # -- collectives
    def all_gather(self, mine: torch.Tensor) -> torch.Tensor:
        """One fixed-length device vector per rank -> ``[world, len]`` (no sync; the caller yields before reading it)."""
        if self.world == 1:
            return mine[None]
        out = torch.empty((self.world, mine.numel()), dtype=mine.dtype, device=self.device)
        dist.all_gather_into_tensor(out, mine.contiguous()[None], group=self.group)
        return out

    def all_reduce_grids(self, count, isum):
        if self.world == 1:
            return count, isum
        grids = torch.stack([count.to(torch.float64), isum])            # counts < 2^53 stay exact
        dist.all_reduce(grids, op=dist.ReduceOp.SUM, group=self.group)
        return grids[0].to(torch.int32), grids[1].contiguous()

    def exchange(self, to_left, to_right, from_left, from_right) -> None:
        """Lists of 1-D tensors: part k of ``to_left`` goes to rank - 1, of ``to_right`` to rank + 1; ``from_*`` are
        preallocated views that receive the neighbours' parts (empty tensors are skipped)."""
        ops, keep = [], []
        if self.rank > 0:
            for t in to_left:
                if t.numel():
                    keep.append(t.contiguous()); ops.append(dist.P2POp(dist.isend, keep[-1], self.rank - 1, group=self.group))
            for t in from_left:
                if t.numel():
                    tmp = torch.empty_like(t); keep.append((t, tmp)); ops.append(dist.P2POp(dist.irecv, tmp, self.rank - 1, group=self.group))
        if self.rank < self.world - 1:
            for t in to_right:
                if t.numel():
                    keep.append(t.contiguous()); ops.append(dist.P2POp(dist.isend, keep[-1], self.rank + 1, group=self.group))
            for t in from_right:
                if t.numel():
                    tmp = torch.empty_like(t); keep.append((t, tmp)); ops.append(dist.P2POp(dist.irecv, tmp, self.rank + 1, group=self.group))
        if ops:
            for req in dist.batch_isend_irecv(ops):
                req.wait()
        for item in keep:
            if isinstance(item, tuple):
                item[0].copy_(item[1])

    # -- the local problem [left halo | owned | right halo]
    def local_problem(self, pts: PointBatch, n_own: int, lo_end: int, hi_start: int, nl: int, nr: int, head: np.ndarray,
                      all_ids: np.ndarray, lbase: int, gbase: int, rbase: int):
        n_loc = nl + n_own + nr
        X = torch.empty(n_loc, dtype=torch.float32, device=self.device)
        Y = torch.empty(n_loc, dtype=torch.float32, device=self.device)
        X[nl:nl + n_own].copy_(pts.x[:n_own])
        Y[nl:nl + n_own].copy_(pts.y[:n_own])
        self.exchange([pts.x[:lo_end], pts.y[:lo_end]], [pts.x[hi_start:n_own], pts.y[hi_start:n_own]],
                      [X[:nl], Y[:nl]], [X[nl + n_own:], Y[nl + n_own:]])
        times, gidx = self.local_index(head, all_ids, nl, n_own, nr, lbase, gbase, rbase)
        return X, Y, times, gidx

    def local_index(self, head, all_ids, nl, n_own, nr, lbase, gbase, rbase):
        n_loc = nl + n_own + nr
        if n_loc == 0:
            return (torch.zeros(0, dtype=torch.float32, device=self.device), torch.zeros(0, dtype=torch.int64, device=self.device))
        times = self.expand_frame_times(self.upload(head), self.upload(all_ids.astype(np.float32)), n_loc)
        gidx = torch.arange(n_loc, dtype=torch.int64, device=self.device)
        gidx[:nl] += lbase
        gidx[nl:nl + n_own] += gbase - nl
        gidx[nl + n_own:] += rbase - nl - n_own
        return times, gidx

    def exchange_cores(self, core, nl: int, n_own: int, nr: int, lo_end: int, hi_start: int) -> None:
        """Halo points take their OWNER's core flags (in place)."""
        own = core[nl:nl + n_own]
        self.exchange([own[:lo_end]], [own[hi_start:]], [core[:nl]], [core[nl + n_own:]])


class CudaEngine(TorchEngineBase):
    """The product engine: numeric stages, packing and collectives through ``libradarb200.so`` on the current CUDA device
    and stream (torch allocates the buffers and provides the stream, nothing else)."""

    wait_before_collective = False          # every block slot has its own communicator and issues on its own stream

    def __init__(self, device_index: Optional[int] = None):
        from . import device as dev

        if not torch.cuda.is_available():
            raise RadarB200Error("no CUDA device: the sharded detection path is GPU only (no CPU fallback)")
        self.dev = dev
        self.device = torch.device("cuda", torch.cuda.current_device() if device_index is None else device_index)
        self._comm_slots = set()

    # -- communicators: one per block slot (library context), created collectively
    def prepare_slots(self, n_slots: int, slot_ctx) -> None:
        import ctypes as C

        from . import _lib

        if self.world == 1:
            return
        for k in range(n_slots):
            if k in self._comm_slots:
                continue
            with slot_ctx(k):
                ctx = _lib.context(self.device.index)
                uid = torch.zeros(128, dtype=torch.uint8)
                if self.rank == 0:
                    buf = (C.c_uint8 * 128)()
                    _lib.check(ctx.lib.rb_comm_unique_id(buf), "rb_comm_unique_id")
                    uid = torch.tensor(list(buf), dtype=torch.uint8)
                if dist.get_backend(self.group) == "nccl":
                    uid = uid.to(self.device)
                dist.broadcast(uid, src=0, group=self.group)         # bootstrap only: the id travels over the caller's group
                raw = bytes(uid.cpu().tolist())
                _lib.check(ctx.lib.rb_comm_init(ctx.handle, raw, self.rank, self.world), "rb_comm_init")
                # one round of every kind of operation, in the same order on all ranks: NCCL sets up its connections
                # (neighbour send/recv channels above all) on first use, and later the slots run unordered
                t = torch.zeros(16, dtype=torch.uint8, device=self.device)
                r = torch.zeros(16, dtype=torch.uint8, device=self.device)
                self.exchange([t[:4]], [t[4:8]], [r[:4]], [r[4:8]])
                self.all_gather(t)
                self.all_reduce_grids(torch.zeros(4, dtype=torch.int32, device=self.device), torch.zeros(4, dtype=torch.float64, device=self.device))
                torch.cuda.current_stream(self.device).synchronize()
            self._comm_slots.add(k)

    def _ctx(self):
        from . import _lib
        return _lib.context(self.device.index)

    def upload(self, arr, dtype=None) -> torch.Tensor:
        """Host array -> device tensor WITHOUT a stream sync: staged in pinned memory (torch's caching host allocator
        recycles the block only after the copy has run) and copied asynchronously."""
        t = torch.from_numpy(np.ascontiguousarray(arr))
        if dtype is not None and t.dtype != dtype:
            t = t.to(dtype)
        pinned = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
        pinned.copy_(t)
        return pinned.to(self.device, non_blocking=True)

    def spoke_to_points(self, echo, cos_tab, sin_tab, range_res, sweep_gain, thr, stride, gpf, cap=None) -> PointBatch:
        return self.dev.spoke_to_points(echo, cos_tab, sin_tab, range_res, sweep_gain, thr, stride, gains_per_frame=gpf, cap=cap)

    # -- the spoke stage, frame offsets and bounds enqueued together WITHOUT a sync: the caller reads the count, the
    #    offsets and the bounds back later (with its first collective), and repeats the launch if ``cap`` was too small
    def spoke_launch(self, echo, cos_tab, sin_tab, range_res, sweep_gain, thr, stride, gpf, cap):
        W = echo.shape[0]
        out = (torch.empty(cap, dtype=torch.float32, device=self.device), torch.empty(cap, dtype=torch.float32, device=self.device),
               torch.empty(cap, dtype=torch.float32, device=self.device), torch.empty(cap, dtype=torch.int32, device=self.device),
               torch.empty(W + 1, dtype=torch.int64, device=self.device))
        self.dev.spoke_to_points_raw(echo, cos_tab, sin_tab, range_res, sweep_gain, thr, stride, cap, out=out)
        off = self.dev.frame_offsets(out[4], W // gpf, gpf)
        b4 = self.dev.bounds_counted(out[0], out[1], out[4][W:])
        return dict(outs=out, off=off, b4=b4)

    def bounds(self, x, y) -> torch.Tensor:
        return self.dev.bounds(x, y)

    def _edges(self, xe: np.ndarray, ye: np.ndarray):
        from . import _lib

        key = (xe.tobytes(), ye.tobytes())
        cache = self.__dict__.setdefault("_edge_cache", {})       # one upload per distinct grid and block slot (stream)
        hit = cache.get(_lib.get_slot())
        if hit is None or hit[0] != key:
            both = self.upload(np.concatenate([xe, ye]))
            hit = cache[_lib.get_slot()] = (key, (both[:len(xe)], both[len(xe):]))
        return hit[1]

    def land_accumulate(self, batch: PointBatch, xe: np.ndarray, ye: np.ndarray):
        d_xe, d_ye = self._edges(xe, ye)
        n = batch.n
        if n == 0:
            return (torch.zeros((len(xe) - 1, len(ye) - 1), dtype=torch.int32, device=self.device),
                    torch.zeros((len(xe) - 1, len(ye) - 1), dtype=torch.float64, device=self.device))
        return self.dev.land_accumulate(batch.x[:n], batch.y[:n], batch.inten[:n], d_xe, d_ye, check=False)

    def land_flag(self):
        """Device int32[1]: a non-integer intensity was seen by land_accumulate (read with the block's next read-back)."""
        return self.dev.land_accumulate_flag(self.device.index)

    def land_cells(self, count, isum, built, persistence, min_intensity):
        return self.dev.land_cells(count, isum, built, persistence, min_intensity)

    def land_filter(self, batch: PointBatch, xe, ye, land) -> PointBatch:
        """Enqueues the filter; the point count of the result is read later (``n`` = -1 until then)."""
        d_xe, d_ye = self._edges(xe, ye)
        return self.dev.land_filter(batch, d_xe, d_ye, land, sync=False)

    def expand_frame_times(self, frame_off, frame_ids, n):
        return self.dev.expand_frame_times(frame_off, frame_ids, n)

    def phases(self, x, y, times, eps_space, eps_time, min_samples, hint=None):
        return self.dev.StDbscanPhases(x, y, None, times, eps_space, eps_time, min_samples, stride=1, n=times.numel(), hint=hint)

    def relabel(self, keys, table_keys, table_ids):
        return self.dev.relabel(keys, table_keys, table_ids)

    # -- packing and collectives: library calls (kernels of csrc/shard.cu, NCCL through csrc/comm.cu)
    def pack_stats(self, raw_off_d, b4_d, cap: int) -> torch.Tensor:
        from ._lib import check, ptr, stream_ptr
        ctx = self._ctx()
        out = torch.empty(7, dtype=torch.float64, device=self.device)
        check(ctx.lib.rb_shard_pack_stats(ctx.handle, ptr(raw_off_d), raw_off_d.numel() - 1, ptr(b4_d), int(cap), ptr(out), stream_ptr()),
              "rb_shard_pack_stats")
        return out

    def pack_layout(self, off_d, ids: np.ndarray, F: int, hh: int) -> torch.Tensor:
        from ._lib import check, ptr, stream_ptr
        ctx = self._ctx()
        out = torch.empty(2 + 4 * hh, dtype=torch.int64, device=self.device)
        ids64 = np.ascontiguousarray(ids, dtype=np.int64)
        check(ctx.lib.rb_shard_pack_layout(ctx.handle, ptr(off_d), int(F), ids64.ctypes.data, int(hh), ptr(out), stream_ptr()),
              "rb_shard_pack_layout")
        return out

    def pack_keys(self, key, gidx, zones, n_loc: int, cap_k: int) -> torch.Tensor:
        from ._lib import check, ptr, stream_ptr
        ctx = self._ctx()
        vec = torch.empty(9 + 2 * cap_k, dtype=torch.int64, device=self.device)
        z = np.ascontiguousarray(np.array(zones, dtype=np.int64).reshape(-1))
        check(ctx.lib.rb_shard_pack_keys(ctx.handle, ptr(key) if n_loc else None, ptr(gidx) if n_loc else None, int(n_loc), z.ctypes.data,
                                         int(cap_k), ptr(vec), stream_ptr()), "rb_shard_pack_keys")
        return vec

    def all_gather(self, mine: torch.Tensor) -> torch.Tensor:
        from ._lib import check, ptr, stream_ptr
        if self.world == 1:
            return mine[None]
        ctx = self._ctx()
        mine = mine.contiguous()
        out = torch.empty((self.world, mine.numel()), dtype=mine.dtype, device=self.device)
        check(ctx.lib.rb_comm_all_gather(ctx.handle, ptr(mine), ptr(out), mine.numel() * mine.element_size(), stream_ptr()),
              "rb_comm_all_gather")
        return out

    def all_reduce_grids(self, count, isum):
        from ._lib import check, ptr, stream_ptr
        if self.world == 1:
            return count, isum
        ctx = self._ctx()
        check(ctx.lib.rb_comm_all_reduce_grids(ctx.handle, ptr(count), ptr(isum), count.numel(), stream_ptr()), "rb_comm_all_reduce_grids")
        return count, isum

    def exchange(self, to_left, to_right, from_left, from_right) -> None:
        import ctypes as C

        from ._lib import check, stream_ptr
        if self.world == 1:
            return
        k = len(to_left)
        assert len(to_right) == k and len(from_left) == k and len(from_right) == k
        ctx = self._ctx()
        vp, i64 = C.c_void_p * k, C.c_int64 * k
        nbytes = lambda ts: i64(*[t.numel() * t.element_size() for t in ts])
        ptrs = lambda ts: vp(*[t.data_ptr() if t.numel() else None for t in ts])
        check(ctx.lib.rb_comm_exchange(ctx.handle, k, ptrs(to_left), nbytes(to_left), ptrs(to_right), nbytes(to_right), ptrs(from_left),
                                       nbytes(from_left), ptrs(from_right), nbytes(from_right), stream_ptr()), "rb_comm_exchange")

    def local_index(self, head, all_ids, nl, n_own, nr, lbase, gbase, rbase):
        from ._lib import check, ptr, stream_ptr
        n_loc = nl + n_own + nr
        times = torch.empty(max(n_loc, 1), dtype=torch.float32, device=self.device)[:n_loc]
        gidx = torch.empty(max(n_loc, 1), dtype=torch.int64, device=self.device)[:n_loc]
        if n_loc:
            ctx = self._ctx()
            h = np.ascontiguousarray(head, dtype=np.int64)
            ids = np.ascontiguousarray(all_ids, dtype=np.float32)
            check(ctx.lib.rb_shard_local_index(ctx.handle, h.ctypes.data, ids.ctypes.data, len(ids), int(nl), int(n_own), int(nr), int(lbase),
                                               int(gbase), int(rbase), ptr(times), ptr(gidx), stream_ptr()), "rb_shard_local_index")
        return times, gidx


# a block that has just enqueued its spoke stage (~2 ms of GPU time for 512 frames) sits out this many scheduler
# rounds: a constant, so the schedule stays identical on every rank
SPOKE_SKIP = 5


# ------------------------------------------------------------------------------------------ result
@dataclass
class ShardResult:
    """Result for the frames owned by this rank (same fields the single-GPU ``DetectionResult`` has)."""
    frame_ids: np.ndarray
    raw: PointBatch
    points: PointBatch
    labels: torch.Tensor
    n_clusters: int                        # GLOBAL number of clusters
    halo_points: Tuple[int, int] = (0, 0)  # points received from the left / right neighbour
    land: Optional[torch.Tensor] = None
    edges: Optional[Tuple[np.ndarray, np.ndarray]] = None

    def to_host(self) -> dict:
        n, p = self.points.n, self.points
        packed = torch.stack([p.x[:n], p.y[:n], p.inten[:n]], dim=1)
        from .device import to_pinned_host
        points, gains, frame_off, labels = to_pinned_host(packed, p.gain[:n], p.frame_off, self.labels[:n])
        return dict(points=points, gains=gains, frame_off=frame_off, labels=labels, frame_ids=self.frame_ids)


# ------------------------------------------------------------------------------------------ driver
class ShardedDetection:
    """Runs the hot path for this rank's block of frames, exchanging what the stages need with the
    other ranks. ``engine`` defaults to :class:`CudaEngine`; ``group`` to the default process group."""

    def __init__(self, config=None, rank: Optional[int] = None, world: Optional[int] = None,
                 device: Optional[int] = None, engine=None, group=None):
        from .pipeline import DetectionConfig

        self.cfg = config or DetectionConfig()
        if self.cfg.min_frames is not None:
            raise RadarB200Error("ShardedDetection does not run the min_frames variant: use RecordingDetection on one GPU")
        self.group = group
        self.rank = dist.get_rank(group) if rank is None else rank
        self.world = dist.get_world_size(group) if world is None else world
        self.engine = engine or CudaEngine(device)
        self.engine.attach(self.rank, self.world, group)
        self.device = self.engine.device
        self.base = None
        if engine is None:
            from .pipeline import DetectionPipeline
            self.base = DetectionPipeline(self.cfg, self.device.index)       # spoke tables + ctx for the bench
        self._cap_hint = 0
        self._gain_cache = None
        self._streams = []                 # one CUDA stream per block slot (run_blocks)
        self._key_cap = 8192               # capacity of the component-key vector (grows on demand)
        self.profile = False               # True: synchronise and record wall-clock per stage in self.timings
        self.timings = {}
        self._t_last = None

    def _tick(self, name: Optional[str]) -> None:
        """Stage timer (diagnostics): time since the previous tick is booked under ``name``."""
        if not self.profile:
            return
        import time
        if self.device.type == "cuda":
            torch.cuda.synchronize(self.device)
        now = time.perf_counter()
        if name is not None and self._t_last is not None:
            self.timings[name] = self.timings.get(name, 0.0) + (now - self._t_last)
        self._t_last = now

    def _pause(self, skip: int = 0, *tensors):
        """What a block's generator yields before it needs the host: ``(event, skip, host tensors)``. The device->host
        copies of ``tensors`` go into pinned memory and the event marks their completion on the block's stream; the
        scheduler resumes the block once the event has fired (``skip``: rounds to sit out first in ordered mode)."""
        if self.device.type != "cuda":
            return None, skip, [t for t in tensors]
        host = []
        for t in tensors:
            h = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
            h.copy_(t, non_blocking=True)
            host.append(h)
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(self.device))
        return ev, skip, host

    # ---- the path -------------------------------------------------------------------------------------
    # The path of one block is a GENERATOR that yields right before every host read-back. Driven alone
    # (run_device) it is a plain sequential pass. run_blocks drives several of them round-robin in ONE host
    # thread: while a block waits for the GPU, the other blocks' next phases are enqueued, so kernels,
    # collectives and host work of different blocks overlap. Every rank follows the same deterministic schedule
    # (the yields and the collectives of a block do not depend on local data), so the collectives of every
    # communicator are issued in the same order everywhere.
    def _gains(self, n_sweeps: int) -> torch.Tensor:
        if self._gain_cache is None or self._gain_cache.numel() != n_sweeps:
            self._gain_cache = self.engine.upload(np.array(list(self.cfg.gains) * (n_sweeps // len(self.cfg.gains)), dtype=np.int32))
        return self._gain_cache

    def _slot(self, k: int):
        """Context of block slot ``k``: its own CUDA stream and library context (scratch, ST-DBSCAN plan, communicator)."""
        import contextlib
        from . import _lib

        if self.device.type != "cuda":
            return contextlib.nullcontext()
        while len(self._streams) <= k:
            self._streams.append(torch.cuda.Stream(self.device))

        @contextlib.contextmanager
        def ctx():
            prev = _lib.set_slot(k)
            try:
                with torch.cuda.stream(self._streams[k]):
                    yield
            finally:
                _lib.set_slot(prev)
        return ctx()

    def run_blocks(self, blocks, keep: bool = True, in_flight: int = 2, ordered: Optional[bool] = None, make_gen=None):
        """Run a sequence of blocks ``(echo, cos_tab, sin_tab, range_res, frame_ids)`` of this rank with up to
        ``in_flight`` of them interleaved (see above). Same results as :meth:`run_device` per block. Returns the
        results in order (``keep=False``: only the last one; earlier ones are released for buffer reuse).

        ``ordered`` (default: what the engine needs): True = the blocks are stepped round-robin and the host WAITS for
        each block's pending read-back in turn - every rank issues all collectives in one global order, which engines
        whose collectives share a communicator need. False = a block is stepped as soon as ITS read-back has arrived
        (event query), whatever the others do: no head-of-line blocking of the one host thread. The order of a
        communicator's collectives is still the block's program order; only the interleaving BETWEEN the slots'
        communicators then differs from rank to rank, which is safe because their kernels can run side by side."""
        import os

        blocks = list(blocks)
        results = [None] * len(blocks)
        if ordered is None:
            ordered = bool(self.engine.wait_before_collective) or os.environ.get("RB_SHARD_ORDERED", "0") == "1"
        active = []                                           # [index, generator, slot, rounds to skip, pending event]
        free = list(range(max(1, in_flight)))[::-1]
        self.engine.prepare_slots(max(1, in_flight), self._slot)
        nxt = 0
        main = torch.cuda.current_stream(self.device) if self.device.type == "cuda" else None
        while active or nxt < len(blocks):
            while free and nxt < len(blocks):                 # start blocks while there is a free slot
                k = free.pop()
                if main is not None:
                    with self._slot(k):
                        torch.cuda.current_stream(self.device).wait_stream(main)
                active.append([nxt, (make_gen or self._run_gen)(*blocks[nxt]), k, 0, None])
                nxt += 1
            progressed = False
            for entry in list(active):                         # one step of every active block that can take one
                i, gen, k, _, ev = entry
                if ordered:
                    if entry[3] > 0 and len(active) > 1:       # it asked to be left alone for a few rounds (its GPU
                        entry[3] -= 1                          # phase is long): the others' steps fill the time
                        continue
                    if ev is not None:
                        ev.synchronize()
                elif ev is not None and not ev.query():
                    continue                                   # its read-back has not arrived yet: somebody else's turn
                progressed = True
                with self._slot(k):
                    try:
                        entry[4], entry[3], _ = next(gen)
                        continue
                    except StopIteration as fin:
                        res = fin.value
                    if main is not None:
                        done = torch.cuda.Event()
                        done.record(torch.cuda.current_stream(self.device))
                        main.wait_event(done)
                active.remove(entry)
                free.append(k)
                if keep or i == len(blocks) - 1:
                    results[i] = res
                del res
            if not ordered and not progressed and active:      # nothing was ready: poll until some block's read-back arrives
                pend = [e[4] for e in active if e[4] is not None]
                spins = 0
                while pend and not any(ev.query() for ev in pend):
                    spins += 1
                    if spins > 20000:                          # (a long GPU phase: stop burning the core, sleep on the oldest)
                        pend[0].synchronize()
                        break
        return [r for r in results if r is not None]

    def run_device(self, echo, cos_tab, sin_tab, range_res, frame_ids: Sequence[int], cluster: bool = True) -> ShardResult:
        """``echo[F,G,S,E]`` = this rank's frames (device tensor of the engine); ``frame_ids`` their ids,
        increasing across ranks (rank r's ids are all smaller than rank r+1's)."""
        from . import _lib

        slot = _lib.get_slot() if self.device.type == "cuda" else 0
        self.engine.prepare_slots(slot + 1, self._slot)
        gen = self._run_gen(echo, cos_tab, sin_tab, range_res, frame_ids, cluster)
        while True:
            try:
                ev, _, _ = next(gen)
                if ev is not None:
                    ev.synchronize()
            except StopIteration as fin:
                return fin.value

    def _run_gen(self, echo, cos_tab, sin_tab, range_res, frame_ids: Sequence[int], cluster: bool = True):
        """One block = three host read-backs (A: point count + every rank's statistics, B: filtered offsets + every
        rank's halo layout, C: every rank's component keys), each preceded by a ``yield``. What the collectives carry
        is assembled ON THE DEVICE by the engine, so nothing between two read-backs waits for the GPU (an engine whose
        collectives share one stream waits for its long GPU phases before it issues them, see ``wait_before_collective``)."""
        cfg, eng = self.cfg, self.engine
        F, G, S, E = echo.shape
        ids = np.asarray(frame_ids, dtype=np.int64)
        sweeps = echo.reshape(F * G, S, E)
        launch = getattr(eng, "spoke_launch", None)
        self._tick(None)
        while True:
            if launch is not None:
                cap = self._cap_hint or max(1, F * G * ((S * E + cfg.point_stride - 1) // max(cfg.point_stride, 1)) // 8)
                h = launch(sweeps, cos_tab, sin_tab, range_res, self._gains(F * G), cfg.intensity_threshold, cfg.point_stride, G, cap)
                outs, raw_off_d, b4_d = h["outs"][:4], h["off"], h["b4"]
            else:                                              # an engine without the split launch (CPU test engine)
                r = eng.spoke_to_points(sweeps, cos_tab, sin_tab, range_res, self._gains(F * G), cfg.intensity_threshold,
                                        cfg.point_stride, G, cap=None)
                cap, outs, raw_off_d = r.n, (r.x, r.y, r.inten, r.gain), r.frame_off
                b4_d = eng.bounds(r.x[:r.n], r.y[:r.n]) if r.n > 0 else torch.zeros(4, dtype=torch.float32, device=self.device)
            if eng.wait_before_collective:
                # The spoke stage is the long GPU phase of a block. With ONE stream for all blocks' collectives, a
                # collective queued behind unfinished work holds up every other block's collectives behind it.
                yield self._pause(SPOKE_SKIP if launch is not None else 0)
            # collective 1: [frames built, points, xmin, xmax, ymin, ymax, capacity] of every rank (exact in float64)
            g_stats = eng.all_gather(eng.pack_stats(raw_off_d, b4_d, cap))
            pause = self._pause(SPOKE_SKIP if (launch is not None and not eng.wait_before_collective) else 0, g_stats, raw_off_d)
            yield pause
            allv, raw_off = (t.numpy() for t in pause[2])      # read-back A
            if (allv[:, 1] <= allv[:, 6]).all():
                break
            # some rank's capacity guess was too small (its points were cut): everybody repeats - all see the same numbers
            self._cap_hint = int(allv[self.rank, 1] * 1.25) + 1024
        raw_off = raw_off.astype(np.int64)
        raw = PointBatch(*outs, raw_off_d, int(raw_off[-1]))
        self._cap_hint = max(self._cap_hint, int(raw.n * 1.25) + 1024)
        self._tick("spoke+stats")

        # ---- land / stationary persistence filter over ALL ranks' frames --------------------------
        pts, land, edges, b4, inexact_d = raw, None, None, None, None
        built, n_all = int(allv[:, 0].sum()), int(allv[:, 1].sum())
        if cfg.land_filter and n_all > 0 and built > cfg.land_min_frames:
            have = allv[allv[:, 1] > 0]
            b4 = np.array([have[:, 2].min(), have[:, 3].max(), have[:, 4].min(), have[:, 5].max()], dtype=np.float32)
            xe, ye = trk.grid_edges_from_bounds(b4, cfg.land_resolution)
            count, isum = eng.land_accumulate(raw, xe, ye)
            inexact_d = eng.land_flag() if hasattr(eng, "land_flag") else None
            # collective 2: counts and intensity sums of all ranks (sums of integers: exact in any order)
            count, isum = eng.all_reduce_grids(count, isum)
            land = eng.land_cells(count, isum, built, cfg.land_persistence, cfg.land_min_intensity)
            if raw.n > 0:
                pts = eng.land_filter(raw, xe, ye, land)       # enqueued; its point count comes with read-back B
            edges = (xe, ye)
        off_d = pts.frame_off

        # collective 3: per rank [points owned, start of the last-hh-frames zone, ids and per-frame counts of the first
        # hh and last hh frames] -> global index bases and both neighbours' halo layouts at once
        h_t = int(math.floor(cfg.eps_time)) if cfg.eps_time >= 0 else 0
        if cluster and self.world > 1 and h_t > F:
            raise RadarB200Error(f"time shard of {F} frames is shorter than the eps_time halo ({h_t} frames)")
        hh = min(h_t, F)
        g_meta = eng.all_gather(eng.pack_layout(off_d, ids, F, hh)) if cluster else None
        pause = self._pause(0, off_d, *([g_meta] if cluster else []), *([inexact_d] if inexact_d is not None else []))
        yield pause
        back = [t.numpy() for t in pause[2]]                   # read-back B
        off = back[0].astype(np.int64)
        meta = back[1] if cluster else None
        if inexact_d is not None and int(back[-1][0]):
            # the per-cell float64 sums of non-integer intensities depend on the order of addition; across ranks the
            # reference's order (all points of all frames, one after the other) cannot be reproduced by a sum of partial sums
            raise RadarB200Error("time-sharded land filter: intensities must be integer valued (radar echoes are 0..255); "
                                 "use the single-GPU path for other data")
        pts.n = int(off[-1])
        self._tick("land+layout")
        labels = torch.empty(0, dtype=torch.int32, device=self.device)
        n_clusters, halo = 0, (0, 0)
        if cluster:
            labels, n_clusters, halo = yield from self._cluster_gen(pts, ids, off, meta, hh, b4)
        return ShardResult(ids, raw, pts, labels, n_clusters, halo, land, edges)

    def _cluster_gen(self, pts: PointBatch, ids: np.ndarray, off: np.ndarray, meta: np.ndarray, hh: int, b4):
        cfg, eng = self.cfg, self.engine
        F = len(ids)
        n_own = pts.n
        lo_end, hi_start = int(off[hh]), int(off[F - hh])          # owned points [0, lo_end) go left, [hi_start, n) right
        bases = np.concatenate([[0], np.cumsum(meta[:, 0])])
        gbase = int(bases[self.rank])
        lids = lcnt = rids = rcnt = np.zeros(0, np.int64)
        lbase = rbase = 0
        if self.rank > 0 and hh:                                    # left halo = the left neighbour's LAST hh frames
            m = meta[self.rank - 1]
            lids, lcnt, lbase = m[2 + 2 * hh:2 + 3 * hh], m[2 + 3 * hh:2 + 4 * hh], int(bases[self.rank - 1] + m[1])
        if self.rank < self.world - 1 and hh:                       # right halo = the right neighbour's FIRST hh frames
            m = meta[self.rank + 1]
            rids, rcnt, rbase = m[2:2 + hh], m[2 + hh:2 + 2 * hh], int(bases[self.rank + 1])
        nl, nr = int(lcnt.sum()), int(rcnt.sum())
        n_loc = nl + n_own + nr
        if int(meta[:, 0].sum()) == 0:
            return torch.empty(0, dtype=torch.int32, device=self.device), 0, (nl, nr)

        # ---- local problem: [left halo | owned | right halo], times = frame ids, global point indices ------
        all_ids = np.concatenate([lids, ids, rids]).astype(np.float32)
        all_cnt = np.concatenate([lcnt, np.diff(off), rcnt]).astype(np.int64)
        head = np.concatenate([[0], np.cumsum(all_cnt)]).astype(np.int64)
        X, Y, times, gidx = eng.local_problem(pts, n_own, lo_end, hi_start, nl, nr, head, all_ids, lbase, gbase, rbase)
        self._tick("halo+prep")

        # every point (own or halo) lies inside the global raw bounds and every time is one of the ids: with that
        # hint the plan needs neither a bounds pass nor a sync
        hint = None
        if b4 is not None and len(all_ids) and np.array_equal(all_ids, np.rint(all_ids)):
            hint = (float(b4[0]), float(b4[1]), float(b4[2]), float(b4[3]), float(all_ids.min()), float(all_ids.max()))
        ph = eng.phases(X, Y, times, cfg.eps_space, cfg.eps_time, cfg.min_samples, hint=hint) if n_loc else None
        core = ph.cores() if n_loc else torch.zeros(0, dtype=torch.uint8, device=self.device)
        # ---- exact core flags of the halo points come from their owners ----------------------------------
        eng.exchange_cores(core, nl, n_own, nr, lo_end, hi_start)
        if n_loc:
            ph.set_cores(core)
            key = ph.components(gidx)
        else:
            key = torch.zeros(0, dtype=torch.int64, device=self.device)

        # ---- stitch (on every rank) -----------------------------------------------------------------------------
        # what the stitch needs from me: the local keys of my four boundary zones (left halo, own first frames, own last
        # frames, right halo - the same points, in the same order, as the neighbours' zones), run-length encoded over the
        # zone's points, and my distinct component keys (= keys of the points that ARE their component's smallest core).
        # The engine builds the fixed-capacity vector on the device; collective 3 all-gathers it.
        zones = ((0, nl), (nl, nl + lo_end), (nl + hi_start, nl + n_own), (nl + n_own, n_loc))
        while True:
            cap_k = self._key_cap
            vec = eng.pack_keys(key, gidx, zones, n_loc, cap_k)
            self._tick("plan..components+pack")
            if eng.wait_before_collective:
                yield self._pause(1)                           # the clustering kernels (~1 ms): same reasoning as for the spoke stage
            g_keys = eng.all_gather(vec)
            pause = self._pause(0 if eng.wait_before_collective else 1, g_keys)
            yield pause
            got = pause[2][0].numpy()                          # read-back C
            sizes = np.diff(got[:, :5], prepend=0, axis=1)
            need = int(sizes.sum(axis=1).max())
            if need <= cap_k:
                break
            self._key_cap = int(need * 1.5) + 1024             # too small somewhere: everybody repeats with more room
        # every rank's zones as runs (key, start) and its distinct component keys
        runs, all_keys = [], []
        for r in range(self.world):
            tot = int(sizes[r].sum())
            cuts = np.cumsum(sizes[r])[:-1]
            k_parts = np.split(got[r, 9:9 + tot], cuts)
            s_parts = np.split(got[r, 9 + cap_k:9 + cap_k + tot], cuts)
            runs.append([(k_parts[z], s_parts[z]) for z in range(4)])
            all_keys.append(k_parts[4])
        # the same boundary points under two ranks' keys: own last frames | left halo, right halo | own first frames
        e = np.zeros(0, np.int64)
        all_segs = [[e, e, e, e] for _ in range(self.world)]
        for r in range(self.world - 1):
            for za, zb in ((2, 0), (3, 1)):
                if got[r, 5 + za] != got[r + 1, 5 + zb]:
                    raise RadarB200Error("stitch: boundary zones of neighbouring ranks do not match")
                all_segs[r][za], all_segs[r + 1][zb] = pair_zone_runs(*runs[r][za], *runs[r + 1][zb])
        tk, ti, ncl = stitch_components(all_segs, all_keys)
        self._tick("stitch")

        # ---- labels of the owned points -------------------------------------------------------------------------
        if n_loc == 0:
            return torch.empty(0, dtype=torch.int32, device=self.device), int(ncl), (nl, nr)
        core_label = eng.relabel(key, eng.upload(tk, torch.int64), eng.upload(ti, torch.int32))
        labels = ph.assign(core_label)
        out = labels[nl:nl + n_own]
        self._tick("relabel+assign")
        return out, int(ncl), (nl, nr)

    # ---- host entries -----------------------------------------------------------------------------------------------
    def _run_host_gen(self, t_echo, angle_units, scale, frame_ids):
        """End-to-end path of one block as a generator: upload on the block's stream, the device path, and the
        read-back of this rank's result into pinned memory (awaited like every other read-back of the block)."""
        F, G, S, E = t_echo.shape
        c, s, r = self.base.spoke_tables(angle_units, scale, F, E)
        up = self.engine.upload
        d_echo = t_echo.to(self.device, non_blocking=True)
        res = yield from self._run_gen(d_echo, up(c), up(s), up(r), frame_ids)
        n, p = res.points.n, res.points
        pause = self._pause(0, p.x[:n], p.y[:n], p.inten[:n], p.gain[:n], p.frame_off, res.labels[:n])
        yield pause
        # copies, not views: the page-locked blocks go back to torch's host cache with this generator, so a caller that
        # keeps its results does not make every later block allocate page-locked memory (device.to_pinned_host)
        x, y, inten, gain, off, labels = (np.array(t.numpy()) for t in pause[2])
        del pause
        out = dict(points=np.stack([x, y, inten], axis=1), gains=gain, frame_off=off, labels=labels, frame_ids=res.frame_ids,
                   n_clusters=res.n_clusters)
        out["h2d_bytes"] = t_echo.numel() * t_echo.element_size() + 3 * c.nbytes
        out["d2h_bytes"] = out["points"].nbytes + gain.nbytes + labels.nbytes + off.nbytes
        return out

    def run_host_blocks(self, host_blocks, in_flight: int = 2, keep: bool = True):
        """``host_blocks``: ``(pinned echo tensor [F,G,S,E], angle_units, scale, frame_ids)`` per block. The blocks run
        interleaved like :meth:`run_blocks`, so the upload of one block overlaps the kernels and the read-back of
        another. Returns the host dictionaries of :meth:`run_host`."""
        if self.base is None:
            raise RadarB200Error("run_host_blocks needs the CUDA engine")
        return self.run_blocks(host_blocks, keep=keep, in_flight=in_flight, make_gen=self._run_host_gen)


    def run_host(self, echo, angle_units, scale, frame_ids: Sequence[int], pinned: Optional[torch.Tensor] = None) -> dict:
        """Host buffers in, host buffers out for this rank's frames: uploads ``echo[F,G,S,E]`` (numpy or a
        pinned torch tensor), runs the sharded device path and reads this rank's result back."""
        if self.base is None:
            raise RadarB200Error("run_host needs the CUDA engine")
        if pinned is not None:
            t_echo = pinned
        else:
            a = np.asarray(echo)
            t_echo = torch.from_numpy(np.ascontiguousarray(a, dtype=np.uint8 if a.dtype == np.uint8 else np.float32))
        F, G, S, E = t_echo.shape
        c, s, r = self.base.spoke_tables(angle_units, scale, F, E)
        d = self.device
        d_echo = t_echo.to(d, non_blocking=True)
        up = self.engine.upload
        res = self.run_device(d_echo, up(c), up(s), up(r), frame_ids)
        out = res.to_host()
        out["n_clusters"] = res.n_clusters
        out["h2d_bytes"] = t_echo.numel() * t_echo.element_size() + 3 * c.nbytes
        out["d2h_bytes"] = out["points"].nbytes + out["gains"].nbytes + out["labels"].nbytes + out["frame_off"].nbytes
        return out


# ------------------------------------------------------------------------------------------ whole recordings
def split_frames(n_frames: int, world: int, rank: int) -> Tuple[int, int]:
    """Frames ``[a, b)`` of rank ``rank`` when ``n_frames`` frames are split into ``world`` contiguous shares whose sizes
    differ by at most one (earlier ranks take the larger ones)."""
    if world < 1 or not 0 <= rank < world or n_frames < 0:
        raise RadarB200Error("split_frames: bad arguments")
    q, r = divmod(int(n_frames), int(world))
    a = rank * q + min(rank, r)
    return a, a + q + (1 if rank < r else 0)


def check_recording_stats(stats: np.ndarray, cluster: bool, h: int) -> None:
    """The decisions of :meth:`ShardedRecording.finish` that can fail, taken from every rank's gathered
    ``[frames, frames built, raw points, x_min, x_max, y_min, y_max, first id, last id]`` (``stats[world, 9]``): every rank
    sees the same numbers, so all raise the same :class:`RadarB200Error` together and none is left in a collective."""
    frames = stats[:, 0].astype(np.int64)
    if int(frames.sum()) == 0:
        raise RadarB200Error("finish() of an empty recording: no rank was fed any frame")
    world = len(stats)
    if cluster and world > 1:
        need = max(int(h), 1)
        short = [r for r in range(world) if frames[r] < need]
        if short:
            raise RadarB200Error(f"rank {short[0]} holds {int(frames[short[0]])} frames, fewer than the {need} that clustering over "
                                 f"{world} ranks needs (max(floor(eps_time), 1)): give every rank at least {need} frames")
        if h > 64:
            raise RadarB200Error(f"an eps_time halo of {h} frames is more than the 64 frames the ranks exchange")
    last, last_rank = None, None
    for r in range(world):
        if frames[r] == 0:
            continue
        first = int(stats[r, 7])
        if last is not None and first <= last:
            raise RadarB200Error(f"frame ids must increase strictly across ranks: rank {r}'s first id {first} is not above rank "
                                 f"{last_rank}'s last id {last}")
        last, last_rank = int(stats[r, 8]), r


def window_payload(head: np.ndarray, entries: Sequence[np.ndarray]) -> np.ndarray:
    """One rank's window encodings as one int64 vector for the all-gather: ``[n_windows | heads (9 per window) | per window
    its keys, then its starts]``; ``head[k]`` = window k's 5 running entry counts and 4 zone lengths
    (``rb_stdbscan_windowed_pass_keys``), ``entries`` = per window its keys and its starts (``head[k, 4]`` each)."""
    head = np.asarray(head, np.int64).reshape(-1, 9)
    return np.concatenate([[len(head)], head.ravel()] + [np.asarray(e, np.int64) for e in entries]).astype(np.int64)


def stitch_windows(payloads: np.ndarray) -> Tuple[np.ndarray, np.ndarray, int]:
    """The key -> cluster id table of a recording whose windows are spread over the ranks: ``payloads[r]`` = rank r's
    :func:`window_payload` (zero padded). The global window list is all ranks' windows in rank order; every pair of
    adjacent windows - inside a rank or across a rank edge - shares two boundary zones (own last frames | the next's left
    halo, right halo | the next's own first frames), whose encodings are paired (:func:`pair_zone_runs`) and stitched
    (:func:`stitch_components`). Every rank computes the same table from the same payloads."""
    heads, runs, all_keys = [], [], []
    for p in np.asarray(payloads, np.int64):
        nw = int(p[0])
        hr = p[1:1 + 9 * nw].reshape(nw, 9)
        at = 1 + 9 * nw
        for k in range(nw):
            tot = int(hr[k, 4])
            keys, starts = p[at:at + tot], p[at + tot:at + 2 * tot]
            at += 2 * tot
            bnd = np.concatenate([[0], hr[k, :5]])
            runs.append([(keys[bnd[z]:bnd[z + 1]], starts[bnd[z]:bnd[z + 1]]) for z in range(4)])
            all_keys.append(keys[bnd[4]:bnd[5]])
            heads.append(hr[k])
    e = np.zeros(0, np.int64)
    segs = [[e, e, e, e] for _ in heads]
    for k in range(len(heads) - 1):
        for za, zb in ((2, 0), (3, 1)):                          # own last | next's left halo, right halo | next's own first
            if heads[k][5 + za] != heads[k + 1][5 + zb]:
                raise RadarB200Error("stitch: boundary zones of neighbouring windows do not match")
            segs[k][za], segs[k + 1][zb] = pair_zone_runs(*runs[k][za], *runs[k + 1][zb])
    tk, ti, ncl = stitch_components(segs, all_keys)
    return np.ascontiguousarray(tk, np.int64), np.ascontiguousarray(ti, np.int32), int(ncl)


def cluster_starts(table_keys: np.ndarray, table_ids: np.ndarray, n_clusters: int) -> np.ndarray:
    """min_frames: every cluster's start, its smallest core index = the first key of its id in the sorted table."""
    start_of = np.full(max(int(n_clusters), 1), -1, np.int64)
    if len(table_ids):
        uid, first = np.unique(table_ids, return_index=True)
        start_of[uid] = np.asarray(table_keys)[first]
    return start_of


class ShardedRecording:
    """One recording detected over several GPUs, one process per GPU (DESIGN.md section 3.11): rank r is fed a contiguous
    share of the recording's frames - all of rank r's frames come before rank r+1's, ids increase strictly across ranks -
    through the feeding calls of :class:`recording.RecordingDetection` (``add_block``, ``add_host_block``,
    ``add_csv_frames``; each rank parses its own share of a CSV tree). :meth:`finish` is a collective that returns every
    rank's :class:`recording.RecordingResult` for its own frames.

    The results of all ranks, concatenated in rank order, equal ``RecordingDetection.finish()`` of one process fed the same
    frames in the same order, bit for bit and id for id: raw and filtered points with their frame offsets; the land grid,
    sums and mask (identical on every rank); ``land_ordered``; labels, core flags and the global ``n_clusters``;
    ``frames_built`` (the recording's). Also with ``DetectionConfig.min_frames`` and ``cluster_3d``. ``world == 1`` is
    exactly :class:`recording.RecordingDetection`.

    Every collective goes through the engine (:class:`CudaEngine`: NCCL by the library; a test engine may swap them),
    one communicator per rank, in one fixed order on every rank."""

    def __init__(self, config=None, rank: Optional[int] = None, world: Optional[int] = None, group=None, engine=None,
                 max_window_points: Optional[int] = None):
        from .recording import RecordingDetection

        self.group = group
        self.rank = dist.get_rank(group) if rank is None else int(rank)
        self.world = dist.get_world_size(group) if world is None else int(world)
        if not 0 <= self.rank < self.world:
            raise RadarB200Error(f"rank {self.rank} of a world of {self.world}")
        self.engine = engine or CudaEngine()
        self.engine.attach(self.rank, self.world, group)
        self.device = self.engine.device
        self.rec = RecordingDetection(config, self.device.index, max_window_points)
        self.cfg = self.rec.cfg
        self._key_cap = 1 << 15
        self._pinned = None
        self.timings = self.rec.timings

    # ---- feeding: RecordingDetection's calls on this rank's share -----------------------------------------------------
    def add_block(self, echo, cos_tab, sin_tab, range_res, frame_ids: Sequence[int]) -> None:
        """:meth:`recording.RecordingDetection.add_block` for the next frames of this rank's share."""
        self.rec.add_block(echo, cos_tab, sin_tab, range_res, frame_ids)

    def add_host_block(self, echo, angle_units, scale, frame_ids: Sequence[int]) -> None:
        """:meth:`recording.RecordingDetection.add_host_block` for the next frames of this rank's share."""
        self.rec.add_host_block(echo, angle_units, scale, frame_ids)

    def add_csv_frames(self, frame_files, frame_ids: Optional[Sequence[int]] = None, **kw) -> None:
        """:meth:`recording.RecordingDetection.add_csv_frames` for the next frames of this rank's share: each rank parses
        its own files. Pass ``frame_ids`` on every rank but the first (the default ids start at 0 on every rank)."""
        self.rec.add_csv_frames(frame_files, frame_ids, **kw)

    @property
    def pipe(self):
        return self.rec.pipe

    @property
    def csv_files(self):
        return self.rec.csv_files

    # ---- host read-backs and small all-gathers ------------------------------------------------------------------------
    def _read(self, *tensors) -> list:
        """Device tensors -> host numpy copies through one pinned buffer of this recording (grown, never shrunk), one sync."""
        sizes = [t.numel() * t.element_size() for t in tensors]
        total = sum((s + 15) // 16 * 16 for s in sizes)
        if self._pinned is None or self._pinned.numel() < total:
            self._pinned = torch.empty(max(total, 4096), dtype=torch.uint8, pin_memory=True)
        views, at = [], 0
        for t, s in zip(tensors, sizes):
            v = self._pinned[at:at + s].view(t.dtype).view(t.shape)
            v.copy_(t, non_blocking=True)
            views.append(v)
            at += (s + 15) // 16 * 16
        torch.cuda.current_stream(self.device).synchronize()
        return [np.array(v.numpy()) for v in views]

    def _gather(self, vec: np.ndarray) -> np.ndarray:
        """One host vector per rank (same length everywhere) -> ``[world, len]`` on every rank."""
        return self._read(self.engine.all_gather(self.engine.upload(np.ascontiguousarray(vec))))[0]

    # ---- the recording ------------------------------------------------------------------------------------------------
    def finish(self, cluster: bool = True):
        """Collective: land grid and filter over all ranks' frames, one ST-DBSCAN labelling of the recording whose
        windows are spread over the ranks; this rank's :class:`recording.RecordingResult` (see the class docstring)."""
        if self.world == 1:
            return self.rec.finish(cluster)
        return self._finish_protocol(cluster)

    def _finish_protocol(self, cluster: bool = True):
        """The protocol of :meth:`finish`. It also runs at ``world == 1``, where every collective is the identity:
        tools/run_sharded_recording.py measures its cost there next to :meth:`recording.RecordingDetection.finish`."""
        import contextlib
        import time

        from . import device as dev
        from .recording import RecordingResult

        rec, cfg, eng, d = self.rec, self.cfg, self.engine, self.device
        if rec._finished:
            raise RadarB200Error("finish() was already called")
        rec._finished = True
        eng.prepare_slots(1, lambda k: contextlib.nullcontext())
        timings = dict(rec.timings)
        t0 = time.perf_counter()

        # ---- 1. what every rank holds: every decision that can fail is taken from these gathered numbers -------------
        ids = np.concatenate(rec._ids) if rec._ids else np.zeros(0, np.int64)
        F = len(ids)
        raw_off = np.concatenate([[0]] + [o[1:] + b for o, b in zip(rec._offs[1:], rec._bases)]).astype(np.int64)
        n_raw = rec._n
        if rec._store is None:
            rec._grow(1)
        xs, ys, iss, gs = rec._store
        raw = dev.PointBatch(xs, ys, iss, gs, torch.from_numpy(raw_off).to(d), n_raw)
        built_here = int(np.count_nonzero(np.diff(raw_off)))
        b4 = rec._b4 if rec._b4 is not None else np.zeros(4, np.float32)
        stats = self._gather(np.array([F, built_here, n_raw, *b4, ids[0] if F else 0, ids[-1] if F else 0], np.float64))
        h = int(math.floor(np.float32(cfg.eps_time))) if cfg.eps_time >= 0 else 0
        check_recording_stats(stats, cluster, h)
        built, n_all = int(stats[:, 1].sum()), int(stats[:, 2].sum())
        have = stats[stats[:, 2] > 0]
        gb4 = (np.array([have[:, 3].min(), have[:, 4].max(), have[:, 5].min(), have[:, 6].max()], np.float32)
               if len(have) else None)
        timings["stats"] = time.perf_counter() - t0

        # ---- 2. land: one grid over the recording, every rank's sums added up -------------------------------------------
        t0 = time.perf_counter()
        pts, land, edges, count, isum, land_ordered = raw, None, None, None, None, False
        if cfg.land_filter and n_all > 0 and built > cfg.land_min_frames:
            xe, ye = dev.arange_edges(gb4[0], gb4[1], cfg.land_resolution), dev.arange_edges(gb4[2], gb4[3], cfg.land_resolution)
            if len(xe) < 2 or len(ye) < 2:
                raise RadarB200Error("degenerate land grid")
            nx, ny = len(xe) - 1, len(ye) - 1
            d_xe, d_ye = eng.upload(xe), eng.upload(ye)
            chunks = rec._chunks(raw_off) if n_raw else []
            count = torch.zeros((nx, ny), dtype=torch.int32, device=d)
            isum = torch.zeros((nx, ny), dtype=torch.float64, device=d)
            rec._land_accumulate(False, chunks, raw_off, d_xe, d_ye, count, isum)
            inexact = self._gather(np.array([1 if rec._land_inexact() else 0], np.int64))
            if not inexact.any():
                eng.all_reduce_grids(count, isum)                # sums of integers: exact in any order
            else:
                # non-integer intensities: the float64 sums depend on the order of addition. The ordered accumulation
                # runs as a chain in rank order - each rank continues from the sums of all ranks before it - and one
                # all-reduce adds the last rank's grids to zeros everywhere else, which is exact
                land_ordered = True
                count.zero_(), isum.zero_()
                grids = [count.view(-1), isum.view(-1)]
                none = [count.new_empty(0), isum.new_empty(0)]
                if self.rank > 0:
                    eng.exchange(none, none, grids, none)
                rec._land_accumulate(True, chunks, raw_off, d_xe, d_ye, count, isum)
                if self.rank < self.world - 1:
                    eng.exchange(none, grids, none, none)
                    count.zero_(), isum.zero_()
                eng.all_reduce_grids(count, isum)
            land = dev.land_cells(count, isum, built, cfg.land_persistence, cfg.land_min_intensity)
            if n_raw:
                fx, fy, fi, fg, f_off, at = rec._land_filter(chunks, raw_off, d_xe, d_ye, land)
            else:
                fx, fy, fi = (torch.empty(1, dtype=torch.float32, device=d) for _ in range(3))
                fg, f_off, at = torch.empty(1, dtype=torch.int32, device=d), np.zeros(F + 1, np.int64), 0
            pts = dev.PointBatch(fx, fy, fi, fg, torch.from_numpy(f_off).to(d), at)
            edges = (xe, ye)
        p_off = raw_off if pts is raw else pts.frame_off.cpu().numpy()
        torch.cuda.current_stream(d).synchronize()
        timings["land"] = time.perf_counter() - t0

        labels = torch.empty(0, dtype=torch.int32, device=d)
        core, cuts, n_clusters = None, None, 0
        if cluster:
            labels, core, cuts, n_clusters = self._cluster(pts, p_off, ids, h, gb4, timings)
        return RecordingResult(ids, raw, pts, labels, n_clusters, land, edges, count, isum, core=core, cuts=cuts,
                               frames_built=built, land_ordered=land_ordered, timings=timings,
                               frame_times=list(rec._times) if rec._csv_frames else None)

    def _cluster(self, pts: PointBatch, p_off: np.ndarray, ids: np.ndarray, h: int, gb4, timings: dict):
        """Steps 3 and 4 of :meth:`finish`: halos, then the three windowed passes with the stitch of every rank's windows."""
        import ctypes as C
        import time

        from ._lib import StdbscanHint, check, ptr, stream_ptr
        from .recording import plan_windows

        cfg, eng, d, rec = self.cfg, self.engine, self.device, self.rec
        ctx = rec.ctx
        t0 = time.perf_counter()
        F = len(ids)
        h = min(h, F)                                            # (more than F only at world 1, without neighbours)
        n_own = int(p_off[-1])
        # ---- 3. layout of every rank's boundary frames; the local problem [left halo | owned | right halo] ------------
        meta = self._read(eng.all_gather(eng.pack_layout(pts.frame_off, ids, F, h)))[0]
        if int(meta[:, 0].sum()) == 0:
            return torch.empty(0, dtype=torch.int32, device=d), None, None, 0
        lids = lcnt = rids = rcnt = np.zeros(0, np.int64)
        if self.rank > 0 and h:                                  # left halo = the left neighbour's last h frames
            m = meta[self.rank - 1]
            lids, lcnt = m[2 + 2 * h:2 + 3 * h], m[2 + 3 * h:2 + 4 * h]
        if self.rank < self.world - 1 and h:                     # right halo = the right neighbour's first h frames
            m = meta[self.rank + 1]
            rids, rcnt = m[2:2 + h], m[2 + h:2 + 2 * h]
        nl, nr = int(lcnt.sum()), int(rcnt.sum())
        n_loc = nl + n_own + nr
        index_base = int(meta[:self.rank, 0].sum()) - nl
        loc_off = np.ascontiguousarray(np.concatenate([[0], np.cumsum(np.concatenate([lcnt, np.diff(p_off), rcnt]))]), dtype=np.int64)
        loc_ids = np.ascontiguousarray(np.concatenate([lids, ids, rids]), dtype=np.float32)
        own_fa, own_fb = len(lids), len(lids) + F
        lo_end, hi_start = int(p_off[h]), int(p_off[F - h])       # owned points [0, lo_end) go left, [hi_start, n_own) right
        dims = 3 if cfg.cluster_3d else 2
        src = [pts.x, pts.y, pts.inten][:dims]
        loc = [torch.empty(max(n_loc, 1), dtype=torch.float32, device=d) for _ in range(dims)]
        for t, s in zip(loc, src):
            t[nl:nl + n_own].copy_(s[:n_own])
        eng.exchange([s[:lo_end] for s in src], [s[hi_start:n_own] for s in src], [t[:nl] for t in loc],
                     [t[nl + n_own:n_loc] for t in loc])
        X, Y, Z = loc[0], loc[1], (loc[2] if dims == 3 else None)
        torch.cuda.current_stream(d).synchronize()
        timings["layout_halos"] = time.perf_counter() - t0

        # ---- 4. this rank's windows over its owned frames; the three passes ----------------------------------------------
        t0 = time.perf_counter()
        cuts = np.ascontiguousarray(plan_windows(loc_off, h, rec.window_budget(n_loc), own=(own_fa, own_fb)), dtype=np.int64)
        n_w = len(cuts) - 1
        hint = None
        if gb4 is not None and Z is None:                        # every point lies in the global raw bounds: no plan syncs
            hint = StdbscanHint()
            hint.lo[0], hint.hi[0], hint.lo[1], hint.hi[1] = (float(v) for v in gb4)
            hint.times_integer = 1
        mf = 0 if cfg.min_frames is None else int(cfg.min_frames)
        lib, hd = ctx.lib, ctx.handle
        common = (hd, ptr(X), ptr(Y), ptr(Z), 1, loc_off.ctypes.data, loc_ids.ctypes.data, len(loc_ids), own_fa, own_fb,
                  cuts.ctypes.data, n_w, index_base, float(cfg.eps_space), float(np.float32(cfg.eps_time)), int(cfg.min_samples), mf,
                  C.byref(hint) if hint is not None else None)
        core = torch.empty(max(n_loc, 1), dtype=torch.uint8, device=d)
        check(lib.rb_stdbscan_windowed_pass_cores(*common, ptr(core), stream_ptr()), "rb_stdbscan_windowed_pass_cores")
        eng.exchange_cores(core[:n_loc], nl, n_own, nr, lo_end, hi_start)  # halo points take their owner's core flags
        torch.cuda.current_stream(d).synchronize()
        timings["pass_cores"] = time.perf_counter() - t0

        t0 = time.perf_counter()
        left, right = int(self.rank > 0), int(self.rank < self.world - 1)

        def encode(k0, n_enc, cap, flag=None):
            vec = torch.empty(n_enc * (9 + 2 * cap), dtype=torch.int64, device=d)
            check(lib.rb_stdbscan_windowed_pass_keys(*common, left, right, ptr(core), k0, n_enc, cap, ptr(vec), ptr(flag), stream_ptr()),
                  "rb_stdbscan_windowed_pass_keys")
            return vec.view(n_enc, 9 + 2 * cap)

        cap = self._key_cap
        flag = torch.zeros(1, dtype=torch.int64, device=d)
        vec = encode(0, n_w, cap, flag)
        head, bad = self._read(vec[:, :9], flag)
        rows = [(vec[k], cap) for k in range(n_w)]
        for k in range(n_w):                                     # a window that outgrew the guess is encoded again alone
            need = int(head[k, 4])
            if need > cap:
                rows[k] = (encode(k, 1, need)[0], need)
        self._key_cap = min(max(self._key_cap, int(head[:, 4].max()) * 5 // 4), 1 << 22)
        parts = []
        for k, (row, c) in enumerate(rows):
            tot = int(head[k, 4])
            parts += [row[9:9 + tot], row[9 + c:9 + c + tot]]
        ent = self._read(*parts) if parts else []
        payload = window_payload(head, ent)
        torch.cuda.current_stream(d).synchronize()
        timings["pass_keys"] = time.perf_counter() - t0

        # ---- every rank's window encodings (sizes first, then the payload), stitched identically on every rank ------------
        t0 = time.perf_counter()
        sizes = self._gather(np.array([len(payload), int(bad[0])], np.int64))
        if sizes[:, 1].any():
            raise RadarB200Error("sharded recording: the global raw bounds do not contain every point of a local problem "
                                 f"(rank {int(np.nonzero(sizes[:, 1])[0][0])}); the result would be invalid")
        width = int(sizes[:, 0].max())
        got = self._gather(np.concatenate([payload, np.zeros(width - len(payload), np.int64)]))
        tk, ti, ncl = stitch_windows(got)
        start_of = cluster_starts(tk, ti, ncl) if mf else np.full(1, -1, np.int64)
        timings["stitch"] = time.perf_counter() - t0

        t0 = time.perf_counter()
        labels = torch.empty(max(n_own, 1), dtype=torch.int32, device=d)
        check(lib.rb_stdbscan_windowed_pass_labels(*common, ptr(core), tk.ctypes.data, ti.ctypes.data, len(tk), start_of.ctypes.data,
                                                   ncl if mf else 0, ptr(labels), stream_ptr()), "rb_stdbscan_windowed_pass_labels")
        timings["pass_labels"] = time.perf_counter() - t0
        return labels[:n_own], core[nl:nl + n_own], cuts - own_fa, int(ncl)
