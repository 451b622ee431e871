"""ctypes binding of ``libradarb200.so`` (the C ABI declared in ``include/radarb200.h``).

There is no fallback: if the shared library is missing or no CUDA device is present, every
entry point raises. PyTorch is used only to allocate device memory and to provide the current
stream; all compute is in the hand-written kernels behind this ABI.
"""
from __future__ import annotations

import ctypes as C
import threading
from pathlib import Path
from typing import Dict, Optional

PKG = Path(__file__).resolve().parent
LIB_PATH = PKG / "libradarb200.so"

c_i32, c_i64, c_f32, c_f64, c_vp = C.c_int, C.c_int64, C.c_float, C.c_double, C.c_void_p


class DbscanStats(C.Structure):
    _fields_ = [("n_points", c_i64), ("n_cells", c_i64), ("n_core", c_i64), ("n_clusters", c_i64),
                ("pair_tests_count", c_i64), ("pair_tests_union", c_i64), ("pair_tests_border", c_i64),
                ("cell_size", c_f64), ("time_bin", c_f64), ("dims", c_i32 * 4), ("time_radius", c_i32), ("tight", c_i32)]


class StdbscanHint(C.Structure):
    _fields_ = [("lo", c_f32 * 4), ("hi", c_f32 * 4), ("times_integer", c_i32)]


class DetectParams(C.Structure):
    _fields_ = [("n_frames", c_i32), ("gains_per_frame", c_i32), ("n_spokes", c_i32), ("n_bins", c_i32),
                ("intensity_threshold", c_f32), ("point_stride", c_i32), ("land_filter", c_i32), ("land_min_frames", c_i32),
                ("land_resolution", c_f64), ("land_persistence", c_f64), ("land_min_intensity", c_f64),
                ("eps_space", c_f64), ("eps_time", c_f32), ("min_samples", c_i32), ("cluster", c_i32), ("echo_u8", c_i32),
                ("cluster_3d", c_i32)]


class DetectBuffers(C.Structure):
    _fields_ = [("x", c_vp), ("y", c_vp), ("inten", c_vp), ("gain", c_vp), ("frame_off", c_vp),
                ("fx", c_vp), ("fy", c_vp), ("finten", c_vp), ("fgain", c_vp), ("f_frame_off", c_vp),
                ("labels", c_vp), ("cap", c_i64),
                ("count", c_vp), ("isum", c_vp), ("land", c_vp), ("max_cells", c_i64),
                ("x_edges", c_vp), ("y_edges", c_vp), ("max_edges", c_i32)]


class ClusterTable(C.Structure):
    _fields_ = [("frame", c_vp), ("label", c_vp), ("first", c_vp), ("count", c_vp), ("start", c_vp),
                ("cx", c_vp), ("cy", c_vp), ("mean_intensity", c_vp)]


class DetectResult(C.Structure):
    _fields_ = [("n_raw", c_i64), ("n_points", c_i64), ("n_clusters", c_i64),
                ("frames_built", c_i32), ("land_applied", c_i32), ("filtered_is_raw", c_i32),
                ("n_x_edges", c_i32), ("n_y_edges", c_i32), ("bounds", c_f32 * 4), ("land_ordered", c_i32)]


#: name -> (restype, argtypes); must list every symbol of include/radarb200.h
SIGNATURES = {
    "rb_version": (c_i32, []),
    "rb_last_error": (C.c_char_p, []),
    "rb_create": (c_i32, [c_i32, C.POINTER(c_vp)]),
    "rb_destroy": (None, [c_vp]),
    "rb_trim": (c_i32, [c_vp]),
    "rb_device_info": (c_i32, [c_vp, C.POINTER(c_i32), C.POINTER(c_i32), C.POINTER(c_i32), C.POINTER(c_i64)]),
    "rb_spoke_to_points": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_i32, c_i32, c_f32, c_i32,
                                   c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_vp]),
    "rb_spoke_to_points_u8": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_i32, c_i32, c_f32, c_i32,
                                      c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_vp]),
    "rb_polar_to_cartesian": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_i64, c_i32, c_vp, c_vp, c_vp]),
    "rb_frame_offsets": (c_i32, [c_vp, c_vp, c_i64, c_i32, c_vp, c_vp]),
    "rb_expand_frame_times": (c_i32, [c_vp, c_vp, c_vp, c_i64, c_i64, c_vp, c_vp]),
    "rb_fuse_max": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_i64, c_f32, c_f32, c_f32, c_i32, c_i32,
                            c_vp, c_vp, c_vp, c_i64, C.POINTER(c_i64), c_vp]),
    "rb_fuse_max_frames": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_i64, c_f64, c_vp, c_vp, c_vp, c_i64, c_vp,
                                   C.POINTER(c_i64), c_vp]),
    "rb_fuse_plan_groups": (c_i64, [c_vp, c_i64, c_i64, c_vp, c_i64]),
    "rb_bounds": (c_i32, [c_vp, c_vp, c_vp, c_i64, c_vp, c_vp]),
    "rb_bounds_counted": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_vp]),
    "rb_land_accumulate": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_i32, c_vp, c_i32, c_vp, c_vp, c_vp]),
    "rb_land_accumulate_status": (c_i32, [c_vp, C.POINTER(c_i32), c_vp]),
    "rb_land_accumulate_status_async": (c_i32, [c_vp, c_vp, c_vp]),
    "rb_land_accumulate_ordered": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_i32, c_vp, c_i32, c_vp, c_vp, c_vp]),
    "rb_land_cells": (c_i32, [c_vp, c_vp, c_vp, c_i64, c_i64, c_f64, c_f64, c_vp, c_vp]),
    "rb_land_filter": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_i64, c_vp, c_i32, c_vp, c_i32,
                               c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "rb_stdbscan": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_i64, c_f64, c_f32, c_i32,
                            c_vp, c_vp, C.POINTER(c_i64), c_vp]),
    "rb_stdbscan_wf": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_i64, c_f64, c_f32, c_i32, c_i32, c_vp, c_vp, C.POINTER(c_i64), c_vp]),
    "rb_stdbscan_last_stats": (c_i32, [c_vp, C.POINTER(DbscanStats)]),
    "rb_stdbscan_plan": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_i64, c_f64, c_f32, c_i32, c_vp]),
    "rb_stdbscan_plan_hinted": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_i64, c_f64, c_f32, c_i32, C.POINTER(StdbscanHint), c_vp]),
    "rb_stdbscan_check": (c_i32, [c_vp, c_vp]),
    "rb_stdbscan_cores": (c_i32, [c_vp, c_vp, c_vp]),
    "rb_stdbscan_set_cores": (c_i32, [c_vp, c_vp, c_vp]),
    "rb_stdbscan_components": (c_i32, [c_vp, c_vp, c_vp, c_vp]),
    "rb_stdbscan_assign": (c_i32, [c_vp, c_vp, c_vp, c_vp]),
    "rb_relabel": (c_i32, [c_vp, c_vp, c_i64, c_vp, c_vp, c_i64, c_vp, c_vp]),
    "rb_detect_block": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, C.POINTER(DetectParams), C.POINTER(DetectBuffers),
                                C.POINTER(DetectResult), c_vp]),
    "rb_cluster_records": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_i64, c_i64, C.POINTER(ClusterTable), c_i64,
                                   c_vp, c_vp, c_vp, C.POINTER(c_i64), C.POINTER(c_i64), c_vp]),
    "rb_arange_edges": (c_i64, [c_f32, c_f32, c_f64, c_vp, c_i64]),
    "rb_stitch_components": (c_i64, [c_vp, c_i64, c_vp, c_vp, c_i64, c_vp, c_vp, c_i64, c_vp]),
    "rb_stdbscan_windowed": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_vp, c_i64, c_vp, c_i64, c_f64, c_f32, c_i32,
                                     C.POINTER(StdbscanHint), c_vp, c_vp, C.POINTER(c_i64), c_vp]),
    "rb_stdbscan_windowed_wf": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_vp, c_i64, c_vp, c_i64, c_f64, c_f32, c_i32, c_i32,
                                        C.POINTER(StdbscanHint), c_vp, c_vp, C.POINTER(c_i64), c_vp]),
    "rb_stdbscan_windowed_pass_cores": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_vp, c_i64, c_i64, c_i64, c_vp, c_i64, c_i64,
                                                c_f64, c_f32, c_i32, c_i32, C.POINTER(StdbscanHint), c_vp, c_vp]),
    "rb_stdbscan_windowed_pass_keys": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_vp, c_i64, c_i64, c_i64, c_vp, c_i64, c_i64,
                                               c_f64, c_f32, c_i32, c_i32, C.POINTER(StdbscanHint), c_i32, c_i32, c_vp, c_i64, c_i64,
                                               c_i64, c_vp, c_vp, c_vp]),
    "rb_stdbscan_windowed_pass_labels": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_vp, c_i64, c_i64, c_i64, c_vp, c_i64, c_i64,
                                                 c_f64, c_f32, c_i32, c_i32, C.POINTER(StdbscanHint), c_vp, c_vp, c_vp, c_i64, c_vp,
                                                 c_i64, c_vp, c_vp]),
    "rb_pair_zone_runs": (c_i64, [c_vp, c_vp, c_i64, c_vp, c_vp, c_i64, c_vp, c_vp, c_i64]),
    "rb_comm_unique_id": (c_i32, [c_vp]),
    "rb_comm_init": (c_i32, [c_vp, c_vp, c_i32, c_i32]),
    "rb_comm_destroy": (c_i32, [c_vp]),
    "rb_comm_info": (c_i32, [c_vp, C.POINTER(c_i32), C.POINTER(c_i32)]),
    "rb_comm_all_gather": (c_i32, [c_vp, c_vp, c_vp, c_i64, c_vp]),
    "rb_comm_all_reduce_sum": (c_i32, [c_vp, c_vp, c_i64, c_i32, c_vp]),
    "rb_comm_all_reduce_grids": (c_i32, [c_vp, c_vp, c_vp, c_i64, c_vp]),
    "rb_comm_exchange": (c_i32, [c_vp, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "rb_shard_pack_stats": (c_i32, [c_vp, c_vp, c_i64, c_vp, c_i64, c_vp, c_vp]),
    "rb_shard_pack_layout": (c_i32, [c_vp, c_vp, c_i64, c_vp, c_i32, c_vp, c_vp]),
    "rb_shard_local_index": (c_i32, [c_vp, c_vp, c_vp, c_i64, c_i64, c_i64, c_i64, c_i64, c_i64, c_i64, c_vp, c_vp, c_vp]),
    "rb_shard_pack_keys": (c_i32, [c_vp, c_vp, c_vp, c_i64, c_vp, c_i64, c_vp, c_vp]),
    "rb_csv_parse_sweep": (c_i32, [c_vp, c_vp, c_i64, c_i32, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "rb_csv_sweeps_lines": (c_i32, [c_vp, c_vp, c_i64, c_vp, c_vp, c_i32, c_i32, c_vp, c_vp, c_vp, c_vp]),
    "rb_csv_parse_sweeps": (c_i32, [c_vp, c_vp, c_i64, c_vp, c_vp, c_i32, c_i32, c_vp, c_i64, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp,
                                    c_vp, c_vp, c_vp]),
    "rb_ply_append_ascii": (c_i32, [C.c_char_p, c_vp, c_vp, c_vp, c_vp, c_i64]),
    "rb_ply_format_ascii": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_i64, c_vp, c_vp, c_vp]),
    "rb_ply_pack_binary": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_vp]),
    "rb_ply_colors_intensity": (c_i32, [c_vp, c_vp, c_i32, c_i64, c_vp, c_i64, c_i32, c_vp, c_vp, c_vp]),
    "rb_ply_colors_gain": (c_i32, [c_vp, c_vp, c_i64, c_vp, c_vp]),
    "rb_synth_echo": (c_i32, [c_vp, c_vp, c_i64, c_i32, c_i32, c_i32, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "rb_set_option": (c_i32, [c_vp, C.c_char_p, c_i64]),
    "rb_get_info": (c_i64, [c_vp, C.c_char_p]),
    "rb_launch_count": (c_i64, [c_vp]),
}

_lib: Optional[C.CDLL] = None
_lock = threading.Lock()


class RadarB200Error(RuntimeError):
    pass


def load() -> C.CDLL:
    """Load the shared library and bind every declared symbol (no compute, works without a GPU)."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not LIB_PATH.exists():
            raise RadarB200Error(
                f"{LIB_PATH} is missing: build it with `python -m radar_point_cloud_tracking_b200.build` "
                "(there is no CPU fallback for this path)")
        lib = C.CDLL(str(LIB_PATH))
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)          # AttributeError if a declared symbol is not exported
            fn.restype = res
            fn.argtypes = args
        _lib = lib
        return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().rb_last_error()
        raise RadarB200Error(f"{what} failed (rc={rc}): {msg.decode() if msg else '?'}")


class Context:
    """One ``rb_ctx`` per CUDA device (per thread of use)."""

    def __init__(self, device: int):
        lib = load()
        h = c_vp()
        check(lib.rb_create(int(device), C.byref(h)), "rb_create")
        self.handle = h
        self.device = int(device)
        self.lib = lib
        sm, maj, mnr, l2 = c_i32(), c_i32(), c_i32(), c_i64()
        check(lib.rb_device_info(h, C.byref(sm), C.byref(maj), C.byref(mnr), C.byref(l2)), "rb_device_info")
        self.sm_count, self.cc, self.l2_bytes = sm.value, (maj.value, mnr.value), l2.value

    def set_option(self, name: str, value: int) -> None:
        check(self.lib.rb_set_option(self.handle, name.encode(), int(value)), f"rb_set_option({name})")

    def info(self, name: str) -> int:
        return int(self.lib.rb_get_info(self.handle, name.encode()))

    def launch_count(self) -> int:
        return int(self.lib.rb_launch_count(self.handle))

    def close(self) -> None:
        if self.handle:
            self.lib.rb_destroy(self.handle)
            self.handle = None

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass


# A ctx is not thread safe and holds per-call state (scratch, the ST-DBSCAN plan, a communicator): one per device, host
# thread and block slot (several blocks interleaved by one thread, sharded.ShardedDetection.run_blocks). The contexts of
# a thread live in ITS thread-local storage: when the thread ends they are released (rb_destroy frees scratch, pinned
# staging and the communicator) instead of piling up under recycled thread ids; `_all_contexts` only observes them.
import weakref

_tls = threading.local()
_all_contexts: "weakref.WeakSet[Context]" = weakref.WeakSet()


def context(device: Optional[int] = None) -> Context:
    """Context of ``device`` (default: torch's current CUDA device) for the calling thread and block slot.
    Raises without a GPU."""
    import torch

    if not torch.cuda.is_available():
        raise RadarB200Error("no CUDA device: the radar-b200 detection path is GPU only (no CPU fallback)")
    if device is None:
        device = torch.cuda.current_device()
    mine = getattr(_tls, "contexts", None)
    if mine is None:
        mine = _tls.contexts = {}
    key = (device, getattr(_tls, "slot", 0))
    ctx = mine.get(key)
    if ctx is None:
        ctx = mine[key] = Context(device)
        with _lock:
            _all_contexts.add(ctx)
    return ctx


def set_slot(slot: int) -> int:
    """Select the block slot of the calling thread (see :func:`context`); returns the previous one."""
    prev = getattr(_tls, "slot", 0)
    _tls.slot = int(slot)
    return prev


def launch_count_all() -> int:
    """Kernel launches of every live context of this process (all devices, threads and block slots)."""
    with _lock:
        live = list(_all_contexts)
    return sum(c.launch_count() for c in live if c.handle)


def get_slot() -> int:
    return getattr(_tls, "slot", 0)


def bind_to_gpu_numa(device: Optional[int] = None) -> Optional[list]:
    """Pin the calling process to the CPU cores next to ``device`` (NVML's ideal CPU affinity of the GPU = the cores of its
    NUMA node). With one process per GPU this keeps every rank's pinned host buffers and its copy threads on the socket
    the GPU hangs off; without it the 8 ranks' host-to-device streams cross the inter-socket link at random and the
    end-to-end rate stops scaling (round 1: 0.43 per-GPU efficiency at 8 GPUs). Call before allocating pinned memory.
    Returns the CPU list, or ``None`` when NVML / the affinity call is unavailable (nothing is changed then)."""
    import os

    import torch

    try:
        import pynvml

        if device is None:
            device = torch.cuda.current_device()
        pynvml.nvmlInit()
        visible = os.environ.get("CUDA_VISIBLE_DEVICES")
        idx = int(visible.split(",")[device]) if visible else device
        h = pynvml.nvmlDeviceGetHandleByIndex(idx)
        n_cpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (n_cpu + 63) // 64)
        cpus = [64 * w + b for w, word in enumerate(words) for b in range(64) if (int(word) >> b) & 1 and 64 * w + b < n_cpu]
        allowed = sorted(set(cpus) & set(os.sched_getaffinity(0)))
        if not allowed:
            return None
        os.sched_setaffinity(0, allowed)
        return allowed
    except Exception:
        return None


def stream_ptr() -> int:
    import torch

    return int(torch.cuda.current_stream().cuda_stream)


def ptr(t) -> Optional[int]:
    """Device pointer of a torch tensor (None -> NULL)."""
    if t is None:
        return None
    return int(t.data_ptr())
