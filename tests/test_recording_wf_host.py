"""CPU-side checks of the PointCloudWorkF variant on recordings: DetectionConfig.min_frames validation and the C entry
rb_stdbscan_windowed_wf in the header, the bindings and the library."""
import ctypes
import re
from pathlib import Path

import numpy as np
import pytest

from radar_point_cloud_tracking_b200 import _lib
from radar_point_cloud_tracking_b200._lib import RadarB200Error
from radar_point_cloud_tracking_b200.pipeline import DetectionConfig

REPO = Path(__file__).resolve().parent.parent


def test_min_frames_default_keeps_the_t4_clustering():
    assert DetectionConfig().min_frames is None
    assert DetectionConfig(eps_time=45.0).min_frames is None          # no limit on eps_time without the variant


@pytest.mark.parametrize("k", [1, 3, np.int64(4), 61])
def test_min_frames_accepts_ints_from_one(k):
    assert DetectionConfig(min_frames=k, eps_time=30.0).min_frames == k


@pytest.mark.parametrize("k", [0, -2, 2.0, 2.5, True, "3"])
def test_min_frames_rejects_non_ints_and_below_one(k):
    with pytest.raises(RadarB200Error):
        DetectionConfig(min_frames=k)


@pytest.mark.parametrize("eps_time", [30.5, 31.0, float("inf"), float("nan")])
def test_min_frames_needs_eps_time_at_most_30(eps_time):
    with pytest.raises(RadarB200Error):
        DetectionConfig(min_frames=2, eps_time=eps_time)


def test_validate_sees_later_changes():
    cfg = DetectionConfig()
    cfg.min_frames = 0
    with pytest.raises(RadarB200Error):
        cfg.validate()
    cfg.min_frames, cfg.eps_time = 2, 40.0
    with pytest.raises(RadarB200Error):
        cfg.validate()


def test_windowed_wf_is_declared_bound_and_exported():
    text = re.sub(r"/\*.*?\*/", "", (REPO / "include" / "radarb200.h").read_text(), flags=re.S)
    decl = re.search(r"int\s+rb_stdbscan_windowed_wf\s*\(([^;]*)\)\s*;", text)
    assert decl is not None
    n_args = len([a for a in decl.group(1).split(",") if a.strip()])
    restype, argtypes = _lib.SIGNATURES["rb_stdbscan_windowed_wf"]
    assert restype is ctypes.c_int32 and len(argtypes) == n_args == 19
    # rb_stdbscan_windowed's arguments with int min_frames after min_samples
    base = _lib.SIGNATURES["rb_stdbscan_windowed"][1]
    assert list(argtypes[:13]) == list(base[:13]) and argtypes[13] is ctypes.c_int32 and list(argtypes[14:]) == list(base[13:])
    assert getattr(ctypes.CDLL(str(_lib.LIB_PATH)), "rb_stdbscan_windowed_wf") is not None
