"""CPU-side checks of max fusion over many frames: the C entry rb_fuse_max_frames in the header and the bindings, the
resolution validated before any device work, and the frame grouping (rb_fuse_plan_groups) against a restatement."""
import re
from pathlib import Path

import numpy as np
import pytest
import torch

from radar_point_cloud_tracking_b200 import _lib, device, fusion
from radar_point_cloud_tracking_b200._lib import RadarB200Error

REPO = Path(__file__).resolve().parent.parent
BAD_RESOLUTIONS = [0, 0.0, -1, -2.5, float("nan"), float("inf"), -float("inf"), "a", None]


@pytest.mark.parametrize("name", ["rb_fuse_max_frames", "rb_fuse_plan_groups"])
def test_symbol_in_header_and_bindings(name):
    header = (REPO / "include" / "radarb200.h").read_text()
    assert re.search(rf"\b{name}\s*\(", header)
    assert name in _lib.SIGNATURES
    assert hasattr(_lib.load(), name)


def _cpu_batch(n=5, frames=2):
    off = torch.tensor(np.linspace(0, n, frames + 1).astype(np.int64))
    z = torch.zeros(n, dtype=torch.float32)
    return device.PointBatch(z, z, z, None, off, n)


@pytest.mark.parametrize("res", BAD_RESOLUTIONS)
def test_resolution_is_checked_before_any_device_work(res):
    with pytest.raises(RadarB200Error, match="grid_resolution"):
        fusion.fuse_frames_max(_cpu_batch(), res)
    with pytest.raises(RadarB200Error, match="grid_resolution"):
        fusion.fuse_points_max({40: (np.zeros(3, np.float32),) * 3}, res)
    with pytest.raises(RadarB200Error, match="grid_resolution"):
        fusion.fuse_csv_frames_max([{40: REPO / "no_such_file.csv"}], res)


@pytest.mark.parametrize("res", [1.0, 2.5, 0.3, 1e-3, 7])
def test_good_resolutions_pass(res):
    assert device.check_resolution(res) == float(res)


def _groups(cells, bound):
    """Consecutive frames while their cells add up to at most ``bound``; a frame above it is a group alone."""
    cuts, s = [0], 0
    for f, c in enumerate(cells):
        if c and s and s + c > bound:
            cuts.append(f)
            s = 0
        s += c
    if len(cells):
        cuts.append(len(cells))
    return np.array(cuts, dtype=np.int64)


@pytest.mark.parametrize("cells,bound,want", [
    ([], 10, [0]),
    ([0, 0, 0], 1, [0, 3]),
    ([4, 4, 4], 8, [0, 2, 3]),
    ([4, 4, 4], 12, [0, 3]),
    ([20, 1, 1], 8, [0, 1, 3]),               # a frame above the bound is a group alone
    ([1, 20, 1], 8, [0, 1, 2, 3]),
    ([0, 20, 0, 3], 8, [0, 3, 4]),            # frames without cells join whichever group is open
    ([5, 0, 0, 5], 5, [0, 3, 4]),
])
def test_plan_groups_known_cases(cells, bound, want):
    assert device.fuse_plan_groups(cells, bound).tolist() == want
    assert _groups(cells, bound).tolist() == want


def test_plan_groups_random_against_restatement():
    rng = np.random.default_rng(3)
    for _ in range(200):
        F = int(rng.integers(0, 60))
        cells = rng.integers(0, 50, F) * (rng.random(F) < 0.8)
        bound = int(rng.integers(1, 120))
        got = device.fuse_plan_groups(cells, bound)
        assert np.array_equal(got, _groups(cells.tolist(), bound))
        for a, b in zip(got[:-1], got[1:]):                    # every group fits, or is one frame with cells
            assert b > a and (cells[a:b].sum() <= bound or np.count_nonzero(cells[a:b]) == 1)


def test_plan_groups_rejects_bad_arguments():
    with pytest.raises(RadarB200Error):
        device.fuse_plan_groups([1, -1], 4)
    with pytest.raises(RadarB200Error):
        device.fuse_plan_groups([1, 1], 0)
