"""Host-side parts of whole-recording detection (no GPU): frame-id and cut validation, the window planner, and the
library's zone pairing against the sharded driver's numpy version."""
import ctypes as C

import numpy as np
import pytest

from radar_point_cloud_tracking_b200 import _lib
from radar_point_cloud_tracking_b200._lib import RadarB200Error
from radar_point_cloud_tracking_b200.recording import check_frame_ids, plan_windows
from radar_point_cloud_tracking_b200.sharded import pair_zone_runs

RB_ERR_ARG = -2


def _windowed_rc(frame_off, ids, cuts, eps_time=2.0):
    """rb_stdbscan_windowed without a context: the input checks run first, so a valid input fails only at 'ctx is NULL'."""
    lib = _lib.load()
    off = np.ascontiguousarray(frame_off, dtype=np.int64)
    fid = np.ascontiguousarray(ids, dtype=np.float32)
    cu = np.ascontiguousarray(cuts, dtype=np.int64)
    rc = lib.rb_stdbscan_windowed(None, None, None, None, 1, off.ctypes.data, fid.ctypes.data, len(fid), cu.ctypes.data, len(cu) - 1,
                                  8.0, float(eps_time), 15, None, None, None, None, None)
    return rc, lib.rb_last_error().decode()


def test_windowed_input_checks():
    off = np.arange(0, 11 * 5, 5)                       # 10 frames of 5 points
    ids = np.arange(10) + 100
    rc, msg = _windowed_rc(off, ids, [0, 4, 10])
    assert rc == RB_ERR_ARG and "ctx is NULL" in msg     # everything about the input is fine
    for bad_ids, what in ((np.r_[ids[:5], ids[4], ids[6:]], "increase"), (ids + 0.5, "integer"), (ids + (1 << 24), "2^24")):
        rc, msg = _windowed_rc(off, bad_ids, [0, 10])
        assert rc == RB_ERR_ARG and what in msg, msg
    for cuts, what in (([0, 5, 5, 10], "increase"), ([1, 10], "from 0"), ([0, 9], "from 0"), ([0, 1, 10], "floor(eps_time)")):
        rc, msg = _windowed_rc(off, ids, cuts)
        assert rc == RB_ERR_ARG and what in msg, msg
    rc, msg = _windowed_rc(off, ids, [0, 2, 10])        # windows of exactly h = 2 frames are fine
    assert "ctx is NULL" in msg
    rc, msg = _windowed_rc(off, ids, [0, 1, 10], eps_time=0.5)
    assert "ctx is NULL" in msg


def test_check_frame_ids():
    assert check_frame_ids([3, 5, 9]).tolist() == [3, 5, 9]
    assert check_frame_ids(np.array([3.0, 4.0]), after=2).tolist() == [3, 4]
    for bad, after in (([1, 1], None), ([2, 1], None), ([1.5, 2], None), ([5, 6], 5), ([1 << 24], None), ([], None)):
        with pytest.raises(RadarB200Error):
            check_frame_ids(bad, after)


@pytest.mark.parametrize("seed", range(6))
def test_plan_windows(seed):
    rng = np.random.default_rng(seed)
    F = int(rng.integers(1, 300))
    per = rng.integers(0, 50, F)
    per[rng.random(F) < 0.1] = 0                         # frames without points
    off = np.concatenate([[0], np.cumsum(per)]).astype(np.int64)
    for h in (0, 1, 2, 5, 7):
        assert plan_windows(off, h, int(off[-1])).tolist() == [0, F]          # fits: one window
        budget = int(rng.integers(1, max(2, off[-1])))
        cuts = plan_windows(off, h, budget)
        assert cuts[0] == 0 and cuts[-1] == F and np.all(np.diff(cuts) > 0)
        if len(cuts) > 2:
            assert np.all(np.diff(cuts) >= max(h, 1))
        for a, b in zip(cuts[:-1], cuts[1:]):
            local = off[min(b + h, F)] - off[max(a - h, 0)]
            shortest = off[min(a + max(h, 1) + h, F)] - off[max(a - h, 0)]
            # within the budget unless even the shortest legal window exceeds it, or the tail had to be merged
            assert local <= budget or shortest > budget or b == F


def _random_rle(rng, length, core):
    """Run-length encoding (keys, starts) of a zone of `length` points whose core pattern is `core`."""
    keys = np.where(core, rng.integers(0, 40, length), -1)
    flag = np.ones(length, bool)
    flag[1:] = keys[1:] != keys[:-1]
    starts = np.flatnonzero(flag)
    return keys[starts].astype(np.int64), starts.astype(np.int64)


@pytest.mark.parametrize("seed", range(20))
def test_pair_zone_runs_matches_numpy(seed):
    rng = np.random.default_rng(seed)
    lib = _lib.load()
    length = int(rng.integers(0, 200))
    core = rng.random(length) < rng.random()
    # runs of equal keys, so that the encodings are short
    ka, sa = _random_rle(rng, length, core)
    kb, sb = _random_rle(rng, length, core)
    want_a, want_b = pair_zone_runs(ka, sa, kb, sb)
    ptr = lambda a: a.ctypes.data if len(a) else None
    m = lib.rb_pair_zone_runs(ptr(ka), ptr(sa), len(ka), ptr(kb), ptr(sb), len(kb), None, None, 0)
    assert m == len(want_a)
    pa, pb = np.zeros(max(m, 1), np.int64), np.zeros(max(m, 1), np.int64)
    assert lib.rb_pair_zone_runs(ptr(ka), ptr(sa), len(ka), ptr(kb), ptr(sb), len(kb), pa.ctypes.data, pb.ctypes.data, m) == m
    assert np.array_equal(pa[:m], want_a) and np.array_equal(pb[:m], want_b)


def test_pair_zone_runs_rejects_disagreeing_cores():
    lib = _lib.load()
    ka, sa = np.array([5, -1], np.int64), np.array([0, 3], np.int64)
    kb, sb = np.array([7], np.int64), np.array([0], np.int64)
    with pytest.raises(RadarB200Error):
        pair_zone_runs(ka, sa, kb, sb)
    assert lib.rb_pair_zone_runs(ka.ctypes.data, sa.ctypes.data, 2, kb.ctypes.data, sb.ctypes.data, 1, None, None, 0) == RB_ERR_ARG


def test_plan_windows_over_empty_frames():
    """Empty frames before a frame larger than the budget: the planner may leave a window whose local problem has no
    points at all (here frames [0, 9) of window 0) - a valid cut that rb_stdbscan_windowed must take."""
    off = np.array([0] * 10 + [100], dtype=np.int64)
    cuts = plan_windows(off, 2, 50)
    assert cuts.tolist() == [0, 7, 10]
    a, b = cuts[0], cuts[1]
    assert off[min(b + 2, 10)] - off[max(a - 2, 0)] == 0
    rc, msg = _windowed_rc(off, np.arange(10), cuts)
    assert "ctx is NULL" in msg                         # accepted by the input checks
