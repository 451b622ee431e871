"""Host-side pieces of the multi-GPU recording (no GPU): frame shares, windows over a rank's owned frames between its
halos, the stitch of window encodings spread over ranks, the decisions taken from the gathered statistics, and the
input checks of the three windowed pass entries."""
import ctypes as C

import numpy as np
import pytest

from radar_point_cloud_tracking_b200 import _lib
from radar_point_cloud_tracking_b200._lib import RadarB200Error
from radar_point_cloud_tracking_b200.recording import plan_windows
from radar_point_cloud_tracking_b200.sharded import (check_recording_stats, cluster_starts, split_frames, stitch_windows,
                                                     window_payload)

RB_ERR_ARG = -2


def test_split_frames():
    for n, world in ((21, 3), (20000, 8), (5, 5), (7, 2), (0, 2)):
        shares = [split_frames(n, world, r) for r in range(world)]
        assert shares[0][0] == 0 and shares[-1][1] == n
        assert all(a[1] == b[0] for a, b in zip(shares[:-1], shares[1:]))
        sizes = [b - a for a, b in shares]
        assert max(sizes) - min(sizes) <= 1 and sizes == sorted(sizes, reverse=True)
    with pytest.raises(RadarB200Error):
        split_frames(10, 2, 2)


@pytest.mark.parametrize("seed", range(6))
def test_plan_windows_over_owned_frames(seed):
    rng = np.random.default_rng(seed)
    for h in (0, 1, 2, 5, 7):
        hl, hr = (h, h) if seed % 3 == 0 else (h, 0) if seed % 3 == 1 else (0, h)
        own = int(rng.integers(max(h, 1), 120))
        F = hl + own + hr
        per = rng.integers(0, 40, F)
        per[rng.random(F) < 0.1] = 0
        off = np.concatenate([[0], np.cumsum(per)]).astype(np.int64)
        fa, fb = hl, hl + own
        assert plan_windows(off, h, int(off[-1]), own=(fa, fb)).tolist() == [fa, fb]       # fits, halos included
        for budget in (1, int(off[-1]) // 7 + 1, int(off[-1]) // 3 + 1, int(off[-1]) - 1):
            cuts = plan_windows(off, h, budget, own=(fa, fb))
            assert cuts[0] == fa and cuts[-1] == fb and np.all(np.diff(cuts) > 0)
            hmin = max(h, 1)
            if len(cuts) > 2:
                assert np.all(np.diff(cuts) >= hmin)
            for a, b in zip(cuts[:-1], cuts[1:]):
                local = off[min(b + h, F)] - off[max(a - h, 0)]                          # the halo frames count
                assert local <= budget or b - a <= 2 * hmin - 1
        # the whole recording as the owned range is plan_windows itself
        assert np.array_equal(plan_windows(off, h, int(off[-1]) // 4 + 1, own=(0, F)), plan_windows(off, h, int(off[-1]) // 4 + 1))
    with pytest.raises(RadarB200Error):
        plan_windows(np.arange(5), 1, 10, own=(3, 3))


# two windows: window 0's own last frames (2 core points, key 0) are window 1's left halo (key 4); window 0's right halo
# (a non-core point, then a core point, key 0) is window 1's own first frames (key 4); window 1 has a second component 9
HEAD0 = [0, 0, 1, 3, 4, 0, 0, 2, 2]
ENT0 = ([0, -1, 0, 0], [0, 0, 1, 0])
HEAD1 = [1, 3, 3, 3, 5, 2, 2, 0, 0]
ENT1 = ([4, -1, 4, 4, 9], [0, 0, 1, 0, 0])


def _pad(rows):
    w = max(len(r) for r in rows)
    return np.stack([np.concatenate([r, np.zeros(w - len(r), np.int64)]) for r in rows])


def test_stitch_windows_across_ranks():
    one = window_payload(np.array([HEAD0, HEAD1]), [*ENT0, *ENT1])
    tk, ti, ncl = stitch_windows(one[None])
    assert tk.tolist() == [0, 4, 9] and ti.tolist() == [0, 0, 1] and ncl == 2
    # the same windows on two ranks (window 0 on rank 0, window 1 on rank 1), padded as the all-gather pads them
    two = _pad([window_payload(np.array([HEAD0]), list(ENT0)), window_payload(np.array([HEAD1]), list(ENT1))])
    for got in (stitch_windows(two), stitch_windows(_pad([two[0], np.array([0], np.int64), two[1]]))):   # a rank without windows
        assert got[0].tolist() == tk.tolist() and got[1].tolist() == ti.tolist() and got[2] == ncl
    assert cluster_starts(tk, ti, ncl).tolist() == [0, 9]
    bad = list(HEAD1)
    bad[5] = 3                                                   # window 1's left halo is longer than window 0's own last
    with pytest.raises(RadarB200Error, match="do not match"):
        stitch_windows(_pad([window_payload(np.array([HEAD0]), list(ENT0)), window_payload(np.array([bad]), list(ENT1))]))


def _stats(frames, first, last, built=None, points=None):
    n = len(frames)
    built = frames if built is None else built
    points = [10 * f for f in frames] if points is None else points
    return np.array([[frames[r], built[r], points[r], 0, 1, 0, 1, first[r], last[r]] for r in range(n)], np.float64)


def test_check_recording_stats():
    check_recording_stats(_stats([5, 9, 7], [0, 5, 14], [4, 13, 20]), True, 5)
    check_recording_stats(_stats([5, 0, 7], [0, 0, 14], [4, 0, 20]), False, 5)           # no clustering: an empty rank is fine
    with pytest.raises(RadarB200Error, match="empty recording"):
        check_recording_stats(_stats([0, 0], [0, 0], [0, 0]), False, 2)
    with pytest.raises(RadarB200Error, match="rank 1 holds 4 frames, fewer than the 5"):
        check_recording_stats(_stats([7, 4, 10], [0, 7, 11], [6, 10, 20]), True, 5)
    with pytest.raises(RadarB200Error, match="fewer than the 1"):
        check_recording_stats(_stats([3, 0], [0, 0], [2, 0]), True, 0)
    with pytest.raises(RadarB200Error, match="rank 2's first id 9 is not above rank 0's last id 9"):
        check_recording_stats(_stats([10, 0, 11], [0, 0, 9], [9, 0, 19]), False, 2)
    with pytest.raises(RadarB200Error, match="64 frames"):
        check_recording_stats(_stats([70, 70], [0, 70], [69, 139]), True, 65)


def _pass_rc(entry, off, ids, own, cuts, eps_time=2.0, extra=()):
    """A pass entry without a context: the input checks run first, so a valid input fails only at 'ctx is NULL'."""
    lib = _lib.load()
    o = np.ascontiguousarray(off, dtype=np.int64)
    f = np.ascontiguousarray(ids, dtype=np.float32)
    cu = np.ascontiguousarray(cuts, dtype=np.int64)
    fn = getattr(lib, entry)
    rc = fn(None, None, None, None, 1, o.ctypes.data, f.ctypes.data, len(f), own[0], own[1], cu.ctypes.data, len(cu) - 1, 0, 8.0,
            float(eps_time), 15, 0, None, *extra)
    return rc, lib.rb_last_error().decode()


def test_pass_entries_input_checks():
    off = np.arange(0, 11 * 5, 5)                                # 10 local frames of 5 points: halo 2 | owned 6 | halo 2
    ids = np.arange(10) + 100
    cores = lambda own, cuts, **kw: _pass_rc("rb_stdbscan_windowed_pass_cores", off, ids, own, cuts, extra=(None, None), **kw)
    rc, msg = cores((2, 8), [2, 5, 8])
    assert rc == RB_ERR_ARG and "ctx is NULL" in msg
    for own, cuts, what in (((2, 8), [0, 5, 10], "from 0"), ((2, 8), [2, 3, 8], "floor(eps_time)"), ((5, 5), [5, 5], "owned frames"),
                            ((2, 11), [2, 11], "owned frames")):
        rc, msg = cores(own, cuts)
        assert rc == RB_ERR_ARG and what in msg, msg
    keys = lambda own, cuts, left, right: _pass_rc("rb_stdbscan_windowed_pass_keys", off, ids, own, cuts,
                                                   extra=(left, right, None, 0, 1, 4, C.c_void_p(1), None, None))
    rc, msg = keys((2, 8), [2, 8], 1, 1)
    assert "ctx is NULL" in msg
    rc, msg = keys((1, 9), [1, 9], 1, 0)                         # one halo frame where eps_time needs two
    assert rc == RB_ERR_ARG and "left halo" in msg, msg
    labels = _pass_rc("rb_stdbscan_windowed_pass_labels", off, ids, (2, 8), [2, 8],
                      extra=(None, None, None, 0, None, 0, None, None))
    assert "ctx is NULL" in labels[1]
