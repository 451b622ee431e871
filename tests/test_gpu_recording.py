"""Whole recordings fed block by block (RecordingDetection) and ST-DBSCAN in time windows (rb_stdbscan_windowed).

Every comparison is bit-exact: a recording fed in blocks equals DetectionPipeline.run_device on all its frames as one
block, and windowed labels / core flags equal rb_stdbscan and the C oracle for every valid choice of windows."""
import math

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle.c_oracle import st_dbscan_c
from radar_point_cloud_tracking_b200 import synthetic as syn
from radar_point_cloud_tracking_b200._lib import RadarB200Error

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def gpu():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (no CPU fallback exists)")
    torch.cuda.set_device(0)
    from radar_point_cloud_tracking_b200 import device as dev
    return dev


def _tables(pipe, spec, F, d):
    c, s, r = pipe.spoke_tables(spec.angle_units(), spec.scale(), F, spec.bins)
    return [torch.from_numpy(t).to(d) for t in (c, s, r)]


def _same_batch(a, b):
    assert a.n == b.n
    n = a.n
    assert torch.equal(a.frame_off, b.frame_off)
    for k in ("x", "y", "inten", "gain"):
        assert torch.equal(getattr(a, k)[:n], getattr(b, k)[:n]), k


def _assert_same(rec, one):
    _same_batch(rec.raw, one.raw)
    _same_batch(rec.points, one.points)
    assert (rec.land is None) == (one.land is None)
    if one.land is not None:
        assert all(np.array_equal(a, b) for a, b in zip(rec.edges, one.edges))
        for k in ("count", "isum", "land"):
            assert torch.equal(getattr(rec, k), getattr(one, k)), k
    assert rec.n_clusters == one.n_clusters
    assert torch.equal(rec.labels, one.labels)


def _record(echo, ids, blocks, cfg, tables, **kw):
    from radar_point_cloud_tracking_b200.recording import RecordingDetection
    rec = RecordingDetection(cfg, 0, **kw)
    G = echo.shape[1]
    a = 0
    for nb in blocks:
        rec.add_block(echo[a:a + nb], *(t[a * G:(a + nb) * G] for t in tables), ids[a:a + nb])
        a += nb
    assert a == echo.shape[0]
    return rec.finish()


@pytest.mark.parametrize("dtype", ["float32", "uint8"])
def test_blocks_equal_one_block(gpu, dtype):
    from radar_point_cloud_tracking_b200.pipeline import DetectionConfig, DetectionPipeline
    spec = syn.SweepSpec(seed=31, frames=100, spokes=512, bins=1024, clutter_p=0.01, land_blobs=3, buoys=4, boats=3)
    echo = gpu.synth_echo(spec)
    if dtype == "uint8":
        echo = echo.to(torch.uint8)
    cfg = DetectionConfig(eps_time=5.0)
    pipe = DetectionPipeline(cfg, 0)
    tabs = _tables(pipe, spec, spec.frames, echo.device)
    ids = np.arange(spec.frames) * 2 + 7
    one = pipe.run_device(echo, *tabs, frame_ids=ids)
    assert one.land is not None and one.n_clusters > 0
    rec = _record(echo, ids, [1, 7, 40, 13, 1, 38], cfg, tabs, max_window_points=one.points.n // 6)
    assert len(rec.cuts) > 3                           # the clustering ran in several windows
    _assert_same(rec, one)
    rec1 = _record(echo, ids, [100], cfg, tabs)
    assert rec1.cuts.tolist() == [0, 100]
    _assert_same(rec1, one)


def test_land_decided_by_the_recording(gpu):
    """14 one-frame blocks, two of them all-zero echoes (frames with no points, and gaps in the ids): 12 frames built
    > 10, so the recording applies the land filter although no block alone would."""
    from radar_point_cloud_tracking_b200.pipeline import DetectionConfig, DetectionPipeline
    spec = syn.SweepSpec(seed=5, frames=14, spokes=512, bins=1024, clutter_p=0.01, land_blobs=3, buoys=3, boats=2)
    echo = gpu.synth_echo(spec)
    echo[3].zero_()
    echo[9].zero_()
    cfg = DetectionConfig()
    pipe = DetectionPipeline(cfg, 0)
    tabs = _tables(pipe, spec, spec.frames, echo.device)
    ids = np.array([0, 1, 2, 5, 6, 7, 8, 20, 21, 22, 23, 24, 40, 41])
    one = pipe.run_device(echo, *tabs, frame_ids=ids)
    rec = _record(echo, ids, [1] * 14, cfg, tabs)
    assert rec.frames_built == 12 and rec.land is not None
    _assert_same(rec, one)
    alone = pipe.run_device(echo[:1], *(t[:len(spec.gains)] for t in tabs), frame_ids=ids[:1])
    assert alone.land is None


def test_non_integer_intensities_take_the_ordered_path(gpu):
    from radar_point_cloud_tracking_b200.pipeline import DetectionConfig, DetectionPipeline
    spec = syn.SweepSpec(seed=8, frames=16, spokes=512, bins=1024, clutter_p=0.01, land_blobs=3, buoys=3, boats=2)
    echo = gpu.synth_echo(spec)
    echo = torch.where(echo > 0, echo + 0.375, echo)
    cfg = DetectionConfig()
    pipe = DetectionPipeline(cfg, 0)
    tabs = _tables(pipe, spec, spec.frames, echo.device)
    ids = np.arange(spec.frames)
    one = pipe.run_device(echo, *tabs, frame_ids=ids)
    rec = _record(echo, ids, [5, 6, 5], cfg, tabs)
    assert rec.land_ordered and rec.land is not None
    _assert_same(rec, one)


# ---------------------------------------------------------------------------------------- windows vs rb_stdbscan / oracle
def _scene(seed, eps_time):
    """Frame-ordered points with gaps in the frame ids, persistent buoys (clusters spanning every window), a moving boat,
    noise, and at every 9th frame c an elongated blob in frames [c, c+3) with a lone point in frame c-1 whose only core
    neighbours are in the blob: a border point whose core neighbours lie in the next window when a window ends at c."""
    rng = np.random.default_rng(seed)
    F = 150
    steps = rng.choice([1, 1, 1, 2], F)                  # gaps of at most 2: the buoys stay connected at eps_time 2
    for c in range(9, F - 3, 9):
        steps[c:c + 3] = 1                              # the lone point's frame and the blob's frames are consecutive
    ids = np.cumsum(steps) + 100
    per = []
    for f in range(F):
        pts = [rng.uniform(0, 200, (int(rng.integers(5, 30)), 2))]
        for cx, cy in ((20, 20), (150, 40), (80, 170)):
            pts.append(np.array([cx, cy]) + rng.normal(0, 0.3, (4, 2)))
        pts.append(np.array([10 + f, 100]) + rng.normal(0, 0.3, (5, 2)))
        per.append(pts)
    for c in range(9, F - 3, 9):
        x0, y0 = 30 + (c * 7) % 140, 130 + (c % 5) * 12
        line = np.stack([x0 + 0.2 * np.arange(15), np.full(15, y0)], 1)
        for f in range(c, c + 3):
            per[f].append(line)
        per[c - 1].append(np.array([[x0 - 0.95, y0]]))
    frames = [np.concatenate(p).astype(np.float32) for p in per]
    off = np.concatenate([[0], np.cumsum([len(p) for p in frames])]).astype(np.int64)
    xy = np.concatenate(frames)
    z = rng.uniform(0, 0.3, len(xy)).astype(np.float32)
    return xy, z, off, ids


def _cut_sets(F, h, rng):
    hm = max(h, 1)
    exact = list(range(0, F - hm, hm)) + [F]
    plus = list(range(0, F - hm - 1, hm + 1)) + [F]
    uneven, a = [0], 0
    while True:
        step = int(rng.integers(hm, 3 * hm + 2))
        if F - (a + step) < hm:
            break
        a += step
        uneven.append(a)
    uneven.append(F)
    return {"h": exact, "h+1": plus, "uneven": uneven, "64": list(range(0, F - 64, 64)) + [F]}


@pytest.mark.parametrize("eps_time", [2.0, 5.0, 7.5])
@pytest.mark.parametrize("dims", [2, 3])
def test_windows_match_stdbscan_and_oracle(gpu, eps_time, dims):
    from radar_point_cloud_tracking_b200.recording import stdbscan_windowed
    xy, zc, off, ids = _scene(int(eps_time * 10) + dims, eps_time)
    d = torch.device("cuda", 0)
    x, y = (torch.from_numpy(np.ascontiguousarray(xy[:, k])).to(d) for k in (0, 1))
    z = torch.from_numpy(zc).to(d) if dims == 3 else None
    t = np.repeat(ids.astype(np.float32), np.diff(off))
    eps_s, ms = 1.0, 6
    coords = np.column_stack([xy, zc]) if dims == 3 else xy
    want, want_core = st_dbscan_c(coords, t, eps_s, eps_time, ms)
    lab, core, ncl = gpu.stdbscan(x, y, z, torch.from_numpy(t).to(d), eps_s, eps_time, ms, want_core=True)
    assert np.array_equal(lab.cpu().numpy(), want) and np.array_equal(core.cpu().numpy(), want_core)
    assert ncl > 3
    h = int(math.floor(eps_time))
    F = len(ids)
    b4 = np.array([xy[:, 0].min(), xy[:, 0].max(), xy[:, 1].min(), xy[:, 1].max()], np.float32)
    for name, cuts in _cut_sets(F, h, np.random.default_rng(h)).items():
        got, gcore, gncl = stdbscan_windowed(x, y, z, off, ids, np.array(cuts), eps_s, eps_time, ms, bounds4=b4)
        assert np.array_equal(got.cpu().numpy(), want), name
        assert np.array_equal(gcore.cpu().numpy(), want_core), name
        assert gncl == ncl, name
    # the lone points: border points (not core, labelled) - some of them end up in the window before their cores
    lone = np.concatenate([np.flatnonzero((xy[off[c - 1]:off[c], 0] == np.float32(30 + (c * 7) % 140 - 0.95))) + off[c - 1]
                           for c in range(9, F - 3, 9)])
    assert len(lone) and np.all(want_core[lone] == 0) and np.all(want[lone] >= 0)
    # a buoy spans every window of the 64-frame cut set
    buoy = want[np.flatnonzero(np.hypot(xy[:, 0] - 20, xy[:, 1] - 20) < 1.5)]
    assert len(set(buoy[buoy >= 0].tolist())) == 1


def test_windows_without_points(gpu):
    """Windows whose whole local problem is empty (a stretch of empty frames longer than a window plus both halos, and
    empty frames before one frame larger than the budget, as plan_windows cuts them) give rb_stdbscan's labels."""
    from radar_point_cloud_tracking_b200.recording import plan_windows, stdbscan_windowed
    xy, _, off, ids = _scene(41, 2.0)
    gap = 30                                            # frames 70 .. 99 lose their points
    keep = np.ones(len(xy), bool)
    keep[off[70]:off[70 + gap]] = False
    per = np.diff(off)
    per[70:70 + gap] = 0
    xy = xy[keep]
    off = np.concatenate([[0], np.cumsum(per)]).astype(np.int64)
    d = torch.device("cuda", 0)
    eps_s, ms = 1.0, 6
    t = np.repeat(ids.astype(np.float32), np.diff(off))
    x, y = (torch.from_numpy(np.ascontiguousarray(xy[:, k])).to(d) for k in (0, 1))
    want, want_core = st_dbscan_c(xy, t, eps_s, 2.0, ms)
    F = len(ids)
    for cuts in ([0, 40, 75, 80, 85, 90, 110, F], list(range(0, F - 2, 2)) + [F]):
        got, gcore, ncl = stdbscan_windowed(x, y, None, off, ids, np.array(cuts), eps_s, 2.0, ms)
        assert np.array_equal(got.cpu().numpy(), want) and np.array_equal(gcore.cpu().numpy(), want_core)
        assert ncl == want.max() + 1
    # ten frames, the first nine empty, the last one above the budget: window 0 = frames [0, 7) has no points
    rng = np.random.default_rng(3)
    pts = (np.array([5.0, 5.0]) + rng.normal(0, 0.3, (100, 2))).astype(np.float32)
    off2 = np.array([0] * 10 + [100], dtype=np.int64)
    ids2 = np.arange(10)
    cuts = plan_windows(off2, 2, 50)
    assert cuts.tolist() == [0, 7, 10]
    x2, y2 = (torch.from_numpy(np.ascontiguousarray(pts[:, k])).to(d) for k in (0, 1))
    want2, core2 = st_dbscan_c(pts, np.full(100, 9, np.float32), eps_s, 2.0, ms)
    got2, gcore2, ncl2 = stdbscan_windowed(x2, y2, None, off2, ids2, cuts, eps_s, 2.0, ms)
    assert np.array_equal(got2.cpu().numpy(), want2) and np.array_equal(gcore2.cpu().numpy(), core2) and ncl2 == 1


def test_windowed_rejects_bad_input(gpu):
    from radar_point_cloud_tracking_b200.recording import stdbscan_windowed
    xy, _, off, ids = _scene(3, 2.0)
    d = torch.device("cuda", 0)
    x, y = (torch.from_numpy(np.ascontiguousarray(xy[:, k])).to(d) for k in (0, 1))
    F = len(ids)
    for o, i, c in ((off, ids, [0, 1, F]), (off, ids[::-1].copy(), [0, F]), (off, ids + 0.5, [0, F]), (off, ids, [0, F // 2, F // 2, F])):
        with pytest.raises(RadarB200Error):
            stdbscan_windowed(x, y, None, o, i, np.array(c), 1.0, 2.0, 6)


def test_recording_errors(gpu):
    from radar_point_cloud_tracking_b200.pipeline import DetectionConfig
    from radar_point_cloud_tracking_b200.recording import RecordingDetection
    spec = syn.SweepSpec(seed=2, frames=4, spokes=256, bins=512, clutter_p=0.01)
    echo = gpu.synth_echo(spec)
    rec = RecordingDetection(DetectionConfig(), 0)
    tabs = _tables(rec.pipe, spec, 2, echo.device)
    rec.add_block(echo[:2], *tabs, [10, 11])
    for bad in ([11, 12], [13, 12], [12.5, 13]):
        with pytest.raises(RadarB200Error):
            rec.add_block(echo[2:], *tabs, bad)
    rec.add_block(echo[2:], *tabs, [12, 14])
    res = rec.finish()
    assert res.frame_ids.tolist() == [10, 11, 12, 14]
    with pytest.raises(RadarB200Error):
        rec.add_block(echo[2:], *tabs, [20, 21])


def test_at_size_config5_windows(gpu):
    """2048 full-size config-5 frames (eps_time 5) in 512-frame blocks: labels in >= 4 windows equal the one-window run;
    the device cluster records equal the reference's host loop on the same recording."""
    from radar_point_cloud_tracking_b200.pipeline import DetectionConfig
    from radar_point_cloud_tracking_b200.recording import RecordingDetection, plan_windows, stdbscan_windowed
    spec = syn.SweepSpec(seed=2025, frames=2048, spokes=2048, bins=1024)
    cfg = DetectionConfig(eps_time=5.0)
    rec = RecordingDetection(cfg, 0)
    tabs = None
    for a in range(0, spec.frames, 512):
        echo = gpu.synth_echo(spec, a, 512)
        if tabs is None:
            tabs = _tables(rec.pipe, spec, 512, echo.device)
        rec.add_block(echo, *tabs, np.arange(a, a + 512))
        del echo
    res = rec.finish()
    assert res.cuts.tolist() == [0, spec.frames] and res.land is not None and res.n_clusters > 0
    p = res.points
    off = p.frame_off.cpu().numpy()
    cuts = plan_windows(off, 5, p.n // 5)
    assert len(cuts) - 1 >= 4
    lab, core, ncl = stdbscan_windowed(p.x, p.y, None, off, res.frame_ids, cuts, cfg.eps_space, cfg.eps_time, cfg.min_samples,
                                       bounds4=None)
    assert ncl == res.n_clusters
    assert torch.equal(lab, res.labels) and torch.equal(core, res.core)
    host = res.to_host()
    dev_c, host_c = res.clusters_by_frame(host), res.clusters_by_frame_host(host)
    assert list(dev_c) == list(host_c)
    for fid in host_c:
        a, b = dev_c[fid], host_c[fid]
        assert [c.cluster_id for c in a] == [c.cluster_id for c in b]
        for ca, cb in zip(a, b):
            assert np.array_equal(ca.points, cb.points) and np.array_equal(ca.centroid, cb.centroid)
