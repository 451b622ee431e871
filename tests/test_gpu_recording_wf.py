"""The PointCloudWorkF ST-DBSCAN variant (min_frames core test + order-dependent border rule) over whole recordings:
rb_stdbscan_windowed_wf, DetectionConfig.min_frames through RecordingDetection and the block pipelines.

Every comparison is bit-exact against rb_stdbscan_wf on the same points with times = frame ids, and the windowed entry
also against the C oracle. Two hand-built scenes pin the case that makes the variant hard in windows: a cluster's start
(its smallest core index over the whole recording) lying outside the part of the cluster that a window sees."""
import math

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle.c_oracle import st_dbscan_c, st_dbscan_wf_c
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


@pytest.fixture(params=["auto", "general"])
def dbscan_mode(request, gpu):
    """Both ST-DBSCAN algorithms: auto (tight-cell buckets, integer times) and the general point-level one."""
    from radar_point_cloud_tracking_b200 import _lib
    ctx = _lib.context(0)
    ctx.set_option("dbscan_mode", 0 if request.param == "auto" else 1)
    yield request.param
    ctx.set_option("dbscan_mode", 0)


def _dev_xy(xy, z=None):
    d = torch.device("cuda", 0)
    x, y = (torch.from_numpy(np.ascontiguousarray(xy[:, k], dtype=np.float32)).to(d) for k in (0, 1))
    return x, y, (torch.from_numpy(np.ascontiguousarray(z, dtype=np.float32)).to(d) if z is not None else None)


def _flat_wf(gpu, x, y, z, off, ids, eps_s, eps_t, ms, mf):
    """rb_stdbscan_wf on the same points, times = frame ids: (labels, core, n_clusters) on the host."""
    t = np.repeat(np.asarray(ids, np.float32), np.diff(off))
    lab, core, ncl = gpu.stdbscan(x, y, z, torch.from_numpy(t).to(x.device), eps_s, eps_t, ms, want_core=True, min_frames=mf)
    return lab.cpu().numpy(), core.cpu().numpy(), ncl


# ---------------------------------------------------------------------------- rb_stdbscan_windowed_wf vs flat and oracle
def _scene(seed):
    """Frame-ordered points: gaps in the frame ids, buoys that miss frames, a slow boat, noise, clumps seen in one frame
    only (core points for T4, not with min_frames >= 2), and a stretch of 32 frames without points."""
    rng = np.random.default_rng(seed)
    F = 180
    ids = np.cumsum(rng.choice([1, 1, 1, 2], F)) + 100
    per = []
    for f in range(F):
        if 100 <= f < 132:
            per.append(np.zeros((0, 2)))
            continue
        pts = [rng.uniform(0, 200, (int(rng.integers(5, 30)), 2))]
        for cx, cy in ((20, 20), (150, 40), (80, 170)):
            if rng.random() < 0.8:
                pts.append(np.array([cx, cy]) + rng.normal(0, 0.3, (4, 2)))
        pts.append(np.array([10 + 0.5 * f, 100]) + rng.normal(0, 0.3, (5, 2)))
        if rng.random() < 0.3:
            pts.append(rng.uniform(20, 180, 2) + rng.normal(0, 0.2, (8, 2)))
        per.append(np.concatenate(pts))
    off = np.concatenate([[0], np.cumsum([len(p) for p in per])]).astype(np.int64)
    xy = np.concatenate(per).astype(np.float32)
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
    return {"one": [0, F], "h": exact, "h+1": plus, "uneven": uneven}


def _empty_windows(off, cuts, h):
    F = len(off) - 1
    return sum(off[min(b + h, F)] == off[max(a - h, 0)] for a, b in zip(cuts[:-1], cuts[1:]))


@pytest.mark.parametrize("min_frames", [2, 3, 4])
@pytest.mark.parametrize("eps_time", [2.0, 5.0, 7.5])
@pytest.mark.parametrize("dims", [2, 3])
def test_windowed_wf_matches_flat_and_oracle(gpu, dbscan_mode, eps_time, dims, min_frames):
    from radar_point_cloud_tracking_b200.recording import stdbscan_windowed
    xy, zc, off, ids = _scene(int(eps_time * 10) + dims + 7 * min_frames)
    x, y, z = _dev_xy(xy, zc if dims == 3 else None)
    eps_s, ms = 1.0, 6
    coords = np.column_stack([xy, zc]) if dims == 3 else xy
    t = np.repeat(ids.astype(np.float32), np.diff(off))
    want, want_core = st_dbscan_wf_c(coords, t, eps_s, eps_time, ms, min_frames)
    flat, flat_core, flat_ncl = _flat_wf(gpu, x, y, z, off, ids, eps_s, eps_time, ms, min_frames)
    assert np.array_equal(flat, want) and np.array_equal(flat_core, want_core.astype(np.uint8))
    assert flat_ncl == want.max() + 1 > 3
    assert not np.array_equal(want, st_dbscan_c(coords, t, eps_s, eps_time, ms)[0])      # the variant labels differently
    h = int(math.floor(eps_time))
    b4 = np.array([xy[:, 0].min(), xy[:, 0].max(), xy[:, 1].min(), xy[:, 1].max()], np.float32)
    sets = _cut_sets(len(ids), h, np.random.default_rng(h + min_frames))
    assert _empty_windows(off, sets["h"], h) > 0
    for name, cuts in sets.items():
        for hint in (b4, None):
            got, gcore, gncl = stdbscan_windowed(x, y, z, off, ids, np.array(cuts), eps_s, eps_time, ms, bounds4=hint,
                                                 min_frames=min_frames)
            assert np.array_equal(got.cpu().numpy(), want), name
            assert np.array_equal(gcore.cpu().numpy(), flat_core), name
            assert gncl == flat_ncl, name


# ---------------------------------------------------------------------- the cluster's start outside a window's component
FA, FB, H, F_SCENE = 4, 8, 2, 13              # window 1 owns frames [4, 8); its local problem is frames [2, 10)


def _stack(x, y):
    return [(x, y), (x, y + 0.1), (x, y + 0.2)]


def _start_scene(kind):
    """Cluster C = branches P (a stack at x = 0) and Q (a stack at x = 10) that a bridge joins only in frames 10 and 11,
    beyond window 1's local problem; cluster D (frames 0-2) comes first. b = a lone point in frame FA whose only core
    neighbour is a point q of Q.
      A: C starts at s in frame FA-1 (P); Q's first core is in frame FA+1, q is a later one (frame FA+2). Window 1 sees
         Q alone, keyed by its first core > b, and q is not that key - yet C started before b: b joins C.
      B: C starts at s in frame FA, after b; q is Q's first core (frame FA+1): window 1's key of Q. C started after b
         and q is not its start: b stays noise.
    Returns points, frame offsets, ids and the indices of b, s and q."""
    frames = [[] for _ in range(F_SCENE)]
    for f in range(3):
        frames[f] += _stack(50.0, 50.0)
    p_first = FA - 1 if kind == "A" else FA
    if kind == "B":
        frames[FA].append((10.0, -1.5))                                  # b, before s in frame FA
    for f in range(p_first, F_SCENE):
        frames[f] += _stack(0.0, 0.0)
    if kind == "A":
        frames[FA].append((10.0, -1.6))                                  # b
    else:
        frames[FA + 1].append((10.0, -0.6))                              # q = Q's first core
    for f in range(FA + 1, F_SCENE):
        frames[f] += _stack(10.0, 0.0)
    if kind == "A":
        frames[FA + 2].append((10.0, -0.7))                              # q, a later core of Q
    for f in (10, 11):
        frames[f] += [(0.4 * k, 0.0) for k in range(1, 25)]              # the bridge
    off = np.concatenate([[0], np.cumsum([len(fr) for fr in frames])]).astype(np.int64)
    xy = np.array([p for fr in frames for p in fr], np.float32)

    def at(f, p):
        return int(off[f]) + frames[f].index(p)
    b = at(FA, (10.0, -1.6) if kind == "A" else (10.0, -1.5))
    s = at(p_first, (0.0, 0.0))
    q = at(FA + 2, (10.0, -0.7)) if kind == "A" else at(FA + 1, (10.0, -0.6))
    return xy, off, np.arange(F_SCENE) + 50, b, s, q


@pytest.mark.parametrize("kind", ["A", "B"])
def test_cluster_start_outside_the_window(gpu, dbscan_mode, kind):
    from radar_point_cloud_tracking_b200.recording import stdbscan_windowed
    xy, off, ids, b, s, q = _start_scene(kind)
    eps_s, eps_t, ms, mf = 1.0, float(H), 5, 2
    t = np.repeat(ids.astype(np.float32), np.diff(off))
    want, want_core = st_dbscan_wf_c(xy, t, eps_s, eps_t, ms, mf)
    assert want_core[s] and want_core[q] and not want_core[b]
    assert want[s] == want[q] == 1 and want.max() == 1                   # D = 0, C = 1 (P and Q joined by the bridge)
    assert q > b and (s < b if kind == "A" else s > b)
    assert want[b] == (1 if kind == "A" else -1)
    x, y, _ = _dev_xy(xy)
    flat, flat_core, flat_ncl = _flat_wf(gpu, x, y, None, off, ids, eps_s, eps_t, ms, mf)
    assert np.array_equal(flat, want) and np.array_equal(flat_core, want_core.astype(np.uint8)) and flat_ncl == 2
    for cuts in ([0, FA, FB, F_SCENE], [0, FA, FB, 10, F_SCENE], [0, F_SCENE]):
        got, gcore, gncl = stdbscan_windowed(x, y, None, off, ids, np.array(cuts), eps_s, eps_t, ms, min_frames=mf)
        got = got.cpu().numpy()
        assert got[b] == want[b], cuts
        assert np.array_equal(got, want) and np.array_equal(gcore.cpu().numpy(), flat_core) and gncl == 2, cuts


# ------------------------------------------------------------------------------------ DetectionConfig.min_frames end to end
def _tables(pipe, spec, F, d):
    c, s, r = pipe.spoke_tables(spec.angle_units(), spec.scale(), F, spec.bins)
    return [torch.from_numpy(t).to(d) for t in (c, s, r)]


def _record(echo, ids, blocks, cfg, tables, **kw):
    from radar_point_cloud_tracking_b200.recording import RecordingDetection
    rec = RecordingDetection(cfg, 0, **kw)
    G = echo.shape[1]
    a = 0
    for nb in blocks:
        rec.add_block(echo[a:a + nb], *(t[a * G:(a + nb) * G] for t in tables), ids[a:a + nb])
        a += nb
    return rec.finish()


def _assert_wf(gpu, res, cfg, core=True):
    """res's labels (and core flags) = rb_stdbscan_wf on its own filtered points with times = its frame ids."""
    p = res.points
    n = p.n
    off = p.frame_off.cpu().numpy()
    lab, fcore, ncl = _flat_wf(gpu, p.x[:n], p.y[:n], p.inten[:n] if cfg.cluster_3d else None, off, res.frame_ids,
                               cfg.eps_space, cfg.eps_time, cfg.min_samples, cfg.min_frames)
    assert res.n_clusters == ncl
    assert np.array_equal(res.labels[:n].cpu().numpy(), lab)
    if core:
        assert np.array_equal(res.core.cpu().numpy(), fcore)
    return lab


SPEC = dict(seed=31, frames=100, spokes=512, bins=1024, clutter_p=0.01, land_blobs=3, buoys=4, boats=3)


@pytest.mark.parametrize("dtype", ["float32", "uint8"])
def test_recording_blocks_and_windows(gpu, dbscan_mode, dtype):
    from radar_point_cloud_tracking_b200.pipeline import DetectionConfig, DetectionPipeline
    spec = syn.SweepSpec(**SPEC)
    echo = gpu.synth_echo(spec)
    if dtype == "uint8":
        echo = echo.to(torch.uint8)
    cfg = DetectionConfig(eps_time=5.0, min_frames=3)
    tabs = _tables(DetectionPipeline(cfg, 0), spec, spec.frames, echo.device)
    ids = np.arange(spec.frames) * 2 + 7
    one = _record(echo, ids, [100], cfg, tabs)
    assert one.cuts.tolist() == [0, 100] and one.land is not None
    lab = _assert_wf(gpu, one, cfg)
    assert one.n_clusters > 0
    t4 = _record(echo, ids, [100], DetectionConfig(eps_time=5.0), tabs)
    assert not np.array_equal(t4.labels.cpu().numpy(), lab)               # min_frames changed the clustering
    rec = _record(echo, ids, [1, 7, 40, 13, 1, 38], cfg, tabs, max_window_points=one.points.n // 6)
    assert len(rec.cuts) > 3
    assert torch.equal(rec.labels, one.labels) and torch.equal(rec.core, one.core) and rec.n_clusters == one.n_clusters


def test_recording_csv_frames(gpu, tmp_path):
    from radar_point_cloud_tracking_b200.pipeline import DetectionConfig
    from radar_point_cloud_tracking_b200.recording import RecordingDetection
    spec = syn.SweepSpec(seed=41, frames=14, spokes=256, bins=512, clutter_p=0.02, land_blobs=2, buoys=3, boats=2)
    files = syn.write_csv_tree(spec, tmp_path)
    cfg = DetectionConfig(eps_time=3.0, min_frames=2)
    res = []
    for k in range(2):                                  # one window, then at most a quarter of the points per window
        rec = RecordingDetection(cfg, 0, max_window_points=res[0].points.n // 4 if res else None)
        rec.add_csv_frames(files, num_echo_columns=spec.bins)
        res.append(rec.finish())
    one, win = res
    assert one.land is not None and one.n_clusters > 0 and one.cuts.tolist() == [0, spec.frames] and len(win.cuts) > 2
    _assert_wf(gpu, one, cfg)
    assert torch.equal(win.labels, one.labels) and torch.equal(win.core, one.core) and win.n_clusters == one.n_clusters


def test_block_pipelines(gpu, dbscan_mode):
    from radar_point_cloud_tracking_b200.pipeline import DetectionConfig, DetectionPipeline, OverlappedPipeline
    spec = syn.SweepSpec(**SPEC)
    echo = gpu.synth_echo(spec)
    cfg = DetectionConfig(eps_time=5.0, min_frames=3)
    pipe = DetectionPipeline(cfg, 0)
    tabs = _tables(pipe, spec, spec.frames, echo.device)
    ids = np.arange(spec.frames) + 3
    dev_res = pipe.run_device(echo, *tabs, frame_ids=ids)
    lab = _assert_wf(gpu, dev_res, cfg, core=False)
    assert dev_res.n_clusters > 0
    staged = pipe.run_device_staged(echo, *tabs, frame_ids=ids)
    _assert_wf(gpu, staged, cfg, core=False)
    assert torch.equal(staged.labels, dev_res.labels)
    host = pipe.run_host(echo.cpu().numpy(), spec.angle_units(), spec.scale(), ids)
    assert np.array_equal(host["labels"], lab) and host["n_clusters"] == dev_res.n_clusters
    G = len(cfg.gains)
    cuts = [0, 30, 31, 70, 100]
    ov = OverlappedPipeline(cfg, 0, workers=2)
    try:
        blocks = [((echo[a:b], *(t[a * G:b * G] for t in tabs)), {"frame_ids": ids[a:b]}) for a, b in zip(cuts[:-1], cuts[1:])]
        outs = ov.map(blocks)
    finally:
        ov.close()
    torch.cuda.synchronize()
    for r in outs:
        _assert_wf(gpu, r, cfg, core=False)


def test_at_size_config5_windows(gpu):
    """2048 full-size config-5 frames (eps_time 5, min_frames 3) in 512-frame blocks: labels and core flags in >= 4
    windows equal the one-window run (rb_stdbscan_wf)."""
    from radar_point_cloud_tracking_b200.pipeline import DetectionConfig
    from radar_point_cloud_tracking_b200.recording import RecordingDetection, plan_windows, stdbscan_windowed
    spec = syn.SweepSpec(seed=2025, frames=2048, spokes=2048, bins=1024)
    cfg = DetectionConfig(eps_time=5.0, min_frames=3)
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
                                       min_frames=cfg.min_frames)
    assert ncl == res.n_clusters
    assert torch.equal(lab, res.labels) and torch.equal(core, res.core)


# ------------------------------------------------------------------------------------------------------------------ errors
def test_errors(gpu):
    import ctypes as C

    from radar_point_cloud_tracking_b200 import _lib
    from radar_point_cloud_tracking_b200.pipeline import DetectionConfig
    from radar_point_cloud_tracking_b200.recording import stdbscan_windowed
    from radar_point_cloud_tracking_b200.sharded import ShardedDetection
    for kw in (dict(min_frames=0), dict(min_frames=2, eps_time=31.0)):
        with pytest.raises(RadarB200Error):
            DetectionConfig(**kw)
    xy, off, ids, *_ = _start_scene("A")
    x, y, _ = _dev_xy(xy)
    n = len(xy)
    lab = torch.full((n,), 7, dtype=torch.int32, device=x.device)
    ctx = _lib.context(0)
    o = np.ascontiguousarray(off, np.int64)
    i = np.ascontiguousarray(ids, np.float32)
    cu = np.array([0, FA, FB, F_SCENE], np.int64)
    for eps_t, mf in ((2.0, 0), (2.0, -1), (31.0, 2), (float("nan"), 2)):
        ncl = C.c_int64(5)
        rc = ctx.lib.rb_stdbscan_windowed_wf(ctx.handle, _lib.ptr(x), _lib.ptr(y), None, 1, o.ctypes.data, i.ctypes.data, len(i),
                                             cu.ctypes.data, len(cu) - 1, 1.0, eps_t, 5, mf, None, _lib.ptr(lab), None, C.byref(ncl),
                                             _lib.stream_ptr())
        assert rc == -2 and ncl.value == 0                               # RB_ERR_ARG, nothing enqueued
        with pytest.raises(RadarB200Error):
            stdbscan_windowed(x, y, None, off, ids, cu, 1.0, eps_t, 5, min_frames=mf)
    torch.cuda.synchronize()
    assert torch.all(lab == 7)
    with pytest.raises(RadarB200Error):                                  # cuts shorter than floor(eps_time) frames
        stdbscan_windowed(x, y, None, off, ids, np.array([0, 1, F_SCENE]), 1.0, 2.0, 5, min_frames=2)
    with pytest.raises(RadarB200Error):
        ShardedDetection(DetectionConfig(min_frames=2), rank=0, world=1, device=0)
