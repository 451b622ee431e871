"""Detection beyond the 0.125 NM range: the radar's range setting (the CSV's Scale column) decides how large the land
grid is, which land accumulation kernel runs, whether the block driver has to renegotiate its grid capacity and how
coarse ST-DBSCAN's cell table becomes.

    0.125 NM (231.5 m)   93 x 94 land cells      shared-memory histogram, first grid guess
    0.25 NM  (463 m)     185 x 186               global atomics, the block driver grows its grid
    1.5 NM   (2778 m)    1103 x 1106 (~10 MB)    global atomics; ST-DBSCAN's general grid coarsens past eps

Every comparison is bit for bit (no tolerance): the numpy / C oracles, or a float64 torch restatement where the oracle
would be too slow. Each test also asserts that it took the path it targets (``land_last_variant``, the pipeline's grid
hint, ``stdbscan_stats()``), so a later change of a threshold cannot silently remove the coverage."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle import numpy_oracle as O
from oracle.c_oracle import st_dbscan_c
from radar_point_cloud_tracking_b200 import synthetic as syn

pytestmark = pytest.mark.gpu

NM = {0.125: 231.5, 0.25: 463.0, 0.5: 926.0, 1.0: 1852.0, 1.5: 2778.0}
SHARED, GLOBAL, ORDERED = 1, 2, 3                     # land_last_variant


@pytest.fixture(scope="module")
def gpu():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (no CPU fallback exists)")
    torch.cuda.set_device(0)
    from radar_point_cloud_tracking_b200 import device as dev
    return dev


@pytest.fixture(params=["auto", "registers"])
def mask_variant(request, gpu):
    """Both spoke mask kernels: the default (TMA-staged whenever the sweep's cells fill 16-byte vectors) and the
    register-staged one."""
    from radar_point_cloud_tracking_b200 import _lib
    ctx = _lib.context(0)
    ctx.set_option("spoke_mask_variant", 0 if request.param == "auto" else 1)
    yield request.param
    ctx.set_option("spoke_mask_variant", 0)


def _info(key):
    from radar_point_cloud_tracking_b200 import _lib
    return _lib.context(0).info(key)


def _ctas_per_sm(nxe, nye):
    """rb_land_accumulate's choice (land.cu): CTAs per SM of the shared-memory histogram, 0 = the global-atomics kernel."""
    smem = (nxe - 1) * (nye - 1) * 8 + (nxe + nye) * 8
    if smem > 220 * 1024:
        return 0
    return 3 if smem <= 72 * 1024 else (2 if smem <= 110 * 1024 else 1)


def _add_at(x, y, inten, xe, ye):
    ix, iy = O.cell_index(x, xe, len(xe) - 1), O.cell_index(y, ye, len(ye) - 1)
    count = np.zeros((len(xe) - 1, len(ye) - 1), np.int32)
    isum = np.zeros(count.shape, np.float64)
    np.add.at(count, (ix, iy), 1)
    np.add.at(isum, (ix, iy), inten)
    return count, isum


def _check_accumulate(gpu, x, y, inten, xe, ye, want_variant):
    d = torch.device("cuda:0")
    count, isum = gpu.land_accumulate(*(torch.from_numpy(np.ascontiguousarray(a)).to(d) for a in (x, y, inten, xe, ye)))
    assert _info("land_last_variant") == want_variant
    want_c, want_s = _add_at(x, y, inten, xe, ye)
    assert np.array_equal(count.cpu().numpy(), want_c)
    assert np.array_equal(isum.cpu().numpy(), want_s)


# ------------------------------------------------------------------------------------------ land accumulation kernels
# cells (nx, ny) on either side of each switch of rb_land_accumulate: 3 | 2 CTAs per SM at 72 KB, 2 | 1 at 110 KB, the
# shared-memory histogram | global atomics at 220 KB, and a multi-MB grid. The grids are not square, so a kernel that
# swapped the axes of the cell index would put points into the wrong cells.
GRIDS = [((90, 100), 3), ((91, 100), 2), ((110, 125), 2), ((110, 126), 1), ((150, 185), 1), ((150, 186), 0), ((700, 900), 0)]


@pytest.mark.parametrize("cells,ctas", GRIDS)
def test_land_accumulate_on_both_sides_of_every_kernel_switch(gpu, cells, ctas):
    """count / isum of rb_land_accumulate against np.add.at over O.cell_index for three kinds of intensities:
    0..255 integers (fast path, no flag), non-integers (the flag sends them to the ordered kernel: np.add.at's sequential
    float64 sums), and negative integers / integers above 65535 (the shared-memory kernel flags them and the ordered
    kernel runs; the global kernel adds them exactly itself)."""
    nx, ny = cells
    rng = np.random.default_rng(nx * 1000 + ny)
    lo_x, lo_y = np.float32(-311.3), np.float32(47.9)
    hi_x, hi_y = np.float32(lo_x + nx * 5 - 2.5), np.float32(lo_y + ny * 5 - 2.5)
    n = 300_000
    x = rng.uniform(lo_x, hi_x, n).astype(np.float32)
    y = rng.uniform(lo_y, hi_y, n).astype(np.float32)
    k = n // 3                                    # runs of consecutive points in one cell (the histogram's run-length adds)
    x[:k] = np.repeat(rng.uniform(lo_x, hi_x, k // 16), 16).astype(np.float32)[:k]
    y[:k] = np.repeat(rng.uniform(lo_y, hi_y, k // 16), 16).astype(np.float32)[:k]
    x[0], x[1], y[0], y[1] = lo_x, hi_x, hi_y, lo_y
    xe, ye = gpu.arange_edges(x.min(), x.max(), 5.0), gpu.arange_edges(y.min(), y.max(), 5.0)
    assert (len(xe) - 1, len(ye) - 1) == (nx, ny) and _ctas_per_sm(len(xe), len(ye)) == ctas
    fast = SHARED if ctas else GLOBAL
    ints = rng.integers(0, 256, n).astype(np.float32)
    _check_accumulate(gpu, x, y, ints, xe, ye, fast)
    frac = (ints + rng.random(n).astype(np.float32) * np.float32(1e-3)).astype(np.float32)
    assert not np.array_equal(frac, np.rint(frac))
    _check_accumulate(gpu, x, y, frac, xe, ye, ORDERED)
    wide = rng.integers(-70_000, 70_000, n).astype(np.float32)
    assert wide.min() < 0 and wide.max() > 65535
    _check_accumulate(gpu, x, y, wide, xe, ye, ORDERED if ctas else GLOBAL)


# ------------------------------------------------------------------------------------------ cell edges
# (lo, hi, resolution) of float32 bounds: integral bounds whose maximum sits on the last edge (np.clip folds it into the
# last cell); a resolution float32 cannot hold (numpy's spacing float32(lo + res) - lo = 3.300048828125); a positive
# lower bound just below 2048, where lo + res crosses into a coarser float32 binade (spacing 4.9998779296875)
AXES = {"integral": (0.0, 10.0, 5.0), "res_3.3": (-2778.3, 2781.7, 3.3), "binade": (2046.0001, 2646.0001, 5.0)}
SPACING = {"integral": 5.0, "res_3.3": 3.300048828125, "binade": 4.9998779296875}
FRAME_SIZES = [0, 1, 1023, 1024, 1025, 4097]        # frame offsets on and beside the 1024-point tiles of the filter


def _edge_values(edges, lo, hi):
    """Every edge as float32, one ulp either side of it, and both bounds."""
    f = edges.astype(np.float32)
    return np.unique(np.concatenate([f, np.nextafter(f, np.float32(-np.inf)), np.nextafter(f, np.float32(np.inf)),
                                     np.float32([lo, hi])]))


@pytest.mark.parametrize("ax,ay,kernel", [("integral", "res_3.3", SHARED), ("binade", "integral", SHARED),
                                          ("res_3.3", "binade", GLOBAL), ("binade", "res_3.3", GLOBAL)])
def test_points_on_and_beside_cell_edges(gpu, ax, ay, kernel):
    """Points exactly on edges, one float32 ulp either side and at both bounds, through rb_land_accumulate (the named
    kernel) and rb_land_filter(want_mask=True) against O.cell_index, O.land_keep_mask and a cumsum of the keep mask."""
    rng = np.random.default_rng(len(ax) * 31 + len(ay))
    d = torch.device("cuda:0")
    edges, vals = [], []
    for a in (ax, ay):
        lo, hi, res = AXES[a]
        lo, hi = np.float32(lo), np.float32(hi)
        e = gpu.arange_edges(lo, hi, res)
        assert np.array_equal(e, O.grid_edges(lo, hi, res)) and e[1] - e[0] == SPACING[a]
        if a == "integral":
            assert e[-1] == hi                                           # the maximum sits on the last edge
        edges.append(e)
        vals.append(_edge_values(e, lo, hi))
    vx, vy = vals
    x = np.concatenate([vx, rng.choice(vx, len(vy)), rng.choice(vx, 8000)])
    y = np.concatenate([rng.choice(vy, len(vx)), vy, rng.choice(vy, 8000)])
    perm = rng.permutation(len(x))
    x, y = x[perm], y[perm]
    xe, ye = edges
    assert (_ctas_per_sm(len(xe), len(ye)) > 0) == (kernel == SHARED)
    inten = rng.integers(0, 256, len(x)).astype(np.float32)
    _check_accumulate(gpu, x, y, inten, xe, ye, kernel)

    n = sum(FRAME_SIZES)
    assert len(x) >= n
    x, y, inten = x[:n], y[:n], inten[:n]
    land = rng.random((len(xe) - 1, len(ye) - 1)) < 0.5
    off = np.concatenate([[0], np.cumsum(FRAME_SIZES)]).astype(np.int64)
    gain = rng.integers(0, 100, n).astype(np.int32)
    batch = gpu.PointBatch(*(torch.from_numpy(a).to(d) for a in (x, y, inten, gain, off)), n)
    out, mask = gpu.land_filter(batch, torch.from_numpy(xe).to(d), torch.from_numpy(ye).to(d),
                                torch.from_numpy(land.astype(np.uint8)).to(d), want_mask=True)
    keep = O.land_keep_mask(np.column_stack([x, y, inten]), land, (xe, ye))
    assert 0 < keep.sum() < n
    assert np.array_equal(mask.cpu().numpy().astype(bool), keep)
    assert out.n == int(keep.sum())
    for got, want in ((out.x, x), (out.y, y), (out.inten, inten), (out.gain, gain)):
        assert np.array_equal(got[:out.n].cpu().numpy(), want[keep])
    assert np.array_equal(out.frame_off.cpu().numpy(), np.concatenate([[0], np.cumsum(keep)])[off])


# ------------------------------------------------------------------------------------------ spoke stage, varying scales
@pytest.mark.parametrize("S,E,frames", [(64, 1024, 3), (33, 130, 4), (257, 512, 2)])
@pytest.mark.parametrize("dtype", ["float32", "uint8"])
def test_spoke_stage_with_per_spoke_and_per_sweep_scales(gpu, mask_variant, S, E, frames, dtype):
    """range_res tables that differ per spoke AND per sweep (the radar ranges and non-round values), several sweeps per
    launch: every sweep against O.sweep_to_points with its own scale array; gains and frame offsets chain."""
    rng = np.random.default_rng(S * E + frames)
    spec = syn.SweepSpec(seed=S + E, frames=frames, spokes=S, bins=E, clutter_p=0.05, land_blobs=1, buoys=1, boats=1)
    W = frames * 3
    echo = syn.synth_echo(spec).reshape(W, S, E)
    ang = spec.angle_units()
    choices = np.float32(list(NM.values()) + [300.7, 1234.567, 5000.25])
    scale = rng.choice(choices, (W, S)).astype(np.float32)
    assert all(len(np.unique(scale[w])) > 1 for w in range(W)) and not np.array_equal(scale[0], scale[1])
    tabs = [O.spoke_tables(ang, scale[w], E) for w in range(W)]
    d = torch.device("cuda:0")
    c, s, r = (torch.from_numpy(np.stack([t[k] for t in tabs]).astype(np.float32)).to(d) for k in range(3))
    gains = [40, 50, 75] * frames
    t = torch.from_numpy(echo if dtype == "float32" else echo.astype(np.uint8)).to(d)
    b = gpu.spoke_to_points(t, c, s, r, torch.tensor(gains, dtype=torch.int32, device=d), 10.0, 3, gains_per_frame=3)
    vec = 16 if dtype == "uint8" else 4
    assert _info("spoke_last_variant") == (2 if mask_variant == "auto" and (S * E) % vec == 0 else 1)
    want = [O.sweep_to_points(echo[w], ang, scale[w], 10.0, 3) for w in range(W)]
    assert b.n == sum(len(w[0]) for w in want) > 0
    for k, f in enumerate(("x", "y", "inten")):
        assert np.array_equal(getattr(b, f)[:b.n].cpu().numpy(), np.concatenate([w[k] for w in want])), f
    assert np.array_equal(b.gain[:b.n].cpu().numpy(), np.concatenate([np.full(len(w[0]), gains[i], np.int32) for i, w in enumerate(want)]))
    per_frame = [sum(len(w[0]) for w in want[3 * f:3 * f + 3]) for f in range(frames)]
    assert list(b.frame_off.cpu().numpy()) == list(np.concatenate([[0], np.cumsum(per_frame)]))


# ------------------------------------------------------------------------------------------ whole blocks at long range
def _torch_land_check(res, frames_built, d):
    """count, isum, land mask, filtered points and frame offsets of a block against a float64 torch restatement
    (bucketize(right=True) == np.digitize) on the block's own raw points."""
    raw, pts = res.raw, res.points
    n = raw.n
    xe, ye = (torch.from_numpy(e).to(d) for e in res.edges)
    ix = (torch.bucketize(raw.x[:n].double(), xe, right=True) - 1).clamp(0, len(xe) - 2)
    iy = (torch.bucketize(raw.y[:n].double(), ye, right=True) - 1).clamp(0, len(ye) - 2)
    cell = ix * (len(ye) - 1) + iy
    cells = (len(xe) - 1) * (len(ye) - 1)
    count = torch.bincount(cell, minlength=cells)
    isum = torch.zeros(cells, dtype=torch.float64, device=d).index_add_(0, cell, raw.inten[:n].double())
    assert torch.equal(count.view(res.count.shape).to(torch.int32), res.count)
    assert torch.equal(isum.view(res.isum.shape), res.isum)
    mean = torch.where(count > 0, isum / count.clamp(min=1), torch.zeros_like(isum))
    land = ((count.double() / max(frames_built, 1)) >= 0.8) & (mean >= 100)
    assert torch.equal(land.view(res.land.shape), res.land.bool()) and bool(land.any())
    keep = ~land[cell]
    assert 0 < pts.n == int(keep.sum()) < n                          # land really was removed
    for f in ("x", "y", "inten", "gain"):
        assert torch.equal(getattr(pts, f)[:pts.n], getattr(raw, f)[:n][keep]), f
    want_off = torch.cat([torch.zeros(1, dtype=torch.int64, device=d), keep.cumsum(0)])[raw.frame_off]
    assert torch.equal(pts.frame_off, want_off)


def _same_batch(a, b):
    assert a.n == b.n and torch.equal(a.frame_off, b.frame_off)
    for k in ("x", "y", "inten", "gain"):
        assert torch.equal(getattr(a, k)[:a.n], getattr(b, k)[:b.n]), k


def _assert_same(a, b):
    _same_batch(a.raw, b.raw)
    _same_batch(a.points, b.points)
    assert all(np.array_equal(u, v) for u, v in zip(a.edges, b.edges))
    for k in ("count", "isum", "land"):
        assert torch.equal(getattr(a, k), getattr(b, k)), k
    assert a.n_clusters == b.n_clusters and torch.equal(a.labels, b.labels)


def _labels_vs_c_oracle(res, ids):
    p = res.points
    times = np.repeat(np.asarray(ids, np.float32), np.diff(p.frame_off.cpu().numpy()))
    coords = torch.stack([p.x[:p.n], p.y[:p.n]], 1).cpu().numpy()
    want, _ = st_dbscan_c(coords, times, 8.0, 2.0, 15)
    assert want.max() >= 1 and np.array_equal(res.labels.cpu().numpy(), want)


@pytest.mark.parametrize("nm,frames", [(0.25, 24), (1.5, 64)])
def test_full_size_block_at_long_range(gpu, nm, frames):
    """Full-size frames (2048 x 1024 x 3 gains) at 0.25 and 1.5 NM from a fresh DetectionPipeline: rb_detect_block finds
    the land grid larger than its first guess and the pipeline grows its hint and runs the block again; a second call
    of the same shape needs no retry. The result equals the stage-by-stage path, the land stage a float64 restatement,
    the labels the C oracle; ST-DBSCAN runs the tight grid at 0.25 NM and the coarsened general grid at 1.5 NM."""
    from radar_point_cloud_tracking_b200.pipeline import DetectionConfig, DetectionPipeline
    spec = syn.SweepSpec(seed=77, frames=frames, scale_m=NM[nm])
    pipe = DetectionPipeline(DetectionConfig(), 0)
    echo = gpu.synth_echo(spec)
    d = echo.device
    tabs = [torch.from_numpy(t).to(d) for t in pipe.spoke_tables(spec.angle_units(), spec.scale(), frames, spec.bins)]
    hint0 = pipe._grid_hint
    l0 = pipe.ctx.launch_count()
    res = pipe.run_device(echo, *tabs)
    l1 = pipe.ctx.launch_count()
    assert _info("land_last_variant") == GLOBAL
    nxe, nye = len(res.edges[0]), len(res.edges[1])
    assert (nxe - 1) * (nye - 1) > hint0[1]                           # the first guess was too small ...
    hint = pipe._grid_hint
    assert hint[1] > hint0[1] and hint[0] >= max(nxe, nye) and hint[1] >= (nxe - 1) * (nye - 1)   # ... and grew
    again = pipe.run_device(echo, *tabs)
    assert pipe._grid_hint == hint and pipe.ctx.launch_count() - l1 < l1 - l0       # no retry the second time
    _assert_same(again, res)
    staged = pipe.run_device_staged(echo, *tabs)
    st = gpu.stdbscan_stats()
    assert _info("land_last_variant") == GLOBAL
    _assert_same(staged, res)
    del echo, tabs
    built = int(np.count_nonzero(np.diff(res.raw.frame_off.cpu().numpy())))
    _torch_land_check(res, built, d)
    _labels_vs_c_oracle(res, np.arange(frames))
    assert st["n_points"] == res.points.n
    if nm == 0.25:
        assert st["tight"] == 1
    else:
        assert st["tight"] == 0 and st["cell_size"] > 8.0             # the general grid coarsened past eps


# ------------------------------------------------------------------------------------------ mixed ranges
MIXED = dict(seed=29, spokes=512, bins=1024, clutter_p=0.006, land_blobs=3, buoys=3, boats=3)


def _oracle_frames(echo, ang, scale_fgs, thr=10.0, stride=4):
    frames = []
    for f in range(echo.shape[0]):
        per_gain = {g: O.sweep_to_points(echo[f, gi], ang, scale_fgs[f, gi], thr, stride) for gi, g in enumerate((40, 50, 75))}
        frames.append(O.fuse_concat(per_gain))
    return frames


def _check_vs_oracle(res, frames, ids, eps_time=2.0, min_samples=15):
    """Spoke stage + gain concatenation, occupancy grid, land cells, keep masks and labels of a result against the
    numpy / C oracle, frame by frame."""
    raw = res.raw
    assert np.array_equal(torch.stack([raw.x[:raw.n], raw.y[:raw.n], raw.inten[:raw.n]], 1).cpu().numpy(),
                          np.concatenate([f[0] for f in frames]))
    assert np.array_equal(raw.gain[:raw.n].cpu().numpy(), np.concatenate([f[1] for f in frames]))
    pts_f = [f[0] for f in frames]
    count, isum, edges = O.occupancy_grid(pts_f)
    assert np.array_equal(res.edges[0], edges[0]) and np.array_equal(res.edges[1], edges[1])
    assert np.array_equal(res.count.cpu().numpy(), count) and np.array_equal(res.isum.cpu().numpy(), isum)
    land = O.land_cells(count, isum, len(pts_f))
    assert land.any() and np.array_equal(res.land.cpu().numpy().astype(bool), land)
    filt = [p[O.land_keep_mask(p, land, edges)] for p in pts_f]
    p = res.points
    assert np.array_equal(torch.stack([p.x[:p.n], p.y[:p.n], p.inten[:p.n]], 1).cpu().numpy(), np.concatenate(filt))
    assert np.array_equal(np.diff(p.frame_off.cpu().numpy()), [len(f) for f in filt])
    times = np.concatenate([np.full(len(f), i, np.float32) for i, f in zip(ids, filt)])
    want, _ = st_dbscan_c(np.concatenate(filt)[:, :2], times, 8.0, eps_time, min_samples)
    assert want.max() >= 1 and np.array_equal(res.labels.cpu().numpy(), want)


def test_block_whose_frames_alternate_range(gpu):
    """[F, G, S] scales: the frames of one block alternate between 0.125 and 0.5 NM, and the 75 gain of every third
    frame runs at 1 NM. Every stage against the oracle; the union's land grid takes the global kernel."""
    from radar_point_cloud_tracking_b200.pipeline import DetectionConfig, DetectionPipeline
    F = 14
    spec = syn.SweepSpec(frames=F, **MIXED)
    echo_d = gpu.synth_echo(spec)
    echo = echo_d.cpu().numpy()
    scale = np.empty((F, 3, spec.spokes), np.float32)
    for f in range(F):
        scale[f] = NM[0.125] if f % 2 == 0 else NM[0.5]
        if f % 3 == 0:
            scale[f, 2] = NM[1.0]
    ang = spec.angle_units()
    pipe = DetectionPipeline(DetectionConfig(), 0)
    tabs = [torch.from_numpy(t).to(echo_d.device) for t in pipe.spoke_tables(np.broadcast_to(ang, scale.shape), scale, F, spec.bins)]
    res = pipe.run_device(echo_d, *tabs)
    assert _info("land_last_variant") == GLOBAL
    _check_vs_oracle(res, _oracle_frames(echo, ang, scale), np.arange(F))


def test_recording_blocks_of_different_ranges_equal_one_block(gpu):
    """A RecordingDetection fed 0.125 NM blocks, then 0.5 NM blocks: one land grid over the union (global kernel) and
    one labelling, equal to run_device on all frames as one block with [F, G, S] scales."""
    from radar_point_cloud_tracking_b200.pipeline import DetectionConfig, DetectionPipeline
    from radar_point_cloud_tracking_b200.recording import RecordingDetection
    F = 14
    spec = syn.SweepSpec(frames=F, **dict(MIXED, seed=30))
    echo = gpu.synth_echo(spec)
    d = echo.device
    ang = spec.angle_units()
    scale = np.full((F, 3, spec.spokes), NM[0.125], np.float32)
    scale[7:] = NM[0.5]
    ids = np.arange(F) * 2 + 1
    cfg = DetectionConfig()
    pipe = DetectionPipeline(cfg, 0)
    tabs = [torch.from_numpy(t).to(d) for t in pipe.spoke_tables(np.broadcast_to(ang, scale.shape), scale, F, spec.bins)]
    one = pipe.run_device(echo, *tabs, frame_ids=ids)
    rec = RecordingDetection(cfg, 0)
    a = 0
    for nb in (4, 3, 4, 3):
        rec.add_block(echo[a:a + nb], *(t[3 * a:3 * (a + nb)] for t in tabs), ids[a:a + nb])
        a += nb
    got = rec.finish()
    assert _info("land_last_variant") == GLOBAL and _ctas_per_sm(len(got.edges[0]), len(got.edges[1])) == 0
    assert one.land is not None and one.n_clusters > 0
    _assert_same(got, one)


def test_csv_tree_with_two_scales(gpu, tmp_path):
    """The same echoes written under two Scale values (0.125 and 1 NM); frames alternate between the trees and one
    frame mixes sweeps of both, all in one parse batch and one spoke launch. add_csv_frames equals add_host_block of the
    decoded echoes with the per-sweep scales, and its labels equal the oracle's."""
    from radar_point_cloud_tracking_b200.pipeline import DetectionConfig
    from radar_point_cloud_tracking_b200.recording import RecordingDetection
    F = 12
    kw = dict(seed=44, frames=F, spokes=96, bins=256, clutter_p=0.03, land_blobs=2, buoys=2, boats=2)
    spec_a, spec_b = syn.SweepSpec(**kw, scale_m=NM[0.125]), syn.SweepSpec(**kw, scale_m=NM[1.0])
    echo = syn.synth_echo(spec_a)
    tree_a = syn.write_csv_tree(spec_a, tmp_path / "a", echo)
    tree_b = syn.write_csv_tree(spec_b, tmp_path / "b", echo)
    scale = np.empty((F, 3, spec_a.spokes), np.float32)
    frames = []
    for f in range(F):
        pick = [(tree_a if (f + gi) % 2 == 0 else tree_b) if f == 5 else (tree_a if f % 2 == 0 else tree_b) for gi in range(3)]
        frames.append({g: pick[gi][f][g] for gi, g in enumerate(spec_a.gains)})
        scale[f] = np.array([spec_a.scale_m if p is tree_a else spec_b.scale_m for p in pick], np.float32)[:, None]
    assert len(np.unique(scale[5])) == 2
    ids = np.arange(F) + 10
    cfg = DetectionConfig(eps_time=4.0, min_samples=6)
    rec = RecordingDetection(cfg, 0)
    rec.add_csv_frames(frames, ids, num_echo_columns=spec_a.bins)
    got = rec.finish()
    assert rec.csv_files["batched"] == 3 * F and len(rec._offs) - 1 == 1          # one batch
    ang = spec_a.angle_units()
    ref = RecordingDetection(cfg, 0)
    ref.add_host_block(echo.astype(np.uint8), np.broadcast_to(ang, scale.shape), scale, ids)
    _assert_same(got, ref.finish())
    _check_vs_oracle(got, _oracle_frames(echo, ang, scale), ids, 4.0, 6)


# ------------------------------------------------------------------------------------------ fusion at 1.5 NM
def test_fuse_frames_max_at_long_range(gpu):
    """fuse_frames_max at 1 m on full-size 1.5 NM frames: ~31 M grid cells per frame, so the frames fall into several
    2^28-cell groups without forcing a smaller bound; frame by frame against O.fuse_max."""
    from radar_point_cloud_tracking_b200.fusion import fuse_frames_max
    F = 18
    spec = syn.SweepSpec(seed=91, frames=F, scale_m=NM[1.5])
    echo = gpu.synth_echo(spec)
    d = echo.device
    c, s, r = (torch.from_numpy(np.ascontiguousarray(np.broadcast_to(t, (3 * F, spec.spokes)))).to(d)
               for t in O.spoke_tables(spec.angle_units(), spec.scale(), spec.bins))
    b = gpu.spoke_to_points(echo.view(3 * F, spec.spokes, spec.bins), c, s, r,
                            torch.tensor([40, 50, 75] * F, dtype=torch.int32, device=d), 5.0, 8, gains_per_frame=3)
    del echo
    got = fuse_frames_max(b, 1.0).frames()
    off = b.frame_off.cpu().numpy()
    x, y, z = (t[:b.n].cpu().numpy() for t in (b.x, b.y, b.inten))
    cells = [(int(np.ceil((x[a:e].max() - x[a:e].min()) / 1.0)) + 1) * (int(np.ceil((y[a:e].max() - y[a:e].min()) / 1.0)) + 1)
             for a, e in zip(off[:-1], off[1:])]
    assert min(cells) > 25_000_000 and len(gpu.fuse_plan_groups(cells, 1 << 28)) - 1 >= 2
    for f in range(F):
        a, e = off[f], off[f + 1]
        want = O.fuse_max({0: (x[a:e], y[a:e], z[a:e])}, 1.0)
        for u, v in zip(got[f], want):
            assert u.dtype == v.dtype and np.array_equal(u, v)
