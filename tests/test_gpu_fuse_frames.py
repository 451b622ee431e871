"""Max fusion of many frames per call (rb_fuse_max_frames, fusion.fuse_frames_max / fuse_csv_frames_max) against the
numpy oracle of fuse_gains_max, the golden of the unmodified function and the per-frame path, bit for bit with dtypes."""
from types import SimpleNamespace

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle import numpy_oracle as O
from radar_point_cloud_tracking_b200 import synthetic as syn
from radar_point_cloud_tracking_b200._lib import RadarB200Error
from tests.common import golden, pipe_inputs

pytestmark = pytest.mark.gpu

RESOLUTIONS = (1.0, 2.5, 0.3, 1.7, 0.05)


@pytest.fixture(scope="module")
def gpu():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (no CPU fallback exists)")
    torch.cuda.set_device(0)
    from radar_point_cloud_tracking_b200 import device, fusion
    return device, fusion


def _same(got, want):
    assert len(got) == 3
    for a, b in zip(got, want):
        assert a.dtype == b.dtype and a.shape == b.shape
        assert np.array_equal(a, b)


def _batch(device, frames):
    """PointBatch of host frames [(x, y, z) float32]."""
    d = torch.device("cuda", 0)
    counts = [len(f[0]) for f in frames]
    off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    cat = [np.concatenate([f[k] for f in frames]).astype(np.float32) if frames else np.zeros(0, np.float32) for k in range(3)]
    x, y, z = (torch.from_numpy(c).to(d) for c in cat)
    return device.PointBatch(x, y, z, None, torch.from_numpy(off).to(d), int(off[-1]))


def _random_frames(seed=7, n_frames=40):
    rng = np.random.default_rng(seed)
    frames = []
    for f in range(n_frames):
        n = int(np.exp(rng.uniform(0, np.log(200_000)))) if f % 9 else 0
        c = rng.uniform(-60, 60, 2)
        ext = rng.uniform(0.5, 90)
        x = (c[0] + rng.uniform(-ext, ext, n)).astype(np.float32)
        y = (c[1] + rng.normal(0, ext / 3, n)).astype(np.float32)
        kind = f % 4
        if kind == 0:
            z = rng.integers(0, 256, n).astype(np.float32)                         # radar echoes, zeros included
        elif kind == 1:
            z = rng.uniform(-50, 200, n).astype(np.float32)                        # non-integer and negative
        else:
            z = rng.choice(np.array([-3.5, 0.0, 0.25, 7.0, 255.0, 1e-30], np.float32), n)
        frames.append((x, y, z))
    frames[3] = (np.array([12.75], np.float32), np.array([-3.5], np.float32), np.array([9.5], np.float32))       # one point
    n = 500
    frames[5] = (np.full(n, 4.25, np.float32), rng.uniform(-20, 20, n).astype(np.float32), rng.uniform(0, 9, n).astype(np.float32))  # x_min == x_max
    frames[6] = (rng.uniform(0, 30, n).astype(np.float32), rng.uniform(0, 30, n).astype(np.float32),
                 -rng.integers(0, 5, n).astype(np.float32))                      # every intensity <= 0: (f64, f64, f32) empties
    frames[7] = (np.zeros(0, np.float32),) * 3                                   # no points: three float64 empties
    frames[8] = (np.array([1.0, 1.0], np.float32), np.array([2.0, 2.0], np.float32), np.array([0.0, -1.0], np.float32))
    frames[-1] = (np.zeros(0, np.float32),) * 3
    return frames


@pytest.mark.parametrize("res", RESOLUTIONS)
def test_random_frames_one_launch_vs_oracle(gpu, res):
    device, fusion = gpu
    frames = _random_frames()
    fused = fusion.fuse_frames_max(_batch(device, frames), res)
    got = fused.frames()
    assert len(got) == len(frames)
    for f, (fr, g) in enumerate(zip(frames, got)):
        _same(g, O.fuse_max({0: fr}, res))
    assert got[7][2].dtype == np.float64 and got[6][2].dtype == np.float32 and len(got[6][0]) == 0
    assert fused.n == int(fused.cell_off[-1].item())
    for f in (0, 3, 5, 10):                                                      # the one-frame entry agrees
        _same(fusion.fuse_points_max({0: frames[f]}, res), got[f])


def _golden_frame():
    spec, echo = pipe_inputs()
    ang, scale = spec.angle_units(), spec.scale()
    per_gain = {g: O.sweep_to_points(echo[0, gi], ang, scale, 5.0, 8) for gi, g in enumerate(spec.gains)}
    parts = [per_gain[g] for g in sorted(per_gain)]
    return tuple(np.concatenate([p[k] for p in parts]).astype(np.float32) for k in range(3))


@pytest.mark.parametrize("where", ["alone", "first", "middle", "last"])
def test_golden_frame_anywhere_in_a_batch(gpu, where):
    device, fusion = gpu
    g = golden("fuse_max")
    frame = _golden_frame()
    others = _random_frames(seed=11, n_frames=9)
    frames = {"alone": [frame], "first": [frame] + others, "middle": others[:4] + [frame] + others[4:],
              "last": others + [frame]}[where]
    k = {"alone": 0, "first": 0, "middle": 4, "last": len(others)}[where]
    for tag, res in (("r1", 1.0), ("r2p5", 2.5)):
        got = fusion.fuse_frames_max(_batch(device, frames), res).frames()
        _same(got[k], (g[f"{tag}_x"], g[f"{tag}_y"], g[f"{tag}_i"]))


@pytest.mark.parametrize("bound", [1, 5000, 300_000])
def test_many_groups_equal_one_group(gpu, bound):
    device, fusion = gpu
    from radar_point_cloud_tracking_b200._lib import context
    frames = _random_frames(seed=23)
    batch = _batch(device, frames)
    want = fusion.fuse_frames_max(batch, 0.3).frames()
    ctx = context(0)
    cells = []
    for fr in frames:                                                          # the grids of this batch, as the oracle sizes them
        if len(fr[0]):
            nx = int(np.ceil((fr[0].max() - fr[0].min()) / 0.3)) + 1
            ny = int(np.ceil((fr[1].max() - fr[1].min()) / 0.3)) + 1
            cells.append(nx * ny)
        else:
            cells.append(0)
    assert len(device.fuse_plan_groups(cells, bound)) - 1 >= 3
    ctx.set_option("fuse_group_cells", bound)
    try:
        assert ctx.info("fuse_group_cells") == bound
        got = fusion.fuse_frames_max(batch, 0.3).frames()
    finally:
        ctx.set_option("fuse_group_cells", 0)
    for a, b in zip(got, want):
        _same(a, b)


def test_full_size_frames_through_the_spoke_stage(gpu):
    device, fusion = gpu
    from radar_point_cloud_tracking_b200.tracker import sweep_tables
    spec = syn.SweepSpec(seed=2026, frames=64)
    F, G, S, E = spec.frames, len(spec.gains), spec.spokes, spec.bins
    d = torch.device("cuda", 0)
    echo = device.synth_echo(spec, device=d).reshape(F * G, S, E)
    c, s, r = sweep_tables(np.tile(spec.angle_units(), (F * G, 1)), np.tile(spec.scale(), (F * G, 1)), E)
    gains = torch.tensor(list(spec.gains) * F, dtype=torch.int32, device=d)
    batch = device.spoke_to_points(echo, *(torch.from_numpy(np.ascontiguousarray(t)).to(d) for t in (c, s, r)), gains, 5.0, 8,
                                   gains_per_frame=G)
    del echo
    got = fusion.fuse_frames_max(batch, 1.0).frames()
    off = batch.frame_off.cpu().numpy()
    x, y, z = (t[:batch.n].cpu().numpy() for t in (batch.x, batch.y, batch.inten))
    assert batch.n > 64 * 1000
    for f in range(F):
        a, b = off[f], off[f + 1]
        _same(got[f], fusion.fuse_points_max({0: (x[a:b], y[a:b], z[a:b])}, 1.0))


def _rewrite(src, dst, fn):
    dst.write_text("\n".join(fn(src.read_text().split("\n"))))
    return dst


def test_csv_tree_vs_fuse_gains_max(gpu, tmp_path, capsys):
    device, fusion = gpu
    E = 256
    a = syn.write_csv_tree(syn.SweepSpec(seed=51, frames=10, spokes=64, bins=E, clutter_p=0.02, land_blobs=2, buoys=3, boats=2), tmp_path / "a")
    b = syn.write_csv_tree(syn.SweepSpec(seed=52, frames=10, spokes=48, bins=E, clutter_p=0.02, land_blobs=2, buoys=3, boats=2), tmp_path / "b")
    odd = tmp_path / "odd"
    odd.mkdir()
    empty, header_only = odd / "20250813_150000_000.csv", odd / "20250813_150000_100.csv"
    empty.write_text("")
    header_only.write_text(a[0][40].read_text().split("\n")[0] + "\n")

    def dec_echo(rows):                                                          # outside the device grammar
        r = rows[7].split(",")
        r[29:37] = ["212.5"] * 8
        return rows[:7] + [",".join(r)] + rows[8:]

    frames = []
    for f in range(10):
        fa, fb = a[f], b[f]
        if f == 1:
            frames.append({40: fa[40], 75: fb[75]})                              # a gain missing; 64 and 48 spokes
        elif f == 2:
            frames.append({40: empty, 50: header_only})                          # no points at all
        elif f == 3:
            frames.append({40: odd / "20250813_150100_000.csv", 50: fa[50], 75: fa[75]})      # cannot be read
        elif f == 4:
            frames.append({50: _rewrite(fa[50], odd / "20250813_150200_000.csv", dec_echo), 75: fb[75]})
        elif f == 5:
            frames.append({})
        else:
            frames.append(dict(fa) if f % 2 else dict(fb))
    t5 = SimpleNamespace(NUM_ECHO_COLUMNS=E, INTENSITY_THRESHOLD=5.0, POINT_STRIDE=8)
    fusion.install(t5)
    sizes = sum(p.stat().st_size for fr in frames for p in fr.values() if p.exists())
    for res in (1.0, 0.3):
        capsys.readouterr()
        timings = {}
        got = fusion.fuse_csv_frames_max(frames, res, batch_bytes=max(4096, sizes // 4), readers=3, _cfg=fusion._config(t5),
                                         timings=timings)
        printed = capsys.readouterr().out
        assert "Error loading" in printed and "20250813_150100_000.csv" in printed
        assert len(got) == len(frames) and timings["fuse"] > 0
        for f, ff in enumerate(frames):
            _same(got[f], t5.fuse_gains_max(ff, res))
        assert len(got[2][0]) == 0 and got[2][2].dtype == np.float64 and got[5][2].dtype == np.float64


def test_csv_tree_small_batches_count(gpu, tmp_path):
    """batch_bytes small enough for at least three batches: the reader's plan, and results equal to one batch."""
    device, fusion = gpu
    from radar_point_cloud_tracking_b200 import csvbatch
    E = 128
    tree = syn.write_csv_tree(syn.SweepSpec(seed=8, frames=6, spokes=40, bins=E, clutter_p=0.03), tmp_path)
    sizes = [[p.stat().st_size for _, p in sorted(fr.items())] for fr in tree]
    bb = csvbatch.aligned(sum(sizes[0])) + 4096
    batches, _ = csvbatch.pack_batches(sizes, bb)
    assert len(batches) >= 3
    cfg = SimpleNamespace(NUM_ECHO_COLUMNS=E, INTENSITY_THRESHOLD=5.0, POINT_STRIDE=8)
    small = fusion.fuse_csv_frames_max(tree, 1.7, batch_bytes=bb, _cfg=cfg)
    whole = fusion.fuse_csv_frames_max(tree, 1.7, _cfg=cfg)
    for x, y in zip(small, whole):
        _same(x, y)


def test_pipe_spec_first_frame_vs_golden(gpu, tmp_path):
    device, fusion = gpu
    spec, echo = pipe_inputs()
    files = syn.write_csv_tree(spec, tmp_path / "data", echo)
    g = golden("fuse_max")
    cfg = SimpleNamespace(NUM_ECHO_COLUMNS=1024, INTENSITY_THRESHOLD=5.0, POINT_STRIDE=8)
    for tag, res in (("r1", 1.0), ("r2p5", 2.5)):
        got = fusion.fuse_csv_frames_max(files, res, _cfg=cfg)
        assert len(got) == spec.frames
        _same(got[0], (g[f"{tag}_x"], g[f"{tag}_y"], g[f"{tag}_i"]))


@pytest.mark.parametrize("res", [0, -1, float("nan"), float("inf")])
def test_bad_resolution_raises(gpu, res):
    device, fusion = gpu
    batch = _batch(device, _random_frames(n_frames=12)[:3])
    with pytest.raises(RadarB200Error):
        fusion.fuse_frames_max(batch, res)
    from radar_point_cloud_tracking_b200._lib import context, ptr, stream_ptr
    import ctypes as C
    ctx = context(0)
    out = torch.empty(max(batch.n, 1), dtype=torch.float64, device=batch.x.device)
    mx = torch.empty(max(batch.n, 1), dtype=torch.float32, device=batch.x.device)
    co = torch.empty(4, dtype=torch.int64, device=batch.x.device)
    total = C.c_int64(0)
    rc = ctx.lib.rb_fuse_max_frames(ctx.handle, ptr(batch.x), ptr(batch.y), ptr(batch.inten), batch.n, ptr(batch.frame_off), 3,
                                    float(res), ptr(out), ptr(out), ptr(mx), batch.n, ptr(co), C.byref(total), stream_ptr())
    assert rc == -2


def test_frame_over_the_grid_limit_names_the_frame(gpu):
    device, fusion = gpu
    frames = _random_frames(n_frames=12)[:4]
    frames[2] = (np.array([0.0, 40000.0], np.float32), np.array([0.0, 40000.0], np.float32), np.array([1.0, 2.0], np.float32))
    with pytest.raises(RadarB200Error, match="frame 2"):
        fusion.fuse_frames_max(_batch(device, frames), 1.0)
    fusion.fuse_frames_max(_batch(device, frames), 40.0)                       # 1001 x 1001 cells: fine
