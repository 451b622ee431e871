"""Parity of the CUDA path (through the C ABI) with the reference: golden fixtures produced by the
unmodified reference, and the CPU oracle on seeded inputs. Bit-exact everywhere (integer / index
work and float32 chains without reassociation); no tolerance is used in this file."""
import ctypes as C

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle import numpy_oracle as O
from oracle.c_oracle import st_dbscan_c
from radar_point_cloud_tracking_b200 import synthetic as syn
from tests.common import (CLUSTER3D_SPEC, DBSCAN_CASES, PIPE_SPEC, SWEEP_CASES, SWEEP_SPEC, digest, golden,
                          pipe_inputs)

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def gpu():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (no CPU fallback exists)")
    torch.cuda.set_device(0)
    from radar_point_cloud_tracking_b200 import device as dev
    return dev


@pytest.fixture(params=["auto", "registers"])
def mask_variant(request, gpu):
    """Run the spoke-to-point tests on both mask kernels: the default (TMA-staged whenever S*E % 4 == 0)
    and the register-staged one."""
    from radar_point_cloud_tracking_b200 import _lib
    ctx = _lib.context(0)
    ctx.set_option("spoke_mask_variant", 0 if request.param == "auto" else 1)
    yield request.param
    ctx.set_option("spoke_mask_variant", 0)


def _expect_variant(mode, cells):
    from radar_point_cloud_tracking_b200 import _lib
    want = 2 if (mode == "auto" and cells % 4 == 0) else 1
    assert _lib.context(0).info("spoke_last_variant") == want


def _tables(dev, spec, n_sweeps, d):
    from radar_point_cloud_tracking_b200.tracker import sweep_tables
    c, s, r = sweep_tables(spec.angle_units(), spec.scale(), spec.bins)
    rep = lambda t: torch.from_numpy(np.ascontiguousarray(np.broadcast_to(t, (n_sweeps, len(t))))).to(d)
    return rep(c), rep(s), rep(r)


def _run_sweeps(dev, echo_np, spec, thr, stride, gains=None, gpf=1, cap=None):
    d = torch.device("cuda:0")
    W = echo_np.shape[0]
    c, s, r = _tables(dev, spec, W, d)
    g = torch.tensor(gains if gains is not None else [0] * W, dtype=torch.int32, device=d)
    return dev.spoke_to_points(torch.from_numpy(echo_np).to(d), c, s, r, g, thr, stride, gains_per_frame=gpf, cap=cap)


# ------------------------------------------------------------------------------- synthetic twin
def test_device_generator_matches_numpy(gpu):
    for scale_m in (231.5, 2778.0):                 # boat positions depend on the range
        spec = syn.SweepSpec(seed=9, frames=3, spokes=40, bins=256, clutter_p=0.02, land_blobs=2, buoys=3, boats=2, scale_m=scale_m)
        assert np.array_equal(gpu.synth_echo(spec).cpu().numpy(), syn.synth_echo(spec))
        part = gpu.synth_echo(spec, first_frame=1, n_frames=2).cpu().numpy()
        assert np.array_equal(part, syn.synth_echo(spec)[1:])


# ------------------------------------------------------------------------------- a1: spoke-to-point
@pytest.mark.parametrize("tag,thr,stride", SWEEP_CASES)
def test_spoke_to_points_vs_reference_golden(gpu, mask_variant, tag, thr, stride):
    g = golden("sweeps")
    spec = syn.SweepSpec(**SWEEP_SPEC)
    echo = syn.synth_sweep(spec, 0, 2)[None]
    b = _run_sweeps(gpu, echo, spec, thr, stride)
    _expect_variant(mask_variant, echo[0].size)
    assert b.n == int(g[f"{tag}_n"])
    x, y, z = (t[:b.n].cpu().numpy() for t in (b.x, b.y, b.inten))
    assert digest(x) + digest(y) + digest(z) == str(g[f"{tag}_digest"])


@pytest.mark.parametrize("S,E,stride,thr", [(7, 100, 3, 4.0), (33, 130, 1, 8.0), (5, 1023, 5, 2.0), (1, 1, 1, -1.0),
                                            (64, 1024, 7, 9.0), (3, 4096, 2, 0.0), (17, 1000, 3, 1.0),
                                            (2200, 1024, 4, 9.0), (4100, 1024, 3, 2.0)])
def test_spoke_to_points_ragged_shapes(gpu, mask_variant, S, E, stride, thr):
    """Sweeps that do not fill tiles / are not multiples of the vector width; several sweeps per
    launch so stride phases restart at each sweep and output offsets chain across sweeps."""
    spec = syn.SweepSpec(seed=3, frames=2, spokes=S, bins=E, clutter_p=0.05, land_blobs=1, buoys=1, boats=1)
    echo = syn.synth_echo(spec).reshape(-1, S, E)
    b = _run_sweeps(gpu, echo, spec, thr, stride, gains=[40, 50, 75] * 2, gpf=3)
    _expect_variant(mask_variant, S * E)
    off = b.frame_off.cpu().numpy()
    want = [O.sweep_to_points(echo[w], spec.angle_units(), spec.scale(), thr, stride) for w in range(6)]
    wx = np.concatenate([w[0] for w in want])
    assert b.n == len(wx)
    assert np.array_equal(b.x[:b.n].cpu().numpy(), wx)
    assert np.array_equal(b.y[:b.n].cpu().numpy(), np.concatenate([w[1] for w in want]))
    assert np.array_equal(b.inten[:b.n].cpu().numpy(), np.concatenate([w[2] for w in want]))
    assert np.array_equal(b.gain[:b.n].cpu().numpy(),
                          np.concatenate([np.full(len(w[0]), [40, 50, 75][i % 3], np.int32) for i, w in enumerate(want)]))
    assert list(off) == [0, sum(len(w[0]) for w in want[:3]), len(wx)]


def test_spoke_to_points_empty_and_capacity(gpu, mask_variant):
    spec = syn.SweepSpec(**SWEEP_SPEC)
    echo = syn.synth_sweep(spec, 0, 0)[None]
    b = _run_sweeps(gpu, echo, spec, 300.0, 4)            # nothing above the threshold
    assert b.n == 0 and list(b.frame_off.cpu().numpy()) == [0, 0]
    want = O.sweep_to_points(echo[0], spec.angle_units(), spec.scale(), 2.0, 2)
    b = _run_sweeps(gpu, echo, spec, 2.0, 2, cap=1000)    # capacity guess too small -> re-run, same answer
    assert b.n == len(want[0]) and np.array_equal(b.x[:b.n].cpu().numpy(), want[0])
    z = torch.zeros((0, 4, 8), dtype=torch.float32, device="cuda:0")
    e = torch.zeros((0, 4), dtype=torch.float32, device="cuda:0")
    b = gpu.spoke_to_points(z, e, e, e, torch.zeros(0, dtype=torch.int32, device="cuda:0"), 1.0, 1)
    assert b.n == 0


def test_full_size_frame_bit_exact(gpu, mask_variant):
    """One full 2048 x 1024 x 3-gain frame (BASELINE shape) against the numpy oracle."""
    spec = syn.SweepSpec(seed=123, frames=1)
    echo = gpu.synth_echo(spec)
    host = echo.cpu().numpy()
    d = echo.device
    c, s, r = _tables(gpu, spec, 3, d)
    for thr, stride in ((10.0, 4), (2.0, 2)):
        b = gpu.spoke_to_points(echo.view(3, spec.spokes, spec.bins), c, s, r,
                                torch.tensor([40, 50, 75], dtype=torch.int32, device=d), thr, stride, gains_per_frame=3)
        per_gain = {g: O.sweep_to_points(host[0, gi], spec.angle_units(), spec.scale(), thr, stride)
                    for gi, g in enumerate(spec.gains)}
        pts, gains = O.fuse_concat(per_gain)
        assert b.n == len(pts)
        got = torch.stack([b.x[:b.n], b.y[:b.n], b.inten[:b.n]], 1).cpu().numpy()
        assert np.array_equal(got, pts) and np.array_equal(b.gain[:b.n].cpu().numpy(), gains)


def test_batch_properties_at_scale(gpu, mask_variant):
    """Size-independent properties on a 24-sweep batch: per-sweep counts = ceil(M/stride), offsets
    monotone, intensities above threshold, idempotent re-run."""
    spec = syn.SweepSpec(seed=5, frames=8)
    echo = gpu.synth_echo(spec)
    d = echo.device
    W = 24
    c, s, r = _tables(gpu, spec, W, d)
    gains = torch.tensor([40, 50, 75] * 8, dtype=torch.int32, device=d)
    flat = echo.view(W, spec.spokes, spec.bins)
    out1 = gpu.spoke_to_points_raw(flat, c, s, r, gains, 10.0, 4, 3_000_000)
    out2 = gpu.spoke_to_points_raw(flat, c, s, r, gains, 10.0, 4, 3_000_000)
    base = out1[4].cpu().numpy()
    m = (flat > 10.0).sum(dim=(1, 2)).cpu().numpy()
    assert np.array_equal(np.diff(base), (m + 3) // 4)
    n = int(base[-1])
    for a, b in zip(out1[:4], out2[:4]):
        assert torch.equal(a[:n], b[:n])
    assert bool((out1[2][:n] > 10.0).all())


def test_spoke_dense_batch_properties(gpu, mask_variant):
    """Dense clutter (thr 2 -> ~70 % of the cells survive), 12 sweeps, stride 2: per-sweep counts against
    torch, order and values against a torch boolean-mask compaction of two sweeps."""
    spec = syn.SweepSpec(seed=8, frames=4)
    echo = gpu.synth_echo(spec).view(12, spec.spokes, spec.bins)
    d = echo.device
    c, s, r = _tables(gpu, spec, 12, d)
    gains = torch.tensor([40, 50, 75] * 4, dtype=torch.int32, device=d)
    b = gpu.spoke_to_points(echo, c, s, r, gains, 2.0, 2, gains_per_frame=3)
    assert b.n > 8_000_000
    m = (echo > 2.0).view(12, -1).sum(dim=1)
    kept = (m + 1) // 2
    assert b.n == int(kept.sum())
    off = b.frame_off.cpu().numpy()
    assert list(off) == [0] + list(np.cumsum(kept.view(4, 3).sum(dim=1).cpu().numpy()))
    base = np.concatenate([[0], np.cumsum(kept.cpu().numpy())])
    for w in (0, 7):
        want = echo[w].reshape(-1)[(echo[w] > 2.0).reshape(-1)][::2]
        assert torch.equal(b.inten[base[w]:base[w + 1]], want)
        assert bool((b.gain[base[w]:base[w + 1]] == gains[w]).all())


def test_spoke_profile_option(gpu):
    from radar_point_cloud_tracking_b200 import _lib
    ctx = _lib.context(0)
    spec = syn.SweepSpec(**SWEEP_SPEC)
    echo = syn.synth_sweep(spec, 0, 2)[None]
    ctx.set_option("spoke_profile", 1)
    try:
        _run_sweeps(gpu, echo, spec, 10.0, 4)
        assert all(ctx.info(k) >= 0 for k in ("spoke_mask_ns", "spoke_offsets_ns", "spoke_emit_ns"))
    finally:
        ctx.set_option("spoke_profile", 0)


# ------------------------------------------------------------------------------- T4 mirror on CSV files
def test_tracker_functions_on_csv_tree_vs_golden(gpu, tmp_path):
    from radar_point_cloud_tracking_b200 import tracker as trk
    g = golden("pipeline_small")
    spec, echo = pipe_inputs()
    files = syn.write_csv_tree(spec, tmp_path, echo)
    x, y, z, gain = trk.load_radar_csv(files[0][50])
    o = g["frame_offsets"]
    frames = [trk.build_frame(ff, i) for i, ff in enumerate(files)]
    assert gain == 50 and all(f is not None for f in frames)
    assert np.array_equal(np.cumsum([0] + [f.num_points for f in frames]), o)
    assert np.array_equal(np.concatenate([f.points for f in frames]), g["points"])
    assert np.array_equal(np.concatenate([f.gains for f in frames]), g["gains"])
    assert frames[0].points.dtype == np.float32 and frames[0].gains.dtype == np.int32
    n40 = int((frames[0].gains == 40).sum())
    assert np.array_equal(x, frames[0].points[n40:n40 + len(x), 0])

    count, isum, (xe, ye) = trk.build_occupancy_grid(frames, trk.LAND_GRID_RESOLUTION)
    assert np.array_equal(xe, g["x_edges"]) and np.array_equal(ye, g["y_edges"])
    assert np.array_equal(count, g["count"]) and count.dtype == np.int32
    assert np.array_equal(isum, g["isum"]) and isum.dtype == np.float64
    land = trk.identify_land_cells(count, isum, len(frames))
    assert land.dtype == bool and np.array_equal(land, g["land"])
    filt = [trk.filter_land_from_frame(f, land, (xe, ye)) for f in frames]
    assert np.array_equal(np.cumsum([0] + [f.num_points for f in filt]), g["filt_offsets"])
    assert np.array_equal(np.concatenate([f.points for f in filt]), g["filt_points"])
    assert np.array_equal(np.concatenate([f.gains for f in filt]), g["filt_gains"])

    for tag, eps_s, eps_t, ms in DBSCAN_CASES:
        clusters = trk.st_dbscan(filt, eps_s, eps_t, ms)
        rec = sorted((fid, c.cluster_id, c.num_points, c.centroid[0], c.centroid[1], c.mean_intensity)
                     for fid, cl in clusters.items() for c in cl)
        assert np.array_equal(np.array(rec, dtype=np.float64).reshape(-1, 6), g[f"clusters_{tag}"])
    # error behaviour of the reference: unreadable file -> empty arrays and gain 0; empty frame -> None
    bad = tmp_path / "gain_40" / "20250101_000000_000.csv"
    bad.write_text("")
    x, y, z, gain = trk.load_radar_csv(bad)
    assert len(x) == 0 and gain == 0
    assert trk.build_frame({40: bad}, 0) is None
    assert trk.st_dbscan([], 8.0, 2.0, 15) == {}


# ------------------------------------------------------------------------------- device pipeline
def test_device_pipeline_vs_golden(gpu):
    from radar_point_cloud_tracking_b200.pipeline import DetectionConfig, DetectionPipeline
    g = golden("pipeline_small")
    spec, echo = pipe_inputs()
    pipe = DetectionPipeline(DetectionConfig())
    out = pipe.run_host(echo, spec.angle_units(), spec.scale())
    assert np.array_equal(out["points"], g["filt_points"]) and np.array_equal(out["gains"], g["filt_gains"])
    assert np.array_equal(out["frame_off"], g["filt_offsets"])
    # device generator + device path gives the same thing
    d_echo = gpu.synth_echo(spec)
    c, s, r = pipe.spoke_tables(spec.angle_units(), spec.scale(), spec.frames, spec.bins)
    res = pipe.run_device(d_echo, *(torch.from_numpy(t).cuda() for t in (c, s, r)))
    assert np.array_equal(res.land.cpu().numpy().astype(bool), g["land"])
    assert np.array_equal(res.count.cpu().numpy(), g["count"]) and np.array_equal(res.isum.cpu().numpy(), g["isum"])
    raw = res.raw
    assert np.array_equal(torch.stack([raw.x[:raw.n], raw.y[:raw.n], raw.inten[:raw.n]], 1).cpu().numpy(), g["points"])
    rec = sorted((fid, c.cluster_id, c.num_points, c.centroid[0], c.centroid[1], c.mean_intensity)
                 for fid, cl in res.clusters_by_frame().items() for c in cl)
    rec = np.array(rec, dtype=np.float64).reshape(-1, 6)
    assert np.array_equal(rec, g["clusters_default"])
    csv = g["clusters_csv"]
    csv = csv[np.lexsort((csv[:, 1], csv[:, 0]))]
    assert np.array_equal(csv.astype(np.float32), rec.astype(np.float32))     # the real CLI's clusters.csv


# ------------------------------------------------------------------------------- a7: ST-DBSCAN
@pytest.fixture(params=["auto", "general"])
def db_mode(request, gpu):
    """Run the ST-DBSCAN tests on both algorithms: auto (tight-cell buckets whenever the times are integers
    and the table fits) and the general point-level one."""
    from radar_point_cloud_tracking_b200 import _lib
    ctx = _lib.context(0)
    ctx.set_option("dbscan_mode", 0 if request.param == "auto" else 1)
    yield request.param
    ctx.set_option("dbscan_mode", 0)


def test_stdbscan_random_cases_vs_reference_golden(gpu, db_mode):
    from radar_point_cloud_tracking_b200.clustering import st_dbscan
    g = golden("stdbscan_random")
    for k in range(24):
        eps_s, eps_t, ms = g[f"c{k}_params"]
        got = st_dbscan(g[f"c{k}_coords"], g[f"c{k}_times"], float(eps_s), float(eps_t), int(ms))
        assert got.dtype == np.int32 and np.array_equal(got, g[f"c{k}_labels"]), k


def test_stdbscan_package_3d_case_vs_golden(gpu, db_mode):
    from radar_point_cloud_tracking_b200.clustering import st_dbscan
    g = golden("package")
    spec3 = syn.SweepSpec(**CLUSTER3D_SPEC)
    pts, tms = [], []
    for gi in range(3):
        x, y, z = O.sweep_to_points(syn.synth_sweep(spec3, 0, gi), spec3.angle_units(), spec3.scale(), 10.0, 2)
        pts.append(np.column_stack((x, y, z)))
        tms.append(np.full(len(x), gi, dtype=np.float32))
    assert np.array_equal(st_dbscan(np.concatenate(pts), np.concatenate(tms), 5.0, 1.0, 10), g["cluster3d_labels"])


def test_stdbscan_known_answers(gpu, db_mode):
    """radar-pipeline-rs/src/processors/clustering.rs:502-597 + edge cases."""
    from radar_point_cloud_tracking_b200.clustering import st_dbscan
    sq = [[0, 0, 0], [1, 0, 0], [0, 1, 0], [1, 1, 0]]
    coords = np.array(sq + [[100 + a, 100 + b, 0] for a, b, _ in sq], dtype=np.float32)
    lab = st_dbscan(coords, np.zeros(8, np.float32), 5.0, 1.0, 2)
    assert list(lab) == [0, 0, 0, 0, 1, 1, 1, 1]
    lab = st_dbscan(np.array(sq, np.float32), np.array([0, 0, 5, 5], np.float32), 5.0, 1.0, 2)
    assert list(lab) == [0, 0, 1, 1]
    lab = st_dbscan(np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [100, 100, 100]], np.float32), np.zeros(4, np.float32), 5.0, 1.0, 3)
    assert list(lab) == [0, 0, 0, -1]
    assert len(st_dbscan(np.zeros((0, 3), np.float32), np.zeros(0, np.float32), 5.0, 1.0, 3)) == 0
    assert list(st_dbscan(np.zeros((1, 3), np.float32), np.zeros(1, np.float32), 5.0, 1.0, 2)) == [-1]
    # duplicates, eps 0, min_samples 1, exact-distance inclusivity (3-4-5 triangle: d == eps)
    dup = np.array([[1, 1], [1, 1], [1, 1], [2, 2]], np.float32)
    assert list(st_dbscan(dup, np.zeros(4, np.float32), 0.0, 0.0, 3)) == [0, 0, 0, -1]
    assert list(st_dbscan(dup, np.zeros(4, np.float32), 0.0, 0.0, 1)) == [0, 0, 0, 1]
    tri = np.array([[0, 0], [3, 4]], np.float32)
    assert list(st_dbscan(tri, np.zeros(2, np.float32), 5.0, 0.0, 2)) == [0, 0]
    assert list(st_dbscan(tri, np.zeros(2, np.float32), 4.999999, 0.0, 2)) == [-1, -1]
    with pytest.raises(Exception):
        st_dbscan(np.array([[0.1, 0.2]], np.float64), np.zeros(1, np.float32), 1.0, 1.0, 1)


@pytest.mark.parametrize("n,frames,eps_s,eps_t,ms,dim", [(60000, 40, 8.0, 2.0, 15, 2), (40000, 3, 5.0, 1.0, 10, 3),
                                                          (30000, 200, 3.0, 0.5, 4, 2), (20000, 6, 6.0, 2.5, 8, 2)])
def test_stdbscan_vs_c_oracle_medium(gpu, db_mode, n, frames, eps_s, eps_t, ms, dim):
    """Larger seeded problems against the C oracle: identical labels and core sets."""
    rng = np.random.default_rng(n + frames)
    span = 400.0
    coords = (rng.random((n, dim)) * span).astype(np.float32)
    k = n // 2
    centres = (rng.random((40, dim)) * span).astype(np.float32)
    coords[:k] = (centres[rng.integers(0, 40, k)] + rng.normal(0, 3.0, (k, dim))).astype(np.float32)
    if eps_t != int(eps_t):
        times = (rng.random(n) * frames).astype(np.float32)
    else:
        times = rng.integers(0, frames, n).astype(np.float32)
    want, want_core = st_dbscan_c(coords, times, eps_s, eps_t, ms)
    d = torch.device("cuda:0")
    flat = torch.from_numpy(coords).to(d).view(-1)
    lab, core, ncl = gpu.stdbscan(flat, flat[1:], flat[2:] if dim == 3 else None, torch.from_numpy(times).to(d),
                                  eps_s, eps_t, ms, stride=dim, n=n, want_core=True)
    assert np.array_equal(core.cpu().numpy().astype(bool), want_core)
    assert np.array_equal(lab.cpu().numpy(), want)
    assert ncl == want.max() + 1
    st = gpu.stdbscan_stats()
    assert st["n_points"] == n and st["pair_tests_count"] > 0
    if db_mode == "general" or eps_t != int(eps_t):
        assert st["tight"] == 0
    elif dim == 2:
        assert st["tight"] == 1                      # (the 3-D case exceeds the bucket budget at this n)


def test_stdbscan_phases_and_global_keys(gpu, db_mode):
    """The phase entry points reproduce rb_stdbscan; component keys follow the caller's global indices;
    overriding core flags changes the components accordingly (what the sharded driver relies on)."""
    rng = np.random.default_rng(77)
    n = 30000
    coords = (rng.random((n, 2)) * 300).astype(np.float32)
    centres = (rng.random((25, 2)) * 300).astype(np.float32)
    coords[: n // 2] = (centres[rng.integers(0, 25, n // 2)] + rng.normal(0, 2.5, (n // 2, 2))).astype(np.float32)
    times = rng.integers(0, 12, n).astype(np.float32)
    want, want_core = st_dbscan_c(coords, times, 6.0, 2.0, 12)
    d = torch.device("cuda:0")
    flat = torch.from_numpy(coords).to(d).view(-1)
    ph = gpu.StDbscanPhases(flat, flat[1:], None, torch.from_numpy(times).to(d), 6.0, 2.0, 12, stride=2, n=n)
    core = ph.cores()
    assert np.array_equal(core.cpu().numpy().astype(bool), want_core)
    gidx = torch.arange(n, dtype=torch.int64, device=d) * 3 + 1000          # any increasing global numbering
    key = ph.components(gidx).cpu().numpy()
    assert np.array_equal(key >= 0, want_core)
    # key = smallest global index among the component's cores  <=>  canonical label order
    for lab in range(want.max() + 1):
        members = np.flatnonzero((want == lab) & want_core)
        assert np.all(key[members] == members.min() * 3 + 1000)
    uniq = np.unique(key[key >= 0])
    table_k = torch.from_numpy(uniq).to(d)
    table_i = torch.arange(len(uniq), dtype=torch.int32, device=d)
    core_label = gpu.relabel(torch.from_numpy(key).to(d), table_k, table_i)
    labels = ph.assign(core_label).cpu().numpy()
    assert np.array_equal(labels, want)
    # demote every core point of cluster 0 that lives at t >= 6: keys/labels follow the new core set
    mod_core = want_core.copy()
    mod_core[(want == 0) & (times >= 6)] = False
    ph.set_cores(torch.from_numpy(mod_core.astype(np.uint8)).to(d))
    key2 = ph.components(None).cpu().numpy()
    assert np.array_equal(key2 >= 0, mod_core)


def test_stdbscan_wrong_hint_is_an_error_not_a_wrong_answer(gpu):
    """A hint box that does not contain every point would clamp points into edge buckets ("same tight cell => neighbour"
    would then be false): the plan flags it on the device and the check fails loudly."""
    from radar_point_cloud_tracking_b200 import RadarB200Error
    rng = np.random.default_rng(2)
    n = 20000
    d = torch.device("cuda:0")
    x = torch.from_numpy((rng.random(n) * 200 - 100).astype(np.float32)).to(d)
    y = torch.from_numpy((rng.random(n) * 200 - 100).astype(np.float32)).to(d)
    t = torch.from_numpy(rng.integers(0, 8, n).astype(np.float32)).to(d)
    good = gpu.StDbscanPhases(x, y, None, t, 5.0, 1.0, 5, n=n, hint=(-100.0, 100.0, -100.0, 100.0, 0.0, 7.0))
    good.cores()
    good.check()                                                      # a box that holds everything: fine
    for bad_hint in ((-100.0, 50.0, -100.0, 100.0, 0.0, 7.0), (-100.0, 100.0, -100.0, 100.0, 0.0, 5.0)):      # x cut / time cut
        bad = gpu.StDbscanPhases(x, y, None, t, 5.0, 1.0, 5, n=n, hint=bad_hint)
        bad.cores()
        with pytest.raises(RadarB200Error, match="hinted box"):
            bad.check()


def test_block_driver_clusters_in_3d_like_t3(gpu):
    """DetectionConfig(cluster_3d=True): rb_detect_block clusters on (x, y, z = intensity), the coordinates
    3_stdbscan_point_clouds.py builds (T3:177-182) - labels against the C oracle on the block's own points."""
    from radar_point_cloud_tracking_b200.pipeline import DetectionConfig, DetectionPipeline
    spec = syn.SweepSpec(seed=36, frames=20, spokes=512, bins=1024, gains=(50,), clutter_p=0.004)
    cfg = DetectionConfig(gains=(50,), land_filter=False, eps_space=5.0, eps_time=1.0, min_samples=10, cluster_3d=True)
    pipe = DetectionPipeline(cfg, 0)
    echo = gpu.synth_echo(spec)
    c, s, r = pipe.spoke_tables(spec.angle_units(), spec.scale(), spec.frames, spec.bins)
    tabs = [torch.from_numpy(t).to(echo.device) for t in (c, s, r)]
    res = pipe.run_device(echo, *tabs)
    staged = pipe.run_device_staged(echo, *tabs)
    p = res.points
    coords = torch.stack([p.x[:p.n], p.y[:p.n], p.inten[:p.n]], 1).cpu().numpy()
    times = np.repeat(np.arange(spec.frames), np.diff(p.frame_off.cpu().numpy())).astype(np.float32)
    want, _ = st_dbscan_c(coords, times, 5.0, 1.0, 10)
    assert p.n > 20000 and want.max() > 5
    assert np.array_equal(res.labels.cpu().numpy(), want) and torch.equal(res.labels, staged.labels)
    flat, _ = st_dbscan_c(coords[:, :2], times, 5.0, 1.0, 10)
    assert not np.array_equal(flat, want)                             # the third coordinate really takes part


def test_stdbscan_sparse_frame_ids_and_coarsening(gpu, db_mode):
    """Frame ids with huge gaps and a tiny eps over a wide extent force the grid to coarsen."""
    from radar_point_cloud_tracking_b200.clustering import st_dbscan
    rng = np.random.default_rng(1)
    coords = (rng.random((5000, 2)) * 20000).astype(np.float32)
    coords[:2500] = (coords[rng.integers(2500, 5000, 2500)] + rng.normal(0, 0.05, (2500, 2))).astype(np.float32)
    times = rng.choice(np.array([0, 1, 2, 1000000, 1000001, 5000000], np.float32), 5000)
    want, _ = st_dbscan_c(coords, times, 0.2, 1.0, 3)
    assert np.array_equal(st_dbscan(coords, times, 0.2, 1.0, 3), want)


# ------------------------------------------------------------------------------- a3 + package transforms
def test_fuse_max_vs_reference_golden(gpu):
    from radar_point_cloud_tracking_b200.fusion import fuse_points_absolute, fuse_points_max
    g = golden("fuse_max")
    spec, echo = pipe_inputs()
    b = _run_sweeps(gpu, echo[0], spec, 5.0, 8, gains=[40, 50, 75], gpf=1)
    off = b.frame_off.cpu().numpy()
    x, y, z = (t[:b.n].cpu().numpy() for t in (b.x, b.y, b.inten))
    per_gain = {gain: (x[off[i]:off[i + 1]], y[off[i]:off[i + 1]], z[off[i]:off[i + 1]]) for i, gain in enumerate(spec.gains)}
    for tag, res in (("r1", 1.0), ("r2p5", 2.5)):
        ox, oy, oi = fuse_points_max(per_gain, res)
        assert ox.dtype == g[f"{tag}_x"].dtype
        assert np.array_equal(ox, g[f"{tag}_x"]) and np.array_equal(oy, g[f"{tag}_y"]) and np.array_equal(oi, g[f"{tag}_i"])
    ax, ay, ai, ag = fuse_points_absolute(per_gain)
    assert digest(ax) + digest(ay) + digest(ai) + digest(ag) == str(g["abs_digest"])


def test_package_transforms_vs_golden(gpu):
    from types import SimpleNamespace
    from radar_point_cloud_tracking_b200.transforms import polar_to_cartesian, sweep_to_point_cloud
    g = golden("package")
    spec = syn.SweepSpec(**SWEEP_SPEC)
    angles = np.deg2rad(spec.angle_units().astype(np.float32) * (360.0 / 8196.0))
    ranges = (spec.scale()[:, None] / spec.bins) * np.arange(spec.bins, dtype=np.float32)
    x, y = polar_to_cartesian(angles, ranges)
    assert digest(x) + digest(y) == str(g["p2c_digest"])
    # known answers of radar-pipeline/tests/test_transforms.py:15-40 (atol 1e-6 in the reference)
    a = np.array([0, np.pi / 2, np.pi], dtype=np.float32)
    x, y = polar_to_cartesian(a, np.ones((3, 1), np.float32))
    np.testing.assert_allclose(x[:, 0], [1, 0, -1], atol=1e-6)
    np.testing.assert_allclose(y[:, 0], [0, 1, 0], atol=1e-6)
    sweep = SimpleNamespace(angles_rad=angles, ranges=ranges, intensities=syn.synth_sweep(spec, 0, 1),
                            scale=spec.scale(), gain=50)
    for tag, thr, stride in (("default", 0.0, 16), ("t10_s4", 10.0, 4)):
        pc = sweep_to_point_cloud(sweep, SimpleNamespace(intensity_threshold=thr, point_stride=stride))
        assert pc.size == int(g[f"s2pc_{tag}_n"])
        assert digest(pc.x) + digest(pc.y) + digest(pc.z) == str(g[f"s2pc_{tag}_digest"])
    assert sweep_to_point_cloud(sweep).size == int(g["s2pc_default_n"])


def test_abi_error_paths(gpu):
    from radar_point_cloud_tracking_b200 import _lib
    ctx = _lib.context(0)
    rc = ctx.lib.rb_bounds(ctx.handle, None, None, 0, None, None)
    assert rc == -2 and b"NULL" in ctx.lib.rb_last_error()
    n = C.c_int64(7)
    assert ctx.lib.rb_stdbscan(ctx.handle, None, None, None, 1, None, 0, 1.0, 1.0, 1, None, None, C.byref(n), None) == 0
    assert n.value == 0 and ctx.launch_count() > 0


# ------------------------------------------------------------------------------- scale / stress properties
def test_stdbscan_dense_clutter_both_algorithms_vs_oracle(gpu):
    """Dense clutter (every point has hundreds of neighbours, BASELINE config 4 in miniature): the tight-cell
    algorithm decides most pairs without a distance test; labels and core flags must still equal the C oracle
    and the general algorithm, point for point."""
    from radar_point_cloud_tracking_b200 import _lib
    rng = np.random.default_rng(404)
    n, frames = 50000, 4
    coords = (rng.random((n, 2)) * 220).astype(np.float32)                 # ~1 point / m^2 / frame-ish
    coords[:4000] = (rng.random((4000, 2)) * 40 + 400).astype(np.float32)    # a second, detached dense patch
    coords[4000:4200] = (rng.random((200, 2)) * 3000 + 1000).astype(np.float32)   # isolated noise
    times = rng.integers(0, frames, n).astype(np.float32)
    want, want_core = st_dbscan_c(coords, times, 12.0, 2.0, 15)
    assert want_core.mean() > 0.9 and want.max() >= 1
    d = torch.device("cuda:0")
    flat = torch.from_numpy(coords).to(d).view(-1)
    ctx = _lib.context(0)
    tests = {}
    for mode in (0, 1):
        ctx.set_option("dbscan_mode", mode)
        try:
            lab, core, ncl = gpu.stdbscan(flat, flat[1:], None, torch.from_numpy(times).to(d), 12.0, 2.0, 15, stride=2, n=n,
                                          want_core=True)
        finally:
            ctx.set_option("dbscan_mode", 0)
        st = gpu.stdbscan_stats()
        assert st["tight"] == (1 if mode == 0 else 0)
        tests[mode] = st["pair_tests_count"] + st["pair_tests_union"] + st["pair_tests_border"]
        assert np.array_equal(core.cpu().numpy().astype(bool), want_core)
        assert np.array_equal(lab.cpu().numpy(), want)
    assert tests[0] * 5 < tests[1]                      # the shortcuts really skip most of the pair tests


def test_land_filter_full_size_vs_torch_float64(gpu):
    """24 full-size fused frames (2048 x 1024 x 3 gains): count grid, land mask and filtered points against a
    torch float64 restatement (bucketize(right=True) == np.digitize) on the same device-resident points."""
    from radar_point_cloud_tracking_b200.pipeline import DetectionConfig, DetectionPipeline
    spec = syn.SweepSpec(seed=77, frames=24)
    pipe = DetectionPipeline(DetectionConfig(), 0)
    echo = gpu.synth_echo(spec)
    c, s, r = pipe.spoke_tables(spec.angle_units(), spec.scale(), spec.frames, spec.bins)
    d = echo.device
    res = pipe.run_device(echo, *(torch.from_numpy(t).to(d) for t in (c, s, r)), cluster=False)
    raw, pts = res.raw, res.points
    n = raw.n
    assert n > 200_000 and res.land is not None and 0 < pts.n < n
    xe, ye = (torch.from_numpy(e).to(d) for e in res.edges)
    x64, y64 = raw.x[:n].double(), raw.y[:n].double()
    ix = (torch.bucketize(x64, xe, right=True) - 1).clamp(0, len(xe) - 2)
    iy = (torch.bucketize(y64, ye, right=True) - 1).clamp(0, len(ye) - 2)
    cell = ix * (len(ye) - 1) + iy
    cells = (len(xe) - 1) * (len(ye) - 1)
    count = torch.bincount(cell, minlength=cells)
    isum = torch.zeros(cells, dtype=torch.float64, device=d).index_add_(0, cell, raw.inten[:n].double())
    assert torch.equal(count.view(res.count.shape).to(torch.int32), res.count)
    assert torch.equal(isum.view(res.isum.shape), res.isum)                 # integer-valued echoes: exact in any order
    frames_built = int(np.count_nonzero(np.diff(raw.frame_off.cpu().numpy())))
    mean = torch.where(count > 0, isum / count.clamp(min=1), torch.zeros_like(isum))
    land = ((count.double() / max(frames_built, 1)) >= 0.8) & (mean >= 100)
    assert torch.equal(land.view(res.land.shape), res.land.bool()) and bool(land.any())
    keep = ~land[cell]
    assert pts.n == int(keep.sum())
    assert torch.equal(pts.x[:pts.n], raw.x[:n][keep]) and torch.equal(pts.inten[:pts.n], raw.inten[:n][keep])
    assert torch.equal(pts.gain[:pts.n], raw.gain[:n][keep])
    off = raw.frame_off
    want_off = torch.cat([torch.zeros(1, dtype=torch.int64, device=d), keep.cumsum(0)])[off]
    assert torch.equal(pts.frame_off, want_off)


def test_land_accumulate_non_integer_intensities_take_the_ordered_path(gpu):
    """np.add.at adds the points of a cell one after the other (T4:388-389). The fast kernel is exact for integer-valued
    intensities and raises a flag otherwise; the ordered kernel then reproduces the sequential float64 sums bit for bit -
    through device.land_accumulate and through the block driver (rb_detect_block, res.land_ordered)."""
    import ctypes as C
    from radar_point_cloud_tracking_b200 import _lib
    rng = np.random.default_rng(61)
    n = 400_000
    x = rng.normal(0, 60, n).astype(np.float32)
    y = rng.normal(0, 60, n).astype(np.float32)
    x[: n // 2] = rng.normal(35, 1.5, n // 2).astype(np.float32)        # half of the points in a handful of cells
    y[: n // 2] = rng.normal(-20, 1.5, n // 2).astype(np.float32)
    inten = (rng.random(n) * 255 + rng.random(n) * 1e-3).astype(np.float32)
    xe, ye = O.grid_edges(x.min(), x.max(), 5.0), O.grid_edges(y.min(), y.max(), 5.0)
    ix, iy = O.cell_index(x, xe, len(xe) - 1), O.cell_index(y, ye, len(ye) - 1)
    count = np.zeros((len(xe) - 1, len(ye) - 1), np.int32)
    isum = np.zeros(count.shape, np.float64)
    np.add.at(count, (ix, iy), 1)
    np.add.at(isum, (ix, iy), inten)
    d = torch.device("cuda:0")
    tx, ty, ti, txe, tye = (torch.from_numpy(a).to(d) for a in (x, y, inten, xe, ye))
    c1, s1 = gpu.land_accumulate(tx, ty, ti, txe, tye)
    assert np.array_equal(c1.cpu().numpy(), count) and np.array_equal(s1.cpu().numpy(), isum)
    # the flag really was what sent it there: check=False leaves the (order dependent) fast result and the raised flag
    c2, s2 = gpu.land_accumulate(tx, ty, ti, txe, tye, check=False)
    assert int(gpu.land_accumulate_flag(0).item()) == 1 and np.array_equal(c2.cpu().numpy(), count)
    assert int(gpu.land_accumulate_flag(0).item()) == 0                    # reading clears it
    # integer-valued intensities: fast path, exact, no flag
    ti_int = torch.from_numpy(np.rint(inten)).to(d)
    c3, s3 = gpu.land_accumulate(tx, ty, ti_int, txe, tye, check=False)
    want = np.zeros(count.shape, np.float64)
    np.add.at(want, (ix, iy), np.rint(inten))
    assert int(gpu.land_accumulate_flag(0).item()) == 0 and np.array_equal(s3.cpu().numpy(), want)


def test_block_driver_with_non_integer_echoes_matches_the_oracle(gpu):
    """A recording whose echoes are not integers through rb_detect_block: the land stage repeats itself with the ordered
    accumulation (res.land_ordered) and grids, mask and filtered points equal the numpy oracle's."""
    from radar_point_cloud_tracking_b200 import _lib
    from radar_point_cloud_tracking_b200.pipeline import DetectionConfig, DetectionPipeline
    spec = syn.SweepSpec(seed=71, frames=14, spokes=128, bins=512, clutter_p=0.01, land_blobs=2, buoys=2, boats=2)
    echo = syn.synth_echo(spec)
    rng = np.random.default_rng(5)
    echo = (echo * np.float32(0.731) + rng.random(echo.shape).astype(np.float32) * np.float32(0.01)).astype(np.float32)
    cfg = DetectionConfig(intensity_threshold=7.0, land_min_intensity=60.0)
    pipe = DetectionPipeline(cfg, 0)
    c, s, r = pipe.spoke_tables(spec.angle_units(), spec.scale(), spec.frames, spec.bins)
    res = pipe.run_device(torch.from_numpy(echo).cuda(), *(torch.from_numpy(t).cuda() for t in (c, s, r)), cluster=False)
    frames = []
    for f in range(spec.frames):
        per_gain = {g: O.sweep_to_points(echo[f, gi], spec.angle_units(), spec.scale(), 7.0, 4) for gi, g in enumerate(spec.gains)}
        frames.append(O.fuse_concat(per_gain)[0])
    count, isum, edges = O.occupancy_grid(frames)
    land = O.land_cells(count, isum, len(frames), min_intensity=60.0)
    assert land.any() and not np.array_equal(isum, np.rint(isum))
    assert np.array_equal(res.count.cpu().numpy(), count) and np.array_equal(res.isum.cpu().numpy(), isum)
    assert np.array_equal(res.land.cpu().numpy().astype(bool), land)
    want = np.concatenate([p[O.land_keep_mask(p, land, edges)] for p in frames])
    p = res.points
    assert np.array_equal(torch.stack([p.x[:p.n], p.y[:p.n], p.inten[:p.n]], 1).cpu().numpy(), want)


def test_pipeline_is_deterministic_at_scale(gpu):
    """Atomics decide only WHICH thread links two components first, never the result: two runs over 48
    full-size frames give identical points and labels; labels are canonical (ids appear in index order)."""
    from radar_point_cloud_tracking_b200.pipeline import DetectionConfig, DetectionPipeline
    spec = syn.SweepSpec(seed=5, frames=48)
    pipe = DetectionPipeline(DetectionConfig(), 0)
    echo = gpu.synth_echo(spec)
    c, s, r = pipe.spoke_tables(spec.angle_units(), spec.scale(), spec.frames, spec.bins)
    tabs = [torch.from_numpy(t).to(echo.device) for t in (c, s, r)]
    a = pipe.run_device(echo, *tabs)
    b = pipe.run_device(echo, *tabs)
    assert a.points.n == b.points.n and a.n_clusters == b.n_clusters > 3
    assert torch.equal(a.labels, b.labels) and torch.equal(a.points.x[:a.points.n], b.points.x[:b.points.n])
    lab = a.labels.cpu().numpy()
    first = [int(np.flatnonzero(lab == k)[0]) for k in range(a.n_clusters)]
    # the first CORE point of cluster k precedes that of cluster k+1; border points may come earlier, so check
    # through the ids' first occurrences being "almost sorted" is not enough - recompute from the core flags
    core = gpu.StDbscanPhases(a.points.x, a.points.y, None,
                              gpu.expand_frame_times(a.points.frame_off, torch.arange(spec.frames, dtype=torch.float32, device=echo.device),
                                                     a.points.n), 8.0, 2.0, 15, n=a.points.n).cores().cpu().numpy().astype(bool)
    first_core = [int(np.flatnonzero((lab == k) & core)[0]) for k in range(a.n_clusters)]
    assert first_core == sorted(first_core) and len(first) == a.n_clusters


@pytest.mark.parametrize("kw", [{}, {"land_filter": False}, {"eps_time": 0.5, "min_samples": 6}])
def test_native_block_driver_equals_staged_path(gpu, kw):
    """rb_detect_block (one call, native host driver, hinted ST-DBSCAN plan) against the same path driven stage
    by stage through the per-function entry points: identical raw points, grids, mask, filtered points, labels."""
    from radar_point_cloud_tracking_b200.pipeline import DetectionConfig, DetectionPipeline
    spec = syn.SweepSpec(seed=19, frames=14, spokes=384, bins=1024, clutter_p=0.006, land_blobs=3, buoys=3, boats=3)
    pipe = DetectionPipeline(DetectionConfig(**kw), 0)
    echo = gpu.synth_echo(spec)
    c, s, r = pipe.spoke_tables(spec.angle_units(), spec.scale(), spec.frames, spec.bins)
    tabs = [torch.from_numpy(t).to(echo.device) for t in (c, s, r)]
    ids = np.arange(100, 100 + spec.frames)
    a = pipe.run_device(echo, *tabs, frame_ids=ids)
    b = pipe.run_device_staged(echo, *tabs, frame_ids=ids)
    assert a.raw.n == b.raw.n > 0 and a.points.n == b.points.n and a.n_clusters == b.n_clusters
    for f in ("x", "y", "inten", "gain"):
        assert torch.equal(getattr(a.raw, f)[:a.raw.n], getattr(b.raw, f)[:b.raw.n])
        assert torch.equal(getattr(a.points, f)[:a.points.n], getattr(b.points, f)[:b.points.n])
    assert torch.equal(a.raw.frame_off, b.raw.frame_off) and torch.equal(a.points.frame_off, b.points.frame_off)
    assert torch.equal(a.labels, b.labels)
    if kw.get("land_filter", True):
        assert np.array_equal(a.edges[0], b.edges[0]) and np.array_equal(a.edges[1], b.edges[1])
        assert torch.equal(a.count, b.count) and torch.equal(a.isum, b.isum) and torch.equal(a.land, b.land)
    else:
        assert a.land is None and a.points.n == a.raw.n
    empty = pipe.run_device(torch.zeros_like(echo), *tabs)              # nothing above the threshold
    assert empty.raw.n == 0 and empty.points.n == 0 and empty.n_clusters == 0 and empty.labels.numel() == 0


def test_overlapped_pipeline_equals_sequential(gpu):
    """Two host threads / CUDA streams / library contexts running blocks concurrently give the per-block results
    of the sequential driver."""
    from radar_point_cloud_tracking_b200.pipeline import DetectionConfig, DetectionPipeline, OverlappedPipeline
    cfg = DetectionConfig()
    specs = [syn.SweepSpec(seed=40 + k, frames=12, spokes=256, bins=1024, clutter_p=0.006, land_blobs=2, buoys=2, boats=2) for k in range(5)]
    pipe = DetectionPipeline(cfg, 0)
    blocks, want = [], []
    for sp in specs:
        echo = gpu.synth_echo(sp)
        c, s, r = pipe.spoke_tables(sp.angle_units(), sp.scale(), sp.frames, sp.bins)
        tabs = [torch.from_numpy(t).to(echo.device) for t in (c, s, r)]
        blocks.append(((echo, *tabs), {}))
        want.append(pipe.run_device(echo, *tabs))
    torch.cuda.synchronize()
    op = OverlappedPipeline(cfg, 0, workers=2)
    try:
        got = op.map(blocks * 2)
        torch.cuda.synchronize()
        assert op.launch_count() > 0
    finally:
        op.close()
    for k, g in enumerate(got):
        w = want[k % len(want)]
        assert g.points.n == w.points.n and g.n_clusters == w.n_clusters
        assert torch.equal(g.labels, w.labels) and torch.equal(g.points.x[:g.points.n], w.points.x[:w.points.n])


@pytest.mark.parametrize("S,E,thr,stride", [(2048, 1024, 10.0, 4), (64, 1024, 9.5, 3), (33, 130, 8.0, 1), (17, 1000, 2.0, 2),
                                            (5, 1023, -1.0, 5), (40, 512, 254.0, 1), (40, 512, 255.0, 1), (40, 512, 0.0, 7)])
def test_spoke_to_points_uint8_equals_float32(gpu, S, E, thr, stride):
    """uint8 echoes (integer compare on four cells at a time, 16-byte bulk copies when S*E % 16 == 0, scalar
    fallback otherwise) give exactly the float32 result: fractional, negative and saturating thresholds."""
    from radar_point_cloud_tracking_b200 import _lib
    spec = syn.SweepSpec(seed=13, frames=2, spokes=S, bins=E, clutter_p=0.02, land_blobs=1, buoys=1, boats=1)
    echo = syn.synth_echo(spec).reshape(-1, S, E)
    echo[0, 0, :min(E, 8)] = [0, 255, 254, 1, 10, 9, 11, 255][:min(E, 8)]
    assert np.array_equal(echo, echo.astype(np.uint8).astype(np.float32))       # the generator emits 0..255 integers
    d = torch.device("cuda:0")
    c, s, r = _tables(gpu, spec, 6, d)
    gains = torch.tensor([40, 50, 75] * 2, dtype=torch.int32, device=d)
    outs = []
    for t in (torch.from_numpy(echo).to(d), torch.from_numpy(echo.astype(np.uint8)).to(d)):
        outs.append(gpu.spoke_to_points(t, c, s, r, gains, thr, stride, gains_per_frame=3))
        want_variant = 2 if (S * E) % (16 if t.dtype == torch.uint8 else 4) == 0 else 1
        assert _lib.context(0).info("spoke_last_variant") == want_variant
    a, b = outs
    assert a.n == b.n and torch.equal(a.frame_off, b.frame_off)
    for f in ("x", "y", "inten", "gain"):
        assert torch.equal(getattr(a, f)[:a.n], getattr(b, f)[:b.n])
    assert (a.n > 0) == (thr < 255.0)


def test_pipeline_uint8_block_equals_float32(gpu):
    from radar_point_cloud_tracking_b200.pipeline import DetectionConfig, DetectionPipeline
    spec = syn.SweepSpec(seed=23, frames=12, spokes=512, bins=1024, clutter_p=0.005)
    pipe = DetectionPipeline(DetectionConfig(), 0)
    echo = gpu.synth_echo(spec)
    c, s, r = pipe.spoke_tables(spec.angle_units(), spec.scale(), spec.frames, spec.bins)
    tabs = [torch.from_numpy(t).to(echo.device) for t in (c, s, r)]
    a = pipe.run_device(echo, *tabs)
    b = pipe.run_device(echo.to(torch.uint8), *tabs)
    assert a.points.n == b.points.n > 0 and a.n_clusters == b.n_clusters > 0
    assert torch.equal(a.labels, b.labels) and torch.equal(a.points.inten[:a.points.n], b.points.inten[:b.points.n])
    h = pipe.run_host(echo.to(torch.uint8).cpu().numpy(), spec.angle_units(), spec.scale())
    assert np.array_equal(h["labels"], a.labels.cpu().numpy()) and h["h2d_bytes"] < echo.numel() * 1.1


# ------------------------------------------------------------------------------- f3: PointCloudWorkF variant
def test_stdbscan_wf_variant_vs_reference_golden(gpu, db_mode):
    """min_frames core test + FIFO border rule: labels identical to the unmodified reference function (golden)."""
    from radar_point_cloud_tracking_b200.clustering import st_dbscan
    g = golden("wf_stdbscan")
    for k in range(int(g["n_cases"])):
        eps_s, eps_t, ms, mf = g[f"c{k}_params"]
        got = st_dbscan(g[f"c{k}_coords"], g[f"c{k}_times"], float(eps_s), float(eps_t), int(ms), min_frames=int(mf))
        assert np.array_equal(got, g[f"c{k}_labels"]), k


@pytest.mark.parametrize("n,frames,eps_s,eps_t,ms,mf", [(60000, 30, 8.0, 2.0, 15, 2), (40000, 12, 6.0, 1.0, 8, 3), (30000, 6, 5.0, 1.5, 6, 2)])
def test_stdbscan_wf_variant_vs_c_oracle_medium(gpu, db_mode, n, frames, eps_s, eps_t, ms, mf):
    from oracle.c_oracle import st_dbscan_wf_c
    rng = np.random.default_rng(n + mf)
    coords = (rng.random((n, 2)) * 400).astype(np.float32)
    centres = (rng.random((40, 2)) * 400).astype(np.float32)
    coords[: n // 2] = (centres[rng.integers(0, 40, n // 2)] + rng.normal(0, 3.0, (n // 2, 2))).astype(np.float32)
    coords = coords[rng.permutation(n)]
    times = rng.integers(0, frames, n).astype(np.float32) if eps_t == int(eps_t) else (rng.random(n) * frames).astype(np.float32)
    want, want_core = st_dbscan_wf_c(coords, times, eps_s, eps_t, ms, mf)
    plain, _ = st_dbscan_c(coords, times, eps_s, eps_t, ms)
    assert (want != plain).any()                                   # the variant really differs from T4 on this case
    d = torch.device("cuda:0")
    flat = torch.from_numpy(coords).to(d).view(-1)
    lab, core, ncl = gpu.stdbscan(flat, flat[1:], None, torch.from_numpy(times).to(d), eps_s, eps_t, ms, stride=2, n=n,
                                  want_core=True, min_frames=mf)
    assert np.array_equal(core.cpu().numpy().astype(bool), want_core)
    assert np.array_equal(lab.cpu().numpy(), want) and ncl == want.max() + 1


def test_stdbscan_partition_is_permutation_invariant_at_scale(gpu):
    """Size-independent property on a full-size block (64 frames, ~150 k points after the land filter): shuffling
    the points changes cluster NUMBERS (ranks of smallest core indices) and which cluster a shared border point
    joins, but not the core set, the partition of the core points or the noise set."""
    from radar_point_cloud_tracking_b200.pipeline import DetectionConfig, DetectionPipeline
    spec = syn.SweepSpec(seed=77, frames=64)
    pipe = DetectionPipeline(DetectionConfig(), 0)
    echo = gpu.synth_echo(spec)
    c, s, r = pipe.spoke_tables(spec.angle_units(), spec.scale(), spec.frames, spec.bins)
    res = pipe.run_device(echo, *(torch.from_numpy(t).to(echo.device) for t in (c, s, r)))
    n = res.points.n
    assert n > 100_000 and res.n_clusters > 5
    d = echo.device
    x, y = res.points.x[:n], res.points.y[:n]
    t = gpu.expand_frame_times(res.points.frame_off, torch.arange(spec.frames, dtype=torch.float32, device=d), n)
    lab1, core1, ncl1 = gpu.stdbscan(x, y, None, t, 8.0, 2.0, 15, n=n, want_core=True)
    assert torch.equal(lab1, res.labels)                         # the block driver's labels are rb_stdbscan's
    perm = torch.randperm(n, device=d, generator=torch.Generator(device=d).manual_seed(3))
    lab2, core2, ncl2 = gpu.stdbscan(x[perm].contiguous(), y[perm].contiguous(), None, t[perm].contiguous(), 8.0, 2.0, 15, n=n,
                                     want_core=True)
    assert ncl1 == ncl2 and torch.equal(core1[perm], core2)
    a, b = lab1[perm].cpu().numpy(), lab2.cpu().numpy()
    cm = core2.cpu().numpy().astype(bool)
    assert np.array_equal(a < 0, b < 0)                          # same noise set
    pairs = np.unique(np.stack([a[cm], b[cm]]), axis=1)          # label map between the two runs on core points
    assert pairs.shape[1] == ncl1 and len(np.unique(pairs[0])) == ncl1 and len(np.unique(pairs[1])) == ncl1


def test_result_read_back_modes_agree_and_results_stay_valid(gpu, monkeypatch):
    dev = gpu
    """device.to_pinned_host: the staging path (default), fresh pinned tensors and plain .cpu() hand out the same arrays;
    arrays of an earlier call are not touched by later calls (the staging buffer is reused, the results are copies)."""
    import torch
    d = torch.device("cuda", 0)
    g = torch.Generator(device="cpu").manual_seed(5)
    ts = [torch.randn(70001, 3, generator=g).to(d), torch.arange(333, dtype=torch.int32, device=d), torch.zeros(0, dtype=torch.int32, device=d),
          torch.randint(0, 255, (1025,), dtype=torch.uint8, generator=g).to(d), torch.arange(129, dtype=torch.int64, device=d)]
    want = [t.cpu().numpy() for t in ts]
    kept = {}
    for mode in ("staging", "pinned", "pageable"):
        monkeypatch.setattr(dev, "HOST_READBACK_MODE", mode)
        kept[mode] = dev.to_pinned_host(*ts)
        for a, b in zip(kept[mode], want):
            assert a.dtype == b.dtype and a.shape == b.shape and np.array_equal(a, b)
    monkeypatch.setattr(dev, "HOST_READBACK_MODE", "staging")
    dev.to_pinned_host(*[t * 0 for t in ts])                          # overwrites the staging buffer
    dev.to_pinned_host(torch.ones(4_000_000, device=d))               # grows it
    for mode in kept:
        for a, b in zip(kept[mode], want):
            assert np.array_equal(a, b)
