"""Whole recordings from sweep CSV files: rb_csv_parse_sweeps (many files per launch) against pandas, and
RecordingDetection.add_csv_frames against the reference's clusters.csv, against add_block of the decoded echoes, and
against the installed drop-in (build_frame per frame, land, st_dbscan) on an irregular tree."""
import io

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from radar_point_cloud_tracking_b200 import synthetic as syn
from radar_point_cloud_tracking_b200._lib import RadarB200Error
from tests.common import golden, pipe_inputs

pytestmark = pytest.mark.gpu

SPEC = dict(seed=77, frames=2, spokes=96, bins=160, clutter_p=0.02, land_blobs=1, buoys=2, boats=2)
LEAD = 32


@pytest.fixture(scope="module")
def gpu():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (no CPU fallback exists)")
    torch.cuda.set_device(0)
    from radar_point_cloud_tracking_b200 import csvbatch, tracker
    return csvbatch, tracker


def _variants(tmp_path, rows, E):
    """The files of test_gpu_csv_ingest.py's variants: (path, expected to stay on the device)."""
    out = []

    def variant(name, new_rows, sep="\n", device=True):
        p = tmp_path / name
        p.write_bytes(sep.join(new_rows).encode())
        out.append((p, device))

    variant("crlf.csv", rows, "\r\n")
    variant("open_tail.csv", rows[:-1])
    r = rows[3].split(",")
    r[5], r[5 + E - 1], r[40] = "", "", "007"
    r[1] = "926.5"
    variant("empties.csv", rows[:3] + [",".join(r)] + rows[4:])
    variant("header_only.csv", [rows[0], ""])
    variant("empty.csv", [""])
    for name, field in (("decimal_echo.csv", "12.5"), ("big_echo.csv", "300"), ("negative_echo.csv", "-3"), ("spaced.csv", " 7")):
        r = rows[5].split(",")
        r[20] = field
        variant(name, rows[:5] + [",".join(r)] + rows[6:], device=False)
    variant("cr_only.csv", rows, "\r", device=False)
    r = rows[6].split(",")
    r[2] = "3\r"
    variant("stray_cr.csv", rows[:6] + [",".join(r)] + rows[7:], device=False)
    variant("blank_line.csv", rows[:4] + [""] + rows[4:], device=False)
    variant("short_row.csv", rows[:4] + [",".join(rows[4].split(",")[:-3])] + rows[5:], device=False)
    return out


def _same_sweep(got, want):
    if want is None:
        assert got is None
        return
    a0, s0, e0, g0 = want
    a1, s1, e1, g1 = got
    e1 = e1.cpu().numpy().astype(np.float32) if isinstance(e1, torch.Tensor) else e1
    assert g0 == g1 and a1.dtype == np.float32 and s1.dtype == np.float32
    assert np.array_equal(a0, a1, equal_nan=True) and np.array_equal(s0, s1, equal_nan=True)
    assert np.array_equal(a0.view(np.uint32), np.asarray(a1).view(np.uint32))
    assert np.array_equal(s0.view(np.uint32), np.asarray(s1).view(np.uint32))
    assert e0.shape == e1.shape and np.array_equal(e0, e1, equal_nan=True)


def test_batch_parser_matches_pandas(gpu, tmp_path):
    cb, trk = gpu
    spec = syn.SweepSpec(**SPEC)
    E = spec.bins
    tree = syn.write_csv_tree(spec, tmp_path / "a")
    short = syn.write_csv_tree(syn.SweepSpec(**dict(SPEC, spokes=40, seed=5)), tmp_path / "b")
    first = next(iter(tree[0].values()))
    rows = first.read_text().split("\n")
    files = [(p, True) for entry in tree for p in entry.values()]
    var = _variants(tmp_path, rows, E)
    # an open tail followed by another file; files of different row counts in between
    files = files[:2] + var + [(p, True) for p in short[0].values()] + files[2:]
    res = cb.parse_files([p for p, _ in files], E)
    assert len(res) == len(files)
    for (p, on_device), r in zip(files, res):
        drop = trk.read_sweep_csv_device(p, E)
        assert (drop is not None and isinstance(drop[2], torch.Tensor)) == (r.sweep is not None and isinstance(r.sweep[2], torch.Tensor)), p.name
        if r.sweep is not None:
            assert isinstance(r.sweep[2], torch.Tensor) == on_device, p.name
        assert ((r.status & ~LEAD) == 0) == (on_device or r.sweep is None), p.name
        _same_sweep(r.sweep, trk.read_sweep_csv(p, E))


def _lead_token(rng, integer):
    nd = int(rng.integers(1, 16))
    digits = "".join(str(int(v)) for v in rng.integers(0, 10, nd))
    k = 0 if integer or nd == 1 else int(rng.integers(1, nd))
    tok = digits if k == 0 else digits[:nd - k] + "." + digits[nd - k:]
    neg = rng.random() < 0.3 and int(digits) != 0
    return ("-" + tok) if neg else tok


def test_leading_fields_match_pandas(gpu, tmp_path):
    cb, trk = gpu
    rng = np.random.default_rng(9)
    E, S = 6, 300
    header = "Status,Scale,Range,Gain,Angle," + ",".join(f"Echo_{i}" for i in range(E))

    def write(name, angles, scales, gain="40"):
        lines = [header] + [f"1,{s},3,{gain},{a}," + ",".join(str(int(v)) for v in rng.integers(0, 256, E)) for a, s in zip(angles, scales)]
        p = tmp_path / name
        p.write_text("\n".join(lines) + "\n")
        return p

    inside = []
    for i, mode in enumerate(("int", "dec", "mixed", "mixed", "mixed")):
        def col():
            return [_lead_token(rng, mode == "int" or (mode == "mixed" and rng.random() < 0.5)) for _ in range(S)]
        inside.append(write(f"in_{i}.csv", col(), col(), gain=str(int(rng.integers(-99999, 99999)))))
    outside = []
    for j, bad in enumerate(("-0", "-0.0", "1e2", "+5", ".5", "5.", "1234567890123456", "", " 5", "0.1234567890123456")):
        for col in ("angle", "scale"):
            a = [_lead_token(rng, False) for _ in range(S)]
            s = [_lead_token(rng, False) for _ in range(S)]
            (a if col == "angle" else s)[int(rng.integers(0, S))] = bad
            outside.append(write(f"out_{j}_{col}.csv", a, s))
    outside.append(write("gain_dec.csv", ["1"] * S, ["2"] * S, gain="40.0"))
    res = cb.parse_files(inside + outside, E)
    for p, r in zip(inside + outside, res):
        want = trk.read_sweep_csv(p, E)
        assert ((r.status & LEAD) != 0) == (p in outside), p.name
        assert (r.status & ~LEAD) == 0 and isinstance(r.sweep[2], torch.Tensor)
        _same_sweep(r.sweep, want)


def _golden_rows(clusters):
    return np.array(sorted((fid, c.cluster_id, c.num_points, c.centroid[0], c.centroid[1], c.mean_intensity)
                           for fid, cl in clusters.items() for c in cl), dtype=np.float64).reshape(-1, 6)


@pytest.fixture(scope="module")
def pipe_tree(tmp_path_factory):
    root = tmp_path_factory.mktemp("pipe") / "data"
    spec, echo = pipe_inputs()
    return spec, echo, syn.write_csv_tree(spec, root, echo)


@pytest.mark.parametrize("tag,kw", [("default", {}),
                                    ("nofilter_eps6", dict(skip_land_filter=True, eps_space=6.0, eps_time=1.0, min_samples=8))])
def test_csv_recording_reproduces_the_reference_clusters_csv(gpu, pipe_tree, tag, kw):
    cb, trk = gpu
    from radar_point_cloud_tracking_b200.pipeline import DetectionConfig
    from radar_point_cloud_tracking_b200.recording import RecordingDetection
    _, _, files = pipe_tree
    p = dict(dict(skip_land_filter=False, eps_space=trk.EPS_SPACE, eps_time=trk.EPS_TIME, min_samples=trk.MIN_SAMPLES), **kw)
    text = str(golden("run_pipeline_csv")[f"{tag}/clusters.csv"])
    want = np.loadtxt(io.StringIO(text), delimiter=",", skiprows=1, ndmin=2)
    want = want[np.lexsort((want[:, 1], want[:, 0]))]
    rec = RecordingDetection(DetectionConfig(land_filter=not p["skip_land_filter"], eps_space=p["eps_space"], eps_time=p["eps_time"],
                                             min_samples=p["min_samples"]), 0)
    rec.add_csv_frames(files)
    res = rec.finish()
    via_tracker = trk.detect_csv_frames(files, **p)
    for clusters in (res.clusters_by_frame(), via_tracker):
        got = _golden_rows(clusters)
        assert len(want) > 0 and got.shape == want.shape
        assert np.array_equal(got[:, :3], want[:, :3])
        assert np.array_equal(got[:, 3:].astype(np.float32), want[:, 3:].astype(np.float32))
    assert res.frame_times == [trk.parse_timestamp(sorted(f.items())[0][1].name) for f in files]


def _same_batch(a, b):
    assert a.n == b.n
    assert torch.equal(a.frame_off, b.frame_off)
    for k in ("x", "y", "inten", "gain"):
        assert torch.equal(getattr(a, k)[:a.n], getattr(b, k)[:b.n]), k


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


def test_csv_frames_equal_decoded_blocks(gpu, pipe_tree):
    from radar_point_cloud_tracking_b200.pipeline import DetectionConfig
    from radar_point_cloud_tracking_b200.recording import RecordingDetection
    cb, _ = gpu
    spec, echo, files = pipe_tree
    ids = np.arange(spec.frames) * 2 + 3
    ref = RecordingDetection(DetectionConfig(), 0)
    ref.add_host_block(echo, spec.angle_units(), spec.scale(), ids)
    one = ref.finish()
    assert one.land is not None and one.n_clusters > 0
    per_frame = max(sum(cb.aligned(p.stat().st_size) for p in f.values()) for f in files)
    for batch in (256 << 20, per_frame):
        rec = RecordingDetection(DetectionConfig(), 0)
        if batch == per_frame:                                     # in two calls, the ids continuing
            rec.add_csv_frames(files[:5], ids[:5], batch_bytes=batch, readers=3)
            rec.add_csv_frames(files[5:], ids[5:], batch_bytes=batch)
            assert len(rec._offs) - 1 == spec.frames                 # one batch (block) per frame
        else:
            rec.add_csv_frames(files, ids, batch_bytes=batch)
            assert len(rec._offs) - 1 == 1                           # one batch
        _assert_same(rec.finish(), one)


def _rewrite(src, dst, fn):
    rows = src.read_text().split("\n")
    dst.write_text("\n".join(fn(rows)))
    return dst


def test_irregular_tree_matches_the_drop_in(gpu, tmp_path, capsys):
    cb, trk = gpu
    from radar_point_cloud_tracking_b200.pipeline import DetectionConfig
    from radar_point_cloud_tracking_b200.recording import RecordingDetection
    E = 256
    a = syn.write_csv_tree(syn.SweepSpec(seed=41, frames=13, spokes=64, bins=E, clutter_p=0.02, land_blobs=2, buoys=3, boats=2), tmp_path / "a")
    b = syn.write_csv_tree(syn.SweepSpec(seed=42, frames=13, spokes=48, bins=E, clutter_p=0.02, land_blobs=2, buoys=3, boats=2), tmp_path / "b",
                           start="20250813_142602")
    odd = tmp_path / "odd"
    odd.mkdir()
    empty1, empty2 = odd / "20250813_150000_000.csv", odd / "20250813_150000_100.csv"
    empty1.write_text(""), empty2.write_text("")

    def dec_echo(rows):
        r = rows[7].split(",")
        r[29:37] = ["212.5"] * 8
        return rows[:7] + [",".join(r)] + rows[8:]

    def lead_out(rows):
        r = rows[3].split(",")
        r[1] = "231.50000000000000001"                         # 20 digits: pandas reads the Scale column
        return rows[:3] + [",".join(r)] + rows[4:]

    frames = []
    for f in range(13):
        fa, fb = a[f], b[f]
        if f == 1:
            frames.append({40: fa[40], 75: fb[75]})             # missing gain 50; 64 and 48 spokes in one frame
        elif f == 2:
            frames.append({40: empty1, 50: empty2})             # no points: the id is consumed
        elif f == 3:
            frames.append({40: odd / "20250813_150100_000.csv", 50: fa[50], 75: fa[75]})      # a missing path
        elif f == 4:
            frames.append(dict(fb))                              # 48 spokes
        elif f == 5:
            frames.append({40: _rewrite(fa[40], odd / "20250813_150200_000.csv", dec_echo), 50: fb[50], 75: fa[75]})
        elif f == 6:
            frames.append({40: fa[40], 50: _rewrite(fa[50], odd / "20250813_150300_000.csv", lead_out)})
        else:
            frames.append(dict(fa) if f % 2 else dict(fb))
    ids = np.arange(13) * 3 + 5
    cfg = DetectionConfig(eps_time=4.0, min_samples=6)
    rec = RecordingDetection(cfg, 0)
    rec.add_csv_frames(frames, ids, num_echo_columns=E)
    res = rec.finish()
    printed = capsys.readouterr().out
    assert "Error loading" in printed and "20250813_150100_000.csv" in printed

    class Cfg:
        NUM_ECHO_COLUMNS, INTENSITY_THRESHOLD, POINT_STRIDE = E, cfg.intensity_threshold, cfg.point_stride
        LAND_PERSISTENCE_THRESHOLD, LAND_GRID_RESOLUTION, LAND_MIN_INTENSITY = cfg.land_persistence, cfg.land_resolution, cfg.land_min_intensity
    built = [fr for fr in (trk.build_frame(ff, int(i), _cfg=Cfg) for ff, i in zip(frames, ids)) if fr is not None]
    assert len(built) == 12 and res.frames_built == 12 and res.land is not None and res.land_ordered
    count, isum, edges = trk.build_occupancy_grid(built, cfg.land_resolution)
    land = trk.identify_land_cells(count, isum, len(built), _cfg=Cfg)
    built = [trk.filter_land_from_frame(fr, land, edges) for fr in built]
    want = trk.st_dbscan(built, cfg.eps_space, cfg.eps_time, cfg.min_samples)
    got = res.clusters_by_frame()
    assert len(want) > 0 and sorted(got) == sorted(int(k) for k in want)
    for fid, cl in want.items():
        g = sorted(got[int(fid)], key=lambda c: c.cluster_id)
        w = sorted(cl, key=lambda c: c.cluster_id)
        assert [c.cluster_id for c in g] == [c.cluster_id for c in w]
        for cg, cw in zip(g, w):
            assert np.array_equal(cg.points, cw.points) and np.array_equal(cg.centroid, cw.centroid)
            assert np.array_equal(cg.intensities, cw.intensities)
    assert res.frame_ids.tolist() == ids.tolist()
    assert res.frame_times[2] == trk.parse_timestamp(empty1.name)


def test_at_size_equals_host_block(gpu, tmp_path):
    from radar_point_cloud_tracking_b200.pipeline import DetectionConfig
    from radar_point_cloud_tracking_b200.recording import RecordingDetection
    spec = syn.SweepSpec(seed=12, frames=2)
    echo = syn.synth_echo(spec)
    files = syn.write_csv_tree(spec, tmp_path, echo)
    ref = RecordingDetection(DetectionConfig(), 0)
    ref.add_host_block(echo.astype(np.uint8), spec.angle_units(), spec.scale(), [0, 1])
    rec = RecordingDetection(DetectionConfig(), 0)
    rec.add_csv_frames(files)
    one, got = ref.finish(), rec.finish()
    assert got.raw.n > 0
    _assert_same(got, one)


def test_csv_input_errors(gpu, pipe_tree):
    from radar_point_cloud_tracking_b200.pipeline import DetectionConfig
    from radar_point_cloud_tracking_b200.recording import RecordingDetection
    _, _, files = pipe_tree
    rec = RecordingDetection(DetectionConfig(), 0)
    rec.add_csv_frames([])                                        # nothing to add
    for bad in ([3, 2], [1]):                                     # ids without frames
        with pytest.raises(RadarB200Error):
            rec.add_csv_frames([], bad)
    with pytest.raises(RadarB200Error):
        rec.add_csv_frames(files[:2], [5, 4])
    with pytest.raises(RadarB200Error):
        rec.add_csv_frames(files[:2], num_echo_columns=0)
    rec.add_csv_frames(files[:2], [5, 6])
    with pytest.raises(RadarB200Error):
        rec.add_csv_frames(files[2:3], [6])                      # ids must continue to increase
    rec.finish()
    with pytest.raises(RadarB200Error):
        rec.add_csv_frames(files[2:3])


def test_slots_grow_for_later_calls(gpu, tmp_path):
    """A first call with little to read (an empty file; a frame missing a gain) must not leave later calls with slots
    too small for their frames: every file of the later full frames (1.2 MB sweeps) is parsed in a batch."""
    cb, _ = gpu
    from radar_point_cloud_tracking_b200.pipeline import DetectionConfig
    from radar_point_cloud_tracking_b200.recording import RecordingDetection
    files = syn.write_csv_tree(syn.SweepSpec(seed=3, frames=3, spokes=512, bins=1024, clutter_p=0.01), tmp_path / "t")
    empty = tmp_path / "20250813_140000_000.csv"
    empty.write_text("")
    per_frame = max(sum(cb.aligned(p.stat().st_size) for p in f.values()) for f in files)
    for first in ([{40: empty}], [{40: files[0][40], 50: files[0][50]}]):
        rec = RecordingDetection(DetectionConfig(), 0)
        rec.add_csv_frames(first)
        small = rec._reader.slot_bytes
        assert small < per_frame
        rec.add_csv_frames(files[1:])
        assert rec._reader.slot_bytes >= per_frame
        assert rec.csv_files == {"batched": len(first[0]) + 3 * (len(files) - 1), "per_file": 0}
        assert rec.finish().frames_built == len(files) - (first[0].get(40) == empty)
