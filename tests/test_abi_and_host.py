"""CPU-side checks: the C-ABI library loads and exports every symbol the header declares, the host
logic (tables, edges, config plumbing) matches the oracle, and the product path refuses to run
without a GPU instead of falling back to anything."""
import ctypes
import re
from pathlib import Path

import numpy as np
import pytest

from oracle import numpy_oracle as O
from radar_point_cloud_tracking_b200 import _lib, synthetic as syn
from radar_point_cloud_tracking_b200 import tracker as trk

REPO = Path(__file__).resolve().parent.parent


def header_symbols():
    text = (REPO / "include" / "radarb200.h").read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(rb_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    lib = _lib.load()
    names = header_symbols()
    assert len(names) >= 18
    assert sorted(_lib.SIGNATURES) == names            # the binding covers the header, nothing more
    raw = ctypes.CDLL(str(_lib.LIB_PATH))
    for n in names:
        assert getattr(raw, n) is not None
    assert lib.rb_version() == 1


def test_library_is_sm100a_only():
    import subprocess
    out = subprocess.run(["cuobjdump", "-lelf", str(_lib.LIB_PATH)], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_\d+a?", out))
    assert archs == {"sm_100a"}, archs


def test_no_gpu_is_a_hard_error():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from radar_point_cloud_tracking_b200.clustering import st_dbscan
    from radar_point_cloud_tracking_b200.pipeline import DetectionPipeline
    with pytest.raises(_lib.RadarB200Error):
        st_dbscan(np.zeros((4, 2), np.float32), np.zeros(4, np.float32), 1.0, 1.0, 2)
    with pytest.raises(_lib.RadarB200Error):
        DetectionPipeline()
    with pytest.raises(_lib.RadarB200Error):
        _lib.context()
    h = ctypes.c_void_p()
    assert _lib.load().rb_create(0, ctypes.byref(h)) != 0 and b"no CUDA device" in _lib.load().rb_last_error()


def test_product_package_never_imports_the_oracle():
    for py in (REPO / "radar_point_cloud_tracking_b200").glob("*.py"):
        src = py.read_text()
        assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), py
        assert "sklearn" not in src and "BallTree" not in src, py


def test_sweep_tables_match_reference_expressions():
    spec = syn.SweepSpec(spokes=2048, bins=1024)
    c, s, r = trk.sweep_tables(spec.angle_units(), spec.scale(), spec.bins)
    oc, os_, or_ = O.spoke_tables(spec.angle_units(), spec.scale(), spec.bins)
    assert c.dtype == np.float32 and np.array_equal(c, oc) and np.array_equal(s, os_) and np.array_equal(r, or_)
    # [W, S] batches give the same rows
    a2 = np.stack([spec.angle_units(), spec.angle_units()[::-1]])
    c2, s2, r2 = trk.sweep_tables(a2, np.stack([spec.scale(), spec.scale() * 2]), 1000)
    assert np.array_equal(c2[0], c) and np.array_equal(s2[1], s[::-1])
    assert np.array_equal(r2[1], (spec.scale() * 2 / 1000).astype(np.float32))


def test_grid_edges_match_numpy_arange_of_float32_bounds():
    rng = np.random.default_rng(0)
    for _ in range(50):
        lo, hi = np.sort(rng.normal(0, 300, 2)).astype(np.float32)
        xe, ye = trk.grid_edges_from_bounds(np.array([lo, hi, lo, hi], np.float32), 5.0)
        assert xe.dtype == np.float64 and np.array_equal(xe, O.grid_edges(lo, hi, 5.0)) and np.array_equal(xe, ye)


def test_parse_timestamp_and_csv_reader(tmp_path):
    dt, ms = trk.parse_timestamp("20250813_142602_181.csv")
    assert (dt.year, dt.second, ms % 1000) == (2025, 2, 181)
    with pytest.raises(ValueError):
        trk.parse_timestamp("nope.csv")
    spec = syn.SweepSpec(seed=1, frames=1, spokes=4, bins=1024, gains=(75,))
    files = syn.write_csv_tree(spec, tmp_path)
    angle, scale, echo, gain = trk.read_sweep_csv(files[0][75])
    assert gain == 75 and echo.shape == (4, 1024) and echo.dtype == np.float32
    assert np.array_equal(echo, syn.synth_echo(spec)[0, 0]) and np.array_equal(angle, spec.angle_units())
    assert trk.read_sweep_csv(tmp_path / "missing.csv") is None


def test_install_reads_reference_globals_at_call_time():
    from types import SimpleNamespace
    ref = SimpleNamespace(RadarFrame=trk.RadarFrame, Cluster=trk.Cluster, NUM_ECHO_COLUMNS=1024,
                          INTENSITY_THRESHOLD=10.0, POINT_STRIDE=4, LAND_PERSISTENCE_THRESHOLD=0.8,
                          LAND_GRID_RESOLUTION=5.0, LAND_MIN_INTENSITY=100)
    trk.install(ref)
    for name in ("load_radar_csv", "build_frame", "build_occupancy_grid", "identify_land_cells",
                 "filter_land_from_frame", "st_dbscan"):
        assert callable(getattr(ref, name))
    ref.INTENSITY_THRESHOLD = 2.0
    assert trk._module_config(ref).INTENSITY_THRESHOLD == 2.0
    assert ref.st_dbscan([], 8.0, 2.0, 15) == {}


def test_synthetic_generator_is_deterministic():
    spec = syn.SweepSpec(seed=3, frames=2, spokes=16, bins=64)
    a, b = syn.synth_echo(spec), syn.synth_echo(spec)
    assert np.array_equal(a, b) and a.dtype == np.float32 and a.min() >= 0 and a.max() <= 255
    assert np.array_equal(a, np.rint(a))


def test_native_arange_edges_match_numpy():
    """rb_arange_edges (host code of the library, used by rb_detect_block) == np.arange on float32 scalar
    bounds, bit for bit - length rule and fill rule of numpy (T4:372-373)."""
    from radar_point_cloud_tracking_b200 import device as dev
    rng = np.random.default_rng(3)
    for _ in range(2000):
        lo, hi = np.sort(rng.normal(0, 400, 2)).astype(np.float32)
        step = float(rng.choice([5.0, 1.0, 2.5, 0.7, 3.3, 10.0]))
        ref = np.arange(lo, hi + step, step)
        got = dev.arange_edges(lo, hi, step)
        assert ref.dtype == np.float64 and np.array_equal(ref, got)
    assert len(dev.arange_edges(3.0, 3.0, 5.0)) == 1 and len(dev.arange_edges(0.0, 10.0, 5.0)) == 3


def test_stitch_components_matches_a_plain_union_find():
    """Native rb_stitch_components (host function) against a dictionary union-find, random component graphs."""
    from radar_point_cloud_tracking_b200.sharded import stitch_components

    rng = np.random.default_rng(5)
    e = np.zeros(0, np.int64)
    for world in (2, 3, 5):
        # rank r sees components keyed by random global indices; neighbouring ranks share boundary points
        keys = [np.unique(rng.integers(0, 10_000, size=rng.integers(1, 40))).astype(np.int64) for _ in range(world)]
        segs = [[e, e, e, e] for _ in range(world)]
        for r in range(world - 1):
            n_last, n_first = int(rng.integers(0, 30)), int(rng.integers(0, 30))
            segs[r][2], segs[r + 1][0] = rng.choice(keys[r], n_last), rng.choice(keys[r + 1], n_last)
            segs[r][3], segs[r + 1][1] = rng.choice(keys[r], n_first), rng.choice(keys[r + 1], n_first)
        tk, ti, ncl = stitch_components(segs, keys)
        parent = {int(k): int(k) for k in np.concatenate(keys)}

        def find(x):
            while parent[x] != x:
                x = parent[x]
            return x
        for r in range(world - 1):
            for a, b in ((segs[r][2], segs[r + 1][0]), (segs[r][3], segs[r + 1][1])):
                for u, v in zip(a.tolist(), b.tolist()):
                    ru, rv = find(u), find(v)
                    if ru != rv:
                        parent[max(ru, rv)] = min(ru, rv)
        roots = sorted({find(k) for k in parent})
        want = {k: roots.index(find(k)) for k in parent}
        assert list(tk) == sorted(parent) and ncl == len(roots)
        assert [want[int(k)] for k in tk] == list(ti)


def test_pair_zone_runs_equals_positional_pairing():
    """The run-length encoded boundary zones of two neighbouring ranks (sharded.pair_zone_runs) give exactly the distinct
    key pairs of the position-by-position pairing of the decoded arrays."""
    from radar_point_cloud_tracking_b200.sharded import pair_zone_runs

    rng = np.random.default_rng(21)

    def encode(keys):
        if len(keys) == 0:
            return np.zeros(0, np.int64), np.zeros(0, np.int64)
        start = np.flatnonzero(np.concatenate([[True], keys[1:] != keys[:-1]]))
        return keys[start], start.astype(np.int64)

    for n in (0, 1, 7, 500, 20000):
        core = rng.random(n) < 0.7
        # two labelings of the same points: components of A are unions of runs, B's are a different coarsening
        a = np.where(core, 1000 + rng.integers(0, 6, n) * 3, -1).astype(np.int64)
        b = np.where(core, 5000 + (rng.integers(0, 4, n) + np.arange(n) // max(n // 3, 1)) * 7, -1).astype(np.int64)
        if n > 50:
            a[10:40] = np.where(core[10:40], 1000, -1)                     # a long run
        pa, pb = pair_zone_runs(*encode(a), *encode(b))
        want = np.unique(np.stack([a[core], b[core]], axis=1), axis=0) if core.any() else np.zeros((0, 2), np.int64)
        assert np.array_equal(np.stack([pa, pb], axis=1), want)
    with pytest.raises(Exception):
        pair_zone_runs(np.array([5, -1]), np.array([0, 3]), np.array([-1, 9]), np.array([0, 3]))      # core sets disagree


def test_clusters_from_records_replays_set_order():
    """device.clusters_from_records (host logic): from a segment table in (frame, label) order with first-occurrence
    indices it rebuilds {frame: [Cluster]} in the iteration order of set(frame_labels) - labels far beyond the set's
    table size, so hash collisions and table growth matter - with member arrays as views of the grouped arrays."""
    from radar_point_cloud_tracking_b200.device import clusters_from_records
    from radar_point_cloud_tracking_b200.tracker import Cluster

    rng = np.random.default_rng(23)
    sizes = [0, 900, 3, 2500, 0, 40]
    K = 700
    pts, labels = [], []
    for n in sizes:
        pts.append(np.column_stack([rng.normal(0, 50, n), rng.normal(0, 50, n), rng.random(n) * 255]).astype(np.float32))
        labels.append((rng.integers(-1, K, n) * (rng.random(n) < 0.8) - (rng.random(n) < 0.1)).clip(-1, K - 1).astype(np.int32))
    off = np.concatenate([[0], np.cumsum(sizes)])
    frame_ids = [11, 12, 13, 14, 15, 16]
    # the table the device would produce, built here with numpy: segments by frame, then label; grouped points stable
    rec = {k: [] for k in ("frame", "label", "first", "count", "start", "cx", "cy", "mean_intensity")}
    gx, gy, gi = [], [], []
    pos = 0
    for f, (p, lab) in enumerate(zip(pts, labels)):
        for l in np.unique(lab):
            m = np.flatnonzero(lab == l)
            rec["frame"].append(f); rec["label"].append(l); rec["first"].append(m[0]); rec["count"].append(len(m))
            if l < 0:
                rec["start"].append(-1); rec["cx"].append(0); rec["cy"].append(0); rec["mean_intensity"].append(0)
                continue
            cen, mi = O.cluster_means_f32(p[m, :2], p[m, 2])
            rec["start"].append(pos); rec["cx"].append(cen[0]); rec["cy"].append(cen[1]); rec["mean_intensity"].append(mi)
            gx.append(p[m, 0]); gy.append(p[m, 1]); gi.append(p[m, 2]); pos += len(m)
    rec = {k: np.array(v, dtype=np.int64 if k == "start" else np.float32 if k in ("cx", "cy", "mean_intensity") else np.int32)
           for k, v in rec.items()}
    rec.update(gx=np.concatenate(gx), gy=np.concatenate(gy), gi=np.concatenate(gi))
    got = clusters_from_records(rec, frame_ids, Cluster)
    want_frames = []
    for f, (p, lab) in enumerate(zip(pts, labels)):
        ids = set(lab)                                                 # the reference's loop, T4:518-534
        ids.discard(-1)
        if not ids:
            continue
        want_frames.append(frame_ids[f])
        g = got[frame_ids[f]]
        assert [c.cluster_id for c in g] == [int(c) for c in ids]      # the set's own iteration order
        for c, cid in zip(g, ids):
            m = lab == cid
            assert np.array_equal(c.points, p[m, :2]) and np.array_equal(c.intensities, p[m, 2])
            assert np.array_equal(c.centroid, np.mean(p[m, :2], axis=0)) and c.mean_intensity == float(np.mean(p[m, 2]))
            assert c.points.base is not None                           # a view into the grouped arrays, not a copy
    assert list(got) == want_frames


def test_read_back_staging_views_and_copies():
    """The result read-back goes through one reusable staging buffer per thread (device.to_pinned_host): views at aligned
    offsets with the tensors' dtypes and shapes, arrays handed out as copies, the buffer reused until it is too small."""
    import torch

    from radar_point_cloud_tracking_b200 import device as dv
    ts = [torch.randn(1000, 3), torch.arange(7, dtype=torch.int32), torch.zeros(0, 3),
          torch.randint(0, 255, (513,), dtype=torch.uint8), torch.arange(5, dtype=torch.int64)]
    total = sum((t.numel() * t.element_size() + 255) & ~255 for t in ts)
    buf = dv._staging_buffer(total, False)
    views = dv._staging_views(buf, ts)
    for v, t in zip(views, ts):
        assert v.dtype == t.dtype and v.shape == t.shape and (t.numel() == 0 or v.data_ptr() % 256 == buf.data_ptr() % 256)
        v.copy_(t)
    for v, t in zip(views, ts):
        assert np.array_equal(v.numpy(), t.numpy())
    assert dv._staging_buffer(16, False) is buf
    bigger = dv._staging_buffer(buf.numel() + 1, False)
    assert bigger is not buf and bigger.numel() > buf.numel()
    out = dv.to_pinned_host(*ts)                                    # host tensors: plain copies
    ts[1][0] = 99
    assert out[1][0] == 0 and all(np.array_equal(o[1:] if i == 1 else o, (t.numpy()[1:] if i == 1 else t.numpy())) for i, (o, t) in enumerate(zip(out, ts)))
