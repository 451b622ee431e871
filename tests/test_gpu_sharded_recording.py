"""ShardedRecording on one B200: worlds of 2 and 3 ranks as spawned processes that all use GPU 0. Every library call runs
on the GPU; the collectives go through gloo on host copies (GlooEngine below: NCCL refuses two ranks on one device), so
the protocol of ShardedRecording.finish runs with the real kernels. Every case is compared with one in-process
RecordingDetection fed the same frames: raw and filtered points with their offsets, land grid, sums and mask,
land_ordered, labels, core flags, n_clusters, frames_built and the cluster records, bit for bit and id for id."""
import multiprocessing as mp
import pickle
import socket
import traceback
from pathlib import Path

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from radar_point_cloud_tracking_b200 import synthetic as syn
from radar_point_cloud_tracking_b200._lib import RadarB200Error

pytestmark = pytest.mark.gpu

SPEC = dict(seed=31, frames=21, spokes=512, bins=1024, clutter_p=0.01, land_blobs=3, buoys=4, boats=3)
CSV_SPEC = dict(seed=41, frames=14, spokes=256, bins=1024, clutter_p=0.02, land_blobs=2, buoys=3, boats=2)
# name -> frames per rank (world 2, world 3), config, echo dtype and scale, window budget as a fraction of the points;
# cut_inside: the budget and the shares are such that windows are cut inside a rank as well as at rank edges
CASES = {
    "f32_e2_windows": dict(shares={2: [10, 11], 3: [5, 9, 7]}, cfg=dict(eps_time=2.0), window_div=10, cut_inside=True),
    "u8_e5": dict(shares={2: [9, 12], 3: [5, 9, 7]}, cfg=dict(eps_time=5.0), dtype="uint8", window_div=3),
    "f32_e7.5_3d": dict(shares={2: [10, 11], 3: [7, 7, 7]}, cfg=dict(eps_time=7.5, cluster_3d=True, eps_space=30.0), window_div=2),
    "u8_e2_3d": dict(shares={2: [10, 11], 3: [5, 9, 7]}, cfg=dict(eps_time=2.0, cluster_3d=True, eps_space=30.0), dtype="uint8",
                     window_div=6, cut_inside=True),
    "wf_e5": dict(shares={2: [10, 11], 3: [5, 9, 7]}, cfg=dict(eps_time=5.0, min_frames=3), window_div=3),
    "wf_e2_3d": dict(shares={2: [10, 11], 3: [5, 9, 7]}, cfg=dict(eps_time=2.0, min_frames=2, cluster_3d=True, eps_space=30.0),
                     window_div=5, cut_inside=True),
    "inexact": dict(shares={2: [10, 11], 3: [5, 9, 7]}, cfg=dict(eps_time=2.0), scale=1.37, window_div=4, cut_inside=True),
    "land_6_6": dict(shares={2: [6, 6], 3: [4, 4, 4]}, cfg=dict(eps_time=2.0), frames=12),
    "no_cluster": dict(shares={2: [10, 11], 3: [5, 9, 7]}, cfg=dict(eps_time=2.0), cluster=False),
}
ERRORS = {
    "short_rank": dict(shares={2: [1, 20], 3: [7, 4, 10]}, cfg=dict(eps_time=5.0), match="fewer than"),
    "ids_back": dict(shares={2: [10, 11], 3: [5, 9, 7]}, cfg=dict(eps_time=2.0), ids_back=True, match="increase strictly across ranks"),
}
BRIDGE_SHARES = {2: [4, 9], 3: [4, 4, 5]}


# ------------------------------------------------------------------------------------------------------------- helpers
def _engine_class():
    import torch.distributed as dist

    from radar_point_cloud_tracking_b200.sharded import CudaEngine, TorchEngineBase

    class GlooEngine(CudaEngine):
        """CudaEngine whose collectives run over gloo on host copies (two ranks on one GPU)."""

        def prepare_slots(self, n_slots, slot_ctx):
            pass

        def all_gather(self, mine):
            if self.world == 1:
                return mine[None]
            h = mine.detach().contiguous().cpu()
            parts = [torch.empty_like(h) for _ in range(self.world)]
            dist.all_gather(parts, h, group=self.group)
            return torch.stack(parts).to(self.device)

        def all_reduce_grids(self, count, isum):
            if self.world == 1:
                return count, isum
            c, s = count.cpu(), isum.cpu()
            dist.all_reduce(c, group=self.group)
            dist.all_reduce(s, group=self.group)
            count.copy_(c)
            isum.copy_(s)
            return count, isum

        def exchange(self, to_left, to_right, from_left, from_right):
            if self.world == 1:
                return
            fl = [torch.empty(t.shape, dtype=t.dtype) for t in from_left]
            fr = [torch.empty(t.shape, dtype=t.dtype) for t in from_right]
            TorchEngineBase.exchange(self, [t.cpu() for t in to_left], [t.cpu() for t in to_right], fl, fr)
            for dst, src in list(zip(from_left, fl)) + list(zip(from_right, fr)):
                if dst.numel():
                    dst.copy_(src)

    return GlooEngine


def _ids(n):
    """Frame ids with gaps."""
    return np.cumsum(np.random.default_rng(5).choice([1, 1, 2, 3], n)) + 40


def _config(case, extra=None):
    from radar_point_cloud_tracking_b200.pipeline import DetectionConfig
    return DetectionConfig(**case["cfg"], **(extra or {}))


def _echo(case):
    from radar_point_cloud_tracking_b200 import device as dev
    spec = syn.SweepSpec(**{**SPEC, "frames": case.get("frames", SPEC["frames"])})
    echo = dev.synth_echo(spec, device=torch.device("cuda", 0))
    if "scale" in case:
        echo = echo * case["scale"]                      # non-integer intensities
    if case.get("dtype") == "uint8":
        echo = echo.to(torch.uint8)
    return spec, echo


def _feed(rec, case, spec, echo, a, b, ids):
    """Frames [a, b) fed as blocks of mixed sizes (1, 3, then the rest in two)."""
    G = echo.shape[1]
    c, s, r = (torch.from_numpy(t).to(echo.device) for t in rec.pipe.spoke_tables(spec.angle_units(), spec.scale(), spec.frames, spec.bins))
    cuts = sorted({a, min(a + 1, b), min(a + 4, b), (a + 4 + b) // 2 if b > a + 4 else b, b})
    for x, y in zip(cuts[:-1], cuts[1:]):
        rec.add_block(echo[x:y], c[x * G:y * G], s[x * G:y * G], r[x * G:y * G], ids[x:y])


def _clusters(res):
    return {int(f): [pickle.dumps([(k, vars(cl)[k]) for k in sorted(vars(cl))]) for cl in cls] for f, cls in res.clusters_by_frame().items()}


def _pack(res, clusters=True):
    """Host copies of everything the contract covers."""
    cpu = lambda t: None if t is None else t.cpu().numpy()
    r, p = res.raw, res.points
    return dict(ids=np.asarray(res.frame_ids), raw=[cpu(t[:r.n]) for t in (r.x, r.y, r.inten, r.gain)], raw_off=cpu(r.frame_off),
                pts=[cpu(t[:p.n]) for t in (p.x, p.y, p.inten, p.gain)], pts_off=cpu(p.frame_off), labels=cpu(res.labels),
                core=cpu(res.core), ncl=res.n_clusters, built=res.frames_built, ordered=res.land_ordered, land=cpu(res.land),
                count=cpu(res.count), isum=cpu(res.isum), edges=res.edges, cuts=res.cuts,
                clusters=_clusters(res) if clusters and res.labels.numel() else None, frame_times=res.frame_times)


def _bridge(kind):
    """test_gpu_recording_wf's scene: cluster C's start s, border point b, q = b's only core neighbour."""
    from tests.test_gpu_recording_wf import _start_scene
    return _start_scene(kind)


# ------------------------------------------------------------------------------------------------------------- worker
def _run_case(name, case, world, rank, engine_cls, window_points):
    from radar_point_cloud_tracking_b200.sharded import ShardedRecording
    spec, echo = _echo(case)
    shares = case["shares"][world]
    a = sum(shares[:rank])
    b = a + shares[rank]
    ids = _ids(spec.frames)
    if case.get("ids_back") and rank == world - 1:
        ids = ids - 20                                   # the last rank's ids start below its left neighbour's
    sr = ShardedRecording(_config(case), rank=rank, world=world, engine=engine_cls(0), max_window_points=window_points)
    _feed(sr, case, spec, echo, a, b, ids)
    return _pack(sr.finish(cluster=case.get("cluster", True)))


def _run_bridge(kind, world, rank, engine_cls):
    from radar_point_cloud_tracking_b200 import device as dev
    from radar_point_cloud_tracking_b200.pipeline import DetectionConfig
    from radar_point_cloud_tracking_b200.sharded import ShardedRecording
    xy, off, ids, *_ = _bridge(kind)
    shares = BRIDGE_SHARES[world]
    fa = sum(shares[:rank])
    fb = fa + shares[rank]
    d = torch.device("cuda", 0)
    sr = ShardedRecording(DetectionConfig(eps_space=1.0, eps_time=2.0, min_samples=5, min_frames=2), rank=rank, world=world,
                          engine=engine_cls(0), max_window_points=40)
    p = xy[off[fa]:off[fb]]
    x, y = (torch.from_numpy(np.ascontiguousarray(p[:, k])).to(d) for k in (0, 1))
    inten = torch.zeros(max(len(p), 1), dtype=torch.float32, device=d)
    gain = torch.zeros(max(len(p), 1), dtype=torch.int32, device=d)
    p_off = (off[fa:fb + 1] - off[fa]).astype(np.int64)
    pts = dev.PointBatch(x, y, inten, gain, torch.from_numpy(p_off).to(d), len(p))
    b4 = np.array([xy[:, 0].min(), xy[:, 0].max(), xy[:, 1].min(), xy[:, 1].max()], np.float32)
    labels, core, cuts, ncl = sr._cluster(pts, p_off, ids[fa:fb], 2, b4, {})
    return dict(labels=labels.cpu().numpy(), core=core.cpu().numpy(), ncl=ncl, cuts=cuts)


def _worker(rank, world, port, out_dir, windows, csv_files):
    import torch.distributed as dist
    torch.cuda.set_device(0)
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    engine_cls = _engine_class()
    out = {}
    try:
        for name, case in CASES.items():
            out[name] = _run_case(name, case, world, rank, engine_cls, windows.get(name))
        for name, case in ERRORS.items():
            try:
                _run_case(name, case, world, rank, engine_cls, None)
                out[name] = None
            except RadarB200Error as e:
                out[name] = str(e)
        for kind in ("A", "B"):
            out["bridge_" + kind] = _run_bridge(kind, world, rank, engine_cls)
        out["csv"] = _run_csv(world, rank, engine_cls, csv_files)
    except BaseException:
        out["__error__"] = traceback.format_exc()
    with open(Path(out_dir) / f"rank{rank}.pkl", "wb") as f:
        pickle.dump(out, f)
    dist.destroy_process_group()


def _csv_config():
    from radar_point_cloud_tracking_b200 import tracker as trk
    from radar_point_cloud_tracking_b200.pipeline import DetectionConfig
    c = trk._module_config()
    return DetectionConfig(intensity_threshold=c.INTENSITY_THRESHOLD, point_stride=c.POINT_STRIDE, land_resolution=c.LAND_GRID_RESOLUTION,
                           land_persistence=c.LAND_PERSISTENCE_THRESHOLD, land_min_intensity=c.LAND_MIN_INTENSITY, eps_space=8.0,
                           eps_time=2.0, min_samples=15)


def _run_csv(world, rank, engine_cls, files):
    from radar_point_cloud_tracking_b200.sharded import ShardedRecording, split_frames
    a, b = split_frames(len(files), world, rank)
    sr = ShardedRecording(_csv_config(), rank=rank, world=world, engine=engine_cls(0))
    sr.add_csv_frames(files[a:b], frame_ids=np.arange(a, b))
    return _pack(sr.finish())


# ------------------------------------------------------------------------------------------------------------- fixtures
@pytest.fixture(scope="module")
def gpu():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (no CPU fallback exists)")
    torch.cuda.set_device(0)


@pytest.fixture(scope="module")
def csv_tree(gpu, tmp_path_factory):
    return syn.write_csv_tree(syn.SweepSpec(**CSV_SPEC), tmp_path_factory.mktemp("csv"))


@pytest.fixture(scope="module")
def references(gpu, csv_tree):
    """One-process RecordingDetection of every case (whole recording, same frames, one block), packed."""
    from radar_point_cloud_tracking_b200.recording import RecordingDetection
    out, windows = {}, {}
    for name, case in CASES.items():
        spec, echo = _echo(case)
        ids = _ids(spec.frames)
        rec = RecordingDetection(_config(case), 0)
        _feed(rec, case, spec, echo, 0, spec.frames, ids)
        res = rec.finish(cluster=case.get("cluster", True))
        out[name] = _pack(res)
        if "window_div" in case:
            windows[name] = max(1, res.points.n // case["window_div"])
    rec = RecordingDetection(_csv_config(), 0)
    rec.add_csv_frames(csv_tree)
    out["csv"] = _pack(rec.finish())
    return out, windows


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.fixture(scope="module", params=[2, 3])
def world_run(request, references, csv_tree, tmp_path_factory):
    """All cases in ``world`` spawned processes on GPU 0; their packed results per rank. The processes are joined with a
    timeout and terminated on every exit path."""
    world = request.param
    _, windows = references
    out_dir = tmp_path_factory.mktemp(f"world{world}")
    ctx = mp.get_context("spawn")
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, str(out_dir), windows, csv_tree)) for r in range(world)]
    try:
        for p in procs:
            p.start()
        for p in procs:
            p.join(timeout=900)
        assert all(p.exitcode == 0 for p in procs), [p.exitcode for p in procs]
    finally:
        for p in procs:
            if p.is_alive():
                p.terminate()
                p.join(timeout=30)
    got = []
    for r in range(world):
        with open(out_dir / f"rank{r}.pkl", "rb") as f:
            res = pickle.load(f)
        assert "__error__" not in res, res.get("__error__")
        got.append(res)
    return world, got


# ------------------------------------------------------------------------------------------------------------- checks
def _cat_off(offs):
    out, base = [np.zeros(1, np.int64)], 0
    for o in offs:
        out.append(o[1:] + base)
        base += int(o[-1])
    return np.concatenate(out)


def _assert_equal(parts, want):
    """The ranks' results in rank order = the one-process result."""
    assert np.array_equal(np.concatenate([p["ids"] for p in parts]), want["ids"])
    for key in ("raw", "pts"):
        for k in range(4):
            assert np.array_equal(np.concatenate([p[key][k] for p in parts]), want[key][k]), key
    assert np.array_equal(_cat_off([p["raw_off"] for p in parts]), want["raw_off"])
    assert np.array_equal(_cat_off([p["pts_off"] for p in parts]), want["pts_off"])
    for p in parts:
        assert p["built"] == want["built"] and p["ordered"] == want["ordered"] and p["ncl"] == want["ncl"]
        for k in ("land", "count", "isum"):
            assert (p[k] is None) == (want[k] is None), k
            if want[k] is not None:
                assert p[k].tobytes() == want[k].tobytes(), k                  # bit for bit (float64 sums included)
        if want["edges"] is not None:
            assert all(np.array_equal(a, b) for a, b in zip(p["edges"], want["edges"]))
    labels = np.concatenate([p["labels"] for p in parts])
    assert np.array_equal(labels, want["labels"])
    if want["core"] is not None:
        assert np.array_equal(np.concatenate([p["core"] for p in parts if p["core"] is not None]), want["core"])
    if want["clusters"] is not None:
        merged = {}
        for p in parts:
            for f, cls in (p["clusters"] or {}).items():
                assert f not in merged
                merged[f] = cls
        assert merged == want["clusters"]


@pytest.mark.parametrize("name", list(CASES))
def test_sharded_recording_equals_one_process(world_run, references, name):
    world, got = world_run
    want = references[0][name]
    parts = [g[name] for g in got]
    _assert_equal(parts, want)
    case = CASES[name]
    if case.get("cluster", True) and not case["cfg"].get("cluster_3d"):
        assert want["ncl"] > 0
    if case.get("cut_inside"):
        assert any(len(p["cuts"]) > 2 for p in parts)                              # windows cut inside a rank too
    if name == "inexact":
        assert want["ordered"] and all(p["ordered"] for p in parts)
    if name == "land_6_6":
        assert want["land"] is not None and all(p["built"] == 12 for p in parts)
        assert all(len(p["ids"]) <= 6 for p in parts)                              # no rank alone exceeds land_min_frames
    if name == "no_cluster":
        assert all(p["labels"].size == 0 for p in parts)


def test_clusters_span_ranks(world_run, references):
    """Some cluster id occurs on both sides of a rank boundary: its cores and borders lie on neighbouring ranks."""
    world, got = world_run
    for name in ("f32_e2_windows", "wf_e5"):
        sides = [set(np.unique(g[name]["labels"])) - {-1} for g in got]
        assert any(sides[r] & sides[r + 1] for r in range(world - 1)), name


def test_csv_tree_over_ranks(world_run, references, csv_tree):
    from radar_point_cloud_tracking_b200 import tracker as trk
    world, got = world_run
    want = references[0]["csv"]
    parts = [g["csv"] for g in got]
    _assert_equal(parts, want)
    assert sum((p["frame_times"] for p in parts), []) == want["frame_times"]
    cfg = _csv_config()
    ref = trk.detect_csv_frames(csv_tree, False, cfg.eps_space, cfg.eps_time, cfg.min_samples)
    flat = {int(f): [pickle.dumps([(k, vars(cl)[k]) for k in sorted(vars(cl))]) for cl in cls] for f, cls in ref.items()}
    merged = {}
    for p in parts:
        merged.update(p["clusters"] or {})
    assert merged == flat


@pytest.mark.parametrize("kind", ["A", "B"])
def test_min_frames_cluster_start_on_an_earlier_rank(world_run, kind):
    from oracle.c_oracle import st_dbscan_wf_c
    world, got = world_run
    xy, off, ids, b, s, q = _bridge(kind)
    t = np.repeat(ids.astype(np.float32), np.diff(off))
    want, want_core = st_dbscan_wf_c(xy, t, 1.0, 2.0, 5, 2)
    parts = [g["bridge_" + kind] for g in got]
    labels = np.concatenate([p["labels"] for p in parts])
    assert np.array_equal(labels, want)
    assert np.array_equal(np.concatenate([p["core"] for p in parts]), want_core.astype(np.uint8))
    assert all(p["ncl"] == 2 for p in parts)
    bounds = np.cumsum([0] + BRIDGE_SHARES[world])
    rank_of = lambda i: int(np.searchsorted(off[bounds], i, side="right")) - 1
    if kind == "A":
        assert rank_of(s) < rank_of(b)                                  # the cluster starts on an earlier rank
    assert labels[b] == (1 if kind == "A" else -1)
    assert any(len(p["cuts"]) > 2 for p in parts)


@pytest.mark.parametrize("name", list(ERRORS))
def test_every_rank_raises_the_same_error(world_run, name):
    world, got = world_run
    msgs = [g[name] for g in got]
    assert msgs[0] is not None and ERRORS[name]["match"] in msgs[0], msgs
    assert all(m == msgs[0] for m in msgs)


def test_world_one_is_recording_detection(gpu, references):
    from radar_point_cloud_tracking_b200.sharded import ShardedRecording
    name = "wf_e5"
    case = CASES[name]
    spec, echo = _echo(case)
    sr = ShardedRecording(_config(case), rank=0, world=1, engine=_engine_class()(0))
    _feed(sr, case, spec, echo, 0, spec.frames, _ids(spec.frames))
    _assert_equal([_pack(sr.finish())], references[0][name])


@pytest.mark.parametrize("eps_time,min_frames", [("2.0", "0"), ("5.0", "3")])
def test_sharded_recording_nccl_equals_one_gpu(eps_time, min_frames):
    """NCCL, the product engine, full-size frames (needs >= 2 GPUs in the box; skipped otherwise)."""
    import subprocess
    import sys
    n = torch.cuda.device_count() if torch.cuda.is_available() else 0
    if n < 2:
        pytest.skip("needs at least 2 GPUs")
    repo = Path(__file__).resolve().parent.parent
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={min(8, n)}", "--master-addr", "127.0.0.1",
           "--master-port", "29543", str(repo / "tools" / "check_sharded_recording.py"), "8", eps_time, min_frames]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=repo)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]
    assert "IDENTICAL to one GPU" in res.stdout
