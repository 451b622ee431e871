"""PLY files of whole recordings written from the device (plyio.write_ply_frames, intensity_rgb, gain_rgb and
fuse_csv_frames_max(..., ply_paths=...)) against the host writers and colour helpers, byte for byte."""
import contextlib
import io
from pathlib import Path
from types import SimpleNamespace

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from radar_point_cloud_tracking_b200 import plyio
from radar_point_cloud_tracking_b200 import synthetic as syn
from radar_point_cloud_tracking_b200._lib import RadarB200Error

pytestmark = pytest.mark.gpu

GOLD = np.load(Path(__file__).parent / "golden" / "ply_golden.npz")
F32 = np.float32
FMAX = np.finfo(F32).max


@pytest.fixture(scope="module")
def gpu():
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device (no CPU fallback exists)")
    torch.cuda.set_device(0)
    return torch.device("cuda", 0)


def _quiet(fn, *a, **k):
    with contextlib.redirect_stdout(io.StringIO()) as out:
        fn(*a, **k)
    return out.getvalue()


def _awkward():
    """Values whose "%.4f" is easy to get wrong."""
    rng = np.random.default_rng(3)
    ties = np.array([k / 2.0 ** m for m in range(5, 15) for k in rng.integers(1, 2 ** 12, 20)], F32)   # v * 1e4 = j + 1/2
    ties = ties[(ties.astype(np.float64) * 1e4) % 1 == 0.5]
    near = np.concatenate([np.nextafter(ties, F32(np.inf)), np.nextafter(ties, F32(-np.inf))])
    big = np.array([2 ** 24, 2 ** 24 + 2, 1e14, 9.9999e13, 2 ** 100, FMAX, 3e38, 1.5e15, 2 ** 127, 123456789012345678901234567890.0], F32)
    with np.errstate(over="ignore"):
        big = np.concatenate([big, np.nextafter(big, F32(0)), np.nextafter(big, F32(np.inf))])
    small = np.array([0.0, -0.0, -1e-5, -4.9e-5, -5e-5, 5e-5, 1.5e-4, 2 ** -149, -(2 ** -149), 1e-40, 1.17e-38, 0.00005, 0.99995,
                      -0.99995, 9.99995, np.inf, -np.inf, np.nan, -np.nan, 1.0, -1.0, 255.0], F32)
    return np.concatenate([ties, -ties, near, -near, big, -big, small])


def _frames(seed=1, n_frames=40, dtype=F32):
    """Frame sizes including empty, one-vertex and large frames; coordinates mixing plain and awkward values."""
    rng = np.random.default_rng(seed)
    aw = _awkward()
    sizes = [int(np.exp(rng.uniform(0, np.log(60_000)))) for _ in range(n_frames)]
    sizes[0], sizes[3], sizes[5], sizes[-1], sizes[7] = 0, 1, 0, 0, 250_000
    n = sum(sizes)
    cols = []
    for k in range(3):
        v = rng.normal(0, 10 ** rng.uniform(-2, 4, n), n).astype(dtype)
        pick = rng.random(n) < 0.05
        v[pick] = rng.choice(aw, int(pick.sum())).astype(dtype)
        cols.append(v)
    rgb = rng.integers(0, 256, (n, 3)).astype(np.uint8)
    rgb[:256, 0] = np.arange(256)                                   # all 256 colour values in every channel
    rgb[256:512, 1] = np.arange(256)
    rgb[512:768, 2] = np.arange(256)
    off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    return cols, rgb, off


def _to_dev(d, *arrs):
    return [torch.from_numpy(np.ascontiguousarray(a)).to(d) for a in arrs]


def _compare(tmp_path, d, cols, rgb, off, binary=False, chunk_bytes=plyio.DEFAULT_CHUNK_BYTES):
    F = len(off) - 1
    got_dir, want_dir = tmp_path / "got", tmp_path / "want"
    got_dir.mkdir(parents=True), want_dir.mkdir(parents=True)
    names = [f"frame_{f:04d}.ply" for f in range(F)]
    x, y, z, c, fo = _to_dev(d, *cols, rgb, off)
    printed = _quiet(plyio.write_ply_frames, [got_dir / s for s in names], x, y, z, c, fo, binary=binary, chunk_bytes=chunk_bytes)
    ref = plyio.write_ply_binary if binary else plyio.write_ply_fast
    want_printed = "".join(_quiet(ref, want_dir / names[f], *(v[off[f]:off[f + 1]] for v in cols), rgb[off[f]:off[f + 1]])
                           for f in range(F))
    assert printed == want_printed
    for s in names:
        assert (got_dir / s).read_bytes() == (want_dir / s).read_bytes(), s
    return got_dir


def test_many_frames_equal_write_ply_fast(gpu, tmp_path):
    cols, rgb, off = _frames()
    _compare(tmp_path, gpu, cols, rgb, off)


def test_many_frames_equal_write_ply_binary(gpu, tmp_path):
    cols, rgb, off = _frames(seed=2)
    _compare(tmp_path, gpu, cols, rgb, off, binary=True)


@pytest.mark.filterwarnings("ignore:overflow encountered in cast")
def test_float64_coordinates_are_cast_to_float32_first(gpu, tmp_path):
    cols, rgb, off = _frames(seed=4, n_frames=9, dtype=np.float64)
    cols[0][:1000] = 0.1 + np.arange(1000) * 1e-9                   # values that change when cast
    cols[1][:5] = [1e300, -1e300, 3.5e38, 1e-50, -1e-50]            # overflow to inf, underflow to 0 in float32
    assert np.any(cols[0].astype(F32).astype(np.float64) != cols[0])
    _compare(tmp_path, gpu, cols, rgb, off)
    _compare(tmp_path / "b", gpu, cols, rgb, off, binary=True)


def test_random_bit_patterns(gpu, tmp_path):
    rng = np.random.default_rng(9)
    v = rng.integers(0, 2 ** 32, 400_000, dtype=np.uint64).astype(np.uint32).view(F32)   # every exponent, NaNs, infinities
    w = v[::-1].copy()
    rgb = rng.integers(0, 256, (len(v), 3)).astype(np.uint8)
    off = np.array([0, 1, 150_000, 150_000, 400_000], np.int64)
    got = _compare(tmp_path, gpu, [v, w, v], rgb, off)
    body = b"".join((got / f"frame_{f:04d}.ply").read_bytes().split(b"end_header\n", 1)[1] for f in range(4)).decode().split("\n")
    for i in rng.integers(0, len(v), 3000).tolist():
        assert body[i] == "%.4f %.4f %.4f %d %d %d" % (float(v[i]), float(w[i]), float(v[i]), *rgb[i]), i


@pytest.mark.parametrize("binary", [False, True])
def test_tiny_chunks_split_frames(gpu, tmp_path, binary):
    cols, rgb, off = _frames(seed=5, n_frames=12)
    unit = plyio.PLY_RECORD_BYTES if binary else plyio.PLY_LINE_MAX
    _compare(tmp_path, gpu, cols, rgb, off, binary=binary, chunk_bytes=unit * 997 + 3)
    cut = [0, 1, 2, 3, 10, 10, 11, 40]
    _compare(tmp_path / "t", gpu, [c[:40] for c in cols], rgb[:40], np.array(cut, np.int64), binary=binary,
             chunk_bytes=unit * 3)


def _golden_cases():
    cases = range(int(GOLD["n_cases"]))
    g = lambda c, k: GOLD[f"c{c}_{k}"]
    off = np.concatenate([[0], np.cumsum([len(g(c, "x")) for c in cases])]).astype(np.int64)
    cat = lambda k: np.concatenate([g(c, k) for c in cases])
    return cases, g, off, cat


def test_golden_cases_in_one_batch(gpu, tmp_path):
    cases, g, off, cat = _golden_cases()
    x, y, z, inten, gains, fo = _to_dev(gpu, cat("x"), cat("y"), cat("z"), cat("inten"), cat("gains"), off)
    rgb_i = plyio.intensity_rgb(inten, fo, normalize=True)
    assert rgb_i.is_cuda and rgb_i.dtype == torch.uint8 and tuple(rgb_i.shape) == (len(inten), 3)
    assert np.array_equal(rgb_i.cpu().numpy(), cat("rgb_i"))
    assert np.array_equal(plyio.gain_rgb(gains).cpu().numpy(), cat("rgb_g"))
    paths = [tmp_path / f"fast{c}.ply" for c in cases]
    printed = _quiet(plyio.write_ply_frames, paths, x, y, z, rgb_i, fo)
    assert printed == "".join(f"  Wrote {len(g(c, 'x')):,} points to fast{c}.ply\n" for c in cases)
    for c in cases:
        assert paths[c].read_bytes() == g(c, "fast").tobytes()


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_intensity_colours_at_the_quarter_boundaries(gpu, dtype):
    q = np.array([0.0, 63.75, 127.5, 191.25, 255.0, 1.0, 254.0, 100.0, 200.0], dtype)
    v = np.concatenate([q, np.nextafter(q, dtype(0)), np.nextafter(q, dtype(255)),
                        np.random.default_rng(1).uniform(0, 255, 100_000).astype(dtype), np.arange(256, dtype=dtype)])
    (dv,) = _to_dev(gpu, v)
    assert np.array_equal(plyio.intensity_rgb(dv).cpu().numpy(), plyio.intensity_to_rgb(v))


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_normalisation_per_frame(gpu, dtype):
    rng = np.random.default_rng(8)
    frames = [np.array([5.0]), np.array([3.0, 9.0]), np.array([9.0, 3.0]), rng.normal(50, 30, 100), np.full(100, 7.0),
              np.concatenate([np.full(99, 4.0), [10.0]]), np.concatenate([[0.0], np.full(99, 4.0)]),   # ties at the percentile
              np.concatenate([np.full(98, 1.0), [2.0, 2.0]]), np.array([]), rng.integers(0, 256, 3000).astype(float),
              rng.uniform(-1e6, 1e6, 5000), np.concatenate([rng.normal(0, 1, 200_000), [1e30, -1e30]]),
              np.array([-0.0, 0.0, 0.0]), rng.normal(0, 1e-30, 77)]
    frames = [f.astype(dtype) for f in frames]
    off = np.concatenate([[0], np.cumsum([len(f) for f in frames])]).astype(np.int64)
    v, fo = _to_dev(gpu, np.concatenate(frames), off)
    got = plyio.intensity_rgb(v, fo, normalize=True).cpu().numpy()
    for f, fr in enumerate(frames):
        want = plyio.intensity_to_rgb(plyio.normalize_intensity(fr)) if len(fr) else np.zeros((0, 3), np.uint8)
        assert np.array_equal(got[off[f]:off[f + 1]], want), f


@pytest.mark.parametrize("vals,normalize", [([0.0, 255.5], False), ([-1e-7, 3.0], False), ([np.nan, 1.0], False),
                                            ([np.inf], False), ([1.0, np.nan, 2.0], True), ([0.0, 1.0, np.inf], True)])
def test_colour_domain_errors_raise(gpu, vals, normalize):
    for dtype in (np.float32, np.float64):
        (v,) = _to_dev(gpu, np.array(vals, dtype))
        with pytest.raises(RadarB200Error, match="NaN or outside"):
            plyio.intensity_rgb(v, normalize=normalize)


def _rewrite(src, dst, fn):
    dst.write_text("\n".join(fn(src.read_text().split("\n"))))
    return dst


def test_fuse_csv_frames_with_ply_paths(gpu, tmp_path, capsys):
    from radar_point_cloud_tracking_b200 import fusion
    E = 256
    a = syn.write_csv_tree(syn.SweepSpec(seed=51, frames=10, spokes=64, bins=E, clutter_p=0.02, land_blobs=2, buoys=3, boats=2), tmp_path / "a")
    b = syn.write_csv_tree(syn.SweepSpec(seed=52, frames=10, spokes=48, bins=E, clutter_p=0.02, land_blobs=2, buoys=3, boats=2), tmp_path / "b")
    odd = tmp_path / "odd"
    odd.mkdir()
    empty, header_only = odd / "20250813_150000_000.csv", odd / "20250813_150000_100.csv"
    empty.write_text("")
    header_only.write_text(a[0][40].read_text().split("\n")[0] + "\n")

    def dec_echo(rows):
        r = rows[7].split(",")
        r[29:37] = ["212.5"] * 8
        return rows[:7] + [",".join(r)] + rows[8:]

    frames = []
    for f in range(10):
        fa, fb = a[f], b[f]
        if f == 1:
            frames.append({40: fa[40], 75: fb[75]})
        elif f == 2:
            frames.append({40: empty, 50: header_only})
        elif f == 3:
            frames.append({40: odd / "20250813_150100_000.csv", 50: fa[50], 75: fa[75]})
        elif f == 4:
            frames.append({50: _rewrite(fa[50], odd / "20250813_150200_000.csv", dec_echo), 75: fb[75]})
        elif f == 5:
            frames.append({})
        else:
            frames.append(dict(fa) if f % 2 else dict(fb))
    t5 = SimpleNamespace(NUM_ECHO_COLUMNS=E, INTENSITY_THRESHOLD=5.0, POINT_STRIDE=8)
    fusion.install(t5)
    cfg = fusion._config(t5)
    sizes = sum(p.stat().st_size for fr in frames for p in fr.values() if p.exists())
    plain = fusion.fuse_csv_frames_max(frames, 1.0, batch_bytes=max(4096, sizes // 4), readers=3, _cfg=cfg)
    out = tmp_path / "ply"
    out.mkdir()
    paths = [out / f"frame_{f:03d}.ply" for f in range(len(frames))]
    capsys.readouterr()
    timings = {}
    got = fusion.fuse_csv_frames_max(frames, 1.0, batch_bytes=max(4096, sizes // 4), readers=3, _cfg=cfg, timings=timings,
                                     ply_paths=paths)
    printed = [ln for ln in capsys.readouterr().out.split("\n") if ln.startswith("  Wrote")]
    assert timings["ply"] > 0 and len(got) == len(plain)
    for g, p in zip(got, plain):
        assert all(u.dtype == w.dtype and np.array_equal(u, w) for u, w in zip(g, p))
    want_dir = tmp_path / "want"
    want_dir.mkdir()
    want_printed = []
    for f, ff in enumerate(frames):
        x, y, m = t5.fuse_gains_max(ff, 1.0)
        want_printed += _quiet(plyio.write_ply_fast, want_dir / paths[f].name, x, y, m, plyio.intensity_to_rgb(m)).rstrip("\n").split("\n")
        assert paths[f].read_bytes() == (want_dir / paths[f].name).read_bytes(), f
    assert printed == want_printed


def test_launches_do_not_depend_on_the_number_of_frames(gpu, tmp_path):
    from radar_point_cloud_tracking_b200._lib import context
    ctx = context(0)
    rng = np.random.default_rng(6)
    n = 64 * 3000
    x, y, z = _to_dev(gpu, *(rng.normal(0, 100, n).astype(F32) for _ in range(3)))
    inten, c = _to_dev(gpu, rng.uniform(0, 200, n).astype(F32), rng.integers(0, 256, (n, 3)).astype(np.uint8))
    counts = []
    for F in (1, 64):
        fo = torch.from_numpy(np.linspace(0, n, F + 1).astype(np.int64)).to(gpu)
        d = tmp_path / f"f{F}"
        d.mkdir()
        for binary in (False, True):
            before = ctx.launch_count()
            rgb = plyio.intensity_rgb(inten, fo, normalize=True)
            _quiet(plyio.write_ply_frames, [d / f"{k}.ply" for k in range(F)], x, y, z, rgb, fo, binary=binary, chunk_bytes=4 << 20)
            counts.append(ctx.launch_count() - before)
    assert counts[:2] == counts[2:] and counts[0] > 0


def test_bad_arguments_raise_before_any_file(gpu, tmp_path):
    n = 10
    x, y, z, c, fo = _to_dev(gpu, np.zeros(n, F32), np.zeros(n, F32), np.zeros(n, F32), np.zeros((n, 3), np.uint8),
                             np.array([0, 4, n], np.int64))
    p = [tmp_path / "a.ply", tmp_path / "b.ply"]
    bad = [
        dict(paths=p[:1]),                                                        # one path for two frames
        dict(frame_off=torch.tensor([0, 5, 4], dtype=torch.int64, device=gpu)),  # decreasing
        dict(frame_off=torch.tensor([0, 4, n + 1], dtype=torch.int64, device=gpu)),   # beyond the vertices
        dict(frame_off=torch.tensor([-1, 4, n], dtype=torch.int64, device=gpu)),
        dict(frame_off=torch.tensor([0, 4, n], dtype=torch.int32, device=gpu)),
        dict(colors=c[:, :2].contiguous()),
        dict(colors=c.to(torch.int32)),
        dict(x=x.to(torch.int32)),
        dict(y=y.reshape(2, 5)),
        dict(chunk_bytes=100),
        dict(chunk_bytes=14, binary=True),
    ]
    for change in bad:
        args = dict(paths=p, x=x, y=y, z=z, colors=c, frame_off=fo)
        args.update(change)
        with pytest.raises(RadarB200Error):
            plyio.write_ply_frames(**args)
        assert not list(tmp_path.iterdir()), change
    with pytest.raises(RadarB200Error):
        plyio.intensity_rgb(torch.zeros(3, dtype=torch.int32, device=gpu))
    with pytest.raises(RadarB200Error):
        plyio.intensity_rgb(torch.zeros(3, device=gpu), torch.tensor([0, 4], dtype=torch.int64, device=gpu))
    with pytest.raises(RadarB200Error):
        plyio.gain_rgb(torch.zeros(3, dtype=torch.int64, device=gpu))


def test_unwritable_path_names_the_file(gpu, tmp_path):
    n = 6
    x, c, fo = _to_dev(gpu, np.arange(n, dtype=F32), np.zeros((n, 3), np.uint8), np.array([0, 2, 4, n], np.int64))
    paths = [tmp_path / "ok0.ply", tmp_path / "missing_dir" / "f1.ply", tmp_path / "ok2.ply"]
    with pytest.raises(RadarB200Error, match="f1.ply"):
        _quiet(plyio.write_ply_frames, paths, x, x, x, c, fo)
