"""PLY writers and colour helpers (SURVEY section 8 f, rank 4) against files written by the unmodified reference
(``tests/golden/make_golden_ply.py``): the bytes on disk must be identical. CPU only - the writers are host code
(``rb_ply_append_ascii`` is a host function of the library)."""
import io
import contextlib
from pathlib import Path

import numpy as np
import pytest

from radar_point_cloud_tracking_b200 import plyio

GOLD = np.load(Path(__file__).parent / "golden" / "ply_golden.npz")


def _quiet(fn, *a):
    with contextlib.redirect_stdout(io.StringIO()) as out:
        fn(*a)
    return out.getvalue()


@pytest.mark.parametrize("case", range(int(GOLD["n_cases"])))
def test_writers_and_colours_match_the_reference(tmp_path, case):
    g = lambda k: GOLD[f"c{case}_{k}"]
    x, y, z = g("x"), g("y"), g("z")
    norm = plyio.normalize_intensity(g("inten"))
    assert norm.dtype == g("norm").dtype and np.array_equal(norm, g("norm"))
    rgb_i = plyio.intensity_to_rgb(norm) if len(x) else np.zeros((0, 3), np.uint8)
    rgb_g = plyio.gain_to_rgb(g("gains"))
    assert np.array_equal(rgb_i, g("rgb_i")) and np.array_equal(rgb_g, g("rgb_g"))
    fast, slow = tmp_path / f"fast{case}.ply", tmp_path / f"slow{case}.ply"
    msg = _quiet(plyio.write_ply_fast, fast, x, y, z, rgb_i)
    _quiet(plyio.write_ply, slow, x, y, z, rgb_g)
    assert msg == f"  Wrote {len(x):,} points to {fast.name}\n"
    assert fast.read_bytes() == g("fast").tobytes()
    assert slow.read_bytes() == g("slow").tobytes()


def test_float64_coordinates_keep_each_writer_s_own_rounding(tmp_path):
    a, b = tmp_path / "f64_slow.ply", tmp_path / "f64_fast.ply"
    _quiet(plyio.write_ply, a, GOLD["d_x"], GOLD["d_y"], GOLD["d_z"], GOLD["d_col"])
    _quiet(plyio.write_ply_fast, b, GOLD["d_x"], GOLD["d_y"], GOLD["d_z"], GOLD["d_col"])
    assert a.read_bytes() == GOLD["d_slow"].tobytes() and b.read_bytes() == GOLD["d_fast"].tobytes()
    assert GOLD["d_slow"].tobytes() != GOLD["d_fast"].tobytes()        # the case does tell the two apart


def test_native_formatter_equals_printf_on_random_and_awkward_floats(tmp_path):
    rng = np.random.default_rng(9)
    bits = rng.integers(0, 2 ** 32, 200_000, dtype=np.uint64).astype(np.uint32)
    v = bits.view(np.float32)                                          # every exponent, NaNs and infinities included
    v = np.concatenate([v, np.array([0.0, -0.0, np.inf, -np.inf, np.nan, 1e14, -1e14, 9.9999e13, 2 ** -149, 0.00005, 0.00015], np.float32)])
    rgb = rng.integers(0, 256, (len(v), 3)).astype(np.uint8)
    p = tmp_path / "awkward.ply"
    _quiet(plyio.write_ply_fast, p, v, v[::-1].copy(), v, rgb)
    body = p.read_bytes().split(b"end_header\n", 1)[1].decode().split("\n")
    assert body[-1] == "" and len(body) == len(v) + 1
    w = v[::-1]
    for i in rng.integers(0, len(v), 4000).tolist() + list(range(len(v) - 11, len(v))):
        assert body[i] == "%.4f %.4f %.4f %d %d %d" % (float(v[i]), float(w[i]), float(v[i]), rgb[i, 0], rgb[i, 1], rgb[i, 2]), i


def test_binary_ply_records(tmp_path):
    """WF:797-827: header + 15-byte little-endian records."""
    rng = np.random.default_rng(4)
    n = 257
    x, y, z = (rng.normal(0, 100, n) for _ in range(3))                # float64 in, float32 on disk
    col = rng.integers(0, 256, (n, 3)).astype(np.uint8)
    p = tmp_path / "b.ply"
    plyio.write_ply_binary(p, x, y, z, col)
    raw = p.read_bytes()
    head, body = raw.split(b"end_header\n", 1)
    assert head.decode().split("\n")[:3] == ["ply", "format binary_little_endian 1.0", f"element vertex {n}"]
    rec = np.frombuffer(body, dtype=np.dtype([("x", "<f4"), ("y", "<f4"), ("z", "<f4"), ("r", "u1"), ("g", "u1"), ("b", "u1")]))
    assert len(body) == 15 * n and np.array_equal(rec["x"], x.astype(np.float32)) and np.array_equal(rec["b"], col[:, 2])
