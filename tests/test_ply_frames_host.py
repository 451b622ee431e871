"""CPU-side checks of the device PLY writer: the new C entries in the header and the bindings, argument validation before
any device work or file creation, and the chunk planning of plyio.write_ply_frames."""
import re
from pathlib import Path

import numpy as np
import pytest
import torch

from radar_point_cloud_tracking_b200 import _lib, fusion, plyio
from radar_point_cloud_tracking_b200._lib import RadarB200Error

REPO = Path(__file__).resolve().parent.parent
NAMES = ["rb_ply_format_ascii", "rb_ply_pack_binary", "rb_ply_colors_intensity", "rb_ply_colors_gain"]


@pytest.mark.parametrize("name", NAMES)
def test_symbol_in_header_and_bindings(name):
    header = (REPO / "include" / "radarb200.h").read_text()
    assert re.search(rf"\b{name}\s*\(", header)
    assert name in _lib.SIGNATURES
    assert hasattr(_lib.load(), name)


def _args(n=4):
    x = torch.zeros(n, dtype=torch.float32)
    return x, x, x, torch.zeros((n, 3), dtype=torch.uint8), torch.tensor([0, n], dtype=torch.int64)


@pytest.mark.parametrize("bad", ["x", "colors", "frame_off", "numpy"])
def test_host_tensors_are_rejected_before_any_file_exists(tmp_path, bad):
    x, y, z, c, off = _args()
    args = {"x": x, "y": y, "z": z, "colors": c, "frame_off": off}
    if bad == "numpy":
        args["x"] = np.zeros(4, np.float32)
    path = tmp_path / "f.ply"
    with pytest.raises(RadarB200Error, match="CUDA tensor"):
        plyio.write_ply_frames([path], **args)
    assert not path.exists() and not list(tmp_path.iterdir())


def test_colours_reject_host_tensors():
    with pytest.raises(RadarB200Error, match="CUDA tensor"):
        plyio.intensity_rgb(torch.zeros(3))
    with pytest.raises(RadarB200Error, match="CUDA tensor"):
        plyio.gain_rgb(torch.zeros(3, dtype=torch.int32))


def test_fuse_csv_frames_checks_the_ply_paths_first(tmp_path):
    with pytest.raises(RadarB200Error, match="PLY paths"):
        fusion.fuse_csv_frames_max([{40: REPO / "no_such_file.csv"}] * 2, 1.0, ply_paths=[tmp_path / "a.ply"])
    assert not list(tmp_path.iterdir())


def _check_plan(off, L):
    chunks = plyio.plan_chunks(np.asarray(off, np.int64), L)
    assert chunks[0][0] == off[0] and chunks[-1][1] == off[-1]
    covered = {}
    last_chunk = []
    for k, (v0, v1, pieces) in enumerate(chunks):
        assert 0 <= v1 - v0 <= L
        if k:
            assert v0 == chunks[k - 1][1]
        assert [p[0] for p in pieces] == sorted(p[0] for p in pieces)
        at = v0
        for f, a, b in pieces:
            assert off[f] <= a <= b <= off[f + 1] and v0 <= a and b <= v1
            if a < b:
                assert a == at                                   # the chunk's lines, in order, no gap
                at = b
            covered.setdefault(f, []).append((a, b))
        assert at == v1 or v1 == v0
    for f in range(len(off) - 1):
        spans = covered[f]
        if off[f] == off[f + 1]:
            assert spans == [(off[f], off[f])]
        else:
            assert spans[0][0] == off[f] and spans[-1][1] == off[f + 1]
            assert all(spans[i][1] == spans[i + 1][0] for i in range(len(spans) - 1))
        last_chunk.append(max(k for k, (_, _, ps) in enumerate(chunks) for p in ps if p[0] == f))
    assert last_chunk == sorted(last_chunk)                      # files complete, and are announced, in frame order
    return chunks


def test_plan_packs_frames_and_splits_at_lines():
    off = [0, 3, 3, 10, 11, 11, 25, 25]
    chunks = _check_plan(off, 4)
    assert [(v0, v1) for v0, v1, _ in chunks] == [(0, 4), (4, 8), (8, 12), (12, 16), (16, 20), (20, 24), (24, 25)]
    assert chunks[0][2] == [(0, 0, 3), (1, 3, 3), (2, 3, 4)]
    assert chunks[-1][2] == [(5, 24, 25), (6, 25, 25)]
    assert plyio.plan_chunks(np.array([0, 5], np.int64), 100)[0][2] == [(0, 0, 5)]


def test_plan_random_offsets():
    rng = np.random.default_rng(5)
    for _ in range(200):
        counts = rng.integers(0, 40, rng.integers(1, 30)) * (rng.random(1) < 0.9)
        off = np.concatenate([[0], np.cumsum(counts)]) + rng.integers(0, 5)
        _check_plan(off.tolist(), int(rng.integers(1, 60)))


def test_plan_without_vertices_is_one_chunk():
    chunks = plyio.plan_chunks(np.array([7, 7, 7], np.int64), 10)
    assert chunks == [(7, 7, [(0, 7, 7), (1, 7, 7)])]
    with pytest.raises(RadarB200Error):
        plyio.plan_chunks(np.array([0, 1], np.int64), 0)
