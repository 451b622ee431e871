"""Host-side pieces of the CSV recording path (csvbatch): batch packing, spoke runs, frame offsets, and the leading-field
rule of rb_csv_parse_sweeps stated in Python against pandas' C parser."""
import io

import numpy as np
import pytest
import torch

from radar_point_cloud_tracking_b200 import csvbatch as cb
from radar_point_cloud_tracking_b200 import device as dev
from radar_point_cloud_tracking_b200._lib import RadarB200Error

K = cb.CSV_CHUNK


def test_frame_offsets_from_sweep_bases():
    sweep_off = np.array([0, 5, 5, 12, 20, 20, 31], np.int64)          # 6 sweeps
    got = cb.frame_offsets(sweep_off, [3, 0, 1, 2, 0])
    assert got.tolist() == [0, 12, 12, 20, 31, 31]
    assert cb.frame_offsets(np.zeros(1, np.int64), [0, 0]).tolist() == [0, 0, 0]
    with pytest.raises(ValueError):
        cb.frame_offsets(sweep_off, [3, 1])


def test_sweep_runs():
    keys = [(64, "u8"), (64, "u8"), (48, "u8"), (48, "f32"), (48, "f32"), (64, "u8")]
    assert cb.sweep_runs(keys) == [(0, 2), (2, 3), (3, 5), (5, 6)]
    assert cb.sweep_runs([]) == []
    assert cb.sweep_runs([1]) == [(0, 1)]


def test_pack_batches_aligned_whole_frames_under_the_cap():
    sizes = [[100, 5000, 4096], [None, 10], [9000], [3 * K, 3 * K], [0]]
    batches, offs = cb.pack_batches(sizes, 5 * K)
    # frame 0: 1 + 2 + 1 chunks = 4; frame 1: 1 chunk (the unreadable file takes the per-file path) -> 5 chunks
    assert offs[0] == [0, K, 3 * K] and offs[1] == [-1, 4 * K]
    # frame 2 (3 chunks) starts a new batch; frame 3 (6 chunks) does not fit with it, and alone only its first file fits
    assert offs[2] == [0] and offs[3] == [0, -1] and offs[4] == [3 * K]
    assert batches == [(0, 2, 5 * K), (2, 3, 3 * K), (3, 5, 3 * K)]
    for fa, fb, nbytes in batches:
        assert nbytes <= 5 * K
        for f in range(fa, fb):
            for o, s in zip(offs[f], sizes[f]):
                assert o == -1 or (o % K == 0 and o + s <= nbytes)
    # the cap never reaches 2^31 bytes
    b, o = cb.pack_batches([[1 << 30], [1 << 30]], 1 << 40)
    assert b == [(0, 1, 1 << 30), (1, 2, 1 << 30)]


def _tokens(rng, n):
    out = []
    for _ in range(n):
        nd = int(rng.integers(1, 16))
        digits = "".join(str(int(v)) for v in rng.integers(0, 10, nd))
        k = int(rng.integers(0, nd)) if rng.random() < 0.6 else 0      # fraction digits (at least one integer digit)
        tok = digits if k == 0 else digits[:nd - k] + "." + digits[nd - k:]
        if rng.random() < 0.4:
            tok = "-" + tok
        out.append(tok)
    return out


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_lead_field_rule_matches_pandas(seed):
    pd = pytest.importorskip("pandas")
    rng = np.random.default_rng(seed)
    toks = _tokens(rng, 4000)
    mixed = pd.read_csv(io.StringIO("v\n" + "\n".join(toks) + "\n"), engine="c")["v"].to_numpy(np.float32)
    ints = [t for t in toks if "." not in t]
    as_int = pd.read_csv(io.StringIO("v\n" + "\n".join(ints) + "\n"), engine="c")["v"].to_numpy(np.float32)
    for src, got in ((toks, mixed), (ints, as_int)):
        for t, g in zip(src, got):
            v = cb.lead_field_value(t)
            if v is None:                                              # only negative zeros leave these tokens
                assert float(t) == 0.0 and t.startswith("-")
                continue
            assert np.float32(v).tobytes() == np.float32(g).tobytes(), t


def test_lead_field_rule_rejects_what_pandas_may_read_differently():
    pd = pytest.importorskip("pandas")
    for t in ("-0", "-0.0", "-000.000", "1e2", "+5", ".5", "5.", "1234567890123456", "1.234567890123456", "", " 5", "5 ", "1.2.3",
              "nan", "-", "0x10", "١"):
        assert cb.lead_field_value(t) is None, t
    for t in ("0", "007", "-5", "12.50", "123456789012345", "-0.00000000000001"):
        assert cb.lead_field_value(t) is not None, t
    assert cb.lead_field_value("5", integer_only=True) == 5 and cb.lead_field_value("5.0", integer_only=True) is None
    # why -0 is excluded: pandas' result for it depends on the rest of the column
    ic = pd.read_csv(io.StringIO("v\n-0\n1\n"), engine="c")["v"].to_numpy(np.float32)
    fc = pd.read_csv(io.StringIO("v\n-0\n1.5\n"), engine="c")["v"].to_numpy(np.float32)
    assert not np.signbit(ic[0]) and np.signbit(fc[0])


def test_batch_wrapper_rejects_misplaced_files():
    """Checked before anything reaches the device: the kernels give a chunk to the last file starting at or before it."""
    text = torch.zeros(4 * K, dtype=torch.uint8)
    for off, ln in (([0, K], [K + 1, 10]),            # overlapping files
                    ([0, 100], [10, 10]),             # unaligned offset
                    ([K, 0], [10, 10]),               # not ascending
                    ([0, 3 * K], [10, K + 1]),        # beyond the text
                    ([0], [10, 10])):                 # one length per file
        with pytest.raises(RadarB200Error):
            dev.csv_parse_sweeps(text, np.array(off), np.array(ln), 8)
