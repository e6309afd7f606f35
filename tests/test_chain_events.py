"""Chain events on the host (LAPF_CHAIN_EVENTS_*, include/lapf.h): the decoder against a plain
per-row decoder, the packed event file and its resume, and the command line's --format events
guard.  No GPU: the buffers are built here in the device's layout."""
import json
import os

import numpy as np
import pytest

from olpefit_b200 import chains


def _random_chain(rows, walkers, cols, dtype, seed):
    """A dense chain in which every row differs from the one before it in one parameter and
    chi-square (thin = 1), and its event buffer."""
    rng = np.random.default_rng(seed)
    P = cols - 1
    dense = np.empty((rows, walkers, cols), dtype=dtype)
    k = rng.integers(0, P, size=(rows, walkers))
    acc = rng.random((rows, walkers)) < 0.4
    row = rng.normal(size=(walkers, cols)).astype(dtype)
    for r in range(rows):
        if r:
            row = row.copy()
            w = np.nonzero(acc[r])[0]
            row[w, k[r, w]] = rng.normal(size=w.size).astype(dtype)
        row[:, P] = rng.normal(size=walkers).astype(dtype)
        dense[r] = row
    codes = (k | (acc << 7)).astype(np.uint8)
    values = np.take_along_axis(dense[..., :P], k[..., None], axis=2)[..., 0]
    pad = -(rows * walkers) % 16
    buf = np.concatenate([dense[0].reshape(-1).view(np.uint8), codes.reshape(-1), np.zeros(pad, np.uint8),
                          np.ascontiguousarray(values).reshape(-1).view(np.uint8),
                          np.ascontiguousarray(dense[..., P]).reshape(-1).view(np.uint8)])
    return dense, buf


def _decode_per_row(buf, rows, walkers, cols, dtype):
    """The layout read one row at a time: row r = row r-1 with column k and chi-square replaced."""
    dt = np.dtype(dtype)
    e = dt.itemsize
    key = buf[:e * walkers * cols].view(dt).reshape(walkers, cols)
    o_code = e * walkers * cols
    o_val = o_code + -(-rows * walkers // 16) * 16
    o_chi = o_val + e * rows * walkers
    out, row = [], key.copy()
    for r in range(rows):
        for w in range(walkers):
            k = buf[o_code + r * walkers + w] & 31
            row[w, k] = buf[o_val + e * (r * walkers + w):o_val + e * (r * walkers + w + 1)].view(dt)[0]
            row[w, cols - 1] = buf[o_chi + e * (r * walkers + w):o_chi + e * (r * walkers + w + 1)].view(dt)[0]
        out.append(row.copy())
    return np.array(out, dtype=dt).reshape(rows, walkers, cols)


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("rows,walkers,cols", [(1, 1, 17), (7, 5, 17), (33, 24, 20), (50, 3, 17)])
def test_decode_events_equals_per_row_decoder(dtype, rows, walkers, cols):
    dense, buf = _random_chain(rows, walkers, cols, dtype, seed=rows * 100 + walkers)
    assert buf.size == chains.event_bytes(rows, walkers, cols, dtype)
    got = chains.decode_events(buf, rows, walkers, cols, dtype)
    assert got.dtype == np.dtype(dtype) and got.shape == (rows, walkers, cols)
    assert got.tobytes() == _decode_per_row(buf, rows, walkers, cols, dtype).tobytes()
    assert got.tobytes() == dense.tobytes()
    assert chains.decode_events(buf[:0], 0, walkers, cols, dtype).shape == (0, walkers, cols)
    with pytest.raises(ValueError):
        chains.decode_events(buf[:-1], rows, walkers, cols, dtype)


def test_decode_events_keeps_nan_and_signed_zero_bits():
    dense, buf = _random_chain(6, 4, 17, np.float64, seed=5)
    buf = buf.copy()
    o_val = 8 * 4 * 17 + 32
    vals = buf[o_val:o_val + 8 * 24].view(np.float64)
    vals[5] = -0.0
    vals[9] = np.nan
    got = chains.decode_events(buf, 6, 4, 17, np.float64)
    assert got.tobytes() == _decode_per_row(buf, 6, 4, 17, np.float64).tobytes()


@pytest.mark.parametrize("dtype", ["float64", "float32"])
def test_event_file_round_trip(tmp_path, dtype):
    W, C = 5, 17
    start = np.random.default_rng(2).normal(size=(W, C))
    base = str(tmp_path / "chains_rank0")
    wr = chains.PackedChainWriter(base, W, C, {"seed": 1}, dtype=dtype, start=start if dtype == "float32" else None,
                                  events=True)
    parts = []
    for i, rows in enumerate((9, 1, 16)):
        dense, buf = _random_chain(rows, W, C, np.dtype(dtype), seed=40 + i)
        wr.append_events(buf, rows)
        parts.append(dense)
    wr.append_events(np.zeros(0, np.uint8), 0)                 # a run that recorded nothing
    wr.close(count=26)
    meta = json.load(open(base + ".json"))
    assert meta["format"] == "events" and meta["rows"] == 26 and meta["dtype"] == dtype
    assert not os.path.exists(base + ".bin")
    want = np.concatenate(parts)
    if dtype == "float32":
        want = start[None] + want.astype(np.float64)
    arr, meta2 = chains.read_packed(base)
    assert arr.dtype == np.float64 and np.array_equal(arr, want) and meta2["count"] == 26
    assert chains.unpack_to_csv(base, str(tmp_path / "csv")) == W
    # the CSV of the event file is the CSV of the same rows written directly
    chains.write_walker_csv(str(tmp_path / "direct.csv"), want[:, 3, :])
    assert open(str(tmp_path / "csv" / "3_finalarray_mpi.csv"), "rb").read() == open(str(tmp_path / "direct.csv"), "rb").read()
    with pytest.raises(ValueError):
        chains.PackedChainWriter(base, W, C, dtype=dtype, resume=True, events=False)   # a row file is not an event file


def test_event_file_resume_drops_a_torn_segment(tmp_path):
    W, C = 3, 17
    base = str(tmp_path / "ev")
    segs = [_random_chain(rows, W, C, np.float64, seed=s) for s, rows in enumerate((4, 6, 5))]
    wr = chains.PackedChainWriter(base, W, C, events=True)
    wr.append_events(segs[0][1], 4)
    wr.append_events(segs[1][1], 6)
    wr.close()
    size = os.path.getsize(base + ".events")
    # an interrupted run: a third segment began to be written, the sidecar was not updated
    with open(base + ".events", "ab") as fh:
        fh.write(b"LAPFEVT1" + np.array([5, W], "<i8").tobytes() + np.array([C, 8], "<i4").tobytes())
        fh.write(segs[2][1][:100].tobytes())
    arr, _ = chains.read_packed(base)
    assert arr.shape == (10, W, C)
    wr = chains.PackedChainWriter(base, W, C, events=True, resume=True)
    assert wr.rows == 10 and os.path.getsize(base + ".events") == size
    wr.append_events(segs[2][1], 5)
    wr.close()
    arr, meta = chains.read_packed(base)
    assert meta["rows"] == 15 and np.array_equal(arr, np.concatenate([s[0] for s in segs]))
    # a complete segment the sidecar does not count (written after the last checkpoint) is dropped too
    json.dump({**meta, "rows": 4}, open(base + ".json", "w"))
    wr = chains.PackedChainWriter(base, W, C, events=True, resume=True)
    wr.close()
    arr, _ = chains.read_packed(base)
    assert np.array_equal(arr, segs[0][0])


def test_format_events_needs_thin_1_before_any_device_is_touched(tmp_path):
    from olpefit_b200 import cli
    with pytest.raises(SystemExit, match="--thin 1"):
        cli.main_step2([str(tmp_path / "N2.20090531.29966.LDIF.fits"), "--format", "events", "--thin", "4"])
