"""Chain files (the step-2 -> step-3 hand-off) and the chain statistics step 3 derives from them.

File layout kept from the reference (SURVEY appendix B):
  <dir>/<N>_apf_results/<w>_finalarray_mpi.csv   apf_step2.py:357-360: no header, first row all
        nan (:278-279), then one row per recorded update: P parameters + chi-square
        (17 columns 2-body, 20 columns 3-body); comma separated, CRLF
  <dir>/<N>_apf_results/<w>_acceptance_rate.csv  apf_step2.py:362-365: str(accept/tries)
  step2a.csv / step2a_acceptance_rate            apf_step2a.py:324,329
plus a packed binary format for batches far beyond what per-walker text files can hold.

Statistics restated from apf_step3.py: ingest (:169-214), Gelman-Rubin (:260-278),
separation / position angle (:255-256,283-291), summary (:436-437).
"""
from __future__ import annotations

import json
import math
import os

import numpy as np

from . import _lib

CSV_LEADING_NAN_ROW = 1
CSV_APPEND = 2

PIXSCALE_PRE2015 = 9.952    # mas / pixel, apf_step3.py:224
PIXSCALE_POST2015 = 9.971   # apf_step3.py:231


# ----------------------------------------------------------------------------------------------
# output directory and file names (apf_step2.py:164-173)
# ----------------------------------------------------------------------------------------------
def split_image_path(image_path: str):
    """(directory with trailing '/', image number) -- apf_step2.py:164-170."""
    d = image_path.split("/")
    directory = ""
    for part in d[:-1]:
        directory = directory + str(part) + "/"
    return directory, d[-1].split(".")[-3]


def results_dir(image_path: str) -> str:
    directory, number = split_image_path(image_path)
    return directory + number + "_apf_results/"


def initial_guess_path(image_path: str) -> str:
    directory, number = split_image_path(image_path)
    return directory + number + "_initialguess"


# ----------------------------------------------------------------------------------------------
# writers
# ----------------------------------------------------------------------------------------------
def write_walker_csv(path, rows, leading_nan=True, append=False):
    """Write (or append) one walker's chain rows [n, P+1] float64 through liblapf's native writer."""
    rows = np.ascontiguousarray(rows, dtype=np.float64)
    if rows.ndim != 2:
        raise ValueError("rows must be [n, columns]")
    flags = (CSV_LEADING_NAN_ROW if leading_nan else 0) | (CSV_APPEND if append else 0)
    _lib.check(_lib.load().lapf_write_chain_csv(os.fsencode(path), rows.ctypes.data, rows.shape[0],
                                                rows.shape[1], rows.shape[1], flags))


_pool = None


def _writer_pool():
    global _pool
    if _pool is None:
        import concurrent.futures as cf
        _pool = cf.ThreadPoolExecutor(max_workers=max(1, min(32, (os.cpu_count() or 1))))
    return _pool


def write_segment_csv(paths, segment, first):
    """Append a time-major chain segment [rows, W, P+1] to the W per-walker files ``paths``.
    One file per walker is the reference's layout (apf_step2.py:357); the walkers' files are
    formatted and written concurrently (the native writer runs outside the GIL)."""
    seg = np.ascontiguousarray(segment, dtype=np.float64)
    nrow, nw, ncol = seg.shape
    lib = _lib.load()
    flags = CSV_LEADING_NAN_ROW if first else CSV_APPEND

    def one(w):
        base = seg.ctypes.data + w * ncol * 8
        return lib.lapf_write_chain_csv(os.fsencode(paths[w]), base, nrow, ncol, nw * ncol, flags)

    if nw == 1:
        _lib.check(one(0))
        return
    for rc in _writer_pool().map(one, range(nw)):
        _lib.check(rc)


def write_acceptance(path, accepts, tries):
    """apf_step2.py:362-365: the numpy repr of total_accept / total_tries."""
    with np.errstate(all="ignore"):
        rate = np.asarray(accepts, dtype=np.float64) / np.asarray(tries, dtype=np.float64)
    with open(path, "w") as fh:
        fh.write(str(rate))


def write_draws_csv(path, walkers, values, rows, names):
    """Posterior draws of one epoch (``GibbsSampler.draws``): a '#' header line naming the columns, then
    one line per filled slot -- walker number, recorded-row index, the P parameters, chi-square --
    sorted by (walker, row).  ``walkers`` [W] are the walkers' numbers, ``values`` [W, K, P+1],
    ``rows`` [W, K] (-1: empty slot).  Values are printed as repr(float): they parse back to the same
    doubles.  Returns the number of lines written after the header."""
    walkers = np.asarray(walkers, dtype=np.int64)
    values = np.asarray(values, dtype=np.float64)
    rows = np.asarray(rows, dtype=np.int64)
    w_idx, k_idx = np.nonzero(rows >= 0)
    order = np.lexsort((rows[w_idx, k_idx], walkers[w_idx]))
    w_idx, k_idx = w_idx[order], k_idx[order]
    with open(path, "w") as fh:
        fh.write("# " + ",".join(["walker", "row"] + list(names)) + "\n")
        for w, k in zip(w_idx.tolist(), k_idx.tolist()):
            fh.write("%d,%d,%s\n" % (walkers[w], rows[w, k], ",".join(map(repr, values[w, k].tolist()))))
    return len(w_idx)


def read_draws_csv(path):
    """(names, walker [n] int64, row [n] int64, values [n, P+1] float64) of a ``write_draws_csv`` file."""
    with open(path) as fh:
        head = fh.readline()
        if not head.startswith("# "):
            raise ValueError("%s: not a draws file" % path)
        names = head[2:].strip().split(",")[2:]
        lines = [ln.split(",") for ln in fh.read().splitlines() if ln]
    walker = np.array([int(x[0]) for x in lines], dtype=np.int64)
    row = np.array([int(x[1]) for x in lines], dtype=np.int64)
    values = np.array([[float(v) for v in x[2:]] for x in lines], dtype=np.float64).reshape(len(lines), len(names))
    return names, walker, row, values


# ----------------------------------------------------------------------------------------------
# chain events (LAPF_CHAIN_EVENTS_*, include/lapf.h): the one place on the host that knows the layout
# ----------------------------------------------------------------------------------------------
EVENT_MAGIC = b"LAPFEVT1"
EVENT_HEADER = 32         # magic, rows (int64), walkers (int64), columns (int32), bytes per value (int32)


def _event_parts(rows, n_walkers, n_cols, itemsize):
    """Byte offsets of (codes, values, chi-square) and the total size of an event buffer."""
    codes = itemsize * n_walkers * n_cols
    values = codes + (rows * n_walkers + 15) // 16 * 16
    chi = values + itemsize * rows * n_walkers
    return codes, values, chi, chi + itemsize * rows * n_walkers


def event_bytes(rows, n_walkers, n_cols, dtype):
    """Size of the event buffer of ``rows`` rows (0 rows: nothing, not even the key)."""
    return _event_parts(rows, n_walkers, n_cols, np.dtype(dtype).itemsize)[3] if rows else 0


def decode_events(buf, rows, n_walkers, n_cols, dtype):
    """The dense chain rows [rows, n_walkers, n_cols] of one event buffer (a uint8 array as
    ``lapf_sampler_run`` wrote it in an event format): float64 values, or float32 differences
    from the starting point -- bit for bit what the dense format of that precision writes.
    Row r is row r-1 with column k replaced by the event's value and the last column by its
    chi-square; vectorised over rows: per column, the last event at or before each row."""
    dt = np.dtype(dtype)
    W, C, R = int(n_walkers), int(n_cols), int(rows)
    if R == 0:
        return np.empty((0, W, C), dtype=dt)
    buf = np.asarray(buf, dtype=np.uint8).reshape(-1)
    o_code, o_val, o_chi, end = _event_parts(R, W, C, dt.itemsize)
    if buf.size < end:
        raise ValueError("event buffer of %d bytes is shorter than the %d of %d rows x %d walkers" % (buf.size, end, R, W))
    key = buf[:o_code].view(dt).reshape(W, C)
    k = (buf[o_code:o_code + R * W] & 31).reshape(R, W)
    values = buf[o_val:o_chi].view(dt).reshape(R, W)
    out = np.empty((R, W, C), dtype=dt)
    out[:, :, C - 1] = buf[o_chi:end].view(dt).reshape(R, W)
    rix = np.arange(1, R + 1, dtype=np.int32)[:, None]
    # blocks of walkers keep each column's gather inside the cache (3x faster at 65,536 walkers)
    for w0 in range(0, W, 256):
        n = min(W, w0 + 256) - w0
        kb, ob = k[:, w0:w0 + n], out[:, w0:w0 + n]
        src = np.empty((R + 1, n), dtype=dt)        # row 0: the key, row 1 + r: the values of event r
        src[1:] = values[:, w0:w0 + n]
        flat, cols = src.reshape(-1), np.arange(n, dtype=np.int32)[None, :]
        for c in range(C - 1):
            src[0] = key[w0:w0 + n, c]
            last = np.maximum.accumulate(np.where(kb == c, rix, 0), axis=0)   # 0: no event of column c yet
            ob[:, :, c] = flat[last * n + cols]
    return out


def _event_segments(path):
    """[(offset of the payload, rows, walkers, columns, bytes per value)] of the complete segments of
    an event file, and the byte size they cover (a torn last segment is not included)."""
    segs, pos = [], 0
    size = os.path.getsize(path)
    with open(path, "rb") as fh:
        while pos + EVENT_HEADER <= size:
            fh.seek(pos)
            head = fh.read(EVENT_HEADER)
            if head[:8] != EVENT_MAGIC:
                raise ValueError("%s: no event segment at byte %d" % (path, pos))
            rows, walkers = (int(v) for v in np.frombuffer(head, dtype="<i8", count=2, offset=8))
            cols, item = (int(v) for v in np.frombuffer(head, dtype="<i4", count=2, offset=24))
            end = pos + EVENT_HEADER + _event_parts(rows, walkers, cols, item)[3]
            if end > size:
                break
            segs.append((pos + EVENT_HEADER, rows, walkers, cols, item))
            pos = end
    return segs, pos


class PackedChainWriter:
    """Packed binary chain: [row][walker][P+1] appended segment by segment to ``<base>.bin`` with a
    JSON sidecar ``<base>.json``; for batches of 10^4..10^6 walkers where one text file per walker
    is not workable.  dtype 'float64' holds the values; 'float32' holds differences from the
    walkers' starting points, which are stored once as float64 in ``<base>.start.bin``
    (LAPF_CHAIN_F32_DELTA).  ``resume=True`` appends to an existing file of the same shape (the
    sidecar tells the row count so far).  ``read_packed`` / ``unpack_to_csv`` convert back.

    ``events=True`` stores the event buffers of an event chain format instead (thin = 1; about a
    seventh of the bytes) in ``<base>.events``, one self-describing segment per ``append_events``:
    a 32-byte header (magic LAPFEVT1, rows, walkers, columns, bytes per value) and the buffer as the
    device wrote it.  Resuming walks the headers and drops a torn last segment."""

    def __init__(self, base, n_walkers, n_cols, meta=None, dtype="float64", start=None, resume=False, events=False):
        self.base, self.n_walkers, self.n_cols = base, int(n_walkers), int(n_cols)
        self.dtype = np.dtype(dtype)
        if self.dtype not in (np.dtype("float64"), np.dtype("float32")):
            raise ValueError("packed chains are float64 or float32 (differences from the start)")
        self.events = bool(events)
        self.path = base + (".events" if self.events else ".bin")
        self.rows = 0
        self.meta = dict(meta or {})
        if resume:
            with open(base + ".json") as fh:
                old = json.load(fh)
            if (old["n_walkers"], old["n_cols"], old["dtype"], old.get("format", "rows")) != (
                    self.n_walkers, self.n_cols, self.dtype.name, "events" if self.events else "rows"):
                raise ValueError("%s holds %s walkers x %s columns of %s (%s): cannot append %d x %d of %s"
                                 % (base, old["n_walkers"], old["n_cols"], old["dtype"], old.get("format", "rows"),
                                    self.n_walkers, self.n_cols, self.dtype.name))
            if self.events:
                # keep the complete segments the sidecar counts; a torn or uncounted tail is dropped
                segs, _ = _event_segments(self.path)
                want = 0
                for off, rows, _, _, item in segs:
                    if self.rows + rows > old["rows"]:
                        break
                    self.rows += rows
                    want = off + _event_parts(rows, self.n_walkers, self.n_cols, item)[3]
                if self.rows != old["rows"]:
                    raise ValueError("%s holds fewer rows than its sidecar says" % self.path)
            else:
                have = os.path.getsize(self.path)
                want = old["rows"] * self.n_walkers * self.n_cols * self.dtype.itemsize
                if have < want:
                    raise ValueError("%s.bin is shorter than its sidecar says" % base)
                self.rows = int(old["rows"])
            self.meta = {**old, **self.meta}
            self.fh = open(self.path, "r+b")
            self.fh.truncate(want)                      # drop a partial segment of an interrupted run
            self.fh.seek(want)
        else:
            self.fh = open(self.path, "wb")
            if self.dtype == np.dtype("float32"):
                if start is None:
                    raise ValueError("float32 chains are differences: the starting points are needed")
                st = np.ascontiguousarray(start, dtype=np.float64)
                assert st.shape == (self.n_walkers, self.n_cols)
                st.tofile(base + ".start.bin")

    def append(self, segment):
        if self.events:
            raise ValueError("an event file takes event buffers (append_events)")
        seg = np.ascontiguousarray(segment, dtype=self.dtype)
        assert seg.shape[1:] == (self.n_walkers, self.n_cols)
        self.fh.write(seg.tobytes())
        self.rows += seg.shape[0]

    def append_events(self, payload, rows):
        """One event buffer of ``rows`` rows, as ``GibbsSampler.run`` / ``ChainStreamer`` return it."""
        if not self.events:
            raise ValueError("a row file takes rows (append)")
        payload = np.asarray(payload, dtype=np.uint8).reshape(-1)
        n = event_bytes(rows, self.n_walkers, self.n_cols, self.dtype)
        if rows == 0:
            return
        if payload.size < n:
            raise ValueError("event buffer of %d bytes, %d rows need %d" % (payload.size, rows, n))
        head = EVENT_MAGIC + np.array([rows, self.n_walkers], dtype="<i8").tobytes() + \
            np.array([self.n_cols, self.dtype.itemsize], dtype="<i4").tobytes()
        self.fh.write(head)
        self.fh.write(payload[:n].tobytes())
        self.rows += int(rows)

    def close(self, **extra):
        self.fh.close()
        self.meta.update(extra)
        self.meta.update({"rows": self.rows, "n_walkers": self.n_walkers, "n_cols": self.n_cols,
                          "dtype": self.dtype.name, "order": "[row][walker][column]",
                          "format": "events" if self.events else "rows",
                          "values": "differences from <base>.start.bin" if self.dtype == np.dtype("float32") else "absolute"})
        with open(self.base + ".json", "w") as fh:
            json.dump(self.meta, fh, indent=1)


def read_packed(base):
    """(chain [rows, walkers, columns] float64, meta) of a packed chain, whatever its storage type."""
    with open(base + ".json") as fh:
        meta = json.load(fh)
    shape = (meta["rows"], meta["n_walkers"], meta["n_cols"])
    dt = np.dtype(meta.get("dtype", "float64"))
    if meta.get("format", "rows") == "events":
        raw = np.memmap(base + ".events", dtype=np.uint8, mode="r")
        parts, have = [], 0
        for off, rows, walkers, cols, _ in _event_segments(base + ".events")[0]:
            if have + rows > shape[0]:
                break
            parts.append(decode_events(raw[off:], rows, walkers, cols, dt))
            have += rows
        if have != shape[0]:
            raise ValueError("%s.events holds fewer rows than its sidecar says" % base)
        arr = np.concatenate(parts, axis=0) if parts else np.empty(shape, dtype=dt)
    else:
        arr = np.fromfile(base + ".bin", dtype=dt, count=int(np.prod(shape))).reshape(shape)
    if dt == np.dtype("float32"):
        start = np.fromfile(base + ".start.bin", dtype=np.float64).reshape(shape[1:])
        arr = start[None] + arr.astype(np.float64)
    return arr, meta


def unpack_to_csv(base, out_dir, walkers=None):
    """Per-walker reference CSVs from a packed chain, so an unmodified apf_step3.py can read them."""
    arr, meta = read_packed(base)
    os.makedirs(out_dir, exist_ok=True)
    ids = range(arr.shape[1]) if walkers is None else walkers
    for w in ids:
        write_walker_csv(os.path.join(out_dir, "%d_finalarray_mpi.csv" % w), arr[:, w, :])
    return len(list(ids))


# ----------------------------------------------------------------------------------------------
# step-3 side: ingest and statistics
# ----------------------------------------------------------------------------------------------
def read_walker_csv(path):
    return np.genfromtxt(path, delimiter=",")


def ingest(input_directory, ncor, additional_burnin=1):
    """apf_step3.py:169-214: load ncor walker files into [length, ncor] arrays per column, drop
    the first ``additional_burnin`` rows (default 1 = the nan row, :81-84), add 1 to the positions
    (FITS pixels are 1-based, :211-214).  Every file must have the same number of rows (:183).
    Returns (columns [n_cols, length-burn, ncor], n_position_columns)."""
    if not additional_burnin:
        additional_burnin = 1
    first = read_walker_csv(os.path.join(input_directory, "0_finalarray_mpi.csv"))
    length, ncols = first.shape
    cols = np.zeros((ncols, length, ncor))
    for i in range(ncor):
        a = first if i == 0 else read_walker_csv(os.path.join(input_directory, "%d_finalarray_mpi.csv" % i))
        if a.shape != (length, ncols):
            raise ValueError("walker %d has %s rows/cols, walker 0 has %s" % (i, a.shape, (length, ncols)))
        cols[:, :, i] = a.T
    cols = cols[:, additional_burnin:length, :]
    npos = 4 if ncols == 17 else 6
    cols[:npos] += 1.0
    return cols, npos


def gelman_rubin(chains, python2_division=True):
    """apf_step3.py:262-276 for one parameter; ``chains`` is [n_rows, n_walkers].  Returns
    (PSRF, RC).  The reference computes (d+3)/(d+1) with d = 16 under Python 2: integer 1."""
    chains = np.asarray(chains, dtype=np.float64)
    n, m = float(chains.shape[0]), float(chains.shape[1])
    w = (1.0 / m) * np.sum(np.std(chains, axis=0) ** 2)
    b = (n / (m - 1.0)) * np.sum((np.mean(chains, axis=0) - np.mean(chains)) ** 2)
    psrf = (((n - 1.0) / n) * w + ((m + 1.0) / (m * n)) * b) / w
    factor = 1.0 if python2_division else 19.0 / 17.0
    return psrf, math.sqrt(factor * psrf)


def gelman_rubin_from_moments(moments, n_rows, n_walkers, python2_division=True):
    """The same statistic from the device-reduced sufficient statistics of ``lapf_sampler_stats``:
    moments[..., 0] = reference value r, [..., 1] = sum of (chain mean - r), [..., 2] = sum of
    (chain mean - r)^2, [..., 3] = sum of chain variances.  Equal-length chains make the overall
    mean the mean of the chain means."""
    mom = np.asarray(moments, dtype=np.float64)
    n, m = float(n_rows), np.asarray(n_walkers, dtype=np.float64)
    s_mean, s_mean2, s_var = mom[..., 1], mom[..., 2], mom[..., 3]
    w = s_var / m
    overall = s_mean / m
    b = (n / (m - 1.0)) * (s_mean2 - m * overall * overall)
    with np.errstate(divide="ignore", invalid="ignore"):   # a parameter that never moved has w = 0
        psrf = (((n - 1.0) / n) * w + ((m + 1.0) / (m * n)) * b) / w
    factor = 1.0 if python2_division else 19.0 / 17.0
    return psrf, np.sqrt(factor * psrf)


def separation_pa(xcs, ycs, xcc, ycc, pixscale=PIXSCALE_PRE2015):
    """apf_step3.py:255-256,283-291 (without the distortion lookup: its FITS tables are not part
    of the checkout): sep = sqrt(dx^2+dy^2)*pixscale [mas], pa = degrees(atan2(-dx, dy))."""
    dy = np.asarray(ycc) - np.asarray(ycs)
    dx = np.asarray(xcc) - np.asarray(xcs)
    return np.sqrt(dy * dy + dx * dx) * pixscale, np.degrees(np.arctan2(-dx, dy))


def summarize(values):
    """median, 16th/84th percentiles, mean, std (apf_step3.py:436-437 uses median and std)."""
    v = np.asarray(values, dtype=np.float64).ravel()
    lo, med, hi = np.percentile(v, [15.865, 50.0, 84.135])
    return {"median": float(med), "lo": float(lo), "hi": float(hi), "mean": float(v.mean()),
            "std": float(v.std())}
