"""Host-side driver of the batched Gibbs-within-Metropolis sampler (apf_step2.py:276-351).

The reference runs one MPI rank per walker (apf_step2.py:54-57); here one ``GibbsSampler`` owns
a batch of independent walkers on one GPU.  Per update and walker the device does exactly what
the reference loop does: pick a parameter uniformly (:302), propose (:306-309), evaluate
model + chi-square (:314-316), accept or reject (:318-327), count, and record a chain row once
count >= burn_in (:342-351).
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from .model import PixelDomain, _stream_ptr


def prior_table(n_frames, nparam, lo=None, hi=None, mu=None, sigma=None):
    """The [F, P, 4] {lo, hi, mu, sigma} table of lapf_sampler_set_priors from per-parameter arrays, each [P]
    (every frame) or [F, P], or None: no bound (-inf / +inf), no Gaussian term (sigma +inf, mu 0)."""
    out = np.empty((n_frames, nparam, 4), dtype=np.float64)
    for i, (v, none) in enumerate(((lo, -np.inf), (hi, np.inf), (mu, 0.0), (sigma, np.inf))):
        if v is None:
            out[..., i] = none
            continue
        a = np.asarray(v.cpu().numpy() if torch.is_tensor(v) else v, dtype=np.float64)
        if a.shape not in ((nparam,), (n_frames, nparam)):
            raise ValueError("prior arrays must be [%d] or [%d, %d], got %s" % (nparam, n_frames, nparam, a.shape))
        out[..., i] = np.broadcast_to(a, (n_frames, nparam))
    return out


class GibbsSampler:
    def __init__(self, domain: PixelDomain, init_params, frame_of=None, *, seed=0, burn_in=0, thin=1,
                 widths=None, id_base=0, id_stride=1, team_warps=0):
        self.lib = _lib.load()
        self.domain = domain
        dev = domain.device
        p = init_params if torch.is_tensor(init_params) else torch.as_tensor(np.asarray(init_params, dtype=np.float64))
        p = p.to(dev, torch.float64).reshape(-1, domain.nparam).contiguous()
        self.n_walkers = int(p.shape[0])
        self.nparam = domain.nparam
        fo = None
        if frame_of is not None:
            fo = frame_of if torch.is_tensor(frame_of) else torch.as_tensor(np.asarray(frame_of, dtype=np.int32))
            fo = fo.to(dev, torch.int32).contiguous()
            if fo.numel() != self.n_walkers:
                raise ValueError("frame_of must have one entry per walker")
        self._keep = (p, fo)   # the library copies init_params; frame_of is only read in create()
        w_arr = None
        if widths is not None:
            w_np = np.ascontiguousarray(widths, dtype=np.float64)
            if w_np.shape != (self.nparam,):
                raise ValueError("widths must have %d entries" % self.nparam)
            w_arr = (C.c_double * self.nparam)(*w_np.tolist())
        cfg = _lib.Config(domain.problem(), self.n_walkers, int(id_base), int(id_stride),
                          int(seed) & 0xFFFFFFFFFFFFFFFF, fo.data_ptr() if fo is not None else None,
                          p.data_ptr(), w_arr, int(burn_in), int(thin), int(team_warps))
        self.burn_in, self.thin = int(burn_in), int(thin)
        self.chain_dtype = torch.float64
        self.events = False
        self._sketch = None
        self._bm = None
        self._draws = None
        handle = C.c_void_p()
        _lib.check(self.lib.lapf_sampler_create(C.byref(cfg), C.byref(handle), _stream_ptr(dev)))
        self._h = handle

    # -- lifetime ------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None):
            torch.cuda.synchronize(self.domain.device)
            self.lib.lapf_sampler_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def reset(self, init_params, seed=0):
        """Start a new batch in this sampler: new starting points and seed; counters, moments
        and the update count return to zero and the initial chi-square is re-evaluated against
        the domain's current pixel buffers (see ``frame.prepare_domain(into=...)``)."""
        dev = self.domain.device
        p = init_params if torch.is_tensor(init_params) else torch.as_tensor(np.asarray(init_params, dtype=np.float64))
        p = p.to(dev, torch.float64).reshape(-1, self.nparam).contiguous()
        if p.shape[0] != self.n_walkers:
            raise ValueError("init_params must have one row per walker")
        self._keep = (p, self._keep[1])
        _lib.check(self.lib.lapf_sampler_reset(self._h, p.data_ptr(), int(seed) & 0xFFFFFFFFFFFFFFFF,
                                               _stream_ptr(dev)))

    def save(self):
        """Checkpoint of the whole batch as a device uint8 tensor (see lapf_sampler_save)."""
        n = int(_lib.check(self.lib.lapf_sampler_checkpoint_bytes(self._h)))
        blob = torch.empty(n, dtype=torch.uint8, device=self.domain.device)
        _lib.check(self.lib.lapf_sampler_save(self._h, blob.data_ptr(), n, _stream_ptr(self.domain.device)))
        return blob

    def load(self, blob):
        """Restore a checkpoint made by ``save`` on a sampler of the same shape: the following runs
        continue the chains bit for bit."""
        blob = blob.to(self.domain.device).contiguous()
        _lib.check(self.lib.lapf_sampler_load(self._h, blob.data_ptr(), blob.numel(), _stream_ptr(self.domain.device)))

    def set_widths(self, widths):
        """New jump widths for the following runs (burn-in tuning; the reference's are fixed)."""
        w_np = np.ascontiguousarray(widths, dtype=np.float64)
        if w_np.shape != (self.nparam,):
            raise ValueError("widths must have %d entries" % self.nparam)
        _lib.check(self.lib.lapf_sampler_set_widths(self._h, (C.c_double * self.nparam)(*w_np.tolist())))

    def set_chain_format(self, fmt: str):
        """'f64': rows are the values themselves (default).  'f32delta': rows are float32 differences
        from the walker's starting point (``start()``) -- half the bytes to drain, and exact to ~1e-7
        of the distance travelled (see include/lapf.h).  'events_f64' / 'events_f32delta' (thin = 1
        only): each run writes the rows of the dense format of that precision as one changed parameter
        and chi-square per row and walker; ``run`` returns that buffer and
        ``chains.decode_events`` rebuilds the rows."""
        code = {"f64": 0, "f32delta": 1, "events_f64": 2, "events_f32delta": 3}[fmt]
        _lib.check(self.lib.lapf_sampler_set_chain_format(self._h, code))
        self.chain_dtype = torch.float32 if code in (1, 3) else torch.float64
        self.events = code >= 2

    def start(self):
        """[W, P+1] float64 device tensor: every walker's starting point and its chi-square."""
        out = torch.empty((self.n_walkers, self.nparam + 1), dtype=torch.float64, device=self.domain.device)
        _lib.check(self.lib.lapf_sampler_start(self._h, out.data_ptr(), _stream_ptr(self.domain.device)))
        return out

    # -- separation / position angle without the chain (apf_step3.py:255-256,283-291,436-437) ---------
    def enable_sketch(self, n_bins=16384, sep_bin=5e-4, pa_bin=2e-3, centers=None):
        """From now on every recorded row enters per-frame histograms of separation (pixels) and
        position angle (degrees) of each companion; call before the first ``run``.  ``centers``:
        [F, nbody-1, 2] centre values (give every rank the same ones), default: the starting point
        of each frame's first walker."""
        dev = self.domain.device
        c = None
        if centers is not None:
            c = centers if torch.is_tensor(centers) else torch.as_tensor(np.asarray(centers, dtype=np.float64))
            c = c.to(dev, torch.float64).reshape(self.domain.n_frames, self.domain.nbody - 1, 2).contiguous()
        _lib.check(self.lib.lapf_sampler_sketch_enable(self._h, int(n_bins), float(sep_bin), float(pa_bin),
                                                       c.data_ptr() if c is not None else None, _stream_ptr(dev)))
        self._sketch = (int(n_bins), float(sep_bin), float(pa_bin))

    def sketch(self):
        """dict(hist [F, nbody-1, 2, n_bins+2] int64, summary [F, nbody-1, 2, 4] float64 (centre, sum,
        sum of squares of value - centre, count), n_bins, sep_bin, pa_bin) as device tensors."""
        if self._sketch is None:
            raise _lib.LapfError("sketches are not enabled")
        dev = self.domain.device
        n_bins, sep_bin, pa_bin = self._sketch
        shape = (self.domain.n_frames, self.domain.nbody - 1, 2)
        hist = torch.empty(shape + (n_bins + 2,), dtype=torch.int32, device=dev)      # uint32 counts
        summ = torch.empty(shape + (4,), dtype=torch.float64, device=dev)
        _lib.check(self.lib.lapf_sampler_sketch(self._h, hist.data_ptr(), summ.data_ptr(), _stream_ptr(dev)))
        return {"hist": hist.long() & 0xFFFFFFFF, "summary": summ, "n_bins": n_bins, "sep_bin": sep_bin, "pa_bin": pa_bin}

    # -- batch means: Monte Carlo standard errors without the chain --------------------------
    def enable_batch_means(self, batch_rows=64, levels=12):
        """From now on every walker keeps batch means of every recorded value at batch lengths
        batch_rows * 2^l rows, l < levels: the chain columns and, if ``enable_sketch`` was called
        before, the separation and position angle of each companion.  Call before the first recorded
        row.  ``stats.batch_means_summary`` turns them into effective sample sizes and standard errors."""
        _lib.check(self.lib.lapf_sampler_batchmeans_enable(self._h, int(batch_rows), int(levels),
                                                           _stream_ptr(self.domain.device)))
        names = list(self._param_names()) + ["chi2"]
        if self._sketch is not None:
            for o in range(1, self.domain.nbody):
                names += ["sep%d" % o, "pa%d" % o]
        self._bm = (int(batch_rows), int(levels), names)

    def _param_names(self):
        from . import layout
        return layout.names(self.domain.nbody)

    def batch_means(self):
        """dict(walker [W, C, levels, 2] (snap, s2), frame [F, C, 1 + levels] (sum over the frame's walkers
        of their row variance, then of the sample variance of their level-l batch means) as float64 device
        tensors, batch_rows, levels, rows (recorded per walker), names [C]) -- see include/lapf.h."""
        if self._bm is None:
            raise _lib.LapfError("batch means are not enabled")
        dev = self.domain.device
        batch_rows, levels, names = self._bm
        c = len(names)
        walker = torch.empty((self.n_walkers, c, levels, 2), dtype=torch.float64, device=dev)
        frame = torch.empty((self.domain.n_frames, c, 1 + levels), dtype=torch.float64, device=dev)
        _lib.check(self.lib.lapf_sampler_batchmeans(self._h, walker.data_ptr(), frame.data_ptr(), _stream_ptr(dev)))
        return {"walker": walker, "frame": frame, "batch_rows": batch_rows, "levels": levels,
                "rows": self.rows_recorded(), "names": names}

    # -- posterior draws: a uniform sample of every walker's recorded rows -----------------------
    def enable_draws(self, per_walker):
        """From now on every walker keeps a uniformly random sample of ``per_walker`` of its recorded
        rows (reservoir sampling on the device, see include/lapf.h).  Call before the first recorded row."""
        _lib.check(self.lib.lapf_sampler_draws_enable(self._h, int(per_walker), _stream_ptr(self.domain.device)))
        self._draws = int(per_walker)

    def draws(self):
        """dict(values [W, K, P+1] float64 (the rows: parameters, chi-square), rows [W, K] int64 (the
        walker's recorded-row index of each slot, -1: empty) as device tensors, per_walker K, filled
        = min(K, rows_recorded()): the slots that hold a row)."""
        if self._draws is None:
            raise _lib.LapfError("draws are not enabled")
        dev, k = self.domain.device, self._draws
        values = torch.empty((self.n_walkers, k, self.nparam + 1), dtype=torch.float64, device=dev)
        rows = torch.empty((self.n_walkers, k), dtype=torch.int64, device=dev)
        _lib.check(self.lib.lapf_sampler_draws(self._h, values.data_ptr(), rows.data_ptr(), _stream_ptr(dev)))
        return {"values": values, "rows": rows, "per_walker": k, "filled": min(k, self.rows_recorded())}

    # -- per-epoch jump widths, tuned on the device ----------------------------------------------
    def set_frame_widths(self, widths=None):
        """From now on the walkers of frame f propose with the jump widths of row f: ``widths`` [F, P]
        (host values), or None for the batch widths in every row.  The first call turns the table on;
        ``set_widths`` is then refused.  See include/lapf.h."""
        nf = self.domain.n_frames
        w_arr = None
        if widths is not None:
            w_np = np.ascontiguousarray(widths.cpu().numpy() if torch.is_tensor(widths) else widths, dtype=np.float64)
            if w_np.shape != (nf, self.nparam):
                raise ValueError("widths must be [%d, %d]" % (nf, self.nparam))
            w_arr = (C.c_double * w_np.size)(*w_np.reshape(-1).tolist())
        _lib.check(self.lib.lapf_sampler_set_frame_widths(self._h, w_arr, _stream_ptr(self.domain.device)))

    def frame_widths(self):
        """[F, P] float64 device tensor: the per-frame jump widths."""
        dev = self.domain.device
        out = torch.empty((self.domain.n_frames, self.nparam), dtype=torch.float64, device=dev)
        _lib.check(self.lib.lapf_sampler_frame_widths(self._h, out.data_ptr(), _stream_ptr(dev)))
        return out

    def frame_counts(self):
        """[F, P, 2] int64 device tensor: per frame and parameter, the tries and accepts of the frame's
        walkers since the last reset (exact integer sums: all-reduce them over ranks)."""
        dev = self.domain.device
        out = torch.empty((self.domain.n_frames, self.nparam, 2), dtype=torch.int64, device=dev)
        _lib.check(self.lib.lapf_sampler_frame_counts(self._h, out.data_ptr(), _stream_ptr(dev)))
        return out

    def adapt_widths(self, counts, target=0.35):
        """One adaptation step of the per-frame widths from cumulative ``frame_counts()`` (summed over
        ranks): each width is scaled by exp(rate - target), clipped to [0.5, 2], where rate is the
        acceptance over the window since the previous step; on the device, without a host sync."""
        c = counts.to(self.domain.device, torch.int64).contiguous()
        if tuple(c.shape) != (self.domain.n_frames, self.nparam, 2):
            raise ValueError("counts must be [%d, %d, 2]" % (self.domain.n_frames, self.nparam))
        _lib.check(self.lib.lapf_sampler_adapt_widths(self._h, c.data_ptr(), float(target), _stream_ptr(self.domain.device)))

    # -- parameter priors: per-epoch boxes and Gaussian terms in the accept rule ------------------
    def set_priors(self, lo=None, hi=None, mu=None, sigma=None):
        """From now on the walkers of frame f see, on parameter j, the box lo <= value <= hi and the Gaussian
        term N(mu, sigma), in chain units.  Each argument is [P] (every frame) or [F, P]; a missing argument
        means none (lo -inf, hi +inf, sigma +inf), and so do those values in an array.  Refused if a walker's
        current state lies outside its box.  See include/lapf.h."""
        table = prior_table(self.domain.n_frames, self.nparam, lo, hi, mu, sigma)
        arr = (C.c_double * table.size)(*table.reshape(-1).tolist())
        _lib.check(self.lib.lapf_sampler_set_priors(self._h, arr, _stream_ptr(self.domain.device)))

    def priors(self):
        """[F, P, 4] float64 device tensor: the table as given, {lo, hi, mu, sigma}."""
        dev = self.domain.device
        out = torch.empty((self.domain.n_frames, self.nparam, 4), dtype=torch.float64, device=dev)
        _lib.check(self.lib.lapf_sampler_priors(self._h, out.data_ptr(), _stream_ptr(dev)))
        return out

    def rows_recorded(self) -> int:
        """Chain rows every walker has recorded since the last reset."""
        n = self.count
        if n < self.burn_in or n < 1:
            return 0
        return (n - self.burn_in) // self.thin + (1 if self.burn_in > 0 else 0)

    # -- the loop ------------------------------------------------------------------------
    @property
    def count(self) -> int:
        return int(self.lib.lapf_sampler_count(self._h))

    @property
    def launches(self) -> int:
        return int(self.lib.lapf_sampler_launches(self._h))

    def rows_for(self, n_updates: int) -> int:
        return int(_lib.check(self.lib.lapf_sampler_rows_for(self._h, int(n_updates))))

    def chain_bytes(self, n_updates: int) -> int:
        """Bytes the next ``run(n_updates)`` records in the current chain format."""
        return int(_lib.check(self.lib.lapf_sampler_chain_bytes(self._h, int(n_updates))))

    def run(self, n_updates: int, record=True, out=None):
        """Advance all walkers by ``n_updates`` updates.  Returns the chain rows recorded by this
        call as a device tensor [rows, n_walkers, P+1] (float64, or float32 differences from
        ``start()`` after ``set_chain_format('f32delta')``; None when record is False).  In an event
        format: (device uint8 tensor of ``chain_bytes(n_updates)`` bytes, rows)."""
        rows = self.rows_for(n_updates)
        if self.events:
            return self._run_events(n_updates, rows, record, out)
        chain = None
        if record:
            if out is not None:
                if out.dtype != self.chain_dtype or out.numel() < rows * self.n_walkers * (self.nparam + 1):
                    raise ValueError("out must be %s and hold %d rows" % (self.chain_dtype, rows))
                chain = out
            else:
                chain = torch.empty((rows, self.n_walkers, self.nparam + 1), dtype=self.chain_dtype,
                                    device=self.domain.device)
        _lib.check(self.lib.lapf_sampler_run(self._h, int(n_updates),
                                             chain.data_ptr() if chain is not None and rows > 0 else None,
                                             rows, _stream_ptr(self.domain.device)))
        if chain is not None and out is not None:
            return chain.reshape(-1)[: rows * self.n_walkers * (self.nparam + 1)].view(
                rows, self.n_walkers, self.nparam + 1)
        return chain

    def _run_events(self, n_updates, rows, record, out):
        nbytes = self.chain_bytes(n_updates)
        buf = None
        if record:
            if out is not None:
                if out.dtype != torch.uint8 or out.numel() < nbytes:
                    raise ValueError("out must be uint8 and hold %d bytes" % nbytes)
                buf = out.reshape(-1)[:nbytes]
            else:
                buf = torch.empty(nbytes, dtype=torch.uint8, device=self.domain.device)
        _lib.check(self.lib.lapf_sampler_run(self._h, int(n_updates), buf.data_ptr() if buf is not None and rows > 0 else None,
                                             rows, _stream_ptr(self.domain.device)))
        return None if buf is None else (buf, rows)

    def state(self):
        """(state [W, P+1], tries [W, P], accepts [W, P]) device tensors: parameters + chi-square,
        total_tries and total_accept of apf_step2.py:276."""
        dev = self.domain.device
        st = torch.empty((self.n_walkers, self.nparam + 1), dtype=torch.float64, device=dev)
        tr = torch.empty((self.n_walkers, self.nparam), dtype=torch.int32, device=dev)
        ac = torch.empty_like(tr)
        _lib.check(self.lib.lapf_sampler_state(self._h, st.data_ptr(), tr.data_ptr(), ac.data_ptr(),
                                               _stream_ptr(dev)))
        return st, tr, ac

    def stats(self, moments=True):
        """Batch statistics reduced on the device (K4).  Returns a dict of device tensors:
        tries[P], accepts[P], min_tries (scalar), exps (scalar: component evaluations, pixels x Gaussian components, really done),
        moments [F, P+1, 4] (reference, sum of centred chain means, of their squares, of chain
        variances), walkers_per_frame [F], rows (scalar)."""
        dev = self.domain.device
        pn, nf = self.nparam, self.domain.n_frames
        tot = torch.empty((2 * pn + 2,), dtype=torch.int64, device=dev)
        mom = torch.empty((nf, pn + 1, 4), dtype=torch.float64, device=dev) if moments else None
        cnt = torch.empty((nf + 1,), dtype=torch.int64, device=dev)
        _lib.check(self.lib.lapf_sampler_stats(self._h, tot.data_ptr(),
                                               mom.data_ptr() if mom is not None else None,
                                               cnt.data_ptr(), _stream_ptr(dev)))
        return {"tries": tot[:pn], "accepts": tot[pn:2 * pn], "min_tries": tot[2 * pn], "exps": tot[2 * pn + 1],
                "moments": mom, "walkers_per_frame": cnt[:nf], "rows": cnt[nf]}


class ChainStreamer:
    """Double-buffered chain output (K3): while the GPU computes segment i+1 into one device
    buffer, segment i travels to pinned host memory on a copy stream and is handed to the caller.
    Replaces the reference's in-memory hstack + whole-file rewrite (apf_step2.py:346-360).

        streamer = ChainStreamer(sampler, max_updates_per_segment)
        seg = streamer.run(n)      # launches n updates; returns the PREVIOUS segment (numpy) or None
        seg = streamer.finish()    # the last segment

    A segment is the rows [rows, W, P+1] of the sampler's chain format, or in an event format the
    tuple (uint8 event buffer, rows) for ``chains.decode_events``.  Buffers are sized in bytes
    (``GibbsSampler.chain_bytes``) and grow if a later segment needs more.
    """

    def __init__(self, sampler: GibbsSampler, max_updates: int):
        self.s = sampler
        self.max_updates = int(max_updates)
        cap = max(16, sampler.chain_bytes(self.max_updates))
        self.dev = [self._device_buffer(cap) for _ in range(2)]
        self.host = [self._host_buffer(cap) for _ in range(2)]
        self.copy_stream = torch.cuda.Stream(device=sampler.domain.device)
        self.done = [torch.cuda.Event(), torch.cuda.Event()]
        self.pending = None          # (buffer index, rows, bytes)
        self.i = 0

    def _device_buffer(self, nbytes):
        return torch.empty(-(-nbytes // 8) * 8, dtype=torch.uint8, device=self.s.domain.device)

    def _host_buffer(self, nbytes):
        return torch.empty(-(-nbytes // 8) * 8, dtype=torch.uint8).pin_memory()

    def _collect(self):
        if self.pending is None:
            return None
        j, rows, nbytes = self.pending
        self.pending = None
        self.done[j].synchronize()
        raw = self.host[j][:nbytes].numpy()
        if self.s.events:
            return raw, rows
        dt = np.float32 if self.s.chain_dtype == torch.float32 else np.float64
        return raw.view(dt).reshape(rows, self.s.n_walkers, self.s.nparam + 1)

    def run(self, n_updates: int):
        if n_updates > self.max_updates:
            raise ValueError("segment longer than the streamer was sized for")
        s, i = self.s, self.i
        compute = torch.cuda.current_stream(s.domain.device)
        compute.wait_event(self.done[i])            # the copy out of dev[i] two segments ago is finished
        nbytes = s.chain_bytes(n_updates)
        if nbytes > self.dev[i].numel():            # host[i] was collected by the previous call
            self.dev[i], self.host[i] = self._device_buffer(nbytes), self._host_buffer(nbytes)
        if s.events:
            _, rows = s.run(n_updates, out=self.dev[i])
        else:
            rows = int(s.run(n_updates, out=self.dev[i].view(s.chain_dtype)).shape[0])
        if nbytes:
            _lib.check(s.lib.lapf_chain_drain(self.dev[i].data_ptr(), self.host[i].data_ptr(), nbytes,
                                              compute.cuda_stream, self.copy_stream.cuda_stream))
        self.done[i].record(self.copy_stream)
        prev = self._collect()                      # overlaps with the segment just launched
        self.pending = (i, rows, nbytes)
        self.i = 1 - i
        return prev

    def finish(self):
        return self._collect()
