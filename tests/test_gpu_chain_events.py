"""Chain events on the device (LAPF_CHAIN_EVENTS_*, include/lapf.h): the same seed through a dense
chain format and the event format of the same precision; the decoded events must be the dense rows
byte for byte, and the codes a trace of every update."""
import math
import os

import numpy as np
import pytest

from oracle import lapf_oracle as orc

pytestmark = pytest.mark.gpu

HEADER = {"itime": 1.0, "coadds": 1, "multisam": 1, "sampmode": 2}
PRECISIONS = [("f64", "events_f64", np.float64), ("f32delta", "events_f32delta", np.float32)]


@pytest.fixture(scope="module")
def gpu():
    import torch
    from olpefit_b200 import chains, frame, sampler, synth
    assert torch.cuda.is_available()
    return {"torch": torch, "chains": chains, "frame": frame, "sampler": sampler, "synth": synth}


def _setup(gpu, nbody, size, n_frames=1):
    synth = gpu["synth"]
    stamps, origins = synth.make_stamps(n_frames, size, nbody)
    dom = gpu["frame"].prepare_domain(stamps, HEADER, origin=origins, nbody=nbody)
    guess = synth.step1_guess(stamps[0], nbody, origin=tuple(origins[0]))
    p0 = gpu["frame"].initial_parameters(stamps[0], guess, nbody, origin=tuple(origins[0]))
    return dom, stamps, origins, p0


def _decode(gpu, out, s, dtype):
    """Dense rows of what ``s.run`` returned in an event format."""
    buf, rows = out
    assert buf.dtype == gpu["torch"].uint8
    return gpu["chains"].decode_events(buf.cpu().numpy(), rows, s.n_walkers, s.nparam + 1, dtype)


def _both(gpu, dom, init, frame_of, runs, dense_fmt, ev_fmt, dtype, sketch=False, **kw):
    """Rows of the dense format and decoded rows of the event format for the same runs, and the
    two samplers' (state, stats, sketch) after them."""
    res = []
    for fmt in (dense_fmt, ev_fmt):
        with gpu["sampler"].GibbsSampler(dom, init, frame_of, **kw) as s:
            if sketch:
                s.enable_sketch(n_bins=512, sep_bin=1e-3, pa_bin=5e-3)
            s.set_chain_format(fmt)
            parts = []
            for n in runs:
                nbytes = s.chain_bytes(n)
                out = s.run(n)
                if fmt == ev_fmt:
                    assert out[0].numel() == nbytes
                    parts.append(_decode(gpu, out, s, dtype))
                else:
                    assert out.numel() * out.element_size() == nbytes
                    parts.append(out.cpu().numpy())
            after = [t.cpu().numpy() for t in s.state()]
            stats = {k: v.cpu().numpy() for k, v in s.stats().items()}
            sk = {k: v.cpu().numpy() for k, v in s.sketch().items() if k in ("hist", "summary")} if sketch else {}
        res.append((np.concatenate(parts), after, stats, sk))
    return res


def _assert_same(dense, events):
    rows_d, st_d, stats_d, sk_d = dense
    rows_e, st_e, stats_e, sk_e = events
    assert rows_d.dtype == rows_e.dtype and rows_d.shape == rows_e.shape
    assert rows_d.tobytes() == rows_e.tobytes()
    for x, y in zip(st_d, st_e):
        assert x.tobytes() == y.tobytes()
    for k in stats_d:
        assert stats_d[k].tobytes() == stats_e[k].tobytes(), k
    for k in sk_d:
        assert sk_d[k].tobytes() == sk_e[k].tobytes(), k


# walkers per CTA item of the batched kernel, as in test_full_size_batch_state_is_consistent_with_k1
@pytest.mark.parametrize("nbody,size,walkers,frames,n_upd", [
    (2, 64, 65536, 100, 12),
    (2, 32, 148 * (2 * 512 + 37), 5, 8),
    (3, 32, 148 * (2 * 512 + 37), 5, 8),
    (3, 64, 148 * (512 + 37), 3, 8),
    (2, 128, 148 * (192 + 29), 3, 6),
    (3, 128, 148 * (144 + 29), 3, 6),
])
def test_events_equal_dense_rows_at_full_occupancy(gpu, nbody, size, walkers, frames, n_upd):
    stamps, origins = gpu["synth"].make_stamps(frames, size, nbody)
    dom = gpu["frame"].prepare_domain(stamps, HEADER, origin=origins, nbody=nbody)
    frame_of = (np.arange(walkers) % frames).astype(np.int32)
    init = np.array([gpu["synth"].truth_parameters(nbody, f) for f in range(frames)])[frame_of]
    for dense_fmt, ev_fmt, dt in PRECISIONS:
        d, e = _both(gpu, dom, init, frame_of, [n_upd], dense_fmt, ev_fmt, dt, seed=31, burn_in=0, thin=1)
        assert d[0].shape == (n_upd, walkers, 3 * nbody + 11)
        _assert_same(d, e)


@pytest.mark.parametrize("nbody,size,team", [(2, 64, 4), (2, 64, 16), (3, 128, 4), (2, 128, 16), (2, 32, 4)])
def test_events_equal_dense_rows_in_team_kernels(gpu, nbody, size, team):
    dom, _, _, p0 = _setup(gpu, nbody, size)
    init = np.tile(p0, (5, 1))
    for dense_fmt, ev_fmt, dt in PRECISIONS:
        d, e = _both(gpu, dom, init, None, [40, 25], dense_fmt, ev_fmt, dt, seed=7, burn_in=0, thin=1, team_warps=team)
        _assert_same(d, e)


@pytest.mark.parametrize("team", [1, 4])
def test_events_with_burn_in_split_runs_and_sketches(gpu, team):
    """burn-in ending inside a run, runs of 7 + 13 + 30 updates against one of 50, and the device
    sketches and moments: all bitwise the dense run's."""
    dom, _, _, p0 = _setup(gpu, 2, 32, n_frames=3)
    walkers = 37 if team == 1 else 6
    frame_of = (np.arange(walkers) % 3).astype(np.int32)
    init = np.array([gpu["synth"].truth_parameters(2, f) for f in range(3)])[frame_of]
    for dense_fmt, ev_fmt, dt in PRECISIONS:
        whole = _both(gpu, dom, init, frame_of, [50], dense_fmt, ev_fmt, dt, sketch=True,
                      seed=77, burn_in=10, thin=1, team_warps=team)
        parts = _both(gpu, dom, init, frame_of, [7, 13, 30], dense_fmt, ev_fmt, dt, sketch=True,
                      seed=77, burn_in=10, thin=1, team_warps=team)
        assert whole[0][0].shape[0] == 41
        _assert_same(*whole)
        _assert_same(*parts)
        _assert_same(whole[1], parts[1])


def test_event_buffers_are_deterministic_and_survive_checkpoints(gpu):
    torch = gpu["torch"]
    dom, _, _, p0 = _setup(gpu, 2, 64)
    walkers = 301                          # rows x walkers not a multiple of 16: the codes are padded
    init = np.tile(p0, (walkers, 1))
    kw = dict(seed=5, burn_in=0, thin=1)
    bufs = []
    for _ in range(2):
        with gpu["sampler"].GibbsSampler(dom, init, **kw) as s:
            s.set_chain_format("events_f32delta")
            torch.cuda.synchronize()
            junk = torch.full((s.chain_bytes(21),), 0xA5, dtype=torch.uint8, device=s.domain.device)
            buf, rows = s.run(21, out=junk)
            bufs.append(buf.cpu().numpy().copy())
    assert rows == 21 and np.array_equal(bufs[0], bufs[1])
    with gpu["sampler"].GibbsSampler(dom, init, **kw) as s:
        s.set_chain_format("events_f64")
        full = _decode(gpu, s.run(50), s, np.float64)
    with gpu["sampler"].GibbsSampler(dom, init, **kw) as a:
        a.set_chain_format("events_f64")
        first = _decode(gpu, a.run(20), a, np.float64)
        blob = a.save()
    with gpu["sampler"].GibbsSampler(dom, np.tile(p0 * 1.01, (walkers, 1)), seed=99, burn_in=0, thin=1) as b:
        b.load(blob)
        b.set_chain_format("events_f64")
        second = _decode(gpu, b.run(30), b, np.float64)
    assert np.concatenate([first, second]).tobytes() == full.tobytes()


def test_chain_streamer_moves_events(gpu):
    dom, _, _, p0 = _setup(gpu, 2, 32, n_frames=2)
    walkers = 600
    frame_of = (np.arange(walkers) % 2).astype(np.int32)
    init = np.tile(p0, (walkers, 1))
    for dense_fmt, ev_fmt, dt in PRECISIONS:
        out = {}
        for fmt in (dense_fmt, ev_fmt):
            with gpu["sampler"].GibbsSampler(dom, init, frame_of, seed=17, burn_in=5, thin=1) as s:
                s.set_chain_format(fmt)
                st = gpu["sampler"].ChainStreamer(s, 20)
                # a segment lives in a pinned buffer that a later call reuses: keep a copy
                keep = lambda x: x if x is None else ((x[0].copy(), x[1]) if isinstance(x, tuple) else x.copy())  # noqa: E731
                segs = [keep(st.run(n)) for n in (4, 20, 20, 13)] + [keep(st.finish())]
                assert segs[0] is None
                if fmt == ev_fmt:
                    segs = [gpu["chains"].decode_events(b, r, walkers, 17, dt) for b, r in segs[1:]]
                out[fmt] = np.concatenate([x for x in segs if x is not None])
        assert out[dense_fmt].shape == (53, walkers, 17)
        assert out[dense_fmt].tobytes() == out[ev_fmt].tobytes()


def test_event_codes_count_tries_and_accepts(gpu):
    """With burn_in = 0 every update is a row: the codes are the complete trace, so per walker and
    parameter they count exactly what the device counters say; a negative log-parameter start yields
    rejected codes only for that parameter."""
    dom, _, _, p0 = _setup(gpu, 2, 32)
    walkers, n_upd, P = 70, 120, 16
    init = np.tile(p0, (walkers, 1))
    init[::7, 7] = -5.0                    # companion amplitude (log10-proposed) negative: never accepted
    with gpu["sampler"].GibbsSampler(dom, init, seed=3, burn_in=0, thin=1) as s:
        s.set_chain_format("events_f64")
        buf, rows = s.run(n_upd)
        _, tries, accepts = (t.cpu().numpy() for t in s.state())
    codes = buf.cpu().numpy()[walkers * 17 * 8:][:rows * walkers].reshape(rows, walkers)
    k, acc = codes & 31, (codes >> 7).astype(bool)
    assert np.all((codes & 0x60) == 0) and k.max() < P
    for w in range(walkers):
        assert np.array_equal(np.bincount(k[:, w], minlength=P), tries[w])
        assert np.array_equal(np.bincount(k[acc[:, w], w], minlength=P), accepts[w])
    neg = np.arange(0, walkers, 7)
    assert tries[neg, 7].sum() > 0 and not acc[:, neg][k[:, neg] == 7].any()
    assert acc[:, neg].any()


def test_decoded_events_replay_the_oracle_with_dense_warps(gpu):
    """The oracle replay of test_dense_warps_replay_oracle_stream from rows rebuilt from events."""
    nbody, size, walkers = 2, 64, 600
    lay = orc.layout_for(nbody)
    dom, stamps, origins, p0 = _setup(gpu, nbody, size)
    n_upd, seed = 160, 4321
    init = np.tile(p0, (walkers, 1))
    with gpu["sampler"].GibbsSampler(dom, init, seed=seed, burn_in=0, thin=1, id_base=11, id_stride=2) as s:
        s.set_chain_format("events_f64")
        chain = _decode(gpu, s.run(n_upd), s, np.float64)
        _, tries, accepts = (t.cpu().numpy() for t in s.state())
    img = stamps[0].astype(np.float64)
    w = orc.weight_map(img, HEADER)
    early = 0
    picks = [0, 1, 15, 16, 17, 259, 511, 512, 517, walkers - 1]
    for wi in picks:
        gid = 11 + 2 * wi
        res = orc.run_chain(img, w, lay, p0, orc.PhiloxStream(seed, gid, lay.nparam), origin=tuple(origins[0]),
                            n_updates=n_upd, burn_in=0, record_trace=True)
        ref, dev = res.rows[1:], chain[:, wi, :]
        same = np.all(np.isclose(dev[:, :-1], ref[:, :-1], rtol=1e-9, atol=1e-12), axis=1)
        first_bad = int(np.argmin(same)) if not same.all() else n_upd
        np.testing.assert_allclose(dev[:first_bad, -1], ref[:first_bad, -1], rtol=1e-5)
        if first_bad == n_upd:
            assert np.array_equal(tries[wi], res.tries) and np.array_equal(accepts[wi], res.accepts)
            continue
        k, new, chi_t, ok = res.trace[first_bad]
        chi_c = ref[first_bad - 1, -1] if first_bad > 0 else orc.chi_squared_weighted(
            img, orc.model_image(p0, lay, size, size, origin=tuple(origins[0])), w)
        u = orc.device_draws(seed, gid, first_bad, lay.nparam)[2]
        margin = abs(math.log(u) + 0.5 * (chi_t - chi_c))
        assert margin <= 0.5 * 1e-5 * (abs(chi_t) + abs(chi_c)), (wi, first_bad, margin)
        early += first_bad < 80
    assert early <= 2


def test_event_formats_need_thin_1(gpu):
    from olpefit_b200 import _lib
    dom, _, _, p0 = _setup(gpu, 2, 32)
    with gpu["sampler"].GibbsSampler(dom, p0[None], seed=1, thin=4) as s:
        for fmt in ("events_f64", "events_f32delta"):
            with pytest.raises(_lib.LapfError, match="error -1"):
                s.set_chain_format(fmt)
        assert s.chain_bytes(8) == 2 * 17 * 8          # the dense format is still in force
        s.set_chain_format("f32delta")
        assert s.chain_bytes(8) == 2 * 17 * 4


def _write_case(tmp_path, tag):
    from olpefit_b200 import frame, synth
    d = tmp_path / ("case%s" % tag)
    d.mkdir()
    img, _ = synth.make_frame(0, 2)
    path = str(d / "N2.20090531.29966.LDIF.fits")
    frame.write_fits(path, img, synth.HEADER)
    with open(str(d / "29966_initialguess"), "w") as fh:
        fh.write(" ".join(str(v) for v in synth.step1_guess(img, 2, sky_xy=(100, 120))) + "\n")
    return path, str(d / "29966_apf_results")


def _read(p):
    with open(p, "rb") as fh:
        return fh.read()


def test_cli_event_file_unpacks_to_the_csv_files_and_resumes(tmp_path):
    from olpefit_b200 import chains, cli
    common = ["--walkers", "4", "--burn-in", "0", "--seed", "21", "--stamp", "32", "--segment", "64", "--quiet"]
    path_c, out_c = _write_case(tmp_path, "_csv")
    assert cli.main_step2([path_c, "--accept-min", "24"] + common) == 0
    path_e, out_e = _write_case(tmp_path, "_events")
    assert cli.main_step2([path_e, "--accept-min", "24", "--format", "events"] + common) == 0
    base = os.path.join(out_e, "chains_rank0")
    assert os.path.exists(base + ".events") and not os.path.exists(base + ".bin")
    assert chains.unpack_to_csv(base, os.path.join(out_e, "csv")) == 4
    for w in range(4):
        assert _read(os.path.join(out_e, "csv", "%d_finalarray_mpi.csv" % w)) == _read(
            os.path.join(out_c, "%d_finalarray_mpi.csv" % w))
    # interrupted and resumed: what the uninterrupted run writes
    for dtype in ("f64", "f32"):
        extra = ["--format", "events", "--chain-dtype", dtype]
        path_w, out_w = _write_case(tmp_path, "_whole_" + dtype)
        assert cli.main_step2([path_w, "--accept-min", "24"] + common + extra) == 0
        whole, meta = chains.read_packed(os.path.join(out_w, "chains_rank0"))
        path_p, out_p = _write_case(tmp_path, "_parts_" + dtype)
        assert cli.main_step2([path_p, "--accept-min", "9", "--checkpoint"] + common + extra) == 0
        part, _ = chains.read_packed(os.path.join(out_p, "chains_rank0"))
        assert 0 < part.shape[0] < whole.shape[0]
        assert cli.main_step2([path_p, "--accept-min", "24", "--resume"] + common + extra) == 0
        both, meta_b = chains.read_packed(os.path.join(out_p, "chains_rank0"))
        assert meta_b["count"] == meta["count"] and meta_b["format"] == "events"
        assert both.shape == whole.shape and both.tobytes() == whole.tobytes()
    with pytest.raises(SystemExit):
        cli.main_step2([path_c, "--format", "events", "--thin", "4"] + common)
