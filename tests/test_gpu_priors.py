"""Parameter priors on the device (lapf_sampler_set_priors / lapf_sampler_priors, include/lapf.h): a neutral
table changes nothing the sampler computes; with boxes and Gaussian terms the chains follow the oracle loop
with the numpy restatement of test_priors in its accept rule; boxes hold for every row, draw and state and
skip the pass in the batched kernel; narrow Gaussian and truncating priors give the expected posteriors;
the self-test marks exactly the box-skipped probes; checkpoints, reset and refusals behave as documented;
and the command line's --prior."""
import json
import os

import numpy as np
import pytest

from oracle import lapf_oracle as orc
from test_gpu_frame_widths import _write_scaled_epochs
from test_priors import outside, run_chain_with_prior

pytestmark = pytest.mark.gpu

HEADER = {"itime": 1.0, "coadds": 1, "multisam": 1, "sampmode": 2}


@pytest.fixture(scope="module")
def gpu():
    import torch
    from olpefit_b200 import _lib, chains, frame, layout, sampler, synth
    assert torch.cuda.is_available()
    return {"torch": torch, "frame": frame, "sampler": sampler, "synth": synth, "lib": _lib, "chains": chains,
            "layout": layout}


def _domain(gpu, nbody, size, n_frames):
    synth = gpu["synth"]
    stamps, origins = synth.make_stamps(n_frames, size, nbody)
    dom = gpu["frame"].prepare_domain(stamps, HEADER, origin=origins, nbody=nbody)
    p_frame = np.array([synth.truth_parameters(nbody, f) for f in range(n_frames)])
    return dom, p_frame, stamps, origins


def _neutral(F, P):
    return np.tile([-np.inf, np.inf, 0.0, np.inf], (F, P, 1))


def _set(s, table):
    s.set_priors(table[..., 0], table[..., 1], table[..., 2], table[..., 3])


def _run(gpu, dom, init, frame_of, runs, *, prior=None, fmt="f64", team=0, burn_in=0, thin=1, seed=7, widths=None,
         extras=True, id_base=0):
    """``prior``: None (off) or an [F, P, 4] table.  Returns (rows or None, everything else as numpy)."""
    torch, chains = gpu["torch"], gpu["chains"]
    out = {}
    with gpu["sampler"].GibbsSampler(dom, init, frame_of, seed=seed, burn_in=burn_in, thin=thin, team_warps=team,
                                     widths=widths, id_base=id_base) as s:
        if extras:
            s.enable_sketch(n_bins=512, sep_bin=1e-3, pa_bin=5e-3)
            s.enable_batch_means(5, 3)
            s.enable_draws(7)
            s.set_frame_widths()
        if prior is not None:
            _set(s, prior)
        if fmt is not None:
            s.set_chain_format(fmt)
        parts = []
        for n in runs:
            r = s.run(n, record=fmt is not None)
            if fmt is not None and not s.events:
                parts.append(r.cpu().numpy())
            elif fmt is not None:
                parts.append(chains.decode_events(r[0].cpu().numpy(), r[1], s.n_walkers, s.nparam + 1, np.float64))
        st, tr, ac = s.state()
        out["state"], out["tries"], out["accepts"] = st.cpu().numpy(), tr.cpu().numpy(), ac.cpu().numpy()
        stt = s.stats()
        out["moments"], out["exps"] = stt["moments"].cpu().numpy(), int(stt["exps"].item())
        if extras:
            sk = s.sketch()
            out["hist"], out["summary"] = sk["hist"].cpu().numpy(), sk["summary"].cpu().numpy()
            bm = s.batch_means()
            out["bm_walker"], out["bm_frame"] = bm["walker"].cpu().numpy(), bm["frame"].cpu().numpy()
            d = s.draws()
            out["draws"], out["draw_rows"] = d["values"].cpu().numpy(), d["rows"].cpu().numpy()
        if prior is not None:
            out["prior"] = s.priors().cpu().numpy()
        torch.cuda.synchronize()
    return (np.concatenate(parts) if parts else None), out


def _same(a, b):
    for key in [k for k in a if k in b and k != "prior"]:
        np.testing.assert_array_equal(np.atleast_1d(a[key]).view(np.uint8), np.atleast_1d(b[key]).view(np.uint8), err_msg=key)


# -- a neutral table is no table ----------------------------------------------------------------------
# the occupancy of test_gpu_frame_widths.test_full_size_table_of_batch_widths_is_the_parent
@pytest.mark.parametrize("nbody,size,walkers,frames,n_upd", [
    (2, 64, 65536, 100, 48),
    (2, 32, 148 * (2 * 512 + 37), 5, 32),
    (3, 32, 148 * (2 * 512 + 37), 5, 32),
    (3, 64, 148 * (512 + 37), 3, 32),
    (2, 128, 148 * (192 + 29), 3, 16),
    (3, 128, 148 * (144 + 29), 3, 16),
])
def test_full_size_neutral_table_is_no_table(gpu, nbody, size, walkers, frames, n_upd):
    dom, p_frame, _, _ = _domain(gpu, nbody, size, frames)
    frame_of = np.arange(walkers) % frames
    init = p_frame[frame_of]
    P = p_frame.shape[1]
    rows0, off = _run(gpu, dom, init, frame_of, [n_upd], burn_in=3)
    rows1, on = _run(gpu, dom, init, frame_of, [n_upd], prior=_neutral(frames, P), burn_in=3)
    np.testing.assert_array_equal(rows0.view(np.int64), rows1.view(np.int64))
    _same(off, on)
    rows2, ev = _run(gpu, dom, init, frame_of, [n_upd // 2, n_upd - n_upd // 2], prior=_neutral(frames, P),
                     fmt="events_f64", burn_in=3)
    np.testing.assert_array_equal(rows0.view(np.int64), rows2.view(np.int64))
    _same(off, ev)
    np.testing.assert_array_equal(on["prior"], _neutral(frames, P))


@pytest.mark.parametrize("team,nbody,size", [(4, 2, 64), (4, 3, 32), (16, 2, 128), (16, 3, 64)])
def test_team_kernels_neutral_table_is_no_table(gpu, team, nbody, size):
    dom, p_frame, _, _ = _domain(gpu, nbody, size, 2)
    frame_of = np.arange(24) % 2
    P = p_frame.shape[1]
    rows0, off = _run(gpu, dom, p_frame[frame_of], frame_of, [70, 41], team=team, burn_in=2)
    rows1, on = _run(gpu, dom, p_frame[frame_of], frame_of, [70, 41], team=team, burn_in=2, prior=_neutral(2, P))
    np.testing.assert_array_equal(rows0.view(np.int64), rows1.view(np.int64))
    _same(off, on)
    rows2, ev = _run(gpu, dom, p_frame[frame_of], frame_of, [111], team=team, burn_in=2, prior=_neutral(2, P),
                     fmt="events_f64")
    np.testing.assert_array_equal(rows0.view(np.int64), rows2.view(np.int64))
    _same(off, ev)


# -- boxes and Gaussian terms -------------------------------------------------------------------------------
def _cutting_table(p_frame, nbody):
    """Boxes around each frame's start that cut through the posterior (a few jump widths wide) on the positions,
    ampratio and a shape parameter, and Gaussian terms on three more; the start lies inside every box."""
    from olpefit_b200 import layout
    F, P = p_frame.shape
    t = _neutral(F, P)
    names = list(layout.names(nbody))
    w, _ = layout.default_widths(nbody)
    for f in range(F):
        p = p_frame[f]
        # the first object's x, the second's y (names[0], names[3]), dx, ampratio
        for j, lo, hi in ((0, -2.0, 1.0), (3, -1.0, 1.5), (names.index("dx"), -3.0, 2.0), (names.index("ampratio"), -2.0, 2.0)):
            t[f, j, :2] = p[j] + lo * w[j], p[j] + hi * w[j]
        j = names.index("sigmax")                                   # a log10-proposed parameter: a relative box
        t[f, j, :2] = p[j] * 10 ** (-2 * w[j]), p[j] * 10 ** (1.5 * w[j])
        for j, dmu, sg in ((1, 0.5, 1.0), (names.index("theta"), 0.3, 2.0), (names.index("sigmay"), 0.4, 1.5)):
            t[f, j, 2:] = p[j] + dmu * w[j] * max(abs(p[j]), 1.0), sg * w[j] * max(abs(p[j]), 1.0)
    return t


def _replay(gpu, rows, tries, accepts, stamps, origins, p_frame, frame_of, table, seed, picks, nbody, n_upd, id_base=0):
    lay = orc.layout_for(nbody)
    for wi in picks:
        f = int(frame_of[wi])
        img = stamps[f].astype(np.float64)
        ref, rt, ra, trace = run_chain_with_prior(img, orc.weight_map(img, HEADER), lay, p_frame[f],
                                                  orc.PhiloxStream(seed, id_base + wi, lay.nparam), table[f],
                                                  origin=tuple(origins[f]), n_updates=n_upd)
        dev = rows[:, wi]
        same = np.all(np.isclose(dev[:, :-1], ref[:, :-1], rtol=1e-9, atol=1e-12), axis=1)
        first_bad = int(np.argmin(same)) if not same.all() else n_upd
        # as in smoke(): FP32 chi-square may flip a borderline accept late, never early
        assert first_bad >= 24, (wi, first_bad, trace[first_bad] if first_bad < n_upd else None)
        np.testing.assert_allclose(dev[:first_bad, -1], ref[:first_bad, -1], rtol=1e-5)
        if first_bad == n_upd:
            np.testing.assert_array_equal(tries[wi], rt)
            np.testing.assert_array_equal(accepts[wi], ra)
        assert sum(1 for k, new, *_ in trace if outside(table[f][k], new)) > 0      # the boxes did cut


@pytest.mark.parametrize("nbody,size,walkers,team", [(2, 64, 600, 0), (2, 32, 600, 0), (2, 128, 24, 16)])
def test_boxes_and_gaussian_terms_replay_the_oracle(gpu, nbody, size, walkers, team):
    dom, p_frame, stamps, origins = _domain(gpu, nbody, size, 2)
    frame_of = np.arange(walkers) % 2
    table = _cutting_table(p_frame, nbody)
    n_upd, seed = 96, 4321
    rows, res = _run(gpu, dom, p_frame[frame_of], frame_of, [n_upd], prior=table, team=team, seed=seed, extras=False)
    picks = sorted({w for w in (0, 1, 2, 31, 32, walkers // 2 + 1, walkers - 1) if w < walkers})
    _replay(gpu, rows, res["tries"], res["accepts"], stamps, origins, p_frame, frame_of, table, seed, picks, nbody, n_upd)


@pytest.mark.parametrize("nbody,size,team", [(2, 64, 0), (3, 32, 0), (2, 128, 0), (2, 64, 4)])
def test_every_row_draw_and_state_lies_inside_the_box(gpu, nbody, size, team):
    dom, p_frame, _, _ = _domain(gpu, nbody, size, 2)
    walkers = 900 if team == 0 else 24
    frame_of = np.arange(walkers) % 2
    table = _cutting_table(p_frame, nbody)
    rows, res = _run(gpu, dom, p_frame[frame_of], frame_of, [150, 77], prior=table, team=team, burn_in=10)
    lo, hi = table[frame_of, :, 0], table[frame_of, :, 1]
    assert np.all((rows[..., :-1] >= lo) & (rows[..., :-1] <= hi))
    st = res["state"][:, :-1]
    assert np.all((st >= lo) & (st <= hi))
    d, dr = res["draws"][..., :-1], res["draw_rows"]
    filled = dr >= 0
    assert filled.all()
    assert np.all((d >= lo[:, None]) & (d <= hi[:, None]))
    assert res["tries"].sum() == walkers * 227                       # a box rejection is a try ...
    np.testing.assert_array_equal(res["prior"], table)


@pytest.mark.parametrize("nbody,size,team", [(2, 64, 0), (2, 32, 0), (3, 128, 0), (2, 64, 4)])
def test_a_closed_box_rejects_every_proposal_without_a_pass(gpu, nbody, size, team):
    dom, p_frame, _, _ = _domain(gpu, nbody, size, 2)
    walkers = 500 if team == 0 else 8
    frame_of = np.arange(walkers) % 2
    table = _neutral(2, p_frame.shape[1])
    table[..., 0] = p_frame
    table[..., 1] = p_frame                                          # lo = hi = the start: every proposal is outside
    rows, res = _run(gpu, dom, p_frame[frame_of], frame_of, [64], prior=table, team=team, extras=False)
    assert res["tries"].sum() == walkers * 64 and res["accepts"].sum() == 0   # tries, never accepts
    np.testing.assert_array_equal(rows[..., :-1], np.broadcast_to(p_frame[frame_of], rows[..., :-1].shape))
    if team == 0:
        assert res["exps"] == 0                                      # the batched kernel skipped every pass
    else:
        assert res["exps"] > 0                                       # the team kernels evaluate and reject


# -- posteriors --------------------------------------------------------------------------------------
def _posterior_rows(gpu, dom, init, j, *, prior=None, widths=None, n=4000, burn=3000, seed=5):
    W = init.shape[0]
    with gpu["sampler"].GibbsSampler(dom, init, np.zeros(W, dtype=np.int32), seed=seed, burn_in=burn, thin=16,
                                     widths=widths) as s:
        if prior is not None:
            _set(s, prior)
        s.run(burn, record=False)
        rows = s.run(n).cpu().numpy()[1:]
    return rows[..., j]                                              # [rows, W]


def _group_mcse(vals, stat, groups=32):
    """stat over all rows, and its Monte Carlo standard error from `groups` groups of whole walkers."""
    parts = [stat(vals[:, g::groups].reshape(-1)) for g in range(groups)]
    return stat(vals.reshape(-1)), float(np.std(parts, ddof=1) / np.sqrt(groups))


def test_narrow_gaussian_and_truncation_give_the_expected_posteriors(gpu):
    from olpefit_b200 import layout
    nbody, size = 2, 64
    dom, p_frame, _, _ = _domain(gpu, nbody, size, 1)
    names = list(layout.names(nbody))
    j = names.index("xcc")
    init = np.tile(p_frame[0], (2048, 1))
    free = _posterior_rows(gpu, dom, init, j)
    m_l, mcse_m = _group_mcse(free, np.mean)
    s_l = float(free.std())
    # a Gaussian prior a fifth of the likelihood's width, centred on its mean: the posterior is the prior
    # (mean mu, std sigma / sqrt(1 + 1/25))
    sg = s_l / 5
    table = _neutral(1, len(names))
    table[0, j, 2:] = m_l, sg
    w, _ = layout.default_widths(nbody)
    w = w.copy()
    w[j] = sg
    narrow = _posterior_rows(gpu, dom, init, j, prior=table, widths=w)
    m_n, mcse_n = _group_mcse(narrow, np.mean)
    assert abs(m_n - m_l) <= 4 * np.hypot(mcse_n, mcse_m / 26), (m_n, m_l, mcse_n)
    assert abs(float(narrow.std()) / sg - 1.0) <= 0.10, (float(narrow.std()), sg)
    # a bound at the free median: the constrained median is the free upper (or lower) quartile
    med = float(np.median(free))
    table = _neutral(1, len(names))
    up = p_frame[0, j] >= med                                        # the start must lie inside the box
    table[0, j, 0 if up else 1] = med
    cut = _posterior_rows(gpu, dom, init, j, prior=table)
    assert np.all(cut >= med) if up else np.all(cut <= med)
    q = 75 if up else 25
    m_c, mcse_c = _group_mcse(cut, np.median)
    q_f, mcse_q = _group_mcse(free, lambda v: np.percentile(v, q))
    assert abs(m_c - q_f) <= 4 * np.hypot(mcse_c, mcse_q), (m_c, q_f, mcse_c, mcse_q)


# -- the self-test ------------------------------------------------------------------------------------
def test_selftest_marks_exactly_the_box_skipped_probes(gpu, tmp_path):
    from olpefit_b200 import layout
    from olpefit_b200.model import _stream_ptr
    nbody, size = 2, 64
    dom, p_frame, _, _ = _domain(gpu, nbody, size, 2)
    W = 700
    frame_of = np.arange(W) % 2
    w, is_log = layout.default_widths(nbody)
    table = _neutral(2, len(w))
    for f in range(2):                                               # boxes that reject about 3/4 of the proposals
        p = p_frame[f]
        a, b = np.where(is_log, p * 10 ** (-0.3 * w), p - 0.3 * w), np.where(is_log, p * 10 ** (0.3 * w), p + 0.3 * w)
        table[f, :, 0], table[f, :, 1] = np.minimum(a, b), np.maximum(a, b)
    dump = str(tmp_path / "selftest.bin")
    with gpu["sampler"].GibbsSampler(dom, p_frame[frame_of], frame_of, seed=9) as s:
        _set(s, table)                                               # runs the self-test with the boxes: no refusal
        os.environ["LAPF_SELFTEST_DUMP"] = dump
        try:
            gpu["lib"].check(s.lib.lapf_sampler_selftest(s._h, _stream_ptr(dom.device)))
        finally:
            del os.environ["LAPF_SELFTEST_DUMP"]
    raw = open(dump, "rb").read()
    U, Wd, P = np.frombuffer(raw[:24], dtype=np.int64)
    body = np.frombuffer(raw[24:], dtype=np.float64)
    n = U * Wd
    probe, chi = body[:3 * n].reshape(U, Wd, 3), body[3 * n:4 * n].reshape(U, Wd)
    kd, nv, chi_t = probe[..., 0], probe[..., 1], probe[..., 2]
    marked = kd < 0
    k = np.where(marked, -1 - kd, kd).astype(int)
    fo = np.broadcast_to(frame_of, (U, Wd))
    lo, hi = table[fo, k, 0], table[fo, k, 1]
    out = ~((nv >= lo) & (nv <= hi))
    np.testing.assert_array_equal(marked, out)
    assert 0.5 < marked.mean() < 0.95, marked.mean()
    np.testing.assert_array_equal(chi_t[~marked].view(np.int64), chi[~marked].view(np.int64))


# -- checkpoints, reset, refusals -----------------------------------------------------------------------
def test_save_and_load_continue_bit_for_bit(gpu):
    dom, p_frame, _, _ = _domain(gpu, 2, 64, 2)
    frame_of = np.arange(600) % 2
    table = _cutting_table(p_frame, 2)
    whole, _ = _run(gpu, dom, p_frame[frame_of], frame_of, [90, 60], prior=table, burn_in=5)
    with gpu["sampler"].GibbsSampler(dom, p_frame[frame_of], frame_of, seed=7, burn_in=5) as s:
        s.enable_sketch(n_bins=512, sep_bin=1e-3, pa_bin=5e-3)
        s.enable_batch_means(5, 3)
        s.enable_draws(7)
        s.set_frame_widths()
        _set(s, table)
        first = s.run(90).cpu().numpy()
        blob = s.save().clone()
    with gpu["sampler"].GibbsSampler(dom, p_frame[frame_of], frame_of, seed=1, burn_in=5) as t:
        t.enable_sketch(n_bins=512, sep_bin=1e-3, pa_bin=5e-3)
        t.enable_batch_means(5, 3)
        t.enable_draws(7)
        t.set_frame_widths()
        _set(t, _neutral(2, 16))
        t.load(blob)
        np.testing.assert_array_equal(t.priors().cpu().numpy(), table)     # the blob's table
        second = t.run(60).cpu().numpy()
    np.testing.assert_array_equal(np.concatenate([first, second]).view(np.int64), whole.view(np.int64))


def _enable(s, opts):
    if "sketch" in opts:
        s.enable_sketch(n_bins=64, sep_bin=1e-3, pa_bin=5e-3)
    if "bm" in opts:
        s.enable_batch_means(5, 2)
    if "draws" in opts:
        s.enable_draws(3)
    if "fw" in opts:
        s.set_frame_widths()


@pytest.mark.parametrize("opts", [(), ("sketch",), ("bm",), ("draws",), ("fw",), ("sketch", "bm", "draws", "fw")])
def test_checkpoints_with_and_without_priors_refuse_each_other(gpu, opts):
    lib = gpu["lib"]
    dom, p_frame, _, _ = _domain(gpu, 2, 32, 2)
    frame_of = np.arange(40) % 2
    init = p_frame[frame_of]
    table = _cutting_table(p_frame, 2)
    blobs = {}
    for on in (False, True):
        with gpu["sampler"].GibbsSampler(dom, init, frame_of, seed=3) as s:
            _enable(s, opts)
            if on:
                _set(s, table)
            s.run(20, record=False)
            blobs[on] = s.save().clone()
    assert blobs[True].numel() == blobs[False].numel() + 32 + 2 * 16 * 4 * 8 * 2
    desc = blobs[True][-(32 + 2 * 16 * 4 * 8 * 2):][:32].cpu().numpy().view(np.int64)
    assert bytes(desc[:1].view(np.uint8)) == b"LAPFPR01" and desc[1:].tolist() == [2, 16, 0]
    for on in (False, True):
        with gpu["sampler"].GibbsSampler(dom, init, frame_of, seed=4) as s:
            _enable(s, opts)
            if on:
                _set(s, table)
            before = s.save().clone()
            with pytest.raises(lib.LapfError):
                s.load(blobs[not on])
            assert gpu["torch"].equal(s.save(), before)               # a refused load changes nothing
            s.load(blobs[on])


def test_reset_keeps_the_table_and_refuses_starts_outside_it(gpu):
    lib, torch = gpu["lib"], gpu["torch"]
    dom, p_frame, _, _ = _domain(gpu, 2, 64, 2)
    frame_of = np.arange(64) % 2
    init = p_frame[frame_of]
    table = _cutting_table(p_frame, 2)
    with gpu["sampler"].GibbsSampler(dom, init, frame_of, seed=3) as s:
        _set(s, table)
        s.run(50, record=False)
        before = s.save().clone()
        bad = init.copy()
        bad[5, 8] = table[1, 8, 1] + 0.5                             # walker 5 (frame 1): ampratio above its box
        with pytest.raises(lib.LapfError, match="frame 1, parameter 8"):
            s.reset(bad, seed=4)
        assert torch.equal(s.save(), before)
        s.reset(init, seed=4)
        np.testing.assert_array_equal(s.priors().cpu().numpy(), table)
        assert s.count == 0
        rows_a = s.run(40).cpu().numpy()
    rows_b, _ = _run(gpu, dom, init, frame_of, [40], prior=table, seed=4, extras=False)
    np.testing.assert_array_equal(rows_a.view(np.int64), rows_b.view(np.int64))


def test_set_priors_refusals(gpu):
    lib, torch = gpu["lib"], gpu["torch"]
    dom, p_frame, _, _ = _domain(gpu, 2, 32, 2)
    frame_of = np.arange(40) % 2
    P = 16
    with gpu["sampler"].GibbsSampler(dom, p_frame[frame_of], frame_of, seed=3) as s:
        with pytest.raises(lib.LapfError):
            s.priors()                                               # no table
        plain = s.save().clone()

        def refused(table, match):
            with pytest.raises(lib.LapfError, match=match):
                _set(s, table)

        for i in range(4):
            t = _neutral(2, P)
            t[1, 3, i] = np.nan
            refused(t, "frame 1, parameter 3 has a nan")
        t = _neutral(2, P)
        t[0, 2, :2] = 5.0, 4.0
        refused(t, "lo 5 > hi 4")
        for sg in (0.0, -1.0, -np.inf):
            t = _neutral(2, P)
            t[1, 4, 3] = sg
            refused(t, "sigma")
        t = _neutral(2, P)
        t[1, 4, 2:] = np.inf, 1.0
        refused(t, "mu inf is not finite")
        t = _neutral(2, P)
        t[1, 4, 3] = 1e-200
        refused(t, "too small")
        t = _neutral(2, P)
        t[1, 8, :2] = p_frame[1, 8] + 0.1, np.inf                    # every walker of frame 1 starts below it
        refused(t, "frame 1, parameter 8")
        with pytest.raises(lib.LapfError):
            s.priors()                                               # nothing was turned on
        assert torch.equal(s.save(), plain)
        t = _cutting_table(p_frame, 2)
        _set(s, t)
        s.run(30, record=False)
        u = t.copy()
        u[0, 0, :2] = p_frame[0, 0] + 1.0, np.inf
        with pytest.raises(lib.LapfError, match="frame 0, parameter 0"):
            _set(s, u)                                               # later calls check the current state too
        np.testing.assert_array_equal(s.priors().cpu().numpy(), t)   # ... and keep the table on refusal
        _set(s, _neutral(2, P))                                      # later calls replace the table
        np.testing.assert_array_equal(s.priors().cpu().numpy(), _neutral(2, P))
        # an infinite box with a Gaussian term of infinite mean is refused only where sigma is finite
        t = _neutral(2, P)
        t[0, 1, 2] = np.inf
        _set(s, t)


# -- the command line ----------------------------------------------------------------------------------
CLI = ["-i", "2a", "--walkers", "8", "--burn-in", "200", "--seed", "29", "--stamp", "64", "--segment", "256", "--quiet"]


def _prior_file(tmp_path, name, p_first, ycc_hi=0.4):
    spec = {"all": {"ampratio": {"min": 0, "max": 1}, "bkgd": {"min": -50.0}, "sigmax2": {"mean": 6.0, "sigma": 0.5}},
            "epochs": {"29960": {"xcc": {"min": p_first[2] - 0.3, "max": p_first[2] + 0.3}},
                       "29962": {"ycc": {"min": -1e9, "max": 1e9 + ycc_hi}}}}
    path = tmp_path / name
    path.write_text(json.dumps(spec))
    return str(path)


def test_cli_prior_writes_summaries_and_every_row_respects_the_boxes(tmp_path):
    from olpefit_b200 import chains, cli, synth
    paths, lst = _write_scaled_epochs(tmp_path, "pr")
    pf = _prior_file(tmp_path, "prior.json", synth.truth_parameters(2, 0))
    assert cli.main_step2([paths[0], "--frames", lst, "--accept-min", "120", "--prior", pf] + CLI) == 0
    table = cli.load_prior_file(pf, 2, ["29960", "29961", "29962"])
    for f, p in enumerate(paths):
        d = chains.results_dir(p)
        summ = json.load(open(d + "step2_summary.json"))
        assert summ["priors"] == cli.prior_summary(table[f], 2)
        assert set(summ["priors"]) == ({"ampratio", "bkgd", "sigmax2", "xcc"} if f == 0 else
                                       {"ampratio", "bkgd", "sigmax2", "ycc"} if f == 2 else {"ampratio", "bkgd", "sigmax2"})
        for w in range(8):
            rows = np.genfromtxt(d + "%d_finalarray_mpi.csv" % w, delimiter=",")[1:, :16]
            assert rows.shape[0] > 0
            assert np.all((rows >= table[f, :, 0]) & (rows <= table[f, :, 1])), (f, w)


def test_cli_prior_resume_needs_the_same_file(tmp_path):
    from olpefit_b200 import chains, cli, synth
    p_first = synth.truth_parameters(2, 0)
    pa, la = _write_scaled_epochs(tmp_path, "whole")
    pf = _prior_file(tmp_path, "prior.json", p_first)
    assert cli.main_step2([pa[0], "--frames", la, "--accept-min", "150", "--prior", pf] + CLI) == 0
    pb, lb = _write_scaled_epochs(tmp_path, "parts")
    assert cli.main_step2([pb[0], "--frames", lb, "--accept-min", "60", "--checkpoint", "--prior", pf] + CLI) == 0
    other = _prior_file(tmp_path, "other.json", p_first, ycc_hi=0.5)
    with pytest.raises(SystemExit, match="other priors"):
        cli.main_step2([pb[0], "--frames", lb, "--accept-min", "150", "--resume", "--prior", other] + CLI)
    assert cli.main_step2([pb[0], "--frames", lb, "--accept-min", "150", "--resume", "--prior", pf] + CLI) == 0
    for a, b in zip(pa, pb):
        da, db = chains.results_dir(a), chains.results_dir(b)
        sa, sb = json.load(open(da + "step2_summary.json")), json.load(open(db + "step2_summary.json"))
        sa.pop("image"), sb.pop("image")
        assert sa == sb
        for w in range(8):
            for name in ("%d_finalarray_mpi.csv", "%d_acceptance_rate.csv"):
                assert open(da + name % w, "rb").read() == open(db + name % w, "rb").read(), (a, name % w)


def test_cli_prior_refuses_a_start_outside_a_box(tmp_path):
    from olpefit_b200 import cli
    paths, lst = _write_scaled_epochs(tmp_path, "out")
    pf = tmp_path / "prior.json"
    pf.write_text(json.dumps({"epochs": {"29961": {"ampratio": {"min": 0.999, "max": 1.0}}}}))
    with pytest.raises(SystemExit, match="epoch 29961 has ampratio"):
        cli.main_step2([paths[0], "--frames", lst, "--accept-min", "50", "--prior", str(pf)] + CLI)
