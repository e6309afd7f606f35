"""Per-epoch jump widths on the device (lapf_sampler_set_frame_widths / frame_counts / adapt_widths,
include/lapf.h): a table of batch widths changes nothing the sampler computes; a row is what the walkers
of its frame propose with; the counts and the adaptation are the numpy restatement of test_frame_widths;
checkpoints, reset and refusals behave as documented; tuning helps epochs of very different brightness;
and the command line's --adapt-per-epoch."""
import json
import os

import numpy as np
import pytest

from oracle import lapf_oracle as orc
from test_frame_widths import adapt_rule

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


def _run(gpu, dom, init, frame_of, runs, *, table=None, fmt="f64", team=0, burn_in=0, thin=1, seed=7, widths=None,
         extras=True, id_base=0):
    """``table``: None (off), "batch" (every row the batch widths) or an [F, P] array.  Returns (rows or None,
    everything else the sampler reports as numpy)."""
    torch, chains = gpu["torch"], gpu["chains"]
    out = {}
    with gpu["sampler"].GibbsSampler(dom, init, frame_of, seed=seed, burn_in=burn_in, thin=thin, team_warps=team,
                                     widths=widths, id_base=id_base) as s:
        if extras:
            s.enable_sketch(n_bins=512, sep_bin=1e-3, pa_bin=5e-3)
            s.enable_batch_means(5, 3)
            s.enable_draws(7)
        if table is not None:
            s.set_frame_widths(None if isinstance(table, str) else table)
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
        out["moments"] = s.stats()["moments"].cpu().numpy()
        if extras:
            sk = s.sketch()
            out["hist"], out["summary"] = sk["hist"].cpu().numpy(), sk["summary"].cpu().numpy()
            bm = s.batch_means()
            out["bm_walker"], out["bm_frame"] = bm["walker"].cpu().numpy(), bm["frame"].cpu().numpy()
            d = s.draws()
            out["draws"], out["draw_rows"] = d["values"].cpu().numpy(), d["rows"].cpu().numpy()
        out["counts"] = s.frame_counts().cpu().numpy()
        if table is not None:
            out["fw"] = s.frame_widths().cpu().numpy()
        torch.cuda.synchronize()
    return (np.concatenate(parts) if parts else None), out


def _same(a, b, keys=None):
    for key in keys or [k for k in a if k in b and k != "fw"]:
        np.testing.assert_array_equal(np.asarray(a[key]).view(np.uint8), np.asarray(b[key]).view(np.uint8), err_msg=key)


# the occupancy of test_gpu_parity.test_full_size_batch_state_is_consistent_with_k1
@pytest.mark.parametrize("nbody,size,walkers,frames,n_upd", [
    (2, 64, 65536, 100, 48),
    (2, 32, 148 * (2 * 512 + 37), 5, 32),
    (3, 32, 148 * (2 * 512 + 37), 5, 32),
    (3, 64, 148 * (512 + 37), 3, 32),
    (2, 128, 148 * (192 + 29), 3, 16),
    (3, 128, 148 * (144 + 29), 3, 16),
])
def test_full_size_table_of_batch_widths_is_the_parent(gpu, nbody, size, walkers, frames, n_upd):
    dom, p_frame, _, _ = _domain(gpu, nbody, size, frames)
    frame_of = np.arange(walkers) % frames
    init = p_frame[frame_of]
    rows0, off = _run(gpu, dom, init, frame_of, [n_upd], burn_in=3)
    rows1, on = _run(gpu, dom, init, frame_of, [n_upd], table="batch", burn_in=3)
    np.testing.assert_array_equal(rows0.view(np.int64), rows1.view(np.int64))
    _same(off, on)
    rows2, ev = _run(gpu, dom, init, frame_of, [n_upd // 2, n_upd - n_upd // 2], table="batch", fmt="events_f64", burn_in=3)
    np.testing.assert_array_equal(rows0.view(np.int64), rows2.view(np.int64))
    _same(off, ev)
    w0, _ = gpu["layout"].default_widths(nbody)
    assert np.array_equal(on["fw"], np.tile(w0, (frames, 1)))


@pytest.mark.parametrize("team,nbody,size", [(4, 2, 64), (4, 3, 32), (16, 2, 128), (16, 3, 64)])
def test_team_kernels_table_of_batch_widths_is_the_parent(gpu, team, nbody, size):
    dom, p_frame, _, _ = _domain(gpu, nbody, size, 2)
    frame_of = np.arange(24) % 2
    rows0, off = _run(gpu, dom, p_frame[frame_of], frame_of, [70, 41], team=team, burn_in=2)
    rows1, on = _run(gpu, dom, p_frame[frame_of], frame_of, [70, 41], team=team, burn_in=2, table="batch")
    np.testing.assert_array_equal(rows0.view(np.int64), rows1.view(np.int64))
    _same(off, on)
    rows2, ev = _run(gpu, dom, p_frame[frame_of], frame_of, [111], team=team, burn_in=2, table="batch", fmt="events_f64")
    np.testing.assert_array_equal(rows0.view(np.int64), rows2.view(np.int64))
    _same(off, ev)


def _rows_table(nbody, F):
    from olpefit_b200 import layout
    w0, _ = layout.default_widths(nbody)
    return np.stack([w0 * s for s in (0.5, 1.7, 3.1)[:F]])


@pytest.mark.parametrize("nbody,size,walkers,team", [(2, 64, 1800, 0), (3, 32, 1800, 0), (2, 128, 700, 0),
                                                     (2, 64, 24, 4), (3, 64, 24, 16)])
def test_each_frame_proposes_with_its_row(gpu, nbody, size, walkers, team):
    dom, p_frame, _, _ = _domain(gpu, nbody, size, 3)
    frame_of = np.arange(walkers) % 3
    init = p_frame[frame_of]
    table = _rows_table(nbody, 3)
    rows, res = _run(gpu, dom, init, frame_of, [40, 23], table=table, team=team, extras=False, id_base=5)
    assert np.array_equal(res["fw"], table)
    for f in range(3):
        ref_rows, ref = _run(gpu, dom, init, frame_of, [63], widths=table[f], team=team, extras=False, id_base=5)
        sel = frame_of == f
        np.testing.assert_array_equal(rows[:, sel].view(np.int64), ref_rows[:, sel].view(np.int64), err_msg=str(f))
        for key in ("state", "tries", "accepts"):
            np.testing.assert_array_equal(res[key][sel], ref[key][sel], err_msg=key)


def test_frame_rows_replay_the_oracle_with_that_rows_widths(gpu):
    nbody, size = 2, 64
    lay = orc.layout_for(nbody)
    dom, p_frame, stamps, origins = _domain(gpu, nbody, size, 3)
    walkers, n_upd, seed = 600, 64, 4321
    frame_of = np.arange(walkers) % 3
    table = _rows_table(nbody, 3)
    rows, _ = _run(gpu, dom, p_frame[frame_of], frame_of, [n_upd], table=table, seed=seed, extras=False)
    for wi in (0, 1, 2, 31, 32, 299, 300, 599):
        f = int(frame_of[wi])
        img = stamps[f].astype(np.float64)
        res = orc.run_chain(img, orc.weight_map(img, HEADER), lay, p_frame[f], orc.PhiloxStream(seed, wi, lay.nparam),
                            origin=tuple(origins[f]), n_updates=n_upd, burn_in=0, widths=table[f])
        dev = rows[:, wi]
        same = np.all(np.isclose(dev[:, :-1], res.rows[1:, :-1], rtol=1e-9, atol=1e-12), axis=1)
        first_bad = int(np.argmin(same)) if not same.all() else n_upd
        # as in smoke(): FP32 chi-square may flip a borderline accept late, never early
        assert first_bad >= 24, (wi, first_bad)
        np.testing.assert_allclose(dev[:first_bad, -1], res.rows[1:first_bad + 1, -1], rtol=1e-5)


def test_frame_counts_are_the_walkers_counters_summed_by_frame(gpu):
    dom, p_frame, _, _ = _domain(gpu, 3, 32, 4)
    frame_of = np.arange(3000) % 4
    frame_of[:17] = 2                                            # uneven frames
    for table in (None, "batch"):
        _, res = _run(gpu, dom, p_frame[frame_of], frame_of, [77], table=table, fmt=None, extras=False)
        want = np.zeros((4, 19, 2), dtype=np.int64)
        np.add.at(want[..., 0], frame_of, res["tries"].astype(np.int64))
        np.add.at(want[..., 1], frame_of, res["accepts"].astype(np.int64))
        np.testing.assert_array_equal(res["counts"], want)


def _ulps(a, b):
    ia, ib = a.view(np.int64), b.view(np.int64)
    return np.abs(ia - ib)


def test_device_adaptation_is_the_numpy_rule(gpu):
    torch = gpu["torch"]
    dom, p_frame, _, _ = _domain(gpu, 2, 32, 3)
    F, P = 3, 16
    rng = np.random.default_rng(4)
    w0 = rng.uniform(1e-3, 1.0, size=(F, P))
    tries = rng.integers(0, 3000, size=(F, P))
    c1 = np.stack([tries, rng.integers(0, tries + 1)], axis=-1)
    c1[0, 5] = 0                                                  # no tries: keeps its width
    c1[2, 4] = [400, 140]                                         # on target
    extra = rng.integers(0, 500, size=(F, P))
    c2 = c1 + np.stack([extra, rng.integers(0, extra + 1)], axis=-1)
    with gpu["sampler"].GibbsSampler(dom, p_frame[np.arange(30) % 3], np.arange(30) % 3, seed=1) as s:
        s.set_frame_widths(w0)
        w, snap = w0, np.zeros_like(c1)
        c3 = c2 + 7
        c4 = c3 + np.array([1000, 0])                             # rate 0 against 0.99: exp(-0.99) clipped to 0.5
        for c, target in ((c1, 0.35), (c2, 0.35), (c2, 0.2), (c3, 0.6), (c4, 0.99)):
            s.adapt_widths(torch.tensor(c, dtype=torch.int64), target)
            w, snap = adapt_rule(w, c, snap, target)
            got = s.frame_widths().cpu().numpy()
            assert _ulps(got, w).max() <= 2, _ulps(got, w).max()
            if c is c1:
                assert got[0, 5] == w0[0, 5] and got[2, 4] == w0[2, 4]        # no tries; on target
            if c is c4:
                np.testing.assert_array_equal(got, 0.5 * w_prev)
            w = w_prev = got                                               # continue from the device's widths


def test_device_adaptation_equals_host_set_widths_at_the_same_counts(gpu):
    dom, p_frame, _, _ = _domain(gpu, 2, 64, 3)
    frame_of = np.arange(900) % 3
    init = p_frame[frame_of]
    steps = [64, 64, 100, 64]
    seen, chains_a = [], []
    with gpu["sampler"].GibbsSampler(dom, init, frame_of, seed=9, burn_in=50) as a:
        a.set_frame_widths()
        for n in steps:
            chains_a.append(a.run(n).cpu().numpy())
            a.adapt_widths(a.frame_counts(), 0.35)
            seen.append(a.frame_widths().cpu().numpy())
        st_a = a.state()[0].cpu().numpy()
    assert not np.array_equal(seen[0], seen[-1])
    chains_b = []
    with gpu["sampler"].GibbsSampler(dom, init, frame_of, seed=9, burn_in=50) as b:
        b.set_frame_widths()
        for n, w in zip(steps, seen):
            chains_b.append(b.run(n).cpu().numpy())
            b.set_frame_widths(w)
        st_b = b.state()[0].cpu().numpy()
    for x, y in zip(chains_a, chains_b):
        np.testing.assert_array_equal(x.view(np.int64), y.view(np.int64))
    np.testing.assert_array_equal(st_a.view(np.int64), st_b.view(np.int64))


def _adapting(s, windows, n):
    out = []
    for _ in range(windows):
        out.append(s.run(n).cpu().numpy())
        s.adapt_widths(s.frame_counts(), 0.35)
    return out


def test_save_and_load_in_burn_in_continue_to_the_same_widths_and_chains(gpu):
    dom, p_frame, _, _ = _domain(gpu, 2, 32, 3)
    frame_of = np.arange(600) % 3
    init = p_frame[frame_of]
    with gpu["sampler"].GibbsSampler(dom, init, frame_of, seed=5, burn_in=400) as a:
        a.set_frame_widths()
        _adapting(a, 2, 64)
        a.run(20)                                                # in the middle of a window
        blob = a.save().clone()
        want = _adapting(a, 3, 44)
        want_w = a.frame_widths().cpu().numpy()
    with gpu["sampler"].GibbsSampler(dom, init, frame_of, seed=5, burn_in=400) as b:
        b.set_frame_widths(np.ones((3, 16)))                     # overwritten by the blob
        b.load(blob)
        got = _adapting(b, 3, 44)
        np.testing.assert_array_equal(b.frame_widths().cpu().numpy(), want_w)
    for x, y in zip(want, got):
        np.testing.assert_array_equal(x.view(np.int64), y.view(np.int64))


def test_reset_refusals_and_checkpoint_layout(gpu):
    lib = gpu["lib"]
    dom, p_frame, _, _ = _domain(gpu, 2, 32, 2)
    frame_of = np.arange(40) % 2
    init = p_frame[frame_of]
    W, P, F = 40, 16, 2
    with gpu["sampler"].GibbsSampler(dom, init, frame_of, seed=3) as s:
        plain = int(s.save().numel())
        # the parent's layout: head, state, shift, moments (2x), exps, tries, accepts
        assert plain == 8 * (2 + 19) + 8 * W * (P + 1) * 4 + 8 * W + 4 * W * P * 2
        plain_blob = s.save().clone()
        with pytest.raises(lib.LapfError):
            s.adapt_widths(s.frame_counts(), 0.35)               # no table
        for bad in (-0.1, float("inf"), float("nan")):
            t = np.ones((F, P))
            t[1, 3] = bad
            with pytest.raises(lib.LapfError):
                s.set_frame_widths(t)
        with pytest.raises(ValueError):
            s.set_frame_widths(np.ones((F + 1, P)))
        s.set_frame_widths()
        with pytest.raises(lib.LapfError):
            s.set_widths(np.ones(P))                             # one source of truth
        for bad in (0.0, 1.0, -0.5, 1.5, float("nan")):
            with pytest.raises(lib.LapfError):
                s.adapt_widths(s.frame_counts(), bad)
        blob = s.save().clone()
        assert blob.numel() == plain + 32 + F * P * 8 * 3
        desc = blob[plain:plain + 32].cpu().numpy().view(np.int64)
        assert bytes(desc[:1].view(np.uint8)) == b"LAPFFW01" and desc[1:].tolist() == [F, P, 0]
        with pytest.raises(lib.LapfError):
            s.load(plain_blob)                                   # no table in the blob
        s.run(300, record=False)
        s.adapt_widths(s.frame_counts(), 0.35)
        w = s.frame_widths().cpu().numpy()
        s.reset(init, seed=3)
        np.testing.assert_array_equal(s.frame_widths().cpu().numpy(), w)     # reset keeps the widths ...
        s.adapt_widths(s.frame_counts(), 0.35)                   # ... and empties the window: no tries, no change
        np.testing.assert_array_equal(s.frame_widths().cpu().numpy(), w)
        s.run(200, record=False)
        c = s.frame_counts()
        s.adapt_widths(c, 0.35)
        want, _ = adapt_rule(w, c.cpu().numpy(), np.zeros((F, P, 2), dtype=np.int64), 0.35)   # window since the reset
        assert _ulps(s.frame_widths().cpu().numpy(), want).max() <= 2
        s.set_frame_widths(np.full((F, P), 0.01))                # later calls replace the widths
        assert (s.frame_widths() == 0.01).all()
    with gpu["sampler"].GibbsSampler(dom, init, frame_of, seed=3) as t:
        with pytest.raises(lib.LapfError):
            t.load(blob)                                         # a table in the blob, none here
        with pytest.raises(lib.LapfError):
            t.frame_widths()
        t.load(plain_blob)
    dom3, p3, _, _ = _domain(gpu, 2, 32, 3)
    with gpu["sampler"].GibbsSampler(dom3, p3[np.arange(40) % 3], np.arange(40) % 3, seed=3) as t:
        t.set_frame_widths()
        with pytest.raises(lib.LapfError):
            t.load(blob)                                         # a table of 2 frames, 3 here


def _scaled_stamps(scales, size=64, nbody=2):
    """Epochs whose objects are `scales` times as bright as a 4000-count star with 1000-count companions (the
    noise model of synth.make_frame)."""
    from olpefit_b200 import synth
    ox, oy = synth.stamp_origin(size, nbody)
    stamps, truths = [], []
    for f, a in enumerate(scales):
        p = synth.truth_parameters(nbody, f)
        p[2 * nbody + 2:3 * nbody + 2] = a * np.array([4000.0, 1000.0, 1000.0][:nbody])
        rng = np.random.default_rng(100 + f)
        t = synth.truth_image(p, nbody, (oy, oy + size, ox, ox + size))
        img = rng.poisson(t + synth.SKY_LEVEL).astype(np.float64) - synth.SKY_LEVEL + rng.normal(0, synth.READ_NOISE, t.shape)
        stamps.append(img.astype(np.float32))
        truths.append(p)
    return np.stack(stamps), np.tile([[ox, oy]], (len(scales), 1)).astype(np.int32), np.stack(truths)


def test_tuning_brings_every_epoch_near_the_target(gpu):
    scales = (0.25, 1.0, 4.0)
    stamps, origins, truths = _scaled_stamps(scales)
    dom = gpu["frame"].prepare_domain(stamps, HEADER, origin=origins, nbody=2)
    frame_of = np.arange(3 * 64) % 3
    burn = 12 * 512
    with gpu["sampler"].GibbsSampler(dom, truths[frame_of], frame_of, seed=13, burn_in=burn) as s:
        s.set_frame_widths()
        c0 = s.frame_counts().cpu().numpy()
        s.run(2048, record=False)
        before = s.frame_counts().cpu().numpy() - c0
        for _ in range(burn // 512 - 4):
            s.run(512, record=False)
            s.adapt_widths(s.frame_counts(), 0.35)
        c1 = s.frame_counts().cpu().numpy()
        s.run(4096, record=False)
        after = s.frame_counts().cpu().numpy() - c1
        w = s.frame_widths().cpu().numpy()
    rate0 = before[..., 1] / before[..., 0]
    rate = after[..., 1] / after[..., 0]
    print("default widths, position acceptance per epoch:", np.round(rate0[:, :4], 3))
    print("tuned, position acceptance per epoch:", np.round(rate[:, :4], 3))
    print("tuned position widths:", w[:, :4])
    assert np.all((rate[:, :4] > 0.2) & (rate[:, :4] < 0.5)), rate[:, :4]
    assert np.all(w[0, :4] > w[2, :4])                           # the faintest epoch takes the longest steps


def _write_scaled_epochs(tmp_path, tag, scales=(0.25, 1.0, 4.0)):
    from olpefit_b200 import chains, frame, synth
    paths = []
    for f, a in enumerate(scales):
        d = tmp_path / ("%s_epoch%d" % (tag, f))
        d.mkdir()
        p = synth.truth_parameters(2, f)
        p[6:8] = a * np.array([4000.0, 1000.0])                 # star and companion, as in _scaled_stamps
        rng = np.random.default_rng(200 + f)
        t = synth.truth_image(p, 2, (0, 1024, 0, 1024))
        img = rng.poisson(t + synth.SKY_LEVEL).astype(np.float64) - synth.SKY_LEVEL + rng.normal(0, synth.READ_NOISE, t.shape)
        path = str(d / ("N2.2009053%d.2996%d.LDIF.fits" % (f, f)))
        frame.write_fits(path, img.astype(np.float32), synth.HEADER)
        os.makedirs(chains.results_dir(path))
        chains.write_walker_csv(chains.results_dir(path) + "step2a.csv", np.concatenate([p, [0.0]])[None])
        paths.append(path)
    lst = tmp_path / (tag + "_frames.txt")
    lst.write_text("\n".join(paths[1:]) + "\n")
    return paths, str(lst)


COMMON = ["-i", "2a", "--walkers", "8", "--burn-in", "1500", "--seed", "29", "--stamp", "64", "--segment", "384",
          "--adapt-per-epoch", "--quiet"]


def test_cli_adapt_per_epoch_writes_widths_and_acceptance(tmp_path):
    from olpefit_b200 import chains, cli, layout
    paths, lst = _write_scaled_epochs(tmp_path, "ape")
    assert cli.main_step2([paths[0], "--frames", lst, "--accept-min", "200", "--no-chains"] + COMMON) == 0
    summ = [json.load(open(chains.results_dir(p) + "step2_summary.json")) for p in paths]
    names = list(layout.names(2))
    w0, _ = layout.default_widths(2)
    for s in summ:
        assert list(s["widths"]) == names and list(s["acceptance"]) == names
        assert all(0.0 <= v <= 1.0 for v in s["acceptance"].values())
    assert summ[0]["widths"]["xcs"] > summ[2]["widths"]["xcs"]         # the faint epoch takes longer steps
    assert summ[0]["widths"] != summ[1]["widths"] != summ[2]["widths"]
    assert [summ[0]["widths"][n] for n in names] != w0.tolist()


def test_cli_adapt_per_epoch_resumes_inside_burn_in(tmp_path):
    from olpefit_b200 import chains, cli
    pa, la = _write_scaled_epochs(tmp_path, "whole")
    assert cli.main_step2([pa[0], "--frames", la, "--accept-min", "200"] + COMMON) == 0
    pb, lb = _write_scaled_epochs(tmp_path, "parts")
    assert cli.main_step2([pb[0], "--frames", lb, "--accept-min", "40", "--checkpoint"] + COMMON) == 0
    first = json.load(open(chains.results_dir(pb[0]) + "step2_summary.json"))
    assert first["updates"] < 1500                               # stopped inside burn-in
    assert cli.main_step2([pb[0], "--frames", lb, "--accept-min", "200", "--resume"] + COMMON) == 0
    for a, b in zip(pa, pb):
        da, db = chains.results_dir(a), chains.results_dir(b)
        sa, sb = json.load(open(da + "step2_summary.json")), json.load(open(db + "step2_summary.json"))
        sa.pop("image"), sb.pop("image")
        assert sa == sb
        for w in range(8):
            for name in ("%d_finalarray_mpi.csv", "%d_acceptance_rate.csv"):
                assert open(da + name % w, "rb").read() == open(db + name % w, "rb").read(), (a, name % w)


def _two_gpus():
    import torch
    return torch.cuda.is_available() and torch.cuda.device_count() >= 2


@pytest.mark.skipif(not _two_gpus(), reason="needs two GPUs")
def test_cli_adapt_per_epoch_on_two_gpus_equals_one_gpu(tmp_path):
    import subprocess
    import sys
    from olpefit_b200 import chains, cli
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    # 3 epochs x 7 walkers over 2 ranks: global walker g = w * 3 + f goes to rank g % 2, so every epoch spans both
    common = ["-i", "2a", "--walkers", "7", "--burn-in", "700", "--seed", "31", "--stamp", "64", "--segment", "256",
              "--accept-min", "80", "--adapt-per-epoch", "--quiet"]
    p1, l1 = _write_scaled_epochs(tmp_path, "one")
    assert cli.main_step2([p1[0], "--frames", l1] + common) == 0
    p2, l2 = _write_scaled_epochs(tmp_path, "two")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", "29631", os.path.join(root, "apf_step2.py"), p2[0], "--frames", l2] + common
    res = subprocess.run(cmd, capture_output=True, text=True, cwd=root, timeout=900)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-4000:]
    for a, b in zip(p1, p2):
        da, db = chains.results_dir(a), chains.results_dir(b)
        for w in range(7):
            assert open(da + "%d_finalarray_mpi.csv" % w, "rb").read() == open(db + "%d_finalarray_mpi.csv" % w, "rb").read()
        sa, sb = json.load(open(da + "step2_summary.json")), json.load(open(db + "step2_summary.json"))
        assert sa["widths"] == sb["widths"] and sa["acceptance"] == sb["acceptance"]
