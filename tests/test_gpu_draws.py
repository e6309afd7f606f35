"""Posterior draws on the device (lapf_sampler_draws, include/lapf.h): the reservoir holds exactly the
dense float64 chain's rows at the indices the numpy restatement in test_draws selects, changes nothing
else the sampler computes, does not depend on how a run is split, checkpointed or recorded, and its
pooled separation / position angle agree with the sketches; plus the command line's draws file."""
import json
import os

import numpy as np
import pytest

from test_draws import reservoir_rows

pytestmark = pytest.mark.gpu

HEADER = {"itime": 1.0, "coadds": 1, "multisam": 1, "sampmode": 2}


@pytest.fixture(scope="module")
def gpu():
    import torch
    from olpefit_b200 import _lib, frame, sampler, stats, synth
    assert torch.cuda.is_available()
    return {"torch": torch, "frame": frame, "sampler": sampler, "stats": stats, "synth": synth, "lib": _lib}


def _domain(gpu, nbody, size, n_frames):
    synth = gpu["synth"]
    stamps, origins = synth.make_stamps(n_frames, size, nbody)
    dom = gpu["frame"].prepare_domain(stamps, HEADER, origin=origins, nbody=nbody)
    p_frame = np.array([synth.truth_parameters(nbody, f) for f in range(n_frames)])
    return dom, p_frame


def _run(gpu, dom, init, frame_of, runs, *, K=None, fmt="f64", team=0, burn_in=0, thin=1, seed=7, bm=None,
         save_after=None, draws_first=True):
    """Runs ``runs`` updates in turn; returns (dense rows or None, everything the sampler reports)."""
    torch = gpu["torch"]
    out = {}
    with gpu["sampler"].GibbsSampler(dom, init, frame_of, seed=seed, burn_in=burn_in, thin=thin, team_warps=team) as s:
        if K is not None and draws_first:
            s.enable_draws(K)
        s.enable_sketch(n_bins=512, sep_bin=1e-3, pa_bin=5e-3)
        if bm is not None:
            s.enable_batch_means(*bm)
        if K is not None and not draws_first:
            s.enable_draws(K)
        if fmt is not None:
            s.set_chain_format(fmt)
        parts = []
        for i, n in enumerate(runs):
            if save_after is not None and i == save_after:
                blob = s.save()
                s.run(5 + 3 * n, record=False)          # wander off, then come back
                s.load(blob)
            r = s.run(n, record=fmt is not None)
            if fmt is not None and not s.events:
                parts.append(r.cpu().numpy())
            elif fmt is not None:
                from olpefit_b200 import chains
                parts.append(chains.decode_events(r[0].cpu().numpy(), r[1], s.n_walkers, s.nparam + 1,
                                                  np.float32 if fmt.endswith("f32delta") else np.float64))
        st, tr, ac = s.state()
        out["state"], out["tries"], out["accepts"] = st.cpu().numpy(), tr.cpu().numpy(), ac.cpu().numpy()
        stt = s.stats()
        out["moments"] = stt["moments"].cpu().numpy()
        out["rows_n"] = int(stt["rows"])
        sk = s.sketch()
        out["hist"], out["summary"] = sk["hist"].cpu().numpy(), sk["summary"].cpu().numpy()
        if bm is not None:
            out["bm"] = s.batch_means()
            out["bm_walker"] = out["bm"]["walker"].cpu().numpy()
        if K is not None:
            d = s.draws()
            out["values"], out["rows"], out["filled"] = d["values"].cpu().numpy(), d["rows"].cpu().numpy(), d["filled"]
            assert d["per_walker"] == K and d["filled"] == min(K, out["rows_n"])
        out["blob_bytes"] = int(s.save().numel())
        torch.cuda.synchronize()
    rows = np.concatenate(parts) if parts else None
    return rows, out


def _check_reservoir(rows, res, K, seed):
    """Row indices are the restatement's; values are the dense rows at them, byte for byte; empty slots
    hold -1 and all-ones NaNs."""
    n, W = rows.shape[0], rows.shape[1]
    want = reservoir_rows(seed, np.arange(W), n, K)
    np.testing.assert_array_equal(res["rows"], want)
    w, k = np.nonzero(want >= 0)
    np.testing.assert_array_equal(res["values"][w, k].view(np.int64), rows[want[w, k], w].view(np.int64))
    w, k = np.nonzero(want < 0)
    assert (res["values"][w, k].view(np.int64) == -1).all()
    assert ((want >= 0).sum(axis=1) == min(K, n)).all()


def _check_unchanged(a, b, rows_a, rows_b):
    for key in ("state", "tries", "accepts", "moments", "hist", "summary"):
        np.testing.assert_array_equal(a[key], b[key], err_msg=key)
    if rows_a is not None:
        np.testing.assert_array_equal(rows_a, rows_b)


@pytest.mark.parametrize("nbody,size,walkers,frames,n_upd,K,thin,burn_in", [
    (2, 64, 65536, 100, 48, 7, 1, 0),
    (2, 32, 148 * (2 * 512 + 37), 5, 32, 1, 1, 3),
    (3, 32, 148 * (2 * 512 + 37), 5, 33, 7, 3, 4),
    (3, 64, 148 * (512 + 37), 3, 32, 40, 1, 0),
    (2, 128, 148 * (192 + 29), 3, 40, 7, 3, 2),
    (3, 128, 148 * (144 + 29), 3, 16, 1, 1, 1),
])
def test_full_size_reservoir_is_the_restated_rows_and_changes_nothing_else(gpu, nbody, size, walkers, frames, n_upd,
                                                                          K, thin, burn_in):
    dom, p_frame = _domain(gpu, nbody, size, frames)
    frame_of = np.arange(walkers) % frames
    rows, res = _run(gpu, dom, p_frame[frame_of], frame_of, [n_upd], K=K, thin=thin, burn_in=burn_in)
    _check_reservoir(rows, res, K, 7)
    rows0, res0 = _run(gpu, dom, p_frame[frame_of], frame_of, [n_upd], thin=thin, burn_in=burn_in)
    _check_unchanged(res, res0, rows, rows0)


@pytest.mark.parametrize("team,nbody,size,K,thin,burn_in", [
    (4, 2, 64, 7, 1, 0), (4, 3, 32, 100, 3, 5), (16, 2, 128, 1, 1, 2), (16, 3, 64, 7, 3, 0),
])
def test_team_kernels_reservoir_is_the_restated_rows(gpu, team, nbody, size, K, thin, burn_in):
    dom, p_frame = _domain(gpu, nbody, size, 2)
    frame_of = np.arange(24) % 2
    rows, res = _run(gpu, dom, p_frame[frame_of], frame_of, [70, 41], K=K, team=team, thin=thin, burn_in=burn_in,
                     bm=(5, 3))
    _check_reservoir(rows, res, K, 7)
    rows0, res0 = _run(gpu, dom, p_frame[frame_of], frame_of, [70, 41], team=team, thin=thin, burn_in=burn_in, bm=(5, 3))
    _check_unchanged(res, res0, rows, rows0)
    np.testing.assert_array_equal(res["bm_walker"], res0["bm_walker"])


def test_reservoir_is_invariant_to_splits_checkpoints_formats_and_recording(gpu):
    dom, p_frame = _domain(gpu, 2, 32, 3)
    frame_of = np.arange(3000) % 3
    init = p_frame[frame_of]
    _, ref = _run(gpu, dom, init, frame_of, [96], K=9)
    for kw in ({"runs": [7, 25, 64]}, {"runs": [40, 56], "save_after": 1}, {"runs": [96], "fmt": "f32delta"},
               {"runs": [50, 46], "fmt": "events_f64"}, {"runs": [33, 63], "fmt": "events_f32delta"},
               {"runs": [96], "fmt": None}, {"runs": [96], "draws_first": False, "bm": (4, 3)}):
        _, res = _run(gpu, dom, init, frame_of, K=9, **kw)
        np.testing.assert_array_equal(res["rows"], ref["rows"], err_msg=str(kw))
        np.testing.assert_array_equal(res["values"].view(np.int64), ref["values"].view(np.int64), err_msg=str(kw))


def test_reset_refusals_and_checkpoint_layout(gpu):
    torch, lib = gpu["torch"], gpu["lib"]
    dom, p_frame = _domain(gpu, 2, 32, 1)
    init = np.repeat(p_frame, 40, axis=0)
    P = 16
    with gpu["sampler"].GibbsSampler(dom, init, seed=3) as s:
        plain = int(s.save().numel())
        for bad in (0, -1, 65537):
            with pytest.raises(lib.LapfError):
                s.enable_draws(bad)
        s.enable_draws(5)
        with pytest.raises(lib.LapfError):
            s.enable_draws(5)                                  # a second call
        blob = s.save()
        assert blob.numel() == plain + 32 + 40 * 5 * (P + 2) * 8
        desc = blob[plain:plain + 32].cpu().numpy().view(np.int64)
        assert bytes(desc[:1].view(np.uint8)) == b"LAPFRS01" and desc[1:].tolist() == [5, P + 1, 0]
        d = s.draws()
        assert (d["rows"] == -1).all() and d["filled"] == 0       # the self-test left the reservoir empty
        s.run(12)
        assert (s.draws()["rows"] >= 0).sum().item() == 40 * 5
        s.reset(init, seed=3)
        d = s.draws()
        assert (d["rows"] == -1).all() and (d["values"].view(torch.int64) == -1).all()
        s.run(3)
        with pytest.raises(lib.LapfError):
            s.load(blob[:plain])                               # a blob without draws is too small
        with gpu["sampler"].GibbsSampler(dom, init, seed=3) as t:
            t.run(2)
            with pytest.raises(lib.LapfError):
                t.enable_draws(4)                              # rows were recorded
        with gpu["sampler"].GibbsSampler(dom, init, seed=3) as t:
            t.enable_draws(4)
            with pytest.raises(lib.LapfError):
                t.load(blob)                                   # large enough, but its descriptor says K = 5
        with gpu["sampler"].GibbsSampler(dom, init, seed=3) as t:
            t.enable_draws(5)
            bad = blob.clone()
            bad[plain + 8] = 6                                 # K in the descriptor
            with pytest.raises(lib.LapfError):
                t.load(bad)
            t.load(blob)
    with gpu["sampler"].GibbsSampler(dom, init, seed=3) as s:
        s.enable_batch_means(4, 3)
        assert int(s.save().numel()) > plain
        s.enable_draws(2)                                      # after batch means: the draws are the last section
        b = s.save()
        assert bytes(b[-(40 * 2 * (P + 2) * 8) - 32:][:8].cpu().numpy()) == b"LAPFRS01"


def test_pooled_draws_agree_with_the_sketch_medians(gpu):
    stats, torch = gpu["stats"], gpu["torch"]
    dom, p_frame = _domain(gpu, 2, 32, 1)
    W, K = 4096, 16
    frame_of = np.zeros(W, dtype=np.int64)
    with gpu["sampler"].GibbsSampler(dom, p_frame[frame_of], frame_of, seed=11, burn_in=2000) as s:
        s.enable_sketch(n_bins=4096, sep_bin=2e-4, pa_bin=1e-3)
        s.enable_batch_means(64, 8)
        s.enable_draws(K)
        for _ in range(4):
            s.run(2048, record=False)
        sk = stats.sketch_summary(s.sketch())
        bm = s.batch_means()
        summ = stats.batch_means_summary(bm, torch.tensor([float(W)], dtype=torch.float64), bm["rows"])
        d = s.draws()
        assert d["filled"] == K and (d["rows"] >= 0).all()
        sep, pa = stats.separation_pa(d["values"].reshape(-1, 17))
        for q, (vals, med, std, mcse, width) in enumerate((
                (sep, sk["sep_q"][0, 0, 1], sk["sep_std"][0, 0], summ["mcse"][0, 17] * stats.PIXSCALE_PRE2015, 2e-4 * stats.PIXSCALE_PRE2015),
                (pa, sk["pa_q"][0, 0, 1], sk["pa_std"][0, 0], summ["mcse"][0, 18], 1e-3))):
            n = vals.numel()
            tol = 4.0 * float(mcse) + 4.0 * 1.2533 * float(std) / np.sqrt(n) + width
            diff = abs(float(vals.median()) - float(med))
            print("quantity", q, "median diff", diff, "tol", tol, "mcse", float(mcse))
            assert diff <= tol


def _write_case(tmp_path, tag):
    from olpefit_b200 import frame, synth
    d = tmp_path / ("2009_2body%s" % tag)
    d.mkdir()
    img, _ = synth.make_frame(0, 2)
    path = str(d / "N2.20090531.29966.LDIF.fits")
    frame.write_fits(path, img, synth.HEADER)
    guess = synth.step1_guess(img, 2, sky_xy=(100, 120))
    with open(str(d / "29966_initialguess"), "w") as fh:
        fh.write(" ".join(str(v) for v in guess) + "\n")
    return path, str(d / "29966_apf_results")


COMMON = ["--walkers", "8", "--burn-in", "0", "--seed", "23", "--stamp", "32", "--segment", "512", "--quiet"]


def test_cli_draws_are_rows_of_the_chain_files(tmp_path):
    from olpefit_b200 import chains, cli
    path_a, out_a = _write_case(tmp_path, "_nochains")
    path_b, out_b = _write_case(tmp_path, "_csv")
    assert cli.main_step2([path_a, "--accept-min", "60", "--no-chains", "--draws", "8"] + COMMON) == 0
    assert cli.main_step2([path_b, "--accept-min", "60", "--format", "csv"] + COMMON) == 0
    assert not os.path.exists(os.path.join(out_b, "step2_draws.csv"))
    names, walker, row, values = chains.read_draws_csv(os.path.join(out_a, "step2_draws.csv"))
    assert len(names) == 17 and names[-1] == "chi2"
    summ = json.load(open(os.path.join(out_a, "step2_summary.json")))
    assert summ["draws"] == {"per_walker": 8, "rows_per_walker": summ["updates"], "count": 64, "file": "step2_draws.csv"}
    assert -1.0 <= summ["sep_pa_companion"]["sep_pa_corr"] <= 1.0
    assert np.bincount(walker).tolist() == [8] * 8
    for w in range(8):
        lines = open(os.path.join(out_b, "%d_finalarray_mpi.csv" % w)).read().splitlines()
        for r, v in zip(row[walker == w], values[walker == w]):
            want = np.array([float(x) for x in lines[r + 1].split(",")])      # line row + 2, counted from 1
            np.testing.assert_array_equal(v.view(np.int64), want.view(np.int64))


def test_cli_draws_survive_checkpoint_and_resume(tmp_path):
    from olpefit_b200 import cli
    path_a, out_a = _write_case(tmp_path, "_whole")
    assert cli.main_step2([path_a, "--accept-min", "160", "--draws", "8", "--no-chains"] + COMMON) == 0
    path_b, out_b = _write_case(tmp_path, "_parts")
    assert cli.main_step2([path_b, "--accept-min", "70", "--draws", "8", "--no-chains", "--checkpoint"] + COMMON) == 0
    assert cli.main_step2([path_b, "--accept-min", "160", "--draws", "8", "--no-chains", "--resume"] + COMMON) == 0
    a = open(os.path.join(out_a, "step2_draws.csv"), "rb").read()
    assert a == open(os.path.join(out_b, "step2_draws.csv"), "rb").read()
    sa = json.load(open(os.path.join(out_a, "step2_summary.json")))
    sb = json.load(open(os.path.join(out_b, "step2_summary.json")))
    assert sa["draws"] == sb["draws"] and sa["sep_pa_companion"] == sb["sep_pa_companion"]


def test_cli_ess_min_with_draws_stops_early_and_fills_the_reservoir(tmp_path):
    from olpefit_b200 import chains, cli
    path, out = _write_case(tmp_path, "_ess")
    accept_min = 5000
    assert cli.main_step2([path, "--accept-min", str(accept_min), "--ess-min", "100", "--draws", "8",
                           "--no-chains"] + COMMON) == 0
    summ = json.load(open(os.path.join(out, "step2_summary.json")))
    assert summ["stop"]["reason"] == "converged" and summ["updates"] < 16 * accept_min
    _, walker, row, _ = chains.read_draws_csv(os.path.join(out, "step2_draws.csv"))
    assert np.bincount(walker).tolist() == [min(8, summ["updates"])] * 8
    assert row.max() < summ["updates"] and summ["draws"]["count"] == 64
