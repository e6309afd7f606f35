"""Batch means on the device (lapf_sampler_batchmeans, include/lapf.h): the per-walker (snap, s2) state
is restated bit for bit from the dense float64 chain by the numpy restatement in test_batch_means, does not depend on
how a run is split, checkpointed or recorded, changes nothing else the sampler computes, and its
standard errors predict the spread of independent group means."""
import json
import os

import numpy as np
import pytest

from test_batch_means import batch_means_frame, batch_means_state

pytestmark = pytest.mark.gpu

HEADER = {"itime": 1.0, "coadds": 1, "multisam": 1, "sampmode": 2}


@pytest.fixture(scope="module")
def gpu():
    import torch
    from olpefit_b200 import frame, sampler, stats, synth
    assert torch.cuda.is_available()
    return {"torch": torch, "frame": frame, "sampler": sampler, "stats": stats, "synth": synth}


def _domain(gpu, nbody, size, n_frames):
    synth = gpu["synth"]
    stamps, origins = synth.make_stamps(n_frames, size, nbody)
    dom = gpu["frame"].prepare_domain(stamps, HEADER, origin=origins, nbody=nbody)
    p_frame = np.array([synth.truth_parameters(nbody, f) for f in range(n_frames)])
    return dom, p_frame


def _sep_pa_centred(rows, centers, frame_of, nbody):
    """Separation (pixels) and position angle (degrees) of every companion minus the frame's sketch centre,
    the angle wrapped to +-180 as record_sketch does: [rows, W, 2 (nbody - 1)]."""
    out = []
    for o in range(1, nbody):
        dx = rows[..., 2 * o] - rows[..., 0]
        dy = rows[..., 2 * o + 1] - rows[..., 1]
        sep = np.sqrt(dx * dx + dy * dy) - centers[frame_of, o - 1, 0]
        pa = np.arctan2(-dx, dy) * 57.29577951308232 - centers[frame_of, o - 1, 1]
        pa = pa - 360.0 * np.rint(pa * (1.0 / 360.0))
        out += [sep, pa]
    return np.stack(out, axis=-1)


def _run(gpu, dom, init, frame_of, runs, *, bm=None, sketch=True, fmt="f64", team=0, burn_in=0, thin=1, seed=7,
         save_after=None):
    """Runs ``runs`` updates in turn; returns (rows or None, everything the sampler reports)."""
    torch = gpu["torch"]
    out = {}
    with gpu["sampler"].GibbsSampler(dom, init, frame_of, seed=seed, burn_in=burn_in, thin=thin, team_warps=team) as s:
        if sketch:
            s.enable_sketch(n_bins=512, sep_bin=1e-3, pa_bin=5e-3)
        if bm is not None:
            s.enable_batch_means(*bm)
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
        out["start"] = s.start().cpu().numpy()
        if sketch:
            sk = s.sketch()
            out["hist"], out["summary"] = sk["hist"].cpu().numpy(), sk["summary"].cpu().numpy()
        if bm is not None:
            b = s.batch_means()
            out["walker"], out["frame"], out["names"] = b["walker"].cpu().numpy(), b["frame"].cpu().numpy(), b["names"]
            assert b["rows"] == out["rows_n"]
        torch.cuda.synchronize()
    rows = np.concatenate(parts) if parts else None
    return rows, out


def _check_against_oracle(rows, res, frame_of, nbody, batch_rows, levels, centers):
    """Columns bit for bit, separation / position angle to 1e-12, and the frame reduction to 1e-12."""
    P = 3 * nbody + 10
    start = res["start"]
    cols = rows - start[None]
    st_cols = batch_means_state(cols, batch_rows, levels)
    np.testing.assert_array_equal(res["walker"][:, :P + 1], st_cols)
    sp = _sep_pa_centred(rows, centers, frame_of, nbody)
    st_sp = batch_means_state(sp, batch_rows, levels)
    # numpy's sqrt / atan2 may differ from the device's in the last bit of the value before it is centred:
    # 1e-12 of the uncentred value per row for the sums, and what that makes of the squared batch sums
    n = rows.shape[0]
    tol = 1e-12 * n * max(np.abs(centers).max(), 1.0)
    np.testing.assert_allclose(res["walker"][:, P + 1:, :, 0], st_sp[..., 0], rtol=1e-12, atol=tol)
    np.testing.assert_allclose(res["walker"][:, P + 1:, :, 1], st_sp[..., 1], rtol=1e-12,
                               atol=2 * tol * np.sqrt(n * st_sp[..., 1].max()) + 1e-300)
    # the frame reduction from walker_out and the running moments
    allv = np.concatenate([cols, sp], axis=-1)
    row_var = allv.var(axis=0)
    per_w = batch_means_frame(res["walker"], row_var, n, batch_rows)
    F = res["frame"].shape[0]
    want = np.stack([per_w[frame_of == f].sum(axis=0) for f in range(F)])
    np.testing.assert_allclose(res["frame"], want, rtol=1e-12, atol=1e-12 * np.abs(want).max())


@pytest.mark.parametrize("nbody,size,walkers,frames,n_upd,batch_rows,thin,burn_in", [
    (2, 64, 65536, 100, 48, 1, 1, 0),
    (2, 32, 148 * (2 * 512 + 37), 5, 32, 5, 1, 3),
    (3, 32, 148 * (2 * 512 + 37), 5, 33, 1, 3, 4),
    (3, 64, 148 * (512 + 37), 3, 32, 5, 1, 0),
    (2, 128, 148 * (192 + 29), 3, 40, 1, 3, 2),
    (3, 128, 148 * (144 + 29), 3, 16, 5, 1, 1),
])
def test_full_size_batch_means_match_oracle_and_change_nothing_else(gpu, nbody, size, walkers, frames, n_upd,
                                                                   batch_rows, thin, burn_in):
    """Every batched shape at full occupancy: the per-walker state is the oracle's restatement of the
    dense chain, and the chain, state, counters, moments and sketches are those of the same run without
    batch means, bit for bit (the update after a boundary row is evaluated as it should be)."""
    dom, p_frame = _domain(gpu, nbody, size, frames)
    frame_of = (np.arange(walkers) % frames).astype(np.int32)
    init = p_frame[frame_of]
    levels = 3
    kw = dict(thin=thin, burn_in=burn_in, seed=31)
    rows, res = _run(gpu, dom, init, frame_of, [n_upd // 2, n_upd - n_upd // 2], bm=(batch_rows, levels), **kw)
    rows0, res0 = _run(gpu, dom, init, frame_of, [n_upd], **kw)
    np.testing.assert_array_equal(rows, rows0)
    for k in ("state", "tries", "accepts", "moments", "hist", "summary"):
        np.testing.assert_array_equal(res[k], res0[k], err_msg=k)
    assert rows.shape[0] >= 2 * batch_rows
    centers = res["summary"][..., 0]
    _check_against_oracle(rows, res, frame_of, nbody, batch_rows, levels, centers)


@pytest.mark.parametrize("team,nbody,size", [(4, 2, 64), (16, 2, 64), (4, 3, 32), (16, 3, 128)])
@pytest.mark.parametrize("batch_rows,thin,burn_in", [(1, 1, 0), (5, 3, 7)])
def test_team_kernels_batch_means_match_oracle(gpu, team, nbody, size, batch_rows, thin, burn_in):
    dom, p_frame = _domain(gpu, nbody, size, 2)
    W = 40
    frame_of = (np.arange(W) % 2).astype(np.int32)
    init = p_frame[frame_of]
    n_upd = 7 + 30 * thin
    kw = dict(thin=thin, burn_in=burn_in, team=team, seed=5)
    rows, res = _run(gpu, dom, init, frame_of, [13, n_upd - 13], bm=(batch_rows, 4), **kw)
    rows0, res0 = _run(gpu, dom, init, frame_of, [n_upd], **kw)
    np.testing.assert_array_equal(rows, rows0)
    for k in ("state", "tries", "accepts", "moments", "hist", "summary"):
        np.testing.assert_array_equal(res[k], res0[k], err_msg=k)
    _check_against_oracle(rows, res, frame_of, nbody, batch_rows, 4, res["summary"][..., 0])


def test_state_is_invariant_to_splits_checkpoints_and_chain_formats(gpu):
    dom, p_frame = _domain(gpu, 2, 64, 3)
    W = 3000
    frame_of = (np.arange(W) % 3).astype(np.int32)
    init = p_frame[frame_of]
    bm = (5, 4)
    _, ref = _run(gpu, dom, init, frame_of, [61], bm=bm, fmt="f64")
    cases = [dict(runs=[17, 44]), dict(runs=[17, 20, 24], save_after=1), dict(runs=[61], fmt="f32delta"),
             dict(runs=[30, 31], fmt="events_f64"), dict(runs=[30, 31], fmt="events_f32delta"),
             dict(runs=[9, 52], fmt=None)]
    for c in cases:
        _, res = _run(gpu, dom, init, frame_of, c.pop("runs"), bm=bm, **c)
        np.testing.assert_array_equal(res["walker"], ref["walker"], err_msg=str(c))
        np.testing.assert_array_equal(res["frame"], ref["frame"], err_msg=str(c))
        np.testing.assert_array_equal(res["moments"], ref["moments"], err_msg=str(c))


def test_reset_selftest_and_refusals(gpu):
    torch = gpu["torch"]
    from olpefit_b200 import _lib
    dom, p_frame = _domain(gpu, 2, 64, 1)
    init = np.tile(p_frame[0], (64, 1))
    S = gpu["sampler"].GibbsSampler
    with S(dom, init, seed=3) as s:
        s.enable_sketch(n_bins=512, sep_bin=1e-3, pa_bin=5e-3)
        s.enable_batch_means(2, 3)
        with pytest.raises(_lib.LapfError):
            s.enable_sketch(n_bins=512, sep_bin=1e-3, pa_bin=5e-3)   # would change the quantities
        s.run(23)
        with pytest.raises(_lib.LapfError):
            s.enable_batch_means(2, 3)                                # rows were recorded
        before = s.batch_means()["walker"].clone()
        _lib.check(s.lib.lapf_sampler_selftest(s._h, None))
        assert torch.equal(s.batch_means()["walker"], before)
        assert float(before.abs().sum()) > 0
        blob = s.save()
        s.reset(init, seed=4)
        assert float(s.batch_means()["walker"].abs().sum()) == 0.0
    for other in ((3, 3), (2, 4)):
        with S(dom, init, seed=3) as s:
            s.enable_sketch(n_bins=512, sep_bin=1e-3, pa_bin=5e-3)
            s.enable_batch_means(*other)
            n = s.save().numel()
            with pytest.raises(_lib.LapfError):
                s.load(torch.cat([blob, torch.zeros(max(0, n - blob.numel()), dtype=torch.uint8, device=blob.device)]))
    with S(dom, init, seed=3) as s:                                    # no sketches: C = P + 1
        s.enable_batch_means(2, 3)
        n = s.save().numel()
        with pytest.raises(_lib.LapfError):
            s.load(torch.cat([blob, torch.zeros(max(0, n - blob.numel()), dtype=torch.uint8, device=blob.device)]))
    with S(dom, init, seed=3, burn_in=10) as s:                        # burn-in rows are not recorded
        s.run(9)
        s.enable_batch_means(1, 2)


def test_mcse_predicts_the_spread_of_group_means(gpu):
    """posterior_2body_s64's configuration with 2048 walkers in 64 groups of 32: the standard deviation
    of the group means of separation and position angle is the MCSE predicted for 32 walkers."""
    torch = gpu["torch"]
    from olpefit_b200 import frame, synth
    ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    z = np.load(os.path.join(ROOT, "tests", "golden", "posterior_2body_s64.npz"))
    size, nbody, epoch = int(z["size"]), int(z["nbody"]), int(z["epoch"])
    ox, oy = (int(v) for v in z["origin"])
    domain = str(z["domain"]) if "domain" in z.files else "stamp"
    if domain == "frame":
        img, _ = synth.make_frame(epoch, nbody)
        dom = frame.prepare_domain(img, HEADER, size=size, cut=(ox, oy), nbody=nbody, whole_frame=True)
    else:
        img, _ = synth.make_frame(epoch, nbody, region=(oy, oy + size, ox, ox + size))
        dom = frame.prepare_domain(img, HEADER, origin=(ox, oy), nbody=nbody)
    G, M = 64, 32
    frame_of = np.zeros(G * M, dtype=np.int32)
    with gpu["sampler"].GibbsSampler(dom, np.tile(z["p0"], (G * M, 1)), frame_of, seed=20261020,
                                     burn_in=int(z["burn"]), thin=int(z["thin"])) as s:
        s.enable_sketch(n_bins=4096, sep_bin=1e-3, pa_bin=5e-3)
        s.enable_batch_means(4, 12)
        s.run(int(z["updates"]), record=False)
        bm = s.batch_means()
    rows = bm["rows"]
    P = 16
    w = bm["walker"]                                   # [W, C, L, 2]
    res = gpu["stats"].batch_means_summary({"frame": bm["frame"], "batch_rows": bm["batch_rows"], "levels": bm["levels"]},
                                          torch.tensor([G * M]), rows)
    assert res["batch_rows_used"] is not None
    b = res["batch_rows_used"]
    lv = int(np.log2(b // bm["batch_rows"]))
    j = rows // b
    means = (w[:, P + 1:P + 3, lv, 0] / (j * b)).cpu().numpy()        # mean of the complete batches per walker
    group = means.reshape(G, M, 2).mean(axis=1)
    spread = group.std(axis=0, ddof=1)
    mcse32 = res["mcse"][0, P + 1:P + 3].cpu().numpy() * np.sqrt(G * M / M)
    print("group spread", spread, "mcse(32)", mcse32, "tau", res["tau"][0, P + 1:P + 3].cpu().numpy(),
          "tau levels", res["tau_levels"][0, P + 1:P + 3].cpu().numpy())
    assert np.all(spread >= 0.7 * mcse32) and np.all(spread <= 1.4 * mcse32), (spread, mcse32)


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


def test_cli_ess_min_stops_before_accept_min(tmp_path):
    from olpefit_b200 import cli
    path, out = _write_case(tmp_path, "_ess")
    accept_min = 5000
    assert cli.main_step2([path, "--accept-min", str(accept_min), "--ess-min", "100"] + COMMON) == 0
    summ = json.load(open(os.path.join(out, "step2_summary.json")))
    print("stop", summ["stop"], "ess", summ["sep_pa_companion"]["sep_mas"]["ess"], summ["sep_pa_companion"]["pa_deg"]["ess"])
    assert summ["stop"]["reason"] == "converged"
    assert summ["stop"]["updates"] == summ["updates"] < 16 * accept_min
    assert summ["sep_pa_companion"]["sep_mas"]["ess"] >= 100 and summ["sep_pa_companion"]["pa_deg"]["ess"] >= 100
    assert summ["batch_rows"] >= 64 and set(summ["ess"]) == set(summ["mcse"]) and len(summ["ess"]) == 16
    lengths = {np.genfromtxt(os.path.join(out, "%d_finalarray_mpi.csv" % w), delimiter=",").shape for w in range(8)}
    assert lengths == {(summ["updates"] + 1, 17)}


def test_cli_unmet_ess_min_writes_the_files_of_a_run_without_it(tmp_path):
    from olpefit_b200 import cli
    path_a, out_a = _write_case(tmp_path, "_plain")
    path_b, out_b = _write_case(tmp_path, "_unmet")
    assert cli.main_step2([path_a, "--accept-min", "40"] + COMMON) == 0
    assert cli.main_step2([path_b, "--accept-min", "40", "--ess-min", "1e12"] + COMMON) == 0
    for w in range(8):
        for name in ("%d_finalarray_mpi.csv" % w, "%d_acceptance_rate.csv" % w):
            assert open(os.path.join(out_a, name), "rb").read() == open(os.path.join(out_b, name), "rb").read(), name
    summ = json.load(open(os.path.join(out_b, "step2_summary.json")))
    assert summ["stop"]["reason"] == "accept_min"
    assert "stop" not in json.load(open(os.path.join(out_a, "step2_summary.json")))


def test_cli_mcse_survives_checkpoint_and_resume(tmp_path):
    from olpefit_b200 import cli
    path_a, out_a = _write_case(tmp_path, "_whole")
    assert cli.main_step2([path_a, "--accept-min", "160", "--mcse"] + COMMON) == 0
    path_b, out_b = _write_case(tmp_path, "_parts")
    assert cli.main_step2([path_b, "--accept-min", "70", "--mcse", "--checkpoint"] + COMMON) == 0
    assert cli.main_step2([path_b, "--accept-min", "160", "--mcse", "--resume"] + COMMON) == 0
    sa = json.load(open(os.path.join(out_a, "step2_summary.json")))
    sb = json.load(open(os.path.join(out_b, "step2_summary.json")))
    assert sa["updates"] == sb["updates"]
    assert np.isfinite(sa["sep_pa_companion"]["sep_mas"]["mcse"])
    assert sa["ess"] == sb["ess"] and sa["mcse"] == sb["mcse"] and sa["batch_rows"] == sb["batch_rows"]
    assert sa["sep_pa_companion"] == sb["sep_pa_companion"]
