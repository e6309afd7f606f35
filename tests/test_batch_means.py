"""Batch means on the host (no GPU): a float64 numpy restatement of the per-walker state of
lapf_sampler_batchmeans (include/lapf.h; tests/test_gpu_batch_means.py pins the device to it bit for
bit) and stats.batch_means_summary recover the autocorrelation time of a known process, per-rank
sums combine to the one-rank summary, and the command line refuses what it cannot do before any
device is touched."""
import os
import socket
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def batch_means_state(values, batch_rows, levels):
    """Per-walker batch-mean state from the recorded values [rows, walkers, C], centred as the device
    centres them (chain column minus the walker's starting point; separation / position angle minus
    the sketch centre): the running sum M1 grows row by row, and at every row count that is a
    multiple of b_l = batch_rows * 2^l, S = M1 - snap_l; s2_l = s2_l + S*S; snap_l = M1.
    Returns [walkers, C, levels, 2] = (snap, s2) in float64."""
    v = np.asarray(values, dtype=np.float64)
    rows, walkers, c = v.shape
    m1 = np.zeros((walkers, c))
    out = np.zeros((walkers, c, levels, 2))
    for r in range(rows):
        m1 = m1 + v[r]
        for lv in range(levels):
            if (r + 1) % (batch_rows << lv) == 0:
                s = m1 - out[:, :, lv, 0]
                out[:, :, lv, 1] = out[:, :, lv, 1] + s * s
                out[:, :, lv, 0] = m1
    return out


def batch_means_frame(state, row_var, rows, batch_rows):
    """Per-walker terms of lapf_sampler_batchmeans' frame_out before the sum over walkers: [walkers, C,
    1 + levels] with [..., 0] = ``row_var`` (population variance of each walker's recorded values) and
    [..., 1 + l] = sample variance of its level-l batch means, (s2 - snap^2/J) / (b^2 (J - 1)) with
    J = rows // b complete batches of b = batch_rows * 2^l rows, 0 where J < 2."""
    state = np.asarray(state, dtype=np.float64)
    walkers, c, levels, _ = state.shape
    out = np.zeros((walkers, c, 1 + levels))
    out[..., 0] = row_var
    for lv in range(levels):
        b = batch_rows << lv
        j = rows // b
        if j >= 2:
            snap, s2 = state[:, :, lv, 0], state[:, :, lv, 1]
            out[..., 1 + lv] = (s2 - snap * snap / j) / (float(b) * float(b) * (j - 1.0))
    return out


def _ar1(n_chains, n_rows, phi, seed):
    rng = np.random.default_rng(seed)
    e = rng.standard_normal((n_rows, n_chains))
    x = np.empty((n_rows, n_chains))
    x[0] = e[0] / np.sqrt(1.0 - phi * phi)
    for t in range(1, n_rows):
        x[t] = phi * x[t - 1] + e[t]
    return x


def _frame_sums(values, batch_rows, levels, groups):
    """lapf_sampler_batchmeans' frame_out restated from values [rows, walkers, C]: walker w in frame groups[w]."""
    st = batch_means_state(values, batch_rows, levels)
    per_w = batch_means_frame(st, values.var(axis=0), values.shape[0], batch_rows)
    n_frames = int(groups.max()) + 1
    return np.stack([per_w[groups == f].sum(axis=0) for f in range(n_frames)]), st


def test_ar1_autocorrelation_time_is_recovered():
    from olpefit_b200 import stats
    phi, rows, chains = 0.9, 1 << 16, 256
    tau_true = (1.0 + phi) / (1.0 - phi)                    # 19
    x = _ar1(chains, rows, phi, 1)
    frame, _ = _frame_sums(x[:, :, None], 16, 12, np.zeros(chains, dtype=int))
    bm = {"frame": torch.tensor(frame), "batch_rows": 16, "levels": 12}
    res = stats.batch_means_summary(bm, torch.tensor([chains]), rows)
    tau = float(res["tau"][0, 0])
    assert tau == pytest.approx(tau_true, rel=0.10), res["tau_levels"]
    assert float(res["ess"][0, 0]) == pytest.approx(chains * rows / tau)
    # the pooled mean's standard error is the one of the process: sqrt(tau var / (M n))
    var = 1.0 / (1.0 - phi * phi)
    assert float(res["mcse"][0, 0]) == pytest.approx(np.sqrt(tau_true * var / (chains * rows)), rel=0.1)
    b = res["batch_rows_used"]
    assert rows // b >= 20 and rows // (2 * b) < 20
    lv = res["tau_levels"][0, 0].numpy()
    assert np.isnan(lv[-1]) and np.all(np.isfinite(lv[: int(np.log2(b // 16)) + 1]))


def test_oracle_state_is_split_invariant_and_no_level_is_nan():
    from olpefit_b200 import stats
    x = _ar1(3, 100, 0.5, 2)[:, :, None]
    st = batch_means_state(x, 5, 3)
    # snap of level l = sum of the first J_l * b_l values
    for lv, b in enumerate((5, 10, 20)):
        j = 100 // b
        np.testing.assert_allclose(st[:, 0, lv, 0], x[: j * b, :, 0].sum(axis=0), rtol=1e-12)
        sums = x[: j * b, :, 0].reshape(j, b, 3).sum(axis=1)
        np.testing.assert_allclose(st[:, 0, lv, 1], (sums ** 2).sum(axis=0), rtol=1e-12)
    frame, _ = _frame_sums(x, 5, 3, np.zeros(3, dtype=int))
    res = stats.batch_means_summary({"frame": torch.tensor(frame), "batch_rows": 5, "levels": 3},
                                    torch.tensor([3]), 100, min_batches=200)
    assert res["batch_rows_used"] is None and bool(torch.isnan(res["ess"]).all())


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, frame_path, out_dir):
    sys.path.insert(0, ROOT)
    os.environ.update({"RANK": str(rank), "LOCAL_RANK": str(rank), "WORLD_SIZE": str(world),
                       "MASTER_ADDR": "127.0.0.1", "MASTER_PORT": str(port)})
    import torch.distributed as td
    from olpefit_b200 import dist, stats
    dist.init(backend="gloo")
    z = np.load(frame_path)
    mine = z["per_rank"][rank]
    frame = dist.allreduce_sum(torch.tensor(mine))
    m = dist.allreduce_sum(torch.tensor(z["walkers_rank"][rank], dtype=torch.float64))
    res = stats.batch_means_summary({"frame": frame, "batch_rows": 4, "levels": 6}, m, int(z["rows"]))
    if rank == 0:
        np.savez(os.path.join(out_dir, "r0.npz"), ess=res["ess"].numpy(), mcse=res["mcse"].numpy(),
                 tau=res["tau"].numpy())
    td.destroy_process_group()


def test_ranks_combine_to_the_one_rank_summary(tmp_path):
    import torch.multiprocessing as mp
    from olpefit_b200 import stats
    rows, walkers, frames = 512, 24, 3
    x = np.stack([_ar1(walkers, rows, 0.6, 3), _ar1(walkers, rows, 0.8, 4)], axis=-1)
    groups = np.arange(walkers) % frames
    whole, _ = _frame_sums(x, 4, 6, groups)
    one = stats.batch_means_summary({"frame": torch.tensor(whole), "batch_rows": 4, "levels": 6},
                                    torch.tensor(np.bincount(groups)), rows)
    # two ranks own the walkers g = rank (mod 2), as dist.shard_ids deals them
    per_rank, wr = [], []
    for r in range(2):
        sel = np.arange(walkers) % 2 == r
        st = batch_means_state(x[:, sel], 4, 6)
        per_w = batch_means_frame(st, x[:, sel].var(axis=0), rows, 4)
        g = groups[sel]
        per_rank.append(np.stack([per_w[g == f].sum(axis=0) for f in range(frames)]))
        wr.append(np.bincount(g, minlength=frames).astype(np.float64))
    path = str(tmp_path / "in.npz")
    np.savez(path, per_rank=np.stack(per_rank), walkers_rank=np.stack(wr), rows=rows)
    mp.spawn(_worker, args=(2, _free_port(), path, str(tmp_path)), nprocs=2, join=True)
    r0 = np.load(str(tmp_path / "r0.npz"))
    for k in ("ess", "mcse", "tau"):
        np.testing.assert_allclose(r0[k], one[k].numpy(), rtol=1e-12, err_msg=k)


def test_command_line_refusals_happen_before_any_device_is_touched(monkeypatch):
    from olpefit_b200 import cli
    import olpefit_b200.dist as dist

    def no_device(*a, **k):
        raise AssertionError("a device was touched")
    monkeypatch.setattr(dist, "init", no_device)
    with pytest.raises(SystemExit) as e:
        cli.main_step2(["x.fits", "--walkers", "1", "--rhat-max", "1.1"])
    assert "2 walkers" in str(e.value)
    for flag in (["--ess-min", "100"], ["--rhat-max", "1.1"], ["--mcse"]):
        with pytest.raises(SystemExit):
            cli.main_step2a(["x.fits"] + flag)
