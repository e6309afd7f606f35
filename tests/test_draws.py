"""Posterior draws (lapf_sampler_draws, include/lapf.h) without a GPU: the numpy restatement of the
reservoir selection that the GPU tests compare the device with, checked against a scalar algorithm R on
the oracle's Philox; its inclusion frequencies and its independence of the update stream; the draws
file round trip; two gloo ranks writing the one-rank file; and the command line's parse-time refusal."""
import os
import socket
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle.lapf_oracle import philox4x32_10  # noqa: E402

MASK = np.uint64(0xFFFFFFFF)
TAG_DRAWS = 0x4C415052   # 'LAPR'
TAG_UPDATES = 0x4C415046  # 'LAPF'


def _philox_np(c0, c1, c2, c3, k0, k1):
    """philox4x32_10 on arrays of uint32 values held in uint64 (broadcasting)."""
    c0, c1, c2, c3, k0, k1 = (np.asarray(v, dtype=np.uint64) & MASK for v in (c0, c1, c2, c3, k0, k1))
    m0, m1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
    w0, w1 = np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)
    s32 = np.uint64(32)
    for _ in range(10):
        p0, p1 = m0 * c0, m1 * c2
        c0, c1, c2, c3 = ((p1 >> s32) ^ c1 ^ k0) & MASK, p1 & MASK, ((p0 >> s32) ^ c3 ^ k1) & MASK, p0 & MASK
        k0, k1 = (k0 + w0) & MASK, (k1 + w1) & MASK
    return c0, c1, c2, c3


def _mulhi64(a, b):
    s32 = np.uint64(32)
    a_lo, a_hi, b_lo, b_hi = a & MASK, a >> s32, b & MASK, b >> s32
    lolo, hilo, lohi, hihi = a_lo * b_lo, a_hi * b_lo, a_lo * b_hi, a_hi * b_hi
    cross = (lolo >> s32) + (hilo & MASK) + (lohi & MASK)
    return hihi + (hilo >> s32) + (lohi >> s32) + (cross >> s32)


def selection_word(seed, gid, n):
    """The 64-bit word r of row n of walker gid (uint64 arrays, broadcasting)."""
    seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    n = np.asarray(n, dtype=np.uint64)
    r0, r1, _, _ = _philox_np(n & MASK, n >> np.uint64(32), np.uint64(seed >> 32), np.uint64(TAG_DRAWS),
                              np.uint64(seed & 0xFFFFFFFF), np.asarray(gid, dtype=np.uint64))
    return r0 | (r1 << np.uint64(32))


def draw_slots(seed, gid, n, K):
    """Reservoir slot (or -1) that recorded row n of walker gid takes among K (int64, broadcasting)."""
    n64 = np.asarray(n, dtype=np.uint64)
    j = _mulhi64(selection_word(seed, gid, n64), n64 + np.uint64(1))
    replaced = np.where(j < np.uint64(K), np.minimum(j, np.uint64(K)).astype(np.int64), -1)
    return np.where(n64 < np.uint64(K), n64.astype(np.int64), replaced)


def reservoir_rows(seed, gids, n_rows, K):
    """[W, K] recorded-row index held by each slot after rows 0 .. n_rows-1 (-1: empty)."""
    gids = np.asarray(gids, dtype=np.uint64)
    out = np.full((gids.size, K), -1, dtype=np.int64)
    w = np.arange(gids.size)
    for n in range(n_rows):
        j = draw_slots(seed, gids, n, K)
        sel = j >= 0
        out[w[sel], j[sel]] = n
    return out


def _scalar_reservoir(seed, gid, n_rows, K, n0=0):
    """Algorithm R with Python integers on the oracle's Philox."""
    slots = [-1] * K
    for n in range(n0, n0 + n_rows):
        if n < K:
            slots[n] = n
            continue
        c = philox4x32_10((n & 0xFFFFFFFF, n >> 32, (seed >> 32) & 0xFFFFFFFF, TAG_DRAWS),
                          (seed & 0xFFFFFFFF, gid & 0xFFFFFFFF))
        j = ((c[0] | (c[1] << 32)) * (n + 1)) >> 64
        if j < K:
            slots[j] = n
    return slots


@pytest.mark.parametrize("seed,K,n_rows", [(7, 1, 40), (0x123456789ABCDEF0, 7, 60), (2 ** 64 - 1, 64, 50)])
def test_vectorised_selection_is_the_scalar_algorithm_r(seed, K, n_rows):
    gids = np.array([0, 1, 2, 5, 77, 65535, 2 ** 32 - 1])
    got = reservoir_rows(seed, gids, n_rows, K)
    want = np.array([_scalar_reservoir(seed, int(g), n_rows, K) for g in gids])
    np.testing.assert_array_equal(got, want)


def test_selection_words_agree_beyond_32_bit_row_indices():
    rng = np.random.default_rng(3)
    n = rng.integers(0, 2 ** 62, size=200, dtype=np.int64)
    gid = rng.integers(0, 2 ** 32, size=200, dtype=np.int64)
    seed = 0xDEADBEEF12345678
    got = draw_slots(seed, gid.astype(np.uint64), n.astype(np.uint64), 2 ** 16)
    for i in range(n.size):
        nn = int(n[i])
        c = philox4x32_10((nn & 0xFFFFFFFF, nn >> 32, seed >> 32, TAG_DRAWS), (seed & 0xFFFFFFFF, int(gid[i])))
        j = ((c[0] | (c[1] << 32)) * (nn + 1)) >> 64
        assert got[i] == (j if j < 2 ** 16 else -1)


def test_every_row_is_kept_with_probability_k_over_n():
    K, n_rows, W = 8, 50, 40000
    res = reservoir_rows(11, np.arange(W), n_rows, K)
    counts = np.bincount(res.reshape(-1), minlength=n_rows)
    p = K / n_rows
    sigma = np.sqrt(W * p * (1 - p))
    assert np.all(np.abs(counts - W * p) < 5 * sigma), (counts, W * p, sigma)
    assert (res >= 0).all() and all(len(set(r)) == K for r in res[:100])


def test_selection_words_are_uncorrelated_with_the_update_uniforms():
    seed, n = 0x0123456789ABCDEF, 200000
    t = np.arange(n, dtype=np.uint64)
    for gid in (0, 12345):
        sel = selection_word(seed, gid, t).astype(np.float64) * 2.0 ** -64
        r0, _, _, r3 = _philox_np(t & MASK, t >> np.uint64(32), np.uint64(seed >> 32), np.uint64(TAG_UPDATES),
                                  np.uint64(seed & 0xFFFFFFFF), np.uint64(gid))
        u = ((r3 << np.uint64(21)) | (r0 & np.uint64(0x1FFFFF))).astype(np.float64) * 2.0 ** -53   # make_draw's uniform
        assert abs(np.corrcoef(sel, u)[0, 1]) < 5 / np.sqrt(n)
        assert abs(sel.mean() - 0.5) < 5 * np.sqrt(1 / 12 / n)


def test_draws_file_round_trips_bit_for_bit(tmp_path):
    from olpefit_b200 import chains
    rng = np.random.default_rng(5)
    W, K, C = 5, 4, 17
    values = rng.normal(size=(W, K, C)) * 10.0 ** rng.integers(-300, 300, size=(W, K, C))
    values[0, 0, :3] = [-0.0, 5e-324, np.finfo(np.float64).max]
    values[1, 2, 4] = np.nan
    rows = np.array([[3, 0, 2, 1], [-1, -1, 7, -1], [0, 1, 2, 3], [9, -1, 4, 6], [-1, -1, -1, -1]])
    walkers = np.array([4, 1, 0, 3, 2])
    names = ["p%d" % i for i in range(C - 1)] + ["chi2"]
    path = str(tmp_path / "step2_draws.csv")
    assert chains.write_draws_csv(path, walkers, values, rows, names) == int((rows >= 0).sum())
    got_names, w, r, v = chains.read_draws_csv(path)
    assert got_names == names
    keys = list(zip(w.tolist(), r.tolist()))
    assert keys == sorted(keys)
    want = {(int(walkers[i]), int(rows[i, k])): values[i, k] for i in range(W) for k in range(K) if rows[i, k] >= 0}
    assert set(keys) == set(want)
    for i, key in enumerate(keys):
        a, b = v[i], want[key]
        assert np.array_equal(np.isnan(a), np.isnan(b))
        np.testing.assert_array_equal(a[~np.isnan(a)].view(np.int64), b[~np.isnan(b)].view(np.int64))
    with open(path) as fh:
        assert fh.readline() == "# " + ",".join(["walker", "row"] + names) + "\n"


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _files(all_v, all_r, n_frames, per_frame, out_dir):
    from olpefit_b200 import chains
    names = ["c%d" % i for i in range(all_v.shape[-1])]
    for f in range(n_frames):
        chains.write_draws_csv(os.path.join(out_dir, "draws_%d.csv" % f), np.arange(per_frame),
                               all_v[f::n_frames], all_r[f::n_frames], names)


def _worker(rank, world, port, in_path, out_dir):
    sys.path.insert(0, ROOT)
    os.environ.update({"RANK": str(rank), "LOCAL_RANK": str(rank), "WORLD_SIZE": str(world),
                       "MASTER_ADDR": "127.0.0.1", "MASTER_PORT": str(port)})
    import torch.distributed as td
    from olpefit_b200 import cli, dist
    dist.init(backend="gloo")
    z = np.load(in_path)
    ids = np.arange(rank, z["values"].shape[0], world)          # dist.shard_ids: rank r owns r, r + world, ...
    n_local = ids.size
    pad = 1 if n_local == 0 else 0                              # a rank without walkers still has a 1-walker sampler
    d = {"values": torch.tensor(np.concatenate([z["values"][ids], np.zeros((pad,) + z["values"].shape[1:])])),
         "rows": torch.tensor(np.concatenate([z["rows"][ids], np.zeros((pad, z["rows"].shape[1]), dtype=np.int64)]))}
    all_v, all_r = cli._gather_draws(d, n_local, rank, world)
    if rank == 0:
        _files(all_v, all_r, int(z["n_frames"]), int(z["per_frame"]), out_dir)
    else:
        assert all_v is None and all_r is None
    td.destroy_process_group()


def test_two_ranks_write_the_one_rank_file(tmp_path):
    import torch.multiprocessing as mp
    from olpefit_b200 import cli
    n_frames, per_frame, K, C = 3, 5, 4, 17
    W = n_frames * per_frame
    rng = np.random.default_rng(9)
    values = rng.normal(size=(W, K, C))
    rows = reservoir_rows(3, np.arange(W), 6, K)
    rows[-4:, 2:] = -1                                          # walkers with fewer rows than slots
    one = tmp_path / "one"
    one.mkdir()
    all_v, all_r = cli._gather_draws({"values": torch.tensor(values), "rows": torch.tensor(rows)}, W, 0, 1)
    _files(all_v, all_r, n_frames, per_frame, str(one))
    two = tmp_path / "two"
    two.mkdir()
    path = str(tmp_path / "in.npz")
    np.savez(path, values=values, rows=rows, n_frames=n_frames, per_frame=per_frame)
    mp.spawn(_worker, args=(2, _free_port(), path, str(two)), nprocs=2, join=True)
    for f in range(n_frames):
        a = open(str(one / ("draws_%d.csv" % f)), "rb").read()
        assert a == open(str(two / ("draws_%d.csv" % f)), "rb").read()
        assert len(a.splitlines()) == 1 + int((rows[f::n_frames] >= 0).sum())


def test_command_line_refuses_draws_below_one_before_any_device_is_touched(monkeypatch, capsys):
    from olpefit_b200 import cli
    import olpefit_b200.dist as dist

    def no_device(*a, **k):
        raise AssertionError("a device was touched")
    monkeypatch.setattr(dist, "init", no_device)
    for k in ("0", "-3"):
        with pytest.raises(SystemExit) as e:
            cli.main_step2(["x.fits", "--draws", k])
        assert e.value.code == 2
        assert "positive integer" in capsys.readouterr().err
    with pytest.raises(SystemExit):
        cli.main_step2a(["x.fits", "--draws", "8"])                # step-2 kinds only
