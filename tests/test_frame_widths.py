"""Per-epoch jump widths (lapf_sampler_adapt_widths, include/lapf.h) without a GPU: the numpy restatement
of the adaptation rule that the GPU tests compare the device with, its properties (a window without
tries keeps the width, a rate on target leaves it bit for bit, the factor is clipped to [0.5, 2], windows
are differences of cumulative counts), and the command line's parse-time refusals."""
import numpy as np
import pytest


def adapt_rule(widths, counts, snap, target):
    """One adaptation step: (new widths [F, P], new snapshot [F, P, 2]) from cumulative counts [F, P, 2]
    (tries, accepts) and the snapshot of the previous step.  Division, subtraction and product are
    float64 operations rounded to nearest, as on the device."""
    w = np.array(widths, dtype=np.float64)
    counts = np.asarray(counts, dtype=np.int64)
    dt = counts[..., 0] - snap[..., 0]
    da = counts[..., 1] - snap[..., 1]
    live = dt > 0
    rate = da[live].astype(np.float64) / dt[live].astype(np.float64)
    w[live] = w[live] * np.minimum(np.maximum(np.exp(rate - target), 0.5), 2.0)
    return w, counts.copy()


def _case(seed=1, F=3, P=16):
    rng = np.random.default_rng(seed)
    w0 = rng.uniform(1e-3, 1.0, size=(F, P))
    tries = rng.integers(0, 5000, size=(F, P))
    acc = rng.integers(0, tries + 1)
    return w0, np.stack([tries, acc], axis=-1)


def test_a_window_without_tries_keeps_the_width():
    w0, c = _case()
    c[0, 3] = [0, 0]
    c[2, :] = 0
    w, snap = adapt_rule(w0, c, np.zeros_like(c), 0.35)
    np.testing.assert_array_equal(w[0, 3], w0[0, 3])
    np.testing.assert_array_equal(w[2], w0[2])
    np.testing.assert_array_equal(snap, c)
    w2, _ = adapt_rule(w, c, snap, 0.35)                         # nothing new since the snapshot: nothing moves
    np.testing.assert_array_equal(w2, w)


def test_a_rate_on_target_leaves_the_width_bit_for_bit():
    w0, _ = _case()
    tries = np.full(w0.shape, 400)
    c = np.stack([tries, tries // 4], axis=-1)                   # 100 / 400 = 0.25 exactly
    w, _ = adapt_rule(w0, c, np.zeros_like(c), 0.25)
    assert np.array_equal(w.view(np.int64), w0.view(np.int64))


def test_the_factor_is_clipped_to_half_and_double():
    w0, _ = _case()
    tries = np.full(w0.shape, 1000)
    # at target 0.35 the factor stays inside the clip: exp(1 - 0.35) = 1.92, exp(0 - 0.35) = 0.70
    for acc, lo, hi in ((tries, 1.91, 1.92), (0 * tries, 0.70, 0.71)):
        c = np.stack([tries, acc], axis=-1)
        w, _ = adapt_rule(w0, c, np.zeros_like(c), 0.35)
        assert np.all((w / w0 > lo) & (w / w0 < hi))
    c = np.stack([tries, tries], axis=-1)
    w, _ = adapt_rule(w0, c, np.zeros_like(c), -1.0)             # exp(2) = 7.4 -> 2
    np.testing.assert_array_equal(w, w0 * 2.0)
    c = np.stack([tries, 0 * tries], axis=-1)
    w, _ = adapt_rule(w0, c, np.zeros_like(c), 0.99)             # exp(-0.99) = 0.37 -> 0.5
    np.testing.assert_array_equal(w, w0 * 0.5)


def test_windows_are_differences_of_cumulative_counts():
    w0, c1 = _case(2)
    _, extra = _case(3)
    c2 = c1 + extra                                              # cumulative: the second window holds `extra`
    w1, s1 = adapt_rule(w0, c1, np.zeros_like(c1), 0.35)
    w2, s2 = adapt_rule(w1, c2, s1, 0.35)
    w_direct, _ = adapt_rule(w1, extra, np.zeros_like(extra), 0.35)
    np.testing.assert_array_equal(w2, w_direct)
    np.testing.assert_array_equal(s2, c2)
    # the window's own rate decides, not the cumulative one
    f, j = np.unravel_index(np.argmax(np.abs(extra[..., 1] / np.maximum(extra[..., 0], 1) - c2[..., 1] / np.maximum(c2[..., 0], 1))), w0.shape)
    rate = extra[f, j, 1] / extra[f, j, 0]
    assert w2[f, j] == w1[f, j] * min(max(np.exp(rate - 0.35), 0.5), 2.0)


def _no_device(monkeypatch):
    import olpefit_b200.dist as dist

    def no_device(*a, **k):
        raise AssertionError("a device was touched")
    monkeypatch.setattr(dist, "init", no_device)


def test_command_line_refuses_adapt_per_epoch_with_adapt_before_any_device_is_touched(monkeypatch):
    from olpefit_b200 import cli
    _no_device(monkeypatch)
    with pytest.raises(SystemExit) as e:
        cli.main_step2(["x.fits", "--adapt-per-epoch", "--adapt"])
    assert "--adapt" in str(e.value.code)


def test_command_line_refuses_adapt_per_epoch_without_burn_in_before_any_device_is_touched(monkeypatch):
    from olpefit_b200 import cli
    _no_device(monkeypatch)
    for run, argv in ((cli.main_step2, ["x.fits", "--adapt-per-epoch", "--burn-in", "0"]),
                      (cli.main_step2_3body, ["x.fits", "--adapt-per-epoch"])):      # the 3-body default burn-in is 0
        with pytest.raises(SystemExit) as e:
            run(argv)
        assert "burn-in" in str(e.value.code)
    with pytest.raises(SystemExit) as e:
        cli.main_step2a(["x.fits", "--adapt-per-epoch", "--burn-in", "100"])          # step-2 kinds only
    assert e.value.code == 2
