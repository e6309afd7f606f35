"""Parameter priors (lapf_sampler_set_priors, include/lapf.h) without a GPU: the numpy restatement of the
accept rule that the GPU tests compare the device with (h computed as on the host, g and the threshold
rounded as on the device), an oracle loop with that rule, the Python table builder, and the command
line's --prior file: parsing, the merge of "all" and "epochs", every parse-time refusal, the start check
and the summary block."""
import json
import math

import numpy as np
import pytest

from oracle import lapf_oracle as orc


def h_of(sigma):
    """h = 0.5 / sigma^2 as lapf_sampler_set_priors computes it on the host; 0 for sigma = +inf (no term)."""
    sigma = np.asarray(sigma, dtype=np.float64)
    with np.errstate(divide="ignore"):
        return np.where(np.isinf(sigma), 0.0, 0.5 / (sigma * sigma))


def prior_g(entry, nv, pk):
    """The Gaussian term of a move pk -> nv under entry {lo, hi, mu, sigma}: h ((nv - mu)^2 - (pk - mu)^2),
    0 where h = 0.  numpy's float64 operations round each result to nearest and never fuse, like the
    device's __dsub_rn / __dmul_rn."""
    h = float(h_of(entry[3]))
    if h == 0.0:
        return 0.0
    dn, dp = np.float64(nv) - np.float64(entry[2]), np.float64(pk) - np.float64(entry[2])
    return float(np.float64(h) * (dn * dn - dp * dp))


def threshold(chi_t, chi_c, g):
    """The right side of the accept test ln u < -0.5 (chi_t - chi_c) - g."""
    return float(np.float64(-0.5) * (np.float64(chi_t) - np.float64(chi_c)) - np.float64(g))


def outside(entry, v):
    """A proposal outside the box (nan is outside every box) is rejected without a trial chi-square."""
    return not (entry[0] <= v <= entry[1])


def run_chain_with_prior(data, weight, layout, p0, stream, table_f, *, origin, n_updates):
    """oracle.run_chain (apf_step2.py:276-351, burn-in 0, thin 1) with the prior in its accept rule: a proposal
    outside its box is a try and a reject; otherwise accept iff ln u < threshold(chi_t, chi_c, g).
    Returns (rows [n_updates, P+1], tries, accepts, trace of (k, new, chi_t, g, ok))."""
    ny, nx = data.shape
    grid = orc.pixel_grid(ny, nx, origin)
    npar = layout.nparam
    is_log = layout.is_log()
    w = np.asarray(layout.widths, dtype=np.float64)

    def chi2(q):
        with np.errstate(all="ignore"):
            return orc.chi_squared_weighted(data, orc.model_image(q, layout, ny, nx, grid=grid), weight)

    p = np.array(p0, dtype=np.float64)
    chi = chi2(p)
    tries, accepts = np.zeros(npar, dtype=np.int64), np.zeros(npar, dtype=np.int64)
    rows, trace = [], []
    for t in range(n_updates):
        k = stream.draw_index(t, npar)
        tries[k] += 1
        new = orc.propose(stream, t, p[k], w[k], is_log[k])
        u = stream.draw_uniform(t)
        if outside(table_f[k], new):
            chi_t, g, ok = float("nan"), 0.0, False
        else:
            trial = p.copy()
            trial[k] = new
            chi_t = chi2(trial)
            g = prior_g(table_f[k], new, p[k])
            ok = bool(math.log(u) < threshold(chi_t, chi, g))
        if ok:
            accepts[k] += 1
            p[k] = new
            chi = chi_t
        trace.append((k, new, chi_t, g, ok))
        rows.append(np.concatenate([p, [chi]]))
    return np.array(rows), tries, accepts, trace


# -- the rule -------------------------------------------------------------------------------------
def test_h_is_computed_as_on_the_host():
    assert h_of(np.inf) == 0.0
    assert h_of(2.0) == 0.125
    s = 0.1
    assert h_of(s) == 0.5 / (s * s)


def test_without_a_term_g_is_zero_even_for_huge_proposals():
    e = (-np.inf, np.inf, 0.0, np.inf)
    assert prior_g(e, 1e308, 3.0) == 0.0                          # h = 0 is never multiplied: 0 * inf would be nan
    assert prior_g(e, np.inf, 3.0) == 0.0
    rng = np.random.default_rng(3)
    for chi_t, chi_c in rng.normal(1e4, 50.0, size=(200, 2)):
        a = threshold(chi_t, chi_c, 0.0)
        b = -0.5 * (chi_t - chi_c)
        assert np.float64(a).view(np.int64) == np.float64(b).view(np.int64)


def test_g_is_the_change_of_the_gaussian_log_density():
    e = (-np.inf, np.inf, 6.4, 0.5)
    assert prior_g(e, 6.4, 6.4) == 0.0
    assert prior_g(e, 6.9, 6.4) == pytest.approx(2.0 * 0.25, rel=1e-12)          # one sigma away: +0.5 nats
    assert prior_g(e, 6.4, 6.9) == pytest.approx(-0.5, rel=1e-12)
    # moving towards mu lowers the threshold's penalty: accepted where the bare ratio would not be
    assert threshold(100.2, 100.0, prior_g(e, 6.4, 7.4)) > threshold(100.2, 100.0, 0.0)


def test_g_and_the_threshold_are_rounded_per_operation():
    # the unfused forms differ from a fused multiply-add in the last bit on some inputs; the restatement
    # must be the unfused one (DESIGN.md 5)
    rng = np.random.default_rng(11)
    for _ in range(500):
        mu, sg = rng.normal(0, 10), rng.uniform(1e-3, 10)
        nv, pk = mu + rng.normal(0, 3 * sg), mu + rng.normal(0, 3 * sg)
        e = (-np.inf, np.inf, mu, sg)
        h = 0.5 / (sg * sg)
        dn, dp = nv - mu, pk - mu
        want = h * ((dn * dn) - (dp * dp))
        assert np.float64(prior_g(e, nv, pk)).view(np.int64) == np.float64(want).view(np.int64)


def test_the_box_includes_its_ends_and_refuses_nan():
    e = (0.0, 1.0, 0.0, np.inf)
    assert not outside(e, 0.0) and not outside(e, 1.0) and not outside(e, 0.5)
    assert outside(e, -1e-300) and outside(e, 1.0000000000000002) and outside(e, float("nan"))
    assert not outside((-np.inf, np.inf, 0.0, np.inf), np.inf)   # an infinite box skips only nan


def test_the_oracle_loop_with_a_neutral_table_is_the_oracle():
    from olpefit_b200 import synth
    lay = orc.layout_for(2)
    stamps, origins = synth.make_stamps(1, 32, 2)
    img = stamps[0].astype(np.float64)
    w = orc.weight_map(img, {"itime": 1.0, "coadds": 1, "multisam": 1, "sampmode": 2})
    p0 = synth.truth_parameters(2, 0)
    table = np.tile([-np.inf, np.inf, 0.0, np.inf], (lay.nparam, 1))
    rows, tries, accepts, _ = run_chain_with_prior(img, w, lay, p0, orc.PhiloxStream(5, 3, lay.nparam), table,
                                                   origin=tuple(origins[0]), n_updates=40)
    ref = orc.run_chain(img, w, lay, p0, orc.PhiloxStream(5, 3, lay.nparam), origin=tuple(origins[0]), n_updates=40)
    np.testing.assert_array_equal(tries, ref.tries)
    np.testing.assert_array_equal(accepts, ref.accepts)
    np.testing.assert_array_equal(rows, ref.rows[1:])


# -- the Python table --------------------------------------------------------------------------------
def test_prior_table_broadcasts_and_fills_none():
    from olpefit_b200.sampler import prior_table
    t = prior_table(3, 4, lo=[0, 1, 2, 3], sigma=np.full((3, 4), 2.0))
    assert t.shape == (3, 4, 4)
    np.testing.assert_array_equal(t[..., 0], np.tile([0, 1, 2, 3], (3, 1)))
    assert np.all(t[..., 1] == np.inf) and np.all(t[..., 2] == 0.0) and np.all(t[..., 3] == 2.0)
    with pytest.raises(ValueError):
        prior_table(3, 4, hi=[1, 2])


# -- the command line's file ---------------------------------------------------------------------------
def _write(tmp_path, spec):
    p = tmp_path / "prior.json"
    p.write_text(json.dumps(spec) if not isinstance(spec, str) else spec)
    return str(p)


EPOCHS = ["29966", "30001"]


def test_parse_merges_all_and_epochs(tmp_path):
    from olpefit_b200 import cli, layout
    names = list(layout.names(2))
    spec = {"all": {"ampratio": {"min": 0, "max": 1}, "bkgd": {"min": 0}, "sigmax2": {"mean": 6.4, "sigma": 0.5},
                    "xcc": {"min": 100.0}},
            "epochs": {"29966": {"xcc": {"min": 519.0, "max": 524.0}}}}
    t = cli.load_prior_file(_write(tmp_path, spec), 2, EPOCHS)
    assert t.shape == (2, 16, 4)
    j = names.index
    for f in range(2):
        np.testing.assert_array_equal(t[f, j("ampratio")], [0, 1, 0, np.inf])
        np.testing.assert_array_equal(t[f, j("bkgd")], [0, np.inf, 0, np.inf])
        np.testing.assert_array_equal(t[f, j("sigmax2")], [-np.inf, np.inf, 6.4, 0.5])
        np.testing.assert_array_equal(t[f, j("xcs")], [-np.inf, np.inf, 0, np.inf])
    np.testing.assert_array_equal(t[0, j("xcc")], [519.0, 524.0, 0, np.inf])       # the epoch's entry replaces "all"
    np.testing.assert_array_equal(t[1, j("xcc")], [100.0, np.inf, 0, np.inf])
    s0 = cli.prior_summary(t[0], 2)
    assert set(s0) == {"ampratio", "bkgd", "sigmax2", "xcc"}
    assert s0["xcc"] == {"min": 519.0, "max": 524.0, "mean": None, "sigma": None}
    assert s0["sigmax2"] == {"min": None, "max": None, "mean": 6.4, "sigma": 0.5}
    assert s0["bkgd"] == {"min": 0.0, "max": None, "mean": None, "sigma": None}
    json.dumps(s0, allow_nan=False)                                 # plain JSON: no Infinity
    assert cli.prior_summary(cli.load_prior_file(_write(tmp_path, {}), 2, EPOCHS)[0], 2) == {}


@pytest.mark.parametrize("spec,message", [
    ({"all": {"nope": {"min": 0}}}, "unknown parameter 'nope'"),
    ({"all": {"bkgd": {"lo": 0}}}, "unknown key 'lo'"),
    ({"epochs": {"12345": {"bkgd": {"min": 0}}}}, "unknown epoch '12345'"),
    ({"all": {"ampratio": {"min": 1, "max": 1}}}, "min 1 >= max 1"),
    ({"all": {"ampratio": {"min": 2, "max": 1}}}, "min 2 >= max 1"),
    ({"all": {"sigmax": {"mean": 1, "sigma": 0}}}, "sigma 0 <= 0"),
    ({"all": {"sigmax": {"mean": 1, "sigma": -2}}}, "sigma -2 <= 0"),
    ({"all": {"sigmax": {"mean": 1}}}, "mean and sigma together"),
    ({"all": {"sigmax": {"sigma": 1}}}, "mean and sigma together"),
    ({"all": {"sigmax": {"min": "a"}}}, "is not a finite number"),
    ({"priors": {}}, "\"all\" and \"epochs\" only"),
    ({"epochs": {"29966": {"ycc": 3}}}, "must be an object"),
    ("{not json", "--prior"),
])
def test_parse_refusals(tmp_path, spec, message):
    from olpefit_b200 import cli
    with pytest.raises(SystemExit) as e:
        cli.load_prior_file(_write(tmp_path, spec), 2, EPOCHS)
    assert message in str(e.value), str(e.value)


def test_refusals_reach_the_command_line_before_the_gpu(tmp_path):
    from olpefit_b200 import cli
    img = tmp_path / "n0001.29966.fits.gz"
    with pytest.raises(SystemExit) as e:
        cli.run("step2", 2, [str(img), "--prior", _write(tmp_path, {"all": {"xyz": {"min": 0}}})])
    assert "unknown parameter 'xyz'" in str(e.value)


def test_start_check_names_the_epoch_and_the_parameter():
    from olpefit_b200 import cli, layout
    t = np.tile([-np.inf, np.inf, 0.0, np.inf], (2, 16, 1))
    starts = np.ones((2, 16))
    cli.check_prior_starts(t, starts, 2, EPOCHS)
    t[1, layout.names(2).index("ampratio"), :2] = [0.0, 0.5]
    with pytest.raises(SystemExit) as e:
        cli.check_prior_starts(t, starts, 2, EPOCHS)
    assert "epoch 30001" in str(e.value) and "ampratio" in str(e.value)
