"""No GPU: the PSIS-LOO definition of literate_b200.loo (K12's) on hand cases, the GPD fit on draws of known shape, the global
and comparison standard errors, compare's refusals, the refusal of imputation replicates, and the command line's refusals and
file names."""
import math
import os

import numpy as np
import pytest
from scipy import stats

from literate_b200 import loo as LO


def _lse(x):
    m = np.max(x)
    return m + math.log(np.sum(np.exp(x - m)))


def test_short_tail_is_left_unsmoothed():
    """20 draws, r_eff 1: M = ceil(min(4, 13.4)) = 4, so T <= 4, k_hat = +inf and lw = x - logsumexp(x)."""
    x = np.random.default_rng(0).normal(size=20)
    lw, k, T = LO.psis_host(x, 1.0)
    assert k == math.inf and T == 4
    np.testing.assert_array_equal(lw, (x - x.max()) - _lse(x - x.max()))


def test_ties_at_the_cutoff_shorten_the_tail():
    """1000 draws, r_eff 1: M = 95; places 884 .. 933 hold the order statistic at S - M - 1 = 904, so the tail is the 66 draws
    above them, not 95."""
    rng = np.random.default_rng(1)
    x = np.sort(rng.normal(size=1000))
    x[1000 - 95 - 1 - 20:1000 - 95 - 1 + 30] = x[1000 - 95 - 1]
    rng.shuffle(x)
    lw, k, T = LO.psis_host(x, 1.0)
    assert T == 1000 - 934 and math.isfinite(k)
    assert abs(_lse(lw)) < 1e-12


def test_constant_column():
    """Equal draws: every x is 0 = the cutoff, the tail is empty, k_hat = +inf and the weights uniform."""
    lw, k, T = LO.psis_host(np.full(500, -3.25), 1.0)
    assert T == 0 and k == math.inf
    np.testing.assert_allclose(lw, -math.log(500), rtol=1e-15)


def test_smoothed_tail_is_truncated_at_zero(monkeypatch):
    """A fit whose quantiles rise above the largest draw (k 0.9, sigma 10): those tail values are truncated at 0 and tie."""
    monkeypatch.setattr(LO, "gpdfit_host", lambda y: (0.9, 10.0))
    x = np.random.default_rng(2).normal(size=2000)
    lw, k, T = LO.psis_host(x, 1.0)
    p = (np.arange(0.5, T) / T)[-1]
    assert math.log(np.expm1(-0.9 * np.log1p(-p)) / 0.9 * 10.0) > 0.0
    top = lw == lw.max()
    assert top.sum() >= 2 and lw.max() == pytest.approx(-_lse(lw - lw.max()), abs=1e-12)


def test_near_zero_k_uses_the_exponential_inverse(monkeypatch):
    """|k_hat| < eps: the tail becomes log(-log1p(-p) sigma + exp(cutoff))."""
    monkeypatch.setattr(LO, "gpdfit_host", lambda y: (1e-17, 0.5))
    x = np.random.default_rng(3).normal(size=2000)
    lw, k, T = LO.psis_host(x, 1.0)
    xs = x - x.max()
    cutoff = np.sort(xs)[2000 - 135 - 1]
    order = np.argsort(xs)[-T:]
    want = np.log(-np.log1p(-(np.arange(0.5, T) / T)) * 0.5 + math.exp(cutoff))
    want[want > 0] = 0
    full = xs.copy()
    full[order] = want
    np.testing.assert_allclose(lw, full - _lse(full), rtol=1e-14, atol=1e-14)
    assert T == 135


@pytest.mark.parametrize("k", [0.1, 0.3, 0.5, 0.7])
def test_gpdfit_recovers_the_shape(k):
    """10^5 GPD(k, sigma 2) draws: k_hat within 4 sampling sd of k; the estimator's asymptotic sd is (1 + k) / sqrt(n) (the
    GPD's Fisher information for k < 1/2, larger beyond it, so the bound stays conservative near 0.7 at this n)."""
    n = 100_000
    y = np.sort(stats.genpareto.rvs(k, scale=2.0, size=n, random_state=np.random.default_rng(int(k * 10))))
    kh, sigma = LO.gpdfit_host(y)
    sd = (1 + k) / math.sqrt(n)
    assert abs(kh - k) < 4 * sd, (kh, k, sd)
    assert abs(sigma - 2.0) < 0.05


def _result(elpd, A=None, n=1000, kind="forward", khat=None):
    elpd = np.asarray(elpd, float)
    nb = len(elpd) // 2
    out = np.full((9, 2, nb), np.nan)
    out[0] = (np.arange(2 * nb) + 3.0).reshape(2, nb) if A is None else np.asarray(A, float).reshape(2, nb)
    out[2] = elpd.reshape(2, nb)
    out[1] = out[2] + 0.5
    out[3] = 0.5
    out[4] = out[2] - 0.1
    out[5] = 0.6
    out[6] = 0.2 if khat is None else np.asarray(khat, float).reshape(2, nb)
    out[7] = 1.0
    out[8] = 50
    return LO.LooResult(kind, 10.0, out, n, np.zeros(2, np.int64))


def test_global_se_and_compare_se_diff():
    """se = sqrt(n var(pointwise, ddof 0)); se_diff the same of the differences; the best model ranks first with 0 difference."""
    a = [-1.0, -2.0, -3.0, -4.5]
    b = [-1.5, -2.0, -3.5, -4.0]
    ra, rb = _result(a), _result(b)
    g = ra.global_row()
    assert g[0] == 4 and g[2] == -10.5 and g[4] == 2.0
    assert g[3] == pytest.approx(math.sqrt(4 * np.var(a)), rel=1e-15)
    rows = LO.compare([rb, ra], ["b", "a"])
    assert [r[1] for r in rows] == ["a", "b"] and rows[0][5] == 0.0 and rows[0][6] == 0.0
    d = np.array(a) - np.array(b)
    assert rows[1][5] == pytest.approx(0.5) and rows[1][6] == pytest.approx(math.sqrt(4 * np.var(d)), rel=1e-15)


def test_k_threshold_and_flags():
    r = _result([-1.0, -2.0, -3.0, -4.0, -5.0, -6.0], khat=[0.1, 0.69, math.inf, 0.8, math.nan, -math.inf], n=10 ** 6)
    assert r.threshold() == pytest.approx(min(1 - 1 / 6, 0.7))
    assert [row[11] for row in r.table()] == ["ok", "ok", "k_inf", "k_high", "k_inf", "k_inf"]      # a NaN fit is never "ok"
    assert r.global_row()[8] == 4
    r.out[:, 0, 1] = np.nan
    assert r.table()[1][11] == "none" and r.global_row()[0] == 5


def test_compare_refusals():
    """Different bin counts, column sets or counts A are refused; different exposures (not part of the result) are not."""
    base = _result([-1.0, -2.0, -3.0, -4.0])
    with pytest.raises(ValueError, match="bins"):
        LO.compare([base, _result([-1.0] * 6)], ["a", "b"])
    other = _result([-1.0, -2.0, -3.0, -4.0])
    other.out[:, 1, 0] = np.nan
    with pytest.raises(ValueError, match="columns"):
        LO.compare([base, other], ["a", "b"])
    A = base.out[0].ravel().copy()
    A[3] = np.nextafter(A[3], 10.0)
    with pytest.raises(ValueError, match="counts"):
        LO.compare([base, _result([-1.0, -2.0, -3.0, -4.0], A=A)], ["a", "b"])
    assert len(LO.compare([base, _result([-1.1, -2.0, -3.0, -4.0])], ["a", "b"])) == 2
    with pytest.raises(ValueError):
        LO.compare([base], ["a"])


def test_mixed_replicates_are_refused():
    assert LO.one_table(None, 1) == 0 and LO.one_table([2, 2, 2], 3) == 2
    with pytest.raises(ValueError, match="one table"):
        LO.one_table([0, 1, 0], 2)
    with pytest.raises(ValueError, match="one table"):
        LO.loo_records_device(None, np.zeros((8, 2, 144)), "forward", np.ones((2, 4, 5)), rep_of_chain=[0, 1])


def test_pointwise_is_the_poisson_log_pmf():
    """l of dense records is scipy's Poisson logpmf of A at r B, 0 where B = 0; A = 0 at r = 0 gives 0 (0 log 0 = 0)."""
    nb = 5
    rng = np.random.default_rng(4)
    rec = np.zeros((4, 3, 16 + 2 * nb))
    rec[..., 0] = np.arange(4)[:, None]
    rec[..., 16:] = rng.uniform(0.1, 0.5, (4, 3, 2 * nb))
    A = np.array([[3, 0, 7, 1, 2], [0, 4, 4, 9, 1]], float)
    B = np.array([[10, 5, 0, 8, 3], [6, 2, 9, 30, 4]], float)
    terms = np.stack([A[0], B[0], A[1], B[1]])
    rec[1, 1, 16 + 1] = 0.0
    ll, act, used, status = LO.pointwise_host(rec, 1, nb, terms, rate_col=16)
    assert used.all() and status.tolist() == [0, 0]
    rates = rec[..., 16:].reshape(4, 3, 2, nb)
    want = np.where(B > 0, stats.poisson.logpmf(A, rates * B), 0.0)
    np.testing.assert_allclose(ll, want, rtol=1e-13, atol=1e-13)
    assert ll[1, 1, 0, 1] == 0.0
    rec[2, 0, 16] = 0.0                                    # A = 3 at rate 0: l = -inf, the record is not used
    _, _, used, status = LO.pointwise_host(rec, 1, nb, terms, rate_col=16)
    assert not used[2, 0] and used.sum() == 11 and status.tolist() == [1, 0]


def test_write_tsv_names(tmp_path):
    r = _result([-1.0, -2.0, -3.0, -4.0], kind="dd")
    paths = r.write_tsv(str(tmp_path))
    assert [os.path.basename(p) for p in paths] == ["loo_dd.tsv", "loo_dd_global.tsv"]
    lines = open(paths[0]).read().splitlines()
    assert lines[0].split("\t")[-1] == "flag" and len(lines) == 5 and lines[1].split("\t")[:2] == ["birth", "10.0"]
    p = LO.write_compare(str(tmp_path / "loo_compare.tsv"), LO.compare([r, _result([-1.0, -2.5, -3.0, -4.0])], ["x", "y"]))
    assert open(p).readline().rstrip("\n").split("\t") == list(LO.COMPARE_HEAD)


def _touch(path, head="it\tlikelihood\n"):
    with open(path, "w") as fh:
        fh.write(head)


def test_command_line_refusals(tmp_path):
    """Refused before any device is opened: a missing directory, one named twice, no logs, TrendRate logs, and a directory whose
    RJMCMC logs have two stems (two runs, e.g. two -out, on one table)."""
    with pytest.raises(SystemExit, match="not a directory"):
        LO.main([str(tmp_path / "nope")])
    empty = tmp_path / "empty"
    empty.mkdir()
    with pytest.raises(SystemExit, match="no RJMCMC"):
        LO.main([str(empty)])
    with pytest.raises(SystemExit, match="twice"):
        LO.main([str(empty), str(empty) + "/"])
    tr = tmp_path / "tr"
    tr.mkdir()
    _touch(str(tr / "t_1.trendrate.log"))
    with pytest.raises(SystemExit, match="TrendRate"):
        LO.main([str(tr)])
    two = tmp_path / "two"
    two.mkdir()
    for stem in ("tableBD_a", "tableBD_b"):
        _touch(str(two / ("%s_chain0_mcmc.log" % stem)))
    with pytest.raises(SystemExit, match="one run"):
        LO.main([str(two)])
    bad = tmp_path / "bad"
    bad.mkdir()
    _touch(str(bad / "x_1.log"), "it\tniche_0\n")
    with pytest.raises(SystemExit, match="not a log name"):
        LO.main([str(bad)])
