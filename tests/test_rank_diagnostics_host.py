"""CPU: the host restatement of the rank-normalised diagnostics (diagnostics.rank_rhat_ess) -- hand-worked ranks, quantiles and
indicators, the scale-mismatch case the plain split R-hat misses, invariances, numpy's quantile bit for bit, and each degenerate
rule."""
import math

import numpy as np
import pytest
from scipy.special import ndtri

from literate_b200 import diagnostics as D


def test_hand_worked_2x6_with_ties():
    x = np.array([[1.0, 3.0, 3.0, 2.0, 5.0, 3.0],
                  [4.0, 1.0, 2.0, 3.0, 6.0, 0.5]])
    _, xs = D._split(x)
    assert np.array_equal(xs, x)                                          # S even: every draw is a split draw
    # sorted: 0.5 1 1 2 2 3 3 3 3 4 5 6 -> ranks 1, 2.5, 2.5, 4.5, 4.5, 7.5 x4, 10, 11, 12
    r = np.array([[2.5, 7.5, 7.5, 4.5, 11, 7.5], [10, 2.5, 4.5, 7.5, 12, 1]])
    z = D.rank_normal(x)
    assert np.allclose(z, ndtri((r - 0.375) / 12.25), rtol=1e-15, atol=1e-15)
    assert z[0, 1] == z[0, 2] == z[0, 5] == z[1, 3]
    assert float(np.median(xs)) == 3.0
    # 12 draws: h = 11 p; q05 = x(0) + (x(1) - x(0)) 0.55 -> the g >= 0.5 branch, q95 = x(10) + (x(11) - x(10)) 0.45
    assert D.quantile_linear(x, 0.05) == 1.0 - (1.0 - 0.5) * (1 - 0.55) == np.quantile(x, 0.05)
    assert D.quantile_linear(x, 0.95) == 5.0 + (6.0 - 5.0) * (11 * 0.95 - 10) == np.quantile(x, 0.95)
    q05, q95 = D.quantile_linear(x, 0.05), D.quantile_linear(x, 0.95)
    assert np.array_equal((xs <= q05), [[False] * 6, [False] * 5 + [True]])
    assert np.array_equal((xs <= q95), [[True] * 6, [True, True, True, True, False, True]])
    out = D.rank_rhat_ess(x)
    assert out["median"] == 3.0 and out["q05"] == q05 and out["q95"] == q95
    assert out["rhat_bulk"] == D.rhat_ess(z)["rhat"] and out["ess_bulk"] == D.rhat_ess(z)["ess"]
    f = np.abs(x - 3.0)
    assert out["rhat_tail"] == D.rhat_ess(D.rank_normal(f))["rhat"]


def test_hand_worked_odd_s_drops_the_middle_draw_but_not_from_the_quantiles():
    x = np.array([[1.0, 3.0, 9.0, 2.0, 5.0],
                  [4.0, 1.0, -7.0, 3.0, 6.0]])
    _, xs = D._split(x)
    assert np.array_equal(xs, [[1, 3, 2, 5], [4, 1, 3, 6]])
    r = np.array([[1.5, 4.5, 3, 7], [6, 1.5, 4.5, 8]])
    assert np.allclose(D.rank_normal(xs), ndtri((r - 0.375) / 8.25), rtol=1e-15, atol=1e-15)
    out = D.rank_rhat_ess(x)
    assert out["median"] == 3.0                                            # (3 + 3) / 2 of the split draws
    assert out["q05"] == np.quantile(x, 0.05) and out["q95"] == np.quantile(x, 0.95)   # -7 and 9 included
    assert out["q05"] < -1 and out["q95"] > 6


def test_scale_mismatch_is_caught_by_the_folded_rhat_and_the_tail_ess():
    rng = np.random.default_rng(2021)
    x = np.concatenate([rng.normal(0, 1, (4, 1000)), rng.normal(0, 3, (4, 1000))])
    plain = D.rhat_ess(x)
    out = D.rank_rhat_ess(x)
    assert plain["rhat"] < 1.005
    assert out["rhat_rank"] > 1.1 and out["rhat_rank"] == out["rhat_tail"] > out["rhat_bulk"]
    assert out["ess_tail"] < plain["ess"] / 4


def _chains(seed, M=4, S=301):
    rng = np.random.default_rng(seed)
    return rng.integers(-20, 21, (M, S)).astype(np.float64) + (np.arange(M) % 2)[:, None]


def test_invariance_under_an_increasing_map_and_a_shift():
    x = _chains(1)
    a, b = D.rank_rhat_ess(x), D.rank_rhat_ess(x ** 3)
    for k in ("rhat_bulk", "ess_bulk", "ess_tail"):
        assert a[k] == b[k], k
    c = D.rank_rhat_ess(x + 1000.0)
    for k in ("rhat_bulk", "rhat_tail", "rhat_rank", "ess_bulk", "ess_tail"):
        assert a[k] == c[k], k
    assert c["median"] == a["median"] + 1000.0


@pytest.mark.parametrize("n", [21, 41, 2001, 20, 37, 1000, 4004])
def test_quantile_bit_identical_to_numpy(n):
    rng = np.random.default_rng(n)
    for x in (rng.normal(size=n), np.round(rng.normal(size=n), 1), rng.integers(0, 3, n).astype(float)):
        for p in (0.05, 0.95):
            q = D.quantile_linear(x, p)
            assert np.float64(q).view(np.int64) == np.float64(np.quantile(x, p)).view(np.int64), (n, p)
    x = rng.normal(size=n)
    x[3] = np.nan
    assert math.isnan(D.quantile_linear(x, 0.05))


def test_degenerate_columns():
    nan_out = lambda o: all(math.isnan(v) for k, v in o.items() if k != "margin")
    assert nan_out(D.rank_rhat_ess(np.full((3, 10), 2.5)))                          # constant
    assert nan_out(D.rank_rhat_ess(np.repeat(np.arange(3.0)[:, None], 10, 1)))      # stuck
    x = np.random.default_rng(0).normal(size=(3, 10))
    x[1, 2] = np.inf
    assert all(math.isnan(v) for k, v in D.rank_rhat_ess(x).items() if k != "margin")
    with pytest.raises(RuntimeError, match="not enough data"):
        D.rank_rhat_ess(np.zeros((2, 3)))


def test_constant_and_stuck_indicators():
    # q95 is the column's maximum (a 0/1 column with many ones): I_0.95 is all ones, a constant indicator with N draws' ESS
    rng = np.random.default_rng(4)
    x = (rng.uniform(size=(4, 200)) < 0.3).astype(float)
    out = D.rank_rhat_ess(x)
    assert D.quantile_linear(x, 0.95) == 1.0 and D.quantile_linear(x, 0.05) == 0.0
    assert math.isnan(D.rhat_ess((x <= 1.0).astype(float))["rhat"])
    e05 = D.rhat_ess((x <= 0.0).astype(float))["ess"]
    assert out["ess_tail"] == min(e05, float(x.size))
    y = x.copy()
    y[:, :] = 0.0
    y[0, 0] = 1.0                                                                 # q05 = q95 = 0: neither indicator constant
    ind = D.rhat_ess((y <= 0.0).astype(float))
    assert D.rank_rhat_ess(y)["ess_tail"] == ind["ess"] and math.isfinite(ind["rhat"])
    # a stuck indicator: every split chain below or above q05 as a whole -> NaN tail ESS
    y = np.concatenate([np.tile(rng.uniform(0, 1, 20), (1, 5)).reshape(1, 100), np.tile(rng.uniform(5, 6, 20), (19, 5)).reshape(19, 100)])
    y[0] = rng.uniform(0, 1, 100)
    ind = (y <= D.quantile_linear(y, 0.05)).astype(float)
    assert D.rhat_ess(ind)["rhat"] == math.inf
    assert math.isnan(D.rank_rhat_ess(y)["ess_tail"])


def test_folded_constant_01_column():
    # a 0/1 column split exactly in half: the median is 0.5, |x - 0.5| is constant, rhat_tail NaN, rhat_rank = rhat_bulk
    rng = np.random.default_rng(5)
    x = np.zeros((4, 100))
    flat = x.ravel()
    flat[rng.permutation(400)[:200]] = 1.0
    out = D.rank_rhat_ess(x)
    assert out["median"] == 0.5 and math.isnan(out["rhat_tail"])
    assert out["rhat_rank"] == out["rhat_bulk"] and math.isfinite(out["rhat_bulk"])


def test_columns_layout():
    x = np.random.default_rng(6).normal(size=(50, 3, 2))
    cols = D.rank_rhat_ess_columns(x)
    assert cols["rhat_rank"][1] == D.rank_rhat_ess(x[:, :, 1].T)["rhat_rank"]
    assert set(cols) == {"median", "q05", "q95", "rhat_bulk", "rhat_tail", "rhat_rank", "ess_bulk", "ess_tail", "margin"}
