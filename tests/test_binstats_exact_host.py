"""CPU: the exact reference of K1 (oracle/k1_exact.py) and the rule that decides which tables may take the int32 entry point.

* the O(n) reference equals the per-bin, per-lineage Fraction restatement bit for bit, edges included (times in (-1, 1),
  te == ts, te < ts, NaN rows, births and deaths on the window's edges, clipping windows, only_dead);
* it equals the oracle's per-bin loop bit for bit on dyadic tables (every shipped table), and the oracle's NumPy sums within
  their own rounding on real-valued ones;
* year_jitter_ok accepts exactly the jitters whose fl(year + jitter) is exact for every int32 year, and forward.as_year_table
  keeps every other jittered table float64.
"""
import math

import numpy as np
import pytest

from conftest import golden_input
from oracle import k1_exact as K, literate_oracle as O
from literate_b200 import engine as E, forward as F, synth


def _counts(ts, te, first_bin, n_bins):
    with np.errstate(invalid="ignore"):
        c = [O.events_in_bin(ts, te, first_bin + j, first_bin + j + 1)[:2] for j in range(n_bins)]
    return np.array([a for a, _ in c], np.int64), np.array([b for _, b in c], np.int64)


def _edge_table(rng, n, lo, hi):
    """Random lifetimes plus rows on every edge the kernel treats separately."""
    ts = rng.uniform(lo, hi, n)
    te = ts + rng.exponential(1.5, n)
    k = n // 4
    ts[:k] = np.floor(ts[:k]); te[:k] = np.ceil(te[:k])                   # on integers: births and deaths on bin edges
    edge = [(-2.0 ** -60, 2.0 ** -60),             # fractions that round to 1 (birth) and to 0 (death)
            (2.0 ** -53, 0.3), (3 * 2.0 ** -53, 0.7),  # ties of rint(x * 2^52): to even
            (-0.3, -1 + 2.0 ** -53), (-1.0, 0.0), (-0.0, 1.0),
            (0.25, 0.25), (1.5, 1.5),                # te == ts
            (2.5, 1.0), (0.1, -0.7),                 # te < ts
            (np.nan, 1.5), (0.5, np.nan), (np.nan, np.nan),
            (lo, hi), (float(math.floor(lo)), lo + 0.5), (hi - 0.5, float(math.ceil(hi))),
            (-np.inf, 0.5), (0.5, np.inf), (-1e10, 1.25), (1.75, 3e9)]
    for i, (s, e) in enumerate(edge):
        ts[k + i], te[k + i] = s, e
    return ts, te


@pytest.mark.parametrize("seed", range(6))
def test_linear_reference_equals_the_literal_one(seed):
    rng = np.random.default_rng(100 + seed)
    ts, te = _edge_table(rng, 240, -4.0, 4.0)
    fb, nb = (-5, 11) if seed % 2 == 0 else (-1, 3)       # the whole table, and a window that cuts it
    ts[-1], te[-1] = float(fb), float(fb) + 0.5           # a birth on first_bin, one on first_bin + n_bins, a death on first_bin
    ts[-2], te[-2] = float(fb + nb), float(fb + nb) + 2.0
    ts[-3], te[-3] = float(fb) - 1.5, float(fb)
    sp, ex, br = K.exact_bin_stats(ts, te, fb, nb)
    assert np.array_equal(br, K.exact_time_at_risk_literal(ts, te, fb, nb))
    wsp, wex = _counts(ts, te, fb, nb)
    assert np.array_equal(sp, wsp) and np.array_equal(ex, wex)
    # only_dead: end_time equal to some te, which is then excluded (te < end_time)
    end = float(np.sort(te[np.isfinite(te)])[len(te) // 2])
    _, _, _, exd, brd = K.exact_bin_stats(ts, te, fb, nb, only_dead=True, end_time=end)
    with np.errstate(invalid="ignore"):
        keep = te < end
    assert np.array_equal(brd, K.exact_time_at_risk_literal(ts[keep], te[keep], fb, nb))
    assert np.array_equal(exd, _counts(ts[keep], te[keep], fb, nb)[1])
    assert (te == end).any() and exd.sum() < ex.sum()


def test_quantization_moves_only_times_inside_minus_one_one():
    """Off the 2^-52 grid only below |t| = 1: 0.3 is not a multiple of 2^-52, 1000.3 is; a fraction that rounds to 1 starts
    the next bin, one that rounds to 0 ends the previous one."""
    from fractions import Fraction
    _, _, br = K.exact_bin_stats(np.array([0.3]), np.array([0.9]), 0, 1)
    assert br[0] == (round(0.9 * 2 ** 52) - round(0.3 * 2 ** 52)) / 2 ** 52
    assert br[0] != float(Fraction(0.9) - Fraction(0.3))
    _, _, br = K.exact_bin_stats(np.array([1000.3]), np.array([1000.9]), 1000, 1)
    assert br[0] == float(Fraction(1000.9) - Fraction(1000.3))
    _, _, br = K.exact_bin_stats(np.array([-2.0 ** -60, 0.0]), np.array([0.5, 2.0 ** -60]), -1, 2)
    assert br.tolist() == [0.0, 0.5]


@pytest.mark.parametrize("name,tbp", [("example_dataTAD.txt", False), ("example_dataTBP.txt", True)])
def test_equals_the_oracle_on_shipped_tables(name, tbp):
    for jitter in (0.5, 0.0, 0.25, 1.0):
        lin = O.read_lineages(golden_input(name), TBP=tbp, death_jitter=jitter)
        w = O.bin_stats(lin.ts, lin.te, only_dead=True)
        g = K.exact_bin_stats(lin.ts, lin.te, w.first_bin, w.n_bins, only_dead=True)
        for a, b in zip(g, (w.sp, w.ex, w.br, w.ex_dead, w.br_dead)):
            assert np.array_equal(a, b), (name, jitter)


def test_equals_the_oracle_on_metal_bands_and_syn_int(metal_path):
    lin = O.read_lineages(metal_path)
    tables = [(lin.ts, lin.te)] + [synth.syn_int(n, replicate=n) for n in (1, 31, 20011)]
    for ts, te in tables:
        w = O.bin_stats(ts, te, only_dead=True)
        g = K.exact_bin_stats(ts, te, w.first_bin, w.n_bins, only_dead=True)
        for a, b in zip(g, (w.sp, w.ex, w.br, w.ex_dead, w.br_dead)):
            assert np.array_equal(a, b), len(ts)
    # quarter years with negative times: dyadic too
    rng = np.random.default_rng(8)
    ts = -40 + rng.integers(0, 160, 3000) / 4.0; te = ts + rng.integers(0, 80, 3000) / 4.0
    w = O.bin_stats(ts, te)
    g = K.exact_bin_stats(ts, te, w.first_bin, w.n_bins)
    assert np.array_equal(g[0], w.sp) and np.array_equal(g[1], w.ex) and np.array_equal(g[2], w.br)


def test_real_valued_tables_within_the_oracles_rounding():
    """syn_real: the oracle's NumPy sums carry ~1e-15 of rounding; the exact sums differ from them by no more than that, and
    do differ (a reference that merely re-did the NumPy sums would not)."""
    ts, te = synth.syn_real(1_000_000)
    sp, ex, br = K.exact_bin_stats(ts, te, 1800, 200)
    w = O.bin_stats_fast(ts, te)
    assert np.array_equal(sp, w.sp) and np.array_equal(ex, w.ex)
    np.testing.assert_allclose(br, w.br, rtol=1e-13, atol=0)
    assert (br != w.br).sum() > 50
    # conservation: every lineage lies inside the window, so the whole time at risk is sum(te - ts) (exactly, in Fractions)
    from fractions import Fraction
    small_ts, small_te = ts[:2000], te[:2000]
    _, _, b = K.exact_bin_stats(small_ts, small_te, 1800, 200)
    tot = sum((Fraction(e) - Fraction(s) for s, e in zip(small_ts.tolist(), small_te.tolist())), Fraction(0))
    assert abs(Fraction(b.sum()) - tot) <= tot * 2 ** -45


ACCEPTED = (0.0, 2.0 ** -22, 0.25, 0.5, 1.0)
REFUSED = (0.1, 0.3, 0.05, 0.001, 1e-14, 2.0 ** -30)


def test_year_jitter_rule():
    for j in ACCEPTED:
        assert E.year_jitter_ok(j), j
        # exact for every admissible year
        for y in (-(2 ** 31 - 3), -1025, -1, 0, 1024, 2020, 2 ** 31 - 3):
            assert float(y) + j - float(y) == j
    for j in REFUSED + (-0.5, 1.5, float("nan"), float("inf")):
        assert not E.year_jitter_ok(j), j
    for j in REFUSED:
        assert any(float(y) + j - float(y) != j for y in (2020, 2 ** 30 + 1, 2 ** 31 - 3)), j


@pytest.mark.filterwarnings("ignore:Four column:FutureWarning")
@pytest.mark.parametrize("jitter", REFUSED)
def test_refused_jitters_keep_tables_float64(jitter):
    ts, te, *_ = F.parse_lineages(golden_input("example_dataTAD.txt"), death_jitter=jitter)
    assert F.as_year_table(ts, te, jitter) is None


@pytest.mark.filterwarnings("ignore:Four column:FutureWarning")
@pytest.mark.parametrize("jitter", ACCEPTED)
def test_accepted_jitters_take_the_int32_table(jitter):
    ts, te, *_ = F.parse_lineages(golden_input("example_dataTAD.txt"), death_jitter=jitter)
    ti, ei = F.as_year_table(ts, te, jitter)
    assert np.array_equal(ti, ts) and np.array_equal(ei + jitter, te)
