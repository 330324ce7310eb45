"""GPU: K6 (TrendRate chains, SURVEY 8 f-4) through the C ABI against the oracle pinned to the unmodified trend_rate.py.

Deterministic parity: statistics (K1 on create_bins' window) bit-exact; likelihood, prior, rates, adequacy and both
proposal kinds with explicit draws within 1e-10 relative (tolerance of the north star, written at each assert).
Chain-level parity is distributional (Philox vs MT19937): posterior means against the committed summaries of 8 unmodified
reference chains (tests/golden/trendrate/posterior/*.json) with the between-chain spread as the Monte-Carlo error.
"""
import json
import os

import numpy as np
import pytest

from oracle import trendrate_oracle as T
from literate_b200 import library as L
from literate_b200 import trend as TR
from test_oracle_trend_golden import TG, _jobs, stage

pytestmark = pytest.mark.gpu
RTOL = 1e-10


def _job(tag):
    return [j for j in _jobs() if j["tag"] == tag][0]


def _setup(device, tmp_path, tag="ex_ramp", n_chains=8, seed=1, const_birth=False, const_death=False, jitter=0.5, rm=0):
    job = _job(tag)
    data, trend_path = stage(job, tmp_path)
    idx = int(job["args"][job["args"].index("-trend_index") + 1])
    ts, te, present, origin = L.parse_ts_te(data, death_jitter=jitter)
    first, nb = L.bin_window(origin, present, rm)
    st = device.bin_stats(ts, te, first_bin=first, n_bins=nb, death_jitter=jitter)
    trend = TR.parse_trend_data(trend_path, idx, rm)
    ots, ote, opresent, oorigin = T.parse_ts_te(data, death_jitter=jitter)
    bins = T.create_bins(oorigin, opresent, ots, ote, rm)
    otrend = T.normalise_trend(T.read_trend_column(trend_path, idx), rm)
    ch = TR.TrendChains(device, st.sp, st.ex, st.br, trend, n_chains, seed, const_birth, const_death)
    return st, bins, trend, otrend, ch


def _random_params(rng, n):
    return np.stack([rng.gamma(1, .2, n) + .002, rng.gamma(1, .2, n) + .002, rng.normal(0, .3, n), rng.normal(0, .3, n),
                     rng.gamma(3, .5, n), rng.gamma(3, .5, n)], axis=1)


@pytest.mark.parametrize("tag,jitter,rm", [("ex_ramp", .5, 0), ("ex_jitter0", 0.0, 0), ("ex_rmfirst", .5, 1), ("metal_ramp", .5, 0)])
def test_statistics_equal_create_bins(device, tmp_path, tag, jitter, rm):
    st, bins, trend, otrend, ch = _setup(device, tmp_path, tag, jitter=jitter, rm=rm)
    assert st.n_bins == bins.n_bins
    assert np.array_equal(st.sp[0], bins.n_spec) and np.array_equal(st.ex[0], bins.n_exti)      # bit-exact
    assert np.array_equal(st.br[0], bins.dt)                                                    # dyadic data: exact
    assert np.array_equal(trend, otrend)


@pytest.mark.parametrize("tag,cb,cd", [("ex_ramp", False, False), ("ex_hump", True, False), ("ex_hump", False, True), ("metal_ramp", False, False)])
def test_state_evaluation_matches_the_oracle(device, tmp_path, tag, cb, cd):
    st, bins, trend, otrend, ch = _setup(device, tmp_path, tag, const_birth=cb, const_death=cd)
    rng = np.random.default_rng(7)
    P = _random_params(rng, 200)
    P[0] = [.1, .1, 0, 0, 1, 1]                    # the initial state (trend_rate.py:141-147)
    P[1, 2] = -5.0                                  # negative alpha: rates floored at SMALL_NUMBER (:80)
    P[2, 3] = -5.0
    out = ch.evaluate(P)
    emp_b, emp_d = bins.n_spec / bins.dt, bins.n_exti / bins.dt
    for i, p in enumerate(P):
        lk, lam, mu = T.likelihood(p, bins, otrend, cb, cd)
        np.testing.assert_allclose(out["lik"][i], lk, rtol=RTOL)
        assert out["prior"][i] == pytest.approx(T.prior(p, exact_scipy=True), rel=RTOL)
        np.testing.assert_allclose(out["rates"][i, 0], lam, rtol=RTOL)
        np.testing.assert_allclose(out["rates"][i, 1], mu, rtol=RTOL)
        np.testing.assert_allclose(out["adequacy"][i], T.adequacy(emp_b, emp_d, lam, mu), rtol=1e-8)
    assert (out["rates"][1, 0] == T.SMALL_NUMBER).any() or cb
    # outside the support of the priors: -inf, like scipy
    bad = np.array([[.0005, .1, 0, 0, 1, 1], [.1, .0009, 0, 0, 1, 1], [.1, .1, 0, 0, -.1, 1], [.1, .1, 0, 0, 1, 0.0]])
    assert np.all(np.isneginf(ch.evaluate(bad)["prior"]))


def test_two_hundred_bins_strided_over_the_lanes(device):
    """n_bins > 32: every lane owns several bins (the strided part of trend_lik / adequacy / records)."""
    rng = np.random.default_rng(5)
    nb = 200
    sp = rng.integers(0, 5000, nb); ex = rng.integers(0, 4000, nb); br = rng.uniform(1000, 90000, nb)
    trend = rng.uniform(0, 1, nb); trend[3] = T.SMALL_NUMBER; trend[77] = 1.0
    bins = T.Bins(1800.0, 2000.5, sp, ex, br)
    ch = TR.TrendChains(device, sp, ex, br, trend, 4, 1)
    P = _random_params(rng, 64)
    out = ch.evaluate(P)
    for i, p in enumerate(P):
        lk, lam, mu = T.likelihood(p, bins, trend)
        np.testing.assert_allclose(out["lik"][i], lk, rtol=RTOL)
        np.testing.assert_allclose(out["rates"][i], [lam, mu], rtol=RTOL)
        np.testing.assert_allclose(out["adequacy"][i], T.adequacy(sp / br, ex / br, lam, mu), rtol=1e-8)
    recs = ch.run(2001, 500)
    assert recs.shape == (5, 4, 16 + 2 * nb)
    for r in recs[:, 0]:
        lk, lam, mu = T.likelihood(r[5:11], bins, trend)
        np.testing.assert_allclose(r[2:4], lk, rtol=RTOL)
        np.testing.assert_allclose(r[16:16 + nb], lam, rtol=RTOL)
        np.testing.assert_allclose(r[16 + nb:], mu, rtol=RTOL)


@pytest.mark.parametrize("nb", [65, 100, 129, 200, 300])
def test_wide_build_gives_the_chains_of_the_one_warp_build(device, nb, monkeypatch):
    """More than 64 bins: the likelihood sums are formed group by group (2 or 4 groups of bins) in a fixed order, which the wide
    build (one warp per group, partial sums exchanged through shared memory once per iteration) reproduces: records and final
    states identical to the one-warp kernel, bit for bit, over split launches."""
    rng = np.random.default_rng(nb)
    sp = rng.integers(0, 5000, nb); ex = rng.integers(0, 4000, nb); br = rng.uniform(1000, 90000, nb)
    trend = np.clip(rng.uniform(0, 1, nb), T.SMALL_NUMBER, 1.0)
    out = []
    for wide in ("0", "1"):
        monkeypatch.setenv("LR_TREND_WIDE", wide)
        ch = TR.TrendChains(device, sp, ex, br, trend, 7, 3)
        recs = [ch.run(n, s) for n, s in ((1501, 100), (1, 1), (998, 7), (3000, 250))]
        out.append((np.concatenate(recs), ch.state()))
    assert np.array_equal(out[0][0], out[1][0]) and np.array_equal(out[0][1], out[1][1])
    assert len(np.unique(out[0][0][:, :, 14])) > 10           # the chains do move (accepted counts grow)


@pytest.mark.parametrize("nb", [1, 2, 33])
def test_few_bins(device, nb):
    rng = np.random.default_rng(40 + nb)
    sp = rng.integers(1, 50, nb); ex = rng.integers(1, 40, nb); br = rng.uniform(50, 500, nb)
    trend = np.clip(rng.uniform(0, 1, nb), T.SMALL_NUMBER, 1.0)
    bins = T.Bins(0.0, nb + 1.5, sp, ex, br)
    ch = TR.TrendChains(device, sp, ex, br, trend, 4, 2)
    recs = ch.run(4001, 1000)
    for r in recs[1:].reshape(-1, recs.shape[-1]):
        lk, lam, mu = T.likelihood(r[5:11], bins, trend)
        np.testing.assert_allclose(r[2:4], lk, rtol=RTOL)
        np.testing.assert_allclose(r[16:], np.concatenate([lam, mu]), rtol=RTOL)
        assert r[4] == pytest.approx(T.prior(r[5:11], exact_scipy=True), rel=RTOL)


def test_replicates_of_the_statistics(device):
    """Imputation replicates: chain c runs on replicate rep_of_chain[c]; states are evaluated on the replicate asked for."""
    rng = np.random.default_rng(9)
    nb, n_rep = 40, 3
    sp = rng.integers(0, 300, (n_rep, nb)); ex = rng.integers(0, 200, (n_rep, nb)); br = rng.uniform(100, 3000, (n_rep, nb))
    trend = np.clip(rng.uniform(0, 1, nb), T.SMALL_NUMBER, 1.0)
    rep_of_chain = np.arange(12) % n_rep
    ch = TR.TrendChains(device, sp, ex, br, trend, 12, 5, rep_of_chain=rep_of_chain)
    P = _random_params(rng, 30)
    rep = rng.integers(0, n_rep, 30)
    out = ch.evaluate(P, rep=rep)
    for i, p in enumerate(P):
        lk, lam, mu = T.likelihood(p, T.Bins(0.0, nb + 1.5, sp[rep[i]], ex[rep[i]], br[rep[i]]), trend)
        np.testing.assert_allclose(out["lik"][i], lk, rtol=RTOL)
    recs = ch.run(1501, 500)
    for c in range(12):
        r = recs[-1, c]
        k = rep_of_chain[c]
        lk, _, _ = T.likelihood(r[5:11], T.Bins(0.0, nb + 1.5, sp[k], ex[k], br[k]), trend)
        np.testing.assert_allclose(r[2:4], lk, rtol=RTOL)
    assert np.array_equal(ch.state()[:, 11], rep_of_chain)


def test_proposals_with_explicit_draws_match_the_oracle(device, tmp_path):
    st, bins, trend, otrend, ch = _setup(device, tmp_path)
    rng = np.random.default_rng(11)
    n = 300
    P = _random_params(rng, n)
    kind = rng.integers(0, 2, n).astype(np.int32)
    on = (rng.uniform(size=(n, 6)) < .5).astype(np.int32)
    draw = np.where(kind[:, None] == 1, rng.normal(size=(n, 6)), rng.uniform(size=(n, 6)))
    out = ch.evaluate(P, kind=kind, on=on, draw=draw)
    for i in range(n):
        if kind[i] == 1:
            q, h = T.normal_given(P[i], on[i], draw[i])
        else:
            q, h = T.multiplier_given(P[i], on[i], draw[i])
        np.testing.assert_allclose(out["params"][i], q, rtol=1e-13)
        assert out["hastings"][i] == pytest.approx(h, rel=1e-11, abs=1e-15)
        lk, _, _ = T.likelihood(q, bins, otrend)
        np.testing.assert_allclose(out["lik"][i], lk, rtol=RTOL)
        assert out["prior"][i] == pytest.approx(T.prior(q, exact_scipy=True), rel=RTOL)
        # untouched parameters come back bit for bit
        assert np.array_equal(out["params"][i][on[i] == 0], P[i][on[i] == 0])


def test_chain_bookkeeping(device, tmp_path):
    """Initial state, forced acceptance of iteration 0, stored likelihoods = likelihoods of the stored parameters, records on
    the sampling grid, counters."""
    st, bins, trend, otrend, ch = _setup(device, tmp_path, n_chains=16, seed=3)
    s0 = ch.state()
    lk, _, _ = T.likelihood(np.array([.1, .1, 0, 0, 1, 1.]), bins, otrend)
    for s in s0:
        assert np.array_equal(s[:6], [.1, .1, 0, 0, 1, 1]) and s[9] == 0 and s[10] == 0
        np.testing.assert_allclose(s[6:8], lk, rtol=RTOL)
        assert s[8] == pytest.approx(T.prior(s[:6], exact_scipy=True), rel=RTOL)
    recs = ch.run(20001, 500)
    assert recs.shape == (41, 16, 16 + 2 * bins.n_bins)
    assert np.all(recs[0, :, 14] == 1)                                       # iteration 0 is always accepted (:176)
    assert not np.all(recs[0, :, 5:11] == np.array([.1, .1, 0, 0, 1, 1]))
    emp_b, emp_d = bins.n_spec / bins.dt, bins.n_exti / bins.dt
    for si in range(0, 41, 4):
        for c in (0, 7, 15):
            r = recs[si, c]
            assert r[0] == si * 500
            lk, lam, mu = T.likelihood(r[5:11], bins, otrend)
            np.testing.assert_allclose(r[2:4], lk, rtol=RTOL)
            assert r[1] == r[2] + r[3]
            assert r[4] == pytest.approx(T.prior(r[5:11], exact_scipy=True), rel=RTOL)
            np.testing.assert_allclose(r[16:16 + bins.n_bins], lam, rtol=RTOL)
            np.testing.assert_allclose(r[11:14], T.adequacy(emp_b, emp_d, lam, mu), rtol=1e-8)
            assert r[5] > .001 and r[6] > .001 and r[9] > 0 and r[10] > 0   # support of the priors
    fin = ch.state()
    assert np.all(fin[:, 9] == 20001) and np.all(fin[:, 10] == recs[-1, :, 14])
    acc = fin[:, 10].mean() / 20001
    assert 0.2 < acc < 0.95


def test_determinism_split_runs_and_sharding(device, tmp_path):
    st, bins, trend, otrend, a = _setup(device, tmp_path, n_chains=32, seed=11)
    ra = a.run(3000, 100)
    mk = lambda n, seed, c0=0: TR.TrendChains(device, st.sp, st.ex, st.br, trend, n, seed, chain_id0=c0)
    b = mk(32, 11)
    rb = np.concatenate([b.run(1000, 100), b.run(1501, 100), b.run(499, 100)])
    assert np.array_equal(ra, rb) and np.array_equal(a.state(), b.state())
    c = mk(8, 11, 16)
    assert np.array_equal(c.run(3000, 100), ra[:, 16:24])
    assert not np.array_equal(mk(32, 12).run(3000, 100), ra)
    big = mk(2048, 11)                     # four warps per CTA
    assert np.array_equal(big.run(3000, 100)[:, :32], ra)


def test_both_sides_constant_is_refused(device, tmp_path):
    from literate_b200._native import NativeError
    with pytest.raises(NativeError, match="binomial"):
        _setup(device, tmp_path, const_birth=True, const_death=True)


def _chain_means(recs, nb, burnin=0.2):
    b = int(burnin * recs.shape[0])
    r = recs[b:]
    cols = {"likelihood": 1, "likelihood_birth": 2, "likelihood_death": 3, "prior": 4, "l_min": 5, "m_min": 6, "alpha": 7,
            "beta": 8, "delta": 9, "gamma": 10}
    out = {k + "_mean": r[:, :, c].mean(0) for k, c in cols.items()}
    out["birth_rate_mean"] = r[:, :, 16:16 + nb].mean(0)
    out["death_rate_mean"] = r[:, :, 16 + nb:16 + 2 * nb].mean(0)
    return out


@pytest.mark.parametrize("tag,base,cd", [("ex_ramp", "ex_ramp", False), ("ex_hump_constD", "ex_hump", True)])
def test_posterior_matches_reference_chains(device, tmp_path, tag, base, cd):
    """128 device chains against 32 unmodified reference chains of the same length: every posterior mean within 3.5 standard
    errors of the difference of the two population means (between-chain variance of both sides); 64 against 8 within 4.5 while
    a fixture still holds the 8 chains of round 1."""
    with open(os.path.join(TG, "posterior", tag + ".json")) as fh:
        ref = json.load(fh)
    strong = len(ref["chains"]) >= 32
    z_max = 3.5 if strong else 4.5
    st, bins, trend, otrend, ch = _setup(device, tmp_path, base, n_chains=128 if strong else 64, seed=2026, const_death=cd)
    recs = ch.run(ref["n_iter"], ref["sample_every"])
    assert recs.shape[0] == len(range(0, ref["n_iter"], ref["sample_every"]))
    mine = _chain_means(recs, bins.n_bins, ref["burnin"])
    for key, a in mine.items():
        b = np.array([c[key] for c in ref["chains"]], dtype=float)
        a = np.asarray(a, dtype=float)
        se = np.sqrt(a.var(0, ddof=1) / len(a) + b.var(0, ddof=1) / len(b))
        if np.all(se == 0):                  # beta and gamma are never updated with a constant death rate (:125-126, :132-133)
            assert cd and key in ("beta_mean", "gamma_mean") and np.array_equal(a.mean(0), b.mean(0))
            continue
        z = np.abs(a.mean(0) - b.mean(0)) / se
        assert np.all(z < z_max), (key, float(np.max(z)), a.mean(0), b.mean(0))


def test_command_line_end_to_end(device, tmp_path, capsys):
    job = _job("ex_ramp")
    data, trend_path = stage(job, tmp_path)
    paths = TR.run(TR.build_parser().parse_args(["-d", data, "-trend_data", trend_path, "-trend_index", "1", "-n", "3001", "-s", "50",
                                                 "-seed", "1", "-chains", "3", "-quiet", "1"]), device=device)
    assert [os.path.basename(p) for p in paths] == ["example3_%d_EXPB_EXPD_1.trendrate.log" % s for s in (1, 2, 3)]
    want = open(os.path.join(TG, "ex_ramp", job["files"][0]), "rb").read().split(b"\r\n")
    for p in paths:
        got = open(p, "rb").read().split(b"\r\n")
        assert got[0] == want[0] and len(got) == len(want)                  # same header, same number of rows
        rows = np.array([l.split(b"\t") for l in got[1:-1]], dtype=float)
        assert np.array_equal(rows[:, 0], np.arange(0, 3001, 50))
        np.testing.assert_allclose(rows[:, 1], rows[:, 2] + rows[:, 5], rtol=1e-15)
    a, b = open(paths[0], "rb").read(), open(paths[1], "rb").read()
    assert a != b


def test_directory_of_imputations(device, tmp_path):
    """-d <directory>: every table is a replicate of one K1 launch; chain k runs on table k % n_tables and logs next to it."""
    job = _job("ex_ramp")
    data, trend_path = stage(job, tmp_path)
    rows = [l.split("\t") for l in open(data).read().splitlines()[1:]]
    d = os.path.join(str(tmp_path), "imputations")
    os.makedirs(d)
    rng = np.random.default_rng(3)
    tables = []
    for i in range(3):
        path = os.path.join(d, "imp_%d.tsv" % i)
        with open(path, "w") as fh:
            fh.write("id\tts\tte\n")
            for j, r in enumerate(rows):
                ts, te = int(r[1]), int(r[2])
                if i and 1996 < ts < 2010 and te - ts > 2 and rng.uniform() < .3:
                    ts += 1                                     # another imputation of the same record, window unchanged
                fh.write("%s\t%d\t%d\n" % (r[0], ts, te))
            if i == 2:
                fh.write("999\t2001\t2005\n")                  # ragged: one more lineage than the others
        tables.append(path)
    paths = TR.run(TR.build_parser().parse_args(["-d", d, "-trend_data", trend_path, "-trend_index", "1", "-n", "2001", "-s", "500",
                                                 "-seed", "5", "-chains", "6", "-quiet", "1"]), device=device)
    assert [os.path.basename(p) for p in paths] == ["imp_%d_%d_EXPB_EXPD_1.trendrate.log" % (k % 3, 5 + k // 3) for k in range(6)]
    otrend = T.normalise_trend(T.read_trend_column(trend_path, 1))
    for k, p in enumerate(paths):
        ts, te, present, origin = T.parse_ts_te(tables[k % 3])
        bins = T.create_bins(origin, present, ts, te)
        got = np.loadtxt(p, skiprows=1)
        assert got.shape[0] == 5
        for row in got:
            lk, lam, mu = T.likelihood(row[6:12], bins, otrend)
            np.testing.assert_allclose(row[3:5], lk, rtol=RTOL)
