"""GPU: tempered ladders of TrendRate (K6) and DDRate (K7) chains.  The reference has no tempering (SURVEY A-15); as for K3
(test_gpu_tempering.py) the checks are self-consistency ones: a chain at beta = 1 is the untempered chain bit for bit, swap
rounds permute the temperatures of a ladder by the one rule K3 uses, the cold members sample the posterior of the reference
chains, chains at beta = 0 sample the prior, and the command lines log only cold rows."""
import os

import numpy as np
import pytest
import torch

from conftest import golden_input
from oracle import ddrate_oracle as D
from oracle import literate_oracle as O
from oracle import trendrate_oracle as TO
from literate_b200 import ddrate as DD
from literate_b200 import engine as E
from literate_b200 import library as L
from literate_b200 import parallel as P
from literate_b200 import trend as TR
from literate_b200._native import NativeError
from test_gpu_ddrate import _setup as dd_setup
from test_gpu_trend import _chain_means, _setup as trend_setup
from test_oracle_ddrate_golden import DG, _jobs as dd_jobs, stage as dd_stage
from test_oracle_trend_golden import TG, _jobs as trend_jobs, stage as trend_stage

pytestmark = pytest.mark.gpu
RTOL = 1e-10
KINDS = ["trend", "dd"]


def _synthetic(device, kind, nb, n, seed, rep_of_chain=None, n_rep=1, chain_id0=0):
    """n chains (global ids from chain_id0) of K6 or K7 on synthetic tables of nb bins (n_rep replicates)."""
    rng = np.random.default_rng(nb + n_rep)
    if kind == "trend":
        br = rng.uniform(1000, 90000, (n_rep, nb)); sp = rng.integers(0, 5000, (n_rep, nb)); ex = rng.integers(0, 4000, (n_rep, nb))
        trend = np.clip(rng.uniform(0, 1, nb), TO.SMALL_NUMBER, 1.0)
        return TR.TrendChains(device, sp, ex, br, trend, n, seed, chain_id0=chain_id0, rep_of_chain=rep_of_chain)
    t = np.arange(nb)
    br = np.stack([20 + 400 / (1 + np.exp(-0.3 * (t - nb / 2))) + rng.uniform(0, 5, nb) for _ in range(n_rep)])
    sp = rng.poisson(br * 0.2); ex = rng.poisson(br * 0.1)
    gts = np.sort(rng.uniform(0, nb * .7, 40)).round(); gte = np.minimum(gts + rng.integers(1, nb + 1, 40), nb) + .5
    return DD.DDChains(device, sp, ex, br, 0.0, nb + 1.5, 3, 2, gts, gte, n, seed, chain_id0=chain_id0, rep_of_chain=rep_of_chain)


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("nb,wide", [(24, "0"), (200, "0"), (200, "1")])
def test_beta_one_is_the_untempered_chain(device, kind, nb, wide, monkeypatch):
    """set_beta(1) changes nothing: records and states bit for bit those of a population that never got a beta, for the
    one-warp and the wide build; the beta field of the records reads 1."""
    monkeypatch.setenv("LR_TREND_WIDE" if kind == "trend" else "LR_DD_WIDE", wide)
    out = []
    for set_beta in (False, True):
        ch = _synthetic(device, kind, nb, 12, 4)
        if set_beta:
            ch.set_beta(1.0)
        recs = np.concatenate([ch.run(n, s) for n, s in ((1501, 100), (998, 7), (2000, 250))])
        out.append((recs, ch.state()))
        assert np.all(recs[..., ch.REC_BETA] == 1.0)
        beta, swaps = ch.temper()
        assert np.all(beta == 1.0) and np.all(swaps == 0)
    assert np.array_equal(out[0][0], out[1][0]) and np.array_equal(out[0][1], out[1][1])


@pytest.mark.parametrize("kind", KINDS)
def test_wide_build_equals_one_warp_build_under_tempering(device, kind, monkeypatch):
    """Ladders with beta < 1, split launches with swap rounds in between: records, states, temperatures and swap counters of
    the wide build (4 warps per chain at 200 bins) equal those of the one-warp build."""
    T, n = 4, 16
    out = []
    for wide in ("0", "1"):
        monkeypatch.setenv("LR_TREND_WIDE" if kind == "trend" else "LR_DD_WIDE", wide)
        ch = _synthetic(device, kind, 200, n, 9)
        ch.set_beta(np.tile(P.temperature_ladder(T, 0.5), n // T))
        recs, rounds = ch.run_tempered(4001, 100, T, 500)
        more, rounds2 = ch.run_tempered(999, 7, T, 333, round0=rounds)
        out.append((np.concatenate([recs, more]), ch.state(), *ch.temper()))
        assert rounds == 8 and rounds2 == 3
    for a, b in zip(out[0], out[1]):
        assert np.array_equal(a, b)
    assert out[0][3][:, 1].sum() > 0 and len(np.unique(out[0][0][..., ch.REC_BETA])) == T


@pytest.mark.parametrize("kind", KINDS)
def test_swap_rounds_permute_temperatures(device, kind):
    T, n = 4, 64
    ch = _synthetic(device, kind, 24, n, 7)
    beta = np.tile(P.temperature_ladder(T, 0.3), n // T)
    ch.set_beta(beta)
    ch.run(2000)
    prev = beta.copy()
    for rnd in range(6):
        s_before = ch.state()
        ch.swap_step(T, rnd)
        now = ch.temper()[0]
        assert np.array_equal(ch.state(), s_before)            # parameters and likelihoods never move between chains
        assert np.array_equal(np.sort(now.reshape(-1, T), axis=1), np.sort(beta.reshape(-1, T), axis=1))   # a permutation per ladder
        for lad in range(n // T):                              # only temperature neighbours of this round's parity exchanged
            a, b = prev[lad * T:(lad + 1) * T], now[lad * T:(lad + 1) * T]
            ra = np.argsort(np.argsort(-a)); rb = np.argsort(np.argsort(-b))
            for i in np.nonzero(ra != rb)[0]:
                assert abs(int(ra[i]) - int(rb[i])) == 1 and min(ra[i], rb[i]) % 2 == rnd % 2
        prev = now
        ch.run(500)
    sw = ch.temper()[1].sum(0)
    assert sw[0] > 0 and 0 < sw[1] <= sw[0] and sw[0] % 2 == 0 and sw[1] % 2 == 0      # both members of a pair count


@pytest.mark.parametrize("kind", KINDS)
def test_swap_outcome_is_independent_of_sharding(device, kind):
    """Two shards of 8 chains fed the gathered (lik, beta) table take the decisions of the 16-chain population, for ladders
    of 4 and for a ladder of 16 that spans both shards (the multi-rank path of parallel.tempered_swap, on one device)."""
    for T in (4, 16):
        beta = np.tile(P.temperature_ladder(T, 0.25), 16 // T)
        whole = _synthetic(device, kind, 24, 16, 3)
        a = _synthetic(device, kind, 24, 8, 3)
        b = _synthetic(device, kind, 24, 8, 3, chain_id0=8)
        for ch, bb in ((whole, beta), (a, beta[:8]), (b, beta[8:])):
            ch.set_beta(bb); ch.run(1500)
        for rnd in range(4):
            whole.swap_step(T, rnd)
            ia = a.swap_info_device(torch.empty((8, 2), dtype=torch.float64, device="cuda"))
            ib = b.swap_info_device(torch.empty((8, 2), dtype=torch.float64, device="cuda"))
            torch.cuda.synchronize()
            table = torch.cat([ia, ib])
            a.swap_apply_device(table, 0, T, rnd); b.swap_apply_device(table, 8, T, rnd)
            torch.cuda.synchronize()
            assert np.array_equal(np.concatenate([a.temper()[0], b.temper()[0]]), whole.temper()[0]), (T, rnd)
            whole.run(300); a.run(300); b.run(300)
        assert np.array_equal(np.concatenate([a.state(), b.state()]), whole.state())
        assert np.array_equal(np.concatenate([a.temper()[1], b.temper()[1]]), whole.temper()[1])
        if T == 16:
            with pytest.raises(NativeError, match="whole ladders"):
                a.swap_step(T, 99)                              # a ladder of 16 does not fit a shard of 8


@pytest.mark.parametrize("kind", KINDS)
def test_refusals(device, kind):
    ch = _synthetic(device, kind, 24, 66, 1)
    for bad in (-0.1, 1.5, np.nan):
        with pytest.raises(NativeError, match=r"outside \[0, 1\]"):
            ch.set_beta(bad)
    with pytest.raises(NativeError, match="whole ladders"):
        ch.swap_step(1, 0)
    with pytest.raises(NativeError, match="2..32"):
        ch.swap_step(33, 0)                                    # 66 chains are whole ladders of 33
    with pytest.raises(NativeError, match="whole ladders"):
        ch.swap_step(4, 0)                                     # 66 is not a multiple of 4
    mixed = _synthetic(device, kind, 24, 8, 1, rep_of_chain=np.arange(8) % 2, n_rep=2)
    with pytest.raises(NativeError, match="replicates"):
        mixed.swap_step(4, 0)
    same = _synthetic(device, kind, 24, 8, 1, rep_of_chain=np.repeat([0, 1], 4), n_rep=2)
    same.set_beta(np.tile(P.temperature_ladder(4), 2))
    same.swap_step(4, 0)                                       # ladders of 4 on one replicate each
    assert np.array_equal(same.state()[:, same.STATE_DOUBLES - (1 if kind == "trend" else 3)], np.repeat([0, 1], 4))


def test_one_swap_rule_for_the_three_samplers(device):
    """One crafted (lik, beta) table, one seed: K3, K6 and K7 objects apply the same permutations for ladders of 2, 4 and 32
    over several rounds, and count the same swaps."""
    n, seed = 64, 5
    rng = np.random.default_rng(8)
    lin = O.read_lineages(golden_input("example_dataTAD.txt"))
    ds = E.Dataset(device, device.bin_stats(lin.ts, lin.te), 0, lin.start_time, lin.end_time)
    k3 = E.Chains(ds, n, seed)
    k6 = _synthetic_seeded(device, "trend", n, seed)
    k7 = _synthetic_seeded(device, "dd", n, seed)
    for ladder in (2, 4, 32):
        lik = rng.normal(-3000, 4, n)
        beta = np.tile(P.temperature_ladder(ladder, 0.05), n // ladder)
        for rnd in range(6):
            table = torch.tensor(np.stack([lik, beta], axis=1), dtype=torch.float64, device="cuda")
            got = []
            for ch in (k3, k6, k7):
                ch.set_beta(beta)
                ch.swap_apply_device(table, 0, ladder, rnd)
                torch.cuda.synchronize()
                got.append(ch.state()[:, E.REC_BETA] if ch is k3 else ch.temper()[0])
            assert np.array_equal(got[0], got[1]) and np.array_equal(got[0], got[2]), (ladder, rnd)
            assert np.array_equal(np.sort(got[0].reshape(-1, ladder), 1), np.sort(beta.reshape(-1, ladder), 1))
            beta = got[0]
            lik = lik + rng.normal(0, 2, n)
    c3 = k3.counters()[:, 8:10]
    assert np.array_equal(c3, k6.temper()[1]) and np.array_equal(c3, k7.temper()[1])
    assert 0 < c3[:, 1].sum() < c3[:, 0].sum()


def _synthetic_seeded(device, kind, n, seed):
    rng = np.random.default_rng(2)
    if kind == "trend":
        return TR.TrendChains(device, rng.integers(0, 50, 10), rng.integers(0, 40, 10), rng.uniform(100, 900, 10),
                              np.linspace(.05, 1, 10), n, seed)
    return DD.DDChains(device, rng.integers(0, 50, 10), rng.integers(0, 40, 10), rng.uniform(100, 900, 10), 0.0, 11.5, 2, 2,
                       None, None, n, seed)


def _z_against_reference(mine, ref, z_max):
    for key, a in mine.items():
        b = np.array([c[key] for c in ref["chains"]], dtype=float)
        a = np.asarray(a, dtype=float)
        se = np.sqrt(a.var(0, ddof=1) / len(a) + b.var(0, ddof=1) / len(b))
        z = np.abs(a.mean(0) - b.mean(0)) / se
        assert np.all(z < z_max), (key, float(np.max(z)), a.mean(0), b.mean(0))


def _run_tempered_cold(ch, n_iter, every, T, swap_every=1000, chunk=50_000):
    """run_tempered in launches of `chunk` iterations (the round counter carried): returns (cold records, swap rounds,
    log-likelihood of the hottest member of every ladder [n_samples, n_ladders])."""
    cold, hottest, done, rounds = [], [], 0, 0
    while done < n_iter:
        k = min(chunk, n_iter - done)
        rt, r = ch.run_tempered(k, every, T, swap_every, round0=rounds)
        rounds += r
        done += k
        cold.append(E.cold_records(rt, T, ch.REC_BETA))
        hot = rt.reshape(rt.shape[0], rt.shape[1] // T, T, -1)
        hottest.append(np.take_along_axis(hot[..., 1], np.argmin(hot[..., ch.REC_BETA], axis=2)[:, :, None], axis=2)[:, :, 0])
    return np.concatenate(cold), rounds, np.concatenate(hottest)


def _check_ladders(ch, cold, hottest):
    """Swap acceptance inside (0.05, 0.999); the hottest members see a flatter likelihood: a lower mean log-likelihood."""
    sw = ch.temper()[1].sum(0)
    assert 0.05 < sw[1] / sw[0] < 0.999, sw
    b = cold.shape[0] // 5
    assert hottest[b:].mean() < cold[b:, :, 1].mean()


def test_cold_trendrate_chains_sample_the_untempered_posterior(device, tmp_path):
    """128 ladders of T = 4 against the 32 unmodified reference chains of ex_ramp: every posterior mean of the cold members
    within 3.5 standard errors (the bound of test_gpu_trend.test_posterior_matches_reference_chains)."""
    import json
    with open(os.path.join(TG, "posterior", "ex_ramp.json")) as fh:
        ref = json.load(fh)
    assert len(ref["chains"]) >= 32
    T, ladders = 4, 128
    st, bins, trend, otrend, ch = trend_setup(device, tmp_path, "ex_ramp", n_chains=T * ladders, seed=2028)
    ch.set_beta(np.tile(P.temperature_ladder(T, 0.1), ladders))
    cold, rounds, hottest = _run_tempered_cold(ch, ref["n_iter"], ref["sample_every"], T)
    assert rounds == ref["n_iter"] // 1000
    _check_ladders(ch, cold, hottest)
    assert cold.shape[0] == len(range(0, ref["n_iter"], ref["sample_every"]))
    _z_against_reference(_chain_means(cold, bins.n_bins, ref["burnin"]), ref, 3.5)


def test_cold_ddrate_chains_sample_the_untempered_posterior(device, tmp_path):
    """128 ladders of T = 4 against the 32 unmodified reference chains of ex_g_mddn (-m_birth 3: the genre term is tempered
    too), every posterior mean within 3.5 standard errors."""
    import json
    with open(os.path.join(DG, "posterior", "ex_g_mddn.json")) as fh:
        ref = json.load(fh)
    assert len(ref["chains"]) >= 32
    T, ladders = 4, 128
    S, ch = dd_setup(device, tmp_path, "ex_g_mddn", mb=3, md=2, n_chains=T * ladders, seed=2029)
    ch.set_beta(np.tile(P.temperature_ladder(T, 0.1), ladders))
    cold, rounds, hottest = _run_tempered_cold(ch, ref["n_iter"], ref["sample_every"], T)
    _check_ladders(ch, cold, hottest)
    r = cold[int(ref["burnin"] * cold.shape[0]):]
    nb = S.n
    cols = {"likelihood": r[:, :, 1], "likelihood_birth": r[:, :, 2], "likelihood_death": r[:, :, 3], "prior": r[:, :, 4],
            "l_f": r[:, :, 5], "l_mul": r[:, :, 6], "k": r[:, :, 7], "x0_abs": r[:, :, 8] + S.origin, "div_0": r[:, :, 9],
            "K_max": r[:, :, 10] + r[:, :, 9], "m_mul": r[:, :, 11], "nuB": r[:, :, 12], "nuD": r[:, :, 13], "g_l1": r[:, :, 14],
            "g_l2": r[:, :, 15], "likelihood_genre": r[:, :, 16]}
    mine = {k + "_mean": v.mean(0) for k, v in cols.items()}
    for i, k in enumerate(["birth_rate", "death_rate", "niche", "niche_frac"]):
        mine[k + "_mean"] = r[:, :, 24 + i * nb:24 + (i + 1) * nb].mean(0)
    _z_against_reference(mine, ref, 3.5)


def _prior_moments(ch, n_iter, every, cols, want, burnin=0.1, chunk=200_000):
    """Runs n_iter iterations sampling every `every`-th; per chain the mean of x and of (x - mean)^2 under the closed-form
    prior must match the prior's mean and variance within 4 standard errors of the between-chain spread."""
    parts, done = [], 0
    while done < n_iter:
        k = min(chunk, n_iter - done)
        parts.append(ch.run(k, every)[:, :, :20].copy())
        done += k
    recs = np.concatenate(parts)
    r = recs[int(burnin * recs.shape[0]):]
    for name, col in cols.items():
        mean, var = want[name]
        x = r[:, :, col]
        m = x.mean(0)
        v = ((x - mean) ** 2).mean(0)
        for got, w in ((m, mean), (v, var)):
            z = abs(got.mean() - w) / (got.std(ddof=1) / np.sqrt(len(got)))
            assert z < 4, (name, got.mean(), w, z)


def test_beta_zero_samples_the_prior(device, tmp_path):
    """Chains fixed at beta = 0, no swaps: the parameters whose moves cross their prior within the budget have the prior's
    moments.  K6: l_min, m_min ~ Gamma(1, scale 10, loc .001), delta, gamma ~ Gamma(3, scale .5) (alpha / beta are skipped:
    their additive steps of .001 cannot cross N(0, 5)).  K7 (-m_birth 3 -m_death 2): the Gamma parameters the multiplier
    moves and m_mul ~ Beta(1, 1.2) (x0 is skipped: its flat prior is improper, DDRatev3.py:139-140)."""
    g1 = lambda s, loc=0.0: (s + loc, s * s)
    g3 = (1.5, 0.75)
    st, bins, trend, otrend, k6 = trend_setup(device, tmp_path, "ex_ramp", n_chains=256, seed=31)
    k6.set_beta(0.0)
    _prior_moments(k6, 1_000_001, 1000, {"l_min": 5, "m_min": 6, "delta": 9, "gamma": 10},
                   {"l_min": g1(10, .001), "m_min": g1(10, .001), "delta": g3, "gamma": g3})
    S, k7 = dd_setup(device, tmp_path, "ex_g_mddn", mb=3, md=2, n_chains=256, seed=32)
    k7.set_beta(0.0)
    k0l = float(np.max(S.bins.dt))
    a, b = 1.0, 1.2
    _prior_moments(k7, 2_000_001, 1000, {"l_f": 5, "l_mul": 6, "k": 7, "div_0": 9, "L": 10, "m_mul": 11, "nuB": 12, "nuD": 13,
                                            "g_l1": 14, "g_l2": 15},
                   {"l_f": g1(10), "l_mul": g1(1), "k": g1(10), "div_0": g1(k0l), "L": g1(k0l), "nuB": g3, "nuD": g3, "g_l1": g1(10),
                    "g_l2": g1(10), "m_mul": (a / (a + b), a * b / ((a + b) ** 2 * (a + b + 1)))})
    assert np.all(k6.temper()[0] == 0.0) and np.all(k7.temper()[1] == 0)


def _imputations(data, tmp_path):
    """A directory of two imputations of `data`: the second moves some birth times by a year inside the same window."""
    d = os.path.join(str(tmp_path), "tables")
    os.makedirs(d)
    rows = [l.split("\t") for l in open(data).read().splitlines()[1:]]
    for i in range(2):
        with open(os.path.join(d, "imp_%d.tsv" % i), "w") as fh:
            fh.write("id\tts\tte\n")
            for j, r in enumerate(rows):
                ts, te = int(float(r[-2])), int(float(r[-1]))
                if i and 1996 < ts < 2010 and te - ts > 2 and j % 3 == 0:
                    ts += 1
                fh.write("%s\t%d\t%d\n" % (r[0], ts, te))
    return d


def _trend_job(tmp_path):
    job = [j for j in trend_jobs() if j["tag"] == "ex_ramp"][0]
    data, trend_path = trend_stage(job, tmp_path)
    return data, trend_path


def test_trendrate_command_line_logs_cold_rows(device, tmp_path, capsys):
    data, trend_path = _trend_job(tmp_path)
    base = ["-trend_data", trend_path, "-trend_index", "1", "-n", "3001", "-s", "50", "-seed", "1", "-chains", "3"]
    plain = TR.run(TR.build_parser().parse_args(["-d", data] + base + ["-quiet", "1"]), device=device)
    plain_rows = [len(open(p).read().splitlines()) for p in plain]
    for p in plain:
        os.rename(p, p + ".plain")
    capsys.readouterr()
    temp = TR.run(TR.build_parser().parse_args(["-d", data] + base + ["-temper", "4", "-swap_every", "200"]), device=device)
    assert "swap rounds" in capsys.readouterr().out
    assert temp == plain and [len(open(p).read().splitlines()) for p in temp] == plain_rows
    otrend = TO.normalise_trend(TO.read_trend_column(trend_path, 1))
    ts, te, present, origin = TO.parse_ts_te(data)
    bins = TO.create_bins(origin, present, ts, te)
    for p in temp:
        assert open(p).readline() == open(p + ".plain").readline()
        for row in np.loadtxt(p, skiprows=1):
            lk, _, _ = TO.likelihood(row[6:12], bins, otrend)
            np.testing.assert_allclose(row[3:5], lk, rtol=RTOL)        # the row's likelihood is the untempered one of its state
    # a directory of tables: every ladder stays on its table
    d = _imputations(data, tmp_path)
    paths = TR.run(TR.build_parser().parse_args(["-d", d] + base[:-1] + ["4", "-temper", "2", "-quiet", "1"]), device=device)
    assert [os.path.basename(p) for p in paths] == ["imp_%d_%d_EXPB_EXPD_1.trendrate.log" % (k % 2, 1 + k // 2) for k in range(4)]
    for k, p in enumerate(paths):
        ts, te, present, origin = TO.parse_ts_te(os.path.join(d, "imp_%d.tsv" % (k % 2)))
        tb = TO.create_bins(origin, present, ts, te)
        for row in np.loadtxt(p, skiprows=1):
            lk, _, _ = TO.likelihood(row[6:12], tb, otrend)
            np.testing.assert_allclose(row[3:5], lk, rtol=RTOL)


def test_ddrate_command_line_logs_cold_rows(device, tmp_path, capsys):
    job = [j for j in dd_jobs() if j["tag"] == "ex_g_mddn"][0]
    data, genre = dd_stage(job, tmp_path)
    base = ["-d", data, "-m_birth", "3", "-g", genre, "-n", "3001", "-s", "50", "-seed", "1", "-chains", "3"]
    plain = DD.run(DD.build_parser().parse_args(base + ["-quiet", "1"]), device=device)
    plain_rows = [len(open(p).read().splitlines()) for p in plain]
    for p in plain:
        os.rename(p, p + ".plain")
    capsys.readouterr()
    temp = DD.run(DD.build_parser().parse_args(base + ["-temper", "4", "-swap_every", "200"]), device=device)
    assert "swap rounds" in capsys.readouterr().out
    assert temp == plain and [len(open(p).read().splitlines()) for p in temp] == plain_rows
    ts, te, present, origin = L.parse_ts_te(data)
    gts, gte, _, _ = L.parse_ts_te(genre)
    S = D.Setup(D.create_bins(origin, present, ts, te, 0), 3, 2, gts, gte)
    for p in temp:
        assert open(p).readline() == open(p + ".plain").readline()
        assert open(p[:-4] + ".div.log").read()                  # the sibling .div.log is written as without -temper
        for row in np.loadtxt(p, skiprows=1):
            q = row[6:17].copy()
            q[3] -= S.origin
            q[5] -= q[4]
            lk = np.asarray(D.likelihood(q, S)[0])
            np.testing.assert_allclose(row[3:5], lk[:2], rtol=RTOL)
            np.testing.assert_allclose(row[2], lk.sum(), rtol=RTOL)
    # a directory of tables: every ladder stays on its table
    d = _imputations(data, tmp_path)
    paths = DD.run(DD.build_parser().parse_args(["-d", d, "-m_birth", "2", "-m_death", "2", "-n", "2001", "-s", "100", "-seed", "1",
                                                 "-chains", "4", "-temper", "2", "-quiet", "1"]), device=device)
    assert [os.path.basename(p) for p in paths] == ["imp_%d_%d_LDDN_MDDN.log" % (k % 2, 1 + k // 2) for k in range(4)]
    tabs = [L.parse_ts_te(os.path.join(d, "imp_%d.tsv" % i)) for i in range(2)]
    present, origin = max(t[2] for t in tabs), min(t[3] for t in tabs)
    for k, p in enumerate(paths):
        ts, te = tabs[k % 2][0], tabs[k % 2][1]
        Sk = D.Setup(D.create_bins(origin, present, ts, te, 0), 2, 2)
        for row in np.loadtxt(p, skiprows=1):
            q = row[6:17].copy()
            q[3] -= Sk.origin
            q[5] -= q[4]
            np.testing.assert_allclose(row[3:5], np.asarray(D.likelihood(q, Sk)[0])[:2], rtol=RTOL)
