"""CPU: the host restatement of split R-hat and ESS (diagnostics.rhat_ess) on worked and simulated cases, and the diagnosed
columns of sample logs written through the product's own writers against the records that produced them."""
import math
import os

import numpy as np
import pytest

from literate_b200 import ddrate as DD
from literate_b200 import diagnostics as D
from literate_b200 import engine as E
from literate_b200 import forward as F
from literate_b200 import plotdd as PD
from literate_b200 import summary as S
from literate_b200 import trend as TR
from test_plotdd_host import synthetic_records, write_logs


def ar1(rng, chains, draws, rho):
    e = rng.normal(size=(chains, draws))
    x = np.empty_like(e)
    x[:, 0] = e[:, 0] / math.sqrt(1.0 - rho * rho)
    for i in range(1, draws):
        x[:, i] = rho * x[:, i - 1] + e[:, i]
    return x


def test_hand_worked_two_chains_of_six():
    # split chains [1 2 3] [4 5 6] [2 4 6] [8 10 12]: means 2 5 4 10, acov(0) 2/3 2/3 8/3 8/3, acov(1) 0; n = 3
    x = np.array([[1., 2, 3, 4, 5, 6], [2, 4, 6, 8, 10, 12]])
    r = D.rhat_ess(x)
    W = 1.5 * (5.0 / 3.0)                                     # n/(n-1) mean_j acov_j(0) = 5/2
    between = 139.0 / 12.0                                    # var(2, 5, 4, 10; ddof 1)
    varp = 2.0 / 3.0 * W + between                            # 53/4
    assert r["mean"] == 5.25
    assert r["sd"] == pytest.approx(math.sqrt(53 / 4), rel=1e-15)
    assert r["rhat"] == pytest.approx(math.sqrt(varp / W), rel=1e-15) and r["rhat"] == pytest.approx(math.sqrt(5.3), rel=1e-15)
    # rho_1 = 43/53; n - 3 = 0: Geyer's loop does not start, max_t = -1, tau = -1 + rho[0] = 0 -> clamped to 1/log10(12)
    assert r["lag"] == -1
    assert r["ess"] == pytest.approx(12 * math.log10(12), rel=1e-15)


@pytest.mark.parametrize("rho", [0.0, 0.5, 0.9])
def test_ar1_chains(rho):
    x = ar1(np.random.default_rng(int(rho * 10) + 3), 64, 4000, rho)
    r = D.rhat_ess(x)
    want = (1 - rho) / (1 + rho)
    assert abs(r["ess"] / x.size / want - 1) < 0.10, (r, want)
    assert r["rhat"] < 1.01
    assert r["lag"] >= 1 and r["lag"] % 2 == 1


def test_shifted_chain_raises_rhat():
    x = np.random.default_rng(5).normal(size=(4, 1000))
    assert D.rhat_ess(x)["rhat"] < 1.01
    x[0] += 1.0
    assert D.rhat_ess(x)["rhat"] > 1.05


def test_antithetic_chain_meets_the_tau_clamp():
    x = ar1(np.random.default_rng(6), 4, 2000, -0.9)
    r = D.rhat_ess(x)
    mn = 8 * 1000
    assert r["ess"] == pytest.approx(mn * math.log10(mn), rel=1e-14)     # tau would be ~0.05 < 1/log10(mn)


def test_odd_draws_drop_the_middle_and_too_few_raise():
    x = np.random.default_rng(7).normal(size=(3, 101))
    want = D.rhat_ess(np.delete(x, 50, axis=1))
    x[:, 50] = np.nan                                         # the dropped draw is never looked at
    assert D.rhat_ess(x) == want
    for s in (1, 2, 3):
        with pytest.raises(RuntimeError, match="not enough data"):
            D.rhat_ess(np.ones((2, s)))
    assert D.rhat_ess(x[:, :5])["lag"] == -1 and np.isfinite(D.rhat_ess(x[:, :5])["ess"])


def test_degenerate_columns():
    r = D.rhat_ess(np.full((3, 40), 0.1))                     # constant: means exactly 0.1, W = 0 and var+ = 0
    assert r["mean"] == pytest.approx(0.1, rel=1e-15) and r["sd"] == 0.0 and math.isnan(r["rhat"]) and math.isnan(r["ess"]) and r["lag"] == -1
    st = np.repeat(np.array([[0.1], [0.2], [0.3]]), 40, axis=1)   # every split chain stuck on its own value
    r = D.rhat_ess(st)
    assert r["rhat"] == math.inf and math.isnan(r["ess"]) and r["lag"] == -1 and r["sd"] > 0
    halves = np.concatenate([np.full((2, 20), 1.0), np.full((2, 20), 2.0)], axis=1)   # stuck within split chains only
    assert D.rhat_ess(halves)["rhat"] == math.inf
    for bad in (np.nan, np.inf, -np.inf):
        x = np.random.default_rng(8).normal(size=(2, 30))
        x[1, 3] = bad
        r = D.rhat_ess(x)
        assert all(math.isnan(r[k]) for k in ("mean", "sd", "rhat", "ess")) and r["lag"] == -1
    assert [D.flag(*v) for v in ((float("nan"), float("nan"), -1, float("nan")), (math.inf, float("nan"), -1, 1.0),
                                 (float("nan"), float("nan"), -1, 1.0), (1.02, 150.0, 7, 1.0), (1.0, 150.0, 7, 1.0),
                                 (1.02, 500.0, 7, 1.0), (1.0, 500.0, 7, 1.0), (1.0, 80.0, -1, 1.0))] == \
        ["nonfinite", "stuck", "const", "rhat+ess", "ess", "rhat", "ok", "ess"]


@pytest.mark.parametrize("kind,genre", [("trendrate", False), ("dd", False), ("dd", True)])
def test_columns_follow_the_log_header(kind, genre):
    nb = 7
    names = [c[0] for c in D.diagnostic_columns(kind, nb, 1850.0, genre)]
    head = TR.header(nb) if kind == "trendrate" else DD.header(nb, 3 if genre else 2)
    assert names == [h for h in head if h != "it"] + ["net_%d" % j for j in range(nb)]
    assert [c[0] for c in D.diagnostic_columns("forward", nb)] == [c for c in F.MCMC_COLS if c not in ("it", "root_age", "death_age")]


def _record_columns(recs, specs, burnin):
    r = recs[S.burnin_index(recs.shape[0], burnin):]
    return PD._host_columns(r.reshape(-1, r.shape[-1]), specs).reshape(r.shape[0], r.shape[1], len(specs))


@pytest.mark.parametrize("kind,variant", [("trendrate", (False, False, False)), ("dd", (0, 2)), ("dd", (3, 1))])
def test_sibling_logs_equal_records(tmp_path, kind, variant):
    nb, origin = 9, 1850.0
    recs = synthetic_records(kind, 45, 3, nb, seed=4)
    paths = write_logs(str(tmp_path), kind, recs, nb, variant, origin)
    genre = kind == "dd" and variant[0] == 3
    cols = D.diagnostic_columns(kind, nb, origin, genre)
    got_kind, names, x = D.log_draws(paths, 0.2)
    assert got_kind == kind and names == [c[0] for c in cols]
    want = _record_columns(recs, [c[1] if np.ndim(c[1]) else (c[1], -1, 1, 0.0) for c in cols], 0.2)
    assert np.array_equal(x, want)
    assert D.find_logs(str(tmp_path)) == {kind: sorted(paths)}


def forward_records(rng, n_samples, n_chains, start, end):
    """Seeded K3-like records: rates, shift times inside (start, end), parameters; field [13] clear so that the log's
    poisson_rate_hp is field [9]."""
    r = np.zeros((n_samples, n_chains, E.LR_REC_DOUBLES))
    r[..., E.REC_IT] = np.arange(n_samples)[:, None] * 10
    r[..., E.REC_LIK] = -rng.uniform(1000, 2000, (n_samples, n_chains))
    r[..., E.REC_PRIOR] = -rng.uniform(1, 20, (n_samples, n_chains))
    r[..., E.REC_LAVG:E.REC_MAVG + 1] = rng.gamma(2.0, 0.1, (n_samples, n_chains, 2))
    r[..., E.REC_GL:E.REC_POI + 1] = rng.gamma(2.0, 1.0, (n_samples, n_chains, 3))
    r[..., E.REC_ADQ:E.REC_ADQ + 3] = rng.uniform(0, 1, (n_samples, n_chains, 3))
    r[..., E.REC_BETA] = 1.0
    for s in range(n_samples):
        for c in range(n_chains):
            for side, (kf, rf, tf) in enumerate(((E.REC_KL, E.REC_L, E.REC_TL), (E.REC_KM, E.REC_M, E.REC_TM))):
                k = int(rng.integers(1, 5))
                r[s, c, kf] = k
                r[s, c, rf:rf + k] = rng.gamma(2.0, 0.1, k)
                r[s, c, tf:tf + k] = np.concatenate([[start], np.sort(rng.uniform(start + 1, end - 1, k - 1))])
    return r


def test_forward_logs_equal_records(tmp_path):
    start, end, M, Sn = 1800.0, 1830.5, 3, 40
    recs = forward_records(np.random.default_rng(9), Sn, M, start, end)
    paths = []
    for c in range(M):
        w = F.ChainLogWriter(os.path.join(str(tmp_path), "t_BD_chain%d" % c), 1, False, start, end, 0, 0.0)
        for s in range(Sn):
            w.write(recs[s, c])
        w.close()
        paths.append(w.mcmc.name)
    kind, names, x = D.log_draws(paths, 0.25)
    edges = np.arange(start, end)
    nb = len(edges) - 1
    assert kind == "forward" and names == [c[0] for c in D.FORWARD_COLS] + sum(D._bin_names(nb), [])
    specs = [c[1] if np.ndim(c[1]) else (c[1], -1, 1, 0.0) for c in D.FORWARD_COLS]
    want = _record_columns(recs, specs, 0.25)
    assert np.array_equal(x[:, :, :len(specs)], want)
    r = recs[S.burnin_index(Sn, 0.25):]
    for c in range(M):
        rr = r[:, c]
        mb = S.marginal_matrix(rr[:, E.REC_L:E.REC_L + E.LR_KMAX], rr[:, E.REC_TL + 1:E.REC_TL + E.LR_KMAX], rr[:, E.REC_KL].astype(int), edges)
        md = S.marginal_matrix(rr[:, E.REC_M:E.REC_M + E.LR_KMAX], rr[:, E.REC_TM + 1:E.REC_TM + E.LR_KMAX], rr[:, E.REC_KM].astype(int), edges)
        assert np.array_equal(x[:, c, len(specs):], np.concatenate([mb, md, mb - md], axis=1))
    assert D.find_logs(str(tmp_path)) == {"forward": sorted(paths)}


def test_logs_of_different_lengths_are_cut(tmp_path):
    recs = synthetic_records("trendrate", 30, 2, 5, seed=1)
    p0 = write_logs(str(tmp_path), "trendrate", recs, 5, (False, False, False), 0.0)
    with open(p0[1]) as fh:
        lines = fh.readlines()
    with open(p0[1], "w") as fh:
        fh.writelines(lines[:-10])
    notes = []
    _, _, x = D.log_draws(p0, 0.2, note=notes.append)
    assert x.shape[0] == 20 - S.burnin_index(20, 0.2) and len(notes) == 1
