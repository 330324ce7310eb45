"""GPU: K9 (lr_chain_diagnostics) against the host restatement diagnostics.rhat_ess -- mean, sd and R-hat to 1e-12, ESS to 1e-9
(relative), lags equal -- on simulated columns, tempered runs of all three samplers, K5's per-bin matrices, and the diagnose
command line on logs of the sampling command lines."""
import math
import os

import numpy as np
import pytest
import torch

from literate_b200 import diagnose as DG
from literate_b200 import diagnostics as D
from literate_b200 import engine as E
from literate_b200 import forward as F
from literate_b200 import parallel as P
from literate_b200 import summary as S
from literate_b200 import synth
from literate_b200 import ddrate as DD
from literate_b200 import trend as TR
from test_gpu_sibling_tempering import _synthetic
from test_oracle_ddrate_golden import _jobs as dd_jobs, stage as dd_stage
from test_oracle_trend_golden import _jobs as trend_jobs, stage as trend_stage

pytestmark = pytest.mark.gpu


def _spec(c):
    return (c, -1, 1, 0.0) if np.ndim(c) == 0 else (tuple(c) + (0.0,))[:4]


def _host_values(recs, specs):
    """[S, chains, w] records -> [S, chains, n_cols] column values, the fp64 operations of the kernel in its order."""
    out = np.empty(recs.shape[:2] + (len(specs),))
    for j, c in enumerate(specs):
        a, b, sg, add = _spec(c)
        v = recs[..., a]
        if b >= 0:
            v = v + recs[..., b] if sg > 0 else v - recs[..., b]
        out[..., j] = v + add if add != 0.0 else v
    return out


def _rel_ok(got, want, rtol):
    both_nan = np.isnan(got) & np.isnan(want)
    same = got == want
    with np.errstate(invalid="ignore"):
        close = np.abs(got - want) <= rtol * np.abs(want)
    return both_nan | same | close


def assert_matches(got, host, names=None):
    """Device outputs (dict of tensors or Diagnostics) against rhat_ess_columns; columns whose Geyer decision lies within 1e-12 of
    zero on the host are excused (returned count)."""
    val = lambda v: v.cpu().numpy() if torch.is_tensor(v) else np.asarray(v)
    g = {k: val(got[k] if isinstance(got, dict) else getattr(got, k)).astype(np.float64) for k in ("mean", "sd", "rhat", "ess", "lag")}
    excused = host["margin"] < 1e-12
    for k, tol in (("mean", 1e-12), ("sd", 1e-12), ("rhat", 1e-12), ("ess", 1e-9)):
        ok = _rel_ok(g[k], host[k], tol) | excused
        assert ok.all(), (k, [(names[i] if names else i, g[k][i], host[k][i]) for i in np.flatnonzero(~ok)[:5]])
    ok = (g["lag"] == host["lag"]) | excused
    assert ok.all(), [(names[i] if names else i, g["lag"][i], host["lag"][i]) for i in np.flatnonzero(~ok)[:5]]
    return int(excused.sum())


def _columns(rng, S, M):
    """records [S, M, 12]: AR(1) 0.5 and 0.9, integers, a constant, per-chain constants (stuck), +-inf, NaN, a shifted chain,
    two noise fields for the spec columns."""
    def ar(rho):
        e = rng.normal(size=(M, S))
        x = np.empty_like(e)
        x[:, 0] = e[:, 0] / math.sqrt(1 - rho * rho)
        for i in range(1, S):
            x[:, i] = rho * x[:, i - 1] + e[:, i]
        return x.T
    r = np.empty((S, M, 12))
    r[..., 0] = ar(0.5)
    r[..., 1] = 1e4 + ar(0.9)
    r[..., 2] = rng.integers(0, 4, (S, M))
    r[..., 3] = 0.1
    r[..., 4] = np.arange(M)[None, :] * 0.25
    r[..., 5] = rng.normal(size=(S, M))
    r[0, rng.integers(0, M), 5] = np.inf if S > 4 else -np.inf          # sample 0: never the dropped middle draw
    r[..., 6] = rng.normal(size=(S, M))
    r[S - 1, rng.integers(0, M), 6] = np.nan
    r[..., 7] = rng.normal(size=(S, M)) + (np.arange(M) == 0)[None, :]
    r[..., 8] = rng.gamma(2.0, 0.1, (S, M))
    r[..., 9] = rng.gamma(2.0, 0.1, (S, M))
    r[..., 10] = -rng.exponential(1.0, (S, M))
    r[..., 11] = 7.0
    return r


SPECS = list(range(11)) + [(8, 9, -1), (8, 9, 1, 1850.0), (0, 10, 1, -3.5), (11, 3, 1)]


@pytest.mark.parametrize("S", [4, 5, 1000, 4001])
@pytest.mark.parametrize("M", [1, 2, 7, 256])
def test_kernel_equals_restatement(device, S, M):
    recs = _columns(np.random.default_rng(S * 1000 + M), S, M)
    d = torch.from_numpy(recs).cuda()
    got = device.chain_diagnostics_device(d, SPECS)
    host = D.rhat_ess_columns(_host_values(recs, SPECS))
    assert assert_matches(got, host) == 0
    assert got["lag"][3].item() == -1 and math.isnan(got["rhat"][3].item())                     # constant
    if M > 1:
        assert got["rhat"][4].item() == math.inf                                                # stuck
    assert math.isnan(got["mean"][5].item()) and math.isnan(got["mean"][6].item())              # +-inf, NaN
    again = device.chain_diagnostics_device(d, SPECS)
    for k in got:
        assert np.array_equal(got[k].cpu().numpy().view(np.int64), again[k].cpu().numpy().view(np.int64)), k


def test_long_and_slow_columns(device):
    rng = np.random.default_rng(3)
    S = 1 << 20
    x = np.empty((S, 2, 2))
    for c in range(2):
        x[:, c, 0] = _ar_filter(rng.normal(size=S), 0.5)        # AR(1) 0.5, 2 chains x 2^20 draws
        x[:, c, 1] = np.cumsum(rng.normal(size=S))             # random walk
    got = device.chain_diagnostics_device(torch.from_numpy(x[..., :1].copy()).cuda(), [0])
    assert assert_matches(got, D.rhat_ess_columns(x[..., :1])) == 0
    slow = np.cumsum(rng.normal(size=(1000, 4, 1)), axis=0)      # Geyer's sequence runs to its end: lag n - 5 for n = 500
    got = device.chain_diagnostics_device(torch.from_numpy(slow).cuda(), [0])
    host = D.rhat_ess_columns(slow)
    assert assert_matches(got, host) == 0 and host["lag"][0] == 495


def _ar_filter(e, rho):
    from scipy.signal import lfilter
    return lfilter([1.0], [1.0, -rho], e)


@pytest.mark.parametrize("kind", ["trend", "dd"])
def test_tempered_siblings(device, kind):
    T, n = 4, 16
    ch = _synthetic(device, kind, 24, n, 9)
    ch.set_beta(np.tile(P.temperature_ladder(T, 0.3), n // T))
    recs, _ = ch.run_tempered(8001, 20, T, 200)
    k = "trendrate" if kind == "trend" else "dd"
    cols = D.diagnostic_columns(k, 24)
    got = D.diagnose_records_device(device, torch.from_numpy(recs).cuda(), k, 24, burnin=0.2, ladder=T)
    cold = E.cold_records(recs, T, ch.REC_BETA)
    cold = cold[S.burnin_index(cold.shape[0], 0.2):]
    assert assert_matches(got, D.rhat_ess_columns(_host_values(cold, [c[1] for c in cols])), got.names) == 0
    bad = recs.copy()
    bad[7, 0:T, ch.REC_BETA] = 0.5
    with pytest.raises(ValueError, match="beta = 1"):
        device.chain_diagnostics_device(torch.from_numpy(bad).cuda(), [5], T, ch.REC_BETA)


def _forward_run(device, n_chains, T=1, n_iter=20001, every=100):
    ts, te = synth.syn_int(20_000)
    stats = device.bin_stats(ts, te)
    start, end = float(ts.min()), float(te.max())
    ds = E.Dataset(device, stats, 0, start, end)
    ch = E.Chains(ds, n_chains * T, 5)
    if T > 1:
        ch.set_beta(np.tile(P.temperature_ladder(T, 0.3), n_chains))
        recs, _ = ch.run_tempered(n_iter, every, T, 500)
    else:
        recs = ch.run(n_iter, every)
    ch.close(); ds.close()
    return recs, start, end


def _forward_host(recs, start, end, burnin):
    r = recs[S.burnin_index(recs.shape[0], burnin):]
    edges = np.arange(start, end)
    vals = _host_values(r, [c[1] for c in D.FORWARD_COLS])
    mats = []
    for c in range(r.shape[1]):
        rr = r[:, c]
        mb = S.marginal_matrix(rr[:, E.REC_L:E.REC_L + E.LR_KMAX], rr[:, E.REC_TL + 1:E.REC_TL + E.LR_KMAX], rr[:, E.REC_KL].astype(int), edges)
        md = S.marginal_matrix(rr[:, E.REC_M:E.REC_M + E.LR_KMAX], rr[:, E.REC_TM + 1:E.REC_TM + E.LR_KMAX], rr[:, E.REC_KM].astype(int), edges)
        mats.append(np.concatenate([mb, md, mb - md], axis=1))
    return np.concatenate([vals, np.stack(mats, axis=1)], axis=2), len(edges) - 1


def test_forward_records_and_marginals(device):
    recs, start, end = _forward_run(device, 8)
    host, nb = _forward_host(recs, start, end, 0.2)
    got = D.diagnose_records_device(device, torch.from_numpy(recs).cuda(), "forward", nb, burnin=0.2, origin=start)
    assert len(got.names) == host.shape[2]
    assert assert_matches(got, D.rhat_ess_columns(host), got.names) == 0


def test_tempered_forward(device):
    T = 4
    recs, start, end = _forward_run(device, 4, T)
    cold = E.cold_records(recs, T)
    host, nb = _forward_host(cold, start, end, 0.2)
    got = D.diagnose_records_device(device, torch.from_numpy(recs).cuda(), "forward", nb, burnin=0.2, ladder=T, origin=start)
    assert assert_matches(got, D.rhat_ess_columns(host), got.names) == 0
    bad = recs.copy()
    bad[-1, :T, E.REC_BETA] = 0.5
    with pytest.raises(ValueError, match="beta = 1"):
        D.diagnose_records_device(device, torch.from_numpy(bad).cuda(), "forward", nb, ladder=T, origin=start)


def test_all_ddrate_columns_within_the_workspace_bound():
    dev = E.Device(0)                                           # a fresh handle: its workspace grows from nothing
    nb = 200
    rng = np.random.default_rng(1)
    brk = 20 + 400 / (1 + np.exp(-0.3 * (np.arange(nb) - nb / 2))) + rng.uniform(0, 5, nb)
    dd = DD.DDChains(dev, rng.poisson(brk * 0.2), rng.poisson(brk * 0.1), brk, 0.0, nb + 1.5, 2, 2, n_chains=64, seed=1)
    dd.run(2000)
    recs = torch.empty((200, 64, dd.rec_doubles), dtype=torch.float64, device="cuda")
    dd.run_device(20000, 100, recs)
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info()[0]
    got = D.diagnose_records_device(dev, recs, "dd", nb, burnin=0.0)
    grown = free0 - torch.cuda.mem_get_info()[0]
    assert grown <= (300 << 20), grown
    cols = D.diagnostic_columns("dd", nb)
    assert len(got.names) == len(cols) > 1011
    host = D.rhat_ess_columns(_host_values(recs.cpu().numpy(), [c[1] for c in cols]))
    assert assert_matches(got, host, got.names) == 0


def test_bad_specs_are_refused(device):
    d = torch.zeros((10, 2, 4), dtype=torch.float64, device="cuda")
    for cols in ([4], [(0, 4, 1)], [(0, 1, 2)], [-1]):
        with pytest.raises(E.NativeError, match="lr_chain_diagnostics"):
            device.chain_diagnostics_device(d, cols)
    with pytest.raises(E.NativeError, match="lr_chain_diagnostics"):
        device.chain_diagnostics_device(d, [0], ladder=2, beta_col=4)
    with pytest.raises(RuntimeError, match="not enough data"):
        device.chain_diagnostics_device(d[:3], [0])


def _write_table(path, ts, te_year):
    with open(path, "w") as fh:
        fh.write("clade\tts\tte\n")
        for i, (a, b) in enumerate(zip(ts, te_year)):
            fh.write("%d\t%d\t%d\n" % (i, a, b))


def _tsv(path):
    rows = [l.rstrip("\n").split("\t") for l in open(path)]
    assert rows[0] == ["column", "mean", "sd", "rhat", "ess", "mcse", "lag", "flag"]
    return {r[0]: r[1:] for r in rows[1:]}


def _check_tsv(path, logs):
    _, names, x = D.log_draws(logs, 0.2)
    host = D.rhat_ess_columns(x)
    tab = _tsv(path)
    assert list(tab) == names
    got = {k: np.array([float(tab[nm][i]) for nm in names]) for i, k in enumerate(("mean", "sd", "rhat", "ess"))}
    got["lag"] = np.array([int(tab[nm][5]) for nm in names])
    assert assert_matches(got, host, names) == 0
    for nm in names:
        fl = tab[nm][6]
        assert fl in D.FLAGS


def test_diagnose_command_line(device, tmp_path):
    fwd = tmp_path / "fwd"
    fwd.mkdir()
    ts, te = synth.syn_int(3000)
    _write_table(str(fwd / "t.tsv"), ts, te - 0.5)
    F.main(["-d", str(fwd / "t.tsv"), "-n", "20000", "-s", "100", "-p", "100000", "-seed", "2", "-chains", "4", "-quiet", "1"])
    job = [j for j in trend_jobs() if j["tag"] == "ex_ramp"][0]
    data, trend_path = trend_stage(job, tmp_path)
    TR.main(["-d", data, "-trend_data", trend_path, "-trend_index", "1", "-n", "3001", "-s", "50", "-seed", "3", "-chains", "4", "-quiet", "1"])
    job = [j for j in dd_jobs() if j["tag"] == "ex_g_mddn"][0]
    data, genre = dd_stage(job, tmp_path)
    DD.main(["-d", data, "-m_birth", "3", "-g", genre, "-n", "3001", "-s", "50", "-seed", "3", "-chains", "4", "-quiet", "1"])
    logdir = str(fwd / "literate_mcmc_logs")
    assert DG.main([logdir]) == [os.path.join(logdir, "diagnostics_forward.tsv")]
    _check_tsv(os.path.join(logdir, "diagnostics_forward.tsv"), D.find_logs(logdir)["forward"])
    out = DG.main([str(tmp_path), "-rhat_max", "1.05", "-ess_min", "100"])
    logs = D.find_logs(str(tmp_path))
    assert sorted(logs) == ["dd", "trendrate"] and len(logs["dd"]) == 4 and len(logs["trendrate"]) == 4
    for kind in logs:
        p = os.path.join(str(tmp_path), "diagnostics_%s.tsv" % kind)
        assert p in out
        _check_tsv(p, logs[kind])


@pytest.mark.parametrize("disagree", [True, False])
def test_tables_that_disagree(device, tmp_path, disagree):
    ts0, te0 = synth.syn_int(5000, replicate=0)
    y0 = te0 - 0.5
    if disagree:
        ts1, y1 = ts0, ts0 + np.floor((y0 - ts0) / 2)          # every lifetime halved: about twice the death rate
    else:
        # the same lineages in another order: two independent replicates would give posteriors about one posterior sd apart,
        # i.e. an R-hat near sqrt(1 + chi2_1 / 2) ~ 1.1 whatever their size, which is a correct answer, not a control
        perm = np.random.default_rng(1).permutation(len(ts0))
        ts1, y1 = ts0[perm], y0[perm]
    _write_table(str(tmp_path / "a.tsv"), ts0, y0)
    _write_table(str(tmp_path / "b.tsv"), ts1, y1)
    F.main(["-d", str(tmp_path), "-n", "40000", "-s", "100", "-p", "100000", "-seed", "4", "-chains", "4", "-quiet", "1",
            "-const_rates", "1"])
    logdir = str(tmp_path / "literate_mcmc_logs")
    DG.main([logdir])
    tab = _tsv(os.path.join(logdir, "diagnostics_forward.tsv"))
    rhat = float(tab["mu_avg"][2])
    assert (rhat > 1.1) if disagree else (rhat < 1.05), rhat
