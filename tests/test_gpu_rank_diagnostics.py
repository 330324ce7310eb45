"""GPU: K10 (lr_rank_transform, lr_rank_diagnostics) against the host restatement diagnostics.rank_rhat_ess -- the transform
itself (ranks, z, median and quantiles bit for bit, indicators), R-hats to 1e-12 and ESS to 1e-9 (relative), tempered and
RJMCMC records with K5's per-bin matrices, all DDRate columns within the workspace bound, a column of 2 M draws, and
`diagnose -rank 1`."""
import math
import os

import numpy as np
import pytest
import torch
from scipy.special import ndtri

from literate_b200 import diagnose as DG
from literate_b200 import diagnostics as D
from literate_b200 import engine as E
from literate_b200 import forward as F
from literate_b200 import parallel as P
from literate_b200 import summary as S
from literate_b200 import synth
from literate_b200 import ddrate as DD
from literate_b200 import trend as TR
from test_gpu_diagnostics import SPECS, _columns, _forward_host, _forward_run, _host_values, _rel_ok, _tsv, _write_table
from test_gpu_sibling_tempering import _synthetic
from test_oracle_ddrate_golden import _jobs as dd_jobs, stage as dd_stage
from test_oracle_trend_golden import _jobs as trend_jobs, stage as trend_stage

pytestmark = pytest.mark.gpu

RHATS = ("rhat_bulk", "rhat_tail", "rhat_rank")
ESSES = ("ess_bulk", "ess_tail")


def bits(a):
    return np.asarray(a, dtype=np.float64).view(np.int64)


def assert_rank_matches(got, host, names=None):
    """Device rank outputs (dict of tensors or Diagnostics) against rank_rhat_ess_columns: median and quantiles bit for bit,
    R-hats to 1e-12, ESS to 1e-9; columns whose Geyer decision lies within 1e-12 of zero on the host are excused."""
    val = lambda v: v.cpu().numpy() if torch.is_tensor(v) else np.asarray(v)
    g = {k: val(got[k] if isinstance(got, dict) else getattr(got, k)).astype(np.float64) for k in E.RANK_FIELDS}
    excused = host["margin"] < 1e-12
    for k in ("median", "q05", "q95"):
        ok = (bits(g[k]) == bits(host[k])) | (np.isnan(g[k]) & np.isnan(host[k]))
        assert ok.all(), (k, [(names[i] if names else i, g[k][i], host[k][i]) for i in np.flatnonzero(~ok)[:5]])
    for k, tol in [(k, 1e-12) for k in RHATS] + [(k, 1e-9) for k in ESSES]:
        ok = _rel_ok(g[k], host[k], tol) | excused
        assert ok.all(), (k, [(names[i] if names else i, g[k][i], host[k][i]) for i in np.flatnonzero(~ok)[:5]])
    return int(excused.sum())


def _z_ref(v):
    """Phi^-1 of the exact ratio (r - 3/8) / (N + 1/4), from the smaller tail (both numerators exact)."""
    return D.rank_normal(v)


def _split_draws(vals):
    """[S, M, cols] -> [2n, M, cols], the split draws in the row order of Z."""
    Sd = vals.shape[0]
    n = Sd // 2
    return np.concatenate([vals[:n], vals[Sd - n:]], axis=0)


@pytest.mark.parametrize("S", [4, 5, 41, 1000, 4001])
@pytest.mark.parametrize("M", [1, 2, 7, 256])
def test_transform(device, S, M):
    recs = _columns(np.random.default_rng(S * 1000 + M + 7), S, M)
    vals = _host_values(recs, SPECS)
    k = len(SPECS)
    Z, quant = device.rank_transform_device(torch.from_numpy(recs).cuda(), SPECS)
    Z, quant = Z.cpu().numpy(), quant.cpu().numpy()
    xs = _split_draws(vals)
    assert Z.shape == (xs.shape[0], M, 4 * k)
    for j in range(k):
        x, xall = xs[..., j], vals[..., j]
        med = np.median(x)
        assert bits(quant[0, j]) == bits(med) or (math.isnan(med) and math.isnan(quant[0, j])), j
        for t, p in ((1, 0.05), (2, 0.95)):
            q = np.quantile(xall, p)
            assert bits(quant[t, j]) == bits(q) or (math.isnan(q) and math.isnan(quant[t, j])), (j, p)
        assert np.array_equal(Z[..., 2 * k + j], (x <= quant[1, j]).astype(float)), j
        assert np.array_equal(Z[..., 3 * k + j], (x <= quant[2, j]).astype(float)), j
        z = Z[..., j]
        order = np.argsort(x.ravel(), kind="stable")                 # NaN last, as the keys order them
        zs, vs = z.ravel()[order], x.ravel()[order]
        assert (np.diff(zs) >= 0).all(), j
        same = (vs[1:] == vs[:-1]) | (np.isnan(vs[1:]) & np.isnan(vs[:-1]))
        assert (zs[1:][same] == zs[:-1][same]).all(), j
        if not np.isnan(x).any():
            ref = _z_ref(x)
            assert (np.abs(z - ref) <= 1e-13 * np.maximum(1.0, np.abs(ref))).all(), j
            if not math.isnan(med):
                f = np.abs(x - med)
                ref = _z_ref(f)
                assert (np.abs(Z[..., k + j] - ref) <= 1e-13 * np.maximum(1.0, np.abs(ref))).all(), j


@pytest.mark.parametrize("S", [4, 5, 41, 1000, 4001])
@pytest.mark.parametrize("M", [1, 2, 7, 256])
def test_diagnostics_equal_restatement(device, S, M):
    recs = _columns(np.random.default_rng(S * 1000 + M), S, M)
    d = torch.from_numpy(recs).cuda()
    got = device.rank_diagnostics_device(d, SPECS)
    host = D.rank_rhat_ess_columns(_host_values(recs, SPECS))
    assert assert_rank_matches(got, host) == 0
    assert math.isnan(got["rhat_rank"][3].item()) and math.isnan(got["median"][3].item())        # constant
    assert math.isnan(got["ess_tail"][5].item()) and math.isnan(got["rhat_rank"][6].item())     # +-inf, NaN
    again = device.rank_diagnostics_device(d, SPECS)
    for k in got:
        assert np.array_equal(bits(got[k].cpu().numpy()), bits(again[k].cpu().numpy())), k


def test_scale_mismatch_on_the_device(device):
    rng = np.random.default_rng(2021)
    x = np.concatenate([rng.normal(0, 1, (4, 1000)), rng.normal(0, 3, (4, 1000))])
    recs = torch.from_numpy(np.ascontiguousarray(x.T[:, :, None])).cuda()
    plain = device.chain_diagnostics_device(recs, [0])
    got = device.rank_diagnostics_device(recs, [0])
    assert plain["rhat"][0].item() < 1.005
    assert got["rhat_rank"][0].item() > 1.1 and got["rhat_rank"][0].item() == got["rhat_tail"][0].item()
    assert got["ess_tail"][0].item() < plain["ess"][0].item() / 4
    assert_rank_matches(got, D.rank_rhat_ess_columns(x.T[:, :, None]))


@pytest.mark.parametrize("kind", ["trend", "dd"])
def test_tempered_siblings(device, kind):
    T, n = 4, 16
    ch = _synthetic(device, kind, 24, n, 9)
    ch.set_beta(np.tile(P.temperature_ladder(T, 0.3), n // T))
    recs, _ = ch.run_tempered(8001, 20, T, 200)
    k = "trendrate" if kind == "trend" else "dd"
    cols = D.diagnostic_columns(k, 24)
    got = D.diagnose_records_device(device, torch.from_numpy(recs).cuda(), k, 24, burnin=0.2, ladder=T, rank=True)
    cold = E.cold_records(recs, T, ch.REC_BETA)
    cold = cold[S.burnin_index(cold.shape[0], 0.2):]
    assert assert_rank_matches(got, D.rank_rhat_ess_columns(_host_values(cold, [c[1] for c in cols])), got.names) == 0
    bad = recs.copy()
    bad[7, 0:T, ch.REC_BETA] = 0.5
    with pytest.raises(ValueError, match="lr_rank_diagnostics: a ladder has no chain at beta = 1"):
        device.rank_diagnostics_device(torch.from_numpy(bad).cuda(), [5], T, ch.REC_BETA)


@pytest.mark.parametrize("T", [1, 4])
def test_forward_records_and_marginals(device, T):
    recs, start, end = _forward_run(device, 8 if T == 1 else 4, T)
    cold = E.cold_records(recs, T) if T > 1 else recs
    host, nb = _forward_host(cold, start, end, 0.2)
    got = D.diagnose_records_device(device, torch.from_numpy(recs).cuda(), "forward", nb, burnin=0.2, ladder=T, origin=start, rank=True)
    assert len(got.names) == host.shape[2]
    assert assert_rank_matches(got, D.rank_rhat_ess_columns(host), got.names) == 0


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
    got = D.diagnose_records_device(dev, recs, "dd", nb, burnin=0.0, rank=True)
    grown = free0 - torch.cuda.mem_get_info()[0]
    assert grown <= (3 << 29), grown
    cols = D.diagnostic_columns("dd", nb)
    assert len(got.names) == len(cols) > 1011
    host = D.rank_rhat_ess_columns(_host_values(recs.cpu().numpy(), [c[1] for c in cols]))
    assert assert_rank_matches(got, host, got.names) == 0


def test_one_column_of_two_million_draws(device):
    rng = np.random.default_rng(9)
    x = np.round(rng.standard_t(3, size=(500, 4096, 1)), 2)          # heavy tails and many ties
    x[:, :7] *= 1.5
    d = torch.from_numpy(x).cuda()
    got = device.rank_diagnostics_device(d, [0])
    assert assert_rank_matches(got, D.rank_rhat_ess_columns(x)) == 0
    Z, quant = device.rank_transform_device(d, [0])
    ref = _z_ref(x[..., 0])
    z = Z[..., 0].cpu().numpy()
    assert (np.abs(z - ref) <= 1e-13 * np.maximum(1.0, np.abs(ref))).all()
    again = device.rank_diagnostics_device(d, [0])
    for k in got:
        assert np.array_equal(bits(got[k].cpu().numpy()), bits(again[k].cpu().numpy())), k


def test_bad_specs_are_refused(device):
    d = torch.zeros((10, 2, 4), dtype=torch.float64, device="cuda")
    for fn in (device.rank_diagnostics_device, device.rank_transform_device):
        name = "lr_rank_diagnostics" if fn == device.rank_diagnostics_device else "lr_rank_transform"
        for cols in ([4], [(0, 4, 1)], [(0, 1, 2)], [-1]):
            with pytest.raises(E.NativeError, match=name):
                fn(d, cols)
        with pytest.raises(E.NativeError, match=name):
            fn(d, [0], ladder=2, beta_col=4)
        with pytest.raises(RuntimeError, match="not enough data"):
            fn(d[:3], [0])


def _check_rank_tsv(path, logs):
    _, names, x = D.log_draws(logs, 0.2)
    host = D.rank_rhat_ess_columns(x)
    rows = [l.rstrip("\n").split("\t") for l in open(path)]
    assert rows[0] == ["column", "median", "q05", "q95", "rhat_rank", "rhat_bulk", "rhat_tail", "ess_bulk", "ess_tail", "flag"]
    tab = {r[0]: r[1:] for r in rows[1:]}
    assert list(tab) == names
    order = ("median", "q05", "q95", "rhat_rank", "rhat_bulk", "rhat_tail", "ess_bulk", "ess_tail")
    got = {k: np.array([float(tab[nm][i]) for nm in names]) for i, k in enumerate(order)}
    assert assert_rank_matches(got, host, names) == 0
    assert all(tab[nm][8] in D.FLAGS for nm in names)


def test_diagnose_command_line_rank(device, tmp_path):
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
    for logdir in (str(fwd / "literate_mcmc_logs"), str(tmp_path)):
        logs = D.find_logs(logdir)
        out = DG.main([logdir, "-rank", "1"])
        plain = {k: open(os.path.join(logdir, "diagnostics_%s.tsv" % k), "rb").read() for k in logs}
        want = []
        for kind in logs:
            p = os.path.join(logdir, "diagnostics_%s.tsv" % kind)
            want += [p, os.path.join(logdir, "diagnostics_%s_rank.tsv" % kind)]
            _check_rank_tsv(want[-1], logs[kind])
        assert out == want
        assert DG.main([logdir]) == want[::2]
        for k in logs:
            assert open(os.path.join(logdir, "diagnostics_%s.tsv" % k), "rb").read() == plain[k]


@pytest.mark.parametrize("disagree", [True, False])
def test_tables_that_disagree_rank(device, tmp_path, disagree):
    ts0, te0 = synth.syn_int(5000, replicate=0)
    y0 = te0 - 0.5
    if disagree:
        ts1, y1 = ts0, ts0 + np.floor((y0 - ts0) / 2)          # every lifetime halved: about twice the death rate
    else:
        perm = np.random.default_rng(1).permutation(len(ts0))   # the same lineages in another order (test_gpu_diagnostics)
        ts1, y1 = ts0[perm], y0[perm]
    _write_table(str(tmp_path / "a.tsv"), ts0, y0)
    _write_table(str(tmp_path / "b.tsv"), ts1, y1)
    F.main(["-d", str(tmp_path), "-n", "40000", "-s", "100", "-p", "100000", "-seed", "4", "-chains", "4", "-quiet", "1",
            "-const_rates", "1"])
    logdir = str(tmp_path / "literate_mcmc_logs")
    DG.main([logdir, "-rank", "1"])
    rows = [l.rstrip("\n").split("\t") for l in open(os.path.join(logdir, "diagnostics_forward_rank.tsv"))]
    rhat = float({r[0]: r for r in rows}["mu_avg"][4])
    assert (rhat > 1.1) if disagree else (rhat < 1.05), rhat
