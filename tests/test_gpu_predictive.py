"""GPU: K11 (lr_predictive_check) and its sampler lr_poisson against their host definitions in literate_b200.predictive --
the sampler draw for draw (except decisions within TIE_TOL of a tie) and against scipy's Poisson law, the kernel on records of
K3 (models 0-3 and a general dataset), K6 and K7 including a tempered run and imputation replicates, the stored bin terms against
the likelihood, a known answer, the check's power on data a constant-rate model cannot fit, the refusals of the entry point, and
the command line on logs of forward.py and ddrate.py against the device path on the same seed (byte-identical tables)."""
import ctypes
import math
import os
import subprocess

import numpy as np
import pytest
import torch
from scipy import stats

from literate_b200 import build
from literate_b200 import engine as E
from literate_b200 import predictive as PP
from literate_b200 import ddrate as DD
from literate_b200 import trend as TR

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    out = os.path.join(str(tmp_path_factory.mktemp("poisson")), "poisson_harness.so")
    cmd = [build._nvcc()] + build.NVCC_FLAGS + ["-shared", os.path.join(HERE, "poisson_harness.cu"), "-o", out]
    p = subprocess.run(cmd, capture_output=True, text=True)
    assert p.returncode == 0, p.stdout + p.stderr
    lib = ctypes.CDLL(out)
    lib.t_poisson.argtypes = [ctypes.c_void_p] * 2 + [ctypes.c_ulonglong] + [ctypes.c_void_p] * 2 + [ctypes.c_longlong]
    lib.t_poisson.restype = ctypes.c_int
    return lib


def _draw(lib, mu, ctr, seed):
    m = torch.from_numpy(np.ascontiguousarray(mu, np.float64)).cuda()
    c = torch.from_numpy(np.ascontiguousarray(ctr, np.uint32).view(np.int32)).cuda()
    y = torch.empty(len(mu), dtype=torch.int64, device="cuda")
    e = torch.empty(len(mu), dtype=torch.int32, device="cuda")
    assert lib.t_poisson(m.data_ptr(), c.data_ptr(), seed, y.data_ptr(), e.data_ptr(), len(mu)) == 0
    torch.cuda.synchronize()
    return y.cpu().numpy(), e.cpu().numpy()


def test_poisson_matches_its_definition(harness):
    """2^20 (counter, mean) pairs, means log-uniform over 1e-8 .. 1e9 plus both sides of the branch at 10: every draw equals the
    host restatement except draws the restatement marks as within TIE_TOL of a tie; out-of-range means give -1."""
    rng = np.random.default_rng(11)
    n = 1 << 20
    mu = np.exp(rng.uniform(math.log(1e-8), math.log(1e9), n))
    mu[:8] = [0.0, 1e-8, np.nextafter(10.0, 0.0), 10.0, 9.5, 10.5, 1e9, 2.0 ** 52]
    ctr = rng.integers(0, 2 ** 32, (n, 4), dtype=np.uint64).astype(np.uint32)
    ctr[:, 2] &= np.uint32((1 << 25) - 1)
    seed = 0x1234567890abcdef
    y, exh = _draw(harness, mu, ctr, seed)
    hy, near, hexh = PP.poisson_host(mu, ctr[:, 0], ctr[:, 1], ctr[:, 2], ctr[:, 3], seed)
    bad = y != hy
    print("lr_poisson: %d of %d draws within TIE_TOL of a tie, %d of them differ" % (near.sum(), n, (bad & near).sum()))
    assert not (bad & ~near).any(), list(zip(mu[bad & ~near][:5], y[bad & ~near][:5], hy[bad & ~near][:5]))
    assert (exh.astype(bool) == hexh).all() and not hexh.any()
    assert y[0] == 0
    bad_mu = np.array([-1.0, np.nan, np.inf, 2.0 ** 53])
    yb, _ = _draw(harness, bad_mu, np.zeros((4, 4), np.uint32), 1)
    assert (yb == -1).all()


@pytest.mark.parametrize("mu", [1e-3, 0.7, 3.0, 9.99, 10.0, 37.5, 1e3, 1e6, 1e9])
def test_poisson_law(harness, mu):
    """2^22 draws at one mean: chi-square against scipy.stats.poisson over bins of expected count >= 20."""
    n = 1 << 22
    ctr = np.zeros((n, 4), np.uint32)
    ctr[:, 0] = np.arange(n, dtype=np.uint32)
    ctr[:, 3] = 77
    y, exh = _draw(harness, np.full(n, mu), ctr, 5)
    assert not exh.any() and (y >= 0).all()
    lo, hi = int(stats.poisson.ppf(1e-7, mu)), int(stats.poisson.isf(1e-7, mu))
    edges = [lo]
    k = lo
    while k <= hi:                                   # group values until each bin expects >= 20 draws
        j = k
        while j <= hi and n * (stats.poisson.cdf(j, mu) - stats.poisson.cdf(edges[-1] - 1, mu)) < 20:
            j += max(1, int(math.sqrt(mu) / 20))
        edges.append(j + 1)
        k = j + 1
    cdf = stats.poisson.cdf(np.array(edges) - 1, mu)
    exp = n * np.diff(cdf)
    exp[0] += n * cdf[0]
    exp[-1] += n * (1 - cdf[-1])
    obs = np.histogram(np.clip(y, edges[0], edges[-1] - 1), bins=edges)[0]
    keep = exp > 0
    chi2 = float(((obs[keep] - exp[keep]) ** 2 / exp[keep]).sum())
    p = stats.chi2.sf(chi2, keep.sum() - 1) if keep.sum() > 1 else 1.0
    assert p > 1e-5, (mu, chi2, keep.sum(), p)


# ------------------------------------------------------------------------------------------ the kernel
def _k3_case(dev, model, n_rep=1, general=False, ladder=1, n=8, seed=3):
    """K3 records of a synthetic table with a real-valued start time (the likelihood's bin mapping differs from np.histogram's)."""
    rng = np.random.default_rng(model + 10 * n_rep)
    start, end = 3.4, 43.7
    nb = 40
    br = rng.uniform(20, 300, (n_rep, nb)); br[:, 5] = 0.0
    sp = rng.poisson(br * np.where(np.arange(nb) < 20, 0.1, 0.25)); ex = rng.poisson(br * 0.1)
    exd, brd = rng.poisson(br * 0.05), br * 0.6
    if general:
        ds = E.Dataset.from_tables(dev, sp.astype(float) + 0.5, (br > 0).astype(float), ex.astype(float), br, sp / np.maximum(br, 1),
                                   ex / np.maximum(br, 1), start, end, model_tag=1)
    else:
        ds = E.Dataset(dev, E.BinStats(3, sp, ex, br, exd, brd), model, start, end)
    rep = np.repeat(np.arange(n) % n_rep, ladder).astype(np.int32)
    ch = E.Chains(ds, n * ladder, seed, E.default_config(1 if general else model), rep_of_chain=rep)
    if ladder > 1:
        ch.set_beta(np.tile([1.0, 0.7, 0.5, 0.3][:ladder], n))
        recs = ch.run_tempered(20000, 50, ladder, 100)[0]
    else:
        recs = ch.run(20000, 50)
    terms = ds.bin_terms().cpu().numpy()
    ch.close(); ds.close()
    return recs, terms, dict(layout=0, n_bins=nb, start_time=start, rep_of_chain=np.arange(n) % n_rep), "forward"


def _dense_case(dev, kind, n_rep=1, ladder=1, n=8, seed=5):
    rng = np.random.default_rng(7 + n_rep)
    nb = 30
    br = rng.uniform(50, 900, (n_rep, nb)); br[:, 3] = 0.0
    sp = rng.poisson(br * 0.2); ex = rng.poisson(br * 0.1)
    rep = np.repeat(np.arange(n) % n_rep, ladder).astype(np.int32)
    if kind == "trendrate":
        ch = TR.TrendChains(dev, sp, ex, br, np.linspace(.05, 1, nb), n * ladder, seed, rep_of_chain=rep)
    else:
        ch = DD.DDChains(dev, sp, ex, br, 0.0, nb + 1.5, 2, 2, None, None, n * ladder, seed, rep_of_chain=rep)
    if ladder > 1:
        ch.set_beta(np.tile([1.0, 0.7, 0.5, 0.3][:ladder], n))
        recs = ch.run_tempered(20000, 50, ladder, 100)[0]
    else:
        recs = ch.run(20000, 50)
    ch.close()
    layout, rate_col, _ = PP.KINDS[kind]
    return recs, PP.stats_terms(sp, ex, br), dict(layout=1, rate_col=rate_col, n_bins=nb, rep_of_chain=np.arange(n) % n_rep), kind


CASES = ["k3_m0", "k3_m1", "k3_m2", "k3_m3", "k3_general", "k3_rep3", "k3_ladder4", "k6", "k6_ladder4", "k7", "k7_rep2"]


def _case(dev, name):
    if name.startswith("k3_m"):
        return _k3_case(dev, int(name[-1]))
    if name == "k3_general":
        return _k3_case(dev, 1, general=True)
    if name == "k3_rep3":
        return _k3_case(dev, 0, n_rep=3, n=9)
    if name == "k3_ladder4":
        return _k3_case(dev, 0, ladder=4)
    kind = "trendrate" if name.startswith("k6") else "dd"
    return _dense_case(dev, kind, n_rep=2 if name.endswith("rep2") else 1, ladder=4 if "ladder" in name else 1)


@pytest.mark.parametrize("name", CASES)
def test_kernel_matches_host_definition(device, name):
    """Repeated calls bit-identical; every int64 output equal, sums of mu / mu^2 / A, per-record deviances and their sums to
    1e-12.  Records the host marks as within TIE_TOL of a tie are made unusable on both sides first (none was in past runs)."""
    recs, terms, kw, kind = _case(device, name)
    ladder = 4 if "ladder" in name else 1
    beta_col = PP.KINDS[kind][2] if ladder > 1 else -1
    b0 = 40
    post = recs[b0:]
    host = PP.predictive_check_host(post, kw["layout"], kw["n_bins"], terms, rate_col=kw.get("rate_col", 0),
                                    start_time=kw.get("start_time", 0.0), rep_of_chain=kw["rep_of_chain"], ladder=ladder,
                                    beta_col=beta_col, chain_id0=0, seed=99)
    t = torch.from_numpy(np.ascontiguousarray(recs)).cuda()
    outs = [device.predictive_check_device(t[b0:], kw["layout"], terms, rate_col=kw.get("rate_col", 0), start_time=kw.get("start_time", 0.0),
                                           rep_of_chain=kw["rep_of_chain"], ladder=ladder, beta_col=beta_col, seed=99, per_record=True)
            for _ in range(2)]
    g = {k: v.cpu().numpy() for k, v in outs[0].items() if k != "terms"}
    for k in g:
        assert np.array_equal(g[k], outs[1][k].cpu().numpy(), equal_nan=True), k
    n_near = int(host["near"].sum())
    print("%s: %d records used, %d near-tie records, status %s" % (name, g["glob_count"][0], n_near, g["status"]))
    if n_near:
        # records with a decision within TIE_TOL of a tie: made unusable on both sides (iteration -1), the rest held exactly
        post = post.copy()
        for s_, c_ in zip(*np.nonzero(host["near"])):
            post[s_, c_ * ladder:(c_ + 1) * ladder, 0] = -1.0
        host = PP.predictive_check_host(post, kw["layout"], kw["n_bins"], terms, rate_col=kw.get("rate_col", 0),
                                        start_time=kw.get("start_time", 0.0), rep_of_chain=kw["rep_of_chain"], ladder=ladder,
                                        beta_col=beta_col, chain_id0=0, seed=99)
        assert not host["near"].any()
        g = {k: v.cpu().numpy() for k, v in device.predictive_check_device(
            torch.from_numpy(np.ascontiguousarray(post)).cuda(), kw["layout"], terms, rate_col=kw.get("rate_col", 0),
            start_time=kw.get("start_time", 0.0), rep_of_chain=kw["rep_of_chain"], ladder=ladder, beta_col=beta_col, seed=99,
            per_record=True).items() if k != "terms"}
    assert g["glob_count"][0] > 0
    for k in ("status", "bin_count", "glob_count"):
        assert np.array_equal(g[k], host[k]), (k, g[k], host[k])
    np.testing.assert_allclose(g["bin_sum"], host["bin_sum"], rtol=1e-12, atol=0)
    np.testing.assert_allclose(g["dev"], host["dev"], rtol=1e-12, atol=1e-300)
    np.testing.assert_allclose(g["glob_sum"], host["glob_sum"], rtol=1e-12)


def test_entry_point_refusals(device):
    """n_bins beyond the draw grid (more than 65535 blocks of 256 bins), rate fields outside the row, replicates out of range."""
    import ctypes as C
    recs = torch.zeros((4, 2, 16 + 2 * 8), dtype=torch.float64, device="cuda")
    terms = torch.ones((1, 4, 8), dtype=torch.float64, device="cuda")
    outs = [torch.zeros(64, dtype=torch.float64, device="cuda") for _ in range(5)]
    status = torch.zeros(3, dtype=torch.int64, device="cuda")

    def call(n_bins, rate_col=16, rep=None):
        r = None if rep is None else np.ascontiguousarray(rep, np.int32)
        return device.lib.lr_predictive_check(device.h, C.c_void_p(recs.data_ptr()), 4, 2, 1, -1, recs.shape[2], 1, rate_col, 0.0, n_bins,
                                              C.c_void_p(terms.data_ptr()), 1, None if r is None else C.c_void_p(r.ctypes.data), 0, 0,
                                              *[C.c_void_p(t.data_ptr()) for t in outs[:4]], None, C.c_void_p(status.data_ptr()), None)
    assert call(8) == 0
    torch.cuda.synchronize()
    assert call(65535 * 256 + 1) == -1 and b"n_bins" in device.lib.lr_last_error()
    assert call(0) == -1
    assert call(8, rate_col=17) == -1 and b"outside the row" in device.lib.lr_last_error()
    assert call(8, rep=[0, 1]) == -1 and b"replicate" in device.lib.lr_last_error()


def test_bin_terms_give_the_likelihood(device):
    """For random K3 states on every model, C + sum_j A log r_j - B r_j over the stored bin terms equals Dataset.evaluate's
    likelihood to 1e-10."""
    rng = np.random.default_rng(4)
    nb, start, end = 40, 3.4, 43.7
    br = rng.uniform(20, 300, nb); br[5] = 0.0
    sp, ex = rng.poisson(br * 0.1), rng.poisson(br * 0.1)
    exd, brd = rng.poisson(br * 0.05), br * 0.6
    for model in range(4):
        ds = E.Dataset(device, E.BinStats(3, sp[None], ex[None], br[None], exd[None], brd[None]), model, start, end)
        T = ds.bin_terms().cpu().numpy()[0]
        m = br > 0
        C = 0.0 if model >= 2 else float(np.sum(np.where(m, (sp + ex if model == 0 else ex) * np.log(np.where(m, br, 1.0)), 0.0)))
        states = []
        for _ in range(50):
            kl, km = rng.integers(1, 6, 2)
            tl = np.sort(rng.uniform(start + 1, end - 1, kl - 1)); tm = np.sort(rng.uniform(start + 1, end - 1, km - 1))
            states.append((rng.uniform(.01, .5, kl), rng.uniform(.01, .5, km), np.r_[start, tl, end], np.r_[start, tm, end]))
        want = ds.evaluate(states)["lik"]
        rec = np.zeros((1, len(states), E.LR_REC_DOUBLES))
        for i, (L, M, tl, tm) in enumerate(states):
            rec[0, i, [E.REC_KL, E.REC_KM]] = len(L), len(M)
            rec[0, i, E.REC_L:E.REC_L + len(L)] = L; rec[0, i, E.REC_TL:E.REC_TL + len(L)] = tl[:-1]
            rec[0, i, E.REC_M:E.REC_M + len(M)] = M; rec[0, i, E.REC_TM:E.REC_TM + len(M)] = tm[:-1]
        rates, ok = PP.bin_rates(rec, 0, nb, start_time=start)
        assert ok.all()
        r = rates[0]
        with np.errstate(divide="ignore"):
            got = C + np.sum(T[0] * np.log(r[:, 0]) - T[1] * r[:, 0], axis=1) + np.sum(np.where(T[2] > 0, T[2] * np.log(r[:, 1]), 0.0) - T[3] * r[:, 1], axis=1)
        np.testing.assert_allclose(got, want, rtol=1e-10)
        ds.close()


def test_point_mass_known_answer(device):
    """10^6 records of one state (a point-mass posterior): every per-bin p_mid within 4 standard errors of the exact mid-p of
    scipy.stats.poisson."""
    nb, S_, M = 12, 10000, 100
    rates_b = np.linspace(0.05, 0.3, nb); rates_d = np.linspace(0.2, 0.02, nb)
    br = np.linspace(10, 400, nb)
    sp = np.round(rates_b * br * np.linspace(0.6, 1.6, nb)); ex = np.round(rates_d * br)
    recs = np.zeros((S_, M, 16 + 2 * nb))
    recs[..., 0] = np.arange(S_)[:, None]
    recs[..., 16:16 + nb] = rates_b; recs[..., 16 + nb:] = rates_d
    terms = PP.stats_terms(sp, ex, br)
    res = PP.predictive_records_device(device, torch.from_numpy(recs).cuda(), "trendrate", terms, burnin=0, seed=3)
    assert int(res.glob_count[0]) == S_ * M
    tab = res.table()
    for side, (A, r) in enumerate(((sp, rates_b), (ex, rates_d))):
        mu = r * br
        exact = stats.poisson.sf(A, mu) + 0.5 * stats.poisson.pmf(A, mu)
        got = np.array([row[6] for row in tab[side * nb:(side + 1) * nb]])
        se = np.sqrt(np.maximum(exact * (1 - exact), 1e-12) / (S_ * M))
        assert np.all(np.abs(got - exact) <= 4 * se + 1e-12), (side, got, exact)
        np.testing.assert_allclose([row[3] for row in tab[side * nb:(side + 1) * nb]], mu, rtol=1e-12)


def test_teeth_constant_rates_miss_a_jump(device):
    """Per-bin counts whose birth rate jumps 4x at mid-window: RJMCMC chains held to constant rates fail the global birth check
    (p < 1e-3) and flag the bins next to the jump; default chains pass it (0.01 < p < 0.99)."""
    rng = np.random.default_rng(21)
    nb = 40
    br = np.full(nb, 400.0)
    sp = rng.poisson(br * np.where(np.arange(nb) < nb // 2, 0.05, 0.2)); ex = rng.poisson(br * 0.1)
    ps = {}
    for const in (1, 0):
        ds = E.Dataset(device, E.BinStats(0, sp[None], ex[None], br[None]), 0, 0.0, float(nb))
        ch = E.Chains(ds, 8, 17, E.default_config(0, const_rates=const))
        recs = ch.run(200000, 200)
        res = PP.predictive_records_device(device, torch.from_numpy(recs).cuda(), "forward", ds.bin_terms(), start_time=0.0, seed=1)
        ch.close(); ds.close()
        ps[const] = res.global_table()[0][4]
        if const:
            flags = [row[7] for row in res.table()[:nb]]
            assert flags[nb // 2 - 1] == "obs_low" and flags[nb // 2] == "obs_high", flags
    print("global birth p: constant rates %.3g, default %.3g" % (ps[1], ps[0]))
    assert ps[1] < 1e-3
    assert 0.01 < ps[0] < 0.99


# ------------------------------------------------------------------------------------------ logs equal records
def _read(d, kind):
    return [open(os.path.join(d, "predictive_%s%s.tsv" % (kind, t)), "rb").read() for t in ("", "_global")]


def test_forward_logs_equal_records(device, tmp_path):
    """forward.py -chains 4 on a shipped table, then the same seed and configuration through engine: the command line's tables
    from the log directory are byte-identical to predictive_records_device's on the device records; a log whose name claims
    another model is refused by the device likelihood."""
    import shutil
    import warnings
    from literate_b200 import forward as F
    src = os.path.join(HERE, "golden", "inputs", "example_dataTAD.txt")
    shutil.copy(src, tmp_path / "example_dataTAD.txt")
    table = str(tmp_path / "example_dataTAD.txt")
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", FutureWarning)
        F.run(F.build_parser().parse_args(["-d", table, "-n", "20000", "-s", "50", "-p", "50", "-seed", "6", "-chains", "4", "-quiet", "1"]),
              device=device)
        ts, te, start, end, _ = F.parse_lineages(table, death_jitter=0.5)
    log_dir = str(tmp_path / "literate_mcmc_logs")
    out_cli, out_dev = tmp_path / "cli", tmp_path / "dev"
    out_cli.mkdir(); out_dev.mkdir()
    PP.check_dir(log_dir, burnin=0.2, seed=0, device=device, out_dir=str(out_cli), note=print)

    stats = device.bin_stats(ts, te, first_bin=int(start), n_bins=int(end) - int(start), death_jitter=0.5, end_time=float(end))
    ds = E.Dataset(device, stats, 0, float(start), float(end))
    ch = E.Chains(ds, 4, 6, E.default_config(0), chain_id0=0, rep_of_chain=np.zeros(4, np.int32))
    recs = ch.run(20000, 50)
    res = PP.predictive_records_device(device, torch.from_numpy(recs).cuda(), "forward", ds.bin_terms(), start_time=float(start),
                                       burnin=0.2, seed=0)
    ch.close(); ds.close()
    res.write_tsv(str(out_dev))
    assert int(res.glob_count[0]) == 4 * (400 - 80)
    assert _read(str(out_cli), "forward") == _read(str(out_dev), "forward")

    # the same logs under another model's name: the device likelihood of the first row disagrees
    bad = tmp_path / "bad"
    bad.mkdir()
    for f in os.listdir(log_dir):
        if "chain0" in f:
            shutil.copy(os.path.join(log_dir, f), bad / f.replace("_BD_", "_BDk_"))
    with pytest.raises(SystemExit, match="likelihood"):
        PP.check_dir(str(bad), device=device)


def test_ddrate_logs_equal_records(device, tmp_path):
    """ddrate.py -chains 4 on a shipped table, then the same seed through engine: byte-identical tables from logs and records."""
    import shutil
    from literate_b200 import library as L
    shutil.copy(os.path.join(HERE, "golden", "trendrate", "example3.tsv"), tmp_path / "example3.tsv")
    argv = ["-d", str(tmp_path / "example3.tsv"), "-m_birth", "2", "-m_death", "2", "-n", "20000", "-s", "50", "-seed", "3",
            "-chains", "4", "-quiet", "1"]
    paths = DD.run(DD.build_parser().parse_args(argv), device=device)
    assert len(paths) == 4
    out_cli, out_dev = tmp_path / "cli", tmp_path / "dev"
    out_cli.mkdir(); out_dev.mkdir()
    PP.check_dir(str(tmp_path), burnin=0.2, seed=0, device=device, out_dir=str(out_cli), note=print)

    args = DD.build_parser().parse_args(argv)
    tables, ts, te, present, origin = L.read_tables(args, exclude="-")
    first_bin, n_bins = L.bin_window(origin, present, 0)
    st = device.bin_stats(ts, te, first_bin=first_bin, n_bins=n_bins, death_jitter=args.death_jitter)
    ch = DD.DDChains(device, st.sp, st.ex, st.br, origin, present, 2, 2, None, None, 4, 3, chain_id0=0, rep_of_chain=np.zeros(4, np.int32))
    recs = ch.run(20000, 50)
    ch.close()
    res = PP.predictive_records_device(device, torch.from_numpy(recs).cuda(), "dd", PP.stats_terms(st.sp, st.ex, st.br), first_edge=0.0,
                                       burnin=0.2, seed=0)
    res.write_tsv(str(out_dev))
    assert int(res.glob_count[0]) == 4 * (400 - 80)
    assert _read(str(out_cli), "dd") == _read(str(out_dev), "dd")
