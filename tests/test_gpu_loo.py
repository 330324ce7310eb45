"""GPU: K12 (lr_loo) against its host definition literate_b200.loo.loo_host on records of K3 (models 0-3, a general dataset, a
ladder of 4), K6 (plus a ladder) and K7; the pointwise log-likelihood against the samplers' own; a known answer from exact Gamma
posteriors; a brute-force LOO by refitting; the comparison's power on a rate jump; and the command line on logs of forward.py and
ddrate.py against the device path on the same seeds (byte-identical tables)."""
import math
import os
import shutil

import numpy as np
import pytest
import torch
from scipy import special

from literate_b200 import engine as E
from literate_b200 import loo as LO
from literate_b200 import predictive as PP
from literate_b200 import ddrate as DD
from literate_b200 import trend as TR

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


def _k3_case(dev, model, n_rep=1, general=False, ladder=1, n=8, seed=3):
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
    return recs, terms, dict(layout=0, n_bins=nb, start_time=start), "forward", np.arange(n) % n_rep


def _dense_case(dev, kind, ladder=1, n=8, seed=5):
    rng = np.random.default_rng(8)
    nb = 30
    br = rng.uniform(50, 900, (1, nb)); br[:, 3] = 0.0
    sp = rng.poisson(br * 0.2); ex = rng.poisson(br * 0.1)
    rep = np.zeros(n * ladder, np.int32)
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
    return recs, PP.stats_terms(sp, ex, br), dict(layout=1, rate_col=PP.KINDS[kind][1], n_bins=nb), kind, np.zeros(n, np.int64)


CASES = ["k3_m0", "k3_m1", "k3_m2", "k3_m3", "k3_general", "k3_ladder4", "k6", "k6_ladder4", "k7"]


def _case(dev, name):
    if name.startswith("k3_m"):
        return _k3_case(dev, int(name[-1]))
    if name == "k3_general":
        return _k3_case(dev, 1, general=True)
    if name == "k3_ladder4":
        return _k3_case(dev, 0, ladder=4)
    return _dense_case(dev, "trendrate" if name.startswith("k6") else "dd", ladder=4 if "ladder" in name else 1)


def _device(dev, recs, kw, terms, ladder, beta_col):
    t = torch.from_numpy(np.ascontiguousarray(recs)).cuda()
    o = dev.loo_device(t, kw["layout"], terms, rate_col=kw.get("rate_col", 0), start_time=kw.get("start_time", 0.0), ladder=ladder,
                       beta_col=beta_col)
    return {k: v.cpu().numpy() for k, v in o.items()}


@pytest.mark.parametrize("name", CASES)
def test_kernel_matches_host_definition(device, name):
    """Repeated calls bit-identical; records used, status and the tail length T equal (T given the device's r_eff, which the
    ceil of M must not turn into another tail); r_eff to 1e-9 (K9 and diagnostics.rhat_ess sum the same autocovariances in
    different orders); lppd, elpd_loo, p_loo, WAIC and k_hat to 1e-9 relative / absolute.  The inputs agree to a few ulp (one
    fp64 log and lgamma each; compensated against pairwise sums), and none of these quantities amplifies that by 10^6: the
    logsumexps and means have condition ~1 and the GPD fit's profile is smooth in b, so 1e-9 leaves room without hiding a
    wrong step, which moves them by 1e-3 or more."""
    recs, terms, kw, kind, rep = _case(device, name)
    ladder = 4 if "ladder" in name else 1
    beta_col = PP.KINDS[kind][2] if ladder > 1 else -1
    post = recs[40:]
    g = [_device(device, post, kw, terms[0], ladder, beta_col) for _ in range(2)]
    for k in g[0]:
        assert np.array_equal(g[0][k], g[1][k], equal_nan=True), k
    out = g[0]["out"]
    host = LO.loo_host(post, kw["layout"], kw["n_bins"], terms[0], rate_col=kw.get("rate_col", 0), start_time=kw.get("start_time", 0.0),
                       ladder=ladder, beta_col=beta_col)
    fixed = LO.loo_host(post, kw["layout"], kw["n_bins"], terms[0], rate_col=kw.get("rate_col", 0), start_time=kw.get("start_time", 0.0),
                        ladder=ladder, beta_col=beta_col, r_eff=out[7])
    print("%s: %d records used, status %s, k_hat max %.3g, r_eff %.3g .. %.3g" % (name, g[0]["n"][0], g[0]["status"],
                                                                               np.nanmax(out[6]), np.nanmin(out[7]), np.nanmax(out[7])))
    assert int(g[0]["n"][0]) == host["n"] > 0
    assert np.array_equal(g[0]["status"], host["status"])
    assert np.array_equal(np.isnan(out), np.isnan(host["out"]))
    np.testing.assert_array_equal(out[0], host["out"][0])
    np.testing.assert_array_equal(out[8], fixed["out"][8])
    np.testing.assert_allclose(out[7], host["out"][7], rtol=1e-9)
    for f in range(1, 7):
        np.testing.assert_allclose(out[f], fixed["out"][f], rtol=1e-9, atol=1e-9, err_msg=LO.FIELDS[f])


def test_imputation_replicates_are_refused(device):
    recs, terms, kw, kind, rep = _k3_case(device, 0, n_rep=3, n=9)
    with pytest.raises(ValueError, match="one table"):
        LO.loo_records_device(device, torch.from_numpy(recs).cuda(), kind, terms, start_time=kw["start_time"], rep_of_chain=rep)


@pytest.mark.parametrize("name", ["k3_m0", "k3_m1", "k3_m2", "k3_m3", "k6", "k7"])
def test_pointwise_sums_to_the_samplers_likelihood(device, name):
    """sum over the columns of l minus the logged likelihood (K3 REC_LIK; K6 and K7 field 1, for K7 likB + likD + likG without a
    genre table) is one constant over the records, to 1e-9 relative to the likelihood."""
    recs, terms, kw, kind, _ = _case(device, name)
    ll, act, used, _ = LO.pointwise_host(recs, kw["layout"], kw["n_bins"], terms[0], rate_col=kw.get("rate_col", 0),
                                         start_time=kw.get("start_time", 0.0))
    assert used.all()
    lik = recs[..., E.REC_LIK if kind == "forward" else 1]
    d = np.where(act, ll, 0.0).sum(axis=(2, 3)) - lik
    assert np.all(np.abs(d - d.flat[0]) <= 1e-9 * np.maximum(1.0, np.abs(lik))), (d.min(), d.max())


def test_known_answer_gamma_posterior(device):
    """One constant rate per side with a Gamma(a, b) prior: iid draws of its exact posterior Gamma(a + sum A, b + sum B) as
    dense records.  Every column's elpd_loo is the log of the negative-binomial predictive of A_j under Gamma(a + sum A - A_j,
    b + sum B - B_j), within 4 Monte Carlo sd (delta method on the harmonic mean of the draws' likelihoods, computed here); k_hat
    stays below the threshold."""
    nb, S_, M = 24, 4096, 256
    rng = np.random.default_rng(9)
    B = rng.uniform(20, 200, (2, nb))
    A = rng.poisson(B * np.array([[0.2], [0.1]])).astype(float)
    a, b = 1.0, 1.0
    recs = np.zeros((S_, M, 16 + 2 * nb))
    recs[..., 0] = np.arange(S_)[:, None]
    draws = []
    for side in range(2):
        r = rng.gamma(a + A[side].sum(), 1.0 / (b + B[side].sum()), (S_, M))
        recs[..., 16 + side * nb:16 + (side + 1) * nb] = r[..., None]
        draws.append(r.ravel())
    terms = np.stack([A[0], B[0], A[1], B[1]])
    res = LO.loo_records_device(device, torch.from_numpy(recs).cuda(), "trendrate", terms, burnin=0)
    assert res.n == S_ * M
    th = res.threshold()
    for side in range(2):
        for j in range(nb):
            al, be = a + A[side].sum() - A[side, j], b + B[side].sum() - B[side, j]
            y, x = A[side, j], B[side, j]
            exact = (special.gammaln(al + y) - special.gammaln(al) - special.gammaln(y + 1) + al * math.log(be / (be + x))
                     + y * math.log(x / (be + x)))
            r = draws[side]
            inv = np.exp(-(y * np.log(r * x) - r * x - special.gammaln(y + 1)) - (-exact))     # 1 / p relative to the answer
            sd = inv.std() / math.sqrt(len(inv)) / inv.mean()
            got = res.out[2, side, j]
            assert abs(got - exact) <= 4 * sd, (side, j, got, exact, sd)
            assert res.out[6, side, j] < th


def test_brute_force_loo_by_refitting(device):
    """A general dataset; for three (side, bin) columns, chains on the table with that column's A and B zeroed give the exact LOO
    predictive (the mean over their cold records of Poisson(A | r B)).  The full run's PSIS elpd_loo agrees within 3.5 standard
    errors: the between-chain errors of the refit mean and of the full run's importance-sampling estimate, combined."""
    rng = np.random.default_rng(12)
    nb, start, end, n = 20, 0.0, 20.0, 16
    br = rng.uniform(100, 400, nb)
    sp = rng.poisson(br * np.where(np.arange(nb) < 10, 0.1, 0.2)).astype(float); ex = rng.poisson(br * 0.1).astype(float)

    def run(Ab, Bb, Ad, Bd, seed):
        ds = E.Dataset.from_tables(device, Ab, Bb, Ad, Bd, sp / br, ex / br, start, end, model_tag=1)
        ch = E.Chains(ds, n, seed, E.default_config(1))
        recs = ch.run(100000, 100)[200:]
        terms = ds.bin_terms().cpu().numpy()[0]
        ch.close(); ds.close()
        return recs, terms

    full, terms = run(sp, br, ex, br, 1)
    res = LO.loo_records_device(device, torch.from_numpy(np.ascontiguousarray(full)).cuda(), "forward", terms, start_time=start, burnin=0)
    ll_full = LO.pointwise_host(full, 0, nb, terms, start_time=start)[0]
    for side, j in ((0, 3), (0, 15), (1, 9)):
        tabs = [sp.copy(), br.copy(), ex.copy(), br.copy()]
        tabs[2 * side][j] = 0.0
        tabs[2 * side + 1][j] = 0.0
        refit, _ = run(*tabs, 7 + j)
        ll = LO.pointwise_host(refit, 0, nb, terms, start_time=start)[0][:, :, side, j]         # l of the held-out count
        per_chain = np.log(np.exp(ll).mean(axis=0))
        exact = math.log(np.exp(ll).mean())
        lf = ll_full[:, :, side, j]
        is_chain = -np.log(np.exp(-lf).mean(axis=0))
        se = math.sqrt(per_chain.var(ddof=1) / n + is_chain.var(ddof=1) / n)
        got = res.out[2, side, j]
        print("column (%d, %d): PSIS %.6f, refit %.6f, se %.3g, k_hat %.3g" % (side, j, got, exact, se, res.out[6, side, j]))
        assert abs(got - exact) <= 3.5 * se


def test_teeth_default_beats_constant_rates_on_a_jump(device):
    """K11's 4x birth-rate jump: default RJMCMC chains beat -const_rates 1 chains by more than 4 se_diff, and the birth bins carry
    90 % of the difference.  The unit is the whole birth side, not the bins next to the jump: the constant-rate chains fit one
    birth rate to both halves, between 0.05 and 0.2, so every birth bin is misfit, while both models fit the death side alike.
    On a table without a jump the two models must agree: their elpd_loo differ by less than 1 (345 with the jump), whichever
    ranks first, so a LOO that over-penalises the shifts (an inflated p_loo) fails.  The criterion is not "within 2 se_diff":
    for nested models that predict alike, the pointwise differences are small and share a sign, so se_diff is small and
    unreliable (Sivula et al. 2022); these seeded chains give 0.17 in favour of the constant rates at se_diff 0.048."""
    rng = np.random.default_rng(21)
    nb = 40
    br = np.full(nb, 400.0)
    for jump in (True, False):
        sp = rng.poisson(br * np.where((np.arange(nb) < nb // 2) | (not jump), 0.05, 0.2)); ex = rng.poisson(br * 0.1)
        res = {}
        for const in (0, 1):
            ds = E.Dataset(device, E.BinStats(0, sp[None], ex[None], br[None]), 0, 0.0, float(nb))
            ch = E.Chains(ds, 8, 17, E.default_config(0, const_rates=const))
            recs = ch.run(200000, 200)
            res[const] = LO.loo_records_device(device, torch.from_numpy(recs).cuda(), "forward", ds.bin_terms(), start_time=0.0)
            ch.close(); ds.close()
        rows = LO.compare([res[0], res[1]], ["default", "const"])
        print("jump %s: %s" % (jump, rows))
        if jump:
            assert rows[0][1] == "default" and rows[1][5] > 4 * rows[1][6]
            d = res[0].out[2, 0] - res[1].out[2, 0]
            assert d.sum() > 0.9 * (res[0].pointwise() - res[1].pointwise()).sum()
        else:
            assert rows[1][5] < 1.0


# ------------------------------------------------------------------------------------------ logs equal records
def _read(d, names):
    return [open(os.path.join(d, f), "rb").read() for f in names]


def test_command_line_equals_records(device, tmp_path):
    """forward.py -chains 4 with -model_BDI 0 and 1 and ddrate.py -chains 4, each in its own directory: the command line's
    loo_<kind>.tsv, loo_<kind>_global.tsv and loo_compare.tsv are byte-identical to those from the engine's device records of the
    same seeds."""
    import warnings
    from literate_b200 import forward as F
    from literate_b200 import library as L
    src = os.path.join(HERE, "golden", "inputs", "example_dataTAD.txt")
    dirs, dev_res = [], []
    for model in (0, 1):
        d = tmp_path / ("m%d" % model)
        d.mkdir()
        shutil.copy(src, d / "example_dataTAD.txt")
        table = str(d / "example_dataTAD.txt")
        with warnings.catch_warnings():
            warnings.simplefilter("ignore", FutureWarning)
            F.run(F.build_parser().parse_args(["-d", table, "-n", "20000", "-s", "50", "-p", "50", "-seed", "6", "-chains", "4", "-quiet",
                                               "1", "-model_BDI", str(model)]), device=device)
            ts, te, start, end, _ = F.parse_lineages(table, death_jitter=0.5)
        dirs.append(str(d / "literate_mcmc_logs"))
        stats = device.bin_stats(ts, te, first_bin=int(start), n_bins=int(end) - int(start), death_jitter=0.5, end_time=float(end))
        ds = E.Dataset(device, stats, model, float(start), float(end))
        ch = E.Chains(ds, 4, 6, E.default_config(model), chain_id0=0, rep_of_chain=np.zeros(4, np.int32))
        recs = ch.run(20000, 50)
        dev_res.append(LO.loo_records_device(device, torch.from_numpy(recs).cuda(), "forward", ds.bin_terms(), start_time=float(start),
                                             burnin=0.2))
        ch.close(); ds.close()
    dd = tmp_path / "dd"
    dd.mkdir()
    shutil.copy(os.path.join(HERE, "golden", "trendrate", "example3.tsv"), dd / "example3.tsv")
    argv = ["-d", str(dd / "example3.tsv"), "-m_birth", "2", "-m_death", "2", "-n", "20000", "-s", "50", "-seed", "3", "-chains", "4",
            "-quiet", "1"]
    assert len(DD.run(DD.build_parser().parse_args(argv), device=device)) == 4
    dirs.append(str(dd))
    args = DD.build_parser().parse_args(argv)
    tables, ts, te, present, origin = L.read_tables(args, exclude="-")
    first_bin, n_bins = L.bin_window(origin, present, 0)
    st = device.bin_stats(ts, te, first_bin=first_bin, n_bins=n_bins, death_jitter=args.death_jitter)
    ch = DD.DDChains(device, st.sp, st.ex, st.br, origin, present, 2, 2, None, None, 4, 3, chain_id0=0, rep_of_chain=np.zeros(4, np.int32))
    recs = ch.run(20000, 50)
    ch.close()
    dev_res.append(LO.loo_records_device(device, torch.from_numpy(recs).cuda(), "dd", PP.stats_terms(st.sp, st.ex, st.br), first_edge=0.0,
                                         burnin=0.2))

    # the two RJMCMC runs
    out = tmp_path / "out"
    out.mkdir()
    got = LO.main(dirs[:2] + ["-out", str(out)], device=device)
    assert len(got) == 2
    ref = tmp_path / "ref"
    ref.mkdir()
    LO.write_compare(str(ref / "loo_compare.tsv"), LO.compare(dev_res[:2], [d + ":forward" for d in dirs[:2]]))
    assert _read(str(out), ["loo_compare.tsv"]) == _read(str(ref), ["loo_compare.tsv"])
    for d, r in zip(dirs, dev_res):
        rd = tmp_path / ("ref_" + os.path.basename(os.path.dirname(d)) + os.path.basename(d))
        rd.mkdir()
        r.write_tsv(str(rd))
        if r.kind == "dd":
            LO.loo_dir(d, device=device)
        names_k = ["loo_%s.tsv" % r.kind, "loo_%s_global.tsv" % r.kind]
        assert _read(d, names_k) == _read(str(rd), names_k)
    # the DDRate run observes the same counts (its table holds the same lineages), so the three compare column by column
    got = LO.main(dirs + ["-out", str(out)], device=device)
    assert len(got) == 3
    LO.write_compare(str(ref / "loo_compare.tsv"), LO.compare(dev_res, [d + ":" + r.kind for d, r in zip(dirs, dev_res)]))
    assert _read(str(out), ["loo_compare.tsv"]) == _read(str(ref), ["loo_compare.tsv"])
