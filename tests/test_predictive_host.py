"""Host side of the posterior predictive check (literate_b200.predictive): the Philox counter layout, the host definition on
hand-computed cases, log packing, model detection and the refusals of the command line.  No GPU needed."""
import math
import os

import numpy as np
import pytest

from literate_b200 import engine as E
from literate_b200 import forward as F
from literate_b200 import predictive as PP
import _device_math as D


def test_philox_and_counter_layout():
    rng = np.random.default_rng(1)
    c = rng.integers(0, 2 ** 32, (5, 1000), dtype=np.uint64).astype(np.uint32)
    assert all(np.array_equal(a, b) for a, b in zip(PP.philox(*c[:4], c[4], c[4] ^ 7), D.philox_ref(*c[:4], c[4], c[4] ^ 7)))
    for ctr, key, want in D.PHILOX_KAT:
        assert tuple(int(v) for v in PP.philox(*ctr, *key)) == want
    c0, c1, c2, c3 = PP.counters(2 ** 33 + 5, 7, 1, 2 ** 32 + 3)
    assert (int(c0), int(c1), int(c2), int(c3)) == (5, 2, 7 | 1 << 24, 3)
    assert PP.u01(np.uint32(0), np.uint32(0)) == 2.0 ** -53
    assert PP.u01(np.uint32(0xffffffff), np.uint32(0xffffffff)) == 1 - 2.0 ** -53


def test_sampler_edges():
    y, near, exh = PP.poisson_host(np.array([0.0, -1.0, np.nan, 2.0 ** 53, 1e-300]), 1, 2, 3, 4, 5)
    assert list(y[:4]) == [0, -1, -1, -1] and y[4] == 0 and not exh.any()
    # the inversion branch is the sequential search itself: with u below exp(-mu) the count is 0
    mu = np.full(4096, 2.5)
    y, _, _ = PP.poisson_host(mu, np.arange(4096), 0, 0, 0, 9)
    x, yy, _, _ = PP.philox(np.arange(4096), 0, 0, 0, np.uint32(9), np.uint32(0))
    u = PP.u01(x, yy)
    assert np.array_equal(y == 0, u <= math.exp(-2.5))


def _dense(rates_b, rates_d, it, nb):
    r = np.zeros((len(it), 1, 16 + 2 * nb))
    r[:, 0, 0] = it
    r[:, 0, 16:16 + nb] = rates_b
    r[:, 0, 16 + nb:] = rates_d
    return r


def test_host_definition_hand_cases():
    """A point mass with B = 0 bins and y = 0 terms: bins with B = 0 take no draw; with A = 0 everywhere D_obs = 2 sum mu; the
    expected count is rate B exactly; a record with a negative rate is skipped."""
    nb = 3
    terms = np.array([[[0, 0, 0], [2.0, 0.0, 4.0], [0, 0, 0], [1.0, 1.0, 0.0]]])
    recs = _dense([0.5, 9.0, 0.25], [0.1, 0.2, 0.3], np.arange(6), nb)
    recs[5, 0, 16] = -1.0
    out = PP.predictive_check_host(recs, 1, nb, terms, rate_col=16)
    assert list(out["status"]) == [1, 0, 0]
    assert list(out["bin_count"][0, 0]) == [5, 0, 5] and list(out["bin_count"][1, 0]) == [5, 5, 0]
    np.testing.assert_allclose(out["bin_sum"][0, 0], [5.0, 0.0, 5.0])
    np.testing.assert_allclose(out["dev"][:5, 0, 0], 2 * (1.0 + 1.0))
    np.testing.assert_allclose(out["dev"][:5, 0, 2], 2 * (0.1 + 0.2))
    assert np.isnan(out["dev"][5]).all()
    assert out["glob_count"][0] == 5
    # A = 0 and every replicate 0 > A never: #(y_rep > A) counts the non-zero draws
    y_pos = out["bin_count"][0, 2]
    assert (y_pos <= out["bin_count"][0, 0]).all() and (out["bin_count"][0, 3] + y_pos == out["bin_count"][0, 0]).all()
    res = PP.PredictiveResult.from_outputs("trendrate", 10.0, out)
    rows = res.table()
    assert rows[1][7] == "none" and rows[0][1] == 10.0 and rows[0][3] == 1.0


def test_k3_bin_mapping_is_the_likelihoods():
    """Segment k starts at bin floor(t_k) - floor(start): with start 3.4 a shift at 5.2 starts bin 2 (np.histogram from 3.4
    would put it in bin 1)."""
    rec = np.zeros((1, 1, E.LR_REC_DOUBLES))
    rec[0, 0, [E.REC_KL, E.REC_KM]] = 2, 1
    rec[0, 0, E.REC_L:E.REC_L + 2] = [1.0, 2.0]
    rec[0, 0, E.REC_TL:E.REC_TL + 2] = [3.4, 5.2]
    rec[0, 0, E.REC_M] = 3.0
    rates, ok = PP.bin_rates(rec, 0, 6, start_time=3.4)
    assert ok.all()
    assert list(rates[0, 0, 0]) == [1.0, 1.0, 2.0, 2.0, 2.0, 2.0] and list(rates[0, 0, 1]) == [3.0] * 6
    rec[0, 0, E.REC_TL + 1] = np.nan
    assert not PP.bin_rates(rec, 0, 6, start_time=3.4)[1].any()


def _records(rng, n, start, end):
    recs = np.zeros((n, E.LR_REC_DOUBLES))
    for i in range(n):
        recs[i, E.REC_IT] = 100 * i
        for kf, rf, tf in ((E.REC_KL, E.REC_L, E.REC_TL), (E.REC_KM, E.REC_M, E.REC_TM)):
            K = int(rng.integers(1, 5))
            recs[i, kf] = K
            recs[i, rf:rf + K] = rng.uniform(0.01, 1, K)
            recs[i, tf] = start
            recs[i, tf + 1:tf + K] = np.sort(rng.uniform(start + 1, end - 1, K - 1))
        recs[i, E.REC_LIK] = rng.normal() * 100
        recs[i, E.REC_PRIOR] = rng.normal()
        recs[i, E.REC_BETA] = 1.0
        recs[i, E.REC_POI_INIT] = 1
    return recs


def _write_logs(tmp, name, recs, start, end, sp, ex, br):
    stem = os.path.join(tmp, name)
    w = F.ChainLogWriter(stem, 0, 0, start, end, end, 0.0)
    for r in recs:
        w.write(r)
    w.close()
    F.write_div_log(stem + "_div.log", sp, ex, br)
    return stem + "_mcmc.log"


def test_log_packing_equals_the_records(tmp_path):
    rng = np.random.default_rng(2)
    start, end = 3.4, 43.7
    recs = _records(rng, 50, start, end)
    path = _write_logs(str(tmp_path), "tab_BD_chain0", recs, start, end, np.ones(40, int), np.ones(40, int), np.ones(40))
    got, s, e = PP.pack_forward_log(path, burnin=0.2)
    assert (s, e) == (start, end) and got.shape == (40, E.LR_REC_DOUBLES)
    want = recs[10:]
    fields = [E.REC_IT, E.REC_LIK, E.REC_KL, E.REC_KM, E.REC_BETA] + list(range(E.REC_L, E.LR_REC_DOUBLES))
    assert np.array_equal(got[:, fields], want[:, fields])


def _host_lik(model, start, end, sp, ex, br, state):
    """C + sum A log r - B r of the -model_BDI tables (models 0-2), in the bin mapping of the likelihood."""
    m = br > 0
    A_b = np.where(m, sp, 0.0) if model <= 1 else sp.astype(float)
    B_b = (np.where(m, 1.0, 0.0) if model == 1 else np.where(m, br, 0.0)) if model <= 1 else br
    A_d = np.where(m, ex, 0.0) if model <= 1 else ex.astype(float)
    B_d = np.where(m, br, 0.0) if model <= 1 else br
    C = 0.0 if model >= 2 else float(np.sum(np.where(m, (sp + ex if model == 0 else ex) * np.log(np.where(m, br, 1.0)), 0.0)))
    L, M, tl, tm = state
    rec = np.zeros((1, 1, E.LR_REC_DOUBLES))
    rec[0, 0, [E.REC_KL, E.REC_KM]] = len(L), len(M)
    rec[0, 0, E.REC_L:E.REC_L + len(L)] = L; rec[0, 0, E.REC_TL:E.REC_TL + len(L)] = tl[:-1]
    rec[0, 0, E.REC_M:E.REC_M + len(M)] = M; rec[0, 0, E.REC_TM:E.REC_TM + len(M)] = tm[:-1]
    r = PP.bin_rates(rec, 0, len(sp), start_time=start)[0][0, 0]
    return C + np.sum(A_b * np.log(r[0]) - B_b * r[0]) + np.sum(A_d * np.log(r[1]) - B_d * r[1])


def test_model_detection(tmp_path):
    rng = np.random.default_rng(3)
    start, end = 3.4, 43.7
    sp, ex, br = rng.integers(0, 30, 40), rng.integers(0, 20, 40), rng.uniform(0, 200, 40)
    br[4] = 0.0
    assert [PP.model_tag(p) for p in ("a_BD_mcmc.log", "a_ID_x_mcmc.log", "a_BDk_chain3_mcmc.log", "a_BDd_mcmc.log", "a_mcmc.log")] == \
        [0, 1, 2, 3, None]
    recs = _records(rng, 20, start, end)
    for model in (0, 1, 2):
        for r in recs:
            kl, km = int(r[E.REC_KL]), int(r[E.REC_KM])
            st = (r[E.REC_L:E.REC_L + kl], r[E.REC_M:E.REC_M + km], np.append(r[E.REC_TL:E.REC_TL + kl], end), np.append(r[E.REC_TM:E.REC_TM + km], end))
            r[E.REC_LIK] = _host_lik(model, start, end, sp, ex, br, st)
        tag = {0: "BD", 1: "ID", 2: "BDk"}[model]
        path = _write_logs(str(tmp_path), "t%d_%s" % (model, tag), recs, start, end, sp, ex, br)
        got, m, s, e, gsp, gex, gbr, id0 = PP.forward_logs([path], 0.2, _host_lik)
        assert m == model and np.array_equal(gsp[0], sp) and np.array_equal(gbr[0], br)
        wrong = _write_logs(str(tmp_path), "w%d_%s" % (model, {0: "ID", 1: "BDk", 2: "BD"}[model]), recs, start, end, sp, ex, br)
        with pytest.raises(ValueError, match="likelihood"):
            PP.forward_logs([wrong], 0.2, _host_lik)
    bdd = _write_logs(str(tmp_path), "d_BDd", recs, start, end, sp, ex, br)
    with pytest.raises(ValueError, match="predictive_records_device"):
        PP.forward_logs([bdd], 0.2, _host_lik)


def test_refusals(tmp_path):
    with pytest.raises(SystemExit):
        PP.main([str(tmp_path), "-p_tail", "0.7"])
    with pytest.raises(SystemExit):
        PP.main([str(tmp_path / "missing")])
    with pytest.raises(SystemExit, match="no RJMCMC or DDRate"):
        PP.check_dir(str(tmp_path))
    with open(tmp_path / "x_1_EXPB_EXPD_1.trendrate.log", "w") as fh:
        fh.write("it\tlikelihood\n0\t1.0\n")
    with pytest.raises(SystemExit, match="predictive_records_device"):
        PP.check_dir(str(tmp_path))
    with pytest.raises(ValueError, match="kind"):
        PP.predictive_records_device(None, np.zeros((4, 1, 20)), "proportion", np.zeros((1, 4, 2)))


def test_chain_ids_follow_the_samplers_naming():
    """Chain k of a run over n_tab tables is table k % n_tab (sorted), run k // n_tab: an imputation directory's logs are put in
    chain order, not file-name order."""
    fw = ["d/imp_1_BD_chain0_mcmc.log", "d/imp_0_BD_chain1_mcmc.log", "d/imp_0_BD_chain0_mcmc.log", "d/imp_1_BD_chain1_mcmc.log"]
    paths, id0 = PP.chain_ids(fw, "forward")
    assert id0 == 0 and paths == ["d/imp_0_BD_chain0_mcmc.log", "d/imp_1_BD_chain0_mcmc.log", "d/imp_0_BD_chain1_mcmc.log",
                                  "d/imp_1_BD_chain1_mcmc.log"]
    assert PP.chain_ids(["d/x_BD_chain2_mcmc.log", "d/x_BD_chain3_mcmc.log"], "forward") == (["d/x_BD_chain2_mcmc.log", "d/x_BD_chain3_mcmc.log"], 2)
    assert PP.chain_ids(["d/x_BD_mcmc.log"], "forward") == (["d/x_BD_mcmc.log"], 0)
    dd = ["a/b_11_LDDN_MDDN.log", "a/a_10_LDDN_MDDN.log", "a/b_10_LDDN_MDDN.log", "a/a_11_LDDN_MDDN.log"]
    paths, id0 = PP.chain_ids(dd, "dd")
    assert id0 == 0 and paths == ["a/a_10_LDDN_MDDN.log", "a/b_10_LDDN_MDDN.log", "a/a_11_LDDN_MDDN.log", "a/b_11_LDDN_MDDN.log"]
    with pytest.raises(ValueError, match="consecutive"):
        PP.chain_ids(["d/x_BD_chain0_mcmc.log", "d/x_BD_chain2_mcmc.log"], "forward")
    with pytest.raises(ValueError, match="log name"):
        PP.chain_ids(["a/run.log"], "dd")


def test_dd_logs_refuse_a_short_div_log(tmp_path):
    """-m_birth 3 zips the statistics with the genre table's: a .div.log shorter than the log's bins is refused."""
    from literate_b200 import ddrate as DD
    nb = 5
    head = DD.header(nb, 2)
    row = [0, 1.0, 1.0, 0.0, 0.0, 0.0] + [0.1] * 11 + [0.2] * (4 * nb) + [0.0, 0.0, 0.0]
    with open(tmp_path / "t_1_LDDN_MDDN.log", "w") as fh:
        fh.write("\t".join(head) + "\n")
        for it in range(10):
            fh.write("\t".join(str(v) for v in [it] + row[1:]) + "\n")
    DD.write_div_log(str(tmp_path / "t_1_LDDN_MDDN.div.log"), np.ones(nb - 2, int), np.ones(nb - 2, int), np.ones(nb - 2))
    with pytest.raises(ValueError, match="div.log holds 3 bins"):
        PP.dd_logs([str(tmp_path / "t_1_LDDN_MDDN.log")])
    DD.write_div_log(str(tmp_path / "t_1_LDDN_MDDN.div.log"), np.ones(nb, int), np.ones(nb, int), np.ones(nb))
    recs, terms, id0 = PP.dd_logs([str(tmp_path / "t_1_LDDN_MDDN.log")], burnin=0.2)
    assert recs.shape == (8, 1, 24 + 4 * nb) and terms.shape == (1, 4, nb) and id0 == 0
    assert (recs[:, 0, 24:24 + 2 * nb] == 0.2).all() and list(recs[:, 0, 0]) == list(range(2, 10))
