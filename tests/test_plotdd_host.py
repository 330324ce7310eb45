"""CPU: plotdd's summaries of TrendRate / DDRate sample logs equal the host restatement on the records that produced them."""
import csv
import os
import re

import numpy as np
import pytest

from literate_b200 import ddrate as DD
from literate_b200 import plotdd as PD
from literate_b200 import trend as TR


def synthetic_records(kind, n_samples, n_chains, n_bins, seed):
    """Seeded K6 / K7 records with the layout of the kernels: rates, parameters, beta = 1; some columns repeat one value or
    three values, so the HPD sees ties."""
    rng = np.random.default_rng(seed)
    w = TR.REC_HEAD + 2 * n_bins if kind == "trendrate" else DD.REC_HEAD + 4 * n_bins
    r = rng.gamma(2.0, 0.1, (n_samples, n_chains, w))
    r[..., 0] = np.arange(n_samples)[:, None] * 100
    r[..., 1:5] = -rng.uniform(100, 200, (n_samples, n_chains, 4))
    head = TR.REC_HEAD if kind == "trendrate" else DD.REC_HEAD
    r[..., head + 1] = 0.25                                                    # a constant bin
    r[..., head + 2] = rng.choice([0.1, 0.2, 0.3], (n_samples, n_chains))       # three distinct values
    r[..., TR.REC_BETA if kind == "trendrate" else DD.REC_BETA] = 1.0
    if kind == "dd":
        r[..., 8] = rng.uniform(-20, 40, (n_samples, n_chains))                # x0 relative to the origin
        r[..., 9] = rng.uniform(10, 50, (n_samples, n_chains))                 # div_0
        r[..., 10] = rng.uniform(100, 900, (n_samples, n_chains))              # L
    return r


def write_logs(tmp, kind, recs, n_bins, variant, origin):
    """The logs the command lines would write for these records, through the product's own names, headers and rows."""
    paths = []
    for k in range(recs.shape[1]):
        if kind == "trendrate":
            const_b, const_d, no_death = variant
            path = TR.log_name(os.path.join(tmp, "table.tsv"), 7 + k, 1, const_b, const_d, no_death)
            head, row = TR.header(n_bins), lambda rec: TR.record_row(rec, n_bins)
        else:
            m_birth, m_death = variant
            stem = DD.log_stem(os.path.join(tmp, "table.tsv"), 7 + k, m_birth, m_death)
            path = stem + ".log"
            head, row = DD.header(n_bins, m_birth), lambda rec: DD.record_row(rec, n_bins, m_birth, origin)
            z = np.zeros(n_bins, dtype=np.int64)
            DD.write_div_log(stem + ".div.log", z, z, np.ones(n_bins))
        with open(path, "w", newline="") as fh:
            w = csv.writer(fh, delimiter="\t")
            w.writerow(head)
            for s in range(recs.shape[0]):
                w.writerow(row(recs[s, k]))
        paths.append(path)
    return paths


def assert_same(a, b):
    assert a.kind == b.kind and a.n_samples == b.n_samples and np.array_equal(a.time, b.time)
    assert list(a.series) == list(b.series) and list(a.params) == list(b.params)
    for tag in a.series:
        assert np.array_equal(a.series[tag]["lo"], b.series[tag]["lo"]) and np.array_equal(a.series[tag]["hi"], b.series[tag]["hi"]), tag
        np.testing.assert_allclose(a.series[tag]["mean"], b.series[tag]["mean"], rtol=1e-12, atol=0)
    for p in a.params:
        assert a.params[p]["lo"] == b.params[p]["lo"] and a.params[p]["hi"] == b.params[p]["hi"], p
        np.testing.assert_allclose(a.params[p]["mean"], b.params[p]["mean"], rtol=1e-12, atol=0)


CASES = [("trendrate", (False, False, False)), ("trendrate", (True, False, False)), ("trendrate", (False, True, True)),
         ("dd", (0, 2)), ("dd", (3, 1))]


@pytest.mark.parametrize("kind,variant", CASES)
def test_logs_equal_records(tmp_path, kind, variant):
    nb, origin = 13, 1850.0
    recs = synthetic_records(kind, 57, 3, nb, seed=len(str(variant)))
    paths = write_logs(str(tmp_path), kind, recs, nb, variant, origin)
    assert PD.find_logs(str(tmp_path)) == {kind: sorted(paths)}          # .div.log files are not sample logs
    assert_same(PD.summarize_logs(paths, 0.2, origin), PD.summarize_records(recs, kind, nb, origin, 0.2))
    for k, p in enumerate(paths):                                         # without -combine: one chain per file
        assert_same(PD.summarize_logs([p], 0.3, origin), PD.summarize_records(recs[:, k], kind, nb, origin, 0.3))
    s = PD.summarize_logs(paths)
    assert np.array_equal(s.time, np.arange(nb)) and s.n_samples == 3 * (57 - PD.S.burnin_index(57, 0.2))
    if kind == "dd":                                                      # the log's transforms of x0 and L
        r = recs[PD.S.burnin_index(57, 0.2):].reshape(-1, recs.shape[-1])
        x0, cap = r[:, 8] + origin, r[:, 10] + r[:, 9]
        lo, hi = PD.S.hpd_columns(np.stack([x0, cap], axis=1))
        got = PD.summarize_logs(paths, 0.2).params
        assert (got["midpoint_x0"]["lo"], got["maxCarryingCap"]["lo"]) == tuple(lo)
        assert (got["midpoint_x0"]["hi"], got["maxCarryingCap"]["hi"]) == tuple(hi)
    assert s.series["birth"]["lo"][1] == s.series["birth"]["hi"][1] == 0.25


def test_ladders_summarise_their_cold_members():
    recs = synthetic_records("dd", 40, 8, 5, seed=3)
    beta = np.tile([1.0, 0.5], (40, 4))
    beta[::3] = beta[::3, ::-1]                                            # the cold member changes from sample to sample
    recs[..., DD.REC_BETA] = beta
    cold = recs.reshape(40, 4, 2, -1)[np.arange(40)[:, None], np.arange(4)[None, :], np.argmax(beta.reshape(40, 4, 2), axis=2)]
    assert_same(PD.summarize_records(recs, "dd", 5, ladder=2), PD.summarize_records(cold, "dd", 5))


def _r_vectors(path):
    out = {}
    for line in open(path):
        m = re.fullmatch(r"(\w+)=c\((.*)\)\n", line)
        if m:
            out[m.group(1)] = [x.strip() for x in m.group(2).split(",")]
    return out


@pytest.mark.parametrize("kind,variant", [CASES[0], CASES[4]])
def test_command_line_writes_r_files(tmp_path, kind, variant):
    nb = 11
    recs = synthetic_records(kind, 30, 2, nb, seed=5)
    paths = write_logs(str(tmp_path), kind, recs, nb, variant, 0.0)
    written = PD.main([str(tmp_path), "-combine", "1", "-origin", "1900"])
    tag = "DD" if kind == "dd" else "trendrate"
    assert written == [os.path.join(str(tmp_path), "COMBINED_%s_plots.r" % tag)]
    per_file = PD.main([str(tmp_path), "-burnin", "0.1"])
    assert per_file == [PD.log_stem(p) + "_plots.r" for p in sorted(paths)]
    for path in written + per_file:
        v = _r_vectors(path)
        series = ["birth_rate", "death_rate", "net_rate"] + (["niche_mean", "nicheFrac_mean"] if kind == "dd" else [])
        for name in ["time"] + series + [s.split("_")[0] + t for s in series for t in ("_minHPD", "_maxHPD")]:
            assert len(v[name]) == nb and all(float(x) == float(x) for x in v[name]), name
        assert len(v["param_mean"]) == len(PD.param_names(kind)) == len(v["params"])
    v = _r_vectors(written[0])
    assert [float(x) for x in v["time"]] == list(1900.5 + np.arange(nb))
    assert PD.find_logs(str(tmp_path)) == {kind: sorted(paths)}           # the R files and combined outputs are not logs
