"""CPU: host side of the DDRate path (literate_b200/ddrate.py) -- log naming, header, row and div.log formatting -- against
the oracle pinned to the unmodified DDRatev3.py.  No GPU work."""
import csv
import io
import os

import numpy as np
import pytest

from oracle import ddrate_oracle as D
from literate_b200 import ddrate as DD
from literate_b200 import library as L
from test_oracle_ddrate_golden import DG, _flag, _jobs, setup_job


@pytest.mark.parametrize("tag", ["ex_g_mddn", "ex_g_rmfirst"])
def test_rows_from_records_are_byte_identical_to_the_reference_log(tag, tmp_path):
    job = [j for j in _jobs() if j["tag"] == tag][0]
    a = job["args"]
    data, S, gbins = setup_job(job, tmp_path)
    rows = D.run_chain(S, 601, 50, _flag(a, "-seed", -1, int), None, exact_scipy=True, collect=True)
    nb = S.n
    buf = io.StringIO(newline="")
    w = csv.writer(buf, delimiter="\t")
    w.writerow(DD.header(nb, 3))
    for r in rows:
        rec = np.zeros(DD.REC_HEAD + 4 * nb)
        rec[0], rec[1], rec[2], rec[3], rec[4] = r[0], r[2], r[3], r[4], r[5]
        rec[5:16] = r[6:17]
        rec[5 + 3] = r[6 + 3] - S.origin            # the chain holds x0 relative to the origin and L without div_0 (:278-279)
        rec[5 + 5] = r[6 + 5] - r[6 + 4]
        rec[16] = r[17]
        rec[DD.REC_HEAD:] = r[18:18 + 4 * nb]
        rec[17:20] = r[18 + 4 * nb:]
        w.writerow(DD.record_row(rec, nb, 3, S.origin))
    want = open(os.path.join(DG, tag, [f for f in job["files"] if not f.endswith(".div.log")][0]), "rb").read()
    got = buf.getvalue().encode().split(b"\r\n")
    ref = want.split(b"\r\n")[:len(got) - 1]
    # adding the origin back to x0 (and div_0 to L) is exact only if the subtraction above was: compare as numbers there
    assert got[0] == ref[0]
    for g, r in zip(got[1:], ref[1:]):
        gf, rf = g.split(b"\t"), r.split(b"\t")
        assert len(gf) == len(rf)
        for k, (x, y) in enumerate(zip(gf, rf)):
            if k in (9, 11):
                assert float(x) == pytest.approx(float(y), rel=1e-14)
            else:
                assert x == y
    stem = DD.log_stem(data, _flag(a, "-seed", -1, int), 3, S.m_death)
    assert sorted(os.path.basename(stem) + e for e in (".log", ".div.log")) == job["files"]
    p = os.path.join(str(tmp_path), "div.log")
    DD.write_div_log(p, S.bins.n_spec, S.bins.n_exti, S.bins.dt, gbins.n_spec, gbins.n_exti, gbins.dt)
    assert open(p, "rb").read() == open(os.path.join(DG, tag, [f for f in job["files"] if f.endswith(".div.log")][0]), "rb").read()


def test_window_and_flags(tmp_path):
    job = _jobs()[0]
    data, S, gbins = setup_job(job, tmp_path)
    ts, te, present, origin = L.parse_ts_te(data)
    first, nb = L.bin_window(origin, present, 0)
    assert (first, nb) == (S.origin, S.n) and present == S.present
    a = DD.build_parser().parse_args(["-d", "x.tsv"])
    assert (a.m_birth, a.m_death, a.n, a.s, a.seed, a.genre_times, a.chains) == (2, 2, 10000000, 1000, -1, "", 1)
    assert DD.log_stem("a/b.tsv", 5, 2, 0) == "a/b_5_LDDN_ML" and DD.log_stem("b.tsv", 5, 0, 1) == "b_5_LL_MDD"
