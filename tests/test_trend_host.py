"""CPU: host side of the TrendRate path (literate_b200/trend.py) -- parsing, bin window, trend normalisation, log naming
and row formatting -- against the oracle pinned to the unmodified trend_rate.py.  No GPU work."""
import csv
import io
import os

import numpy as np
import pytest

from oracle import trendrate_oracle as T
from literate_b200 import library as L
from literate_b200 import trend as TR
from test_oracle_trend_golden import TG, _flag, _jobs, setup_job, stage


@pytest.mark.parametrize("job", _jobs(), ids=lambda j: j["tag"])
def test_parsing_and_window_equal_the_oracle(job, tmp_path):
    a = job["args"]
    data, trend_path = stage(job, tmp_path)
    rm, jit = _flag(a, "-rm_first_bin", 0.0), _flag(a, "-death_jitter", 0.5)
    ts, te, present, origin = L.parse_ts_te(data, death_jitter=jit)
    ots, ote, opresent, oorigin = T.parse_ts_te(data, death_jitter=jit)
    assert np.array_equal(ts, ots) and np.array_equal(te, ote) and (present, origin) == (opresent, oorigin)
    bins = T.create_bins(oorigin, opresent, ots, ote, rm)
    first, nb = L.bin_window(origin, present, rm)
    assert nb == bins.n_bins and first == bins.origin
    idx = _flag(a, "-trend_index", 0, int)
    assert np.array_equal(TR.parse_trend_data(trend_path, idx, rm), T.normalise_trend(T.read_trend_column(trend_path, idx), rm))


def test_rows_from_records_are_byte_identical_to_the_reference_log(tmp_path):
    """The same numbers give the same text: records built from the oracle's sampled rows, written by the product's
    writer, reproduce the unmodified reference's log byte for byte."""
    job = [j for j in _jobs() if j["tag"] == "ex_hump"][0]
    a = job["args"]
    data, bins, trend, idx, flags = setup_job(job, tmp_path)
    rows = T.run_chain(bins, trend, _flag(a, "-n", 0, int), _flag(a, "-s", 1000, int), _flag(a, "-seed", -1, int), None,
                       exact_scipy=True, collect=True, **flags)
    nb = bins.n_bins
    buf = io.StringIO(newline="")
    w = csv.writer(buf, delimiter="\t")
    w.writerow(TR.header(nb))
    for r in rows:
        rec = np.zeros(TR.REC_HEAD + 2 * nb)
        rec[0], rec[1], rec[2], rec[3], rec[4] = r[0], r[2], r[3], r[4], r[5]
        rec[5:11] = r[6:12]
        rec[TR.REC_HEAD:] = r[12:12 + 2 * nb]
        rec[11:14] = r[12 + 2 * nb:]
        w.writerow(TR.record_row(rec, nb))
    want = open(os.path.join(TG, job["tag"], job["files"][0]), "rb").read()
    assert buf.getvalue().encode() == want
    name = TR.log_name(data, 2, idx, flags["const_birth"], flags["const_death"], flags["no_death"])
    assert os.path.basename(name) == job["files"][0]


def test_flags_follow_the_reference_parser():
    p = TR.build_parser()
    a = p.parse_args(["-d", "x.tsv", "-trend_data", "t.tsv", "-const_B", "0", "-no_death", "False"])
    assert a.const_B is True and a.no_death is True and a.const_D is False      # argparse type=bool: any non-empty string
    assert (a.n, a.s, a.p, a.seed, a.death_jitter, a.trend_index, a.chains) == (10000000, 1000, 1000, -1, .5, 0, 1)
    with pytest.raises(SystemExit):
        L.bin_window(1994.25, 2017.5)
