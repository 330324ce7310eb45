"""GPU: K8 (lr_column_hpd) against summary.hpd_columns, and plotdd's device summaries of K6 / K7 records against the host
restatement -- HPD bounds bit for bit (NaN equal; the sign of a zero is free), means to 1e-12 of the host's (1e-14 of the correctly
rounded mean for the kernel alone)."""
import math
import os

import numpy as np
import pytest
import torch

from literate_b200 import ddrate as DD
from literate_b200 import engine as E
from literate_b200 import library as L
from literate_b200 import parallel as P
from literate_b200 import plotdd as PD
from literate_b200 import summary as S
from literate_b200 import trend as TR
from test_gpu_sibling_tempering import _synthetic
from test_oracle_ddrate_golden import _jobs as dd_jobs, stage as dd_stage
from test_oracle_trend_golden import _jobs as trend_jobs, stage as trend_stage
from test_plotdd_host import assert_same

pytestmark = pytest.mark.gpu


def _kernel(device, x, level, cols=None, mask_col=-1):
    d = torch.from_numpy(np.ascontiguousarray(x)).cuda()
    out = device.column_hpd_device(d, range(x.shape[1]) if cols is None else cols, level, mask_col)
    torch.cuda.synchronize()
    return [t.cpu().numpy() for t in out]


def _correct_mean(h):
    """Per column the correctly rounded sum (math.fsum) over n; columns holding inf or NaN as numpy has them.  (numpy's mean over
    axis 0 adds the rows one after another: on 262 143 draws of 0.1, 0.2, 0.3 it is 1.5e-12 off, relatively.)"""
    with np.errstate(invalid="ignore"):
        out = h.mean(axis=0)
    for j in range(h.shape[1]):
        if np.all(np.isfinite(h[:, j])):
            out[j] = math.fsum(h[:, j]) / h.shape[0]
    return out


def _check(device, x, level, cols=None, mask_col=-1, host=None):
    mean, lo, hi, n = _kernel(device, x, level, cols, mask_col)
    h = x if host is None else host
    wlo, whi = S.hpd_columns(h, level)
    assert np.array_equal(lo, wlo, equal_nan=True) and np.array_equal(hi, whi, equal_nan=True)
    np.testing.assert_allclose(mean, _correct_mean(h), rtol=1e-14, atol=0)
    assert n[0] == h.shape[0]
    again = _kernel(device, x, level, cols, mask_col)
    assert all(np.array_equal(a, b, equal_nan=True) and np.array_equal(np.signbit(a), np.signbit(b)) for a, b in zip(again, (mean, lo, hi, n)))


def _columns(rng, n):
    """Continuous, three-valued, constant, with +-inf, with NaN, mixed -0.0 / +0.0, negative."""
    x = np.stack([rng.gamma(2.0, 0.1, n), rng.choice([0.1, 0.2, 0.3], n), np.full(n, 0.25), rng.normal(5, 1, n),
                  rng.choice([-0.0, 0.0, 1.0], n), -rng.exponential(1.0, n)], axis=1)
    x[rng.random(n) < 0.02, 3] = np.inf
    x[rng.random(n) < 0.02, 3] = -np.inf
    nan = x[:, 0].copy()
    nan[rng.random(n) < 0.03] = np.nan
    return np.concatenate([x, nan[:, None]], axis=1)


@pytest.mark.parametrize("n", [2, 39, 40, 1000, 262_143])
@pytest.mark.parametrize("level", [0.5, 0.95, 0.99, 1.0])
def test_kernel_equals_hpd_columns(device, n, level):
    rng = np.random.default_rng(n)
    x = _columns(rng, n)
    if int(round(level * n)) < 2:
        with pytest.raises(RuntimeError, match="not enough data"):
            _kernel(device, x, level)
        return
    _check(device, x, level)


def test_one_row_is_not_enough(device):
    with pytest.raises(RuntimeError, match="not enough data"):
        _kernel(device, np.ones((1, 3)), 0.95)
    x = np.ones((10, 3))
    x[:, 2] = 0.0
    x[4, 2] = 1.0                                                           # one row passes the mask: rint(0.95) = 1
    with pytest.raises(RuntimeError, match="not enough data"):
        _kernel(device, x, 0.95, mask_col=2)


def test_many_rows_and_groups(device):
    rng = np.random.default_rng(11)
    _check(device, _columns(rng, 4_200_000)[:, [0, 1, 4]], 0.95)           # more than 4 M rows
    x = rng.gamma(2.0, 0.1, (5000, 70))                                     # more columns than one group (32)
    x[:, 40] = 3.0
    _check(device, x, 0.95)


def test_column_specs_and_mask(device):
    rng = np.random.default_rng(12)
    x = rng.gamma(2.0, 0.1, (20_000, 9))
    x[:, 8] = (rng.random(20_000) < 0.3).astype(float)
    cols = [0, (1, 2, -1), (3, 4, 1), (5, -1, 1, 1850.0), (6, 7, 1, -3.5)]
    host = np.stack([x[:, 0], x[:, 1] - x[:, 2], x[:, 3] + x[:, 4], x[:, 5] + 1850.0, (x[:, 6] + x[:, 7]) + -3.5], axis=1)
    _check(device, x, 0.95, cols, host=host)
    keep = x[:, 8] == 1.0
    _check(device, x, 0.95, cols, mask_col=8, host=host[keep])


def test_bad_columns_are_refused(device):
    d = torch.zeros((10, 4), dtype=torch.float64, device="cuda")
    for cols in ([4], [(0, 4, 1)], [(0, 1, 2)], [-1]):
        with pytest.raises(E.NativeError, match="lr_column_hpd"):
            device.column_hpd_device(d, cols)
    with pytest.raises(E.NativeError, match="lr_column_hpd"):
        device.column_hpd_device(d, [0], level=1.5)


@pytest.mark.parametrize("kind", ["trend", "dd"])
@pytest.mark.parametrize("nb", [24, 200])
def test_device_summary_of_records(device, kind, nb):
    ch = _synthetic(device, kind, nb, 16, 5)
    rec = torch.empty((ch.records_per_run(20001, 100), 16, ch.rec_doubles), dtype=torch.float64, device="cuda")
    ch.run_device(20001, 100, rec)
    torch.cuda.synchronize()
    k = "trendrate" if kind == "trend" else "dd"
    for origin in (0.0, 1850.0):
        assert_same(PD.summarize_records_device(device, rec, k, nb, origin), PD.summarize_records(rec.cpu().numpy(), k, nb, origin))


@pytest.mark.parametrize("kind", ["trend", "dd"])
def test_cold_members_of_ladders(device, kind):
    T, n = 4, 16
    ch = _synthetic(device, kind, 24, n, 9)
    ch.set_beta(np.tile(P.temperature_ladder(T, 0.3), n // T))
    recs, _ = ch.run_tempered(8001, 50, T, 200)
    k = "trendrate" if kind == "trend" else "dd"
    dev = PD.summarize_records_device(device, torch.from_numpy(recs).cuda(), k, 24, cold_only=True)
    assert len(np.unique(recs[..., ch.REC_BETA])) == T
    assert_same(dev, PD.summarize_records(E.cold_records(recs, T, ch.REC_BETA), k, 24))
    assert_same(dev, PD.summarize_records(recs, k, 24, ladder=T))


def test_trendrate_command_line_to_plotdd(device, tmp_path):
    job = [j for j in trend_jobs() if j["tag"] == "ex_ramp"][0]
    data, trend_path = trend_stage(job, tmp_path)
    TR.main(["-d", data, "-trend_data", trend_path, "-trend_index", "1", "-n", "3001", "-s", "50", "-seed", "3", "-chains", "8", "-quiet", "1"])
    ts, te, present, origin = L.parse_ts_te(data)
    first, nb = L.bin_window(origin, present)
    st = device.bin_stats(ts, te, first_bin=first, n_bins=nb)
    ch = TR.TrendChains(device, st.sp, st.ex, st.br, TR.parse_trend_data(trend_path, 1), 8, 3)
    rec = torch.empty((ch.records_per_run(3001, 50), 8, ch.rec_doubles), dtype=torch.float64, device="cuda")
    ch.run_device(3001, 50, rec)
    torch.cuda.synchronize()
    out = PD.main([str(tmp_path), "-combine", "1", "-origin", repr(origin)])
    assert out == [os.path.join(str(tmp_path), "COMBINED_trendrate_plots.r")]
    logs = PD.find_logs(str(tmp_path))["trendrate"]
    assert len(logs) == 8
    assert_same(PD.summarize_logs(logs, 0.2, origin), PD.summarize_records_device(device, rec, "trendrate", nb, origin))


def test_ddrate_command_line_to_plotdd(device, tmp_path):
    job = [j for j in dd_jobs() if j["tag"] == "ex_g_mddn"][0]
    data, genre = dd_stage(job, tmp_path)
    DD.main(["-d", data, "-m_birth", "3", "-g", genre, "-n", "3001", "-s", "50", "-seed", "3", "-chains", "8", "-quiet", "1"])
    ts, te, present, origin = L.parse_ts_te(data)
    gts, gte, _, _ = L.parse_ts_te(genre)
    first, nb = L.bin_window(origin, present)
    st = device.bin_stats(ts, te, first_bin=first, n_bins=nb)
    ch = DD.DDChains(device, st.sp, st.ex, st.br, origin, present, 3, 2, gts, gte, 8, 3)
    rec = torch.empty((ch.records_per_run(3001, 50), 8, ch.rec_doubles), dtype=torch.float64, device="cuda")
    ch.run_device(3001, 50, rec)
    torch.cuda.synchronize()
    out = PD.main([str(tmp_path), "-combine", "1", "-origin", repr(origin)])
    assert out == [os.path.join(str(tmp_path), "COMBINED_DD_plots.r")]
    logs = PD.find_logs(str(tmp_path))["dd"]
    assert len(logs) == 8
    assert_same(PD.summarize_logs(logs, 0.2, origin), PD.summarize_records_device(device, rec, "dd", nb, origin))
