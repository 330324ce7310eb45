"""GPU: K1 against its exact reference (oracle/k1_exact.py) -- no tolerance anywhere.

sp, ex and ex_dead equal, br and br_dead the same bits as the correctly rounded exact sums, through every entry point
(lr_bin_stats_host, lr_bin_stats on device tables with a padded row pitch, lr_bin_accumulate + lr_bin_finalize) and every
build (general, lane-private where it fits, the automatic choice twice so that the table-kind hint can switch it), on the
tables where a fixed-point pass goes wrong: real-valued times (whose low bits are not zero), sorted tables (run-length and
warp-merge paths), the automatic lane-private threshold, times in (-1, 1) and negative years, lineages far outside the window
and at +-inf, the shared-memory limits of both builds, one bin whose lane words carry into the third word, ragged replicates,
lineage shards finalized once, and the int32 year path.
"""
import numpy as np
import pytest

from conftest import golden_input
from oracle import k1_exact as K
from literate_b200 import _native as N, engine as E, forward as F, synth

pytestmark = pytest.mark.gpu

GENERAL, LANES = "k1_bin_kernel", "k1_bin_lanes_kernel"
NAMES = ("sp", "ex", "br", "ex_dead", "br_dead")


def _want(ts2, te2, fb, nb, end):
    rows = [K.exact_bin_stats(ts2[r], te2[r], fb, nb, only_dead=True, end_time=end) for r in range(ts2.shape[0])]
    return tuple(np.stack([row[k] for row in rows]) for k in range(5))


def _assert_exact(got, want, what):
    for name, g, w in zip(NAMES, got, want):
        g = np.asarray(g)
        assert g.shape == w.shape, (what, name)
        same = g.view(np.int64) == w.view(np.int64)
        if not same.all():
            bad = np.argwhere(~same)
            i = tuple(bad[0])
            raise AssertionError("%s: %s differs in %d bins, first %s: got %r want %r" % (what, name, len(bad), i, g[i], w[i]))


def _end_time(te):
    """A death time of the table itself: only_dead keeps te < end_time strictly."""
    f = np.sort(te[np.isfinite(te)])
    return float(f[int(0.6 * (len(f) - 1))])


def _expect(build, entry, nb, n, n_rep, pitch, hint):
    """The build lr_bin_accumulate must pick (its stated rule)."""
    if build == "general":
        return GENERAL
    fits = nb <= 439 and (entry == "host" or n_rep == 1 or pitch % 2 == 0)
    if build == "lanes":
        return LANES if fits else GENERAL
    if entry == "host":
        return GENERAL
    pays = (nb <= 310 and n >= 250_000) or (hint == 1 and n >= 50_000)
    return LANES if fits and pays else GENERAL


def _set_build(monkeypatch, build):
    if build == "auto":
        monkeypatch.delenv("LR_K1_LANES", raising=False)
    else:
        monkeypatch.setenv("LR_K1_LANES", "1" if build == "lanes" else "0")


def _run_entry(dev, entry, build, ts2, te2, dts, dte, fb, nb, end, pitch):
    """One entry point, the full and the extinct-only statistics; every K1 pass checked for the build it ran."""
    import torch
    n_rep, n = ts2.shape
    if entry == "host":
        hint = dev.bin_table_hint()
        r = dev.bin_stats(ts2, te2, first_bin=fb, n_bins=nb, only_dead=True, end_time=end, fe_ref=0.5)
        assert dev.bin_last_build() == _expect(build, entry, nb, n, n_rep, pitch, hint), (entry, build)
        return (r.sp, r.ex, r.br, r.ex_dead, r.br_dead)
    out = []
    for dead in (False, True):
        torch.cuda.synchronize()
        hint = dev.bin_table_hint()
        if entry == "device":
            res = dev.bin_stats_device(dts, dte, fb, nb, fe_ref=1.0, dead_only=dead, end_time=end)
        else:
            acc = dev.new_accumulators(n_rep, nb, dts.device)
            dev.bin_accumulate_device(dts, dte, fb, nb, acc, fe_ref=0.5, dead_only=dead, end_time=end)
            res = dev.bin_finalize_device(acc, nb, fe_ref=0.5)
        assert dev.bin_last_build() == _expect(build, entry, nb, n, n_rep, pitch, hint), (entry, build, dead)
        torch.cuda.synchronize()
        out.append([x.cpu().numpy() for x in res])
    return (out[0][0], out[0][1], out[0][2], out[1][1], out[1][2])


def _to_device(ts2, te2, pitch):
    import torch
    n_rep, n = ts2.shape
    dts = torch.full((n_rep, pitch), float("nan"), dtype=torch.float64, device="cuda")
    dte = torch.full((n_rep, pitch), float("nan"), dtype=torch.float64, device="cuda")
    dts[:, :n] = torch.from_numpy(ts2).cuda(); dte[:, :n] = torch.from_numpy(te2).cuda()
    return dts[:, :n], dte[:, :n]


def _check_all(dev, monkeypatch, ts, te, fb, nb, end=None, want=None, pitch=None, what=""):
    """Every entry point under every build, bit for bit against the exact reference.  A 1-D table is binned as two replicates
    (the table and its reverse), so that the device entries see a padded row pitch."""
    ts2 = np.ascontiguousarray(ts if ts.ndim == 2 else np.stack([ts, ts[::-1]]))
    te2 = np.ascontiguousarray(te if te.ndim == 2 else np.stack([te, te[::-1]]))
    n_rep, n = ts2.shape
    if end is None:
        end = _end_time(te2[0])
    if want is None:
        want = _want(ts2, te2, fb, nb, end)
    if pitch is None:
        pitch = (n + 7) // 2 * 2
    dts, dte = _to_device(ts2, te2, pitch)
    for build in ("general", "lanes", "auto"):
        _set_build(monkeypatch, build)
        for entry in ("host", "device", "accumulate"):
            for rnd in range(2 if build == "auto" else 1):
                got = _run_entry(dev, entry, build, ts2, te2, dts, dte, fb, nb, end, pitch)
                _assert_exact(got, want, (what, build, entry, rnd))
    return want


def _scatter(rng, ts, te, rows):
    """Put hand-made rows at spread-out positions (head, tiles and tail of the segments)."""
    ts, te = ts.copy(), te.copy()
    idx = rng.choice(len(ts), len(rows), replace=False)
    for i, (s, e) in zip(idx, rows):
        ts[i], te[i] = s, e
    return ts, te


def test_bench_size_real_valued_shuffled_and_sorted(device, monkeypatch):
    """syn_real at 1M lineages: shuffled, sorted by birth (run-length / warp-merge path of the birth side), by death."""
    ts, te = synth.syn_real(1_000_000)
    end = _end_time(te)
    want = None
    for name, o in (("shuffled", np.arange(len(ts))), ("by birth", np.argsort(ts, kind="stable")),
                    ("by death", np.argsort(te, kind="stable"))):
        want = _check_all(device, monkeypatch, ts[o], te[o], 1800, 200, end=end, want=want, what=name)


@pytest.mark.parametrize("n", [49_999, 50_001])
def test_either_side_of_the_lane_private_threshold(device, monkeypatch, n):
    ts, te = synth.syn_real(n, replicate=n)
    _check_all(device, monkeypatch, ts, te, 1800, 200, what=n)
    # a real-valued table leaves the hint at 1: the second automatic pass takes the lane-private build from 50 000 on
    import torch
    monkeypatch.delenv("LR_K1_LANES", raising=False)
    t, e = _to_device(ts[None, :], te[None, :], n)
    for _ in range(2):
        device.bin_stats_device(t, e, 1800, 200, fe_ref=1.0)
        torch.cuda.synchronize()
    assert device.bin_table_hint() == 1
    assert device.bin_last_build() == (LANES if n >= 50_000 else GENERAL)


def test_times_inside_minus_one_one_and_negative_years(device, monkeypatch):
    """A TBP table near the present (times in [0, 1) and fractions that quantize to the grid) and a table of BCE years
    (the automatic window starts at int(min ts), so some lineages are born before it)."""
    rng = np.random.default_rng(41)
    n = 60_000
    ts = rng.uniform(0, 30, n); ts[: n // 3] = rng.uniform(0, 1, n // 3)
    te = ts + rng.exponential(2.0, n); te[: n // 6] = ts[: n // 6] + rng.uniform(0, 1e-3, n // 6)
    ts, te = _scatter(rng, ts, te, [(2.0 ** -60, 2.0 ** -59), (0.0, 2.0 ** -53), (2.0 ** -53, 3 * 2.0 ** -53), (0.3, 0.9),
                                    (0.0, 1.0), (1 - 2.0 ** -54, 1.0), (0.5, 0.5)])
    fb, nb = E.window(ts, te)
    assert fb == 0
    _check_all(device, monkeypatch, ts, te, fb, nb, what="near the present")
    ts = rng.uniform(-800.0, 50.0, n); te = ts + rng.exponential(20.0, n)
    ts, te = _scatter(rng, ts, te, [(-0.3, -2.0 ** -60), (-2.0 ** -60, 0.7), (-1.0, -1 + 2.0 ** -53), (-0.5 - 2.0 ** -54, -0.25),
                                    (-3.0, -1.0), (-1.5, 0.0), (-2.0, -2.0), (-7.25, -9.0)])
    fb, nb = E.window(ts, te)
    assert fb > np.min(ts)
    _check_all(device, monkeypatch, ts, te, fb, nb, what="BCE years")


FAR = [(-3e9, 1900.5), (-np.inf, 1850.25), (1900.3, 5e9), (1900.7, np.inf), (-np.inf, np.inf), (-5e9, -4e9), (3e9, 4e9),
       (-np.inf, -np.inf), (np.inf, np.inf), (1e300, 1e301), (-1e300, 1799.5), (np.nan, 1900.5), (1850.5, np.nan),
       (-2.0 ** 31 - 0.5, 2.0 ** 31 + 0.5), (2.0 ** 31, 2.0 ** 31 + 1), (-2.0 ** 31 - 1, -2.0 ** 31)]


def test_lineages_far_outside_the_window(device, monkeypatch):
    """|t| beyond 2^31 and +-inf: __double2int_rd / ru saturate, and the bin index must still fall outside the window;
    windows at both ends of the admissible first_bin (|first_bin| < 2^30)."""
    rng = np.random.default_rng(43)
    ts, te = synth.syn_real(100_000, replicate=5)
    ts, te = _scatter(rng, ts, te, FAR * 4)
    _check_all(device, monkeypatch, ts, te, 1800, 200, what="1800")
    for fb in (2 ** 30 - 1, -(2 ** 30 - 1)):
        nb = 100
        s = fb + rng.uniform(-5, nb + 5, 60_000); e = s + rng.exponential(10.0, 60_000)
        rows = [(fb - 0.5, float(fb)), (float(fb), fb + 0.5), (float(fb + nb), fb + nb + 1.0)] + \
               [(a + (fb - 1800 if np.isfinite(a) and abs(a) < 1e4 else 0), b + (fb - 1800 if np.isfinite(b) and abs(b) < 1e4 else 0))
                for a, b in FAR]
        s, e = _scatter(rng, s, e, rows)
        _check_all(device, monkeypatch, s, e, fb, nb, what=fb)


@pytest.mark.parametrize("nb", [1, 310, 311, 439, 440, 6000])
def test_window_sizes(device, monkeypatch, nb):
    """One bin; the widest windows of the 4-deep (310) and 2-deep (439) lane-private build and one bin more; 6000 bins
    (general build only).  Lineages before, across and after the window."""
    rng = np.random.default_rng(nb)
    n = 60_000
    ts = 1000 + rng.uniform(-2, nb + 2, n); te = ts + rng.exponential(max(nb / 8, 0.7), n)
    _check_all(device, monkeypatch, ts, te, 1000, nb, what=nb)


def test_one_bin_every_lineage_fractions_near_one(device, monkeypatch):
    """24M lineages in ONE bin with both fractions near 1: every lane's two fraction words of the lane-private build wrap
    (> 4096 additions of ~2^52 per CTA and lane) into the shared third word; the general build's 96-bit chains carry into their
    top word; the finalized sum needs the sticky rounding of the 128-bit conversion."""
    import torch
    rng = np.random.default_rng(47)
    n = 24_000_000
    te = 11.0 - rng.uniform(0, 1e-6, n)
    ts = te - 1e-9 - rng.uniform(0, 1e-3, n)
    end = float(np.median(te))
    want = _want(ts[None, :], te[None, :], 9, 3, end)
    assert want[0][0, 1] == n and want[2][0, 1] > 2.0 ** 13
    dts, dte = torch.from_numpy(ts).cuda()[None, :], torch.from_numpy(te).cuda()[None, :]
    for build in ("general", "lanes", "auto"):
        _set_build(monkeypatch, build)
        for entry in ("host", "device", "accumulate"):
            got = _run_entry(device, entry, build, ts[None, :], te[None, :], dts, dte, 9, 3, end, n)
            _assert_exact(got, want, (build, entry))


def test_ragged_replicates_with_nan_padding_and_odd_pitch(device, monkeypatch):
    """Five replicates of different lengths padded with NaN rows; the device entries get an odd row pitch (the scalar load
    path of the general build; the lane-private one needs 16-byte rows and is not taken)."""
    n_rep, n = 5, 3001
    ts = np.full((n_rep, n), np.nan); te = np.full((n_rep, n), np.nan)
    for r in range(n_rep):
        m = n - 211 * r
        ts[r, :m], te[r, :m] = synth.syn_real(m, replicate=60 + r)
    _check_all(device, monkeypatch, ts, te, 1800, 200, end=_end_time(te[0]), pitch=n, what="ragged")


def test_lineage_shards_finalized_once(device, monkeypatch):
    """parallel.bin_stats_lineage_sharded across ranks: shards of one real-valued table accumulated by different builds into
    one block with one fe_ref, finalized once -> the exact statistics of the whole table; another order, the same bits."""
    import torch
    ts, te = synth.syn_real(300_000, replicate=9)
    rng = np.random.default_rng(53)
    o = rng.permutation(len(ts)); ts, te = ts[o], te[o]
    end = _end_time(te)
    want = _want(ts[None, :], te[None, :], 1800, 200, end)
    t, e = torch.from_numpy(ts).cuda(), torch.from_numpy(te).cuda()
    cuts = [0, 100_000, 200_002, 300_000]
    shards = [(t[a:b], e[a:b]) for a, b in zip(cuts[:-1], cuts[1:])]
    results = []
    for order, builds in (((0, 1, 2), ("general", "lanes", "auto")), ((2, 0, 1), ("lanes", "auto", "general"))):
        acc = device.new_accumulators(1, 200, t.device); accd = device.new_accumulators(1, 200, t.device)
        for k, build in zip(order, builds):
            _set_build(monkeypatch, build)
            device.bin_accumulate_device(shards[k][0], shards[k][1], 1800, 200, acc, fe_ref=0.5)
            device.bin_accumulate_device(shards[k][0], shards[k][1], 1800, 200, accd, fe_ref=0.5, dead_only=True, end_time=end)
            if build != "auto":
                assert device.bin_last_build() == (GENERAL if build == "general" else LANES)
        sp, ex, br = device.bin_finalize_device(acc, 200, fe_ref=0.5)
        _, exd, brd = device.bin_finalize_device(accd, 200, fe_ref=0.5)
        torch.cuda.synchronize()
        got = tuple(x.cpu().numpy() for x in (sp, ex, br, exd, brd))
        _assert_exact(got, want, order)
        results.append(got)
    for a, b in zip(*results):
        assert a.view(np.int64).tolist() == b.view(np.int64).tolist()


# ---------------------------------------------------------------- int32 years
ACCEPTED = (0.0, 2.0 ** -22, 0.25, 0.5, 1.0)
REFUSED = (0.1, 0.3, 0.05, 0.001, 1e-14, 2.0 ** -30)
LIM = 2 ** 31 - 3                      # the largest |year| forward.as_year_table admits


def _year_tables():
    """(name, ts [n_rep, n] int32, te, first_bin, n_bins): negative years, years at the int32 limits, YEAR_PAD rows,
    windows at |first_bin| = 2^30 - 1."""
    rng = np.random.default_rng(61)
    out = []
    n = 20_011
    ty = rng.integers(-700, 300, n); ey = ty + rng.integers(-3, 60, n)
    edge = [(LIM, LIM), (-LIM, -LIM + 5), (-LIM, LIM), (LIM - 10, LIM), (-LIM, -400), (-400, LIM), (-400, -400), (-401, -402)]
    for i, (a, b) in enumerate(edge):
        ty[7 * i + 3], ey[7 * i + 3] = a, b
    out.append(("BCE years, cut window", ty[None, :], ey[None, :], -400, 500))
    for fb in (2 ** 30 - 1, -(2 ** 30 - 1)):
        ty = fb + rng.integers(-5, 60, n); ey = ty + rng.integers(-1, 30, n)
        for i, (a, b) in enumerate(edge[:6]):
            ty[5 * i + 1], ey[5 * i + 1] = a, b
        out.append(("first_bin %d" % fb, ty[None, :], ey[None, :], fb, 50))
    n_rep, n = 5, 3001
    T = np.full((n_rep, n), E.YEAR_PAD, dtype=np.int64); Ee = np.full((n_rep, n), E.YEAR_PAD, dtype=np.int64)
    for r in range(n_rep):
        m = n - 211 * r
        s, e = synth.syn_int(m, replicate=70 + r)
        T[r, :m], Ee[r, :m] = s, e - 0.5
    out.append(("ragged, YEAR_PAD", T, Ee, 1800, 200))
    return [(name, a.astype(np.int32), b.astype(np.int32), fb, nb) for name, a, b, fb, nb in out]


@pytest.mark.parametrize("jitter", ACCEPTED)
def test_int32_years_exact(device, jitter):
    """lr_bin_stats_host_i32 and lr_bin_accumulate_i32 give the exact statistics of the fp64 table (ts, te + jitter)."""
    import torch
    for name, ti, ei, fb, nb in _year_tables():
        ts = ti.astype(np.float64); te = ei.astype(np.float64) + jitter
        pad = ti == E.YEAR_PAD
        ts[pad] = np.nan; te[pad] = np.nan                   # a ragged replicate's padding as the fp64 table holds it
        end = _end_time(te[0])
        want = _want(ts, te, fb, nb, end)
        r = device.bin_stats(ti, ei, first_bin=fb, n_bins=nb, death_jitter=jitter, only_dead=True, end_time=end)
        _assert_exact((r.sp, r.ex, r.br, r.ex_dead, r.br_dead), want, (name, jitter, "host"))
        dti, dei = torch.from_numpy(ti).cuda(), torch.from_numpy(ei).cuda()
        res = []
        for dead in (False, True):
            acc = device.new_accumulators(ti.shape[0], nb, dti.device)
            device.bin_accumulate_device(dti, dei, fb, nb, acc, death_jitter=jitter, dead_only=dead, end_time=end)
            res.append(device.bin_finalize_device(acc, nb, fe_ref=E.fe_ref_for_jitter(jitter)))
        torch.cuda.synchronize()
        got = [x.cpu().numpy() for x in res[0]] + [x.cpu().numpy() for x in res[1][1:]]
        _assert_exact(got, want, (name, jitter, "accumulate"))


@pytest.mark.parametrize("jitter", REFUSED)
def test_int32_years_refuse_inexact_jitters(device, jitter):
    """A jitter whose fl(year + jitter) is not year + jitter for every int32 year: the int32 pass would count every death with
    the wrong fraction (or in the wrong bin), so the C ABI refuses it and names death_jitter; the Python entries raise."""
    import torch
    ti = np.array([1990, 2000, 2010], np.int32); ei = np.array([1995, 2001, 2010], np.int32)
    sp = np.empty((1, 30), np.int64); ex = np.empty_like(sp); br = np.empty((1, 30))
    rc = device.lib.lr_bin_stats_host_i32(device.h, N.np_ptr(ti), N.np_ptr(ei), 3, 3, 1, 1990, 30, float(jitter), 0, 2011.0,
                                          N.np_ptr(sp), N.np_ptr(ex), N.np_ptr(br))
    assert rc != 0 and "death_jitter" in device.lib.lr_last_error().decode()
    dti, dei = torch.from_numpy(ti).cuda(), torch.from_numpy(ei).cuda()
    acc = device.new_accumulators(1, 30, dti.device)
    import ctypes as C
    rc = device.lib.lr_bin_accumulate_i32(device.h, C.c_void_p(dti.data_ptr()), C.c_void_p(dei.data_ptr()), 3, 3, 1, 1990, 30,
                                          float(jitter), 0, 2011.0, C.c_void_p(acc.data_ptr()), None)
    assert rc != 0 and "death_jitter" in device.lib.lr_last_error().decode()
    torch.cuda.synchronize()
    assert int(acc.abs().sum()) == 0
    with pytest.raises(ValueError, match="death_jitter"):
        device.bin_stats(ti, ei, death_jitter=jitter)
    with pytest.raises(ValueError, match="death_jitter"):
        device.bin_accumulate_device(dti, dei, 1990, 30, acc, death_jitter=jitter)


@pytest.mark.parametrize("jitter,int32_path", [(0.1, False), (1e-14, False), (0.5, True)])
def test_command_line_binning_of_jittered_tables(device, tmp_path, jitter, int32_path):
    """What forward does with -death_jitter J on the example TAD table: parse_lineages, as_year_table, Device.bin_stats.
    The statistics are the exact ones of the jittered table whichever path it takes; 0.1 and 1e-14 must stay float64 (the
    int32 pass would count every death with fraction J instead of fl(year + J) - year, and for 1e-14 put deaths in the wrong
    bin)."""
    path = golden_input("example_dataTAD.txt", tmp_path)
    with pytest.warns(FutureWarning):
        ts, te, start, end, _ = F.parse_lineages(path, death_jitter=jitter)
    years = F.as_year_table(ts, te, jitter)
    fb, nb = int(start), int(end) - int(start)
    st = device.bin_stats(*(years if years is not None else (ts, te)), first_bin=fb, n_bins=nb, death_jitter=jitter,
                          only_dead=True, end_time=float(end))
    want = K.exact_bin_stats(ts, te, fb, nb, only_dead=True, end_time=float(end))
    _assert_exact((st.sp[0], st.ex[0], st.br[0], st.ex_dead[0], st.br_dead[0]), want, jitter)
    assert (years is not None) == int32_path
