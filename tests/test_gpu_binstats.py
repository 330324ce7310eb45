"""GPU: K1 (lineages -> per-bin statistics) through the C ABI against the oracle.

Bar: counts bit-exact always; br bit-exact against the exact reference (oracle/k1_exact.py: the correctly rounded exact
sum the kernel promises) for any data -- equal to the oracle's own NumPy sums for dyadic data (all shipped data: integer
years + .5), within their rounding for real-valued times.  tests/test_gpu_binstats_exact.py runs every entry point and build.
"""
import numpy as np
import pytest

from conftest import golden_input
from oracle import k1_exact as K, literate_oracle as O
from literate_b200 import synth

pytestmark = pytest.mark.gpu


@pytest.fixture(params=["auto", "general", "lanes"])
def k1_build(request, monkeypatch):
    """The two builds of the real-valued path (k1_bin_kernel / k1_bin_lanes_kernel, LR_K1_LANES) and the automatic choice."""
    if request.param != "auto":
        monkeypatch.setenv("LR_K1_LANES", "1" if request.param == "lanes" else "0")
    else:
        monkeypatch.delenv("LR_K1_LANES", raising=False)
    return request.param


def _exact(ts, te, first_bin, n_bins, only_dead=False):
    return K.exact_bin_stats(ts, te, first_bin, n_bins, only_dead=only_dead, end_time=np.max(te))


def _check(dev, ts, te, jitter, only_dead=True):
    got = dev.bin_stats(ts, te, death_jitter=jitter, only_dead=only_dead)
    want = O.bin_stats(ts, te, only_dead=only_dead)
    assert got.first_bin == want.first_bin and got.n_bins == want.n_bins
    assert (got.sp[0] == want.sp).all() and (got.ex[0] == want.ex).all()
    if only_dead:
        assert (got.ex_dead[0] == want.ex_dead).all()
    exact = _exact(ts, te, want.first_bin, want.n_bins, only_dead)
    pairs = [(got.br[0], exact[2])] + ([(got.br_dead[0], exact[4])] if only_dead else [])
    for g, w in pairs:
        assert (g == w).all()


def test_example_tad_and_tbp(device):
    for name, tbp in (("example_dataTAD.txt", False), ("example_dataTBP.txt", True)):
        lin = O.read_lineages(golden_input(name), TBP=tbp)
        _check(device, lin.ts, lin.te, 0.5)
        lin0 = O.read_lineages(golden_input(name), TBP=tbp, death_jitter=0.0)
        _check(device, lin0.ts, lin0.te, 0.0)


def test_metal_bands(device, metal_path):
    lin = O.read_lineages(metal_path)
    _check(device, lin.ts, lin.te, 0.5)
    got = device.bin_stats(lin.ts, lin.te)
    assert got.sp.sum() == 27495 and got.ex.sum() == 16191 and got.br.sum() == 95426.5


def test_random_integer_and_real(device, k1_build):
    rng = np.random.default_rng(11)
    for n in (1, 2, 31, 257, 4097, 20011):
        ts, te = synth.syn_int(n, replicate=n)
        _check(device, ts, te, 0.5)
        ts, te = synth.syn_real(n, replicate=n)
        _check(device, ts, te, 0.0)
        # a wrong fe_ref hint must not change the result
        a = device.bin_stats(ts, te, fe_ref=0.5)
        b = device.bin_stats(ts, te, fe_ref=1.0)
        assert (a.br == b.br).all() and (a.sp == b.sp).all() and (a.ex == b.ex).all()
    # quarter-year data: fractional but dyadic -> still bit-exact
    n = 5000
    ts = 1900 + rng.integers(0, 160, n) / 4.0
    te = ts + rng.integers(0, 80, n) / 4.0
    te[0] = 1945.0
    _check(device, ts, te, 0.0)


def test_sorted_real_valued_tables_take_the_warp_merge(device, k1_build):
    """Tables sorted by birth (or death) time: the lanes of a warp hit one bin, the fractions are summed across the warp
    (MATCH.ALL + REDUX) before one carry chain.  The sums are integers: the result must be the SAME BITS as for the shuffled
    table, whatever mix of merged and per-lane updates a warp ends up doing (bin boundaries, half-sorted tables)."""
    rng = np.random.default_rng(17)
    n = 300_000
    ts, te = synth.syn_real(n, replicate=3)
    ref = device.bin_stats(ts, te, death_jitter=0.0)
    want = O.bin_stats_fast(ts, te)
    assert (ref.sp[0] == want.sp).all() and (ref.ex[0] == want.ex).all()
    assert (ref.br[0] == _exact(ts, te, want.first_bin, want.n_bins)[2]).all()
    orders = {"by birth": np.argsort(ts), "by death": np.argsort(te), "first half by birth": np.r_[np.argsort(ts[:n // 2]), n // 2 + rng.permutation(n - n // 2)],
              "runs of 40": np.argsort(np.floor(ts) * 1e6 + np.arange(n) // 40 % 7)}
    for name, o in orders.items():
        got = device.bin_stats(ts[o], te[o], death_jitter=0.0)
        assert (got.sp == ref.sp).all() and (got.ex == ref.ex).all() and (got.br == ref.br).all(), name
    # quarter-year data sorted by birth: fractional, dyadic -> bit-exact against the reference arithmetic
    ts = np.sort(1900 + rng.integers(0, 400, 50_000) / 4.0); te = ts + rng.integers(1, 200, 50_000) / 4.0
    _check(device, ts, te, 0.0)


def test_degenerate_inputs(device, k1_build):
    # all extant, single bin
    ts = np.array([10.0, 10.0, 10.0]); te = np.array([11.5, 11.5, 11.5])
    _check(device, ts, te, 0.5)
    # ts == te (zero time at risk), te < ts (malformed rows still count as events in the reference), NaN rows
    ts = np.array([5.0, 7.0, 9.0, 6.5, 8.0, 5.0, np.nan]); te = np.array([12.5, 7.0, 6.0, 6.5, np.nan, 5.5, 9.5])
    got = device.bin_stats(ts, te, first_bin=5, n_bins=7)
    with np.errstate(invalid="ignore"):
        for j in range(7):
            assert O.events_in_bin(ts, te, 5 + j, 6 + j) == (got.sp[0, j], got.ex[0, j], got.br[0, j]), j
    # sorted input: every lane of a warp hits the same bin
    ts = np.repeat(np.arange(1900.0, 1950.0), 300); te = ts + 3.5
    _check(device, ts, te, 0.5)
    # unsorted real values with many lineages born and dying in the same bin
    rng = np.random.default_rng(3)
    ts = 50 + rng.uniform(0, 20, 3000); te = ts + rng.uniform(0, 0.7, 3000); te[0] = 71.25
    _check(device, ts, te, 0.0)


def test_explicit_window_with_lineages_outside(device, k1_build):
    """first_bin / n_bins given by the caller (lineage-sharded use): lineages born before the window,
    dying after it, or entirely outside are clipped exactly as get_br clips them (:111-116)."""
    rng = np.random.default_rng(21)
    n = 4000
    ts = np.floor(rng.uniform(80, 140, n)); te = ts + np.floor(rng.exponential(10, n)) + 0.5
    first, nb = 100, 25
    got = device.bin_stats(ts, te, first_bin=first, n_bins=nb)
    for j in range(nb):
        a, b, c = O.events_in_bin(ts, te, first + j, first + j + 1)
        assert (got.sp[0, j], got.ex[0, j], got.br[0, j]) == (a, b, c)


def test_many_bins_and_single_bin(device, k1_build):
    """Window sizes at both ends: one bin, and 6000 one-year bins (216 KB of shared histograms, one CTA per SM)."""
    ts = np.array([3.0, 3.0, 3.25]); te = np.array([3.5, 4.5, 3.75])
    _check(device, ts, te, 0.5, only_dead=False)
    rng = np.random.default_rng(31)
    n = 50_000
    ts = np.floor(rng.uniform(0, 6000, n)); te = np.minimum(ts + np.floor(rng.exponential(40, n)), 6000) + 0.5
    ts[0], te[0] = 0.0, 6000.5
    got = device.bin_stats(ts, te)
    want = O.bin_stats_fast(ts, te)
    assert got.n_bins == 6000 and (got.sp[0] == want.sp).all() and (got.ex[0] == want.ex).all() and (got.br[0] == want.br).all()
    for j in (0, 1234, 5999):
        assert O.events_in_bin(ts, te, j, j + 1) == (got.sp[0, j], got.ex[0, j], got.br[0, j])


def test_too_many_bins_is_refused_with_a_message(device):
    from literate_b200.engine import NativeError
    ts = np.array([0.0, 10.0]); te = np.array([7000.5, 20.5])
    with pytest.raises(NativeError, match="n_bins <= "):
        device.bin_stats(ts, te)


def test_replicates_and_ragged_pitch(device, k1_build):
    import torch
    n_rep, n = 5, 3001      # odd n: rows are not 16-byte aligned -> scalar load path for odd replicates
    ts = np.empty((n_rep, n)); te = np.empty((n_rep, n))
    for r in range(n_rep):
        ts[r], te[r] = synth.syn_int(n, replicate=100 + r)
    got = device.bin_stats(ts, te)
    for r in range(n_rep):
        want = O.bin_stats_fast(ts[r], te[r])
        assert (got.sp[r] == want.sp).all() and (got.ex[r] == want.ex).all() and (got.br[r] == want.br).all()
    # device-pointer entry point with a padded row pitch
    dts = torch.zeros((n_rep, n + 5), dtype=torch.float64, device="cuda"); dte = torch.zeros_like(dts)
    dts[:, :n] = torch.from_numpy(ts).cuda(); dte[:, :n] = torch.from_numpy(te).cuda()
    sp, ex, br = device.bin_stats_device(dts[:, :n], dte[:, :n], got.first_bin, got.n_bins)
    torch.cuda.synchronize()
    assert (sp.cpu().numpy() == got.sp).all() and (ex.cpu().numpy() == got.ex).all() and (br.cpu().numpy() == got.br).all()


def test_full_size_one_million(device, k1_build):
    """BASELINE cfg3 size: 1M lineages x 200 bins against the O(N) oracle, plus size-independent checks."""
    n = 1_000_000
    ts, te = synth.syn_int(n)
    got = device.bin_stats(ts, te)
    want = O.bin_stats_fast(ts, te)
    assert got.n_bins == 200
    assert (got.sp[0] == want.sp).all() and (got.ex[0] == want.ex).all() and (got.br[0] == want.br).all()
    # conservation: every lineage is born once inside the window; total time at risk = sum of clipped lifetimes
    assert got.sp.sum() == n
    assert got.br.sum() == np.sum(np.minimum(te, 2000.0) - ts)
    # three spot-checked bins against the reference formulation itself
    for j in (0, 77, 199):
        assert O.events_in_bin(ts, te, 1800 + j, 1801 + j) == (got.sp[0, j], got.ex[0, j], got.br[0, j])
    # linearity: binning the two halves separately and adding gives the same integers
    h1 = device.bin_stats(ts[: n // 2], te[: n // 2], first_bin=1800, n_bins=200)
    h2 = device.bin_stats(ts[n // 2:], te[n // 2:], first_bin=1800, n_bins=200)
    assert ((h1.sp + h2.sp) == got.sp).all() and ((h1.ex + h2.ex) == got.ex).all() and ((h1.br + h2.br) == got.br).all()
    tr, er = synth.syn_real(n)
    got = device.bin_stats(tr, er, death_jitter=0.0)
    want = O.bin_stats_fast(tr, er)
    assert (got.sp[0] == want.sp).all() and (got.ex[0] == want.ex).all()
    assert (got.br[0] == _exact(tr, er, 1800, 200)[2]).all()
    again = device.bin_stats(tr, er, death_jitter=0.0)
    assert (again.br == got.br).all()          # run-to-run deterministic (integer accumulation)


def test_empty_table_through_the_c_abi(device):
    """n = 0: nothing is launched, the accumulators stay zero and finalise to empty bins; the host wrapper refuses it."""
    import torch
    acc = device.new_accumulators(1, 10, torch.device("cuda", 0))
    e = torch.empty((1, 0), dtype=torch.float64, device="cuda")
    device.bin_accumulate_device(e, e, 100, 10, acc)
    sp, ex, br = device.bin_finalize_device(acc, 10)
    torch.cuda.synchronize()
    assert int(sp.sum()) == 0 and int(ex.sum()) == 0 and float(br.sum()) == 0.0
    with pytest.raises(ValueError):
        device.bin_stats(np.empty(0), np.empty(0))


def test_full_size_hundred_million_lineages(device):
    """BASELINE cfg5 size on one GPU: 1e8 lineages (1.6 GB) generated on the device; size-independent checks
    (every lineage born once inside the window, total time at risk conserved exactly for half-integer data, the two
    halves add up to the whole, a second pass gives the same integers)."""
    import torch
    n = 100_000_000
    ts, te = synth.syn_int_device(n, 1, torch.device("cuda", 0))
    ts, te = ts[:, :n], te[:, :n]
    sp, ex, br = device.bin_stats_device(ts, te, 1800, 200)
    torch.cuda.synchronize()
    assert int(sp.sum()) == n
    want = (torch.minimum(te, torch.tensor(2000.0, device="cuda", dtype=torch.float64)) - ts).sum()
    assert float(br.sum()) == float(want)
    alive_at_end = int((te > 2000.0).sum())
    assert int(ex.sum()) == n - alive_at_end
    h = n // 2
    a = device.bin_stats_device(ts[:, :h], te[:, :h], 1800, 200)
    b = device.bin_stats_device(ts[:, h:], te[:, h:], 1800, 200)
    torch.cuda.synchronize()
    assert torch.equal(a[0] + b[0], sp) and torch.equal(a[1] + b[1], ex) and torch.equal(a[2] + b[2], br)
    sp2, ex2, br2 = device.bin_stats_device(ts, te, 1800, 200)
    torch.cuda.synchronize()
    assert torch.equal(sp2, sp) and torch.equal(br2, br)


def test_int32_year_tables_give_the_same_statistics(device, metal_path):
    """lr_bin_stats_host_i32 / lr_bin_accumulate_i32: integer years as int32 (8 bytes per lineage), the death jitter of
    LiteRateForward.py:471 added by the kernel.  Same statistics as the fp64 entry points on the jittered table, bit for
    bit: shipped tables, jitters that are multiples of 2^-22 in [0, 1] (0, 0.25, 0.5, 1: the int32 entry points refuse any other),
    extinct-only statistics, lineages outside / before the window, te < ts,
    ragged replicates padded with YEAR_PAD, row pitches that are not multiples of four, one lineage."""
    import torch
    from literate_b200 import engine as E
    rng = np.random.default_rng(5)
    for path in (golden_input("example_dataTAD.txt"), metal_path):
        for jitter in (0.5, 0.0, 1.0, 0.25):
            lin = O.read_lineages(path, death_jitter=jitter)
            ty, ey = lin.ts.astype(np.int32), (lin.te - jitter).astype(np.int32)
            assert (ty == lin.ts).all() and (ey + jitter == lin.te).all()
            a = device.bin_stats(lin.ts, lin.te, death_jitter=jitter, only_dead=True)
            b = device.bin_stats(ty, ey, death_jitter=jitter, only_dead=True)
            assert a.first_bin == b.first_bin and a.n_bins == b.n_bins
            for x, y in ((a.sp, b.sp), (a.ex, b.ex), (a.br, b.br), (a.ex_dead, b.ex_dead), (a.br_dead, b.br_dead)):
                assert np.array_equal(x, y), (path, jitter)
    # explicit window smaller than the data (births before / after the window, deaths beyond it), lineages with te < ts and te == ts
    for n in (1, 3, 5, 127, 128, 129, 1023, 20011):
        ty = rng.integers(1880, 2030, n).astype(np.int32)
        ey = (ty + rng.integers(-3, 40, n)).astype(np.int32)
        for jitter in (0.5, 0.0):
            a = device.bin_stats(ty.astype(np.float64), ey + jitter, first_bin=1900, n_bins=100, death_jitter=jitter, only_dead=True, end_time=2001.0)
            b = device.bin_stats(ty, ey, first_bin=1900, n_bins=100, death_jitter=jitter, only_dead=True, end_time=2001.0)
            for x, y in ((a.sp, b.sp), (a.ex, b.ex), (a.br, b.br), (a.ex_dead, b.ex_dead), (a.br_dead, b.br_dead)):
                assert np.array_equal(x, y), (n, jitter)
    # replicates of different lengths: NaN rows in the fp64 table, YEAR_PAD in the int32 one
    n_rep, n = 5, 3001
    T = np.full((n_rep, n), np.nan); Ee = np.full((n_rep, n), np.nan)
    Ti = np.full((n_rep, n), E.YEAR_PAD, dtype=np.int32); Ei = np.full((n_rep, n), E.YEAR_PAD, dtype=np.int32)
    for r in range(n_rep):
        m = n - 211 * r
        ts, te = synth.syn_int(m, replicate=40 + r)
        T[r, :m], Ee[r, :m] = ts, te
        Ti[r, :m], Ei[r, :m] = ts.astype(np.int32), (te - 0.5).astype(np.int32)
    a = device.bin_stats(T, Ee, first_bin=1800, n_bins=200, end_time=2000.5)
    b = device.bin_stats(Ti, Ei, first_bin=1800, n_bins=200, death_jitter=0.5, end_time=2000.5)
    assert np.array_equal(a.sp, b.sp) and np.array_equal(a.ex, b.ex) and np.array_equal(a.br, b.br)
    # device entry point, full bench size of one replicate, raw accumulators compared word for word
    tdev = torch.device("cuda:0")
    ts, te = synth.syn_int_device(1_000_000, 3, tdev)
    ts, te = ts[:, :1_000_000], te[:, :1_000_000]
    ti, ei = ts.to(torch.int32).contiguous(), (te - 0.5).to(torch.int32).contiguous()
    acc_a = device.new_accumulators(3, 200, tdev); acc_b = device.new_accumulators(3, 200, tdev)
    device.bin_accumulate_device(ts, te, 1800, 200, acc_a, fe_ref=0.5)
    device.bin_accumulate_device(ti, ei, 1800, 200, acc_b, death_jitter=0.5)
    torch.cuda.synchronize()
    assert bool((acc_a == acc_b).all())


def _same_accumulators(a, b):
    """Raw accumulator blocks of two passes over the same table: the counters word for word, the two fixed-point sums as the
    integers their (low 32 bits, rest) row pairs encode -- how a sum is split over the pair depends on where a pass flushed."""
    assert np.array_equal(a[:, [0, 1, 6, 7]], b[:, [0, 1, 6, 7]])
    for lo, hi in ((2, 3), (4, 5)):
        va = a[:, lo].astype(object) + a[:, hi].astype(object) * (1 << 32)
        vb = b[:, lo].astype(object) + b[:, hi].astype(object) * (1 << 32)
        assert (va == vb).all()


def test_lane_private_build_is_bit_identical_and_carries_into_the_third_word(device, monkeypatch):
    """k1_bin_lanes_kernel against k1_bin_kernel on tables that stress what is new in it: one bin that takes every lineage
    (each lane's high word overflows after 4096 additions of fractions near 1 -> the shared third word), extant-heavy tables
    (deaths outside the window go to the spare bin), only_dead, negative times, an odd number of bins, several replicates."""
    import torch
    rng = np.random.default_rng(5)
    n = 600_000
    cases = {
        "one bin, fractions near 1": (10 + 1 - rng.uniform(0, 1e-3, n), 10 + 1 - rng.uniform(0, 1e-6, n) + 0.0),
        "mostly extant": (1900 + rng.uniform(0, 101, n), np.where(rng.uniform(size=n) < 0.9, 2001.0, 1900 + rng.uniform(0, 101, n))),
        "negative times": (-60 + rng.uniform(0, 37, n), -60 + rng.uniform(0, 37, n) + rng.exponential(5, n)),
    }
    ts, te = cases["one bin, fractions near 1"]
    cases["one bin, fractions near 1"] = (np.minimum(ts, te - 1e-9), te)
    ts, te = cases["mostly extant"]
    cases["mostly extant"] = (np.minimum(ts, te), np.maximum(ts, te))
    for name, (ts, te) in cases.items():
        res = {}
        for build in ("0", "1"):
            monkeypatch.setenv("LR_K1_LANES", build)
            for dead in (False, True):
                kw = dict(first_bin=10, n_bins=1, end_time=11.5) if name.startswith("one bin") else {}
                res[build, dead] = device.bin_stats(ts, te, death_jitter=0.0, only_dead=dead, **kw)
        for dead in (False, True):
            a, b = res["0", dead], res["1", dead]
            assert a.n_bins == b.n_bins and (a.sp == b.sp).all() and (a.ex == b.ex).all() and (a.br == b.br).all(), (name, dead)
            if dead:
                assert (a.ex_dead == b.ex_dead).all() and (a.br_dead == b.br_dead).all(), name
        got = res["1", False]
        if name.startswith("one bin"):
            assert got.sp[0, 0] == n and got.ex[0, 0] == n
            assert got.br[0, 0] == _exact(ts, te, 10, 1)[2][0]
            continue
        want = O.bin_stats_fast(ts, te)
        assert (got.sp[0] == want.sp).all() and (got.ex[0] == want.ex).all(), name
        assert (got.br[0] == _exact(ts, te, want.first_bin, want.n_bins)[2]).all(), name
    # replicates with a ragged pitch, device entry point, raw accumulators
    tdev = torch.device("cuda:0")
    n_rep, n, ld, nb = 5, 70_001, 70_004, 37
    t = torch.full((n_rep, ld), float("nan"), dtype=torch.float64, device=tdev)
    e = torch.full((n_rep, ld), float("nan"), dtype=torch.float64, device=tdev)
    t[:, :n] = torch.from_numpy(100 + rng.uniform(0, nb, (n_rep, n))).to(tdev)
    e[:, :n] = t[:, :n] + torch.from_numpy(rng.exponential(6, (n_rep, n))).to(tdev)
    accs = []
    for build in ("0", "1"):
        monkeypatch.setenv("LR_K1_LANES", build)
        acc = device.new_accumulators(n_rep, nb, tdev)
        device.bin_accumulate_device(t[:, :n], e[:, :n], 100, nb, acc, fe_ref=1.0)
        torch.cuda.synchronize()
        accs.append(acc.cpu().numpy().copy())
    _same_accumulators(accs[0], accs[1])
    # the widest window the lane-private build fits (439 bins), and one bin more (general build either way)
    for nb in (439, 440):
        n = 150_000
        ts = 1000 + rng.uniform(0, nb, n); te = np.minimum(ts + rng.exponential(30, n), 1000.0 + nb)
        res = []
        for build in ("0", "1"):
            monkeypatch.setenv("LR_K1_LANES", build)
            res.append(device.bin_stats(ts, te, death_jitter=0.0, first_bin=1000, n_bins=nb))
        assert (res[0].sp == res[1].sp).all() and (res[0].ex == res[1].ex).all() and (res[0].br == res[1].br).all(), nb
        want = O.bin_stats_fast(ts, te)
        assert (res[1].sp[0] == want.sp[:nb]).all() and (res[1].ex[0] == want.ex[:nb]).all(), nb
    # 48 M lineages in ONE bin with fractions near 1: every lane's high word wraps (5 000 additions of ~2^20 per CTA and lane)
    n = 48_000_000
    g = torch.Generator(device=tdev); g.manual_seed(9)
    e = 11.0 - torch.rand(n, dtype=torch.float64, device=tdev, generator=g) * 1e-6
    t = e - 1e-9 - torch.rand(n, dtype=torch.float64, device=tdev, generator=g) * 1e-3
    accs = []
    for build in ("0", "1"):
        monkeypatch.setenv("LR_K1_LANES", build)
        acc = device.new_accumulators(1, 3, tdev)
        device.bin_accumulate_device(t, e, 9, 3, acc, fe_ref=1.0)
        torch.cuda.synchronize()
        accs.append(acc.cpu().numpy().copy())
    _same_accumulators(accs[0], accs[1])
    assert accs[0][0, 0, 1] == n and accs[0][0, 1, 1] == n
    sp, ex, br = device.bin_finalize_device(torch.from_numpy(accs[1]).to(tdev), 3, fe_ref=1.0)
    # every lineage lies in [10, 11]: the exact time at risk is sum((te - 10) * 2^52 - (ts - 10) * 2^52), integers below 2^52
    from fractions import Fraction
    d = ((e - 10.0) * 2.0 ** 52).to(torch.int64) - ((t - 10.0) * 2.0 ** 52).to(torch.int64)
    want = float(Fraction(int((d & ((1 << 26) - 1)).sum()) + (int((d >> 26).sum()) << 26), 1 << 52))
    assert float(br[0, 1]) == want and float(br[0, 0]) == 0.0 and float(br[0, 2]) == 0.0


def test_choice_of_build(device, monkeypatch):
    """lr_bin_accumulate (device tables): the lane-private build for every table of >= 250 000 lineages up to 310 bins, for real-valued
    tables of >= 50 000 up to 439 (the previous pass tells the kind), the general build otherwise; the host-buffer entry points always
    run the general build."""
    import torch
    monkeypatch.delenv("LR_K1_LANES", raising=False)
    tdev = torch.device("cuda:0")
    rng = np.random.default_rng(2)
    for nb, real, n, want in ((200, False, 260_000, "k1_bin_lanes_kernel"), (200, False, 100_000, "k1_bin_kernel"), (310, True, 260_000, "k1_bin_lanes_kernel"),
                              (311, False, 260_000, "k1_bin_kernel"), (311, True, 60_000, "k1_bin_lanes_kernel"), (200, True, 40_000, "k1_bin_kernel"),
                              (439, True, 60_000, "k1_bin_lanes_kernel"), (440, True, 60_000, "k1_bin_kernel")):
        ts = np.floor(rng.uniform(0, nb, n)); te = ts + np.floor(rng.exponential(10, n)) + 0.5
        if real:
            ts = ts + rng.uniform(0, 1, n); te = ts + rng.exponential(10, n)
        t, e = torch.from_numpy(ts).to(tdev), torch.from_numpy(te).to(tdev)
        for _ in range(2):                                   # the first pass records the kind of table, the second uses it
            got = device.bin_stats_device(t, e, 0, nb, fe_ref=0.5)
            torch.cuda.synchronize()
        assert device.bin_last_build() == want, (nb, real, n)
        wantst = O.bin_stats_fast(ts, te)
        assert (got[0][0].cpu().numpy() == wantst.sp[:nb]).all(), (nb, real)
    device.bin_stats(ts, te, death_jitter=0.0)               # host entry
    assert device.bin_last_build() == "k1_bin_kernel"


def test_the_pass_remembers_the_kind_of_table(device, monkeypatch):
    """lr_bin_table_hint: 1 after a table with fractional times, 0 after integer years -- what the next pass chooses its build by."""
    monkeypatch.delenv("LR_K1_LANES", raising=False)
    ts, te = synth.syn_real(50_000, replicate=1)
    for _ in range(2):                     # the second pass runs the lane-private build, which records the kind as well
        device.bin_stats(ts, te, death_jitter=0.0)
        device.sync()
        assert device.bin_table_hint() == 1
    ts, te = synth.syn_int(50_000, replicate=1)
    for _ in range(2):
        device.bin_stats(ts, te, death_jitter=0.5)
        device.sync()
        assert device.bin_table_hint() == 0
