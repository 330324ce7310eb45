"""GPU: K7 (DDRate chains, SURVEY 8 f-4) through the C ABI against the oracle pinned to the unmodified DDRatev3.py.

Deterministic parity (1e-10 relative, the north star's tolerance): the three likelihood terms, prior, per-bin rates / niche
/ niche fraction, genre-window statistics (exact counts), the multiplier move and both sliding-window moves with explicit
draws, for every (m_birth, m_death) the functions of the reference define.  Chain-level parity is distributional: 64 device
chains against the committed summaries of 8 unmodified reference chains (-m_birth 3, the configuration that runs as shipped).
"""
import json
import os

import numpy as np
import pytest

from oracle import ddrate_oracle as D
from literate_b200 import ddrate as DD
from literate_b200 import library as L
from test_oracle_ddrate_golden import DG, _jobs, stage

pytestmark = pytest.mark.gpu
RTOL = 1e-10


def _job(tag):
    return [j for j in _jobs() if j["tag"] == tag][0]


def _setup(device, tmp_path, tag="ex_g_mddn", mb=3, md=2, n_chains=8, seed=1, rm=0):
    job = _job(tag)
    data, genre = stage(job, tmp_path)
    ts, te, present, origin = L.parse_ts_te(data)
    first, nb = L.bin_window(origin, present, rm)
    st = device.bin_stats(ts, te, first_bin=first, n_bins=nb)
    gts, gte, _, _ = L.parse_ts_te(genre)
    bins = D.create_bins(origin, present, ts, te, rm)
    assert np.array_equal(st.sp[0], bins.n_spec) and np.array_equal(st.ex[0], bins.n_exti) and np.array_equal(st.br[0], bins.dt)
    S = D.Setup(bins, mb, md, gts, gte)
    ch = DD.DDChains(device, st.sp[0], st.ex[0], st.br[0], bins.origin, present, mb, md, gts if mb == 3 else None,
                     gte if mb == 3 else None, n_chains, seed)
    return S, ch


def _random_params(rng, n, S):
    span = S.present - S.origin
    return np.stack([rng.gamma(2, .2, n), rng.gamma(2, .5, n), rng.gamma(2, .5, n), rng.uniform(0, span * .98, n), rng.gamma(2, 5, n),
                     rng.gamma(2, 30, n), rng.uniform(0, 1, n), rng.gamma(3, .5, n), rng.gamma(3, .5, n), rng.gamma(2, .5, n),
                     rng.gamma(2, .5, n)], axis=1)


@pytest.mark.parametrize("mb,md", [(3, 2), (3, 1), (3, 0), (2, 2), (2, 1), (1, 2), (1, 1), (0, 0), (0, 2), (1, 0)])
def test_state_evaluation_matches_the_oracle(device, tmp_path, mb, md):
    S, ch = _setup(device, tmp_path, mb=mb, md=md)
    rng = np.random.default_rng(100 + 10 * mb + md)
    P = _random_params(rng, 120, S)
    P[0] = D.initial_args(S)
    P[1, 6] = 1.7                  # m_mul > 1: death rates floored at SMALL_NUMBER where they turn negative (:79)
    out = ch.evaluate(P)
    emp_b, emp_d = S.bins.n_spec / S.bins.dt, S.bins.n_exti / S.bins.dt
    for i, p in enumerate(P):
        lk, birth, death, niche, nf = D.likelihood(p, S)
        np.testing.assert_allclose(out["lik"][i], lk, rtol=RTOL)
        want = D.prior(p, S, exact_scipy=True)
        assert out["prior"][i] == (pytest.approx(want, rel=RTOL) if np.isfinite(want) else want)
        np.testing.assert_allclose(out["series"][i], [birth, death, niche, nf], rtol=RTOL)
        np.testing.assert_allclose(out["adequacy"][i], D.adequacy(emp_b, emp_d, birth, death), rtol=1e-8)
        if mb == 3:
            assert tuple(out["genre"][i]) == pytest.approx(D.genre_stats(S, p[3]), rel=1e-13)
            assert out["genre"][i][0] == D.genre_stats(S, p[3])[0] and out["genre"][i][2] == D.genre_stats(S, p[3])[2]   # counts exact
    bad = np.tile(D.initial_args(S), (5, 1))
    bad[0, 0] = -.1; bad[1, 3] = S.present - S.origin; bad[2, 6] = 1.0; bad[3, 7] = 0.0; bad[4, 5] = -1.0
    assert np.all(np.isneginf(ch.evaluate(bad)["prior"]))


def test_first_bin_removed_and_metal_bands(device, tmp_path):
    """-rm_first_bin moves the origin (create_bins, literate_library.py:247-252): midpoint prior, initial x0 and the genre
    windows follow; the metal-band table has 32 bins (one per lane) and counts in the thousands."""
    for tag, rm in (("ex_g_rmfirst", 1), ("metal_g_mddn", 0)):
        S, ch = _setup(device, tmp_path, tag, rm=rm, n_chains=4)
        assert np.array_equal(ch.state()[0, :11], D.initial_args(S))
        rng = np.random.default_rng(77)
        P = _random_params(rng, 40, S)
        out = ch.evaluate(P)
        for i, p in enumerate(P):
            lk, birth, death, niche, nf = D.likelihood(p, S)
            np.testing.assert_allclose(out["lik"][i], lk, rtol=RTOL)
            want = D.prior(p, S, exact_scipy=True)
            assert out["prior"][i] == (pytest.approx(want, rel=RTOL) if np.isfinite(want) else want)
            assert tuple(out["genre"][i]) == pytest.approx(D.genre_stats(S, p[3]), rel=1e-13)
        r = ch.run(3001, 1000)[-1, 0]
        lk, _, _, _, _ = D.likelihood(r[5:16], S)
        np.testing.assert_allclose([r[2], r[3], r[16]], lk, rtol=RTOL)


@pytest.mark.parametrize("nb,mb,md", [(200, 3, 2), (200, 1, 1), (33, 2, 2), (1, 2, 2), (5, 3, 0)])
def test_bin_counts_from_one_to_two_hundred(device, nb, mb, md):
    """n_bins > 32: every lane owns several bins (the first 32 go through the cached logarithms, the rest through dd_bin);
    n_bins = 1: a single lane carries the whole likelihood."""
    rng = np.random.default_rng(1000 + nb + mb)
    t = np.arange(nb)
    br = 20 + 400 / (1 + np.exp(-0.3 * (t - nb / 2))) + rng.uniform(0, 5, nb)
    sp = rng.poisson(br * 0.2); ex = rng.poisson(br * 0.1)
    gts = np.sort(rng.uniform(0, nb * .7, 40)).round(); gte = np.minimum(gts + rng.integers(1, nb + 1, 40), nb) + .5
    bins = D.Bins(0.0, nb + 1.5, sp, ex, br)
    S = D.Setup(bins, mb, md, gts, gte)
    ch = DD.DDChains(device, sp, ex, br, 0.0, nb + 1.5, mb, md, gts if mb == 3 else None, gte if mb == 3 else None, 6, 3)
    P = _random_params(rng, 40, S)
    out = ch.evaluate(P)
    for i, p in enumerate(P):
        lk, birth, death, niche, nf = D.likelihood(p, S)
        np.testing.assert_allclose(out["lik"][i], lk, rtol=RTOL)
        np.testing.assert_allclose(out["series"][i], [birth, death, niche, nf], rtol=RTOL)
    recs = ch.run(6001, 1000)
    assert recs.shape == (7, 6, 24 + 4 * nb)
    for r in recs[1:, ::2].reshape(-1, recs.shape[-1]):
        lk, birth, death, niche, nf = D.likelihood(r[5:16], S)
        np.testing.assert_allclose([r[2], r[3], r[16]], lk, rtol=RTOL)
        np.testing.assert_allclose(r[24:].reshape(4, nb), [birth, death, niche, nf], rtol=RTOL)
        assert r[4] == pytest.approx(D.prior(r[5:16], S, exact_scipy=True), rel=RTOL)


@pytest.mark.parametrize("nb,mb,md", [(65, 3, 2), (100, 2, 1), (129, 1, 2), (200, 3, 2), (200, 0, 0), (300, 3, 1)])
def test_wide_build_gives_the_chains_of_the_one_warp_build(device, nb, mb, md, monkeypatch):
    """More than 64 bins and few chains: 2 or 4 warps share a chain's bins (k7_dd_kernel<2> and <4>), exchange the per-bin terms and add
    them in the one-warp kernel's order -- records and final states identical, bit for bit, over split launches."""
    rng = np.random.default_rng(77 + nb + mb)
    t = np.arange(nb)
    br = 20 + 400 / (1 + np.exp(-0.3 * (t - nb / 2))) + rng.uniform(0, 5, nb)
    sp = rng.poisson(br * 0.2); ex = rng.poisson(br * 0.1)
    gts = np.sort(rng.uniform(0, nb * .7, 40)).round(); gte = np.minimum(gts + rng.integers(1, nb + 1, 40), nb) + .5
    out = []
    for wide in ("0", "1"):
        monkeypatch.setenv("LR_DD_WIDE", wide)
        ch = DD.DDChains(device, sp, ex, br, 0.0, nb + 1.5, mb, md, gts if mb == 3 else None, gte if mb == 3 else None, 7, 5)
        recs = [ch.run(n, s) for n, s in ((1501, 100), (1, 1), (998, 7), (3000, 250))]
        out.append((np.concatenate(recs), ch.state()))
    assert np.array_equal(out[0][0], out[1][0]) and np.array_equal(out[0][1], out[1][1])


def test_proposals_with_explicit_draws_match_the_oracle(device, tmp_path):
    S, ch = _setup(device, tmp_path)
    rng = np.random.default_rng(12)
    n = 300
    P = _random_params(rng, n, S)
    kind = rng.integers(0, 3, n).astype(np.int32)
    on = (rng.uniform(size=(n, 11)) < .4).astype(np.int32)
    draw = rng.uniform(size=(n, 11))
    P[:20, 6] = rng.uniform(0, .02, 20); P[20:40, 6] = rng.uniform(.98, 1, 20)     # m_mul near both reflecting ends
    P[40:50, 3] = rng.uniform(0, .7, 10)                                             # x0 near 0: the abs() branch
    out = ch.evaluate(P, kind=kind, on=on, draw=draw)
    for i in range(n):
        q, h = P[i].copy(), 0.0
        if kind[i] == 0:
            q, h = D.multiplier_given(P[i], on[i], draw[i])
        elif kind[i] == 1:
            q[3] = D.sliding_window_given(q[3], draw[i, 3], S.present, 1.5)
        else:
            q[6] = D.sliding_window_given(q[6], draw[i, 6], 1, .05)
        np.testing.assert_allclose(out["params"][i], q, rtol=1e-13)
        assert out["hastings"][i] == pytest.approx(h, rel=1e-11, abs=1e-15)
        lk, _, _, _, _ = D.likelihood(q, S)
        np.testing.assert_allclose(out["lik"][i], lk, rtol=RTOL)
        want = D.prior(q, S, exact_scipy=True)
        assert out["prior"][i] == (pytest.approx(want, rel=RTOL) if np.isfinite(want) else want)


@pytest.mark.parametrize("mb,md", [(3, 2), (2, 1), (1, 0)])
def test_chain_bookkeeping(device, tmp_path, mb, md):
    """Initial state, forced acceptance of iteration 0, stored terms = terms of the stored parameters (the cached sides and
    the cached genre statistics), records on the sampling grid."""
    S, ch = _setup(device, tmp_path, mb=mb, md=md, n_chains=16, seed=3)
    s0 = ch.state()
    init = D.initial_args(S)
    lk, _, _, _, _ = D.likelihood(init, S)
    for s in s0:
        assert np.array_equal(s[:11], init) and s[15] == 0
        np.testing.assert_allclose(s[11:14], lk, rtol=RTOL)
        assert s[14] == pytest.approx(D.prior(init, S, exact_scipy=True), rel=RTOL)
    recs = ch.run(20001, 500)
    nb = S.n
    assert recs.shape == (41, 16, 24 + 4 * nb) and np.all(recs[0, :, 20] == 1)
    emp_b, emp_d = S.bins.n_spec / S.bins.dt, S.bins.n_exti / S.bins.dt
    for si in range(0, 41, 4):
        for c in (0, 7, 15):
            r = recs[si, c]
            assert r[0] == si * 500
            p = r[5:16]
            lk, birth, death, niche, nf = D.likelihood(p, S)
            np.testing.assert_allclose([r[2], r[3], r[16]], lk, rtol=RTOL)
            assert r[1] == pytest.approx(r[2] + r[3] + r[16], rel=1e-15)
            assert r[4] == pytest.approx(D.prior(p, S, exact_scipy=True), rel=RTOL)
            np.testing.assert_allclose(r[24:].reshape(4, nb), [birth, death, niche, nf], rtol=RTOL)
            np.testing.assert_allclose(r[17:20], D.adequacy(emp_b, emp_d, birth, death), rtol=1e-8)
    fin = ch.state()
    assert np.all(fin[:, 15] == 20001) and np.all(fin[:, 16] == recs[-1, :, 20])
    if mb == 3:
        for s in fin[:4]:
            assert tuple(s[17:21]) == pytest.approx(D.genre_stats(S, s[3]), rel=1e-13)
    assert 0.05 < fin[:, 16].mean() / 20001 < 0.95


def test_determinism_split_runs_and_sharding(device, tmp_path):
    S, a = _setup(device, tmp_path, n_chains=32, seed=11)
    ra = a.run(3000, 100)
    mk = lambda n, seed, c0=0: DD.DDChains(device, S.bins.n_spec, S.bins.n_exti, S.bins.dt, S.origin, S.present, 3, 2, S.gts, S.gte,
                                           n, seed, chain_id0=c0)
    b = mk(32, 11)
    rb = np.concatenate([b.run(1000, 100), b.run(1501, 100), b.run(499, 100)])
    assert np.array_equal(ra, rb) and np.array_equal(a.state(), b.state())
    assert np.array_equal(mk(8, 11, 16).run(3000, 100), ra[:, 16:24])
    assert not np.array_equal(mk(32, 12).run(3000, 100), ra)
    assert np.array_equal(mk(2048, 11).run(3000, 100)[:, :32], ra)


def test_unsupported_models_are_refused(device, tmp_path):
    from literate_b200._native import NativeError
    with pytest.raises(NativeError, match="NameError"):
        _setup(device, tmp_path, mb=2, md=-1)


@pytest.mark.parametrize("tag,md", [("ex_g_mddn", 2), ("ex_g_mdd", 1)])
def test_posterior_matches_reference_chains(device, tmp_path, tag, md):
    """128 device chains against 32 unmodified reference chains of the same length: every posterior mean within 3.5 standard
    errors of the difference of the two population means (between-chain variance of both sides); 64 against 8 within 4.5 while
    a fixture still holds the 8 chains of round 1."""
    with open(os.path.join(DG, "posterior", tag + ".json")) as fh:
        ref = json.load(fh)
    strong = len(ref["chains"]) >= 32
    z_max = 3.5 if strong else 4.5
    S, ch = _setup(device, tmp_path, "ex_g_mddn", mb=3, md=md, n_chains=128 if strong else 64, seed=2027)
    recs = ch.run(ref["n_iter"], ref["sample_every"])
    r = recs[int(ref["burnin"] * recs.shape[0]):]
    nb = S.n
    cols = {"likelihood": r[:, :, 1], "likelihood_birth": r[:, :, 2], "likelihood_death": r[:, :, 3], "prior": r[:, :, 4],
            "l_f": r[:, :, 5], "l_mul": r[:, :, 6], "k": r[:, :, 7], "x0_abs": r[:, :, 8] + S.origin, "div_0": r[:, :, 9],
            "K_max": r[:, :, 10] + r[:, :, 9], "m_mul": r[:, :, 11], "nuB": r[:, :, 12], "nuD": r[:, :, 13], "g_l1": r[:, :, 14],
            "g_l2": r[:, :, 15], "likelihood_genre": r[:, :, 16]}
    mine = {k + "_mean": v.mean(0) for k, v in cols.items()}
    for i, k in enumerate(["birth_rate", "death_rate", "niche", "niche_frac"]):
        mine[k + "_mean"] = r[:, :, 24 + i * nb:24 + (i + 1) * nb].mean(0)
    for key, a in mine.items():
        b = np.array([c[key] for c in ref["chains"]], dtype=float)
        a = np.asarray(a, dtype=float)
        se = np.sqrt(a.var(0, ddof=1) / len(a) + b.var(0, ddof=1) / len(b))
        z = np.abs(a.mean(0) - b.mean(0)) / se
        assert np.all(z < z_max), (key, float(np.max(z)), a.mean(0), b.mean(0))


def test_command_line_end_to_end(device, tmp_path):
    job = _job("ex_g_mddn")
    data, genre = stage(job, tmp_path)
    paths = DD.run(DD.build_parser().parse_args(["-d", data, "-m_birth", "3", "-g", genre, "-n", "3001", "-s", "50", "-seed", "1",
                                                 "-chains", "2", "-quiet", "1"]), device=device)
    assert [os.path.basename(p) for p in paths] == ["example3_%d_GLDDN_MDDN.log" % s for s in (1, 2)]
    files = {f: open(os.path.join(DG, "ex_g_mddn", f), "rb").read() for f in job["files"]}
    want = files["example3_1_GLDDN_MDDN.log"].split(b"\r\n")
    for p in paths:
        got = open(p, "rb").read().split(b"\r\n")
        assert got[0] == want[0] and len(got) == len(want)
        rows = np.array([l.split(b"\t") for l in got[1:-1]], dtype=float)
        assert rows.shape[1] == len(want[1].split(b"\t")) and np.array_equal(rows[:, 0], np.arange(0, 3001, 50))
        assert open(p[:-4] + ".div.log", "rb").read() == files["example3_1_GLDDN_MDDN.div.log"]      # statistics: byte-identical
    # a model the reference cannot start (NameError at :48) but whose functions are defined
    paths = DD.run(DD.build_parser().parse_args(["-d", data, "-m_birth", "2", "-m_death", "1", "-n", "501", "-s", "100", "-seed", "4",
                                                 "-quiet", "1"]), device=device)
    assert os.path.basename(paths[0]) == "example3_4_LDDN_MDD.log"
    assert len(open(paths[0]).read().splitlines()) == 7


def test_replicates_and_directory_of_imputations(device, tmp_path):
    """Replicate axis of K7 (PRIOR_K0_L = the replicate's own max br) and -d <directory> of the command line."""
    rng = np.random.default_rng(21)
    nb, n_rep = 40, 3
    t = np.arange(nb)
    br = np.stack([20 + (300 + 60 * r) / (1 + np.exp(-0.3 * (t - nb / 2))) + rng.uniform(0, 5, nb) for r in range(n_rep)])
    sp = rng.poisson(br * 0.2); ex = rng.poisson(br * 0.1)
    rep_of_chain = np.arange(9) % n_rep
    ch = DD.DDChains(device, sp, ex, br, 0.0, nb + 1.5, 2, 2, None, None, 9, 4, rep_of_chain=rep_of_chain)
    setups = [D.Setup(D.Bins(0.0, nb + 1.5, sp[r], ex[r], br[r]), 2, 2) for r in range(n_rep)]
    P = _random_params(rng, 30, setups[0])
    rep = rng.integers(0, n_rep, 30)
    out = ch.evaluate(P, rep=rep)
    for i, p in enumerate(P):
        lk, birth, death, niche, nf = D.likelihood(p, setups[rep[i]])
        np.testing.assert_allclose(out["lik"][i], lk, rtol=RTOL)
        assert out["prior"][i] == pytest.approx(D.prior(p, setups[rep[i]], exact_scipy=True), rel=RTOL)
    recs = ch.run(3001, 1000)
    for c in range(9):
        r = recs[-1, c]
        S = setups[rep_of_chain[c]]
        lk, _, _, _, _ = D.likelihood(r[5:16], S)
        np.testing.assert_allclose([r[2], r[3], r[16]], lk, rtol=RTOL)
        assert r[4] == pytest.approx(D.prior(r[5:16], S, exact_scipy=True), rel=RTOL)
    assert np.array_equal(ch.state()[:, 21], rep_of_chain)
    # the command line on a directory: two imputations of the example table
    job = _job("ex_g_mddn")
    data, genre = stage(job, tmp_path)
    rows = [l.split("\t") for l in open(data).read().splitlines()[1:]]
    d = os.path.join(str(tmp_path), "imputations")
    os.makedirs(d)
    for i in range(2):
        with open(os.path.join(d, "imp_%d.tsv" % i), "w") as fh:
            fh.write("id\tts\tte\n")
            for r in rows:
                ts_, te_ = int(r[1]), int(r[2])
                if i and 1996 < ts_ < 2010 and te_ - ts_ > 2 and rng.uniform() < .3:
                    ts_ += 1
                fh.write("%s\t%d\t%d\n" % (r[0], ts_, te_))
    paths = DD.run(DD.build_parser().parse_args(["-d", d, "-m_birth", "3", "-g", genre, "-n", "1001", "-s", "500", "-seed", "3", "-chains", "4",
                                                 "-quiet", "1"]), device=device)
    assert [os.path.basename(p) for p in paths] == ["imp_%d_%d_GLDDN_MDDN.log" % (k % 2, 3 + k // 2) for k in range(4)]
    gts, gte, _, _ = L.parse_ts_te(genre)
    for k, p in enumerate(paths):
        ts, te, present, origin = L.parse_ts_te(os.path.join(d, "imp_%d.tsv" % (k % 2)))
        S = D.Setup(D.create_bins(origin, present, ts, te), 3, 2, gts, gte)
        got = np.loadtxt(p, skiprows=1)
        assert got.shape[0] == 3
        for row in got:
            args = row[6:17].copy(); args[3] -= S.origin; args[5] -= args[4]
            lk, _, _, _, _ = D.likelihood(args, S)
            np.testing.assert_allclose([row[3], row[4], row[17]], lk, rtol=1e-9)
