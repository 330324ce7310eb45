"""GPU: the shared sampler arithmetic of lr_common.cuh, on the device, against exact or high-precision references.

Every chain of K3 (RJMCMC), K6 (TrendRate) and K7 (DDRate) takes its random numbers and accept decisions from these helpers, and
K8-K10 their compensated sums and sort keys.  The chain tests compare builds with each other (which share the helpers) or
posteriors within the between-chain spread (which a half-step bias in a uniform hides), so the helpers are held here one by one,
through tests/device_math_harness.cu (one kernel per helper, applied elementwise):

* philox4x32_10: Random123's known-answer vectors, and 2^20 random (counter, key) tuples against the uint64 restatement;
* u01: exactly (k + 1/2) 2^-52, strictly inside (0, 1);
* exp_small: bit for bit the exact emulation of its fma Horner scheme, and within 1 ulp of exp (mpmath, 200 bits) over the
  log-multiplier window of K3, K6 and K7 and over +-0.1;
* mh_bracket with mh_accept_gt (K6, K7) and mh_accept_ge (K3): the decision of the plain double comparison with the device's
  own log(u), in every binade of u01, at log(u) and its neighbours, at the bracket's edges, at NaN and +-inf;
* normal_f32: within the error bound that follows from the documented bounds of __logf, sqrtf and cospif and the float rounding
  of its arguments, against mpmath; and over all 2^24 angle codes its values are symmetric about 0;
* lr_sum: within 2 ulp of the correctly rounded sum (math.fsum), infinities and NaN as a plain sum gives them, repeatable;
* lr_key / lr_val: an order-preserving bijection, -0.0 before +0.0, NaN last;
* warp_sum_first(v, K): the bits of warp_sum(v) when lanes >= K hold zeros.
Everything that needs many draws runs in one launch.
"""
import ctypes
import math
from fractions import Fraction

import mpmath
import numpy as np
import pytest

import _device_math as D

pytestmark = pytest.mark.gpu

C_P, C_LL, C_I, C_D = ctypes.c_void_p, ctypes.c_longlong, ctypes.c_int, ctypes.c_double
SIGNATURES = {
    "t_philox": [C_P, C_P, C_LL], "t_u01": [C_P, C_P, C_LL], "t_exp_small": [C_P, C_P, C_LL], "t_bracket": [C_P, C_P, C_LL],
    "t_accept": [C_P, C_P, C_P, C_P, C_P, C_LL], "t_normal": [C_P, C_P, C_P, C_LL], "t_normal_angles": [C_D, C_P],
    "t_lr_sum": [C_P, C_P, C_P, C_I], "t_key": [C_P, C_P, C_P, C_LL], "t_warp_sum": [C_P, C_P, C_P, C_I],
}


@pytest.fixture(scope="module")
def H(tmp_path_factory):
    import torch
    lib = ctypes.CDLL(D.compile_harness(tmp_path_factory.mktemp("device_math")))
    for name, args in SIGNATURES.items():
        getattr(lib, name).argtypes = args
        getattr(lib, name).restype = C_I
    torch.cuda.init()
    return lib


def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _empty(n, dtype):
    import torch
    return torch.empty(n, dtype=dtype, device="cuda")


def _run(fn, *args):
    """One launch of a harness kernel (tensors as device pointers), waited for."""
    import torch
    rc = fn(*[C_P(a.data_ptr()) if isinstance(a, torch.Tensor) else a for a in args])
    assert rc == 0, "launch failed: cudaError %d" % rc
    torch.cuda.synchronize()


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint64)


# ---- Philox-4x32-10 ----------------------------------------------------------------------------------------------------------
def _philox_dev(H, tuples):
    import torch
    t = np.asarray(tuples, np.uint64).astype(np.uint32).view(np.int32)
    out = _empty(4 * len(t), torch.int32)
    _run(H.t_philox, _dev(t), out, len(t))
    return out.cpu().numpy().view(np.uint32).reshape(-1, 4)


def test_philox_known_answers(H):
    got = _philox_dev(H, [c + k for c, k, _ in D.PHILOX_KAT])
    assert [tuple(int(v) for v in r) for r in got] == [want for _, _, want in D.PHILOX_KAT]


def test_philox_random_tuples(H):
    """2^20 random (counter, key) tuples: a device-only mistake in mul.hi or a shift shows here and not in the host build."""
    a = np.random.default_rng(11).integers(0, 2 ** 32, (1 << 20, 6), dtype=np.uint64)
    want = np.stack(D.philox_ref(*a.T), axis=1)
    assert np.array_equal(_philox_dev(H, a), want)


# ---- u01 ---------------------------------------------------------------------------------------------------------------------
def test_u01_is_exact_and_inside(H):
    import torch
    rng = np.random.default_rng(12)
    edges = [(0, 0), (0xffffffff, 0xffffffff), (0, 0xfff), (0xffffffff, 0xfff), (0, 0x1000), (0xffffffff, 0xfffff000),
             (0x80000000, 0), (0x7fffffff, 0xffffffff), (1, 0), (0, 0x80000000)]
    hl = np.concatenate([np.array(edges, np.uint64), rng.integers(0, 2 ** 32, (1 << 16, 2), dtype=np.uint64)])
    out = _empty(len(hl), torch.float64)
    _run(H.t_u01, _dev(hl.astype(np.uint32).view(np.int32)), out, len(hl))
    got = out.cpu().numpy()
    bad = [(hex(int(h)), hex(int(lo)), float(g)) for (h, lo), g in zip(hl, got) if Fraction(float(g)) != D.u01_exact(h, lo)]
    assert not bad, bad[:8]
    assert got[0] == 2.0 ** -53 and got[1] == 1 - 2.0 ** -53 and got[2] == got[0] and got[4] == 3 * 2.0 ** -53
    assert (got > 0).all() and (got < 1).all()


# ---- exp_small ---------------------------------------------------------------------------------------------------------------
def test_exp_small(H):
    """Bit for bit the Horner scheme with correctly rounded fmas (coefficients parsed from lr_common.cuh), and within 1 ulp of
    exp over >= 10^5 points of the multiplier window, its ends and +-0.1; exp_small(0) = 1."""
    import torch
    x = D.exp_small_points(np.random.default_rng(13), 1 << 17)
    out = _empty(len(x), torch.float64)
    _run(H.t_exp_small, _dev(x), out, len(x))
    got = out.cpu().numpy()
    assert got[x == 0.0].tolist() == [1.0, 1.0]
    coef = [float(s) for s in D.exp_small_literals()]
    emu = np.array([D.exp_small_emulated(float(v), coef) for v in x])
    diff = np.flatnonzero(_bits(got) != _bits(emu))
    assert diff.size == 0, [(float(x[i]), float(got[i]), float(emu[i])) for i in diff[:8]]
    mpmath.mp.prec = 200
    err = np.array([D.ulp_error(float(g), mpmath.exp(mpmath.mpf(float(v)))) for g, v in zip(got, x)])
    print("exp_small on the device: worst error %.3f ulp over %d points" % (err.max(), len(x)))
    assert err.max() <= 1.0, (float(x[err.argmax()]), float(err.max()))


# ---- accept decisions --------------------------------------------------------------------------------------------------------
def _accept_uniforms(rng):
    """u01 values (2k + 1) 2^-53 in every binade from 2^-53 to 1 - 2^-53: its first and last value and 40 random ones, plus
    2^14 uniformly random ones and the neighbours of 1/2."""
    ks = []
    for b in range(1, 54):                      # u in [2^-b, 2^(1-b)): k in [2^(52-b), 2^(53-b) - 1] (b = 53: k = 0)
        lo, hi = (2 ** (52 - b), 2 ** (53 - b) - 1) if b < 53 else (0, 0)
        ks += [lo, hi] + [int(v) for v in rng.integers(lo, hi + 1, 40, dtype=np.uint64)]
    ks += [int(v) for v in rng.integers(0, 2 ** 52, 1 << 14, dtype=np.uint64)]
    ks += [2 ** 51 - 1, 2 ** 51, 2 ** 51 + 1]
    k = np.array(ks, np.uint64)
    return (2 * k + 1).astype(np.float64) * 2.0 ** -53


def _neighbours(v, n):
    """v and its n neighbours on each side (doubles)."""
    out, up, dn = [v], v, v
    for _ in range(n):
        up, dn = np.nextafter(up, np.inf), np.nextafter(dn, -np.inf)
        out += [up, dn]
    return out


def test_accept_decisions_are_the_double_comparison(H):
    """mh_accept_gt(x, u) == (x > log u) and K3's mh_accept_ge(x, u, lo, hi, log) == (x >= log u), log u the double logarithm of
    the same kernel: at log u and 4 ulp around it, at the bracket's edges and their neighbours, at NaN and +-inf.  The bracket
    only decides where the double logarithm need not be taken, so the plain double comparison is the reference."""
    import torch
    u = _accept_uniforms(np.random.default_rng(14))
    br = _empty(3 * len(u), torch.float64)
    _run(H.t_bracket, _dev(u), br, len(u))
    lo, hi, logu = br.cpu().numpy().reshape(-1, 3).T
    assert (lo <= logu).all() and (logu <= hi).all(), "the bracket misses log(u)"
    cols = np.stack(_neighbours(logu, 4) + _neighbours(lo, 1) + _neighbours(hi, 1)
                    + [np.full_like(u, np.nan), np.full_like(u, np.inf), np.full_like(u, -np.inf)], axis=1)
    x = cols.ravel()
    uu = np.repeat(u, cols.shape[1])
    gt, ge = _empty(len(x), torch.int8), _empty(len(x), torch.int8)
    lg = _empty(len(x), torch.float64)
    _run(H.t_accept, _dev(x), _dev(uu), gt, ge, lg, len(x))
    gt, ge, lg = gt.cpu().numpy().astype(bool), ge.cpu().numpy().astype(bool), lg.cpu().numpy()
    assert np.array_equal(_bits(lg), _bits(np.repeat(logu, cols.shape[1])))
    with np.errstate(invalid="ignore"):
        bad_gt, bad_ge = np.flatnonzero(gt != (x > lg)), np.flatnonzero(ge != (x >= lg))
    assert bad_gt.size == 0, [(float(uu[i]), float(x[i]), float(lg[i]), bool(gt[i])) for i in bad_gt[:8]]
    assert bad_ge.size == 0, [(float(uu[i]), float(x[i]), float(lg[i]), bool(ge[i])) for i in bad_ge[:8]]
    # reported, not asserted: how often the device's double log differs from the correctly rounded one
    mpmath.mp.prec = 200
    off = sum(float(mpmath.log(mpmath.mpf(float(v)))) != float(g) for v, g in zip(u, logu))
    print("device log(u): %d of %d values differ from the correctly rounded logarithm" % (off, len(u)))


# ---- normal_f32 --------------------------------------------------------------------------------------------------------------
LOGF_ABS = 2.0 ** -21.41        # __logf: maximum absolute error on [0.5, 2]
LOGF_ULP = 3.0                  # __logf: maximum ulp error elsewhere
COSPIF_ULP = 1.0                # cospif: maximum ulp error


def _normal_bound(u1, k):
    """Reference sqrt(-2 log u1) cos(2 pi (k + 1/2) / 2^24) at 200 bits, and the largest |normal_f32(u1, k << 8) - reference|
    the documented bounds allow:
      uf = (float)u1; lf = __logf(uf) within LOGF_ABS of log uf on [.5, 2], LOGF_ULP ulp elsewhere; L = -2 lf (exact):
        |L - (-2 log u1)| <= EL = 2 (|log(uf / u1)| + e_log)
      r = sqrtf(L): |sqrt L - R| <= min(sqrt(EL), EL / (R + sqrt(max(R^2 - EL, 0)))) -- absolute where R is tiny (u1 -> 1) --
        plus the rounding 2^-24 sqrt(L)
      a = fl(fl(k + .5) 2^-23): k + .5 rounds for k >= 2^23, off by |a - (k + .5) 2^-23|
      c = cospif(a): COSPIF_ULP ulp of its result, plus pi |a - exact| from the angle
      z = fl(r c): 2^-24 relative."""
    mp = mpmath.mpf
    uf = float(np.float32(u1))
    R = mpmath.sqrt(-2 * mpmath.log(mp(u1)))
    theta = 2 * mpmath.pi * (mp(int(k)) + mp(0.5)) / 2 ** 24
    C = mpmath.cos(theta)
    Z = R * C
    lnuf = abs(float(mpmath.log(mp(uf))))
    e_log = LOGF_ABS if 0.5 <= uf <= 2.0 else LOGF_ULP * 2.0 ** -23 * lnuf / (1 - LOGF_ULP * 2.0 ** -23)
    EL = 2 * (abs(float(mpmath.log(mp(uf) / mp(u1)))) + e_log)
    Rf = float(R)
    ds = min(math.sqrt(EL), EL / (Rf + math.sqrt(max(Rf * Rf - EL, 0.0)))) if Rf > 0 else math.sqrt(EL)
    dr = ds + 2.0 ** -24 * (Rf + ds)
    af = float(np.float32(np.float32(k) + np.float32(0.5)) * np.float32(2.0 ** -23))
    da = math.pi * abs(float(mp(af) - (mp(int(k)) + mp(0.5)) / 2 ** 23))
    Cf = abs(float(C))
    dc = COSPIF_ULP * 2.0 ** -23 * (Cf + da) + da + 2.0 ** -149
    bound = dr * (Cf + dc) + Rf * dc + 2.0 ** -24 * (Rf + dr) * (Cf + dc)
    return Z, bound * (1 + 1e-9)                # the margin covers the double arithmetic of the bound itself


def test_normal_f32_within_its_error_bound(H):
    import torch
    rng = np.random.default_rng(15)
    n = 20000
    u1 = (2 * rng.integers(0, 2 ** 52, n, dtype=np.uint64) + 1).astype(np.float64) * 2.0 ** -53
    k = rng.integers(0, 2 ** 24, n, dtype=np.uint64)
    # u1 -> 1 (r tiny: the absolute error of -2 log u1 dominates), the smallest u1, the float rounding boundaries of 1/2 and 1,
    # and the angle codes where k + 0.5 starts to round
    eu = [1 - 2.0 ** -53, 1 - 2.0 ** -40, 1 - 2.0 ** -26, 1 - 2.0 ** -25, 1 - 3 * 2.0 ** -26, 1 - 2.0 ** -24, 1 - 2.0 ** -23,
          1 - 2.0 ** -22, 1 - 2.0 ** -20, 1 - 2.0 ** -16, 2.0 ** -53, 0.5 - 2.0 ** -53, 0.5 - 2.0 ** -26, 0.5, 0.5 + 2.0 ** -53,
          0.25 - 2.0 ** -53]
    ek = [0, 1, 2 ** 22 - 1, 2 ** 22, 2 ** 23 - 1, 2 ** 23, 2 ** 23 + 1, 3 * 2 ** 22, 2 ** 24 - 2, 2 ** 24 - 1]
    u1 = np.concatenate([np.repeat(eu, len(ek)), np.tile(eu, 4), u1])
    k = np.concatenate([np.tile(np.array(ek, np.uint64), len(eu)), rng.integers(0, 2 ** 24, len(eu) * 4, dtype=np.uint64), k])
    bits = (k << np.uint64(8)) | rng.integers(0, 256, len(k), dtype=np.uint64)       # the low 8 bits are not used
    out = _empty(len(u1), torch.float64)
    _run(H.t_normal, _dev(u1), _dev(bits.astype(np.uint32).view(np.int32)), out, len(u1))
    z = out.cpu().numpy()
    mpmath.mp.prec = 200
    worst, bad = 0.0, []
    for a, kk, g in zip(u1, k, z):
        Z, b = _normal_bound(float(a), int(kk))
        e = float(abs(mpmath.mpf(float(g)) - Z)) if np.isfinite(g) else math.inf
        worst = max(worst, e / b)
        if not e <= b:
            bad.append((float(a), int(kk), float(g), float(Z), b))
    print("normal_f32: worst error %.3f of its bound over %d draws" % (worst, len(z)))
    assert not bad, bad[:8]


@pytest.mark.parametrize("u1", [0.3, 2.0 ** -53, 0.5 + 2.0 ** -53, 1 - 2.0 ** -22, 1 - 2.0 ** -53])
def test_normal_f32_angles_are_symmetric(H, u1):
    """For a fixed u1 the values over all 2^24 angle codes are a multiset equal to its own negation -- what makes K6's normal
    step a symmetric proposal.  For k >= 2^23, (float)k + 0.5f rounds to even, so those codes land on the even multiples of
    2^-23 (twice each, the ends once): a lattice that is still symmetric about 3/2."""
    import torch
    z = _empty(1 << 24, torch.float64)
    _run(H.t_normal_angles, C_D(u1), z)
    s = torch.sort(z).values
    assert torch.isfinite(s).all()
    assert torch.equal(s, -s.flip(0))


# ---- lr_sum ------------------------------------------------------------------------------------------------------------------
def _sum_cases():
    rng = np.random.default_rng(16)
    ln = np.exp(rng.standard_normal(1_000_000))
    return {
        "tenths": np.full(1_000_000, 0.1),
        "column_0.1_0.2_0.3": np.tile([0.1, 0.2, 0.3], 333_334),
        "alternating_1e16_and_1": np.tile([1e16, 1.0, -1e16, 1.0], 25_000),
        "lognormal_sorted": np.sort(ln),
        "lognormal_shuffled": ln,
        "loglik_-3.5e6_sd3": rng.normal(-3.5e6, 3.0, 1_000_000),
    }


SPECIAL_SUMS = [[1.0, math.inf, 2.0], [1.0, -math.inf, -2.0], [math.inf, -math.inf], [1.0, math.nan, 2.0],
                [math.inf, 1.0, math.nan], [1.7976931348623157e308, 1.7976931348623157e308, -1.7976931348623157e308],
                [-1.7976931348623157e308, -1.7976931348623157e308, 1.0], [math.inf, math.inf], []]


def test_lr_sum(H):
    """Within 2 ulp of the correctly rounded sum on every column, twice with the same bits; a sum that meets +-inf or NaN
    gives what the plain sum in order gives.

    A-priori bound of Neumaier's sum (u = 2^-53): u|S| + O(n u^2) sum|x|, printed per case in ulp of S.  It is below an ulp
    for every column but the alternating one (1e16, 1, -1e16, 1, ...), where the second term is large; there every rounding
    error of s is an integer below 2^53 and their sum c is exact, so the result is the correctly rounded sum all the same."""
    import torch
    cases = _sum_cases()
    seqs = list(cases.values()) + [np.array(s, np.float64) for s in SPECIAL_SUMS]
    off = np.concatenate([[0], np.cumsum([len(s) for s in seqs])]).astype(np.int64)
    v = _dev(np.concatenate(seqs))
    o = _dev(off)
    first, second = _empty(len(seqs), torch.float64), _empty(len(seqs), torch.float64)
    _run(H.t_lr_sum, v, o, first, len(seqs))
    _run(H.t_lr_sum, v, o, second, len(seqs))
    got = first.cpu().numpy()
    assert np.array_equal(_bits(got), _bits(second.cpu().numpy()))
    u = 2.0 ** -53
    for (name, x), g in zip(cases.items(), got):
        S = math.fsum(x)
        A = math.fsum(np.abs(x))
        bound = (u * abs(S) + 2 * len(x) * u * u * A) / math.ulp(S)
        err = abs(g - S) / math.ulp(S)
        print("lr_sum %-24s error %.2f ulp, a-priori bound %.3g ulp" % (name, err, bound))
        assert err <= 2.0, (name, g, S, err)
    for s, g in zip(SPECIAL_SUMS, got[len(cases):]):
        plain = 0.0
        for t in s:
            plain += t
        assert (math.isnan(g) and math.isnan(plain)) or g == plain, (s, g, plain)


# ---- lr_key / lr_val ---------------------------------------------------------------------------------------------------------
DMAX, DMIN_DENORM = 1.7976931348623157e308, 5e-324
SPECIALS = [-math.inf, -DMAX, -1.0, -DMIN_DENORM, -0.0, 0.0, DMIN_DENORM, 1.0, DMAX, math.inf]
NAN_BITS = [0x7ff8000000000000, 0xfff8000000000000, 0x7ff0000000000001, 0xfff0000000000001, 0x7fffffffffffffff,
            0xffffffffffffffff, 0x7ff4000000000000]


def _keys(H, x):
    import torch
    key, back = _empty(len(x), torch.int64), _empty(len(x), torch.float64)
    _run(H.t_key, _dev(x), key, back, len(x))
    return key.cpu().numpy().view(np.uint64), back.cpu().numpy()


def _rank(v):
    """Position of a double in the order lr_key promises: by value, -0.0 before +0.0, every NaN last and equal."""
    if math.isnan(v):
        return (2, 0.0, 0)
    return (0, v, 0 if math.copysign(1.0, v) < 0 else 1)


def test_lr_key_orders_the_specials(H):
    x = np.array(SPECIALS + [0.0] * len(NAN_BITS))
    x[len(SPECIALS):] = np.array(NAN_BITS, np.uint64).view(np.float64)
    key, back = _keys(H, x)
    for i in range(len(x)):
        for j in range(len(x)):
            ri, rj = _rank(float(x[i])), _rank(float(x[j]))
            assert (key[i] < key[j]) == (ri < rj) and (key[i] == key[j]) == (ri == rj), (x[i], x[j], hex(key[i]), hex(key[j]))
    assert (key[len(SPECIALS):] == np.uint64(0xffffffffffffffff)).all()
    n = len(SPECIALS)
    assert np.array_equal(_bits(back[:n]), _bits(x[:n]))


def test_lr_key_roundtrip_and_order_of_random_bits(H):
    b = np.random.default_rng(17).integers(0, 2 ** 64, 1_000_000, dtype=np.uint64)
    x = b.view(np.float64)
    key, back = _keys(H, x)
    fin = ~np.isnan(x)
    assert np.array_equal(_bits(back[fin]), b[fin])
    assert (key[~fin] == np.uint64(0xffffffffffffffff)).all()
    s = x[fin][np.argsort(key[fin], kind="stable")]
    assert (np.diff(s) >= 0).all()
    assert np.unique(key[fin]).size == fin.sum()                            # distinct doubles, distinct keys


# ---- warp_sum_first ----------------------------------------------------------------------------------------------------------
def test_warp_sum_first_is_warp_sum(H):
    import torch
    rng = np.random.default_rng(18)
    K = np.repeat(np.arange(1, 33, dtype=np.int32), 16)
    v = rng.standard_normal((len(K), 32)) * 10.0 ** rng.integers(-8, 9, (len(K), 32))
    v[np.arange(32)[None, :] >= K[:, None]] = 0.0
    out = _empty(64 * len(K), torch.float64)
    _run(H.t_warp_sum, _dev(v), _dev(K), out, len(K))
    o = out.cpu().numpy().reshape(len(K), 2, 32)
    full, first = o[:, 0, :], o[:, 1, :]
    assert (_bits(full) == _bits(full[:, :1])).all()                 # the butterfly leaves the same bits in every lane
    bad = np.flatnonzero((_bits(first) != _bits(full[:, :1])).any(axis=1))
    assert bad.size == 0, [(int(K[i]), full[i, 0], first[i].tolist()) for i in bad[:4]]
