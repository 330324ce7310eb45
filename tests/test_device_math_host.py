"""CPU: what of the shared sampler arithmetic of lr_common.cuh can be checked without a device.

* philox4x32_10 is __host__ __device__: a host program built with nvcc from lr_common.cuh (tests/device_math_harness.cu) gives
  Random123's known-answer vectors bit for bit, and the uint64 restatement of the round function on random tuples;
* exp_small, emulated exactly from the coefficients of the c_exp_small initialiser as lr_common.cuh spells them: the
  coefficients are 1/n! to 16 significant digits, exp_small(0) is 1, and the result is within 1 ulp of exp (mpmath, 200 bits)
  over the log-multiplier window of K3, K6 and K7 and over +-0.1.
"""
import math
import subprocess
from fractions import Fraction

import mpmath
import numpy as np
import pytest

import _device_math as D


@pytest.fixture(scope="module")
def philox_host(tmp_path_factory):
    exe = D.compile_harness(tmp_path_factory.mktemp("device_math_host"), host_main=True)

    def run(rows):
        inp = "".join(" ".join("%08x" % v for v in r) + "\n" for r in rows)
        p = subprocess.run([exe], input=inp, capture_output=True, text=True, check=True)
        return [tuple(int(w, 16) for w in line.split()) for line in p.stdout.splitlines()]
    return run


def test_philox_known_answers_on_the_host(philox_host):
    got = philox_host([c + k for c, k, _ in D.PHILOX_KAT])
    assert got == [want for _, _, want in D.PHILOX_KAT]


def test_philox_host_build_equals_the_restatement(philox_host):
    rng = np.random.default_rng(7)
    a = rng.integers(0, 2 ** 32, (2000, 6), dtype=np.uint64)
    a[:6] = np.eye(6, dtype=np.uint64) * 0xffffffff                  # one word set at a time
    want = np.stack(D.philox_ref(*a.T), axis=1)
    assert np.array_equal(np.array(philox_host(a.tolist()), np.uint64), want.astype(np.uint64))


def test_restatement_gives_the_known_answers():
    for c, k, want in D.PHILOX_KAT:
        assert tuple(int(v) for v in D.philox_ref(*c, *k)) == want


def _sig16(q, rounded):
    """q (a positive Fraction) to 16 significant decimal digits, exactly: rounded to nearest, or truncated."""
    e = math.floor(math.log10(q))
    while Fraction(10) ** e > q:
        e -= 1
    while Fraction(10) ** (e + 1) <= q:
        e += 1
    unit = Fraction(10) ** (e - 15)
    return (round(q / unit) if rounded else math.floor(q / unit)) * unit


def test_exp_small_coefficients_are_reciprocal_factorials():
    """c_exp_small[k] is 1/n!, n = 11 - k, rounded to 16 significant digits (a shorter literal: its trailing zeros dropped).
    Most terms are too small to move the result by an ulp on |x| <= 0.1, so only this pins a mistyped digit there.

    1/4! is the one literal truncated instead of rounded (4.166666666666666e-2): its double is 1 ulp below the one nearest 1/24,
    which moves x^4 / 24 by less than 6e-22 on |x| <= 0.1, far below the final rounding (the emulation below stays within
    0.55 ulp).  It stays as it is: a correctly rounded coefficient would change the last bit of a rare multiplier, and from
    there the chains of K3, K6 and K7."""
    lits = D.exp_small_literals()
    assert len(lits) == 12
    for k, s in enumerate(lits):
        n = 11 - k
        assert Fraction(s) == _sig16(Fraction(1, math.factorial(n)), rounded=n != 4), (n, s)


def test_exp_small_emulated_within_one_ulp():
    """The exact emulation of exp_small against exp at 200 bits, over the window LN_MULT (u - 1/2) of the u01 values, its
    ends and +-0.1: at most 1 ulp (truncation of the Taylor series < 2e-21, i.e. the fma roundings only)."""
    coef = [float(s) for s in D.exp_small_literals()]
    assert D.exp_small_emulated(0.0, coef) == 1.0
    x = D.exp_small_points(np.random.default_rng(3), 20000)
    assert np.abs(x).max() <= 0.1
    mpmath.mp.prec = 200
    worst = max(D.ulp_error(D.exp_small_emulated(v, coef), mpmath.exp(mpmath.mpf(float(v)))) for v in x)
    print("exp_small, exact emulation: worst error %.3f ulp over %d points" % (worst, len(x)))
    assert worst <= 1.0
