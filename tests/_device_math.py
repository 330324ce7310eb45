"""Exact host references of the sampler arithmetic in literate_b200/csrc/lr_common.cuh, and the build of its test harness
tests/device_math_harness.cu (test_device_math_host.py, test_gpu_device_math.py)."""
import os
import re
import subprocess
from fractions import Fraction

import mpmath
import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)
HARNESS = os.path.join(HERE, "device_math_harness.cu")
COMMON = os.path.join(REPO, "literate_b200", "csrc", "lr_common.cuh")

LN_MULT = 0.19062035960864987          # 2 log(1.1): the log-multiplier window of K3, K6 and K7 (LR_LN_MULT, TR_LN_MULT, DD_LN_MULT)

# Random123's known-answer vectors of Philox-4x32-10 (kat_vectors): counter, key -> output
PHILOX_KAT = [
    ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0), (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
]


def compile_harness(out_dir, host_main=False):
    """nvcc with the library's own flags: the shared library of the harness kernels, or (host_main) its host Philox program.
    Skips when there is no nvcc."""
    from literate_b200 import build
    try:
        nvcc = build._nvcc()
    except RuntimeError:
        pytest.skip("nvcc not found")
    out = os.path.join(str(out_dir), "device_math_host" if host_main else "device_math_harness.so")
    cmd = [nvcc] + build.NVCC_FLAGS + (["-DLR_HARNESS_HOST_MAIN"] if host_main else ["-shared"]) + [HARNESS, "-o", out]
    p = subprocess.run(cmd, capture_output=True, text=True)
    assert p.returncode == 0, " ".join(cmd) + "\n" + p.stdout + p.stderr
    return out


def philox_ref(c0, c1, c2, c3, k0, k1):
    """Philox-4x32-10 (Salmon et al., SC'11) on uint32 arrays, restated with uint64 products: (x, y, z, w) as uint32 arrays."""
    m = np.uint64(0xffffffff)
    c = [np.asarray(v, np.uint64) for v in (c0, c1, c2, c3)]
    k0, k1 = np.asarray(k0, np.uint64), np.asarray(k1, np.uint64)
    for _ in range(10):
        p0, p1 = np.uint64(0xD2511F53) * c[0], np.uint64(0xCD9E8D57) * c[2]       # < 2^64: exact
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & m, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & m]
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & m, (k1 + np.uint64(0xBB67AE85)) & m
    return tuple(v.astype(np.uint32) for v in c)


def u01_exact(hi, lo):
    """(k + 1/2) 2^-52, k = the 52 kept bits of (hi, lo): all of hi, the top 20 bits of lo."""
    return Fraction((int(hi) << 20) | (int(lo) >> 12), 2 ** 52) + Fraction(1, 2 ** 53)


def exp_small_literals():
    """The initialiser of c_exp_small in lr_common.cuh, as the source spells it (strings, highest order first)."""
    with open(COMMON) as fh:
        src = fh.read()
    m = re.search(r"c_exp_small\[(\d+)\]\s*=\s*\{(.*?)\};", src, re.S)
    assert m, "c_exp_small not found in lr_common.cuh"
    lits = [t.strip() for t in re.sub(r"/\*.*?\*/", "", m.group(2)).split(",")]
    assert len(lits) == int(m.group(1))
    return lits


def exp_small_emulated(x, coef):
    """exp_small's Horner scheme with every fma correctly rounded: p = fl(p x + c), exactly."""
    fx = Fraction(x)
    p = coef[0]
    for c in coef[1:]:
        p = float(Fraction(p) * fx + Fraction(c))
    return p


def ulp_at(v):
    """Spacing of the doubles at the real number v (an mpf), in the binade of v itself."""
    if v == 0:
        return 2.0 ** -1074
    _, e = mpmath.frexp(v)                     # v = m 2^e, |m| in [1/2, 1)
    return 2.0 ** max(int(e) - 53, -1074)


def ulp_error(got, ref):
    """|got - ref| in units of the last place at ref (ref an mpf)."""
    return float(abs(mpmath.mpf(got) - ref)) / ulp_at(ref)


def exp_small_points(rng, n):
    """n points of the log-multiplier window LN_MULT (u - 1/2), u a u01 value, plus both ends of the window, +-0.1 and 0."""
    k = rng.integers(0, 2 ** 52, n, dtype=np.uint64)
    u = (2 * k + 1).astype(np.float64) * 2.0 ** -53            # (k + 1/2) 2^-52, exact: 2k + 1 < 2^53
    x = LN_MULT * (u - 0.5)
    ends = [LN_MULT * (2.0 ** -53 - 0.5), LN_MULT * ((1 - 2.0 ** -53) - 0.5)]
    edges = ends + [np.nextafter(e, 0.0) for e in ends] + [0.1, -0.1, np.nextafter(0.1, 0), np.nextafter(-0.1, 0), 0.0, -0.0,
                                                         2.0 ** -30, -(2.0 ** -30), 1e-300, -1e-300]
    return np.concatenate([np.array(edges), x])
