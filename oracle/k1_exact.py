"""Exact reference of K1 (lineages -> per-bin sp, ex, br) under the kernel's stated arithmetic.

Restates precompute_events / get_br (LiteRateForward.py:111-123, :529-549) the way include/literate_b200.h (L2) promises
them:

* counts come from the raw doubles: births ts in [t0, t1), deaths te in (t0, t1]; rows with te <= ts or NaN still count
  as events but carry no time at risk;
* time at risk uses quantized endpoints, a birth at floor(ts) + q(ts - floor(ts)) and a death at
  (ceil(te) - 1) + q(te - (ceil(te) - 1)), with q(x) = rint(x * 2^52) / 2^52 and the difference taken in fp64.  For
  |t| >= 1 this is the identity (the difference is exact and already on the 2^-52 grid); it only moves times in (-1, 1);
* br[j] = sum_i max(0, min(hi_i, t1) - max(lo_i, t0)) summed exactly and rounded once, to nearest.

exact_bin_stats is O(n); exact_time_at_risk_literal is the same definition per bin and per lineage in Fractions, for a
few hundred lineages, and exists to check the O(n) version.
"""
from __future__ import annotations

import math
from fractions import Fraction

import numpy as np

FIX_SHIFT = 52
FIX = 1 << FIX_SHIFT
_LIMB = 26                      # fractions <= 2^52 split into 26 + 27 bits: a per-bin limb sum stays below 2^53 in float64
MAX_LINEAGES = 1 << 26


def _q(x):
    """rint(x * 2^52) of fp64 fractions in [0, 1], as int64 (ties to even, as the kernel's rounding)."""
    return np.rint(x * float(FIX)).astype(np.int64)


def _exact_sums(bins, vals, n_bins):
    """Per-bin exact sums (Python ints) of non-negative int64 values <= 2^52."""
    lo = (vals & ((1 << _LIMB) - 1)).astype(np.float64)
    hi = (vals >> _LIMB).astype(np.float64)
    s_lo = np.bincount(bins, weights=lo, minlength=n_bins)[:n_bins].astype(np.int64)
    s_hi = np.bincount(bins, weights=hi, minlength=n_bins)[:n_bins].astype(np.int64)
    return [int(a) + (int(b) << _LIMB) for a, b in zip(s_lo, s_hi)]


def _one(ts, te, first_bin, n_bins):
    T0, T1 = float(first_bin), float(first_bin) + float(n_bins)
    with np.errstate(invalid="ignore"):
        born = (ts >= T0) & (ts < T1)
        died = (te > T0) & (te <= T1)
        live = te > ts
    sp = np.bincount((np.floor(ts[born]) - first_bin).astype(np.int64), minlength=n_bins)[:n_bins].astype(np.int64)
    ex = np.bincount((np.ceil(te[died]) - 1 - first_bin).astype(np.int64), minlength=n_bins)[:n_bins].astype(np.int64)

    # time at risk: each live lineage is an interval between two points (bin, fraction in 2^-52 units) of the window,
    # a start with fraction in [0, 2^52) and an end with fraction in (0, 2^52]
    s, e = ts[live], te[live]
    ia = np.zeros(len(s), np.int64); fs = np.zeros(len(s), np.int64)
    ib = np.full(len(s), n_bins - 1, np.int64); fe = np.full(len(s), FIX, np.int64)
    m = (s >= T0) & (s < T1)
    ia[s >= T1] = n_bins                # born after the window: starts at its end
    if m.any():
        fl = np.floor(s[m])
        ia[m] = fl.astype(np.int64) - first_bin
        fs[m] = _q(s[m] - fl)
    m = (e > T0) & (e <= T1)
    ib[e <= T0] = -1                    # died before the window: ends at its start
    if m.any():
        c1 = np.ceil(e[m]) - 1.0
        ib[m] = c1.astype(np.int64) - first_bin
        fe[m] = _q(e[m] - c1)
    up = fs == FIX                      # a birth fraction that rounds to 1: the start of the next bin
    ia[up] += 1; fs[up] = 0
    down = fe == 0                      # a death fraction that rounds to 0: the end of the previous bin
    ib[down] -= 1; fe[down] = FIX
    keep = (ia < ib) | ((ia == ib) & (fs < fe))         # false for lineages that end before / start after the window
    ia, fs, ib, fe = ia[keep], fs[keep], ib[keep], fe[keep]
    same = ia == ib
    d = ~same
    bins = np.concatenate([ia[same], ia[d], ib[d]])
    vals = np.concatenate([fe[same] - fs[same], FIX - fs[d], fe[d]])
    part = _exact_sums(bins, vals, n_bins)
    # whole years of the bins strictly between the two ends (difference array)
    full = np.bincount(ia[d] + 1, minlength=n_bins + 1) - np.bincount(ib[d], minlength=n_bins + 1)
    full = np.cumsum(full)[:n_bins]
    br = np.array([float(Fraction(p + (int(f) << FIX_SHIFT), FIX)) for p, f in zip(part, full)], dtype=np.float64)
    return sp, ex, br


def exact_bin_stats(ts, te, first_bin, n_bins, only_dead=False, end_time=None):
    """(sp, ex, br) of one table over bins [first_bin + j, first_bin + j + 1), j < n_bins; with only_dead also
    (ex_dead, br_dead) of the lineages with te < end_time (:531-532; end_time defaults to max te)."""
    ts = np.ascontiguousarray(ts, dtype=np.float64).ravel()
    te = np.ascontiguousarray(te, dtype=np.float64).ravel()
    if ts.shape != te.shape:
        raise ValueError("ts and te must have the same length")
    if len(ts) > MAX_LINEAGES:
        raise ValueError("at most 2^26 lineages: the limb sums must stay exact in float64")
    first_bin, n_bins = int(first_bin), int(n_bins)
    sp, ex, br = _one(ts, te, first_bin, n_bins)
    if not only_dead:
        return sp, ex, br
    if end_time is None:
        end_time = np.max(te)
    with np.errstate(invalid="ignore"):
        keep = te < end_time
    _, exd, brd = _one(ts[keep], te[keep], first_bin, n_bins)
    return sp, ex, br, exd, brd


def _q_literal(x):
    return Fraction(round(x * FIX), FIX)


def exact_time_at_risk_literal(ts, te, first_bin, n_bins):
    """br of the same definition, bin by bin and lineage by lineage in exact rationals (a few hundred lineages at most)."""
    out = []
    ends = []
    for s, e in zip(np.asarray(ts, dtype=np.float64).tolist(), np.asarray(te, dtype=np.float64).tolist()):
        if not e > s:
            continue
        lo = s if math.isinf(s) else math.floor(s) + _q_literal(s - math.floor(s))
        hi = e if math.isinf(e) else (math.ceil(e) - 1) + _q_literal(e - (math.ceil(e) - 1))
        ends.append((lo, hi))
    for j in range(int(n_bins)):
        t0, t1 = int(first_bin) + j, int(first_bin) + j + 1
        tot = Fraction(0)
        for lo, hi in ends:
            d = min(hi, t1) - max(lo, t0)
            if d > 0:
                tot += d
        out.append(float(tot))
    return np.array(out, dtype=np.float64)
