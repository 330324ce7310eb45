"""Posterior predictive checks of the per-bin births and deaths of a run (K11, lr_predictive_check).

Every likelihood of the three samplers is  C + sum_j [A^b_j log lambda_j - B^b_j lambda_j] + sum_j [A^d_j log mu_j - B^d_j mu_j]
with event weights A and exposures B per bin (RJMCMC: engine.Dataset.bin_terms; TrendRate / DDRate: sp, br, ex, br of their
statistics).  The model it states is: given a posterior draw, the count of side s in bin j is Poisson(rate_sj B_sj).  For every
post-burn-in record and every bin with B > 0 one replicate count is drawn from that model and compared with the observed A:

  per side and bin   p_mid = (#(y_rep > A) + #(y_rep == A) / 2) / n over the n records used ("obs_high" below p_tail: the data
                     hold more events than the model predicts; "obs_low" above 1 - p_tail), with the expected count, the mean
                     replicate and the predictive sd sqrt(E[mu] + Var[mu]) of the Poisson mixture
  per record         the Poisson deviance D(y, mu) = 2 sum_j [y log(y / mu) - (y - mu)] (0 log 0 = 0) of the observed and of the
                     replicated counts, per side and in total; p = #(D_rep >= D_obs) / n

The exposure B is held at its observed value, as the likelihood holds it: no new lineage table is simulated, so the check asks
whether the counts are Poisson around the fitted rates given the time at risk, not whether the whole process reproduces the data.

predictive_check_host is the definition, step for step (as diagnostics.rhat_ess is for K9): the Philox counter layout, the
sampler, the per-bin rates, the deviances and the counts.  The command line

    python -m literate_b200.predictive <log dir> [-burnin .2] [-seed 0] [-p_tail .025]

checks the RJMCMC logs (*_mcmc.log with their _sp_rates / _ex_rates / _div.log) and DDRate logs (with their .div.log) of a
directory and writes predictive_<kind>.tsv and predictive_<kind>_global.tsv there.  Logs are put in chain order and given the
chain ids of the run that wrote them from their names (chain_ids), so a directory gives the tables the device records give.
The bin_start of DDRate logs is the bin number: neither file holds the window's origin.
"""
from __future__ import annotations

import argparse
import math
import os
import re
from dataclasses import dataclass

import numpy as np

from . import _native as N
from . import engine as E
from . import summary as S

KINDS = {"forward": (0, 0, E.REC_BETA), "trendrate": (1, 16, 15), "dd": (1, 24, 21)}   # kind -> (layout, rate_col, beta field)
POIS_SEARCH, POIS_ATTEMPTS, POIS_MU_MAX = 256, 64, 2.0 ** 52      # lr_poisson (lr_common.cuh)
TIE_TOL = 2.0 ** -44          # a decision this close (relative to its operands) may go either way between exp / log / lgamma builds
MODEL_TAGS = {"BD": 0, "ID": 1, "BDk": 2, "BDd": 3}              # forward.MODEL_SUFFIX
IT_MAX = 9.2e18


# ------------------------------------------------------------------------------------------ the sampler
def philox(c0, c1, c2, c3, k0, k1):
    """Philox-4x32-10 (lr_common.cuh philox4x32_10) on uint32 arrays -> (x, y, z, w) uint32 arrays."""
    m = np.uint64(0xffffffff)
    c = [np.asarray(v).astype(np.uint64) for v in (c0, c1, c2, c3)]
    k0, k1 = np.asarray(k0).astype(np.uint64), np.asarray(k1).astype(np.uint64)
    for _ in range(10):
        p0, p1 = np.uint64(0xD2511F53) * c[0], np.uint64(0xCD9E8D57) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & m, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & m]
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & m, (k1 + np.uint64(0xBB67AE85)) & m
    return tuple(v.astype(np.uint32) for v in c)


def u01(hi, lo):
    """(k + 1/2) 2^-52 of the 52 bits k = hi, top 20 bits of lo (u01 of lr_common.cuh), exactly."""
    k = (np.asarray(hi).astype(np.uint64) << np.uint64(20)) | (np.asarray(lo).astype(np.uint64) >> np.uint64(12))
    return (2 * k + 1).astype(np.float64) * 2.0 ** -53


def counters(it, j, side, chain):
    """K11's Philox counter of (record iteration, bin, side, global chain id) at attempt 0: (c0, c1, c2, c3) uint32 arrays.
    Attempt a sets bits 25.. of c2; the key is (seed low 32 bits, seed high 32 bits)."""
    it = np.asarray(it).astype(np.int64).astype(np.uint64)
    c2 = np.asarray(j).astype(np.uint32) | (np.asarray(side).astype(np.uint32) << np.uint32(24))
    return ((it & np.uint64(0xffffffff)).astype(np.uint32), (it >> np.uint64(32)).astype(np.uint32), c2,
            (np.asarray(chain).astype(np.int64).astype(np.uint64) & np.uint64(0xffffffff)).astype(np.uint32))


def poisson_host(mu, c0, c1, c2, c3, seed):
    """lr_poisson restated: arrays mu and counters (c2 with bits 25.. clear) -> (count int64, near bool, exhausted bool).
    near: a decision of the draw lies within TIE_TOL of a tie (relative to the operands of its comparison), where an exp, log or
    lgamma a few ulp apart may decide it the other way.  Count -1: mu outside [0, 2^52] (no draw)."""
    mu = np.asarray(mu, np.float64)
    c0, c1, c2, c3 = (np.broadcast_to(np.asarray(c, np.uint32), mu.shape) for c in (c0, c1, c2, c3))
    k0, k1 = np.uint32(seed & 0xffffffff), np.uint32((seed >> 32) & 0xffffffff)
    y = np.zeros(mu.shape, np.int64)
    near = np.zeros(mu.shape, bool)
    exh = np.zeros(mu.shape, bool)
    y[~((mu >= 0.0) & (mu <= POIS_MU_MAX))] = -1
    # inversion by sequential search
    i = np.nonzero(((mu > 0.0) & (mu < 10.0)).ravel())[0]
    flat = lambda a: a.reshape(-1)
    yf, nf, ef, mf = flat(y), flat(near), flat(exh), flat(mu)
    if len(i):
        x, yy, _, _ = philox(flat(c0)[i], flat(c1)[i], flat(c2)[i], flat(c3)[i], k0, k1)
        u, m = u01(x, yy), mf[i]
        p = np.exp(-m)
        F = p.copy()
        k = np.zeros(len(i), np.int64)
        nr = np.abs(u - F) <= TIE_TOL * u
        act = u > F
        while act.any():
            stop = act & (k == POIS_SEARCH)
            ef[i[stop]] = True
            k[stop] = 0
            act &= ~stop
            a = np.nonzero(act)[0]
            k[a] += 1
            p[a] = p[a] * m[a] / k[a].astype(np.float64)
            F[a] = F[a] + p[a]
            nr[a] |= np.abs(u[a] - F[a]) <= TIE_TOL * u[a]
            act[a] = u[a] > F[a]
        yf[i], nf[i] = k, nr
    # PTRS
    i = np.nonzero(((mu >= 10.0) & (mu <= POIS_MU_MAX)).ravel())[0]
    if len(i):
        m = mf[i]
        slam, loglam = np.sqrt(m), np.log(m)
        b = 0.931 + 2.53 * slam
        a = -0.059 + 0.02483 * b
        invalpha = 1.1239 + 1.1328 / (b - 3.4)
        vr = 0.9277 - 3.6224 / (b - 2.0)
        lia = np.log(invalpha)
        out = np.zeros(len(i), np.int64)
        nr = np.zeros(len(i), bool)
        act = np.ones(len(i), bool)
        for att in range(POIS_ATTEMPTS):
            q = np.nonzero(act)[0]
            if not len(q):
                break
            g = i[q]
            x, yy, z, w = philox(flat(c0)[g], flat(c1)[g], flat(c2)[g] | np.uint32(att << 25), flat(c3)[g], k0, k1)
            U, V = u01(x, yy) - 0.5, u01(z, w)
            us = 0.5 - np.abs(U)
            kd = np.floor((2.0 * a[q] / us + b[q]) * U + m[q] + 0.43)
            acc = (us >= 0.07) & (V <= vr[q])
            rej = ~acc & ((kd < 0.0) | ((us < 0.013) & (V > us)))
            t = ~acc & ~rej
            if t.any():
                qt = q[t]
                lv, lb = np.log(V[t]), np.log(a[qt] / (us[t] * us[t]) + b[qt])
                lg = np.array([math.lgamma(v) for v in (kd[t] + 1.0)])
                lhs = (lv + lia[qt]) - lb
                rhs = (-m[qt] + kd[t] * loglam[qt]) - lg
                mag = np.abs(lv) + np.abs(lia[qt]) + np.abs(lb) + m[qt] + np.abs(kd[t] * loglam[qt]) + np.abs(lg) + 1.0
                nr[qt] |= np.abs(lhs - rhs) <= TIE_TOL * mag
                acc[t] = lhs <= rhs
            out[q[acc]] = kd[acc].astype(np.int64)
            act[q[acc]] = False
        ef[i[act]] = True
        out[act] = 0
        yf[i], nf[i] = out, nr
    return y, near, exh


# ------------------------------------------------------------------------------------------ the check, host definition
def _cold_rows(records, ladder, beta_col):
    """[S, M T, w] -> rows [S, M, w] and missing [S, M]: the first member of every ladder with field beta_col == 1.0."""
    S_, nk, w = records.shape
    if ladder == 1:
        return records, np.zeros((S_, nk), bool)
    r = records.reshape(S_, nk // ladder, ladder, w)
    hit = r[..., beta_col] == 1.0
    idx = np.argmax(hit, axis=2)
    return np.take_along_axis(r, idx[:, :, None, None], axis=2)[:, :, 0, :], ~hit.any(axis=2)


def bin_rates(rows, layout, n_bins, rate_col=0, start_time=0.0):
    """Per-bin rates [S, M, 2, n_bins] of records rows [S, M, w] and whether each record's rates are usable [S, M] (layout 0: K in
    1..32, finite shift times whose bins do not decrease).  Layout 0 (RJMCMC): segment k of a side starts at bin
    floor(t_k) - floor(start_time) clamped to [0, n_bins] (slot 0 at bin 0) and bin j takes the last segment starting at or before
    it -- the likelihood's own mapping (bin_of_time / side_stats), not np.histogram's.  Layout 1: the fields
    [rate_col, rate_col + n_bins) and the next n_bins."""
    Sh = rows.shape[:2]
    if layout == 1:
        return rows[..., rate_col:rate_col + 2 * n_bins].reshape(Sh + (2, n_bins)), np.ones(Sh, bool)
    s0f = math.floor(start_time)
    out = np.zeros(Sh + (2, n_bins))
    ok = np.ones(Sh, bool)
    j = np.arange(n_bins)
    for side, (kf, rf, tf) in enumerate(((E.REC_KL, E.REC_L, E.REC_TL), (E.REC_KM, E.REC_M, E.REC_TM))):
        kd = rows[..., kf]
        valid = (kd >= 1) & (kd <= 32) & (kd == np.floor(kd))
        K = np.where(valid, kd, 1).astype(np.int64)
        t = rows[..., tf:tf + 32]
        inside = (np.arange(32) >= 1) & (np.arange(32) < K[..., None])
        fin = np.isfinite(t) | ~inside
        jb = np.where(inside & fin, np.clip(np.floor(np.where(fin, t, 0.0)) - s0f, 0, n_bins), 0).astype(np.int64)
        jb = np.where(inside, jb, n_bins + 1)                                  # slots >= K never start a bin
        jb[..., 0] = 0
        order = np.all(np.where(inside[..., 1:], jb[..., 1:] >= jb[..., :-1], True), axis=-1)
        ok &= valid & fin.all(axis=-1) & order
        slot = (jb[..., None, 1:] <= j[:, None]).sum(axis=-1)                  # [S, M, n_bins]
        out[..., side, :] = np.take_along_axis(rows[..., rf:rf + 32], slot, axis=-1)
    return out, ok


def predictive_check_host(records, layout, n_bins, terms, rate_col=0, start_time=0.0, rep_of_chain=None, ladder=1, beta_col=-1,
                          chain_id0=0, seed=0):
    """K11 on host records [n_samples, n_chains * ladder, w] (after the burn-in): the definition lr_predictive_check computes.
    terms [n_rep, 4, n_bins]: A^b, B^b, A^d, B^d; rep_of_chain [n_chains] (None: 0).  Returns a dict of the kernel's outputs --
    bin_count int64 [2, 4, n_bins] (used, sum y_rep, #(y_rep > A), #(y_rep == A)), bin_sum [2, 3, n_bins] (sum mu, mu^2, A),
    glob_count int64 [4] (used, #(D_rep >= D_obs) birth, death, total), glob_sum [6], dev [S, M, 4] (NaN where not used), status
    int64 [3] -- plus near [S, M]: records with a draw or a deviance comparison within TIE_TOL of a tie (sums are exactly rounded
    (math.fsum) where the kernel's are compensated in its own fixed order)."""
    records = np.asarray(records, np.float64)
    terms = np.asarray(terms, np.float64).reshape(-1, 4, n_bins)
    rows, missing = _cold_rows(records, ladder, beta_col)
    S_, M = rows.shape[:2]
    rep = np.zeros(M, np.int64) if rep_of_chain is None else np.asarray(rep_of_chain, np.int64)
    rates, ok = bin_rates(rows, layout, n_bins, rate_col, start_time)
    T = terms[rep]                                                              # [M, 4, nb]
    A = np.stack([T[:, 0], T[:, 2]], axis=1)[None]                              # [1, M, 2, nb]
    B = np.stack([T[:, 1], T[:, 3]], axis=1)[None]
    has = np.broadcast_to(B > 0.0, rates.shape)
    with np.errstate(invalid="ignore", over="ignore"):
        mu = rates * B
    mu_ok = np.where(has, (mu >= 0.0) & (mu <= POIS_MU_MAX), True).all(axis=(2, 3))
    it = rows[..., 0]
    ok &= (it >= 0.0) & (it < IT_MAX) & mu_ok
    used = ok & ~missing
    status = np.array([int((~ok & ~missing).sum()), 0, int(missing.sum())], np.int64)
    draw = has & used[..., None, None]
    s_i, c_i, side_i, j_i = np.nonzero(draw)
    c = counters(np.where(used, it, 0.0)[s_i, c_i], j_i, side_i, chain_id0 + c_i)
    y_d, near_d, exh_d = poisson_host(mu[draw], *c, seed)
    status[1] = int(exh_d.sum())
    y = np.zeros(rates.shape, np.int64)
    y[draw] = y_d
    near = np.zeros((S_, M), bool)
    np.logical_or.at(near, (s_i, c_i), near_d)
    Ab = np.broadcast_to(A, rates.shape)
    yd = y.astype(np.float64)
    bin_count = np.zeros((2, 4, n_bins), np.int64)
    bin_count[:, 0] = draw.sum(axis=(0, 1))
    bin_count[:, 1] = np.where(draw, y, 0).sum(axis=(0, 1))
    bin_count[:, 2] = (draw & (yd > Ab)).sum(axis=(0, 1))
    bin_count[:, 3] = (draw & (yd == Ab)).sum(axis=(0, 1))
    bin_sum = np.zeros((2, 3, n_bins))
    for side in range(2):
        for jj in range(n_bins):
            sel = draw[:, :, side, jj]
            m_ = mu[:, :, side, jj][sel]
            bin_sum[side, 0, jj] = math.fsum(m_)
            bin_sum[side, 1, jj] = math.fsum(m_ * m_)
            bin_sum[side, 2, jj] = math.fsum(Ab[:, :, side, jj][sel])

    def term(yv, m_):
        with np.errstate(divide="ignore", invalid="ignore"):
            return np.where(yv == 0.0, m_, yv * np.log(yv / m_) - (yv - m_))
    dev = np.full((S_, M, 4), np.nan)
    glob_count = np.zeros(4, np.int64)
    sums = [[] for _ in range(6)]
    for s_, c_ in zip(*np.nonzero(used)):
        D = []
        for side in range(2):
            sel = draw[s_, c_, side]
            m_ = mu[s_, c_, side][sel]
            D += [2.0 * math.fsum(term(Ab[s_, c_, side][sel], m_)), 2.0 * math.fsum(term(yd[s_, c_, side][sel], m_))]
        D += [D[0] + D[2], D[1] + D[3]]
        dev[s_, c_] = D[:4]
        glob_count += [1, D[1] >= D[0], D[3] >= D[2], D[5] >= D[4]]
        for k in range(6):
            sums[k].append(D[k])
        if any(abs(D[2 * k + 1] - D[2 * k]) <= 1e-9 * max(abs(D[2 * k]), abs(D[2 * k + 1])) for k in range(3)):
            near[s_, c_] = True
    glob_sum = np.array([math.fsum(v) for v in sums])
    return {"bin_count": bin_count, "bin_sum": bin_sum, "glob_count": glob_count, "glob_sum": glob_sum, "dev": dev,
            "status": status, "near": near}


# ------------------------------------------------------------------------------------------ results
@dataclass
class PredictiveResult:
    """The outputs of one check (K11 or its host definition) and the tables formed from them."""
    kind: str
    first_edge: float              # bin_start of bin 0: the RJMCMC run's start time; for device records of TrendRate / DDRate what the
                                   # caller gives (the window's origin); 0.0 for DDRate logs, which do not hold the origin (bin numbers)
    bin_count: np.ndarray          # int64 [2, 4, n_bins]
    bin_sum: np.ndarray            # [2, 3, n_bins]
    glob_count: np.ndarray         # int64 [4]
    glob_sum: np.ndarray           # [6]
    status: np.ndarray             # int64 [3]
    dev: np.ndarray = None         # [S, M, 4] per-record deviances, when asked for

    @classmethod
    def from_outputs(cls, kind, first_edge, out):
        return cls(kind, float(first_edge), *(np.asarray(out[k]) for k in ("bin_count", "bin_sum", "glob_count", "glob_sum", "status")),
                   None if out.get("dev") is None else np.asarray(out["dev"]))

    def table(self, p_tail=0.025):
        """Rows (side, bin start, observed, expected, mean_rep, sd_rep, p_mid, flag) of every side and bin; observed is the mean
        of A over the records used (A itself when every chain runs on one replicate); bins without a draw are flagged "none"."""
        rows = []
        for side, name in enumerate(("birth", "death")):
            for j in range(self.bin_count.shape[2]):
                n = int(self.bin_count[side, 0, j])
                if n == 0:
                    rows.append((name, self.first_edge + j, math.nan, math.nan, math.nan, math.nan, math.nan, "none"))
                    continue
                e = float(self.bin_sum[side, 0, j]) / n
                var = e + max(float(self.bin_sum[side, 1, j]) / n - e * e, 0.0)
                p = (int(self.bin_count[side, 2, j]) + 0.5 * int(self.bin_count[side, 3, j])) / n
                flag = "obs_high" if p < p_tail else ("obs_low" if p > 1.0 - p_tail else "ok")
                rows.append((name, self.first_edge + j, float(self.bin_sum[side, 2, j]) / n, e, int(self.bin_count[side, 1, j]) / n,
                             math.sqrt(var), p, flag))
        return rows

    def global_table(self):
        """Rows (part, records, mean_D_obs, mean_D_rep, p) for birth, death and total; p = #(D_rep >= D_obs) / records."""
        n = int(self.glob_count[0])
        return [(name, n, float(self.glob_sum[2 * k]) / n if n else math.nan, float(self.glob_sum[2 * k + 1]) / n if n else math.nan,
                 int(self.glob_count[1 + k]) / n if n else math.nan) for k, name in enumerate(("birth", "death", "total"))]

    def write_tsv(self, out_dir, p_tail=0.025):
        """predictive_<kind>.tsv and predictive_<kind>_global.tsv in out_dir; returns their paths."""
        f = lambda v: v if isinstance(v, str) else (str(v) if isinstance(v, int) else repr(float(v)))
        paths = [os.path.join(out_dir, "predictive_%s.tsv" % self.kind), os.path.join(out_dir, "predictive_%s_global.tsv" % self.kind)]
        heads = [("side", "bin_start", "observed", "expected", "mean_rep", "sd_rep", "p_mid", "flag"),
                 ("part", "records", "mean_D_obs", "mean_D_rep", "p")]
        for path, head, rows in zip(paths, heads, (self.table(p_tail), self.global_table())):
            with open(path, "w") as fh:
                fh.write("\t".join(head) + "\n")
                for r in rows:
                    fh.write("\t".join(f(v) for v in r) + "\n")
        return paths

    def summary_line(self, p_tail=0.025):
        g = self.global_table()
        flagged = sum(r[7] in ("obs_high", "obs_low") for r in self.table(p_tail))
        return "%s: %d records, deviance p birth %.4g death %.4g total %.4g; %d of %d side-bins outside [%g, %g]" % (
            self.kind, g[0][1], g[0][4], g[1][4], g[2][4], flagged, 2 * self.bin_count.shape[2], p_tail, 1 - p_tail)


# ------------------------------------------------------------------------------------------ device
def predictive_records_device(dev, records, kind, terms, start_time=0.0, first_edge=None, burnin=0.2, ladder=1, seed=0,
                              rep_of_chain=None, chain_id0=0, per_record=False):
    """K11 on a float64 CUDA tensor of records [n_samples, n_chains * ladder, w] of K3 ("forward"), K6 ("trendrate") or K7 ("dd")
    after removing the burn-in of every chain (summary.burnin_index).  terms [n_rep, 4, n_bins] (torch or numpy): the per-bin
    A^b, B^b, A^d, B^d (RJMCMC: Dataset.bin_terms(); TrendRate / DDRate: sp, br, ex, br of the statistics the sampler was created
    on, see stats_terms); start_time: the RJMCMC run's start time (its bin mapping); first_edge: start of bin 0 in the tables
    (default start_time).  ladder > 1: checked over the cold members.  -> PredictiveResult (dev with per_record)."""
    import torch
    if kind not in KINDS:
        raise ValueError("kind must be one of %s" % ", ".join(KINDS))
    layout, rate_col, beta_col = KINDS[kind]
    b0 = S.burnin_index(records.shape[0], burnin)
    out = dev.predictive_check_device(records[b0:], layout, terms, rate_col=rate_col, start_time=start_time, rep_of_chain=rep_of_chain,
                                      ladder=ladder, beta_col=beta_col if ladder > 1 else -1, chain_id0=chain_id0, seed=seed,
                                      per_record=per_record)
    host = {k: (v.cpu().numpy() if isinstance(v, torch.Tensor) else v) for k, v in out.items()}
    return PredictiveResult.from_outputs(kind, start_time if first_edge is None else first_edge, host)


def stats_terms(sp, ex, br):
    """The per-bin terms of the Keiding likelihood of TrendRate and DDRate: [n_rep, 4, n_bins] = sp, br, ex, br."""
    sp, ex, br = (np.atleast_2d(np.asarray(a, np.float64)) for a in (sp, ex, br))
    return np.ascontiguousarray(np.stack([sp, br, ex, br], axis=1))


# ------------------------------------------------------------------------------------------ logs
def chain_ids(paths, kind):
    """The logs of one run in chain order and the global id of the first: the samplers log chain k of a run over n_tab tables
    as table k % n_tab (tables in sorted order), run i = k // n_tab -- forward.py as <table><model><out>[_chain<i>]_mcmc.log,
    ddrate.py as <table>_<seed + i><model>.log (i counted from the lowest seed among the logs).  K11 keys its draws by the chain
    id, so the logs give the draws of the device records they were written from.  Refuses names outside these patterns and
    logs that are not consecutive chains of one run.  Returns (sorted paths, first chain id)."""
    keys = [log_key(p, kind) for p in paths]
    stems = sorted({k[0] for k in keys})
    i0 = 0 if kind == "forward" else min(k[1] for k in keys)
    ids = [(i - i0) * len(stems) + stems.index(st) for st, i in keys]
    order = np.argsort(ids, kind="stable")
    ids = [ids[o] for o in order]
    if ids != list(range(ids[0], ids[0] + len(ids))):
        raise ValueError("the logs are not consecutive chains of one run (chains %s)" % ids)
    return [paths[o] for o in order], ids[0]


def log_key(path, kind):
    """(stem, run index) of a log name: forward.py's <table><model><out>[_chain<i>]_mcmc.log -> (<table><model><out>, i), ddrate.py's
    <table>_<seed><model>.log -> (<table><model>, seed).  Logs of one run share the stems of its tables."""
    b = os.path.basename(path)
    m = re.match(r"(.*?)(?:_chain(\d+))?_mcmc\.log$", b) if kind == "forward" else re.match(r"(.*)_(\d+)(_[A-Z]+_M[A-Z]+)\.log$", b)
    if not m:
        raise ValueError("%s: not a log name of the sampler (%s)" % (path, "<table><model><out>[_chain<i>]_mcmc.log" if kind == "forward"
                                                                         else "<table>_<seed><model>.log"))
    return (m.group(1), int(m.group(2) or 0)) if kind == "forward" else (m.group(1) + m.group(3), int(m.group(2)))


def model_tag(path):
    """-model_BDI of an RJMCMC log from its file name (the _BD / _ID / _BDk / _BDd of forward.MODEL_SUFFIX), or None."""
    toks = os.path.basename(path)[:-len("_mcmc.log")].split("_")
    tags = [MODEL_TAGS[t] for t in toks if t in MODEL_TAGS]
    return tags[-1] if tags else None


def _read_div(path):
    tbl = np.loadtxt(path, delimiter="\t", skiprows=1, ndmin=2)
    return tbl[:, 0].astype(np.int64), tbl[:, 1].astype(np.int64), tbl[:, 2].astype(np.float64)


def pack_forward_log(path, burnin=0.2):
    """The post-burn-in rows of an RJMCMC log and its _sp_rates / _ex_rates logs as K3 records [n, LR_REC_DOUBLES]: iteration,
    logged likelihood, K_l, K_m, beta 1, the rates and shift times (slot 0 = the logged start time).  Rates and times are printed
    with repr, so the fields are exactly those of the records the log was written from.  Returns (records, start_time, end_time)."""
    head = open(path).readline().rstrip("\r\n").split("\t")
    tbl = np.loadtxt(path, delimiter="\t", skiprows=1, ndmin=2)
    idx = {h: i for i, h in enumerate(head)}
    stem = path[:-len("mcmc.log")]
    b0 = S.burnin_index(tbl.shape[0], burnin)
    recs = np.zeros((tbl.shape[0] - b0, E.LR_REC_DOUBLES))
    start, end = float(tbl[0, idx["root_age"]]), float(tbl[0, idx["death_age"]])
    for side, (tag, kf, rf, tf) in enumerate((("sp_rates.log", E.REC_KL, E.REC_L, E.REC_TL), ("ex_rates.log", E.REC_KM, E.REC_M, E.REC_TM))):
        with open(stem + tag) as fh:
            lines = fh.read().splitlines()
        if len(lines) != tbl.shape[0]:
            raise ValueError("%s holds %d rows, %s %d" % (stem + tag, len(lines), path, tbl.shape[0]))
        for r, line in enumerate(lines[b0:]):
            v = [float(x) for x in line.split("\t")]
            K = (len(v) + 1) // 2
            recs[r, kf] = K
            recs[r, rf:rf + K] = v[:K]
            recs[r, tf] = start
            recs[r, tf + 1:tf + K] = v[K:]
    recs[:, E.REC_IT] = tbl[b0:, idx["it"]]
    recs[:, E.REC_LIK] = tbl[b0:, idx["likelihood"]]
    recs[:, E.REC_BETA] = 1.0
    return recs, start, end


def check_forward_model(path, model, recs, start, end, sp, ex, br, lik_of):
    """Refuses a log whose logged likelihood of its first used row is not what the -model_BDI of its name and its div.log give
    (lik_of(model, start, end, sp, ex, br, state) -> likelihood, state = (L, M, timesL, timesM) as Dataset.evaluate takes)."""
    if model is None:
        raise ValueError("%s: no model tag (_BD, _ID, _BDk, _BDd) in the file name" % path)
    if model == 3:
        raise ValueError("%s: -model_BDI 3 (_BDd) logs cannot be checked from their div.log, which lacks the extinct-only "
                         "statistics; use predictive.predictive_records_device on the device records" % path)
    r = recs[0]
    kl, km = int(r[E.REC_KL]), int(r[E.REC_KM])
    state = (r[E.REC_L:E.REC_L + kl], r[E.REC_M:E.REC_M + km], np.append(r[E.REC_TL:E.REC_TL + kl], end),
             np.append(r[E.REC_TM:E.REC_TM + km], end))
    lik = float(lik_of(model, start, end, sp, ex, br, state))
    if not abs(lik - r[E.REC_LIK]) <= 1e-9 * max(1.0, abs(lik)):
        raise ValueError("%s: the logged likelihood %r is not the model %d likelihood %r of its div.log (a -pyrate_output log, a "
                         "different div.log or another model)" % (path, float(r[E.REC_LIK]), model, lik))


def _device_lik(dev):
    def lik_of(model, start, end, sp, ex, br, state):
        ds = E.Dataset(dev, E.BinStats(0, sp[None], ex[None], br[None]), model, start, end)
        try:
            return ds.evaluate([state])["lik"][0]
        finally:
            ds.close()
    return lik_of


def forward_logs(paths, burnin=0.2, lik_of=None):
    """RJMCMC logs (one per chain) -> (records [n, chains, LR_REC_DOUBLES], model, start, end, sp, ex, br [chains, n_bins], first
    chain id): chains in the order of chain_ids, every log on its own div.log (its replicate), chains cut to the shortest, the
    model confirmed per log (check_forward_model)."""
    paths, id0 = chain_ids(paths, "forward")
    packs, stats, models = [], [], set()
    for p in paths:
        recs, start, end = pack_forward_log(p, burnin)
        sp, ex, br = _read_div(p[:-len("mcmc.log")] + "div.log")
        m = model_tag(p)
        check_forward_model(p, m, recs, start, end, sp, ex, br, lik_of)
        packs.append((recs, start, end)); stats.append((sp, ex, br)); models.add(m)
    if len(models) != 1 or len({(s, e) for _, s, e in packs}) != 1 or len({s[0].shape for s in stats}) != 1:
        raise ValueError("the logs of a check must share the model and the time window")
    n = min(len(r) for r, _, _ in packs)
    return (np.stack([r[:n] for r, _, _ in packs], axis=1), models.pop(), packs[0][1], packs[0][2],
            *(np.stack(v) for v in zip(*stats)), id0)


def dd_logs(paths, burnin=0.2):
    """DDRate logs (one per chain) -> (records [n, chains, LR_DD_REC_HEAD + 4 n_bins] holding the iteration, beta 1 and the logged
    birth and death rates where K7 writes them, terms [chains, 4, n_bins] of each log's .div.log, first chain id): chains in the
    order of chain_ids, cut to the shortest.  Refuses a .div.log with fewer rows than the log has bins (-m_birth 3 writes the
    statistics zipped with the genre table's, so a shorter genre window cuts them) and logs of different bin counts."""
    from . import ddrate as DD
    paths, id0 = chain_ids(paths, "dd")
    recs, terms = [], []
    for p in paths:
        head = open(p).readline().rstrip("\r\n").split("\t")
        tbl = np.loadtxt(p, delimiter="\t", skiprows=1, ndmin=2)
        idx = {h: i for i, h in enumerate(head)}
        nb = sum(h.startswith("l_") and h[2:].isdigit() for h in head)
        tbl = tbl[S.burnin_index(tbl.shape[0], burnin):]
        r = np.zeros((tbl.shape[0], N.LR_DD_REC_HEAD + 4 * nb))
        r[:, 0] = tbl[:, idx["it"]]
        r[:, DD.REC_BETA] = 1.0
        r[:, N.LR_DD_REC_HEAD:N.LR_DD_REC_HEAD + 2 * nb] = tbl[:, idx["l_0"]:idx["l_0"] + 2 * nb]
        recs.append(r)
        sp, ex, br = _read_div(p[:-len(".log")] + ".div.log")
        if len(sp) < nb:
            raise ValueError("%s: its .div.log holds %d bins, the log %d (a genre table over a shorter window cuts the statistics); "
                             "use predictive.predictive_records_device with stats_terms(sp, ex, br)" % (p, len(sp), nb))
        terms.append(stats_terms(sp[:nb], ex[:nb], br[:nb])[0])
    if len({t.shape for t in terms}) != 1:
        raise ValueError("the DDRate logs of a check must have the same bins")
    n = min(len(r) for r in recs)
    return np.stack([r[:n] for r in recs], axis=1), np.stack(terms), id0


def check_dir(log_dir, burnin=0.2, seed=0, p_tail=0.025, device=None, out_dir=None, note=print):
    """The command line's work: every checkable kind of a log directory -> {kind: PredictiveResult}, tables written to out_dir
    (default log_dir)."""
    import torch
    from . import diagnostics as D
    logs = D.find_logs(log_dir)
    if "trendrate" in logs:
        raise SystemExit("TrendRate logs: trend_rate.py writes no statistics beside its log; use "
                         "predictive.predictive_records_device on the device records with stats_terms(sp, ex, br)")
    if not logs:
        raise SystemExit("no RJMCMC or DDRate sample logs in " + log_dir)
    dev = device if device is not None else E.Device(0)
    td = torch.device("cuda", dev.index)
    out = {}
    for kind, paths in logs.items():
        if kind == "forward":
            try:
                recs, model, start, end, sp, ex, br, id0 = forward_logs(paths, burnin, _device_lik(dev))
            except ValueError as e:
                raise SystemExit(str(e))
            ds = E.Dataset(dev, E.BinStats(0, sp, ex, br), model, start, end)
            terms = ds.bin_terms()
            res = predictive_records_device(dev, torch.from_numpy(recs).to(td), "forward", terms, start_time=start, burnin=0,
                                            seed=seed, rep_of_chain=np.arange(recs.shape[1], dtype=np.int32), chain_id0=id0)
            ds.close()
        else:
            try:
                recs, terms, id0 = dd_logs(paths, burnin)
            except ValueError as e:
                raise SystemExit(str(e))
            # neither a DDRate log nor its .div.log holds the window's origin: the table numbers the bins from 0
            res = predictive_records_device(dev, torch.from_numpy(recs).to(td), "dd", terms, first_edge=0.0, burnin=0, seed=seed,
                                            rep_of_chain=np.arange(recs.shape[1], dtype=np.int32), chain_id0=id0)
        res.write_tsv(out_dir or log_dir, p_tail)
        note(res.summary_line(p_tail))
        out[kind] = res
    return out


def main(argv=None):
    ap = argparse.ArgumentParser(prog="python -m literate_b200.predictive",
                                 description="posterior predictive checks of the per-bin births and deaths of the sample logs of a directory")
    ap.add_argument("log_dir")
    ap.add_argument("-burnin", type=float, default=0.2, help="fraction (< 1) or number of rows of every log dropped first")
    ap.add_argument("-seed", type=int, default=0, help="seed of the replicate draws")
    ap.add_argument("-p_tail", type=float, default=0.025, help="bins with p_mid below it or above 1 - it are flagged")
    ap.add_argument("-device", type=int, default=0)
    a = ap.parse_args(argv)
    if not (0.0 < a.p_tail < 0.5):
        raise SystemExit("-p_tail must be in (0, 0.5)")
    if a.seed < 0 or a.seed >= 2 ** 64:
        raise SystemExit("-seed must be in [0, 2^64)")
    if not os.path.isdir(a.log_dir):
        raise SystemExit("not a directory: " + a.log_dir)
    check_dir(a.log_dir, a.burnin, a.seed, a.p_tail, E.Device(a.device))


if __name__ == "__main__":
    main()
