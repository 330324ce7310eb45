"""PSIS-LOO, WAIC and model comparison of runs over their per-bin births and deaths (K12, lr_loo).

The observation is the count A of side s (birth, death) in bin j, the unit K11 checks.  Given a posterior draw every sampler here
models it as Poisson(rate_sj B_sj) with the exposure B held at its observed value, so the pointwise log-likelihood of a column
with B > 0 is the full Poisson log pmf

    l_sj = A log(r B) - r B - lgamma(A + 1)            (A log(r B) = 0 for A = 0)

Summed over the columns it is the sampler's likelihood plus a constant of the run.  Because l is a normalised pmf of the count, two
runs on the same table compare even when their likelihood constants or exposures differ (model 1 holds B = 1 on the birth side).
DDRate's genre term is not a per-bin count: the posterior conditions on it, but it is not a compared observation.

Per column, over the S used draws of all chains (a LOO pools them, so every chain must run on the same table):
  r_eff      ESS / S, the "mean" ESS of diagnostics.rhat_ess (K9) of exp(l - max l) over the chains; 1 when that is NaN
  PSIS       ArviZ's _psislw / _gpdfit / _gpinv (psis_host, gpdfit_host): k_hat and log weights lw
  elpd_loo   logsumexp(l + lw);  lppd = logsumexp(l) - log S;  p_loo = lppd - elpd_loo
  WAIC       p_waic = var(l, ddof 1);  elpd_waic = lppd - p_waic
Globally the sums over the columns, se = sqrt(n var(pointwise, ddof 0)) as ArviZ computes it, and the columns whose k_hat exceeds
min(1 - 1 / log10 S, 0.7) (Vehtari et al. 2024).  compare() ranks runs of one table as az.compare does.

loo_host is the definition, step for step.  The command line

    python -m literate_b200.loo <dir> [<dir> ...] [-burnin .2] [-out <dir>] [-device 0]

reads the RJMCMC and DDRate logs of each directory (one run per directory) through predictive.py's readers, writes
loo_<kind>.tsv and loo_<kind>_global.tsv there and, with more than one model, loo_compare.tsv to -out (default the first
directory).  DDRate logs number their bins from 0, as in K11.
"""
from __future__ import annotations

import argparse
import math
import os
from dataclasses import dataclass

import numpy as np

from . import engine as E
from . import predictive as P
from . import summary as S

LOG_TINY = float(np.log(np.finfo(float).tiny))
EPS = float(np.finfo(float).eps)
FIELDS = ("A", "lppd", "elpd_loo", "p_loo", "elpd_waic", "p_waic", "k_hat", "r_eff", "tail")


# ------------------------------------------------------------------------------------------ the definition
def logsumexp(x):
    x = np.asarray(x, np.float64)
    m = x.max()
    return float(m + np.log(np.sum(np.exp(x - m))))


def gpdfit_host(y):
    """Zhang and Stephens' fit of a generalised Pareto distribution to the ascending exceedances y [T] (ArviZ's _gpdfit):
    m = 30 + floor(sqrt(T)) grid points b_i = 1/y_T + (1 - sqrt(m / (i - 1/2))) / (3 y_[T/4 + 1/2]), k_i = mean log1p(-b_i y),
    L_i = T (log(-b_i / k_i) - k_i - 1), w_i = 1 / sum_l exp(L_l - L_i) (those below 10 eps dropped, the rest renormalised),
    b = sum w_i b_i, k = mean log1p(-b y), sigma = -k / b, and k shrunk to (T k + 5) / (T + 10).  Returns (k, sigma)."""
    y = np.asarray(y, np.float64)
    n = len(y)
    m = 30 + int(n ** 0.5)
    b = 1 - np.sqrt(m / (np.arange(1, m + 1, dtype=float) - 0.5))
    b /= 3 * y[int(n / 4 + 0.5) - 1]
    b += 1 / y[-1]
    k = np.log1p(-b[:, None] * y).mean(axis=1)
    L = n * (np.log(-(b / k)) - k - 1)
    with np.errstate(over="ignore"):                 # exp(L_l - L_i) = inf gives the weight 0, as it should
        w = 1 / np.exp(L - L[:, None]).sum(axis=1)
    keep = w >= 10 * EPS
    w, b = w[keep], b[keep]
    w /= w.sum()
    bh = np.sum(b * w)
    kk = np.log1p(-bh * y).mean()
    sigma = -kk / bh
    return float((n * kk + 5.0) / (n + 10)), float(sigma)


def psis_host(log_ratios, r_eff=1.0):
    """Pareto-smoothed log weights of log importance ratios [S] (ArviZ's _psislw; for LOO the ratios are -l):
      a. x = ratios - max; M = ceil(min(0.2 S, 3 sqrt(S / r_eff)))
      b. cutoff = max(x_(S-M-1), log(DBL_MIN)) (ascending, 0-based); the tail is {x > cutoff}, T its size (T <= M with ties)
      c. T <= 4: k_hat = +inf, no smoothing
      d. else the GPD fit of y = exp(x_tail) - exp(cutoff), ascending (gpdfit_host)
      e. k_hat finite: the sorted tail becomes log(sigma expm1(-k log1p(-p)) / k + exp(cutoff)), p = (t - 1/2) / T
         (-log1p(-p) sigma for |k| < eps; NaN for sigma <= 0), and x[x > 0] = 0
      f. lw = x - logsumexp(x)
    r_eff is taken as given, so that a test can hand over the device's.  Returns (lw [S], k_hat, T)."""
    x = np.array(log_ratios, np.float64)
    n = len(x)
    x = x - x.max()
    M = int(math.ceil(min(0.2 * n, 3 * math.sqrt(n / r_eff))))
    cutoff = max(float(np.sort(x)[n - M - 1]), LOG_TINY)
    tail = np.nonzero(x > cutoff)[0]
    T = len(tail)
    k = math.inf
    if T > 4:
        order = tail[np.argsort(x[tail], kind="stable")]
        ec = math.exp(cutoff)
        k, sigma = gpdfit_host(np.exp(x[order]) - ec)
        if math.isfinite(k):
            p = np.arange(0.5, T) / T
            if sigma <= 0:
                g = np.full(T, np.nan)
            elif abs(k) < EPS:
                g = -np.log1p(-p) * sigma
            else:
                g = np.expm1(-k * np.log1p(-p)) / k * sigma
            x[order] = np.log(g + ec)
            x[x > 0] = 0
    return x - logsumexp(x), k, T


def pointwise_host(records, layout, n_bins, terms, rate_col=0, start_time=0.0, ladder=1, beta_col=-1):
    """l [S, M, 2, n_bins] of records [S, M ladder, w] on terms [4, n_bins] (0 where B = 0), the columns with B > 0 [2, n_bins], the
    used records [S, M] (K11's rule and every l of the record finite) and status int64 [2] (skipped, no member at beta = 1)."""
    records = np.asarray(records, np.float64)
    terms = np.asarray(terms, np.float64).reshape(4, n_bins)
    rows, missing = P._cold_rows(records, ladder, beta_col)
    rates, ok = P.bin_rates(rows, layout, n_bins, rate_col, start_time)
    A, B = terms[[0, 2]], terms[[1, 3]]
    act = B > 0.0
    lg = np.array([[math.lgamma(a + 1.0) if h else 0.0 for a, h in zip(ar, hr)] for ar, hr in zip(A, act)])
    with np.errstate(invalid="ignore", over="ignore", divide="ignore"):
        mu = rates * B
        ll = np.where(A == 0.0, 0.0, A * np.log(mu)) - mu - lg
    ll = np.where(act, ll, 0.0)
    mu_ok = np.where(act, (mu >= 0.0) & (mu <= P.POIS_MU_MAX) & np.isfinite(ll), True).all(axis=(2, 3))
    it = rows[..., 0]
    ok &= (it >= 0.0) & (it < P.IT_MAX) & mu_ok
    used = ok & ~missing
    return ll, act, used, np.array([int((~ok & ~missing).sum()), int(missing.sum())], np.int64)


def loo_host(records, layout, n_bins, terms, rate_col=0, start_time=0.0, ladder=1, beta_col=-1, r_eff=None):
    """K12 on host records [n_samples, n_chains * ladder, w] (after the burn-in) of one table, terms [4, n_bins]: the definition
    lr_loo computes.  r_eff [2, n_bins] replaces the r_eff of step 1 when given.  Returns a dict: out [9, 2, n_bins] (A, lppd,
    elpd_loo, p_loo, elpd_waic, p_waic, k_hat, r_eff, T; NaN where B = 0), n (records used), status int64 [2]."""
    from . import diagnostics as D
    ll, act, used, status = pointwise_host(records, layout, n_bins, terms, rate_col, start_time, ladder, beta_col)
    terms = np.asarray(terms, np.float64).reshape(4, n_bins)
    out = np.full((9, 2, n_bins), np.nan)
    n = int(used.sum())
    for side, j in zip(*np.nonzero(act)):
        out[0, side, j] = terms[2 * side, j]
        if n < 2:
            continue
        col = ll[:, :, side, j]
        l = col[used]
        if r_eff is not None:
            reff = float(r_eff[side, j])
        else:
            w = np.where(used, np.exp(col - l.max()), np.nan)
            ess = D.rhat_ess(w.T)["ess"]
            reff = 1.0 if ess != ess else ess / n
        lw, k, T = psis_host(-l, reff)
        lppd = logsumexp(l) - math.log(n)
        elpd = logsumexp(l + lw)
        pw = float(np.var(l, ddof=1))
        out[1:, side, j] = [lppd, elpd, lppd - elpd, lppd - pw, pw, k, reff, T]
    return {"out": out, "n": n, "status": status}


# ------------------------------------------------------------------------------------------ results
@dataclass
class LooResult:
    """The outputs of one LOO (K12 or its host definition) and the tables formed from them."""
    kind: str
    first_edge: float              # bin_start of bin 0 (0.0 for DDRate logs, which number their bins)
    out: np.ndarray                # [9, 2, n_bins]
    n: int                         # records used
    status: np.ndarray             # int64 [2]

    @property
    def columns(self):
        """[2, n_bins] bool: the columns with B > 0."""
        return ~np.isnan(self.out[0])

    def threshold(self):
        """min(1 - 1 / log10 S, 0.7): the k_hat above which a column's PSIS estimate is unreliable (Vehtari et al. 2024)."""
        return min(1.0 - 1.0 / math.log10(self.n), 0.7) if self.n > 1 else math.nan

    def flags(self):
        """Per side and bin: "none" (B = 0), "k_inf" (k_hat not finite: a tail of at most 4 draws or a failed fit, so the weights
        are not smoothed and the estimate is not reliable), "k_high" (k_hat above the threshold) or "ok"."""
        th = self.threshold()
        k = self.out[6]
        return np.where(~self.columns, "none", np.where(~np.isfinite(k), "k_inf", np.where(k > th, "k_high", "ok")))

    def table(self):
        """Rows (side, bin_start, observed, lppd, elpd_loo, p_loo, elpd_waic, p_waic, k_hat, r_eff, tail, flag) of every side
        and bin."""
        fl = self.flags()
        rows = []
        for side, name in enumerate(("birth", "death")):
            for j in range(self.out.shape[2]):
                v = [float(x) for x in self.out[:8, side, j]]
                t = self.out[8, side, j]
                rows.append((name, self.first_edge + j, *v, int(t) if t == t else math.nan, str(fl[side, j])))
        return rows

    def pointwise(self, f="elpd_loo"):
        return self.out[FIELDS.index(f)][self.columns]

    def global_row(self):
        """(columns, records, elpd_loo, se_elpd_loo, p_loo, elpd_waic, se_elpd_waic, p_waic, k_high, k_threshold)."""
        c = int(self.columns.sum())
        e, w = self.pointwise("elpd_loo"), self.pointwise("elpd_waic")
        se = lambda v: math.sqrt(len(v) * float(np.var(v))) if len(v) else math.nan
        fl = self.flags()
        return (c, int(self.n), float(e.sum()), se(e), float(self.pointwise("p_loo").sum()), float(w.sum()), se(w),
                float(self.pointwise("p_waic").sum()), int(((fl == "k_high") | (fl == "k_inf")).sum()), self.threshold())

    def write_tsv(self, out_dir):
        """loo_<kind>.tsv and loo_<kind>_global.tsv in out_dir; returns their paths."""
        paths = [os.path.join(out_dir, "loo_%s.tsv" % self.kind), os.path.join(out_dir, "loo_%s_global.tsv" % self.kind)]
        heads = [("side", "bin_start", "observed", "lppd", "elpd_loo", "p_loo", "elpd_waic", "p_waic", "k_hat", "r_eff", "tail", "flag"),
                 ("columns", "records", "elpd_loo", "se_elpd_loo", "p_loo", "elpd_waic", "se_elpd_waic", "p_waic", "k_high",
                  "k_threshold")]
        for path, head, rows in zip(paths, heads, (self.table(), [self.global_row()])):
            _write(path, head, rows)
        return paths

    def summary_line(self):
        g = self.global_row()
        return "%s: %d records, %d columns, elpd_loo %.6g (se %.3g), p_loo %.4g, elpd_waic %.6g; %d columns with k_hat > %.3g" % (
            self.kind, g[1], g[0], g[2], g[3], g[4], g[5], g[8], g[9])


def _fmt(v):
    return v if isinstance(v, str) else (str(v) if isinstance(v, (int, np.integer)) else repr(float(v)))


def _write(path, head, rows):
    with open(path, "w") as fh:
        fh.write("\t".join(head) + "\n")
        for r in rows:
            fh.write("\t".join(_fmt(v) for v in r) + "\n")


def compare(results, names=None):
    """az.compare-style ranking of LooResults of one table: rows (rank, model, elpd_loo, se, p_loo, elpd_diff, se_diff, k_high),
    best first; elpd_diff = best - this, se_diff = sqrt(n var(pointwise difference, ddof 0)).  Refuses results whose
    observations differ: a different number of bins, a different set of columns, or A not equal bit for bit (exposures may
    differ)."""
    names = list(names) if names is not None else ["model%d" % i for i in range(len(results))]
    if len(results) < 2 or len(names) != len(results):
        raise ValueError("compare needs at least two results and one name per result")
    r0 = results[0]
    for name, r in zip(names[1:], results[1:]):
        if r.out.shape != r0.out.shape:
            raise ValueError("%s: %d bins, %s: %d; results of different tables do not compare" % (names[0], r0.out.shape[2], name, r.out.shape[2]))
        if not np.array_equal(r.columns, r0.columns):
            raise ValueError("%s and %s hold different columns (bins with B > 0); they do not compare" % (names[0], name))
        if r.out[0][r.columns].tobytes() != r0.out[0][r0.columns].tobytes():
            raise ValueError("%s and %s observe different counts A; they do not compare" % (names[0], name))
    pts = [r.pointwise("elpd_loo") for r in results]
    tot = [float(p.sum()) for p in pts]
    order = sorted(range(len(results)), key=lambda i: -tot[i])
    best = order[0]
    rows = []
    for rank, i in enumerate(order):
        g = results[i].global_row()
        d = pts[best] - pts[i]
        se_diff = 0.0 if i == best else math.sqrt(len(d) * float(np.var(d)))
        rows.append((rank, names[i], tot[i], g[3], g[4], tot[best] - tot[i], se_diff, g[8]))
    return rows


COMPARE_HEAD = ("rank", "model", "elpd_loo", "se", "p_loo", "elpd_diff", "se_diff", "k_high")


def write_compare(path, rows):
    _write(path, COMPARE_HEAD, rows)
    return path


# ------------------------------------------------------------------------------------------ device
def one_table(rep_of_chain, n_rep):
    """The replicate every chain runs on; refuses chains on more than one (imputation replicates are different data)."""
    reps = {0} if rep_of_chain is None else set(int(r) for r in np.asarray(rep_of_chain).ravel())
    if len(reps) != 1:
        raise ValueError("a LOO pools the draws of every chain, so every chain must run on one table; these run on replicates %s"
                         % sorted(reps))
    r = reps.pop()
    if not 0 <= r < n_rep:
        raise ValueError("replicate %d outside the %d of the terms" % (r, n_rep))
    return r


def loo_records_device(dev, records, kind, terms, start_time=0.0, first_edge=None, burnin=0.2, ladder=1, rep_of_chain=None):
    """K12 on a float64 CUDA tensor of records [n_samples, n_chains * ladder, w] of K3 ("forward"), K6 ("trendrate") or K7 ("dd")
    after removing the burn-in of every chain (summary.burnin_index).  terms [n_rep, 4, n_bins] or [4, n_bins] as for
    predictive.predictive_records_device; every chain must run on one replicate (rep_of_chain).  -> LooResult."""
    import torch
    if kind not in P.KINDS:
        raise ValueError("kind must be one of %s" % ", ".join(P.KINDS))
    layout, rate_col, beta_col = P.KINDS[kind]
    t = torch.as_tensor(terms, dtype=torch.float64)
    if t.dim() == 2:
        t = t[None]
    r = one_table(rep_of_chain, t.shape[0])
    b0 = S.burnin_index(records.shape[0], burnin)
    out = dev.loo_device(records[b0:], layout, t[r], rate_col=rate_col, start_time=start_time, ladder=ladder,
                         beta_col=beta_col if ladder > 1 else -1)
    return LooResult(kind, float(start_time if first_edge is None else first_edge), out["out"].cpu().numpy(), int(out["n"].item()),
                     out["status"].cpu().numpy())


# ------------------------------------------------------------------------------------------ logs
def dir_logs(log_dir):
    """{kind: sample logs} of a directory that holds one run per kind; refuses TrendRate logs (trend_rate.py writes no statistics
    beside them), a directory without logs, and logs of one kind with more than one stem (table, model and -out: chain_ids
    would read two runs on one table as two tables of one run, and a LOO would pool two models' draws)."""
    from . import diagnostics as D
    logs = D.find_logs(log_dir)
    if "trendrate" in logs:
        raise SystemExit("TrendRate logs: trend_rate.py writes no statistics beside its log; use loo.loo_records_device on the "
                         "device records with predictive.stats_terms(sp, ex, br)")
    if not logs:
        raise SystemExit("no RJMCMC or DDRate sample logs in " + log_dir)
    for kind, paths in logs.items():
        try:
            stems = sorted({P.log_key(p, kind)[0] for p in paths})
        except ValueError as e:
            raise SystemExit(str(e))
        if len(stems) != 1:
            raise SystemExit("%s: the %s logs of one directory must be one run (one table, model and -out); found %s"
                             % (log_dir, kind, ", ".join(stems)))
    return logs


def loo_dir(log_dir, burnin=0.2, device=None, note=print):
    """The LOO of every kind of run in a log directory (dir_logs) -> {kind: LooResult}; the tables are written there."""
    import torch
    logs = dir_logs(log_dir)
    dev = device if device is not None else E.Device(0)
    td = torch.device("cuda", dev.index)
    out = {}
    for kind, paths in logs.items():
        try:
            if kind == "forward":
                recs, model, start, end, sp, ex, br, _ = P.forward_logs(paths, burnin, P._device_lik(dev))
                if not all(np.array_equal(a[0], a[i]) for a in (sp, ex, br) for i in range(len(a))):
                    raise ValueError("%s: the div.log tables of the chains differ; a LOO needs one table" % log_dir)
                ds = E.Dataset(dev, E.BinStats(0, sp[:1], ex[:1], br[:1]), model, start, end)
                try:
                    terms = ds.bin_terms()
                finally:
                    ds.close()
                res = loo_records_device(dev, torch.from_numpy(recs).to(td), "forward", terms, start_time=start, burnin=0)
            else:
                recs, terms, _ = P.dd_logs(paths, burnin)
                if not all(np.array_equal(terms[0], t) for t in terms):
                    raise ValueError("%s: the .div.log tables of the chains differ; a LOO needs one table" % log_dir)
                # neither a DDRate log nor its .div.log holds the window's origin: the table numbers the bins from 0
                res = loo_records_device(dev, torch.from_numpy(recs).to(td), "dd", terms[:1], first_edge=0.0, burnin=0)
        except ValueError as e:
            raise SystemExit(str(e))
        res.write_tsv(log_dir)
        note(res.summary_line())
        out[kind] = res
    return out


def main(argv=None, device=None, note=print):
    ap = argparse.ArgumentParser(prog="python -m literate_b200.loo",
                                 description="PSIS-LOO and WAIC of the per-bin births and deaths of the runs of log directories, "
                                             "and their comparison")
    ap.add_argument("log_dir", nargs="+", help="one run per directory")
    ap.add_argument("-burnin", type=float, default=0.2, help="fraction (< 1) or number of rows of every log dropped first")
    ap.add_argument("-out", default=None, help="directory of loo_compare.tsv (default: the first log directory)")
    ap.add_argument("-device", type=int, default=0)
    a = ap.parse_args(argv)
    for d in a.log_dir:
        if not os.path.isdir(d):
            raise SystemExit("not a directory: " + d)
    if len({os.path.realpath(d) for d in a.log_dir}) != len(a.log_dir):
        raise SystemExit("a directory is named twice")
    for d in a.log_dir:
        dir_logs(d)
    dev = device if device is not None else E.Device(a.device)
    names, results = [], []
    for d in a.log_dir:
        for kind, res in loo_dir(d, a.burnin, dev, note).items():
            names.append("%s:%s" % (d, kind))
            results.append(res)
    if len(results) > 1:
        try:
            rows = compare(results, names)
        except ValueError as e:
            raise SystemExit(str(e))
        out_dir = a.out or a.log_dir[0]
        write_compare(os.path.join(out_dir, "loo_compare.tsv"), rows)
        for r in rows:
            note("%d  %-40s elpd_loo %.6g  elpd_diff %.4g  se_diff %.3g  k_high %d" % (r[0], r[1], r[2], r[5], r[6], r[7]))
    return dict(zip(names, results))


if __name__ == "__main__":
    main()
