"""Convergence diagnostics over the chains of a run: split R-hat and the "mean" effective sample size (Vehtari et al. 2021, section
3; Stan's and ArviZ's rhat(method="split") and ess(method="mean")) of every logged column -- what the reference's notebooks check
in Tracer one log at a time ("ESS >= 200 per parameter"), for thousands of chains at once and with a multi-chain R-hat.

  rhat_ess                  host restatement of the estimator on one column x [chains, draws], step for step: the definition
                            K9 (lr_chain_diagnostics) computes and the reference of the tests
  diagnostic_columns        the (name, record spec) list of a sampler's records, in log column order
  diagnose_records_device   K9 on device-resident records (RJMCMC: plus the per-bin marginal rates of K5's matrices)
  diagnose_logs             K9 on the post-burn-in rows of sample logs, one log per chain
  rank_rhat_ess             host restatement of the rank-normalised R-hat and bulk and tail ESS (Vehtari et al. 2021, section
                            4; ArviZ's rhat(method="rank"), ess(method="bulk" / "tail")): the definition K10
                            (lr_rank_diagnostics) computes; diagnose_records_device and diagnose_logs add it with rank=True

  python -m literate_b200.diagnose <dir> [-burnin .2] [-rhat_max 1.01] [-ess_min 200] [-device 0] [-rank 0]
"""
from __future__ import annotations

import math
import os
from dataclasses import dataclass

import numpy as np

from . import ddrate as DD
from . import engine as E
from . import plotdd as PD
from . import summary as S
from . import trend as TR

KINDS = ("forward", "trendrate", "dd")
FORWARD_COLS = [("posterior", (E.REC_LIK, E.REC_PRIOR, 1, 0.0)), ("likelihood", E.REC_LIK), ("prior", E.REC_PRIOR),
                ("lambda_avg", E.REC_LAVG), ("mu_avg", E.REC_MAVG), ("K_l", E.REC_KL), ("K_m", E.REC_KM),
                ("gamma_rate_hp_BI", E.REC_GL), ("gamma_rate_hp_D", E.REC_GM), ("poisson_rate_hp", E.REC_POI)]
FLAGS = ("ok", "rhat", "ess", "rhat+ess", "const", "stuck", "nonfinite")


# ------------------------------------------------------------------------------------------ the estimator
def rhat_ess(x):
    """Split R-hat and "mean" ESS of one column x [chains, draws] (draws in sampling order) -> dict of floats mean, sd, rhat, ess,
    lag (Geyer's max_t; -1 for degenerate columns) and margin (host only: the smallest |value| a decision of Geyer's sequence
    turned on, so that tests can tell a tie from a difference).

      1. n = floor(S / 2); split chain 2c = draws [0, n) of chain c, 2c + 1 = draws [S - n, S) (an odd S drops the middle draw);
         m = 2 M.  S < 4: RuntimeError("not enough data").
      2. mean_j of each split chain (exactly its value when all its draws are equal); acov_j(t) = (1/n) sum_{i < n-t} d_ij d_{i+t,j},
         d = x - mean_j.
      3. W = n/(n-1) mean_j acov_j(0); var+ = (n-1)/n W + var_j(mean_j, ddof 1) (exactly 0 when all mean_j are equal);
         R-hat = sqrt(var+ / W); sd = sqrt(var+); mean = the mean of the m n draws used.
      4. rho_0 = 1, rho_t = 1 - (W - mean_j acov_j(t)) / var+.
      5. Geyer's initial positive sequence: rho[0] = 1, rho[1] = rho_1, even = 1, odd = rho_1, t = 1; while t < n - 3 and
         even + odd > 0: even, odd = rho_{t+1}, rho_{t+2}; if even + odd >= 0 store them at t+1, t+2; t += 2.  max_t = t - 2; if
         even > 0: rho[max_t + 1] = even.
      6. Initial monotone sequence: for t = 1, 3, ... while t <= max_t - 2: if rho[t+1] + rho[t+2] > rho[t-1] + rho[t], both
         become (rho[t-1] + rho[t]) / 2.
      7. tau = -1 + 2 sum_{t <= max_t} rho[t] + rho[max_t + 1], at least 1 / log10(m n); ESS = m n / tau; lag = max_t.
      8. A non-finite draw: every output NaN, lag -1.  W = 0 and var+ = 0 (constant): R-hat NaN, ESS NaN, lag -1.  W = 0 and
         var+ > 0 (every split chain stuck on its own value): R-hat +inf, ESS NaN, lag -1.
    Sums are exact where the device compensates them (math.fsum), so the two agree to rounding."""
    x = np.asarray(x, dtype=np.float64)
    if x.ndim == 1:
        x = x[None, :]
    M, Sd = x.shape
    if Sd < 4:
        raise RuntimeError("not enough data")
    n = Sd // 2
    s = np.stack([x[:, :n], x[:, Sd - n:]], axis=1).reshape(2 * M, n)         # row 2c: first half of chain c, 2c + 1: second half
    m = s.shape[0]
    nan = float("nan")
    if not np.all(np.isfinite(s)):
        return {"mean": nan, "sd": nan, "rhat": nan, "ess": nan, "lag": -1, "margin": math.inf}
    mean = math.fsum(s.ravel()) / (m * n)
    mj = np.array([r[0] if r.min() == r.max() else math.fsum(r) / n for r in s])
    d = s - mj[:, None]

    def mean_acov(t):
        return np.mean(np.sum(d[:, :n - t] * d[:, t:], axis=1) / n)

    W = n / (n - 1) * mean_acov(0)
    if np.all(mj == mj[0]):
        between = 0.0
    else:
        xbar = math.fsum(mj) / m
        between = math.fsum((mj - xbar) ** 2) / (m - 1)
    varp = (n - 1) / n * W + between
    sd = math.sqrt(varp)
    if W == 0.0:
        return {"mean": mean, "sd": sd, "rhat": nan if varp == 0.0 else math.inf, "ess": nan, "lag": -1, "margin": math.inf}
    rhat = math.sqrt(varp / W)
    rho_hat = lambda t: 1.0 - (W - mean_acov(t)) / varp
    rho = np.zeros(n + 1)
    rho[0] = 1.0
    rho[1] = rho_hat(1)
    even, odd, t = 1.0, rho[1], 1
    margin, stored = abs(even + odd), True          # every pair sum is a decision (> 0, >= 0), and so is the last even if unstored
    while t < n - 3 and even + odd > 0:
        even, odd = rho_hat(t + 1), rho_hat(t + 2)
        margin = min(margin, abs(even + odd))
        stored = even + odd >= 0
        if stored:
            rho[t + 1], rho[t + 2] = even, odd
        t += 2
    max_t = t - 2
    if even > 0:
        rho[max_t + 1] = even
    if not stored:
        margin = min(margin, abs(even))
    t = 1
    while t <= max_t - 2:
        if rho[t + 1] + rho[t + 2] > rho[t - 1] + rho[t]:
            rho[t + 1] = rho[t + 2] = (rho[t - 1] + rho[t]) / 2
        t += 2
    tau = -1.0 + 2.0 * np.sum(rho[:max_t + 1]) + rho[max_t + 1]
    tau = max(tau, 1.0 / math.log10(m * n))
    return {"mean": mean, "sd": sd, "rhat": rhat, "ess": m * n / tau, "lag": int(max_t), "margin": margin}


def rhat_ess_columns(x):
    """rhat_ess of every column of x [draws, chains, columns] (the layout of records and of diagnose_logs) -> dict of arrays."""
    x = np.asarray(x, dtype=np.float64)
    rows = [rhat_ess(x[:, :, j].T) for j in range(x.shape[2])]
    return {k: np.array([r[k] for r in rows]) for k in ("mean", "sd", "rhat", "ess", "lag", "margin")}


def _split(x):
    x = np.asarray(x, dtype=np.float64)
    if x.ndim == 1:
        x = x[None, :]
    M, Sd = x.shape
    if Sd < 4:
        raise RuntimeError("not enough data")
    n = Sd // 2
    return x, np.concatenate([x[:, :n], x[:, Sd - n:]], axis=1)


def rank_normal(v):
    """Phi^-1((r - 3/8) / (N + 1/4)) of the average ranks r (1-based, ties averaged) of the N values v, any shape.  The ratio and
    its complement (N + 5/8 - r) / (N + 1/4) have exact numerators; the smaller one goes to ndtri, so that the most extreme ranks
    of millions of draws keep full precision (ndtri(1 - eps) cannot)."""
    from scipy.special import ndtri
    from scipy.stats import rankdata
    v = np.asarray(v, dtype=np.float64)
    r = rankdata(v.ravel(), method="average").reshape(v.shape)
    N = v.size
    num, rest, den = r - 0.375, N + 0.625 - r, N + 0.25
    return np.where(num <= rest, ndtri(num / den), -ndtri(rest / den))


def quantile_linear(x, p):
    """np.quantile(x, p) with numpy's default "linear" method, restated step for step as K10 computes it: h = (N - 1) p,
    lo = floor(h), g = h - lo; a + (b - a) g when g < 0.5, else b - (b - a)(1 - g); NaN if x holds a NaN."""
    v = np.sort(np.asarray(x, dtype=np.float64).ravel())
    if np.isnan(v[-1]):
        return float("nan")
    N = v.size
    h = (N - 1) * p
    if h >= N - 1:
        a = b = v[-1]
        g = h + 1.0
    else:
        lo = math.floor(h)
        a, b, g = v[lo], v[lo + 1], h - lo
    d = b - a
    return float(b - d * (1.0 - g)) if g >= 0.5 else float(a + d * g)


def rank_rhat_ess(x):
    """Rank-normalised split R-hat and bulk and tail ESS of one column x [chains M, draws S] -> dict of floats median, q05, q95,
    rhat_bulk, rhat_tail, rhat_rank, ess_bulk, ess_tail and margin (host only: the smallest margin of the four rhat_ess calls).
    ArviZ's _rhat_rank, _ess_bulk and _ess_tail in the order they compute:

      1. n = S // 2, N = 2 M n; xs [M, 2n] = draws [0, n) and [S - n, S) of each chain (an odd S drops the middle draw, as
         rhat_ess does), so that rhat_ess(xs-shaped matrix) splits it into exactly these 2M split chains.  S < 4: RuntimeError.
      2. rhat_ess(x) non-finite, constant or stuck: every output NaN (+-inf draws included).
      3. z = Phi^-1((r - 3/8) / (N + 1/4)) of the average ranks r of xs among the N split draws (rank_normal);
         rhat_bulk, ess_bulk = rhat_ess(z).
      4. median = np.median(xs) ((a + b) / 2 of the middle two, N is even); f = |xs - median|; rhat_tail = rhat_ess(z of f)
         (NaN when f is constant, e.g. a 0/1 column split exactly in half).
      5. rhat_rank = max(rhat_bulk, rhat_tail), a NaN rhat_tail ignored (a stuck z of f gives +inf, which wins).
      6. q_p = np.quantile(x, p) over all M S draws (middle draws included; quantile_linear) for p = 0.05, 0.95; I_p = (xs <= q_p)
         as 0.0 / 1.0; ESS_p = rhat_ess(I_p)["ess"], N when I_p is constant (as ArviZ), NaN when it is stuck;
         ess_tail = min(ESS_0.05, ESS_0.95), NaN if either is.
    One chain (M = 1) is allowed, as in rhat_ess; ArviZ returns NaN for its rank R-hat instead."""
    x, xs = _split(x)
    nan = float("nan")
    keys = ("median", "q05", "q95", "rhat_bulk", "rhat_tail", "rhat_rank", "ess_bulk", "ess_tail")
    base = rhat_ess(x)
    if not math.isfinite(base["rhat"]):
        out = dict.fromkeys(keys, nan)
        out["margin"] = math.inf
        return out
    N = xs.size
    bulk = rhat_ess(rank_normal(xs))
    med = float(np.median(xs))
    tail = rhat_ess(rank_normal(np.abs(xs - med)))
    rb, rt = bulk["rhat"], tail["rhat"]
    margins = [bulk["margin"], tail["margin"]]
    q, ess = [], []
    for p in (0.05, 0.95):
        qp = quantile_linear(x, p)
        ind = rhat_ess((xs <= qp).astype(np.float64))
        const = math.isnan(ind["rhat"])
        ess.append(float(N) if const else ind["ess"])
        margins.append(ind["margin"])
        q.append(qp)
    return {"median": med, "q05": q[0], "q95": q[1], "rhat_bulk": rb, "rhat_tail": rt,
            "rhat_rank": rb if math.isnan(rt) else max(rb, rt), "ess_bulk": bulk["ess"],
            "ess_tail": nan if math.isnan(ess[0]) or math.isnan(ess[1]) else min(ess), "margin": min(margins)}


def rank_rhat_ess_columns(x):
    """rank_rhat_ess of every column of x [draws, chains, columns] -> dict of arrays."""
    x = np.asarray(x, dtype=np.float64)
    rows = [rank_rhat_ess(x[:, :, j].T) for j in range(x.shape[2])]
    return {k: np.array([r[k] for r in rows]) for k in rows[0]}


def flag(rhat, ess, lag, mean, rhat_max=1.01, ess_min=200.0):
    """ok | rhat | ess | rhat+ess | const | stuck | nonfinite of one column's diagnostics (lag is -1 for these three, but also for
    a regular column of fewer than 10 draws per chain, where Geyer's sequence stops at once)."""
    if not math.isfinite(mean):
        return "nonfinite"
    if rhat == math.inf:
        return "stuck"
    if math.isnan(rhat):
        return "const"
    bad = [tag for tag, b in (("rhat", rhat > rhat_max), ("ess", ess < ess_min)) if b]
    return "+".join(bad) if bad else "ok"


# ------------------------------------------------------------------------------------------ columns
def _bin_names(n_bins):
    return [("l_%d" % j) for j in range(n_bins)], [("m_%d" % j) for j in range(n_bins)], [("net_%d" % j) for j in range(n_bins)]


def diagnostic_columns(kind, n_bins, origin=0.0, genre=False):
    """(name, spec) of every diagnosed column of a sampler's records, in log column order (the spec as for
    Device.chain_diagnostics_device: a field, or (a, b, sign, add) = row[a] +- row[b] + add, one fp64 operation each).

      forward    posterior (= likelihood + prior), likelihood, prior, lambda_avg, mu_avg, K_l, K_m, gamma_rate_hp_BI,
                 gamma_rate_hp_D, poisson_rate_hp: the *_mcmc.log columns but it and the constants root_age and death_age.
                 Caveat: while record field [13] is set, the log writes the constant starting value as poisson_rate_hp
                 (forward.ChainLogWriter.write) where the record holds field [9]; logs and records agree on the other rows.
                 The per-bin marginal rates are not record fields: diagnose_records_device adds them from K5's matrices.
      trendrate  every column of the *.trendrate.log but it, then the net rate l_j - m_j per bin
      dd         every column of the DDRate log but it (genre_lik with genre, i.e. -m_birth 3), then the net rate per bin; the
                 parameters under the log's transforms (plotdd.column_specs: midpoint_x0 = x0 + origin, maxCarryingCap = L + div_0)
    """
    if kind == "forward":
        return list(FORWARD_COLS)
    if kind not in ("trendrate", "dd"):
        raise ValueError("kind must be 'forward', 'trendrate' or 'dd'")
    head = TR.REC_HEAD if kind == "trendrate" else DD.REC_HEAD
    log = TR.header(n_bins) if kind == "trendrate" else DD.header(n_bins, 3 if genre else 0)
    f = lambda s, j: head + s * n_bins + j
    cols = [("posterior", (1, 4, 1, 0.0)), (log[2], 1), (log[3], 2), (log[4], 3), (log[5], 4)]
    if kind == "trendrate":
        cols += [(p, 5 + i) for i, p in enumerate(TR.PARAMS)]
        series = 2
    else:
        cols += list(zip(PD.DD_PARAMS, PD.column_specs("dd", n_bins, origin)[-DD.NPAR:]))
        if genre:
            cols.append(("genre_lik", 16))
        series = 4
    tags = ["l_", "m_", "niche_", "nicheFrac_"][:series]
    cols += [("%s%d" % (tag, j), f(s, j)) for s, tag in enumerate(tags) for j in range(n_bins)]
    adq = 11 if kind == "trendrate" else 17
    cols += [(name, adq + i) for i, name in enumerate(("corr_coeff", "rsquared", "gelman_r2"))]
    cols += [("net_%d" % j, (f(0, j), f(1, j), -1, 0.0)) for j in range(n_bins)]
    return cols


# ------------------------------------------------------------------------------------------ results
@dataclass
class Diagnostics:
    kind: str
    names: list
    mean: np.ndarray
    sd: np.ndarray
    rhat: np.ndarray
    ess: np.ndarray
    lag: np.ndarray               # int, -1 for degenerate columns
    n_chains: int
    n_draws: int                  # per chain, after the burn-in
    # rank-normalised diagnostics (rank_rhat_ess; None unless asked for)
    median: np.ndarray = None
    q05: np.ndarray = None
    q95: np.ndarray = None
    rhat_bulk: np.ndarray = None
    rhat_tail: np.ndarray = None
    rhat_rank: np.ndarray = None
    ess_bulk: np.ndarray = None
    ess_tail: np.ndarray = None

    @property
    def mcse(self):
        with np.errstate(invalid="ignore", divide="ignore"):
            return self.sd / np.sqrt(self.ess)

    def flags(self, rhat_max=1.01, ess_min=200.0):
        return [flag(r, e, l, m, rhat_max, ess_min) for r, e, l, m in zip(self.rhat, self.ess, self.lag, self.mean)]

    def rank_flags(self, rhat_max=1.01, ess_min=200.0):
        """The flags of the rank diagnostics, in the vocabulary of FLAGS: const, stuck and nonfinite as flags() gives them; else
        rhat when rhat_rank > rhat_max, ess when min(ess_bulk, ess_tail) < ess_min or ess_tail is NaN."""
        out = []
        for fl, rr, eb, et in zip(self.flags(rhat_max, ess_min), self.rhat_rank, self.ess_bulk, self.ess_tail):
            if fl in ("const", "stuck", "nonfinite"):
                out.append(fl)
                continue
            bad = [tag for tag, b in (("rhat", rr > rhat_max), ("ess", math.isnan(et) or min(eb, et) < ess_min)) if b]
            out.append("+".join(bad) if bad else "ok")
        return out

    def write_rank_tsv(self, path, rhat_max=1.01, ess_min=200.0):
        """column median q05 q95 rhat_rank rhat_bulk rhat_tail ess_bulk ess_tail flag: one row per column, values as repr."""
        with open(path, "w") as fh:
            fh.write("column\tmedian\tq05\tq95\trhat_rank\trhat_bulk\trhat_tail\tess_bulk\tess_tail\tflag\n")
            cols = (self.median, self.q05, self.q95, self.rhat_rank, self.rhat_bulk, self.rhat_tail, self.ess_bulk, self.ess_tail)
            for i, fl in enumerate(self.rank_flags(rhat_max, ess_min)):
                fh.write("\t".join([self.names[i]] + [repr(float(v[i])) for v in cols] + [fl]) + "\n")
        return path

    def write_tsv(self, path, rhat_max=1.01, ess_min=200.0):
        """column mean sd rhat ess mcse lag flag: one row per column, values as repr (nan, inf)."""
        with open(path, "w") as fh:
            fh.write("column\tmean\tsd\trhat\tess\tmcse\tlag\tflag\n")
            for i, fl in enumerate(self.flags(rhat_max, ess_min)):
                vals = [repr(float(v[i])) for v in (self.mean, self.sd, self.rhat, self.ess, self.mcse)]
                fh.write("\t".join([self.names[i]] + vals + [str(int(self.lag[i])), fl]) + "\n")
        return path


def _pack(kind, names, parts, n_chains, n_draws, rank_parts=None):
    cat = {k: np.concatenate([p[k].cpu().numpy() for p in parts]) for k in ("mean", "sd", "rhat", "ess", "lag")}
    d = Diagnostics(kind, list(names), cat["mean"], cat["sd"], cat["rhat"], cat["ess"], cat["lag"].astype(np.int64), n_chains, n_draws)
    if rank_parts is not None:
        for k in E.RANK_FIELDS:
            setattr(d, k, np.concatenate([p[k].cpu().numpy() for p in rank_parts]))
    return d


# ------------------------------------------------------------------------------------------ device records
def cold_records_device(records, ladder, col):
    """engine.cold_records on the device: [S, n_chains, w] -> [S, n_chains // ladder, w], per ladder and sample the first member
    with beta = 1 (a copy of 1/ladder of the records).  ValueError when a ladder has none."""
    import torch
    Sn, nc, w = records.shape
    r = records.reshape(Sn, nc // ladder, ladder, w)
    hit = r[..., col] == 1.0
    if not bool(hit.any(dim=2).all()):
        raise ValueError("a ladder has no chain at beta = 1")
    idx = hit.to(torch.int8).argmax(dim=2)
    return torch.gather(r, 2, idx[:, :, None, None].expand(Sn, nc // ladder, 1, w))[:, :, 0, :]


def diagnose_records_device(dev, records, kind, n_bins, burnin=0.2, ladder=1, origin=0.0, bins=True, genre=False, rank=False):
    """K9 on a float64 CUDA tensor of records [n_samples, n_chains * ladder, rec_doubles] of K3 ("forward"), K6 ("trendrate") or
    K7 ("dd"): the columns of diagnostic_columns after removing the burn-in of every chain -> Diagnostics.  ladder > 1: tempered
    ladders, diagnosed over their cold members (K6 / K7: K9 picks them; K3: gathered on the device first).  origin: the run's
    origin (DDRate's midpoint_x0; RJMCMC: the first bin edge, the run's start time).  bins (forward): the per-bin birth, death and
    net marginal rates l_j, m_j, net_j of n_bins unit bins from origin, from lr_marginal_rates matrices in chunks of at most 1 GB,
    as summary.summarize_records_device expands them.  rank: the rank-normalised diagnostics too (K10 on the same columns, the
    Diagnostics fields median .. ess_tail)."""
    b0 = S.burnin_index(records.shape[0], burnin)
    post = records[b0:]
    cols = diagnostic_columns(kind, n_bins, origin, genre)
    names, specs = [c[0] for c in cols], [c[1] for c in cols]
    n_chains = records.shape[1] // ladder
    if kind != "forward":
        beta = TR.REC_BETA if kind == "trendrate" else DD.REC_BETA
        out = dev.chain_diagnostics_device(post, specs, ladder, beta if ladder > 1 else -1)
        rk = [dev.rank_diagnostics_device(post, specs, ladder, beta if ladder > 1 else -1)] if rank else None
        return _pack(kind, names, [out], n_chains, post.shape[0], rk)
    if ladder > 1:
        post = cold_records_device(post, ladder, E.REC_BETA)
    post = post.contiguous()
    parts = [dev.chain_diagnostics_device(post, specs)]
    rparts = [dev.rank_diagnostics_device(post, specs)] if rank else None
    if bins:
        import torch
        Sn, M = post.shape[0], post.shape[1]
        bnames, dnames, nnames = _bin_names(n_bins)
        per = {"l": [], "m": [], "net": []}
        rper = {"l": [], "m": [], "net": []}
        for _, cnt, mb, md in S.marginal_chunks(dev, post, origin, n_bins):
            mat = torch.cat([mb, md], dim=1).reshape(Sn, M, 2 * cnt)
            del mb, md
            mspecs = list(range(2 * cnt)) + [(j, cnt + j, -1) for j in range(cnt)]
            r = dev.chain_diagnostics_device(mat, mspecs)
            rr = dev.rank_diagnostics_device(mat, mspecs) if rank else None
            for k, sl in (("l", slice(0, cnt)), ("m", slice(cnt, 2 * cnt)), ("net", slice(2 * cnt, 3 * cnt))):
                per[k].append({f: v[sl] for f, v in r.items()})
                if rank:
                    rper[k].append({f: v[sl] for f, v in rr.items()})
            del mat
        parts += per["l"] + per["m"] + per["net"]
        if rank:
            rparts += rper["l"] + rper["m"] + rper["net"]
        names += bnames + dnames + nnames
    return _pack(kind, names, parts, n_chains, post.shape[0], rparts)


# ------------------------------------------------------------------------------------------ logs
def log_kind(path):
    """"forward" for an RJMCMC *_mcmc.log, else plotdd.log_kind ("trendrate", "dd" or None)."""
    if os.path.basename(path).endswith("mcmc.log"):
        return "forward"
    return PD.log_kind(path)


def _forward_log(path, burnin, bins):
    head = open(path).readline().rstrip("\r\n").split("\t")
    tbl = np.loadtxt(path, delimiter="\t", skiprows=1, ndmin=2)
    idx = {h: i for i, h in enumerate(head)}
    b0 = S.burnin_index(tbl.shape[0], burnin)
    col = lambda name: tbl[b0:, idx[name]]
    names = [c[0] for c in FORWARD_COLS]
    cols = [col(nm) for nm in names]
    edges = None
    if bins:
        root_age, death_age = float(np.mean(tbl[:, idx["root_age"]])), float(np.mean(tbl[:, idx["death_age"]]))
        edges = np.arange(root_age, death_age)
        mats = []
        for tag in ("sp_rates.log", "ex_rates.log"):
            rates, shifts, K = S._read_ragged(path.replace("mcmc.log", tag))
            k0 = S.burnin_index(len(K), burnin)
            mats.append(S.marginal_matrix(rates[k0:], shifts[k0:], K[k0:], edges))
        nb = len(edges) - 1
        cols += [mats[0][:, j] for j in range(nb)] + [mats[1][:, j] for j in range(nb)] + [mats[0][:, j] - mats[1][:, j] for j in range(nb)]
        names += sum(_bin_names(nb), [])
    return names, np.stack(cols, axis=1), edges


def _sibling_log(path, kind, burnin):
    head, n_bins, col = PD.read_log(path, burnin)
    names = [c[0] for c in diagnostic_columns(kind, n_bins, 0.0, "genre_lik" in head)]
    return names, np.stack([col(nm) for nm in names], axis=1), None


def log_draws(paths, burnin=0.2, bins=True, note=print):
    """The post-burn-in rows of sample logs of one kind (one log per chain) as (kind, names, x [draws, chains, columns]): the
    diagnosed columns in diagnostic_columns order, RJMCMC's per-bin marginal rates (summary.marginal_matrix, bins from the
    logged root_age and death_age) appended with `bins`, the net rate l_j - m_j formed as the kernel does.  Chains of different
    lengths are cut to the shortest (said through `note`)."""
    paths = [paths] if isinstance(paths, str) else list(paths)
    kinds = {log_kind(p) for p in paths}
    if len(kinds) != 1 or None in kinds:
        raise ValueError("diagnose_logs needs sample logs of one kind (*_mcmc.log, *.trendrate.log or DDRate logs)")
    kind = kinds.pop()
    blocks = [_forward_log(p, burnin, bins) if kind == "forward" else _sibling_log(p, kind, burnin) for p in paths]
    if len({tuple(b[0]) for b in blocks}) != 1:
        raise ValueError("the logs have different columns (bins)")
    lens = [b[1].shape[0] for b in blocks]
    if len(set(lens)) > 1:
        note("chains of %d to %d draws after the burn-in: every chain cut to the shortest" % (min(lens), max(lens)))
    k = min(lens)
    return kind, blocks[0][0], np.stack([b[1][:k] for b in blocks], axis=1)


def diagnose_logs(paths, burnin=0.2, device=None, bins=True, note=print, rank=False):
    """K9 on the post-burn-in rows of sample logs of one kind, one log per chain (log_draws) -> Diagnostics.  device: an
    engine.Device (None: device 0).  rank: the rank-normalised diagnostics too (K10)."""
    import torch
    kind, names, x = log_draws(paths, burnin, bins, note)
    dev = device if device is not None else E.Device(0)
    t = torch.from_numpy(np.ascontiguousarray(x)).to(torch.device("cuda", dev.index))
    out = dev.chain_diagnostics_device(t, list(range(x.shape[2])))
    rk = [dev.rank_diagnostics_device(t, list(range(x.shape[2])))] if rank else None
    return _pack(kind, names, [out], x.shape[1], x.shape[0], rk)


def find_logs(log_dir):
    """{kind: sorted sample logs} of a directory: *_mcmc.log as summary.main finds them, TrendRate / DDRate logs as
    plotdd.find_logs (combined outputs excluded)."""
    import glob
    out = {}
    fw = sorted(f for f in glob.glob(os.path.join(log_dir, "*mcmc.log")) if not os.path.basename(f).startswith("COMBINED"))
    if fw:
        out["forward"] = fw
    for k, v in PD.find_logs(log_dir).items():
        out[k] = v
    return out
