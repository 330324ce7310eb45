"""Posterior summaries of RJMCMC output: number-of-shifts posterior, per-bin marginal rates with 95 % HPD, shift
frequencies with Bayes-factor thresholds, net rate -- the numbers plotRJforward.v3.py derives from the four log files
(plotRJforward.v3.py:92-139, :142-196, :234-262, :292-305), and its log combiner (:307-350, utilities/logCombiner.py).

SURVEY 8(f-1/f-2): host-side consumers of the hot path's output.  Everything is vectorised over samples (the reference
parses and histograms one text row at a time), works either on the log files or directly on the sample records a run
delivers (no text round trip for thousands of chains), and writes an `_RTT_plots.r` file that defines the same R
variables (unique/counts, time, birth_rate, birth_minHPD, ..., net_rate, ...) followed by plain base-R plots.
"""
from __future__ import annotations

import glob
import os
import sys
from dataclasses import dataclass, field

import numpy as np

from . import engine as E


# ------------------------------------------------------------------------------------------ building blocks
def burnin_index(n, burnin):
    """First kept sample: a fraction < 1 of the rows, never more than 90 % (plotRJforward.v3.py:107-108, :293)."""
    return min(int(burnin * n), int(0.9 * n)) if burnin < 1 else int(burnin)


def hpd_columns(x, level=0.95):
    """Narrowest interval holding `level` of the samples, per column (calcHPD, plotRJforward.v3.py:12-28):
    x [n, m] -> (lo [m], hi [m])."""
    x = np.sort(np.asarray(x, dtype=np.float64), axis=0)
    n = x.shape[0]
    n_in = int(round(level * n))
    if n_in < 2:
        raise RuntimeError("not enough data")
    width = x[n_in - 1:] - x[:n - n_in + 1]
    i = np.argmin(width, axis=0)                      # first narrowest window, as the reference's strict '<'
    cols = np.arange(x.shape[1])
    return x[i, cols], x[i + n_in - 1, cols]


def marginal_matrix(rates, shifts, K, edges):
    """Per-bin rate of every sample.  rates [n, Kmax], shifts [n, Kmax-1] (padded), K [n] number of rates, edges: the
    histogram edges np.arange(root_age, death_age).  Bin j takes rates[#shifts falling in bins 0..j] -- np.histogram
    semantics (half-open bins, last one closed, shifts outside the edges ignored), plotRJforward.v3.py:111-121.
    Oldest bin first (the reference stores the reverse and reverses again on output)."""
    rates, shifts, K = np.asarray(rates, float), np.asarray(shifts, float), np.asarray(K)
    n, nb = rates.shape[0], len(edges) - 1
    valid = np.arange(shifts.shape[1])[None, :] < (K[:, None] - 1)
    s = np.where(valid, shifts, np.inf)
    inside = s >= edges[0]
    upper = edges[1:][None, None, :]
    below = (s[:, :, None] < upper)
    below[:, :, -1] = s <= edges[-1]                  # the last bin of np.histogram is closed
    idx = np.sum(below & inside[:, :, None], axis=1)  # [n, nb] cumulative number of shifts
    return np.take_along_axis(rates, idx, axis=1)


def shift_histogram(shifts, K, edges):
    """Counts of sampled shift times per bin over all samples (plotRJforward.v3.py:166-176)."""
    valid = np.arange(shifts.shape[1])[None, :] < (np.asarray(K)[:, None] - 1)
    return np.histogram(np.asarray(shifts)[valid], bins=edges)[0]


def prior_shift_frequency(t_start, t_end, edges, n_sim=100000, seed=0):
    """Expected per-bin frequency of a shift under the prior (get_prior_shift, plotRJforward.v3.py:58-89): Poisson rate
    ~ Gamma(2, 1), K ~ Poisson | K > 0, K-1 shift times uniform inside the window shrunk by 1 at both ends, configurations
    with two times closer than 1 discarded.  Returns (mean frequency, bf2, bf6).  Seeded (the reference is not)."""
    g = np.random.default_rng(seed)
    lam = g.gamma(2.0, 1.0, n_sim)
    k = g.poisson(lam)
    ok = k > 0
    while not ok.all():                               # first positive draw of the reference's 1000-long vector
        redo = ~ok
        k[redo] = g.poisson(lam[redo])
        ok = k > 0
    lo, hi = min(t_end - 1, t_start + 1), max(t_end - 1, t_start + 1)
    kept, times = 0, []
    for kk in np.unique(k):
        m = int(np.sum(k == kk))
        if kk == 1:
            if abs(t_end - t_start) >= 1:
                kept += m
            continue
        sh = g.uniform(lo, hi, (m, kk - 1))
        fr = np.sort(np.concatenate([np.full((m, 1), min(t_start, t_end)), sh, np.full((m, 1), max(t_start, t_end))], axis=1), axis=1)
        good = np.min(np.diff(fr, axis=1), axis=1) >= 1
        kept += int(good.sum())
        times.append(sh[good].ravel())
    times = np.concatenate(times) if times else np.empty(0)
    prior = float(np.mean(np.histogram(times, bins=edges)[0] / max(kept, 1)))
    bf = lambda thr: (np.exp(thr / 2) * prior / (1 - prior)) / (np.exp(thr / 2) * prior / (1 - prior) + 1)   # calcBF :53-55
    return prior, float(bf(2)), float(bf(6))


# ------------------------------------------------------------------------------------------ containers
@dataclass
class SideSummary:
    time: np.ndarray              # bin mid-points
    mean: np.ndarray              # per-bin mean rate
    hpd_lo: np.ndarray
    hpd_hi: np.ndarray
    shift_freq: np.ndarray        # per-bin frequency of a sampled shift
    n_samples: int
    k_values: np.ndarray
    k_counts: np.ndarray
    marginal: np.ndarray = field(repr=False, default=None)   # [n_samples, n_bins]


@dataclass
class Summary:
    name: str
    root_age: float
    death_age: float
    birth: SideSummary
    death: SideSummary
    net_mean: np.ndarray
    net_lo: np.ndarray
    net_hi: np.ndarray
    prior_freq: float = None
    bf2: float = None
    bf6: float = None
    div: np.ndarray = None        # [n_bins, 3] of div.log, if known

    def flags(self, side: SideSummary):
        """(BF2, BF6) vectors of plotRJforward.v3.py:185-193: the mean rate where the shift frequency is in [bf2, bf6) / >= bf6."""
        f = side.shift_freq
        b2 = np.where((f >= self.bf2) & (f < self.bf6), side.mean, np.nan)
        b6 = np.where(f >= self.bf6, side.mean, np.nan)
        return b2, b6


def _side(rates, shifts, K, edges, k_all):
    M = marginal_matrix(rates, shifts, K, edges)
    lo, hi = hpd_columns(M)
    vals, counts = np.unique(k_all, return_counts=True)
    return SideSummary(time=(edges - 0.5)[1:], mean=M.mean(0), hpd_lo=lo, hpd_hi=hi,
                       shift_freq=shift_histogram(shifts, K, edges) / float(len(K)), n_samples=len(K),
                       k_values=vals.astype(float), k_counts=counts, marginal=M)


def _finish(name, root_age, death_age, b, d, bf_seed, div=None):
    n = min(b.marginal.shape[0], d.marginal.shape[0])
    net = b.marginal[:n] - d.marginal[:n]
    nlo, nhi = hpd_columns(net)
    out = Summary(name, root_age, death_age, b, d, net.mean(0), nlo, nhi, div=div)
    if bf_seed is not None:
        edges = np.arange(root_age, death_age)
        out.prior_freq, out.bf2, out.bf6 = prior_shift_frequency(death_age, root_age, edges, seed=bf_seed)
    return out


# ------------------------------------------------------------------------------------------ from records / from logs
def summarize_records(records, start_time, end_time, burnin=0.2, name="chains", bf_seed=0, div=None):
    """records [n_samples, n_chains, 144] (or [n, 144]) of cold chains -> Summary, all chains pooled after removing the
    burn-in of each (what `-combine 1` does to log files, plotRJforward.v3.py:307-350)."""
    r = np.asarray(records)
    if r.ndim == 2:
        r = r[:, None, :]
    b0 = burnin_index(r.shape[0], burnin)
    r = r[b0:].reshape(-1, r.shape[-1])
    edges = np.arange(start_time, end_time)
    KL, KM = r[:, E.REC_KL].astype(int), r[:, E.REC_KM].astype(int)
    b = _side(r[:, E.REC_L:E.REC_L + E.LR_KMAX], r[:, E.REC_TL + 1:E.REC_TL + E.LR_KMAX], KL, edges, KL)
    d = _side(r[:, E.REC_M:E.REC_M + E.LR_KMAX], r[:, E.REC_TM + 1:E.REC_TM + E.LR_KMAX], KM, edges, KM)
    return _finish(name, float(start_time), float(end_time), b, d, bf_seed, div)


def hpd_device(x, level=0.95):
    """hpd_columns on the device: x a CUDA tensor [n, m] -> (lo [m], hi [m]) CUDA tensors.  Same rule as calcHPD
    (plotRJforward.v3.py:12-28): the FIRST narrowest window of round(level n) sorted values (torch.argmin returns the first
    minimum).  Sorting is torch's (device plumbing); the values are the kernel's."""
    import torch
    s, _ = torch.sort(x, dim=0)
    n = s.shape[0]
    n_in = int(round(level * n))
    if n_in < 2:
        raise RuntimeError("not enough data")
    width = s[n_in - 1:] - s[:n - n_in + 1]
    i = torch.argmin(width, dim=0, keepdim=True)
    return s.gather(0, i)[0], s.gather(0, i + (n_in - 1))[0]


def marginal_chunks(dev, records, first_edge, n_bins, budget=1 << 30):
    """K5's per-sample marginal rates of device-resident records [..., 144] (lr_marginal_rates), a range of bins at a time so
    that each matrix takes at most `budget` bytes (one bin at least): yields (lo, cnt, birth, death), birth and death float64
    CUDA tensors [n_records, cnt] for the bins [lo, lo + cnt).  A caller that deletes a chunk before taking the next holds one."""
    n = records.numel() // E.LR_REC_DOUBLES
    step = max(1, min(n_bins, int(budget // (8 * max(n, 1)))))
    for lo in range(0, n_bins, step):
        cnt = min(step, n_bins - lo)
        yield (lo, cnt) + tuple(dev.marginal_rates_device(records, first_edge, n_bins, lo, cnt))


def summarize_records_device(dev, records, start_time, end_time, burnin=0.2, hpd=False, hpd_bytes=1 << 30):
    """Means, shift frequencies and number-of-rates counts of device-resident records (a float64 CUDA tensor
    [n_samples, n_chains, 144]) without bringing them to the host (K5, lr_summarize_records).  With ``hpd`` the 95 % HPD
    intervals of the birth, death and net rates as well: the per-sample matrix is expanded on the device a range of bins at a
    time (lr_marginal_rates; at most ``hpd_bytes`` per matrix) and its columns are sorted there.  Returns a dict of NumPy arrays."""
    b0 = burnin_index(records.shape[0], burnin)
    post = records[b0:].contiguous()
    nb = len(np.arange(start_time, end_time)) - 1
    sr, sc, kc, n = dev.summarize_records_device(post, start_time, nb)
    sr, sc, kc = sr.cpu().numpy(), sc.cpu().numpy(), kc.cpu().numpy()
    out = {"n_samples": n, "time": (np.arange(start_time, end_time) - 0.5)[1:]}
    for side, name in ((0, "birth"), (1, "death")):
        k = np.nonzero(kc[side])[0]
        out[name] = {"mean": sr[side] / n, "shift_freq": sc[side] / float(n), "k_values": (k + 1).astype(float), "k_counts": kc[side][k]}
    out["net_mean"] = out["birth"]["mean"] - out["death"]["mean"]
    if hpd:
        import torch
        parts = {"birth": [], "death": [], "net": []}
        for _, _, mb, md in marginal_chunks(dev, post, start_time, nb, hpd_bytes):
            for name, m in (("birth", mb), ("death", md), ("net", mb - md)):
                parts[name].append(torch.stack(hpd_device(m)))
            del mb, md
        for name in parts:
            lohi = torch.cat(parts[name], dim=1).cpu().numpy()
            tgt = out[name] if name != "net" else out
            tgt["hpd_lo" if name != "net" else "net_lo"], tgt["hpd_hi" if name != "net" else "net_hi"] = lohi[0], lohi[1]
    return out


def _read_ragged(path):
    """sp_rates.log / ex_rates.log: rows `rates... shifts...` -> padded (rates, shifts, K)."""
    rows = [np.array(l.split(), dtype=np.float64) for l in open(path) if l.strip()]
    n, kmax = len(rows), max((len(r) + 1) // 2 for r in rows)
    rates, shifts, K = np.zeros((n, kmax)), np.zeros((n, max(kmax - 1, 1))), np.zeros(n, dtype=int)
    for i, r in enumerate(rows):
        k = (len(r) + 1) // 2
        K[i] = k
        rates[i, :k] = r[:k]
        shifts[i, :k - 1] = r[k:]
    return rates, shifts, K


def summarize_logs(mcmc_log, burnin=0.2, bf_seed=0):
    """One `*_mcmc.log` and its three siblings -> Summary (plot_marginal_rates' per-file body, plotRJforward.v3.py:376-419)."""
    head = open(mcmc_log).readline().split()
    tbl = np.loadtxt(mcmc_log, skiprows=1, ndmin=2)
    root_age = float(np.mean(tbl[:, head.index("root_age")]))
    death_age = float(np.mean(tbl[:, head.index("death_age")]))
    edges = np.arange(root_age, death_age)
    sides = []
    for tag, col in (("sp_rates.log", "K_l"), ("ex_rates.log", "K_m")):
        rates, shifts, K = _read_ragged(mcmc_log.replace("mcmc.log", tag))
        b0 = burnin_index(len(K), burnin)
        kcol = tbl[burnin_index(len(tbl), burnin):, head.index(col)]
        sides.append(_side(rates[b0:], shifts[b0:], K[b0:], edges, kcol))
    div_path = mcmc_log.replace("mcmc.log", "div.log")
    div = np.loadtxt(div_path, skiprows=1, ndmin=2) if os.path.exists(div_path) else None
    return _finish(os.path.splitext(os.path.basename(mcmc_log))[0], root_age, death_age, sides[0], sides[1], bf_seed, div)


def combine_logs(mcmc_files, out_dir, burnin=0.2, thin=1, stem="COMBINED"):
    """Concatenate the post-burn-in rows of several chains into <stem>_{mcmc,sp_rates,ex_rates,div}.log
    (plotRJforward.v3.py:307-350; utilities/logCombiner.py, thinner.py): `it` renumbered from 0, div.log averaged."""
    mcmc_files = sorted(mcmc_files)
    header, rows = None, []
    for f in mcmc_files:
        lines = open(f).read().splitlines()
        header = lines[0]
        body = lines[1:]
        rows += body[int(burnin * len(body)):][::thin]
    with open(os.path.join(out_dir, stem + "_mcmc.log"), "w") as o:
        o.write(header + "\n")
        for i, l in enumerate(rows):
            o.write("\t".join([str(i)] + l.split("\t")[1:]) + "\n")
    for tag in ("sp_rates.log", "ex_rates.log"):
        rows = []
        for f in mcmc_files:
            body = [l for l in open(f.replace("mcmc.log", tag)).read().splitlines()]
            rows += body[int(burnin * len(body)):][::thin]
        with open(os.path.join(out_dir, stem + "_" + tag), "w") as o:
            o.write("\n".join(rows) + "\n")
    div = np.mean([np.loadtxt(f.replace("mcmc.log", "div.log"), skiprows=1, ndmin=2) for f in mcmc_files], axis=0)
    with open(os.path.join(out_dir, stem + "_div.log"), "w") as o:
        o.write("sp_events\tex_events\tbr_length\n")
        for a, b, c in div:
            o.write("%s\t%s\t%s\n" % (repr(float(a)), repr(float(b)), repr(float(c))))
    return os.path.join(out_dir, stem + "_mcmc.log")


# ------------------------------------------------------------------------------------------ imputation replicates
ENVELOPE_ROWS = ("ed_mean", "ed_min", "ed_max", "eb_mean", "eb_min", "eb_max", "nd_mean", "nd_min", "nd_max")


def imputation_envelope(div_tables):
    """utilities/imputation_averager.py:23-61 on stacked div.log tables [n_rep, n_bins, 3] (sp_events, ex_events, br_length):
    mean / min / max over the replicates of the empirical death rate ex/br, the empirical birth rate sp/br and the net
    diversity br.  Returns a dict of nine [n_bins] vectors (ENVELOPE_ROWS).  Host restatement; the device path is
    engine.Device.imputation_envelope_device on K1's output."""
    t = np.asarray(div_tables, dtype=np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        ed, eb, nd = t[:, :, 1] / t[:, :, 2], t[:, :, 0] / t[:, :, 2], t[:, :, 2]
    out = {}
    for tag, m in (("ed", ed), ("eb", eb), ("nd", nd)):
        out[tag + "_mean"], out[tag + "_min"], out[tag + "_max"] = m.mean(axis=0), m.min(axis=0), m.max(axis=0)
    return out


def _averager_r_vec(name, v):
    """print_R_vec of utilities/imputation_averager.py:8-21 (its own variant: no NA for vectors shorter than three)."""
    if len(v) == 0:
        return "%s=c()" % name
    if len(v) == 1:
        return "%s=c(%s)" % (name, v[0])
    if len(v) == 2:
        return "%s=c(%s,%s)" % (name, v[0], v[1])
    w = ["NA" if np.isnan(x) else x for x in v]
    return "%s=c(%s, " % (name, w[0]) + "".join("%s," % x for x in w[1:-1]) + "%s)" % w[-1]


def format_imputation_envelope(env):
    """The text utilities/imputation_averager.py prints (:39-61), byte for byte (np.set_printoptions(suppress=True, precision=3)
    for the three net-diversity arrays, as :5-6)."""
    lines = []
    for title, tag in (("EMPIRICAL DEATH", "ed"), ("EMPIRICAL BIRTH", "eb")):
        lines.append(title)
        for k in ("mean", "min", "max"):
            lines.append(_averager_r_vec("%s_%s" % (tag, k), env["%s_%s" % (tag, k)]))
    lines.append("NET DIVERSITY")
    with np.printoptions(suppress=True, precision=3):
        for k in ("mean", "min", "max"):
            lines.append(str(env["nd_" + k]))
    return "\n".join(lines) + "\n"


def imputation_average_logs(log_dir):
    """The whole utility: every *div.log under `log_dir` (glob order, like the reference) -> the printed text."""
    files = glob.glob(log_dir + "/*div.log")
    if not files:
        raise SystemExit("no *div.log under " + log_dir)
    tables = [np.loadtxt(f, skiprows=1, ndmin=2) for f in files]
    return format_imputation_envelope(imputation_envelope(np.stack(tables)))


# ------------------------------------------------------------------------------------------ R output
def r_vec(name, v):
    """`name=c(a, b,c,...)` exactly as print_R_vec formats it (plotRJforward.v3.py:31-50), NaN -> NA."""
    v = list(v)
    f = lambda x: "NA" if isinstance(x, float) and np.isnan(x) else str(x)
    if len(v) == 0:
        return "%s=c()" % name
    if len(v) <= 2:
        return "%s=c(%s)" % (name, ",".join(str(x) for x in v))
    body = f(v[0]) + ", " + ",".join(f(x) for x in v[1:])
    if all(f(x) == "NA" for x in v):
        return "%s=as.numeric(c(%s))" % (name, body)
    return "%s=c(%s)" % (name, body)


def write_r(summaries, path, TBP=False):
    """<path>: R script with the reference's variable names; plots in base R."""
    out = ["pdf(file='%s',width=12, height=8)" % (os.path.splitext(path)[0] + ".pdf"), "par(mfrow=c(2,4))", "library(scales)"]
    for s in summaries:
        off = s.death_age if TBP else 0.0
        out.append("###%s###" % s.name)
        for side, prefix, col in ((s.birth, "birth", "#4c4cec"), (s.death, "death", "#e34a33")):
            out += ["#Number Shifts", r_vec("unique", [np.float64(x) for x in side.k_values]), r_vec("counts", [int(x) for x in side.k_counts]),
                    "plot(unique,counts,type = 'h', xlim = c(0,%s), ylab = 'Frequency', xlab = 'n. shifts',lwd=5,col='%s')"
                    % (max(s.birth.k_values.max(), s.death.k_values.max()) + 1, col),
                    "#%s rate Plot" % prefix.capitalize(), r_vec("time", [np.float64(x) for x in side.time - off]),
                    r_vec(prefix + "_rate", [np.float64(x) for x in side.mean]), r_vec(prefix + "_minHPD", [np.float64(x) for x in side.hpd_lo]),
                    r_vec(prefix + "_maxHPD", [np.float64(x) for x in side.hpd_hi]),
                    "plot(time,%s_rate,type='n',ylim=c(0,%s),ylab='%s rate',xlab='Time',main='%s')" % (prefix, 1.1 * np.nanmax(side.hpd_hi), prefix.capitalize(), s.name),
                    "polygon(c(time, rev(time)), c(%s_maxHPD, rev(%s_minHPD)), col = alpha('%s',0.3), border = NA)" % (prefix, prefix, col),
                    "lines(time,%s_rate, col = '%s', lwd=2)" % (prefix, col),
                    "#Frequency of shifts", r_vec(prefix + "_counts", [np.float64(x) for x in side.shift_freq]),
                    "plot(time,%s_counts,type = 'h', ylim=c(0,%s), ylab = 'Frequency of rate shift', xlab = 'Time',lwd=5,col='%s')"
                    % (prefix, max(float(side.shift_freq.max()), 0.2), col)]
            if s.bf2 is not None:
                b2, b6 = s.flags(side)
                out += ["bf2 = %s" % s.bf2, "bf6 = %s" % s.bf6, "abline(h=bf2, lty=2)", "abline(h=bf6, lty=2)",
                        r_vec(prefix + "_BF2", [float(x) for x in b2]), r_vec(prefix + "_BF6", [float(x) for x in b6])]
            if prefix == "birth":
                out += ["#Net Rate", r_vec("net_rate", [np.float64(x) for x in s.net_mean]), r_vec("net_minHPD", [np.float64(x) for x in s.net_lo]),
                        r_vec("net_maxHPD", [np.float64(x) for x in s.net_hi]),
                        "plot(time,net_rate,type='n',ylim=c(%s,%s),ylab='Net Rate',xlab='Time')" % (min(0, 1.1 * np.nanmin(s.net_lo)), 1.1 * np.nanmax(s.net_hi)),
                        "polygon(c(time, rev(time)), c(net_maxHPD, rev(net_minHPD)), col = alpha('#32CD32',0.3), border = NA)",
                        "lines(time,net_rate, col = '#32CD32', lwd=2)", "abline(h=0,lty=2)"]
        if s.div is not None:
            out += ["#Net Diversity", r_vec("net_diversity", [np.float64(x) for x in s.div[:, 2]]),
                    "plot(time,net_diversity,type = 'l', ylab = 'Net Diversity', xlab = 'Time',lwd=2, col= '#32CD32')"]
    out.append("n <- dev.off()")
    with open(path, "w") as fh:
        fh.write("\n".join(out) + "\n")
    return path


def main(argv=None):
    import argparse
    p = argparse.ArgumentParser(prog="plotRJforward")          # the reference's options, plotRJforward.v3.py:433-437
    p.add_argument('input_data', metavar='<path to log files>', type=str)
    p.add_argument('-combine', metavar='0', type=int, default=0)
    p.add_argument('-logT', metavar='1', type=int, default=0)
    p.add_argument('-burnin', metavar='.2', type=float, default=.2)
    p.add_argument('-TBP', default=False, action='store_true')
    p.add_argument('-imputations', metavar='0', type=int, default=0,
                   help='1: print the envelopes of the empirical rates and net diversity over the *div.log files of the directory '
                        '(utilities/imputation_averager.py) and stop')
    a = p.parse_args(argv)
    if a.imputations == 1:
        sys.stdout.write(imputation_average_logs(a.input_data))
        return
    files = sorted(f for f in glob.glob("%s/*mcmc.log" % a.input_data) if not os.path.basename(f).startswith("COMBINED"))
    if not files:
        raise SystemExit("no *mcmc.log under " + a.input_data)
    print("found", len(files), "log files...\n")
    burnin = a.burnin
    if a.combine == 1:
        files, burnin = [combine_logs(files, a.input_data, burnin)], 0
    sums = [summarize_logs(f, burnin) for f in files]
    out = (os.path.join(a.input_data, "COMBINED") if a.combine == 1 else files[0].replace("_mcmc.log", "")) + "_RTT_plots.r"
    write_r(sums, out, TBP=a.TBP)
    print("Plots saved in %s" % out)


if __name__ == "__main__":
    main()
