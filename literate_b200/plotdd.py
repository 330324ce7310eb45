"""Posterior summaries of TrendRate and DDRate runs (the step the reference leaves to plotDD.py): per bin the mean and 95 % HPD
band of the birth, death and net rate (DDRate: also niche and niche fraction), and the mean and HPD interval of every model
parameter under the log header's names.  Three ways in, one result (PlotSummary):

  summarize_records         host restatement on sample records (numpy, summary.hpd_columns) -- the reference of the tests
  summarize_records_device  the same from device-resident records with K8 (lr_column_hpd): the records are never copied
  summarize_logs            from the *.trendrate.log / DDRate *.log files the command lines write

Burn-in is removed per chain (per file), then the chains are pooled, as summary.summarize_records does.  The columns are those
of the logs: net rate l_j - m_j, DDRate's midpoint_x0 = x0 + origin and maxCarryingCap = L + div_0 (ddrate.record_row), each
one fp64 operation, so the three paths see the same values.

  python -m literate_b200.plotdd <dir> [-burnin .2] [-combine 1] [-origin Y]     -> <log stem>_plots.r / COMBINED_<kind>_plots.r
"""
from __future__ import annotations

import glob
import os
import re
from dataclasses import dataclass

import numpy as np

from . import ddrate as DD
from . import engine as E
from . import summary as S
from . import trend as TR

KINDS = ("trendrate", "dd")
DD_PARAMS = DD.header(0, 0)[6:6 + DD.NPAR]          # the log's names: midpoint_x0, initCarryingCap, maxCarryingCap, ...
LEVEL = 0.95


@dataclass
class PlotSummary:
    name: str
    kind: str                     # "trendrate" or "dd"
    time: np.ndarray              # bin index, or origin + i + 0.5
    n_samples: int                # pooled samples after the burn-in
    series: dict                  # "birth", "death", "net" (+ "niche", "nicheFrac") -> {"mean", "lo", "hi"} arrays [n_bins]
    params: dict                  # parameter name of the log header -> {"mean", "lo", "hi"} floats


def series_names(kind):
    return ["birth", "death", "net"] + (["niche", "nicheFrac"] if kind == "dd" else [])


def param_names(kind):
    return list(TR.PARAMS) if kind == "trendrate" else list(DD_PARAMS)


def bin_time(n_bins, origin=None):
    return np.arange(n_bins, dtype=np.float64) if origin is None else origin + np.arange(n_bins) + 0.5


def column_specs(kind, n_bins, origin=0.0):
    """(a, b, sign, add) of every output column in the record layout (lr_column_hpd): the per-bin series, then the parameters."""
    if kind not in KINDS:
        raise ValueError("kind must be 'trendrate' or 'dd'")
    head, nser = (TR.REC_HEAD, 2) if kind == "trendrate" else (DD.REC_HEAD, 4)
    f = lambda s, j: head + s * n_bins + j
    cols = [(f(0, j), -1, 1, 0.0) for j in range(n_bins)] + [(f(1, j), -1, 1, 0.0) for j in range(n_bins)]
    cols += [(f(0, j), f(1, j), -1, 0.0) for j in range(n_bins)]                                    # net rate l_j - m_j
    cols += [(f(s, j), -1, 1, 0.0) for s in range(2, nser) for j in range(n_bins)]                  # niche, niche fraction
    if kind == "trendrate":
        cols += [(5 + i, -1, 1, 0.0) for i in range(len(TR.PARAMS))]
    else:
        par = [(5 + i, -1, 1, 0.0) for i in range(DD.NPAR)]
        par[3] = (8, -1, 1, float(origin))                                                          # midpoint_x0 = x0 + origin
        par[5] = (10, 9, 1, 0.0)                                                                    # maxCarryingCap = L + div_0
        cols += par
    return cols


def _host_columns(rows, specs):
    """The columns of lr_column_hpd on host rows [n, w], with the same fp64 operations in the same order."""
    out = np.empty((rows.shape[0], len(specs)))
    for j, (a, b, sg, add) in enumerate(specs):
        v = rows[:, a]
        if b >= 0:
            v = v + rows[:, b] if sg > 0 else v - rows[:, b]
        if add != 0.0:
            v = v + add
        out[:, j] = v
    return out


def _pack(name, kind, n_bins, time, n, mean, lo, hi):
    out = PlotSummary(name, kind, time, int(n), {}, {})
    for s, tag in enumerate(series_names(kind)):
        sl = slice(s * n_bins, (s + 1) * n_bins)
        out.series[tag] = {"mean": mean[sl], "lo": lo[sl], "hi": hi[sl]}
    base = len(series_names(kind)) * n_bins
    for i, p in enumerate(param_names(kind)):
        out.params[p] = {"mean": float(mean[base + i]), "lo": float(lo[base + i]), "hi": float(hi[base + i])}
    return out


def _summarize_host(name, kind, n_bins, time, X):
    lo, hi = S.hpd_columns(X, LEVEL)
    return _pack(name, kind, n_bins, time, X.shape[0], X.mean(axis=0), lo, hi)


def _beta_col(kind):
    return TR.REC_BETA if kind == "trendrate" else DD.REC_BETA


def summarize_records(records, kind, n_bins, origin=0.0, burnin=0.2, ladder=1, name="chains"):
    """records [n_samples, n_chains, rec_doubles] (or [n_samples, rec_doubles]) of K6 ("trendrate") or K7 ("dd") -> PlotSummary
    (host).  ladder > 1: tempered ladders of that many chains, summarised over their cold members (engine.cold_records).
    origin: the run's origin (DDRate's midpoint_x0 is x0 + origin in the log); time = origin + i + 0.5."""
    r = np.asarray(records, dtype=np.float64)
    if r.ndim == 2:
        r = r[:, None, :]
    if ladder > 1:
        r = E.cold_records(r, ladder, _beta_col(kind))
    rows = r[S.burnin_index(r.shape[0], burnin):].reshape(-1, r.shape[-1])
    return _summarize_host(name, kind, n_bins, bin_time(n_bins, origin), _host_columns(rows, column_specs(kind, n_bins, origin)))


def summarize_records_device(dev, records, kind, n_bins, origin=0.0, burnin=0.2, cold_only=False, name="chains"):
    """The same from a float64 CUDA tensor of records [n_samples, n_chains, rec_doubles] on `dev` (an engine.Device): one K8
    call over every column.  cold_only: only records written at beta = 1 count (tempered ladders; the cold member of a ladder
    changes from sample to sample)."""
    if records.dim() == 2:
        records = records[:, None, :]
    w = records.shape[-1]
    rows = records[S.burnin_index(records.shape[0], burnin):].reshape(-1, w)
    mean, lo, hi, n = dev.column_hpd_device(rows, column_specs(kind, n_bins, origin), LEVEL, _beta_col(kind) if cold_only else -1)
    return _pack(name, kind, n_bins, bin_time(n_bins, origin), int(n.item()), mean.cpu().numpy(), lo.cpu().numpy(), hi.cpu().numpy())


# ------------------------------------------------------------------------------------------ logs
def log_kind(path):
    """"trendrate" for *.trendrate.log, "dd" for a DDRate sample log (a *.log with a niche_0 column that is not a .div.log),
    else None."""
    base = os.path.basename(path)
    if base.endswith(".trendrate.log"):
        return "trendrate"
    if base.endswith(".log") and not base.endswith(".div.log"):
        with open(path) as fh:
            if "niche_0" in fh.readline().rstrip("\r\n").split("\t"):
                return "dd"
    return None


def log_stem(path):
    return path[:-len(".trendrate.log")] if path.endswith(".trendrate.log") else path[:-len(".log")]


def read_log(path, burnin):
    """The post-burn-in rows of a TrendRate / DDRate sample log -> (header, n_bins, col): col(name) is the column of that header
    name, or for net_<j> the net rate l_<j> - m_<j> formed as the kernels do."""
    with open(path) as fh:
        head = fh.readline().rstrip("\r\n").split("\t")
    tbl = np.loadtxt(path, delimiter="\t", skiprows=1, ndmin=2)
    tbl = tbl[S.burnin_index(tbl.shape[0], burnin):]
    idx = {h: i for i, h in enumerate(head)}

    def col(name):
        if name.startswith("net_"):
            return tbl[:, idx["l_" + name[4:]]] - tbl[:, idx["m_" + name[4:]]]
        return tbl[:, idx[name]]
    return head, sum(1 for h in head if re.fullmatch(r"l_\d+", h)), col


def _log_columns(path, kind, burnin):
    """The post-burn-in rows of one log as the columns of column_specs."""
    _, n_bins, col = read_log(path, burnin)
    tags = ("l", "m", "net") + (("niche", "nicheFrac") if kind == "dd" else ())
    names = ["%s_%d" % (t, j) for t in tags for j in range(n_bins)] + param_names(kind)
    return np.stack([col(nm) for nm in names], axis=1), n_bins


def summarize_logs(paths, burnin=0.2, origin=None, name=None):
    """Sample logs of one kind (each a chain: its burn-in removed, then pooled) -> PlotSummary.  time: the bin index, or
    origin + i + 0.5 given the run's origin."""
    paths = [paths] if isinstance(paths, str) else list(paths)
    kinds = {log_kind(p) for p in paths}
    if len(kinds) != 1 or None in kinds:
        raise ValueError("summarize_logs needs *.trendrate.log files or DDRate sample logs, of one kind")
    kind = kinds.pop()
    blocks = [_log_columns(p, kind, burnin) for p in paths]
    if len({nb for _, nb in blocks}) != 1:
        raise ValueError("the logs have different numbers of bins")
    n_bins = blocks[0][1]
    name = name or os.path.basename(log_stem(paths[0]))
    return _summarize_host(name, kind, n_bins, bin_time(n_bins, origin), np.concatenate([b for b, _ in blocks]))


def find_logs(log_dir):
    """{kind: sorted sample logs} of a directory (combined outputs excluded)."""
    out = {}
    for f in sorted(glob.glob(os.path.join(log_dir, "*.log"))):
        k = log_kind(f)
        if k is not None and not os.path.basename(f).startswith("COMBINED"):
            out.setdefault(k, []).append(f)
    return out


# ------------------------------------------------------------------------------------------ R output
R_NAMES = {"birth": ("birth_rate", "Birth rate", "#4c4cec"), "death": ("death_rate", "Death rate", "#e34a33"),
           "net": ("net_rate", "Net rate", "#32CD32"), "niche": ("niche_mean", "Niche", "#8c6bb1"),
           "nicheFrac": ("nicheFrac_mean", "Niche fraction", "#feb24c")}


def write_r(s: PlotSummary, path):
    """<path>: R script with the vectors time, <series>_rate / _mean, _minHPD, _maxHPD and the parameter table, plotted in base R
    (as summary.write_r)."""
    f = lambda v: [np.float64(x) for x in v]
    out = ["pdf(file='%s',width=12, height=8)" % (os.path.splitext(path)[0] + ".pdf"), "par(mfrow=c(2,3))", "library(scales)",
           "###%s###" % s.name, "# %d posterior samples" % s.n_samples, S.r_vec("time", f(s.time))]
    for tag in series_names(s.kind):
        var, label, colr = R_NAMES[tag]
        stem = var.rsplit("_", 1)[0]
        v = s.series[tag]
        lo = min(0.0, 1.1 * float(np.nanmin(v["lo"]))) if np.isfinite(np.nanmin(v["lo"])) else 0.0
        hi = 1.1 * float(np.nanmax(v["hi"])) if np.isfinite(np.nanmax(v["hi"])) else 1.0
        out += ["#%s" % label, S.r_vec(var, f(v["mean"])), S.r_vec(stem + "_minHPD", f(v["lo"])), S.r_vec(stem + "_maxHPD", f(v["hi"])),
                "plot(time,%s,type='n',ylim=c(%s,%s),ylab='%s',xlab='Time',main='%s')" % (var, lo, hi, label, s.name),
                "polygon(c(time, rev(time)), c(%s_maxHPD, rev(%s_minHPD)), col = alpha('%s',0.3), border = NA)" % (stem, stem, colr),
                "lines(time,%s, col = '%s', lwd=2)" % (var, colr)]
        if tag == "net":
            out.append("abline(h=0,lty=2)")
    names = list(s.params)
    out += ["#Parameters", "params=c(%s)" % ", ".join("'%s'" % p for p in names),
            S.r_vec("param_mean", f(s.params[p]["mean"] for p in names)),
            S.r_vec("param_minHPD", f(s.params[p]["lo"] for p in names)),
            S.r_vec("param_maxHPD", f(s.params[p]["hi"] for p in names)),
            "print(data.frame(params, param_mean, param_minHPD, param_maxHPD))", "n <- dev.off()"]
    with open(path, "w") as fh:
        fh.write("\n".join(out) + "\n")
    return path


def main(argv=None):
    import argparse
    p = argparse.ArgumentParser(prog="plotdd")
    p.add_argument('input_data', metavar='<path to log files>', type=str)
    p.add_argument('-burnin', metavar='.2', type=float, default=.2)
    p.add_argument('-combine', metavar='0', type=int, default=0)
    p.add_argument('-origin', metavar='Y', type=float, default=None, help='first bin edge of the run: time = Y + i + 0.5 (default: bin index)')
    a = p.parse_args(argv)
    logs = find_logs(a.input_data)
    if not logs:
        raise SystemExit("no *.trendrate.log or DDRate sample log under " + a.input_data)
    written = []
    for kind, files in logs.items():
        print("found", len(files), "%s log files..." % kind)
        if a.combine == 1:
            tag = "DD" if kind == "dd" else "trendrate"
            written.append(write_r(summarize_logs(files, a.burnin, a.origin, name="COMBINED_" + tag),
                                   os.path.join(a.input_data, "COMBINED_%s_plots.r" % tag)))
        else:
            written += [write_r(summarize_logs([f], a.burnin, a.origin), log_stem(f) + "_plots.r") for f in files]
    for w in written:
        print("Plots saved in %s" % w)
    return written


if __name__ == "__main__":
    main()
