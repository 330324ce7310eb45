"""TrendRate on the GPU (SURVEY 8 f-4): host mirror and drop-in command line of trend_rate.py.

Same flags as the reference (literate_library.core_arguments :290-308 plus trend_rate.py:34-38), same input parsing
(pandas, tab-separated, 3 or 4 columns), same bins (unit bins from the first birth time, last one dropped), same log file
name, header and row layout (trend_rate.py:110-118, :191).  The statistics come from K1 (`lr_bin_stats`), the chains run in
K6 (`lr_trend_*`); this module parses, launches and writes text.  There is no CPU path.

New flags: -chains (independent chains, one warp each; chain k is named like a reference run with seed + k), -device,
-quiet, -temper.  -d may name a directory of tables (stochastic imputations of one data set, as for literate_b200.forward): every
table is a replicate binned in the same K1 launch over the common window, chain k runs on table k % n_tables and writes
next to that table.  Under torchrun the chains are block-partitioned over the ranks; a chain keeps its name and its Philox
stream whatever the number of GPUs.
-temper T > 1 (with -swap_every, -temper_delta, as for literate_b200.forward; new, the reference has no tempering): every
logged chain is the cold member (beta = 1, the reference's chain) of a ladder of T Metropolis-coupled chains, all on its
table; only cold samples reach the logs, whose names, headers and rows are those of an untempered run.

  python -m literate_b200.trend -d table.tsv -trend_data trend.tsv -trend_index 1 -n 1000000 -s 1000 -seed 1 -chains 256
"""
from __future__ import annotations

import csv
import ctypes as C
import os
import time

import numpy as np

from . import _native as N
from . import engine as E
from . import library as L
from . import parallel as P
from .library import bin_window, parse_ts_te  # noqa: F401  (parse_ts_te: callers of this module keep importing it from here)

BANNER = "\n\n             TrendRate - 20190205  (literate_b200: B200-native path)\n"
SMALL_NUMBER = 0.000000000000001                         # trend_rate.py:55
PARAMS = ["l_min", "m_min", "alpha", "beta", "delta", "gamma"]
REC_HEAD = N.LR_TREND_REC_HEAD
REC_BETA = 15                                            # record field of the chain's inverse temperature


def _flag(v):
    """argparse ``type=bool`` of the reference (trend_rate.py:36-38): any non-empty string is True."""
    return bool(v)


def build_parser():
    def own(p):                                                       # trend_rate.py:34-38
        p.add_argument('-trend_data', metavar='<path to trend file>', type=str, default="",
                       help='Input trend file should be columns tab-separated with headers. No missing values.')
        p.add_argument('-trend_index', type=int, help='Column of trend in trend file.', default=0, metavar=0)
        p.add_argument('-const_B', type=_flag, help='F) Vary rates with trend T) Constant rates', default=False, metavar=False)
        p.add_argument('-const_D', type=_flag, help='F) Vary rates with trend T) Constant rates', default=False, metavar=False)
        p.add_argument('-no_death', type=_flag, help='F) Calculate death rate T) Likelihood based on births only', default=False, metavar=False)
    return L.build_parser("trend_rate.py", own)


def parse_trend_data(path, index, rm_first_bin=0):
    """trend_rate.parse_trend_data (:58-69): column `index`, last bin dropped, min-max scaled, zeros -> SMALL_NUMBER."""
    import pandas as pd
    trend = pd.read_csv(path, sep="\t").iloc[:, index].to_numpy().astype(np.float64)
    trend = trend[:-1]
    if rm_first_bin:
        trend = trend[1:]
    lo, hi = np.min(trend), np.max(trend)
    trend = (trend - lo) / (hi - lo)
    trend[trend == 0] = SMALL_NUMBER
    return trend


class TrendChains(L.ChainObject):
    """lr_trend_t: the per-bin table and a population of independent TrendRate chains on one device."""
    PREFIX, STATE_DOUBLES, REC_BETA = "trend", N.LR_TREND_STATE_DOUBLES, REC_BETA

    def __init__(self, dev: E.Device, sp, ex, br, trend, n_chains, seed, const_birth=False, const_death=False, chain_id0=0,
                 rep_of_chain=None):
        sp, ex, br, rep = self._inputs(sp, ex, br, rep_of_chain, n_chains)
        trend = np.ascontiguousarray(trend, dtype=np.float64)
        if not (sp.shape == ex.shape == br.shape) or trend.shape != (sp.shape[1],):
            raise ValueError("sp, ex, br must be [n_rep, n_bins] and trend [n_bins] (the reference fails to broadcast, trend_rate.py:82)")
        self.dev, self.n_chains, self.n_rep, self.n_bins = dev, int(n_chains), sp.shape[0], sp.shape[1]
        t = C.c_void_p()
        N.check(dev.lib.lr_trend_create_host(dev.h, self.n_rep, self.n_bins, N.np_ptr(sp), N.np_ptr(ex), N.np_ptr(br), N.np_ptr(trend),
                                             int(bool(const_birth)), int(bool(const_death)), self.n_chains,
                                             C.c_uint64(int(seed) & (2**64 - 1)), int(chain_id0), N.np_ptr(rep), C.byref(t)),
                "lr_trend_create_host")
        self._created(t)

    def evaluate(self, params, rep=None, kind=None, on=None, draw=None):
        """Parity entry point: likelihood, prior, rates and adequacy of explicit parameter vectors [n, 6], optionally after one
        proposal with explicit draws.  Returns a dict of host arrays."""
        params = np.ascontiguousarray(np.atleast_2d(params), dtype=np.float64)
        n = params.shape[0]
        rep_a = None if rep is None else np.ascontiguousarray(rep, dtype=np.int32)
        kind_a = on_a = draw_a = None
        if kind is not None:
            kind_a = np.ascontiguousarray(kind, dtype=np.int32)
            on_a = np.ascontiguousarray(on, dtype=np.int32)
            draw_a = np.ascontiguousarray(draw, dtype=np.float64)
            assert kind_a.shape == (n,) and on_a.shape == (n, 6) and draw_a.shape == (n, 6)
        out = {"params": np.empty((n, 6)), "hastings": np.empty(n), "lik": np.empty((n, 2)), "prior": np.empty(n),
               "rates": np.empty((n, 2, self.n_bins)), "adequacy": np.empty((n, 3))}
        N.check(self.dev.lib.lr_trend_eval_host(self.t, n, N.np_ptr(rep_a), N.np_ptr(params), N.np_ptr(kind_a), N.np_ptr(on_a),
                                                N.np_ptr(draw_a), N.np_ptr(out["params"]), N.np_ptr(out["hastings"]),
                                                N.np_ptr(out["lik"]), N.np_ptr(out["prior"]), N.np_ptr(out["rates"]),
                                                N.np_ptr(out["adequacy"])), "lr_trend_eval_host")
        return out


def log_name(path, seed, trend_index, const_birth, const_death, no_death):
    out = "_CONB" if const_birth else "_EXPB"              # trend_rate.py:104-108
    if no_death:
        out += "_ND"
    elif const_death:
        out += "_COND"
    else:
        out += "_EXPD"
    return "%s_%s%s_%s.trendrate.log" % (os.path.splitext(path)[0], seed, out, trend_index)      # :110


def header(n_bins):
    head = ["it", "posterior", "likelihood", "likelihood_birth", "likelihood_death", "prior"] + PARAMS      # :113-116
    head += ["l_%s" % i for i in range(n_bins)] + ["m_%s" % i for i in range(n_bins)]
    return head + ["corr_coeff", "rsquared", "gelman_r2"]


def record_row(rec, n_bins):
    """One log row (trend_rate.py:191) from a sample record."""
    lik, prior = float(rec[1]), float(rec[4])
    return [int(rec[0]), lik + prior, lik, float(rec[2]), float(rec[3]), prior] + [float(x) for x in rec[5:11]] + \
           [float(x) for x in rec[REC_HEAD:REC_HEAD + 2 * n_bins]] + [float(x) for x in rec[11:14]]


def run(args, device=None):
    """Everything trend_rate.py does after argument parsing; returns the list of log paths of this rank."""
    rank, local_rank, world = P.env_world()
    lead = rank == 0
    if not lead:
        args.quiet = 1
    if lead:
        print(BANNER)
    no_death = bool(args.no_death)
    const_birth = bool(args.const_B)
    const_death = True if no_death else bool(args.const_D)            # :42-45
    seed = L.seed_and_chains(args, world)
    if const_birth and const_death:
        raise SystemExit("-const_B with -const_D / -no_death leaves the additive move without a parameter: the reference stops "
                         "with ValueError in np.random.binomial (trend_rate.py:129-134, :168)")
    tables, ts, te, present, origin = L.read_tables(args, exclude=args.trend_data)
    n_tab = len(tables)
    first_bin, n_bins = bin_window(origin, present, args.rm_first_bin)
    trend = parse_trend_data(args.trend_data, args.trend_index, args.rm_first_bin)
    if len(trend) != n_bins:
        raise SystemExit("the trend table must hold one row per unit bin from the first birth time plus one (%d rows); it has %d"
                         % (n_bins + 1 + (1 if args.rm_first_bin else 0), len(trend) + 1 + (1 if args.rm_first_bin else 0)))
    dev = device if device is not None else E.Device(local_rank if world > 1 else args.device)
    t0 = time.time()
    stats = dev.bin_stats(ts, te, first_bin=first_bin, n_bins=n_bins, death_jitter=args.death_jitter)
    t_bin = time.time() - t0
    sp, ex, br = stats.sp, stats.ex, stats.br
    if lead:                                                           # print_empirical_rates, literate_library.py:260-265
        with np.errstate(divide="ignore", invalid="ignore"), np.printoptions(suppress=True, precision=3):
            print("EMPIRICAL BIRTH RATES:"); print(sp[0] / br[0])
            print("EMPIRICAL DEATH RATES:"); print(ex[0] / br[0])
            print("TREND", trend)

    c0, n_local = P.shard_range(args.chains, world, rank)
    chain_id0, n_dev, rep_of_chain, beta = L.ladders(args, c0, n_local, n_tab)
    chains = TrendChains(dev, sp, ex, br, trend, n_dev, seed, const_birth, const_death, chain_id0=chain_id0, rep_of_chain=rep_of_chain)
    if beta is not None:
        chains.set_beta(beta)
    paths, files, writers = [], [], []
    for k in range(c0, c0 + n_local):
        path = log_name(tables[k % n_tab], seed + k // n_tab, args.trend_index, const_birth, const_death, no_death)
        fh = open(path, "w", newline="")
        w = csv.writer(fh, delimiter="\t")
        w.writerow(header(n_bins))
        paths.append(path); files.append(fh); writers.append(w)

    t_run, rounds = L.sample_and_write(chains, args.n, args.s, files, writers, lambda rec: record_row(rec, n_bins),
                                       lambda rec: print(int(rec[0]), rec[1], rec[5:11]), args.quiet, args.temper, args.swap_every)  # :187
    if not args.quiet:
        acc = chains.state()[:, 10].sum() / max(1, n_dev * args.n)
        print("literate_b200: %d TrendRate chains x %d iterations in %.3f s (%.3g it/s, acceptance %.3f); binning %.4f s"
              % (n_dev, args.n, t_run, n_dev * args.n / max(t_run, 1e-9), acc, t_bin))
        if args.temper > 1:
            swaps = chains.temper()[1].sum(0)
            print("literate_b200: %d swap rounds, %.3f of the proposed temperature swaps accepted" % (rounds, swaps[1] / max(swaps[0], 1)))
    chains.close()
    return paths


def main(argv=None):
    args = build_parser().parse_args(argv)
    if args.d == "" or args.trend_data == "":
        raise SystemExit("use -d <table of lineages> -trend_data <trend table>")
    run(args)


if __name__ == "__main__":
    main()
