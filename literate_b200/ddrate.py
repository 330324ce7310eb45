"""DDRate on the GPU (SURVEY 8 f-4): host mirror and drop-in command line of DDRatev3.py.

Same flags as the reference (literate_library.core_arguments :290-308 plus DDRatev3.py:25-29), same parsing, bins and
output: ``<stem>_<seed><_LL|_LDD|_LDDN|_GLDDN><_ML|_MDD|_MDDN>.log`` with the header of :159-167 and the rows of :285-287,
and the sibling ``.div.log`` (:170-183).  The statistics come from K1 (`lr_bin_stats`), the chains run in K7 (`lr_dd_*`);
this module parses, launches and writes text.  There is no CPU path.

As shipped the reference only starts with ``-m_birth 3 -g <genre table>`` (NameError at :48 otherwise); here -m_birth 0, 1
and 2 run what its functions define for them.  -m_birth -1 / -m_death -1 (NameError at :192-195) are refused.
New flags: -chains (chain k is named like a reference run with seed + k), -device, -quiet.  -d may name a directory of tables
(stochastic imputations of one data set): one replicate each over the common window, chain k on table k % n_tables.
-temper T > 1 (with -swap_every, -temper_delta, as for literate_b200.forward; the reference has no tempering): every logged
chain is the cold member (beta = 1, the reference's chain) of a ladder of T Metropolis-coupled chains, all on its table; the
heated members temper the whole likelihood, genre term included.  Only cold samples reach the logs, whose names, headers and
rows are those of an untempered run.
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
from .library import bin_window, parse_ts_te

BANNER = "\n\n             DDRate  (literate_b200: B200-native path)\n"
PARAMS = ["l_f", "l_mul", "k", "x0", "div_0", "L", "m_mul", "nuB", "nuD", "g_lambda1", "g_lambda2"]
REC_HEAD, NPAR = N.LR_DD_REC_HEAD, N.LR_DD_NPAR
REC_BETA = 21                                            # record field of the chain's inverse temperature


def build_parser():
    def own(p):                                                       # DDRatev3.py:25-29
        p.add_argument('-m_birth', type=int, help='0) use const b rates 1) DD birth 2) niche dep DD b', default=2, metavar=2)
        p.add_argument('-m_death', type=int, help='-1) fixed d rate 0) use const d rates 1) DD death 2) niche dep DD d', default=2, metavar=2)
        p.add_argument('-fix_birth', type=float, help='Fix birth rate (with -m_birth -1)', default=0.1, metavar=0.1)
        p.add_argument('-fix_death', type=float, help='Fix death rate (with -m_death -1)', default=0.1, metavar=0.1)
        p.add_argument('--genre_times', '-g', type=str, help='Genre Data File', default='', metavar='')
    return L.build_parser("DDRatev3.py", own)


class DDChains(L.ChainObject):
    """lr_dd_t: the per-bin table, the genre table and a population of independent DDRate chains on one device."""
    PREFIX, STATE_DOUBLES, REC_BETA = "dd", N.LR_DD_STATE_DOUBLES, REC_BETA

    def __init__(self, dev: E.Device, sp, ex, br, origin, present, m_birth=2, m_death=2, gts=None, gte=None, n_chains=1, seed=1,
                 chain_id0=0, rep_of_chain=None):
        sp, ex, br, rep = self._inputs(sp, ex, br, rep_of_chain, n_chains)
        if not (sp.shape == ex.shape == br.shape):
            raise ValueError("sp, ex, br must be [n_bins] or [n_rep, n_bins]")
        self.dev, self.n_chains, self.n_rep, self.n_bins = dev, int(n_chains), sp.shape[0], sp.shape[1]
        self.m_birth, self.m_death, self.origin = int(m_birth), int(m_death), float(origin)
        ng = 0
        if gts is not None:
            gts = np.ascontiguousarray(gts, dtype=np.float64)
            gte = np.ascontiguousarray(gte, dtype=np.float64)
            ng = len(gts)
        t = C.c_void_p()
        N.check(dev.lib.lr_dd_create_host(dev.h, self.n_rep, self.n_bins, N.np_ptr(sp), N.np_ptr(ex), N.np_ptr(br), float(origin),
                                          float(present), self.m_birth, self.m_death, N.np_ptr(gts), N.np_ptr(gte), ng, self.n_chains,
                                          C.c_uint64(int(seed) & (2**64 - 1)), int(chain_id0), N.np_ptr(rep), C.byref(t)), "lr_dd_create_host")
        self._created(t)

    def evaluate(self, params, kind=None, on=None, draw=None, rep=None):
        """Parity entry point: the three likelihood terms, prior, per-bin series, adequacy and genre statistics of explicit
        parameter vectors [n, 11], optionally after one proposal with explicit draws."""
        params = np.ascontiguousarray(np.atleast_2d(params), dtype=np.float64)
        n = params.shape[0]
        rep_a = None if rep is None else np.ascontiguousarray(rep, dtype=np.int32)
        kind_a = on_a = draw_a = None
        if kind is not None:
            kind_a = np.ascontiguousarray(kind, dtype=np.int32)
            on_a = np.ascontiguousarray(on, dtype=np.int32)
            draw_a = np.ascontiguousarray(draw, dtype=np.float64)
            assert kind_a.shape == (n,) and on_a.shape == (n, NPAR) and draw_a.shape == (n, NPAR)
        out = {"params": np.empty((n, NPAR)), "hastings": np.empty(n), "lik": np.empty((n, 3)), "prior": np.empty(n),
               "series": np.empty((n, 4, self.n_bins)), "adequacy": np.empty((n, 3)), "genre": np.empty((n, 4))}
        N.check(self.dev.lib.lr_dd_eval_host(self.t, n, N.np_ptr(rep_a), N.np_ptr(params), N.np_ptr(kind_a), N.np_ptr(on_a), N.np_ptr(draw_a),
                                             N.np_ptr(out["params"]), N.np_ptr(out["hastings"]), N.np_ptr(out["lik"]),
                                             N.np_ptr(out["prior"]), N.np_ptr(out["series"]), N.np_ptr(out["adequacy"]),
                                             N.np_ptr(out["genre"])), "lr_dd_eval_host")
        return out


def log_stem(path, seed, m_birth, m_death):
    out = {0: "_LL", 1: "_LDD", 2: "_LDDN", 3: "_GLDDN"}[m_birth]                 # DDRatev3.py:146-153
    out += "_ML" if m_death <= 0 else ("_MDD" if m_death == 1 else "_MDDN")
    return "%s_%s%s" % (os.path.splitext(path)[0], seed, out)


def header(n_bins, m_birth):
    head = ["it", "posterior", "likelihood", "likelihood_death", "likelihood_genre", "prior", "l_f", "l_mul", "steepness_k",
            "midpoint_x0", "initCarryingCap", "maxCarryingCap", "m_mul", "nuB", "nuD", "g_l1", "g_l2"]       # :159-161
    if m_birth == 3:
        head += ["genre_lik"]
    for tag in ("l_", "m_", "niche_", "nicheFrac_"):
        head += ["%s%s" % (tag, i) for i in range(n_bins)]
    return head + ["corr_coeff", "rsquared", "gelman_r2"]


def record_row(rec, n_bins, m_birth, origin):
    """One log row (:277-287) from a sample record: x0 becomes a calendar time, L the maximum carrying capacity."""
    lik, prior = float(rec[1]), float(rec[4])
    a = [float(x) for x in rec[5:5 + NPAR]]
    a[3] = float(np.float64(a[3]) + origin)
    a[5] = float(np.float64(a[5]) + np.float64(a[4]))
    row = [int(rec[0]), lik + prior, lik, float(rec[2]), float(rec[3]), prior] + a
    if m_birth == 3:
        row += [float(rec[16])]
    return row + [float(x) for x in rec[REC_HEAD:REC_HEAD + 4 * n_bins]] + [float(x) for x in rec[17:20]]


def write_div_log(path, sp, ex, br, gsp=None, gex=None, gbr=None):
    """:170-183: header with \\n, csv rows with \\r\\n; zip stops at the shorter of the two tables."""
    with open(path, "w", newline="") as fh:
        if gsp is None:
            fh.write('sp_events\tex_events\tbr_length\n')
            rows = zip(sp.tolist(), ex.tolist(), [np.float64(x) for x in br])
        else:
            fh.write('sp_events\tex_events\tbr_length\tg_sp_events\tg_ex_events\tg_br_length\n')
            rows = zip(sp.tolist(), ex.tolist(), [np.float64(x) for x in br], gsp.tolist(), gex.tolist(), [np.float64(x) for x in gbr])
        w = csv.writer(fh, delimiter='\t')
        for row in rows:
            w.writerow(row)


def run(args, device=None):
    """Everything DDRatev3.py does after argument parsing; returns the list of sample-log paths of this rank."""
    rank, local_rank, world = P.env_world()
    lead = rank == 0
    if not lead:
        args.quiet = 1
    if lead:
        print(BANNER)
    if args.m_birth not in (0, 1, 2, 3) or args.m_death not in (0, 1, 2):
        raise SystemExit("-m_birth must be 0..3 and -m_death 0..2 (the fixed-rate models -1 stop with NameError in the reference, "
                         "DDRatev3.py:192-195)")
    if args.m_birth == 3 and not args.genre_times:
        raise SystemExit("-m_birth 3 needs the genre table: -g <file> (DDRatev3.py:36-38)")
    seed = L.seed_and_chains(args, world)
    tables, ts, te, present, origin = L.read_tables(args, exclude=args.genre_times or "-")
    n_tab = len(tables)
    first_bin, n_bins = bin_window(origin, present, args.rm_first_bin)
    dev = device if device is not None else E.Device(local_rank if world > 1 else args.device)
    t0 = time.time()
    stats = dev.bin_stats(ts, te, first_bin=first_bin, n_bins=n_bins, death_jitter=args.death_jitter)
    sp, ex, br = stats.sp, stats.ex, stats.br
    gts = gte = gstats = None
    if args.m_birth == 3:
        gts, gte, gpresent, gorigin = parse_ts_te(args.genre_times, args.TBP, args.first_year, args.last_year, args.death_jitter)
        gfirst, gnb = bin_window(gorigin, gpresent, args.rm_first_bin)
        gstats = dev.bin_stats(gts, gte, first_bin=gfirst, n_bins=gnb, death_jitter=args.death_jitter)
    t_bin = time.time() - t0
    if args.rm_first_bin:
        origin += 1                                        # create_bins, literate_library.py:247-252
    if lead:
        print(origin, present)
        with np.errstate(divide="ignore", invalid="ignore"), np.printoptions(suppress=True, precision=3):
            print("EMPIRICAL BIRTH RATES:"); print(sp[0] / br[0])
            print("EMPIRICAL DEATH RATES:"); print(ex[0] / br[0])

    c0, n_local = P.shard_range(args.chains, world, rank)
    chain_id0, n_dev, rep_of_chain, beta = L.ladders(args, c0, n_local, n_tab)
    chains = DDChains(dev, sp, ex, br, origin, present, args.m_birth, args.m_death, gts, gte, n_dev, seed, chain_id0=chain_id0,
                      rep_of_chain=rep_of_chain)
    if beta is not None:
        chains.set_beta(beta)
    paths, files, writers = [], [], []
    for k in range(c0, c0 + n_local):
        r = k % n_tab
        stem = log_stem(tables[r], seed + k // n_tab, args.m_birth, args.m_death)
        fh = open(stem + ".log", "w", newline="")
        w = csv.writer(fh, delimiter="\t")
        w.writerow(header(n_bins, args.m_birth))
        paths.append(stem + ".log"); files.append(fh); writers.append(w)
        if gstats is None:
            write_div_log(stem + ".div.log", sp[r], ex[r], br[r])
        else:
            write_div_log(stem + ".div.log", sp[r], ex[r], br[r], gstats.sp[0], gstats.ex[0], gstats.br[0])

    t_run, rounds = L.sample_and_write(chains, args.n, args.s, files, writers, lambda rec: record_row(rec, n_bins, args.m_birth, origin),
                                       lambda rec: print(int(rec[0]), rec[1], rec[5:5 + NPAR]), args.quiet, args.temper,
                                       args.swap_every)       # :280
    if not args.quiet:
        acc = chains.state()[:, 16].sum() / max(1, n_dev * args.n)
        print("literate_b200: %d DDRate chains x %d iterations in %.3f s (%.3g it/s, acceptance %.3f); binning %.4f s"
              % (n_dev, args.n, t_run, n_dev * args.n / max(t_run, 1e-9), acc, t_bin))
        if args.temper > 1:
            swaps = chains.temper()[1].sum(0)
            print("literate_b200: %d swap rounds, %.3f of the proposed temperature swaps accepted" % (rounds, swaps[1] / max(swaps[0], 1)))
    chains.close()
    return paths


def main(argv=None):
    args = build_parser().parse_args(argv)
    if args.d == "":
        raise SystemExit("use -d <table of lineages> [-m_birth 3 -g <genre table>]")
    run(args)


if __name__ == "__main__":
    main()
