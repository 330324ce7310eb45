"""Drop-in command line for the RJMCMC birth-death path of LiteRateForward.py.

Same 21 flags, same input parsing (TAD / -TBP, 3 or 4 columns, trailing tabs, CRLF), same output
directory, file names, headers and row layout (LiteRateForward.py:376-512, :321-359, :558-564).
All numerical work (binning, likelihood, proposals, accept step) happens in the CUDA kernels of
libliterate_b200.so; this module parses, launches and writes text.

New flags (absent from the reference): -chains, -device, -launch_iters, -real_move_shift, -temper,
-swap_every, -temper_delta, -quiet.
With -chains 1 (default) file names are exactly the reference's; with more chains each chain k
writes <stem><model><out>_chain<k>_{mcmc,sp_rates,ex_rates,div}.log, which plotRJforward.v3.py's
`*mcmc.log` glob and its .replace('mcmc.log', ...) still resolve.
With -temper T > 1 every logged chain is the cold member (beta = 1, the reference's chain) of a ladder of T
Metropolis-coupled chains; only cold samples reach the logs (SURVEY A-15).
-d may name a directory of tables (stochastic imputations of one data set): each table is a replicate binned in the same
kernel launch, chain k runs on table k % n_tables and writes <table stem><model><out>[_chain<j>]_*.log.
Under torchrun (one process per GPU) the chains are block-partitioned over the ranks; chain k keeps its name and
its Philox stream whatever the number of GPUs.
"""
from __future__ import annotations

import argparse
import csv
import glob
import os
import sys
import time
from warnings import warn

import numpy as np

from . import engine as E
from . import parallel as P

BANNER = "\n\n             LiteRate - 20200206  (literate_b200: B200-native RJMCMC path)\n"
MODEL_SUFFIX = {0: "_BD", 1: "_ID", 2: "_BDk", 3: "_BDd"}          # :422-427
MCMC_COLS = ["it", "posterior", "likelihood", "prior", "lambda_avg", "mu_avg", "K_l", "K_m", "root_age", "death_age",
             "gamma_rate_hp_BI", "gamma_rate_hp_D", "poisson_rate_hp"]   # :496-502
ADEQUACY_COLS = ["corr_coeff", "rsquared", "gelman_r2"]


def build_parser():
    """The reference's parser (:376-401), flag for flag, plus the new multi-chain flags."""
    p = argparse.ArgumentParser(prog="LiteRateForward.py")
    p.add_argument('-v', action='version', version='%(prog)s')
    p.add_argument('-d', type=str, help='data file', default="", metavar="")
    p.add_argument('-n', type=int, help='n. MCMC iterations', default=10000000, metavar=10000000)
    p.add_argument('-p', type=int, help='print frequency', default=1000, metavar=1000)
    p.add_argument('-s', type=int, help='sampling frequency', default=1000, metavar=1000)
    p.add_argument('-seed', type=int, help='seed (set to -1 to make it random)', default=-1, metavar=-1)
    p.add_argument('-const_rates', type=int, help="set to: 1 for constant B/I and D rates", default=0, metavar=0)
    p.add_argument('-const_death_rate', type=int, help="set to: 1 for constant D rates", default=0, metavar=0)
    p.add_argument('-model_BDI', type=int, help='0: birth-death; 1: immigration-death; 2 birth-death (Keiding likelihood); '
                   '3 Keiding likelihood, only no extant', default=0, metavar=0)
    p.add_argument('-TBP', help='Default is AD. Include for TBP.', default=False, action='store_true')
    p.add_argument('-pyrate_output', help='Make output PyRate-compatible', default=False, action='store_true')
    p.add_argument('-first_year', type=int, help='different start of the dataset (TAD only)', default=-1, metavar=-1)
    p.add_argument('-last_year', type=int, help='different end of the dataset (TAD only)', default=-1, metavar=-1)
    p.add_argument('-death_jitter', type=float, help='amount to jitter death times', default=.5, metavar=.5)
    p.add_argument('-use_rate_HP', type=int, help='0: no hyper-prior on rates, 1: hyper-prior on rates', default=1, metavar=1)
    p.add_argument('-Poisson_prior', type=float, help='0: use hyper-prior on n. shifts, >0: fixed prior on n. shifts', default=0, metavar=0)
    p.add_argument('-rm_first_bin', type=float, help='if set to 1 it removes the first time bin', default=0, metavar=0)
    p.add_argument('-calc_adequacy', type=int, help='if set to 1 calculates and log to file adequacy', default=1, metavar=1)
    p.add_argument('-update_fraction', type=float, help='', default=0.75, metavar=0.75)
    p.add_argument('-out', type=str, help='output name suffix', default="", metavar="")
    p.add_argument('-rev_se', type=int, help='reversed order of ts and te in input file', default=0, metavar=0)
    p.add_argument('-proportion', type=int, help='turns ts and te into independent immigration processes (the flag of '
                   'LiteRateForward-proportion.py; output files are then named <table>_PR_seed<seed>)', default=0, metavar=0)
    # ---- not in the reference
    p.add_argument('-chains', type=int, help='number of independent chains run concurrently on the GPU', default=1, metavar=1)
    p.add_argument('-device', type=int, help='CUDA device index', default=0, metavar=0)
    p.add_argument('-launch_iters', type=int, help='iterations per kernel launch (0: choose)', default=0, metavar=0)
    p.add_argument('-real_move_shift', type=int, help='1: move-shift really moves the shift (the reference proposes the '
                   'current state, LiteRateForward.py:184-185)', default=0, metavar=0)
    p.add_argument('-temper', type=int, help='temperatures per logged chain (1: no tempering, as the reference)', default=1, metavar=1)
    p.add_argument('-swap_every', type=int, help='iterations between temperature-swap rounds', default=1000, metavar=1000)
    p.add_argument('-temper_delta', type=float, help='ladder beta_k = 1/(1 + delta k)', default=0.1, metavar=0.1)
    p.add_argument('-quiet', type=int, help='1: no per-iteration progress on stdout', default=0, metavar=0)
    return p


def parse_lineages(path, TBP=False, rev_se=0, first_year=-1, last_year=-1, death_jitter=0.5):
    """TSV -> (ts, te, start_time, end_time, true_root_age), LiteRateForward.py:439-476.

    -first_year raises IndexError in the reference whenever it filters anything (:460-461); the intended
    order of literate_library.parse_ts_te (literate_library.py:216-222) is implemented instead.
    """
    tbl = np.genfromtxt(path, skip_header=1)
    if tbl.ndim == 1:
        tbl = tbl[None, :]
    if tbl.shape[1] == 4:
        warn('Four column (with clade) LiteRate input is deprecated. Use three columns.', FutureWarning)
        ts_y, te_y = tbl[:, 2], tbl[:, 3]
    elif rev_se:
        ts_y, te_y = tbl[:, 2], tbl[:, 1]
    else:
        ts_y, te_y = tbl[:, 1], tbl[:, 2]
    if TBP:
        root = np.max(ts_y)
        ts, te = root - ts_y, root - te_y
    else:
        root = 0
        if first_year != -1:
            keep = ts_y >= first_year
            ts_y, te_y = ts_y[keep], te_y[keep]
        if last_year != -1:
            keep = ts_y <= last_year
            ts, te = ts_y[keep], te_y[keep] + 0.0
            te[te > last_year] = last_year
        else:
            ts, te = ts_y, te_y
    te = te + death_jitter
    ts = np.ascontiguousarray(ts, dtype=np.float64)
    te = np.ascontiguousarray(te, dtype=np.float64)
    return ts, te, np.min(ts), np.max(te), root


def as_year_table(ts, te, death_jitter):
    """(ts, te) as parse_lineages returns them -> int32 YEARS (ts, te - jitter) if the table is one of integer years (every table
    the reference ships) and the jitter is one the int32 entry point reproduces exactly (E.year_jitter_ok: a multiple of
    2^-22 in [0, 1], such as the default .5), else None.  The int32 entry point of K1 takes half the bytes and adds the jitter
    itself; the statistics are the same bit for bit.  Other jitters (-death_jitter 0.1, say) give fl(year + jitter) a
    fraction that differs from year to year, so such tables stay float64."""
    if not E.year_jitter_ok(death_jitter):
        return None
    ok = ~np.isnan(ts)
    ey = te - death_jitter
    lim = float(np.iinfo(np.int32).max - 1)
    if not (np.all(np.isnan(te) == ~ok) and np.all(np.abs(ts[ok]) < lim) and np.all(np.abs(ey[ok]) < lim)):
        return None
    ti, ei = np.where(ok, ts, 0.0).astype(np.int32), np.where(ok, ey, 0.0).astype(np.int32)
    if not (np.array_equal(ti[ok], ts[ok]) and np.array_equal(ei[ok] + death_jitter, te[ok])):
        return None
    ti[~ok] = E.YEAR_PAD; ei[~ok] = E.YEAR_PAD
    return ti, ei


def _fmt(x):
    """str() of what the reference puts in a row: Python ints stay ints, floats use the shortest repr
    (str(np.float64) == repr(float) for every finite value)."""
    if isinstance(x, (int, np.integer)):
        return str(int(x))
    return repr(float(x))


def write_div_log(path, sp, ex, br):
    """div.log (:558-564): header ends in '\\n', the csv.writer rows in '\\r\\n'."""
    with open(path, "w", newline="") as fh:
        fh.write('sp_events\tex_events\tbr_length\n')
        w = csv.writer(fh, delimiter='\t')
        for a, b, c in zip(sp.tolist(), ex.tolist(), br.tolist()):
            w.writerow((a, b, repr(float(c))))


class ChainLogWriter:
    """The three per-chain log files of :493-512 and their rows (:321-359)."""

    def __init__(self, stem, calc_adequacy, pyrate_output, start_time, end_time, true_root_age, poisson_prior):
        self.calc_adequacy, self.pyrate = calc_adequacy, pyrate_output
        self.start_time, self.end_time, self.root = start_time, end_time, true_root_age
        self.poisson_prior = poisson_prior
        self.mcmc = open(stem + "_mcmc.log", "w")
        self.sp = open(stem + "_sp_rates.log", "w")
        self.ex = open(stem + "_ex_rates.log", "w")
        self.mcmc.write('\t'.join(MCMC_COLS + (ADEQUACY_COLS if calc_adequacy else [])) + '\n')

    def write(self, rec):
        kl, km = int(rec[E.REC_KL]), int(rec[E.REC_KM])
        L, M = rec[E.REC_L:E.REC_L + kl], rec[E.REC_M:E.REC_M + km]
        sL, sM = rec[E.REC_TL + 1:E.REC_TL + kl], rec[E.REC_TM + 1:E.REC_TM + km]
        lik, prior = rec[E.REC_LIK], rec[E.REC_PRIOR]
        if self.pyrate:       # :325-326: root_age, root_age - max(timesLA) (= root - end_time)
            ages = [_fmt(self.root), _fmt(np.float64(self.root - self.end_time))]
            sL, sM = self.root - sL, self.root - sM
        else:
            ages = [_fmt(np.float64(self.start_time)), _fmt(np.float64(self.end_time))]
        if rec[E.REC_POI_INIT]:   # Poi_lambda_rjHP is still the Python constant of :220-221
            poi = "1" if self.poisson_prior == 0 else repr(float(self.poisson_prior))
        else:
            poi = repr(float(rec[E.REC_POI]))
        row = [str(int(rec[E.REC_IT])), repr(float(lik + prior)), repr(float(lik)), repr(float(prior)),
               repr(float(rec[E.REC_LAVG])), repr(float(rec[E.REC_MAVG])), str(kl), str(km)] + ages + \
              [repr(float(rec[E.REC_GL])), repr(float(rec[E.REC_GM])), poi]
        if self.calc_adequacy:
            row += [repr(float(v)) for v in rec[E.REC_ADQ:E.REC_ADQ + 3]]
        self.mcmc.write('\t'.join(row) + '\n')
        self.sp.write('\t'.join([repr(float(v)) for v in L] + [repr(float(v)) for v in sL]) + '\n')
        self.ex.write('\t'.join([repr(float(v)) for v in M] + [repr(float(v)) for v in sM]) + '\n')

    def flush(self):
        self.mcmc.flush(); self.sp.flush(); self.ex.flush()

    def close(self):
        self.mcmc.close(); self.sp.close(); self.ex.close()


def _print_state(rec, end_time, calc_adequacy):
    """The progress block of :362-370 (chain 0)."""
    L, M, tL, tM = E.record_to_state(rec, end_time)
    with np.printoptions(suppress=True, precision=3):
        print(int(rec[E.REC_IT]), rec[E.REC_LIK], rec[E.REC_PRIOR])
        print("\tsp.times:", tL)
        print("\tex.times:", tM)
        print("\tsp.rates:", L)
        print("\tex.rates:", M)
        if calc_adequacy:
            print("\tR^2:", rec[E.REC_ADQ + 1])


def run(args, device=None):
    """Everything LiteRateForward.py does after argument parsing; returns the list of mcmc.log paths."""
    rank, local_rank, world = P.env_world()
    lead = rank == 0
    if not lead:
        args.quiet = 1
    if lead:
        print(BANNER)
    if args.seed == -1:                                   # :405-407
        rseed = int(np.random.randint(0, 9999))
        if world > 1:
            raise SystemExit("give -seed explicitly when running on several GPUs (every rank must use the same one)")
    else:
        rseed = args.seed
    if args.model_BDI not in MODEL_SUFFIX:
        raise SystemExit("-model_BDI must be 0, 1, 2 or 3")
    if args.chains < 1:
        raise SystemExit("-chains must be >= 1")
    if not (1 <= args.temper <= 32):
        raise SystemExit("-temper must be 1..32")
    if args.chains < world:
        raise SystemExit("-chains must be at least the number of GPUs")
    out_name = MODEL_SUFFIX[args.model_BDI] + args.out
    only_dead = args.model_BDI == 3
    if args.proportion == 1:
        return _run_proportion(args, rseed, device, lead, world, rank, local_rank)

    # -d may name a DIRECTORY of tables (stochastic imputations of one data set, the reference's "100 chains on 100
    # imputations" workflow, 3_interpreting_literate_results_final.ipynb:208): every table is one replicate, binned in the
    # same K1 launch over a common time window; chain k runs on replicate k % n_tables.
    if os.path.isdir(args.d):
        tables = sorted(f for f in glob.glob(os.path.join(args.d, "*")) if os.path.isfile(f) and f.lower().endswith((".tsv", ".txt")))
        if not tables:
            raise SystemExit("no .tsv/.txt table in " + args.d)
        out_dir = args.d.rstrip("/")
    else:
        tables = [args.d]
        out_dir = os.path.dirname(args.d)                 # :479-491
        if out_dir == "":
            out_dir = os.getcwd()
    parsed = [parse_lineages(f, args.TBP, args.rev_se, args.first_year, args.last_year, args.death_jitter) for f in tables]
    n_tab = len(parsed)
    if args.chains == 1 and n_tab > 1:
        args.chains = n_tab                               # default: one chain per table
    if args.chains % n_tab:
        raise SystemExit("-chains must be a multiple of the number of tables (%d)" % n_tab)
    start_time, end_time = min(p[2] for p in parsed), max(p[3] for p in parsed)
    true_root_age = parsed[0][4]
    n_max = max(len(p[0]) for p in parsed)
    ts = np.full((n_tab, n_max), np.nan); te = np.full((n_tab, n_max), np.nan)      # NaN rows carry no event and no time at risk
    for i, p in enumerate(parsed):
        ts[i, :len(p[0])], te[i, :len(p[1])] = p[0], p[1]
    file_names = [os.path.splitext(os.path.basename(f))[0] for f in tables]
    file_name = file_names[0]
    out_dir = "%s/literate_mcmc_logs" % (out_dir)
    try:
        os.mkdir(out_dir)
    except OSError as e:
        if lead:
            print(e)

    dev = device if device is not None else E.Device(local_rank if world > 1 else args.device)
    t0 = time.time()
    years = as_year_table(ts, te, args.death_jitter)            # integer years: 8 bytes per lineage over PCIe instead of 16
    stats = dev.bin_stats(*(years if years is not None else (ts, te)), first_bin=int(start_time), n_bins=int(end_time) - int(start_time),
                          death_jitter=args.death_jitter, only_dead=only_dead, end_time=float(end_time))
    t_bin = time.time() - t0
    sp, ex, br = stats.sp[0], stats.ex[0], stats.br[0]
    if lead:
        print(ex.tolist())                                     # :526-527
        print(br.sum(), range(stats.first_bin, stats.first_bin + stats.n_bins))
        if only_dead:
            print(len(stats.ex_dead[0]), len(sp))
    if args.rm_first_bin:
        # The reference drops element 0 of the three vectors (:552-556) but keeps an n_bins+1 long rate index and
        # dies with IndexError at the first likelihood; here the window itself starts one bin later.
        stats = E.BinStats(stats.first_bin + 1, stats.sp[:, 1:], stats.ex[:, 1:], stats.br[:, 1:],
                           None if stats.ex_dead is None else stats.ex_dead[:, 1:],
                           None if stats.br_dead is None else stats.br_dead[:, 1:])
        sp, ex, br = stats.sp[0], stats.ex[0], stats.br[0]
        start_time = np.float64(np.floor(start_time) + 1)

    if args.calc_adequacy and lead:                        # print_empirical_rates, literate_library.py:260-266
        with np.errstate(divide="ignore", invalid="ignore"), np.printoptions(suppress=True, precision=3):
            print("EMPIRICAL BIRTH RATES:"); print(sp / br)
            print("EMPIRICAL DEATH RATES:"); print(ex / br)

    ds = E.Dataset(dev, stats, args.model_BDI, float(start_time), float(end_time))
    cfg = E.default_config(args.model_BDI, args.const_rates, args.const_death_rate, args.use_rate_HP, args.Poisson_prior,
                           args.update_fraction, args.real_move_shift)
    # this rank's block of the logged chains; every logged chain is a ladder of T device chains with consecutive ids
    T = args.temper
    c0, n_local = P.shard_range(args.chains, world, rank)
    rep_of_chain = np.repeat(np.arange(c0, c0 + n_local) % n_tab, T).astype(np.int32)      # logged chain k -> table k % n_tab
    chains = E.Chains(ds, n_local * T, rseed, cfg, chain_id0=c0 * T, rep_of_chain=rep_of_chain)
    if T > 1:
        chains.set_beta(np.tile(P.temperature_ladder(T, args.temper_delta), n_local))

    writers, paths = [], []
    for k in range(c0, c0 + n_local):
        r = k % n_tab
        st = "%s/%s%s" % (out_dir, file_names[r], out_name)
        if args.chains > n_tab:
            st += "_chain%d" % (k // n_tab)
        writers.append(ChainLogWriter(st, args.calc_adequacy, args.pyrate_output, start_time, end_time, true_root_age,
                                      args.Poisson_prior))
        paths.append(st + "_mcmc.log")
        write_div_log(st + "_div.log", stats.sp[r], stats.ex[r], stats.br[r])     # every *mcmc.log has its sibling div.log

    s_freq, p_freq = max(1, args.s), max(1, args.p)
    every = int(np.gcd(s_freq, p_freq))
    per_launch = args.launch_iters
    if per_launch <= 0:
        # keep one launch's records under ~256 MB
        max_rec = max(1, (256 << 20) // (n_local * T * E.LR_REC_DOUBLES * 8))
        per_launch = max(every, min(max_rec * every, 2_000_000))
    per_launch = max(every, per_launch // every * every)
    done, rounds = 0, 0
    t_run = time.time()

    def emit(recs):
        for r in range(recs.shape[0]):
            it = int(recs[r, 0, E.REC_IT])
            if it % s_freq == 0:
                for k in range(n_local):
                    writers[k].write(recs[r, k])
            if it % p_freq == 0 and not args.quiet:
                _print_state(recs[r, 0], float(end_time), args.calc_adequacy)
        for w in writers:
            w.flush()

    if T > 1:
        while done < args.n:
            n_it = min(per_launch, args.n - done)
            recs, r = chains.run_tempered(n_it, every, T, max(1, args.swap_every), round0=rounds)
            rounds += r
            emit(E.cold_records(recs, T))
            done += n_it
    else:
        # Double-buffered: the text of launch k is formatted and written while launch k+1 runs on the device (formatting
        # tens of millions of shortest-repr floats is the slower half for many chains).
        import torch
        tdev = torch.device("cuda", dev.index)
        pending = None
        while done < args.n or pending is not None:
            nxt = None
            if done < args.n:
                n_it = min(per_launch, args.n - done)
                n_rec = chains.records_per_run(n_it, every)              # host-side arithmetic: does not wait for the device
                buf = torch.empty((n_rec, n_local, E.LR_REC_DOUBLES), dtype=torch.float64, device=tdev)
                if pending is not None:
                    dev.sync()                                           # the previous launch (on the handle's stream) has written `pending`
                    host_prev = pending.cpu().numpy()
                    pending = None
                else:
                    host_prev = None
                chains.run_device(n_it, every, buf, stream="handle")     # asynchronous
                done += n_it
                nxt = buf
                if host_prev is not None:
                    emit(host_prev)
            else:
                dev.sync()
                emit(pending.cpu().numpy())
                pending = None
            if nxt is not None:
                pending = nxt
    t_run = time.time() - t_run
    for w in writers:
        w.close()
    cnt = chains.counters().sum(0)
    _warn_capacity(chains)
    if not args.quiet:
        print("literate_b200: %d chains x %d iterations in %.3f s (%.3g it/s, %.3g likelihood evaluations/s); binning %.4f s"
              % (n_local * T, args.n, t_run, n_local * T * args.n / max(t_run, 1e-9), cnt[2] / max(t_run, 1e-9), t_bin))
        if T > 1:
            print("literate_b200: %d swap rounds, %.3f of the proposed temperature swaps accepted" % (rounds, cnt[9] / max(cnt[8], 1)))
    chains.close(); ds.close()
    return paths


def _run_proportion(args, rseed, device, lead, world, rank, local_rank):
    """`-proportion 1` (LiteRateForward-proportion.py): other statistics and likelihood tables, the same chains and log rows."""
    from . import proportion as PR
    if os.path.isdir(args.d):
        raise SystemExit("-proportion 1 takes one table")
    if args.temper != 1:
        raise SystemExit("-proportion 1 does not combine with -temper")
    ts, te, start_time, end_time = PR.read_series(args.d, args.death_jitter)
    sp, ex, kn, kd = PR.series_stats(ts, te, start_time, end_time)
    if lead:
        print(te)                                              # :487
        print(sp, ex, kn, kd)                                  # :599
    out_dir = os.path.dirname(args.d) or os.getcwd()
    out_dir = "%s/literate_mcmc_logs" % out_dir
    try:
        os.mkdir(out_dir)
    except OSError as e:
        if lead:
            print(e)
    file_name = os.path.splitext(os.path.basename(args.d))[0]
    out_name = "_PR" + "_seed" + str(args.seed) + args.out          # :442-445 (the seed as given, -1 included)
    if args.rm_first_bin:
        sp, ex, kn, kd = sp[1:], ex[1:], kn[1:], kd[1:]            # :607-613 (the reference then dies in the rate index, as without the flag)
        start_time = float(np.floor(start_time) + 1)
    dev = device if device is not None else E.Device(local_rank if world > 1 else args.device)
    ds = E.Dataset.from_tables(dev, start_time=start_time, end_time=end_time, model_tag=1, **PR.likelihood_tables(sp, ex, kn, kd))
    cfg = E.default_config(1, args.const_rates, args.const_death_rate, args.use_rate_HP, args.Poisson_prior, args.update_fraction,
                           args.real_move_shift)
    c0, n_local = P.shard_range(args.chains, world, rank)
    chains = E.Chains(ds, n_local, rseed, cfg, chain_id0=c0)
    writers, paths = [], []
    for k in range(c0, c0 + n_local):
        st = "%s/%s%s" % (out_dir, file_name, out_name) + ("_chain%d" % k if args.chains > 1 else "")
        writers.append(ChainLogWriter(st, args.calc_adequacy, args.pyrate_output, start_time, end_time, 0, args.Poisson_prior))
        paths.append(st + "_mcmc.log")
        PR.write_div_log(st + "_div.log", sp, ex, kn, kd)
    s_freq, p_freq = max(1, args.s), max(1, args.p)
    every = int(np.gcd(s_freq, p_freq))
    per_launch = max(every, (args.launch_iters if args.launch_iters > 0 else 1_000_000) // every * every)
    done = 0
    t_run = time.time()
    while done < args.n:
        n_it = min(per_launch, args.n - done)
        recs = chains.run(n_it, every)
        for r in range(recs.shape[0]):
            it = int(recs[r, 0, E.REC_IT])
            if it % s_freq == 0:
                for k in range(n_local):
                    writers[k].write(recs[r, k])
            if it % p_freq == 0 and not args.quiet:
                _print_state(recs[r, 0], float(end_time), args.calc_adequacy)
        done += n_it
    t_run = time.time() - t_run
    for w in writers:
        w.close()
    _warn_capacity(chains)
    if not args.quiet:
        print("literate_b200: %d chains x %d iterations in %.3f s (%.3g it/s)" % (n_local, args.n, t_run, n_local * args.n / max(t_run, 1e-9)))
    chains.close(); ds.close()
    return paths


def _warn_capacity(chains):
    """An add-shift proposal on a side that already holds LR_KMAX rates is rejected on the device; the reference would have
    evaluated it (its only bound is the spacing guard, LiteRateForward.py:290, i.e. K <= n_bins).  Tell the user if that happened."""
    rej = int(chains.counters()[:, 7].sum())
    if rej:
        warn("literate_b200: %d add-shift proposals were rejected because a side already held LR_KMAX = %d rates; "
             "the reference has no such limit below n_bins, so this run may differ from it in the far tail of the number of shifts"
             % (rej, E.LR_KMAX), RuntimeWarning)


def main(argv=None):
    args = build_parser().parse_args(argv)
    if args.d == "":
        raise SystemExit("no input file: use -d <table of lineages>")
    run(args)


if __name__ == "__main__":
    main()
