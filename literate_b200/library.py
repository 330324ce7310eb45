"""What the TrendRate and DDRate command lines share, as the reference keeps it in literate_library.py: the table parser
(parse_ts_te), the unit bins (create_bins), the core flags (core_arguments) and the seed rule (set_seed), plus the host
plumbing of their chain objects (K6 lr_trend_t, K7 lr_dd_t), their tempered ladders (-temper) and the sampling loop that
writes their logs.
"""
from __future__ import annotations

import argparse
import ctypes as C
import glob
import os
import time
from warnings import warn

import numpy as np

from . import _native as N
from . import engine as E
from . import parallel as P


def parse_ts_te(path, TBP=False, first_year=-1, last_year=-1, death_jitter=0.5):
    """literate_library.parse_ts_te (:196-229) -> (ts, te, present, origin); the same pandas parser as the reference."""
    import pandas as pd
    t = pd.read_csv(path, delimiter="\t").to_numpy()
    if t.shape[1] == 4:
        warn('Four column (with clade) LiteRate input is deprecated. Use three columns.', FutureWarning)
        ts_y, te_y = t[:, 2], t[:, 3]
    else:
        ts_y, te_y = t[:, 1], t[:, 2]
    ts_y = np.asarray(ts_y, dtype=np.float64)
    te_y = np.asarray(te_y, dtype=np.float64).copy()
    if TBP:
        if first_year != -1:
            keep = ts_y <= first_year
            ts_y, te_y = ts_y[keep], te_y[keep]
        if last_year != -1:                      # (the reference masks te with the already filtered ts, :210-211)
            keep = ts_y >= last_year
            ts_y, te_y = ts_y[keep], te_y[keep]
            te_y[te_y < last_year] = last_year
        root = np.max(ts_y)
        ts, te = root - ts_y, root - te_y
    else:
        if first_year != -1:
            keep = ts_y >= first_year
            ts_y, te_y = ts_y[keep], te_y[keep]
        if last_year != -1:
            keep = ts_y <= last_year
            ts_y, te_y = ts_y[keep], te_y[keep]
            te_y[te_y > last_year] = last_year
        ts, te = ts_y, te_y
    te = te + death_jitter
    return ts, te, float(np.max(te)), float(np.min(ts))


def bin_window(origin, present, rm_first_bin=0):
    """(first_bin, n_bins) of literate_library.create_bins (:231-257): unit bins over np.arange(origin, present + 1), the
    last one always dropped, the first one too with -rm_first_bin."""
    if origin != np.floor(origin):
        raise SystemExit("the first birth time (%r) is not an integer: the unit bins of create_bins would not be aligned with "
                         "the integer bin edges K1 works on" % origin)
    n_edges = len(np.arange(origin, present + 1))
    n_bins = n_edges - 2
    first = int(origin)
    if rm_first_bin:
        first, n_bins = first + 1, n_bins - 1
    if n_bins < 1:
        raise SystemExit("the time window holds no bin after dropping the last one")
    return first, n_bins


def build_parser(prog, add_own):
    """The flags of literate_library.core_arguments (:290-308), then the script's own (add_own(parser)), then -chains,
    -device, -quiet and the tempering flags of literate_b200.forward (-temper, -swap_every, -temper_delta)."""
    p = argparse.ArgumentParser(prog=prog)
    p.add_argument('-v', action='version', version='%(prog)s')
    p.add_argument('-d', type=str, help='data file', default="", metavar="")
    p.add_argument('-n', type=int, help='n. MCMC iterations', default=10000000, metavar=10000000)
    p.add_argument('-p', type=int, help='print frequency', default=1000, metavar=1000)
    p.add_argument('-s', type=int, help='sampling frequency', default=1000, metavar=1000)
    p.add_argument('-seed', type=int, help='seed (set to -1 to make it random)', default=-1, metavar=-1)
    p.add_argument('-TBP', help='Default is AD. Include for TBP.', default=False, action='store_true')
    p.add_argument('-first_year', type=int, help='different start of the dataset', default=-1, metavar=-1)
    p.add_argument('-last_year', type=int, help='different end of the dataset', default=-1, metavar=-1)
    p.add_argument('-death_jitter', type=float, help='amount to jitter death times', default=.5, metavar=.5)
    p.add_argument('-rm_first_bin', type=float, help='if set to 1 it removes the first time bin', default=0, metavar=0)
    p.add_argument('-print_emp', help='Prints empirical rates', default=False, action='store_true')
    add_own(p)
    # ---- not in the reference
    p.add_argument('-chains', type=int, help='number of independent chains run concurrently on the GPU', default=1, metavar=1)
    p.add_argument('-device', type=int, help='CUDA device index', default=0, metavar=0)
    p.add_argument('-quiet', type=int, help='1: no per-sample progress on stdout', default=0, metavar=0)
    p.add_argument('-temper', type=int, help='temperatures per logged chain (1: no tempering, as the reference)', default=1, metavar=1)
    p.add_argument('-swap_every', type=int, help='iterations between temperature-swap rounds', default=1000, metavar=1000)
    p.add_argument('-temper_delta', type=float, help='ladder beta_k = 1/(1 + delta k)', default=0.1, metavar=0.1)
    return p


def seed_and_chains(args, world):
    """set_seed (literate_library.py:282-288): -seed -1 draws the seed; with several GPUs every rank must be given the same
    one.  There must be at least one chain per GPU, and -temper must be 1..32 (checked before any device is touched)."""
    if not (1 <= args.temper <= 32):
        raise SystemExit("-temper must be 1..32")
    if args.seed == -1:
        if world > 1:
            raise SystemExit("give -seed explicitly when running on several GPUs (every rank must use the same one)")
        seed = int(np.random.randint(0, 9999))
    else:
        seed = args.seed
    if args.chains < max(1, world):
        raise SystemExit("-chains must be >= 1 and at least the number of GPUs")
    return seed


def read_tables(args, exclude):
    """The tables of -d: one file, or every .tsv/.txt file of a directory (stochastic imputations of one data set) except
    `exclude`, one replicate each over the common window.  -chains 1 becomes one chain per table, and -chains must be a
    multiple of the number of tables.  Returns (tables, ts, te, present, origin), ts / te NaN-padded [n_tables, n_max]."""
    if os.path.isdir(args.d):
        tables = sorted(f for f in glob.glob(os.path.join(args.d, "*")) if os.path.isfile(f) and f.lower().endswith((".tsv", ".txt"))
                        and os.path.abspath(f) != os.path.abspath(exclude))
        if not tables:
            raise SystemExit("no .tsv/.txt table in " + args.d)
    else:
        tables = [args.d]
    parsed = [parse_ts_te(f, args.TBP, args.first_year, args.last_year, args.death_jitter) for f in tables]
    n_tab = len(parsed)
    if args.chains == 1 and n_tab > 1:
        args.chains = n_tab
    if args.chains % n_tab:
        raise SystemExit("-chains must be a multiple of the number of tables (%d)" % n_tab)
    present, origin = max(p[2] for p in parsed), min(p[3] for p in parsed)
    n_max = max(len(p[0]) for p in parsed)
    ts = np.full((n_tab, n_max), np.nan); te = np.full((n_tab, n_max), np.nan)      # NaN rows carry no event and no time at risk
    for i, p in enumerate(parsed):
        ts[i, :len(p[0])], te[i, :len(p[1])] = p[0], p[1]
    return tables, ts, te, present, origin


class ChainObject(E.Tempered):
    """A population of independent chains of one of the sibling samplers on one device: the C entry points
    lr_<PREFIX>_* of lr_trend_t (K6) and lr_dd_t (K7), tempered ladders included (engine.Tempered).  Subclasses create the
    object and set dev, n_chains, n_bins and t; REC_BETA is the field of beta in their records."""
    STATE_DOUBLES = 0
    REC_BETA = 0

    def _handle(self):
        return self.t

    @staticmethod
    def _inputs(sp, ex, br, rep_of_chain, n_chains):
        """sp, ex, br as [n_rep, n_bins] arrays of the C types and the replicate of every chain (None: replicate 0)."""
        sp = np.ascontiguousarray(np.atleast_2d(sp), dtype=np.int64)
        ex = np.ascontiguousarray(np.atleast_2d(ex), dtype=np.int64)
        br = np.ascontiguousarray(np.atleast_2d(br), dtype=np.float64)
        rep = None
        if rep_of_chain is not None:
            rep = np.ascontiguousarray(rep_of_chain, dtype=np.int32)
            if rep.shape != (int(n_chains),):
                raise ValueError("rep_of_chain must have one entry per chain")
        return sp, ex, br, rep

    def _created(self, t):
        self.t = t
        self.rec_doubles = int(self._lr("record_doubles")(self.n_bins))

    def close(self):
        if getattr(self, "t", None):
            self._lr("destroy")(self.t)
            self.t = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def records_per_run(self, n_iter, sample_every):
        return int(self._lr("records_per_run")(self.t, int(n_iter), int(sample_every)))

    def run(self, n_iter, sample_every=0):
        """n_iter iterations of every chain; returns records [n_samples, n_chains, rec_doubles] (host) or None."""
        name = "lr_%s_run_host" % self.PREFIX
        if sample_every and sample_every > 0:
            out = np.empty((self.records_per_run(n_iter, sample_every), self.n_chains, self.rec_doubles), dtype=np.float64)
            N.check(self._lr("run_host")(self.t, int(n_iter), int(sample_every), N.np_ptr(out)), name)
            return out
        N.check(self._lr("run_host")(self.t, int(n_iter), 0, None), name)
        return None

    def run_device(self, n_iter, sample_every, records, stream=None):
        """Asynchronous: `records` is a float64 CUDA tensor [n_samples, n_chains, rec_doubles] or None."""
        st = C.c_void_p(None) if isinstance(stream, str) and stream == "handle" else E._stream_ptr(stream)
        ptr = C.c_void_p(records.data_ptr()) if records is not None else None
        N.check(self._lr("run")(self.t, int(n_iter), int(sample_every) if records is not None else 0, ptr, st), "lr_%s_run" % self.PREFIX)

    def state(self):
        out = np.empty((self.n_chains, self.STATE_DOUBLES), dtype=np.float64)
        N.check(self._lr("state_host")(self.t, N.np_ptr(out)), "lr_%s_state_host" % self.PREFIX)
        return out

    def temper(self):
        """(beta [n_chains], temperature swaps proposed / accepted int64 [n_chains, 2]) of every chain."""
        beta = np.empty(self.n_chains, dtype=np.float64)
        swaps = np.empty((self.n_chains, 2), dtype=np.int64)
        N.check(self._lr("temper_host")(self.t, N.np_ptr(beta), N.np_ptr(swaps)), "lr_%s_temper_host" % self.PREFIX)
        return beta, swaps


def ladders(args, c0, n_local, n_tab):
    """Device chains of this rank's logged chains [c0, c0 + n_local): with -temper T every logged chain k is the ladder of
    device chains [k T, (k + 1) T), all on table k % n_tab.  Returns (chain_id0, n_chains, rep_of_chain, beta or None)."""
    T = args.temper
    rep_of_chain = np.repeat(np.arange(c0, c0 + n_local) % n_tab, T).astype(np.int32)
    beta = np.tile(P.temperature_ladder(T, args.temper_delta), n_local) if T > 1 else None
    return c0 * T, n_local * T, rep_of_chain, beta


def sample_and_write(chains, n_iter, s, files, writers, row, progress, quiet, ladder=1, swap_every=1000):
    """Runs n_iter iterations of every chain, sampling every s-th, in launches of at most ~256 MB of records and 4M
    iterations; every sample of logged chain k becomes the log row row(rec) of writers[k], and unless quiet progress(rec) of
    chain 0 goes to stdout.  ladder > 1: the chains are ladders of `ladder` consecutive chains with a swap round every
    swap_every iterations (run_tempered, the round counter carried across launches), and only the cold member of each
    ladder is logged.  Closes the files; returns (wall time of the run, swap rounds done)."""
    n_dev = chains.n_chains
    s_freq = max(1, s)
    max_rec = max(1, (256 << 20) // (n_dev * chains.rec_doubles * 8))
    per_launch = max(s_freq, min(max_rec * s_freq, 4_000_000) // s_freq * s_freq)
    done = rounds = 0
    t_run = time.time()
    while done < n_iter:
        n_it = min(per_launch, n_iter - done)
        if ladder > 1:
            recs, r = chains.run_tempered(n_it, s_freq, ladder, max(1, swap_every), round0=rounds)
            rounds += r
            recs = E.cold_records(recs, ladder, chains.REC_BETA)
        else:
            recs = chains.run(n_it, s_freq)
        done += n_it
        n_local = recs.shape[1]
        for r in range(recs.shape[0]):
            for k in range(n_local):
                writers[k].writerow(row(recs[r, k]))
            if not quiet:
                progress(recs[r, 0])
        for fh in files:
            fh.flush()
    t_run = time.time() - t_run
    for fh in files:
        fh.close()
    return t_run, rounds
