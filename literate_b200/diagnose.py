"""Convergence diagnostics of the sample logs in a directory: split R-hat and effective sample size of every logged column over
the chains of each kind of run (K9, literate_b200.diagnostics).

  python -m literate_b200.diagnose <dir> [-burnin .2] [-rhat_max 1.01] [-ess_min 200] [-device 0] [-rank 0]

For each kind (RJMCMC *_mcmc.log, *.trendrate.log, DDRate logs) every log of that kind in <dir> is one chain of the set (the set
`-combine 1` pools).  Burn-in is removed per chain; chains of different lengths are cut to the shortest.  Writes
<dir>/diagnostics_<kind>.tsv with the columns `column mean sd rhat ess mcse lag flag` (mcse = sd / sqrt(ess); flag ok | rhat |
ess | rhat+ess | const | stuck | nonfinite) and prints a short report per kind.  With -rank 1 it also writes
<dir>/diagnostics_<kind>_rank.tsv with the rank-normalised diagnostics (K10, diagnostics.rank_rhat_ess), the columns
`column median q05 q95 rhat_rank rhat_bulk rhat_tail ess_bulk ess_tail flag`, and prints one more line per kind.
"""
from __future__ import annotations

import argparse
import os

import numpy as np

from . import diagnostics as D
from . import engine as E


def _extreme(values, names, pick):
    v = np.asarray(values, dtype=np.float64)
    ok = ~np.isnan(v)
    if not ok.any():
        return float("nan"), "-"
    i = int(np.flatnonzero(ok)[pick(v[ok])])
    return float(v[i]), names[i]


def main(argv=None):
    p = argparse.ArgumentParser(prog="diagnose")
    p.add_argument('input_data', metavar='<path to log files>', type=str)
    p.add_argument('-burnin', metavar='.2', type=float, default=.2)
    p.add_argument('-rhat_max', metavar='1.01', type=float, default=1.01)
    p.add_argument('-ess_min', metavar='200', type=float, default=200.0)
    p.add_argument('-device', metavar='0', type=int, default=0)
    p.add_argument('-rank', metavar='0', type=int, default=0, help='1: also the rank-normalised R-hat and bulk / tail ESS')
    a = p.parse_args(argv)
    logs = D.find_logs(a.input_data)
    if not logs:
        raise SystemExit("no *_mcmc.log, *.trendrate.log or DDRate sample log under " + a.input_data)
    dev = E.Device(a.device)
    written = []
    for kind, files in logs.items():
        d = D.diagnose_logs(files, a.burnin, dev, note=lambda s, k=kind: print("%s: %s" % (k, s)), rank=bool(a.rank))
        path = d.write_tsv(os.path.join(a.input_data, "diagnostics_%s.tsv" % kind), a.rhat_max, a.ess_min)
        flags = d.flags(a.rhat_max, a.ess_min)
        r, rn = _extreme(d.rhat, d.names, np.argmax)
        e, en = _extreme(d.ess, d.names, np.argmin)
        print("%s: %d chains x %d draws; worst R-hat %.4f (%s), lowest ESS %.1f (%s); %d of %d columns flagged; %s"
              % (kind, d.n_chains, d.n_draws, r, rn, e, en, sum(f != "ok" for f in flags), len(flags), path))
        written.append(path)
        if a.rank:
            rpath = d.write_rank_tsv(os.path.join(a.input_data, "diagnostics_%s_rank.tsv" % kind), a.rhat_max, a.ess_min)
            rflags = d.rank_flags(a.rhat_max, a.ess_min)
            r, rn = _extreme(d.rhat_rank, d.names, np.argmax)
            e, en = _extreme(d.ess_tail, d.names, np.argmin)
            print("%s: rank-normalised: worst R-hat %.4f (%s), lowest tail ESS %.1f (%s); %d of %d columns flagged; %s"
                  % (kind, r, rn, e, en, sum(f != "ok" for f in rflags), len(rflags), rpath))
            written.append(rpath)
    return written


if __name__ == "__main__":
    main()
