"""K10 (lr_rank_diagnostics) on one GPU, next to K9's plain call and to a torch route timed in the same run.

  (a) K7 records of diag_bench.py (a): 4096 chains x 500 samples x 200 bins, every column of diagnostics.diagnostic_columns("dd")
  (b) K3 records of diag_bench.py (b): 4096 chains x 500 samples on 200 bins, the record columns and the 600 per-bin marginal
      rates (K5 matrices, diagnostics.diagnose_records_device with and without rank=True)

  python tools/rank_diag_bench.py [reps]
Prints the card's name, power limit and clock, then per workload K9's time, K10's time (CUDA events around calls that return when
their outputs are written) and the torch route's: per chunk of columns torch.sort of the split draws, searchsorted ranks (left and
right side, the average of ties), torch.special.ndtri, the median and quantiles from sorted columns, the folded values sorted and
ranked the same way, the indicators, then K9 on the 4 columns per column and the degenerate rules on the host.  The outputs of
the torch route are compared with K10's.
"""
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import numpy as np
import torch

from literate_b200 import ddrate as DD, diagnostics as D, engine as E, synth
from diag_bench import timed

CHUNK = 1 << 30


def _z(sorted_, v, N):
    lo = torch.searchsorted(sorted_, v, side="left")
    hi = torch.searchsorted(sorted_, v, side="right")
    r = lo.double() + 0.5 * (hi - lo + 1).double()
    num, rest, den = r - 0.375, N + 0.625 - r, N + 0.25
    return torch.where(num <= rest, torch.special.ndtri(num / den), -torch.special.ndtri(rest / den))


def _quantile(s, p):
    n = s.shape[0]
    h = (n - 1) * p
    lo = int(np.floor(h))
    a, b, g = s[lo], s[min(lo + 1, n - 1)], h - lo
    d = b - a
    return b - d * (1.0 - g) if g >= 0.5 else a + d * g


def torch_route(dev, values_of, n_cols, S_, M):
    """values_of(c0, c1) -> float64 CUDA tensor [S, M, c1 - c0]; returns dict of numpy arrays as rank_diagnostics_device"""
    n = S_ // 2
    N = 2 * n * M
    step = max(1, CHUNK // (8 * S_ * M * 10))
    out = {k: np.empty(n_cols) for k in E.RANK_FIELDS}
    for c0 in range(0, n_cols, step):
        c1 = min(n_cols, c0 + step)
        k = c1 - c0
        x = values_of(c0, c1)
        xs = torch.cat([x[:n], x[S_ - n:]], dim=0)                      # [2n, M, k], the rows of Z
        Z = torch.empty((2 * n, M, 4 * k), dtype=torch.float64, device=x.device)
        quant = torch.empty((3, k), dtype=torch.float64, device=x.device)
        finite = torch.isfinite(xs).reshape(N, k).all(dim=0).cpu().numpy()
        for j in range(k):
            v = xs[..., j].reshape(-1)
            s = torch.sort(v).values
            med = (s[N // 2 - 1] + s[N // 2]) / 2
            sa = torch.sort(x[..., j].reshape(-1)).values
            q05, q95 = _quantile(sa, 0.05), _quantile(sa, 0.95)
            Z[..., j] = _z(s, v, N).view(2 * n, M)
            f = (v - med).abs()
            Z[..., k + j] = _z(torch.sort(f).values, f, N).view(2 * n, M)
            Z[..., 2 * k + j] = (xs[..., j] <= q05).double()
            Z[..., 3 * k + j] = (xs[..., j] <= q95).double()
            quant[0, j], quant[1, j], quant[2, j] = med, q05, q95
        r9 = dev.chain_diagnostics_device(Z, list(range(4 * k)))
        rh, es = r9["rhat"].cpu().numpy(), r9["ess"].cpu().numpy()
        qn = quant.cpu().numpy()
        for j in range(k):
            c = c0 + j
            rb, rt = rh[j], rh[k + j]
            if not finite[j] or not np.isfinite(rb):
                for f_ in E.RANK_FIELDS:
                    out[f_][c] = np.nan
                continue
            e = [float(N) if np.isnan(rh[(2 + t) * k + j]) else es[(2 + t) * k + j] for t in (0, 1)]
            out["median"][c], out["q05"][c], out["q95"][c] = qn[0, j], qn[1, j], qn[2, j]
            out["rhat_bulk"][c], out["rhat_tail"][c] = rb, rt
            out["rhat_rank"][c] = rb if np.isnan(rt) else max(rb, rt)
            out["ess_bulk"][c] = es[j]
            out["ess_tail"][c] = np.nan if np.isnan(e[0]) or np.isnan(e[1]) else min(e)
    return out


def compare(k10, tr):
    g = {k: (k10[k].cpu().numpy() if isinstance(k10, dict) else np.asarray(getattr(k10, k))) for k in E.RANK_FIELDS}
    parts = []
    for k in E.RANK_FIELDS:
        a, b = g[k], tr[k]
        both = np.isnan(a) & np.isnan(b)
        ok = np.isfinite(a) & np.isfinite(b)
        rel = float(np.max(np.abs(a[ok] - b[ok]) / np.maximum(np.abs(b[ok]), 1e-300))) if ok.any() else 0.0
        parts.append("%s %.1e%s" % (k, rel, "" if (both | ok | (a == b)).all() else " (NaN differs in %d)" % int((~(both | ok | (a == b))).sum())))
    return "torch route vs K10, max rel diff: " + ", ".join(parts)


def report(label, ms9, ms10, ms_t, cmp):
    print("%s: K9 %.1f ms (runs %s); K10 %.1f ms (runs %s); torch route %.1f ms; %s"
          % (label, min(ms9), ["%.1f" % x for x in ms9], min(ms10), ["%.1f" % x for x in ms10], ms_t, cmp))


def main(reps=3):
    dev = E.Device(0)
    tdev = torch.device("cuda:0")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    print("GPU:", torch.cuda.get_device_name(0), "|", q.stdout.strip())
    # ---- (a) K7 records, every diagnosed column
    nb = 200
    rng = np.random.default_rng(1)
    t = np.arange(nb)
    brk = 20 + 400 / (1 + np.exp(-0.3 * (t - nb / 2))) + rng.uniform(0, 5, nb)
    dd = DD.DDChains(dev, rng.poisson(brk * 0.2), rng.poisson(brk * 0.1), brk, 0.0, nb + 1.5, 2, 2, n_chains=4096, seed=1)
    dd.run(3000)
    recs = torch.empty((500, 4096, dd.rec_doubles), dtype=torch.float64, device=tdev)
    dd.run_device(50000, 100, recs)
    torch.cuda.synchronize()
    specs = [c[1] for c in D.diagnostic_columns("dd", nb)]
    _, ms9 = timed(lambda: dev.chain_diagnostics_device(recs, specs), reps)
    out_a, ms10 = timed(lambda: dev.rank_diagnostics_device(recs, specs), reps)
    again = dev.rank_diagnostics_device(recs, specs)
    same = all(bool(torch.equal(out_a[k].view(torch.int64), again[k].view(torch.int64))) for k in out_a)

    def vals(c0, c1):
        parts = []
        for c in specs[c0:c1]:
            a, b, sg, add = (c, -1, 1, 0.0) if np.ndim(c) == 0 else (tuple(c) + (0.0,))[:4]
            v = recs[..., a]
            if b >= 0:
                v = v + recs[..., b] if sg > 0 else v - recs[..., b]
            parts.append(v + add if add != 0.0 else v)
        return torch.stack(parts, dim=2)

    t0 = time.perf_counter(); tr = torch_route(dev, vals, len(specs), 500, 4096); torch.cuda.synchronize()
    ms_t = (time.perf_counter() - t0) * 1e3
    report("(a) K7: 4096 chains x 500 samples, %d columns (%.1f GB of records)" % (len(specs), recs.numel() * 8 / 1e9), ms9, ms10, ms_t,
           compare(out_a, tr) + "; repeated K10 call bit-identical: %s" % same)
    del recs, dd
    torch.cuda.empty_cache()
    # ---- (b) K3 records, record columns and per-bin marginals
    ts, te = synth.syn_int_device(1_000_000, 1, tdev)
    sp, ex, br = dev.bin_stats_device(ts[:, :1_000_000], te[:, :1_000_000], 1800, 200)
    torch.cuda.synchronize()
    ds = E.Dataset.from_device(dev, sp, ex, br, 0, 1800.0, 2000.5)
    ch = E.Chains(ds, 4096, 1)
    ch.run(3000)
    rec = torch.empty((500, 4096, 144), dtype=torch.float64, device=tdev)
    ch.run_device(50000, 100, rec, stream="handle"); dev.sync()
    _, ms9 = timed(lambda: D.diagnose_records_device(dev, rec, "forward", 200, burnin=0.0, origin=1800.0), reps)
    out_b, msr = timed(lambda: D.diagnose_records_device(dev, rec, "forward", 200, burnin=0.0, origin=1800.0, rank=True), reps)
    ms10 = [b - a for a, b in zip(sorted(ms9), sorted(msr))]
    fcols = [c[1] for c in D.FORWARD_COLS]

    def vals_b(c0, c1):
        parts = []
        for c in range(c0, c1):
            if c < len(fcols):
                a, b, sg, add = (fcols[c], -1, 1, 0.0) if np.ndim(fcols[c]) == 0 else (tuple(fcols[c]) + (0.0,))[:4]
                parts.append(rec[..., a] + rec[..., b] if b >= 0 else rec[..., a])
            else:
                j, side = (c - len(fcols)) % 200, (c - len(fcols)) // 200
                mb, md = dev.marginal_rates_device(rec, 1800.0, 200, j, 1)
                parts.append((mb if side == 0 else md if side == 1 else mb - md).reshape(500, 4096))
        return torch.stack(parts, dim=2)

    t0 = time.perf_counter(); tr = torch_route(dev, vals_b, len(out_b.names), 500, 4096); torch.cuda.synchronize()
    ms_t = (time.perf_counter() - t0) * 1e3
    report("(b) K3: 4096 chains x 500 samples, %d record + 600 per-bin columns (K10 = diagnose_records_device with rank minus "
           "without, both including the K5 matrices)" % len(fcols), ms9, ms10, ms_t, compare(out_b, tr))


if __name__ == "__main__":
    main(int(sys.argv[1]) if len(sys.argv) > 1 else 3)
