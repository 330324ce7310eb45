"""K8 (lr_column_hpd) against torch.sort HPD intervals on one GPU, outputs compared bit for bit in the same run.

  (a) the K5 workload of k5_bench.py: 4096 chains x 500 samples of K3 records, birth, death and net rate over 200 bins, the
      per-sample matrices in the chunks summary.summarize_records_device hands to summary.hpd_device (at most 1 GB each); K8
      on the same chunks is what summary.hpd_device would do on it
  (b) K7 records of 4096 chains x 500 samples x 200 bins (13.5 GB), all 1011 columns of a DDRate log; torch.sort on gathered
      column chunks of at most 1 GB, K8 straight on the records

  python tools/hpd_bench.py [reps]
CUDA-event times, old and new alternated; prints the card's name and power limit.  Bytes: K8 reads the matrix nine times
(eight radix-select passes and the gather); GB/s = those bytes over the kernel time.
"""
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from literate_b200 import ddrate as DD, engine as E, plotdd as PD, synth

CHUNK = 1 << 30


def hpd_sort(x, level=0.95):
    """The body of summary.hpd_device: torch.sort of every column, then the first narrowest window."""
    s, _ = torch.sort(x, dim=0)
    n = s.shape[0]
    n_in = int(round(level * n))
    width = s[n_in - 1:] - s[:n - n_in + 1]
    i = torch.argmin(width, dim=0, keepdim=True)
    return s.gather(0, i)[0], s.gather(0, i + (n_in - 1))[0]


def timed(fn, reps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    out = fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        a.record(); fn(); b.record(); torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
    return out, ms


def same(a, b):
    return all(bool(((x == y) | (torch.isnan(x) & torch.isnan(y))).all()) for x, y in zip(a, b))


def compare(label, old, new, reps, read_bytes):
    """old / new: callables returning (lo, hi) over the whole workload; alternated reps times."""
    t_old, t_new, o, nw = [], [], None, None
    for _ in range(reps):
        o, ms = timed(old, 1); t_old += ms
        nw, ms = timed(new, 1); t_new += ms
    eq = same(o, nw)
    mo, mn = min(t_old), min(t_new)
    print("%s: torch.sort %.1f ms (runs %s), K8 %.1f ms (runs %s), speed-up %.2fx, bounds bit-identical: %s; K8 reads %.1f GB = %.0f GB/s"
          % (label, mo, ["%.1f" % t for t in t_old], mn, ["%.1f" % t for t in t_new], mo / mn, eq, read_bytes / 1e9, read_bytes / (mn * 1e-3) / 1e9))
    return eq


def main(reps=3):
    dev = E.Device(0)
    tdev = torch.device("cuda:0")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    print("GPU:", torch.cuda.get_device_name(0), "|", q.stdout.strip())
    ok = True
    # ---- (a) K5 workload
    ts, te = synth.syn_int_device(1_000_000, 1, tdev)
    sp, ex, br = dev.bin_stats_device(ts[:, :1_000_000], te[:, :1_000_000], 1800, 200)
    torch.cuda.synchronize()
    ds = E.Dataset.from_device(dev, sp, ex, br, 0, 1800.0, 2000.5)
    ch = E.Chains(ds, 4096, 1)
    ch.run(3000)
    rec = torch.empty((500, 4096, 144), dtype=torch.float64, device=tdev)
    ch.run_device(50000, 100, rec, stream="handle"); dev.sync()
    n = rec.shape[0] * rec.shape[1]
    step = max(1, min(200, CHUNK // (8 * n)))
    mats = []
    for lo in range(0, 200, step):
        mb, md = dev.marginal_rates_device(rec, 1800.0, 200, lo, min(step, 200 - lo))
        mats += [mb, md, mb - md]
    torch.cuda.synchronize()
    old = lambda: [hpd_sort(m) for m in mats]
    new = lambda: [dev.column_hpd_device(m, range(m.shape[1]))[1:3] for m in mats]
    flat = lambda f: lambda: tuple(torch.cat(p) for p in zip(*f()))
    ok &= compare("(a) K5: %d records x 200 bins x birth/death/net, %d chunks" % (n, len(mats)), flat(old), flat(new), reps,
                  9 * 8 * n * 600)
    del mats, rec, ch, ds
    torch.cuda.empty_cache()
    # ---- (b) K7 records, every column of the log
    nb = 200
    rng = np.random.default_rng(1)
    t = np.arange(nb)
    brk = 20 + 400 / (1 + np.exp(-0.3 * (t - nb / 2))) + rng.uniform(0, 5, nb)
    dd = DD.DDChains(dev, rng.poisson(brk * 0.2), rng.poisson(brk * 0.1), brk, 0.0, nb + 1.5, 2, 2, n_chains=4096, seed=1)
    dd.run(3000)
    recs = torch.empty((500, 4096, dd.rec_doubles), dtype=torch.float64, device=tdev)
    dd.run_device(50000, 100, recs)
    torch.cuda.synchronize()
    rows = recs.reshape(-1, dd.rec_doubles)
    specs = PD.column_specs("dd", nb, 1800.0)
    k = max(1, CHUNK // (8 * rows.shape[0]))

    def old_b():
        los, his = [], []
        for c0 in range(0, len(specs), k):
            part = specs[c0:c0 + k]
            cols = []
            for a, b, sg, add in part:
                v = rows[:, a]
                if b >= 0:
                    v = v + rows[:, b] if sg > 0 else v - rows[:, b]
                cols.append(v + add if add != 0.0 else v)
            lo, hi = hpd_sort(torch.stack(cols, dim=1))
            los.append(lo); his.append(hi)
        return torch.cat(los), torch.cat(his)

    def new_b():
        _, lo, hi, _ = dev.column_hpd_device(rows, specs)
        return lo, hi

    ok &= compare("(b) K7: %d records x %d columns (%.1f GB of records)" % (rows.shape[0], len(specs), recs.numel() * 8 / 1e9),
                  old_b, new_b, reps, 9 * 8 * rows.shape[0] * len(specs))
    if not ok:
        raise SystemExit("K8 and torch.sort disagree")


if __name__ == "__main__":
    main(int(sys.argv[1]) if len(sys.argv) > 1 else 3)
