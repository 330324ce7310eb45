"""K9 (lr_chain_diagnostics) on one GPU, against a torch.fft route timed in the same run.

  (a) K7 records of hpd_bench.py (b): 4096 chains x 500 samples x 200 bins, every column of diagnostics.diagnostic_columns("dd")
  (b) K3 records of hpd_bench.py (a): 4096 chains x 500 samples on 200 bins, the record columns and the 600 per-bin marginal
      rates (K5 matrices, diagnostics.diagnose_records_device)
  (c) (a) as ladders of 4: every sample's cold member is (a)'s record of the chain (its position rotates), the three hot members
      hold other chains' records at beta 0.5; K9 picks the cold members, so the outputs must equal (a)'s bit for bit

  python tools/diag_bench.py [reps]
Prints the card's name and power limit, K9's time (CUDA events around the call, which returns when the outputs are written), the
lag blocks run, the largest lag, and the bytes K9 reads (a model: the moments pass reads every used value once, a CTA of a lag
block its draws plus a halo of its lags) over the time.  The fft route: the columns gathered, centred per split chain, the
autocovariances of all lags by rfft / irfft over 2n points, summed over split chains on the device; sections 3-7 of
diagnostics.rhat_ess on the host.  Its outputs are compared with K9's.
"""
import math
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from literate_b200 import ddrate as DD, diagnostics as D, engine as E, summary as S, synth

CHUNK = 1 << 30


def blocks_for(max_lag, n):
    """lag blocks of K9 (widths 16, 32, ... 4096) until the block holding lag max_lag + 2"""
    t1, w, k = 0, 16, 0
    while True:
        t1 = min(t1 + w, n)
        k += 1
        if t1 > max_lag + 2 or t1 >= n:
            return k
        w = min(2 * w, 4096)


def k9_bytes(m, n, n_cols, n_blocks):
    b, w, total = 0, 16, float(m * n * n_cols * 8)
    for _ in range(n_blocks):
        cl = min(w, 64)
        total += math.ceil(w / cl) * (2 * 64 + cl) / 64 * m * n * n_cols * 8
        w = min(2 * w, 4096)
    return total


def timed(fn, reps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    out = fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        a.record(); out = fn(); b.record(); torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
    return out, ms


def geyer_host(rho_of, n, m):
    """sections 5-7 of rhat_ess given rho_t (a callable) -> (ess, lag)"""
    rho = np.zeros(n + 1)
    rho[0], rho[1] = 1.0, rho_of(1)
    even, odd, t = 1.0, rho[1], 1
    while t < n - 3 and even + odd > 0:
        even, odd = rho_of(t + 1), rho_of(t + 2)
        if even + odd >= 0:
            rho[t + 1], rho[t + 2] = even, odd
        t += 2
    max_t = t - 2
    if even > 0:
        rho[max_t + 1] = even
    t = 1
    while t <= max_t - 2:
        if rho[t + 1] + rho[t + 2] > rho[t - 1] + rho[t]:
            rho[t + 1] = rho[t + 2] = (rho[t - 1] + rho[t]) / 2
        t += 2
    tau = max(-1.0 + 2.0 * np.sum(rho[:max_t + 1]) + rho[max_t + 1], 1.0 / math.log10(m * n))
    return m * n / tau, max_t


def fft_route(values_of, n_cols, S_, M):
    """values_of(c0, c1) -> float64 CUDA tensor [S, M, c1 - c0] of the columns; returns dict of numpy arrays"""
    n = S_ // 2
    m = 2 * M
    step = max(1, CHUNK // (8 * S_ * M * 6))
    out = {k: np.empty(n_cols) for k in ("mean", "sd", "rhat", "ess", "lag")}
    for c0 in range(0, n_cols, step):
        c1 = min(n_cols, c0 + step)
        x = values_of(c0, c1)
        sp = torch.stack([x[:n], x[S_ - n:]], dim=2).permute(1, 2, 0, 3).reshape(m, n, c1 - c0)   # [m, n, cols], split chain 2c, 2c + 1
        mean = sp.mean(dim=(0, 1))
        mj = sp.mean(dim=1)
        d = sp - mj[:, None, :]
        f = torch.fft.rfft(d, n=2 * n, dim=1)
        ac = torch.fft.irfft(f.real ** 2 + f.imag ** 2, n=2 * n, dim=1)[:, :n] / n          # acov_j(t)
        macov = ac.mean(dim=0).cpu().numpy()                                                  # [n, cols]
        between = mj.var(dim=0, unbiased=True).cpu().numpy()
        mean = mean.cpu().numpy()
        for j in range(c1 - c0):
            W = n / (n - 1) * macov[0, j]
            varp = (n - 1) / n * W + between[j]
            c = c0 + j
            out["mean"][c], out["sd"][c] = mean[j], math.sqrt(varp) if varp >= 0 else float("nan")
            if not np.isfinite(W) or W <= 0:
                out["rhat"][c], out["ess"][c], out["lag"][c] = float("nan"), float("nan"), -1
                continue
            out["rhat"][c] = math.sqrt(varp / W)
            out["ess"][c], out["lag"][c] = geyer_host(lambda t: 1.0 - (W - macov[t, j]) / varp, n, m)
    return out


def compare(k9, ff):
    g = {k: k9[k].cpu().numpy() if not hasattr(k9, "names") else getattr(k9, k) for k in ("rhat", "ess", "lag")}
    ok = np.isfinite(g["ess"]) & np.isfinite(ff["ess"])
    rel = lambda a, b: float(np.max(np.abs(a[ok] - b[ok]) / np.abs(b[ok]))) if ok.any() else 0.0
    return ("fft vs K9 over %d columns: R-hat max rel diff %.2e, ESS max rel diff %.2e, lags differ in %d"
            % (int(ok.sum()), rel(g["rhat"], ff["rhat"]), rel(g["ess"], ff["ess"]), int(np.sum(g["lag"][ok] != ff["lag"][ok]))))


def report(label, ms_k9, out, m, n, n_cols, ms_fft, cmp):
    lag = np.asarray(out["lag"].cpu().numpy() if isinstance(out, dict) else out.lag)
    mx = int(lag.max())
    nb = blocks_for(mx, n)
    by = k9_bytes(m, n, n_cols, nb)
    t = min(ms_k9)
    print("%s: K9 %.1f ms (runs %s), %d lag blocks, largest lag %d, reads %.1f GB (model) = %.0f GB/s; torch.fft route %.1f ms "
          "(device and host); %s" % (label, t, ["%.1f" % x for x in ms_k9], nb, mx, by / 1e9, by / (t * 1e-3) / 1e9, ms_fft, cmp))


def main(reps=3):
    dev = E.Device(0)
    tdev = torch.device("cuda:0")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
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
    cols = D.diagnostic_columns("dd", nb)
    specs = [c[1] for c in cols]
    out_a, ms = timed(lambda: dev.chain_diagnostics_device(recs, specs), reps)

    def vals(c0, c1):
        parts = []
        for c in specs[c0:c1]:
            a, b, sg, add = (c, -1, 1, 0.0) if np.ndim(c) == 0 else (tuple(c) + (0.0,))[:4]
            v = recs[..., a]
            if b >= 0:
                v = v + recs[..., b] if sg > 0 else v - recs[..., b]
            parts.append(v + add if add != 0.0 else v)
        return torch.stack(parts, dim=2)

    t0 = time.perf_counter(); ff = fft_route(vals, len(specs), 500, 4096); torch.cuda.synchronize(); ms_f = (time.perf_counter() - t0) * 1e3
    report("(a) K7: 4096 chains x 500 samples, %d columns (%.1f GB of records)" % (len(specs), recs.numel() * 8 / 1e9), ms, out_a,
           8192, 250, len(specs), ms_f, compare(out_a, ff))
    # ---- (c) the same as ladders of 4
    T = 4
    w = dd.rec_doubles
    lad = torch.empty((500, 4096 * T, w), dtype=torch.float64, device=tdev).view(500, 4096, T, w)
    pos = (torch.arange(500, device=tdev)[:, None] + torch.arange(4096, device=tdev)[None, :]) % T
    for k in range(T):
        lad[:, :, k] = torch.roll(recs, shifts=k + 1, dims=1)
        lad[:, :, k, DD.REC_BETA] = 0.5
    lad.scatter_(2, pos[:, :, None, None].expand(500, 4096, 1, w), recs[:, :, None, :])
    lad = lad.view(500, 4096 * T, w)
    out_c, ms = timed(lambda: dev.chain_diagnostics_device(lad, specs, T, DD.REC_BETA), reps)
    same = all(bool(torch.equal(out_a[k].view(torch.int64), out_c[k].view(torch.int64))) for k in out_a)
    report("(c) K7 as ladders of 4: %d device chains (%.1f GB of records)" % (4096 * T, lad.numel() * 8 / 1e9), ms, out_c, 8192, 250,
           len(specs), float("nan"), "outputs bit-identical to (a): %s" % same)
    del lad, recs, dd
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
    out_b, ms = timed(lambda: D.diagnose_records_device(dev, rec, "forward", 200, burnin=0.0, origin=1800.0), reps)
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

    t0 = time.perf_counter(); ff = fft_route(vals_b, len(out_b.names), 500, 4096); torch.cuda.synchronize(); ms_f = (time.perf_counter() - t0) * 1e3
    report("(b) K3: 4096 chains x 500 samples, %d record + 600 per-bin columns (K9 and the K5 matrices)" % len(fcols), ms, out_b,
           8192, 250, len(out_b.names), ms_f, compare({k: torch.from_numpy(np.asarray(getattr(out_b, k), dtype=np.float64)) for k in ("rhat", "ess", "lag")}, ff))


if __name__ == "__main__":
    main(int(sys.argv[1]) if len(sys.argv) > 1 else 3)
