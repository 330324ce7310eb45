"""Tempered TrendRate (K6) and DDRate (K7) ladders:
    python tools/sibling_temper_bench.py [iters] [T,T,...] [n_bins,...] [out.json]

For 256 logged chains x T temperatures (ladders of T consecutive chains, beta_k = 1/(1 + 0.1 k)) and a swap round every
1000 iterations -- what `-temper T -swap_every 1000` runs -- reports per sampler, bin count and T:
  wall_s            wall time of run_tempered (records every 1000 iterations, as -s 1000), host clock around synchronised work
  cold_it_per_s     iterations of the 256 cold chains per second of wall time; cold_samples_per_s the logged samples
  swap_acceptance   accepted / proposed temperature swaps
  swap_share        share of wall_s spent in swap rounds (swap_step, synchronised on both sides)
  boundary_share    share of wall_s lost to the launch boundaries run_tempered adds: wall_s - swap time - the time of the
                    same iterations and records in one launch per 20 000 iterations
Synthetic tables (those of tools/k6_bench.py and tools/k7_bench.py).  Prints one line per case; with out.json also writes
all results there as JSON.
"""
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from literate_b200 import ddrate as DD, engine as E, parallel as P, trend as TR

iters = int(sys.argv[1]) if len(sys.argv) > 1 else 20000
temps = [int(c) for c in (sys.argv[2] if len(sys.argv) > 2 else "1,2,4,8").split(",")]
bins_list = [int(c) for c in (sys.argv[3] if len(sys.argv) > 3 else "24,200").split(",")]
N_LOG, EVERY, SWAP_EVERY, PLAIN_LAUNCH = 256, 1000, 1000, 20000
dev = E.Device(0)
rng = np.random.default_rng(1)


def make(kind, nb, n):
    if kind == "k6":
        br = rng.uniform(50, 500, nb)
        trend = np.clip(np.linspace(0, 1, nb) + 0.05 * rng.normal(size=nb), 1e-15, 1.0)
        sp = rng.poisson(br * (0.1 + 0.2 * trend)); ex = rng.poisson(br * (0.05 + 0.1 * trend))
        return lambda: TR.TrendChains(dev, sp, ex, br, trend, n, 1)
    t = np.arange(nb)
    br = 20 + 400 / (1 + np.exp(-0.3 * (t - nb / 2))) + rng.uniform(0, 5, nb)
    sp = rng.poisson(br * 0.2); ex = rng.poisson(br * 0.1)
    gts = np.sort(rng.uniform(0, nb * .7, 40)).round(); gte = np.minimum(gts + rng.integers(1, nb, 40), nb) + .5
    return lambda: DD.DDChains(dev, sp, ex, br, 0.0, nb + 1.5, 3, 2, gts, gte, n, 1)


res = {"gpu": torch.cuda.get_device_name(0), "iters": iters, "logged_chains": N_LOG, "swap_every": SWAP_EVERY}
try:
    import subprocess
    res["power_limit"] = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                                        capture_output=True, text=True).stdout.strip()
except Exception as e:                                     # noqa: BLE001
    res["power_limit"] = "unknown (%s)" % e
print(res, flush=True)
for kind in ("k6", "k7"):
    for nb in bins_list:
        for T in temps:
            n = N_LOG * T
            mk = make(kind, nb, n)
            beta = np.tile(P.temperature_ladder(T, 0.1), N_LOG)
            # the same iterations and records in long launches: the reference point of the boundary cost
            plain = mk()
            plain.set_beta(beta)
            plain.run(2000)
            dev.sync()
            t0 = time.perf_counter()
            done = 0
            while done < iters:
                k = min(PLAIN_LAUNCH, iters - done)
                plain.run(k, EVERY)
                done += k
            dev.sync()
            t_plain = time.perf_counter() - t0
            plain.close()

            ch = mk()
            ch.set_beta(beta)
            ch.run(2000)
            t_swap = [0.0]

            def swap(rnd):
                dev.sync()
                a = time.perf_counter()
                ch.swap_step(T, rnd)
                dev.sync()
                t_swap[0] += time.perf_counter() - a

            dev.sync()
            t0 = time.perf_counter()
            if T > 1:
                recs, rounds = ch.run_tempered(iters, EVERY, T, SWAP_EVERY, swap=swap)
                cold = E.cold_records(recs, T, ch.REC_BETA)
            else:
                cold, rounds = ch.run(iters, EVERY), 0
            dev.sync()
            wall = time.perf_counter() - t0
            sw = ch.temper()[1].sum(0)
            key = "%s_%dbins_T%d" % (kind, nb, T)
            res[key] = {"wall_s": wall, "cold_it_per_s": N_LOG * iters / wall, "cold_samples_per_s": cold.shape[0] * cold.shape[1] / wall,
                        "device_chains": n, "swap_rounds": rounds, "swap_acceptance": float(sw[1] / max(sw[0], 1)),
                        "swap_share": t_swap[0] / wall, "boundary_share": max(0.0, wall - t_swap[0] - t_plain) / wall,
                        "plain_wall_s": t_plain}
            print(key, res[key], flush=True)
            ch.close()
if len(sys.argv) > 4:
    with open(sys.argv[4], "w") as fh:
        json.dump(res, fh, indent=1)
