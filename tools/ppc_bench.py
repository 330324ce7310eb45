"""K11 timing: the posterior predictive check on the K5 workload -- 256 chains x 8 000 records of real RJMCMC output on the
syn-int statistics (1 M lineages, 200 bins), 2.4 GB of records -- against the NumPy definition on a subsample, scaled.  Prints one
JSON line with the card's name and power limit, read in the same run.  python tools/ppc_bench.py [--reps 5] [--host-records 2000]"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from literate_b200 import engine as E, predictive as PP, synth


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        name, power = [s.strip() for s in q.stdout.splitlines()[0].split(",")]
        return name, power
    except Exception as e:                       # the timing stands without it, but says so
        return torch.cuda.get_device_name(0), "unknown (%s)" % type(e).__name__


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--host-records", type=int, default=2000)
    a = ap.parse_args()
    dev = E.Device(0)
    tdev = torch.device("cuda:0")
    ts, te = synth.syn_int_device(1_000_000, 1, tdev)
    sp, ex, br = dev.bin_stats_device(ts, te, 1800, 200)
    torch.cuda.synchronize()
    ds = E.Dataset.from_device(dev, sp, ex, br, 0, 1800.0, 2000.5)
    ch = E.Chains(ds, 256, 1)
    ch.run(3000)
    rec = torch.empty((8000, 256, E.LR_REC_DOUBLES), dtype=torch.float64, device=tdev)
    ch.run_device(800000, 100, rec, stream="handle")
    dev.sync()
    terms = ds.bin_terms()
    kw = dict(layout=0, start_time=1800.0, seed=7)
    for _ in range(2):
        dev.predictive_check_device(rec, terms=terms, **kw)
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for _ in range(a.reps):
        out = dev.predictive_check_device(rec, terms=terms, **kw)
    ev[1].record()
    torch.cuda.synchronize()
    ms = ev[0].elapsed_time(ev[1]) / a.reps
    draws = int(out["bin_count"][:, 0].sum())
    # the NumPy definition on the first host_records records of chain order, scaled by draws
    sub = rec[: max(4, a.host_records // 256)].cpu().numpy()
    tm = terms.cpu().numpy()
    t0 = time.perf_counter()
    h = PP.predictive_check_host(sub, 0, 200, tm, start_time=1800.0, seed=7)
    host_s = time.perf_counter() - t0
    host_draws = int(h["bin_count"][:, 0].sum())
    name, power = card()
    print(json.dumps({"bench": "k11_predictive", "records": int(rec.shape[0] * rec.shape[1]), "bins": 200, "draws": draws,
                      "kernel_ms": round(ms, 3), "draws_per_s": draws / (ms * 1e-3), "numpy_s_scaled": host_s * draws / max(host_draws, 1),
                      "numpy_draws_per_s": host_draws / host_s, "speedup": (host_s * draws / max(host_draws, 1)) / (ms * 1e-3),
                      "status": out["status"].cpu().tolist(), "gpu": name, "power_limit": power}))


if __name__ == "__main__":
    main()
