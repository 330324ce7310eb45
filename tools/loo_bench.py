"""K12 timing: PSIS-LOO and WAIC on the K5 workload -- 256 chains x 8 000 records of real RJMCMC output on the syn-int statistics
(1 M lineages, 200 bins; 2.05 M records x 200 bins x 2 sides) -- and on K7 records (256 DDRate chains x 2 000 records on the
same statistics), with the split into pointwise, sort, K9 and fit from a separate torch.profiler pass, and the NumPy definition
on a subsample of records, scaled linearly by records (stated as scaled).  Prints one JSON line with the card's name and power
limit, read in the same run.  python tools/loo_bench.py [--reps 3] [--host-records 10240]"""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import torch

from literate_b200 import engine as E, ddrate as DD, loo as LO, predictive as PP, synth
from ppc_bench import card

# k12_exp_kernel forms K9's input, so it counts with K9
PARTS = (("pointwise", ("k12_scan", "k12_number", "k12_init", "k12_point", "k12_fill")), ("sort", ("k10_",)), ("k9", ("k9_", "k12_exp")),
         ("fit", ("k12_tail", "k12_grid", "k12_fit")))


def split(fn):
    """Kernel time per part of one call, from torch.profiler's CUDA activities (a pass of its own)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    ms = {k: 0.0 for k, _ in PARTS}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        for k, keys in PARTS:
            if any(s in e.key for s in keys):
                ms[k] += t / 1000.0
    return {k: round(v, 3) for k, v in ms.items()}


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for _ in range(reps):
        out = fn()
    ev[1].record()
    torch.cuda.synchronize()
    return ev[0].elapsed_time(ev[1]) / reps, out


def case(name, dev, rec, kw, terms, reps, host_records):
    fn = lambda: dev.loo_device(rec, terms=terms, **kw)
    ms, out = timed(fn, reps)
    parts = split(fn)
    M = rec.shape[1]
    sub = rec[: max(4, host_records // M)].cpu().numpy()
    t0 = time.perf_counter()
    LO.loo_host(sub, kw["layout"], terms.shape[1], terms.cpu().numpy(), rate_col=kw.get("rate_col", 0), start_time=kw.get("start_time", 0.0))
    host_s = time.perf_counter() - t0
    R = rec.shape[0] * M
    return {"case": name, "records": R, "bins": int(terms.shape[1]), "columns": int((terms[[1, 3]] > 0).sum()),
            "used": int(out["n"].item()), "status": out["status"].cpu().tolist(), "kernel_ms": round(ms, 3), "split_ms": parts,
            "numpy_s_scaled": host_s * R / (sub.shape[0] * M), "numpy_records": int(sub.shape[0] * M),
            "speedup": host_s * R / (sub.shape[0] * M) / (ms * 1e-3)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--host-records", type=int, default=10240)
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
    terms = ds.bin_terms()[0].contiguous()
    res = [case("k3_k5_workload", dev, rec, dict(layout=0, start_time=1800.0), terms, a.reps, a.host_records)]
    ch.close(); ds.close()
    del rec
    s, e, b = (x.cpu().numpy() for x in (sp, ex, br))
    dch = DD.DDChains(dev, s, e, b, 0.0, 201.5, 2, 2, None, None, 256, 3)
    drec = torch.from_numpy(dch.run(200000, 100)).to(tdev)
    dch.close()
    dterms = torch.from_numpy(PP.stats_terms(s, e, b)[0]).to(tdev)
    res.append(case("k7", dev, drec, dict(layout=1, rate_col=PP.KINDS["dd"][1]), dterms, a.reps, a.host_records))
    name, power = card()
    print(json.dumps({"bench": "k12_loo", "cases": res, "gpu": name, "power_limit": power}))


if __name__ == "__main__":
    main()
