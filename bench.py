#!/usr/bin/env python
"""bench.py -- RJMCMC iterations/s (all chains) at 1M lineages, and the K1 HBM roofline.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--dump-outputs DIR]    # the CUDA arm (one JSON line on rank 0)
    python bench.py --impl reference [--steps K] [--warmup W]      # the CPU arm (oracle port, all host cores)

Workload (BASELINE.json configs[2]): synthetic 1M lineages x 200 one-year bins, 256 chains on one B200,
-model_BDI 0, every chain on its own stochastic-imputation replicate of the table (the reference's published
workflow is "100 chains on 100 imputations"), i.e. 256 x 1M lineages = 4.1 GB of (ts, te) per step -- larger
than the 126 MB L2, so no flush is needed between steps.  One STEP = one pass of the hot path over that batch:

    K1  lineages -> per-bin (births, deaths, time at risk) for all replicates        lr_bin_accumulate + lr_bin_finalize
    K2  prefix tables of the likelihood                                               lr_dataset_create
    K3  ITERS iterations of every chain, one sample record every SAMPLE iterations    lr_chains_create + lr_chains_run

value = chains x ITERS / step time with (ts, te) resident in HBM; e2e = the same through the host-buffer API
(pinned host ts/te in, sample records out) with the copies inside the timed region.  With N GPUs every rank
runs its own 256 chains on its own replicates (weak scaling, no data-path collective).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

N_LINEAGES = 1_000_000
N_BINS = 200
FIRST_BIN = 1800
CHAINS = 256
ITERS = 100_000          # iterations of every chain per step
SAMPLE = 1000            # the reference's default -s
METRIC = "RJMCMC iters/sec (all chains) at 1M lineages"
UNIT = "it/s"


def _args():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=10)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    p.add_argument("--chains", type=int, default=CHAINS, help="chains per GPU (default: the configuration the metric is quoted on)")
    p.add_argument("--lineages", type=int, default=N_LINEAGES)
    p.add_argument("--iters", type=int, default=ITERS)
    p.add_argument("--shared-dataset", type=int, default=0, help="1: all chains share one replicate (n_rep = 1)")
    p.add_argument("--real", type=int, default=0, help="1: real-valued times (syn-real, -death_jitter 0) instead of integer years")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--no-real-roofline", action="store_true", help="skip K1 on the real-valued tables (roofline_real, roofline_real_sorted)")
    p.add_argument("--no-multi", action="store_true", help="N > 1: skip BASELINE configs[3]/[4] (multi_gpu)")
    p.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed (rank 0's sample records and per-bin "
                                                           "statistics) as DIR/<name>.npy in float64, to compare two builds output for output")
    a = p.parse_args()
    if a.steps < 1:
        p.error("--steps must be at least 1")
    return a


def _workload(a, n_gpus):
    n_rep = 1 if a.shared_dataset else a.chains
    return {
        "workload": "syn-%s %d lineages x %d one-year bins, %d chains/GPU, %s, model_BDI 0, %d it/chain/step, sample every %d"
                    % ("real" if a.real else "int", a.lineages, N_BINS, a.chains,
                       "one imputation replicate per chain" if n_rep > 1 else "one shared table", a.iters, SAMPLE),
        "lineages": a.lineages, "bins": N_BINS, "chains_per_gpu": a.chains, "replicates_per_gpu": n_rep,
        "iters_per_chain_per_step": a.iters, "sample_every": SAMPLE,
        "parallelism": "chains sharded over %d GPU(s), no collective" % n_gpus,
        "l2": "inputs (%.2f GB per step) larger than L2, no flush" % (16.0 * a.lineages * n_rep / 1e9)
              if 16.0 * a.lineages * n_rep > 256e6 else "L2 flushed (512 MB memset) before every step",
    }


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        self.t = threading.Thread(target=self._read, daemon=True)
        self.t.start()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [x.strip() for x in line.split(",")]))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        rows = [r for (t, r) in self.rows if t0 <= t <= t1 and len(r) >= 8] or [r for (_, r) in self.rows if len(r) >= 8]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm = [float(r[1]) for r in rows]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(r[4 + k].lower().startswith("active") for r in rows)]
        pw = [float(r[3]) for r in rows if r[3].replace(".", "", 1).isdigit()]
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": float(rows[0][2]), "reasons": reasons,
                "samples": len(rows), "power_w_max": max(pw) if pw else None}


def _peaks():
    try:
        with open(os.path.join(REPO, "MEASURED_PEAKS.json")) as fh:
            return float(json.load(fh)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (copy kernel, read+write)"
    except Exception:
        return 6650.0, "fallback 6.65 TB/s of B200_PROFILING.md (MEASURED_PEAKS.json absent)"


DUMP_BYTES = 60 << 20    # array data of --dump-outputs; the index files and .npy headers stay within the remaining 4 MB of 64 MB


def _dump_outputs(out_dir, arrays):
    """Saves every (name, array, axis) as out_dir/<name>.npy in float64.  Past DUMP_BYTES in all, every array keeps the same
    fraction of its slices along `axis`, picked with a fixed seed (so two runs keep the same ones); <name>_index.npy lists them."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    total = 8 * sum(x.size for _, x, _ in arrays)
    for name, x, axis in arrays:
        x = np.asarray(x, dtype=np.float64)
        if total > DUMP_BYTES:
            n = x.shape[axis]
            keep = np.sort(np.random.default_rng(0).choice(n, max(1, n * DUMP_BYTES // total), replace=False))
            x = np.take(x, keep, axis=axis)
            np.save(os.path.join(out_dir, name + "_index.npy"), keep.astype(np.float64))
        np.save(os.path.join(out_dir, name + ".npy"), x)


def _sha16(path):
    import hashlib
    with open(path, "rb") as fh:
        return hashlib.sha256(fh.read()).hexdigest()[:16]


def _traffic(a, kind=None):
    """dram bytes per K1 launch from the committed ncu --set full capture of this workload -- only while the capture is of
    the kernel source that is being timed (profiles/k1_traffic.json records the digest of k1_binstats.cu); otherwise null."""
    try:
        with open(os.path.join(REPO, "profiles", "k1_traffic.json")) as fh:
            t = json.load(fh)
        if t.get("k1_binstats_cu_sha16") != _sha16(os.path.join(REPO, "literate_b200", "csrc", "k1_binstats.cu")):
            print("bench.py: profiles/k1_traffic.json was captured from another build of k1_binstats.cu -- roofline.traffic left null "
                  "(re-capture with ncu --set full and tools/profile_to_json.py)", file=sys.stderr)
            return None
        key = "%s_%d_x_%d" % (kind or ("real" if a.real else "int"), a.lineages, 1 if a.shared_dataset else a.chains)
        return t.get(key)
    except Exception:
        return None


def _k3_instructions():
    """warp instructions per chain iteration of K3 on the bench workload, from the committed ncu capture (profiles/k3_instructions.json),
    only while the capture is of the sources being timed."""
    try:
        with open(os.path.join(REPO, "profiles", "k3_instructions.json")) as fh:
            t = json.load(fh)
        dig = "+".join(_sha16(os.path.join(REPO, "literate_b200", "csrc", f)) for f in ("k3_chains.cu", "k3_team.cuh", "chain_device.cuh", "lr_common.cuh"))
        return t["warp_instructions_per_iteration"] if t.get("sources_sha16") == dig else None
    except Exception:
        return None


# ------------------------------------------------------------------------------------------ CPU arm
def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from oracle import cpu_baseline as CB
    cores = os.cpu_count() or 1
    n_rep = 1 if a.shared_dataset else a.chains
    bins, iters = 2, 4000
    for _ in range(a.warmup):
        CB.run_sample(cores, a.lineages, N_BINS, n_rep, a.chains, a.iters, SAMPLE, bins=1, iters=500)
    t0 = time.perf_counter()
    res = [CB.run_sample(cores, a.lineages, N_BINS, n_rep, a.chains, a.iters, SAMPLE, bins=bins, iters=iters, seed0=1 + 97 * k)
           for k in range(a.steps)]
    wall = time.perf_counter() - t0
    full = statistics.mean(r["whole_workload_s"] for r in res)
    value = a.chains * a.iters / full
    sample = ("per step every one of %d worker processes bins %d of the %d unit bins of one %d-lineage replicate with the reference's "
              "per-bin NumPy formulation and runs %d RJMCMC iterations of one chain (scipy priors, adequacy on, sampling every %d); "
              "extrapolated linearly to %d replicates x %d bins and %d chains x %d iterations" %
              (cores, bins, N_BINS, a.lineages, iters, SAMPLE, n_rep, N_BINS, a.chains, a.iters))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": 1e3 * wall / max(a.steps, 1), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": _workload(a, a.gpus),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                         "loop_it_per_s_1core": statistics.mean(r["it_per_s_loop_1core"] for r in res),
                         "binning_s_per_bin_1core": statistics.mean(r["s_per_bin_1core"] for r in res),
                         "whole_workload_s": full},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)
    return 0


# ------------------------------------------------------------------------------------------ multi-GPU configurations
def _multi_gpu_configs(dev, tdev, rank, world, nb):
    """BASELINE configs[4] (lineage axis sharded, per-bin sufficient statistics combined by an NCCL all-reduce) and configs[3]
    (4096 tempered chains sharded over the ranks, ladders that span ranks, one all-gather per swap round), timed with CUDA
    events, max over ranks.  Returns the `multi_gpu` object of the JSON line (same on every rank)."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from literate_b200 import engine as E, parallel as P, synth

    def tmax(x):
        t = torch.tensor([x], dtype=torch.float64, device=tdev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0])

    out = {"world": world}
    # ---- configs[4]: 1e8 lineages, contiguous 1/world slice per rank, K1 + int64 SUM all-reduce + finalize
    n_total = 100_000_000
    s0, cnt = P.shard_range(n_total, world, rank)
    ts, te = synth.syn_int_device(cnt, 1, tdev, seed=synth.BASE_SEED + 17 * rank)
    ts, te = ts[:, :cnt], te[:, :cnt]
    evs = []
    for k in range(8):
        acc = dev.new_accumulators(1, nb, tdev)
        a, b, c = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        a.record()
        dev.bin_accumulate_device(ts, te, FIRST_BIN, nb, acc, fe_ref=0.5)
        b.record()
        P.allreduce_accumulators(acc)
        sp, ex, br = dev.bin_finalize_device(acc, nb, fe_ref=0.5)
        c.record()
        if k >= 3:
            evs.append((a, b, c))
    torch.cuda.synchronize()
    k1 = tmax(statistics.median(a.elapsed_time(b) for a, b, c in evs))
    tot = tmax(statistics.median(a.elapsed_time(c) for a, b, c in evs))
    births_ok = int(sp.sum()) == n_total                      # every lineage is born once inside the window
    # in-run equality: a 4M-lineage table every rank can generate; shards all-reduced == rank 0 binning the whole table itself
    n_chk = 4_000_000
    cts, cte = synth.syn_int_device(n_chk, 1, tdev, seed=synth.BASE_SEED + 999)
    c0, cc = P.shard_range(n_chk, world, rank)
    acc_sh = dev.new_accumulators(1, nb, tdev)
    dev.bin_accumulate_device(cts[:, c0:c0 + cc].contiguous(), cte[:, c0:c0 + cc].contiguous(), FIRST_BIN, nb, acc_sh, fe_ref=0.5)
    P.allreduce_accumulators(acc_sh)
    acc_full = dev.new_accumulators(1, nb, tdev)
    dev.bin_accumulate_device(cts[:, :n_chk], cte[:, :n_chk], FIRST_BIN, nb, acc_full, fe_ref=0.5)
    eq = torch.tensor([1.0 if bool((acc_sh == acc_full).all()) else 0.0], dtype=torch.float64, device=tdev)
    dist.all_reduce(eq, op=dist.ReduceOp.MIN)
    out["cfg5_lineage_sharded"] = {
        "lineages": n_total, "per_gpu": cnt, "bins": nb, "k1_ms": k1, "k1_allreduce_finalize_ms": tot,
        "aggregate_GBps_k1": 16.0 * n_total / (k1 * 1e-3) / 1e9, "aggregate_GBps_incl_allreduce": 16.0 * n_total / (tot * 1e-3) / 1e9,
        "allreduce_bytes": int(acc.numel() * 8), "collective": "NCCL all_reduce(SUM) of int64 accumulators, once per dataset",
        "births_conserved": births_ok,
        "allreduced_equals_single_gpu_accumulators": bool(eq[0] == 1.0), "equality_check_lineages": n_chk}
    del ts, te, cts, cte

    # ---- configs[3]: 4096 tempered chains (+ half a ladder per rank so that every rank boundary cuts a ladder), strong scaling
    iters, swap_every, ladder = 100_000, 1000, 32
    nl = 4096 // world // ladder * ladder + ladder // 2
    total = nl * world
    c0 = rank * nl
    g = synth.syn_int_device(1_000_000, 1, tdev)
    sp, ex, br = dev.bin_stats_device(g[0][:, :1_000_000], g[1][:, :1_000_000], FIRST_BIN, nb)
    ds = E.Dataset.from_device(dev, sp, ex, br, 0, float(FIRST_BIN), float(FIRST_BIN + nb) + 0.5)
    ch = E.Chains(ds, nl, seed=77, chain_id0=c0)
    ch.set_beta(P.temperature_ladder(ladder, 0.025)[np.arange(c0, c0 + nl) % ladder])
    ch.run_device(2000, 0, None)
    torch.cuda.synchronize(); dist.barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for rnd in range(iters // swap_every):
        ch.run_device(swap_every, 0, None)
        P.tempered_swap(ch, c0, ladder, rnd)              # (lik, beta) table -> all-gather (16 B per chain) -> every rank applies the round
    b.record()
    torch.cuda.synchronize()
    ms = tmax(a.elapsed_time(b))
    cnts = ch.counters().sum(0)
    tc = torch.tensor([float(cnts[8]), float(cnts[9])], dtype=torch.float64, device=tdev)
    dist.all_reduce(tc)
    out["cfg4_tempered"] = {"chains": total, "per_gpu": nl, "ladder": ladder, "ladders_span_ranks": True, "iters_per_chain": iters,
                            "swap_every": swap_every, "device_ms": ms, "it_per_s": total * iters / (ms * 1e-3), "scaling": "strong",
                            "swap_acceptance": float(tc[1] / max(float(tc[0]), 1.0)),
                            "collective": "NCCL all_gather of (likelihood, beta), 16 B per chain per swap round; temperatures move, states do not"}
    ch.close(); ds.close()
    return out


# ------------------------------------------------------------------------------------------ CUDA arm
def run_cuda(a):
    import numpy as np
    import torch
    import torch.distributed as dist
    from literate_b200 import engine as E, synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; literate_b200 has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    tdev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=tdev)
    n_gpus = world

    bound_cpus = E.bind_host_to_gpu(local)                 # pinned buffers below are first-touched on the GPU's NUMA node
    dev = E.Device(local)
    n, nb, chains = a.lineages, N_BINS, a.chains
    n_rep = 1 if a.shared_dataset else chains
    fe_ref = 1.0 if a.real else 0.5
    end_time = float(FIRST_BIN + nb) + (0.0 if a.real else 0.5)
    rep0 = rank * n_rep                                    # every rank has its own replicates and chain ids
    gen = synth.syn_real_device if a.real else synth.syn_int_device
    ts, te = gen(n, n_rep, tdev, seed=synth.BASE_SEED + 1000 * rank)
    ts, te = ts[:, :n], te[:, :n]
    rep_of_chain = (np.arange(chains) % n_rep).astype(np.int32)
    n_rec = (a.iters + SAMPLE - 1) // SAMPLE
    records = torch.empty((n_rec, chains, E.LR_REC_DOUBLES), dtype=torch.float64, device=tdev)
    acc = dev.new_accumulators(n_rep, nb, tdev)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=tdev) if 16.0 * n * n_rep <= 256e6 else None
    stream = torch.cuda.Stream(device=tdev)
    cfg = E.default_config(0)
    k1_ms, k3_ms = [], []
    k1_build = ["k1_bin_kernel"]
    last_stats = [None]                                    # (sp, ex, br) of the latest step, for --dump-outputs

    def step(k, timed):
        """One pass of the hot path with device-resident lineages."""
        if flush is not None:
            flush.zero_()
        acc.zero_()
        e0, e1, e2, e3 = (torch.cuda.Event(enable_timing=True) for _ in range(4))
        e0.record()
        dev.bin_accumulate_device(ts, te, FIRST_BIN, nb, acc, fe_ref=fe_ref, stream=stream.cuda_stream)
        e1.record()
        k1_build[0] = dev.bin_last_build()
        sp, ex, br = dev.bin_finalize_device(acc, nb, fe_ref=fe_ref, stream=stream.cuda_stream)
        last_stats[0] = (sp, ex, br)
        ds = E.Dataset.from_device(dev, sp, ex, br, 0, float(FIRST_BIN), end_time, stream=stream.cuda_stream)
        ch = E.Chains(ds, chains, seed=2026 + k, cfg=cfg, chain_id0=rank * chains, rep_of_chain=rep_of_chain)
        e2.record()
        ch.run_device(a.iters, SAMPLE, records, stream=stream.cuda_stream)
        e3.record()
        return (e0, e1, e2, e3), ds, ch

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    with torch.cuda.stream(stream):
        for k in range(a.warmup):
            _, ds, ch = step(k, False)
            torch.cuda.synchronize()
            ch.close(); ds.close()
        barrier()
        clocks = ClockSampler(local)
        clocks.start()
        launches0 = dev.kernel_launches
        t_wall0 = time.perf_counter()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        keep = []
        for k in range(a.steps):
            keep.append(step(a.warmup + k, True))
        g1.record()
        barrier()
        t_wall1 = time.perf_counter()
        total_ms = g0.elapsed_time(g1)
        launches = dev.kernel_launches - launches0
        lik_evals = 0
        # the timed output is checked, not just produced: every chain delivered its samples, and the likelihood and prior of the
        # states the LAST step logged (every 10th sample of every chain) are recomputed from the logged rates / shift times by the
        # batched state evaluator (lr_state_eval_host, itself held to the oracle at 1e-10 by tests/test_gpu_likelihood.py)
        rec = records.cpu().numpy()
        assert np.all(rec[:, :, E.REC_IT] == (np.arange(n_rec) * SAMPLE)[:, None]) and np.all(np.isfinite(rec[:, :, E.REC_LIK]))
        last_ds = keep[-1][1]
        pick = rec[5::10].reshape(-1, rec.shape[-1])
        reps = np.tile(rep_of_chain, len(rec[5::10]))
        states = [E.record_to_state(r, end_time) for r in pick]
        ev = last_ds.evaluate(states, gamma_rate=pick[:, [E.REC_GL, E.REC_GM]], poi_lambda=pick[:, E.REC_POI], rep=reps)
        assert np.allclose(ev["lik"], pick[:, E.REC_LIK], rtol=1e-10, atol=0), "timed output: logged likelihood differs from the state's"
        assert np.allclose(ev["prior_rates"] + pick[:, E.REC_POIA], pick[:, E.REC_PRIOR], rtol=1e-9, atol=1e-9), "timed output: logged prior differs"
        k_l_mean, k_m_mean = float(rec[n_rec // 2:, :, E.REC_KL].mean()), float(rec[n_rec // 2:, :, E.REC_KM].mean())
        for (e0, e1, e2, e3), ds, ch in keep:
            k1_ms.append(e0.elapsed_time(e1))
            k3_ms.append(e2.elapsed_time(e3))
            lik_evals += int(ch.counters()[:, 2].sum())
            ch.close(); ds.close()

        # ---------------- e2e: host buffers through the public API, copies inside the timed region
        e2e = None
        if not a.no_e2e:
            hts = torch.empty((n_rep, n), dtype=torch.float64, pin_memory=True); hts.copy_(ts)
            hte = torch.empty((n_rep, n), dtype=torch.float64, pin_memory=True); hte.copy_(te)
            hrec = torch.empty((n_rec, chains, E.LR_REC_DOUBLES), dtype=torch.float64, pin_memory=True)
            nts, nte, nrec = hts.numpy(), hte.numpy(), hrec.numpy()

            # the public streaming API: engine.Pipeline double-buffers consecutive batches (tables of step k+1 are copied and
            # binned while the chains of step k run); every step's H2D copy and D2H read are inside the timed region,
            # which ends when the last step's records are on the host
            pipe = E.Pipeline(local)

            def e2e_push(k):
                return pipe.push(nts, nte, chains, a.iters, SAMPLE, seed=4052 + k, cfg=cfg, first_bin=FIRST_BIN, n_bins=nb,
                                 death_jitter=0.0 if a.real else 0.5, start_time=float(FIRST_BIN), end_time=end_time,
                                 rep_of_chain=rep_of_chain, chain_id0=rank * chains, out=hrec)
            for k in range(max(1, min(a.warmup, 2))):
                e2e_push(k)
            pipe.flush(out=hrec)
            barrier()
            n_e2e = a.steps                          # as many steps as the device-timed value; the last step's chains cannot overlap a copy
            t0 = time.perf_counter()
            for k in range(n_e2e):
                tp = time.perf_counter()
                e2e_push(100 + k)
                if os.environ.get("LR_BENCH_DEBUG"):
                    print("push %d: %.1f ms" % (k, 1e3 * (time.perf_counter() - tp)), file=sys.stderr, flush=True)
            tp = time.perf_counter()
            pipe.flush(out=hrec)
            tq = time.perf_counter()
            torch.cuda.synchronize()
            e2e_s = time.perf_counter() - t0
            if os.environ.get("LR_BENCH_DEBUG"):
                print("flush %.1f ms, sync %.1f ms, total %.1f ms" % (1e3 * (tq - tp), 1e3 * (time.perf_counter() - tq), 1e3 * e2e_s), file=sys.stderr, flush=True)
            assert np.all(nrec[:, :, E.REC_IT] == (np.arange(n_rec) * SAMPLE)[:, None]) and np.all(np.isfinite(nrec[:, :, E.REC_LIK]))
            e2e = [e2e_s / n_e2e, 16 * n * n_rep + 4 * chains, int(nrec.nbytes) + 24 * n_rep * nb]
            # ---- the same through the compact entry point: the table held on the host as int32 YEARS (what a parser of the
            # integer-year tables the reference ships produces), te jittered by the kernel -- half the bytes over PCIe
            if not a.real:
                hti = torch.empty((n_rep, n), dtype=torch.int32, pin_memory=True); hti.copy_(ts.to(torch.int32))
                hei = torch.empty((n_rep, n), dtype=torch.int32, pin_memory=True); hei.copy_((te - 0.5).to(torch.int32))
                nti, nei = hti.numpy(), hei.numpy()

                def e2e_push_i32(k):
                    return pipe.push(nti, nei, chains, a.iters, SAMPLE, seed=4052 + k, cfg=cfg, first_bin=FIRST_BIN, n_bins=nb,
                                     death_jitter=0.5, start_time=float(FIRST_BIN), end_time=end_time,
                                     rep_of_chain=rep_of_chain, chain_id0=rank * chains, out=hrec)
                e2e_push_i32(0); pipe.flush(out=hrec)
                barrier()
                t0 = time.perf_counter()
                for k in range(n_e2e):
                    e2e_push_i32(100 + k)
                pipe.flush(out=hrec)
                torch.cuda.synchronize()
                e2e_i32_s = time.perf_counter() - t0
                assert np.all(nrec[:, :, E.REC_IT] == (np.arange(n_rec) * SAMPLE)[:, None]) and np.all(np.isfinite(nrec[:, :, E.REC_LIK]))
                e2e += [e2e_i32_s / n_e2e, 8 * n * n_rep + 4 * chains]
                del hti, hei
            pipe.close()
            del hts, hte, hrec
        cl = clocks.stop(t_wall0, t_wall1)

        # ---------------- the sibling samplers of SURVEY 8 f-4 on the statistics of replicate 0 (reported beside the metric, not part of it)
        siblings = None
        if rank == 0:
            from literate_b200 import trend as TR, ddrate as DD
            sp, ex, br = (x[0].cpu().numpy() for x in dev.bin_finalize_device(acc, nb, fe_ref=fe_ref, stream=stream.cuda_stream))
            trend = np.clip(np.linspace(0.0, 1.0, nb), 1e-15, 1.0)
            sib_iters = 20000
            siblings = {"chains": chains, "bins": nb, "iterations": sib_iters}
            for name, mk in (("k6_trend_it_per_s", lambda: TR.TrendChains(dev, sp, ex, br, trend, chains, 7)),
                             ("k7_ddrate_it_per_s", lambda: DD.DDChains(dev, sp, ex, br, float(FIRST_BIN), end_time, 2, 2, None, None, chains, 7))):
                sc = mk()
                sc.run(2000)
                srec = torch.empty((sc.records_per_run(sib_iters, SAMPLE), chains, sc.rec_doubles), dtype=torch.float64, device=tdev)
                s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s0.record(); sc.run_device(sib_iters, SAMPLE, srec, stream=stream.cuda_stream); s1.record()
                torch.cuda.synchronize()
                siblings[name] = chains * sib_iters / (s0.elapsed_time(s1) * 1e-3)
                assert bool(torch.isfinite(srec[:, :, 1]).all())
                sc.close()

        # ---------------- K1 on real-valued tables (fp64 fractions through the carry chains), shuffled and sorted by birth year:
        # the orderings real TSVs come in.  Reported beside the roofline of the integer-year workload the metric is quoted on.
        real_roof = None
        if world == 1 and not a.real and not a.no_real_roofline:
            del ts, te
            torch.cuda.empty_cache()
            real_roof = {}
            rts, rte = synth.syn_real_device(n, n_rep, tdev, seed=synth.BASE_SEED + 7919)
            for tag in ("roofline_real", "roofline_real_sorted"):
                if tag == "roofline_real_sorted":
                    for r in range(n_rep):                      # sort every replicate by birth time (te follows)
                        o = torch.argsort(rts[r, :n])
                        rts[r, :n] = rts[r, :n][o]; rte[r, :n] = rte[r, :n][o]
                    del o
                vts, vte = rts[:, :n], rte[:, :n]
                acc.zero_()
                for _ in range(2):
                    dev.bin_accumulate_device(vts, vte, FIRST_BIN, nb, acc, fe_ref=1.0, stream=stream.cuda_stream)
                    torch.cuda.synchronize()         # the first pass records that the table carries fractions; later passes read it
                real_build = dev.bin_last_build()
                evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(5)]
                for e0, e1 in evs:
                    e0.record(); dev.bin_accumulate_device(vts, vte, FIRST_BIN, nb, acc, fe_ref=1.0, stream=stream.cuda_stream); e1.record()
                torch.cuda.synchronize()
                ms = statistics.mean(e0.elapsed_time(e1) for e0, e1 in evs)
                real_roof[tag] = ms
            del rts, rte, vts, vte
            torch.cuda.empty_cache()

        # ---------------- BASELINE configs[3] and configs[4]: only meaningful on several GPUs, measured in the same run
        multi = None
        if world > 1 and not a.no_multi:
            multi = _multi_gpu_configs(dev, tdev, rank, world, nb)

    t = torch.tensor([total_ms, e2e[0] if e2e else 0.0, e2e[3] if e2e and len(e2e) > 3 else 0.0], dtype=torch.float64, device=tdev)
    tot = torch.tensor([float(lik_evals), float(launches)], dtype=torch.float64, device=tdev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    total_ms, e2e_step_s, e2e_i32_step_s = float(t[0]), float(t[1]), float(t[2])
    if rank == 0:
        peak, peak_src = _peaks()
        k1 = statistics.mean(k1_ms)
        algo_bytes = 16.0 * n * n_rep
        achieved = algo_bytes / (k1 * 1e-3) / 1e9
        value = n_gpus * chains * a.iters * a.steps / (total_ms * 1e-3)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": n_gpus, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": total_ms / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": _workload(a, n_gpus), "clocks": cl,
            "gpu_launches": int(tot[1]),
            "output_check": {"states_re_evaluated": int(len(pick)), "likelihood_rel_tol": 1e-10, "mean_K_l": k_l_mean, "mean_K_m": k_m_mean,
                             "note": "likelihood and prior of states logged by the last timed step recomputed by lr_state_eval_host; "
                                     "posterior parity on these statistics: tests/test_gpu_chains.py (32 oracle chains)"},
            "lik_evals_per_s": float(tot[0]) / (total_ms * 1e-3),
            "kernels": {"k1_kernel": k1_build[0], "k1_bin_kernel_ms": k1, "k3_run_kernel_ms": statistics.mean(k3_ms),
                        "k3_ns_per_iteration_per_chain": 1e6 * statistics.mean(k3_ms) / a.iters,
                        "k3_bound": "instruction issue: teams of 8 warps evaluate consecutive iterations of one chain speculatively "
                                    "(no DRAM traffic in the loop; roofline_k3, profiles/)",
                        "k1_share_of_step": k1 * a.steps / total_ms, "k3_share_of_step": sum(k3_ms) / total_ms},
            "roofline": {"kernel": k1_build[0] + " (lineages -> per-bin births/deaths/time at risk)", "bound": "hbm", "achieved": achieved,
                         "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": _traffic(a),
                         "algorithmic_bytes_per_launch": algo_bytes, "peak_source": peak_src, "ms_per_launch": k1},
        }
        # K3 against the instruction-issue peak (it touches no DRAM): warp instructions per chain iteration from the committed
        # ncu capture of this build x iterations/s measured here / (SMs x 4 schedulers x SM clock measured here)
        k3_ipi = _k3_instructions()
        k3_rate = chains * a.iters / (statistics.mean(k3_ms) * 1e-3)            # one GPU's chains
        clk = (cl.get("sm_mhz") or 1965.0) * 1e6
        line["roofline_k3"] = {"kernel": "K3 chain loop (k3_team_kernel + continuation passes)", "bound": "issue",
                               "warp_instructions_per_iteration": k3_ipi,
                               "achieved": k3_ipi * k3_rate if k3_ipi else None, "peak": dev.sm_count * 4 * clk, "unit": "warp-instructions/s",
                               "frac": (k3_ipi * k3_rate) / (dev.sm_count * 4 * clk) if k3_ipi else None,
                               "source": "profiles/k3_instructions.json (ncu smsp__inst_executed.sum of the K3 kernels of one bench step / chain iterations)"}
        line["kernels"]["k3_issue_frac"] = line["roofline_k3"]["frac"]
        if real_roof:
            for tag, ms in real_roof.items():
                ach = algo_bytes / (ms * 1e-3) / 1e9
                line[tag] = {"kernel": real_build, "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                             "traffic": _traffic(a, ("realsorted" if tag.endswith("sorted") else "real") + "_lanes") if real_build == "k1_bin_lanes_kernel" else None,
                             "ms_per_launch": ms, "algorithmic_bytes_per_launch": algo_bytes,
                             "table": "syn-real %d lineages x %d replicates, %s" % (n, n_rep, "sorted by birth time" if tag.endswith("sorted") else "shuffled")}
        if multi:
            line["multi_gpu"] = multi
        if siblings:
            line["siblings"] = siblings
        if e2e:
            line["e2e"] = {"value": n_gpus * chains * a.iters / e2e_step_s, "unit": UNIT, "h2d_bytes_per_step": e2e[1],
                           "d2h_bytes_per_step": e2e[2], "ms_per_step": 1e3 * e2e_step_s,
                           "h2d_GBps_per_rank": e2e[1] / e2e_step_s / 1e9,
                           "host_table": "fp64 (ts, te), 16 B per lineage: the arrays the reference's parser holds (LiteRateForward.py:440-471)",
                           "cpu_affinity": "GPU-local CPUs (%d of %d)" % (len(bound_cpus), os.cpu_count()) if bound_cpus else "unchanged (NVML reports no GPU-local subset)"}
            if len(e2e) > 3 and e2e_i32_step_s > 0:
                line["e2e_i32"] = {"value": n_gpus * chains * a.iters / e2e_i32_step_s, "unit": UNIT, "h2d_bytes_per_step": e2e[4],
                                   "d2h_bytes_per_step": e2e[2], "ms_per_step": 1e3 * e2e_i32_step_s,
                                   "h2d_GBps_per_rank": e2e[4] / e2e_i32_step_s / 1e9,
                                   "host_table": "int32 years, 8 B per lineage (lr_bin_stats_host_i32; the kernel adds the death jitter)"}
        if n_gpus == 1 and not a.no_cpu_baseline:
            from oracle import cpu_baseline as CB
            cores = os.cpu_count() or 1
            bins, iters = 2, 4000
            r = CB.run_sample(cores, n, nb, n_rep, chains, a.iters, SAMPLE, bins=bins, iters=iters)
            line["cpu_baseline"] = {
                "value": r["value"], "unit": UNIT, "cores": cores, "kind": "port",
                "sample": "one pass: each of %d worker processes bins %d of %d bins of one %d-lineage replicate (reference's per-bin NumPy "
                          "formulation) and runs %d iterations of one chain (scipy priors); extrapolated linearly to the whole workload"
                          % (cores, bins, nb, n, iters),
                "loop_it_per_s_1core": r["it_per_s_loop_1core"], "binning_s_per_bin_1core": r["s_per_bin_1core"],
                "whole_workload_s": r["whole_workload_s"]}
        if a.dump_outputs:
            sp, ex, br = (x.cpu().numpy() for x in last_stats[0])
            _dump_outputs(a.dump_outputs, [("records", rec, 1), ("sp_events_bin", sp, 0), ("ex_events_bin", ex, 0), ("br_length_bin", br, 0)])
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    args = _args()
    # stdout carries exactly one JSON line: native libraries that print there (NCCL's version banner) go to stderr
    sys.stdout.flush()
    _json_fd = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(_json_fd, "w")
    sys.exit(run_reference(args) if args.impl == "reference" else run_cuda(args))
