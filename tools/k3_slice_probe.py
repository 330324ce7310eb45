"""Time-sliced teams (k3_team_slot_kernel) against one CTA per chain on the bench statistics (1M lineages x 200 bins).
python tools/k3_slice_probe.py [iters] [slice_us] > probe.json   -- M it/s per population with LR_TEAM_SLICE_US = 0 and = slice_us,
alternated (the last line is the JSON summary).

149 chains run (nearly) every chain as a lone team of 16, 278 mostly as one of two teams of 8 on an SM; 256 is the bench
population; 148, 296 and 512 are outside the sliced range (LR_TEAM_SLICE_US changes nothing there: the spread of the measurement)."""
import json, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from literate_b200 import engine as E, synth

iters = int(sys.argv[1]) if len(sys.argv) > 1 else 100000
slice_us = sys.argv[2] if len(sys.argv) > 2 else "2000"
dev = E.Device(0)
sm = dev.sm_count
tdev = torch.device("cuda:0")
n, nb, n_rep = 1_000_000, 200, 4
ts, te = synth.syn_int_device(n, n_rep, tdev)
sp, ex, br = dev.bin_stats_device(ts[:, :n], te[:, :n], 1800, nb)
torch.cuda.synchronize()
ds = E.Dataset.from_device(dev, sp, ex, br, 0, 1800.0, 2000.5)
res = {"gpu": torch.cuda.get_device_name(0), "sm": sm, "iters": iters, "slice_us": int(slice_us)}


def run(nch, slicing):
    os.environ["LR_TEAM_SLICE_US"] = slice_us if slicing else "0"
    ch = E.Chains(ds, nch, 1, cfg=E.default_config(0), rep_of_chain=np.arange(nch) % n_rep)
    ch.run(2048)                                     # the first 2048 iterations go to the latency-optimised build
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    l0 = dev.kernel_launches
    a.record(); ch.run_device(iters, 0, None); b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b)
    st = ch.state()
    assert (st[:, E.REC_IT] == 2048 + iters).all()
    ch.close()
    return {"ms": ms, "M_it_per_s": nch * iters / (ms * 1e3), "it_per_us_per_sm": nch * iters / (ms * 1e3) / sm,
            "launches": dev.kernel_launches - l0}


for rep in range(2):
    for nch in (148, 149, 256, 278, 296, 512):
        for slicing in (False, True):
            r = run(nch, slicing)
            res.setdefault("%d_%s" % (nch, "sliced" if slicing else "off"), []).append(r)
            print(nch, "sliced" if slicing else "off", r, flush=True)
print(json.dumps(res))
