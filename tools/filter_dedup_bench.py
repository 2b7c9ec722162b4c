"""B200WavePoolFilteredPlugin with one Butterworth configuration on a 16-channel run: the filter plan gives one
wfb_filter_cfg for all channels, so wfb_filter_pool takes the uniform kernel (coefficients as kernel parameters).
Before configurations were deduplicated the plan held one per channel, which selects the multi-configuration kernel;
WFB_BW_UNIFORM=0 selects that kernel for the same plan, so both are timed here (alternating, CUDA-event timed device
work of ops.filter_pool on the resident run without its copy to the host: the plan and wfb_filter_pool) and their outputs compared.

    python tools/filter_dedup_bench.py [--records 2000000] [--samples 800] [--reps 5]
"""
import argparse
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from waveformanalysis_b200 import engine, ops
from waveformanalysis_b200.channel_config import unique_channels
from waveformanalysis_b200.plugins.filtering import channel_filter_configs

ap = argparse.ArgumentParser()
ap.add_argument("--records", type=int, default=2_000_000)
ap.add_argument("--samples", type=int, default=800)
ap.add_argument("--reps", type=int, default=5)
args = ap.parse_args()

card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True).stdout.strip()
run = engine.DeviceRun.synth(args.records, args.samples, 16, dt_ns=4, seed=99, with_rows=True)
rec = run.records_to_host()[: run.n]
pool = run.pool_to_host()
opts = {"filter_type": "BW", "lowcut": 0.01, "highcut": 0.1, "fs": 0.25, "filter_order": 4}
configs, default = channel_filter_configs(unique_channels(rec["board"], rec["channel"]), opts, None, "run")
res = engine.DeviceRun.from_host(rec, pool)
lens = np.unique(rec["event_length"])
n_cfg = ops.filter_plan(res, configs)["n_cfg"]


def once(uniform: bool):
    os.environ["WFB_BW_UNIFORM"] = "1" if uniform else "0"
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    d_out = ops._filter_launch(res, ops.filter_plan(res, configs, lengths=lens), res.pool_len, res.lmax)
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b), d_out


once(True), once(False)  # warm-up
times = {True: [], False: []}
out = {}
for _ in range(args.reps):
    for u in (True, False):
        ms, out[u] = once(u)
        times[u].append(ms)
same = bool(torch.equal(out[True].view(torch.int32), out[False].view(torch.int32)))
print(f"{card} | {args.records} records x {args.samples} samples, 16 channels, BW order 4: {len(configs)} channels -> {n_cfg} configuration(s)")
for u, name in ((False, "multi-configuration kernel (what one configuration per channel selected)"), (True, "uniform kernel (deduplicated plan)")):
    t = np.array(times[u])
    print(f"  {name}: plan + filter {np.median(t):.2f} ms median (min {t.min():.2f}, max {t.max():.2f}) over {len(t)} calls")
print(f"  outputs byte-identical: {same}")
