#!/usr/bin/env python
"""Time ops.group_hit_windows (the hit_grouped event table) with the device table (wfb_hit_event_table) against the
host table it replaced (a 7-key np.lexsort plus np.bincount / np.minimum.at / np.maximum.at over every hit, kept below
as ``group_hit_windows_host_table``), on one GPU:

    python tools/hit_table_bench.py [--min-hits 10000000] [--reps 3]

The hits are the threshold hits of a synthetic run (DeviceRun.synth, 800 samples per record, threshold 15), grown until
there are at least --min-hits of them; hit_merge runs with merge_gap_ns 0 and 50 and the grouping with time_window_ns
100.  Both versions see the same host arrays and run alternately; every call ends with its results on the host.  The two
results must be identical.  Prints the GPU name and power limit with the times."""
import argparse
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from waveformanalysis_b200 import ops
from waveformanalysis_b200.dtypes import THRESHOLD_HIT_DTYPE
from waveformanalysis_b200.engine import DeviceRun
from waveformanalysis_b200.ops import _dev, _empty, _lib, _ptr, _stream

ap = argparse.ArgumentParser()
ap.add_argument("--min-hits", type=int, default=10_000_000)
ap.add_argument("--reps", type=int, default=3)
args = ap.parse_args()
L, NCH, THR, WINDOW = 800, 16, 15.0, 100.0


def group_hit_windows_host_table(hits, time_window_ns, component_rows=None, component_hits=None):
    """ops.group_hit_windows as it was before wfb_hit_event_table: device grouping, host event table."""
    lib = _lib.load()
    names = hits.dtype.names
    sn, en = ("sample_start", "sample_end") if "sample_start" in names else ("edge_start", "edge_end")
    nh = len(hits)
    d_ts = _dev(hits["timestamp"].astype(np.int64))
    d_dt, d_rid = _dev(hits["dt"].astype(np.int32)), _dev(hits["record_id"].astype(np.int64))
    order = torch.empty(nh, dtype=torch.int64, device="cuda")
    ev = torch.empty(nh, dtype=torch.int64, device="cuda")
    n_ev = torch.zeros(1, dtype=torch.int64, device="cuda")
    ws = _empty(lib.wfb_group_workspace_bytes(nh))
    bad = np.flatnonzero((hits[sn] < 0) | (hits[en] < 0))
    if len(bad):
        dt_ps = hits["dt"].astype(np.float64) * 1e3
        pos = hits["position"].astype(np.float64)
        h0 = hits["timestamp"].astype(np.float64) + (hits[sn].astype(np.int32) - pos) * dt_ps
        h1 = hits["timestamp"].astype(np.float64) + (hits[en].astype(np.int32) - pos) * dt_ps
        cdt = component_hits["dt"].astype(np.float64) * 1e3
        cpos = component_hits["position"].astype(np.float64)
        c0 = component_hits["timestamp"].astype(np.float64) + (component_hits["edge_start"].astype(np.int32) - cpos) * cdt
        c1 = component_hits["timestamp"].astype(np.float64) + (component_hits["edge_end"].astype(np.int32) - cpos) * cdt
        idx = component_rows["hit_index"].astype(np.int64)
        for m in bad.tolist():
            o, c = int(hits["component_offset"][m]), int(hits["component_count"][m])
            h0[m] = c0[idx[o:o + c]].min()
            h1[m] = c1[idx[o:o + c]].max()
        a0, a1 = _dev(h0), _dev(h1)
        _lib.check(lib.wfb_group_abs_windows(_ptr(d_ts), _ptr(a0), _ptr(a1), _ptr(d_dt), _ptr(d_rid), nh, float(time_window_ns), _ptr(order),
                                             _ptr(ev), _ptr(n_ev), _ptr(ws), ws.numel(), _stream()), "wfb_group_abs_windows")
    else:
        d_pos = _dev(hits["position"].astype(np.int64))
        d_s, d_e = _dev(hits[sn].astype(np.int32)), _dev(hits[en].astype(np.int32))
        a0 = torch.empty(nh, dtype=torch.float64, device="cuda")
        a1 = torch.empty(nh, dtype=torch.float64, device="cuda")
        _lib.check(lib.wfb_group_hit_windows(_ptr(d_ts), _ptr(d_pos), _ptr(d_s), _ptr(d_e), _ptr(d_dt), _ptr(d_rid), nh, float(time_window_ns),
                                             _ptr(order), _ptr(ev), _ptr(a0), _ptr(a1), _ptr(n_ev), _ptr(ws), ws.numel(), _stream()),
                   "wfb_group_hit_windows")
    event_of_hit = ev.cpu().numpy()
    abs0, abs1 = a0.cpu().numpy(), a1.cpu().numpy()
    n_events = int(n_ev.item())
    morder = np.lexsort((hits["record_id"].astype(np.int64), hits["timestamp"].astype(np.int64), abs0, hits["dt"].astype(np.int32),
                         hits["channel"].astype(np.int16), hits["board"].astype(np.int16), event_of_hit))
    counts = np.bincount(event_of_hit, minlength=n_events)
    offsets = np.zeros(n_events + 1, dtype=np.int64)
    np.cumsum(counts, out=offsets[1:])
    tmin = np.full(n_events, np.inf)
    tmax = np.full(n_events, -np.inf)
    np.minimum.at(tmin, event_of_hit, abs0)
    np.maximum.at(tmax, event_of_hit, abs1)
    t_min, t_max = tmin.astype(np.int64), tmax.astype(np.int64)
    return dict(event_id=np.arange(n_events, dtype=np.int64), t_min=t_min, t_max=t_max, dt_ns=(t_max - t_min) / 1e3,
                n_hits=counts.astype(np.int64), offsets=offsets, members=morder.astype(np.int64), event_of_hit=event_of_hit,
                order=order.cpu().numpy())


def synth_hits(min_hits: int) -> np.ndarray:
    n = 1_000_000
    while True:
        run = DeviceRun.synth(n, L, NCH, seed=2026, with_rows=False)
        res = run.features_hits(threshold=THR, hit_cap=1024, features=False)
        total = int(res["total"].item())
        if total >= min_hits:
            out = {"hits": torch.empty((total + 16) * 60, dtype=torch.uint8, device="cuda")}
            run.features_hits(threshold=THR, hit_cap=total + 16, features=False, out=out)
            run.check()
            return out["hits"][: total * 60].cpu().numpy().view(THRESHOLD_HIT_DTYPE).copy()
        n = int(n * min_hits / max(total, 1) * 1.05) + 1
        del run, res
        torch.cuda.empty_cache()


def timed(fn, *a):
    torch.cuda.synchronize()
    t = time.perf_counter()
    out = fn(*a)
    torch.cuda.synchronize()
    return time.perf_counter() - t, out


gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True).stdout.strip()
hits = synth_hits(args.min_hits)
print(f"GPU: {gpu} | {len(hits)} threshold hits, time_window_ns {WINDOW}")
for gap in (0.0, 50.0):
    _, merged, comps = ops.hit_merge(hits, merge_gap_ns=gap)
    call = (merged, WINDOW, comps, hits)
    new_out = ops.group_hit_windows(*call)  # warm-up of both, and the identity check
    old_out = group_hit_windows_host_table(*call)
    for k in ("event_id", "t_min", "t_max", "dt_ns", "n_hits", "offsets", "members", "event_of_hit", "order"):
        assert new_out[k].dtype == old_out[k].dtype and np.array_equal(new_out[k], old_out[k]), k
    t_new, t_old = [], []
    for _ in range(args.reps):
        t_old.append(timed(group_hit_windows_host_table, *call)[0])
        t_new.append(timed(ops.group_hit_windows, *call)[0])
    sizes = new_out["n_hits"]
    print(f"merge_gap_ns {gap:g}: {len(merged)} hit_merged rows ({int((merged['sample_start'] < 0).sum())} across records), "
          f"{len(sizes)} events (max {int(sizes.max())} members) | ops.group_hit_windows: host table "
          f"{1e3 * min(t_old):.0f} ms (median {1e3 * np.median(t_old):.0f}), device table {1e3 * min(t_new):.0f} ms "
          f"(median {1e3 * np.median(t_new):.0f}) over {args.reps} alternating calls | results identical")
