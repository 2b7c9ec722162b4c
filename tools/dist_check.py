#!/usr/bin/env python
"""Multi-GPU parity check of the time-sharded pipeline (run under torchrun, one rank per GPU, NCCL):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 tools/dist_check.py \
        [--records-per-rank 2000000] [--verify 1]

Every rank generates ITS time shard of one synthetic run on its GPU, runs the fused features + hits pass and then
hit_merge (merge_gap_ns = 50) -> hit_grouped (time_window_ns = 100) with ``distributed.merge_group_sharded``: the hit
rows never leave the device, the ranks exchange their boundary zones (one all_gather of 2 x 4096 rows per rank) and
two counts.  With --verify 1 rank 0 additionally processes the WHOLE run on its own GPU and checks that the ranks'
feature rows, hit rows, merged rows (after the channel-major assembly) and event ids equal the single-GPU ones byte
for byte; at sizes that no single GPU holds (--verify 0) the check is structural: counts add up, every rank's windows
lie between its cuts, event ids are contiguous across ranks.

--source v1725 starts from files instead: every rank writes its own V1725 .bin files (file i seeded by i, board i, all
16 channels, --samples per waveform; every file spans the same time range, so the exchange moves (P - 1) / P of every
rank's records), builds its time shard with ``distributed.build_records_sharded_v1725`` and runs the same fused ->
merge_group_sharded path.  It reports the time of every ingest stage, the exchange bytes and rate, the merge kernel's
rate against its algorithmic bytes (4 L + 252 per record), the peak device memory, and the GPU name and power limit;
with --verify 1 rank 0 rebuilds all files on one GPU and checks records, pool, features, hits, merged rows and event
ids byte for byte.

--source raw does the same from raw digitizer rows, as a rank gets them from the reference's format_reader: every rank
generates its --groups-per-rank per-channel groups (group g seeded by g alone, board g // 16, channel g % 16, --samples
per row, or 3/4 of that in odd groups with --mixed-widths; every group spans the same time range) and builds its time
shard with ``distributed.build_records_sharded``.  It reports the same figures; with --verify 1 rank 0 rebuilds all
groups with ops.build_records (one width) or ops.build_records_ragged (several) and checks the same outputs.

--events adds the df -> df_events -> df_paired leg on the same shards: ``distributed.df_sharded`` on the rank's feature
rows, then ``distributed.events_sharded`` (time_window_ns = pair window = 100, 2 paired channels).  It reports the time of
every stage (each ended by a device synchronize), gathered_bytes, the event counts and the peak device memory of the leg;
with --verify 1 rank 0 runs the single-GPU chain (df columns, wfb_group_time_window, wfb_event_table, wfb_pair_events
on the whole run) and checks the gathered df columns, event table, members and df_paired columns byte for byte.

--hit-events adds the hit_grouped event table on the rows merge_group_sharded left on every rank:
``distributed.hit_events_sharded`` with the device backend (wfb_hit_event_table).  It reports the table's stage time
(ended by a device synchronize), the events and member rows of every rank and the peak extra device memory of the stage;
with --verify 1 every rank gathers the hit_grouped frame of the whole run (``distributed.gather_hit_grouped_frame``) and
rank 0 checks it against ``ops.group_hit_windows`` on the single-GPU hit_merged rows, packaged as B200HitGroupedPlugin
does.

--peaks adds the wave_pool_filtered -> hit -> waveform_width -> s1_s2 leg on a positive-pulse copy of every rank's
shard (samples and baselines mirrored around the 14-bit mid-scale, as bench.py's c3 leg makes them: waveform_width keeps
only peaks above the row's baseline): ``distributed.peaks_sharded`` with the SG filter (11 / 2), hit (height 8, width
2), waveform_width (0.25 GHz) and s1_s2 on the shard's basic_features.  It reports the row counts, the time of every
stage (each ended by a device synchronize) and the peak extra device memory of the leg; with --verify 1 rank 0 runs
the same chain on the whole run (the rank-order concatenation of the shards) and checks the gathered filtered pool,
hit, waveform_width and s1_s2 rows byte for byte.

--peaks --channels runs the leg as a detector whose channels are not configured alike: the polarity comes from a
channel map (even channels positive, odd channels left unknown; ``ops.apply_polarity``, its time reported as
``polarity``) instead of marking every record positive, and the filter from ``B200WavePoolFilteredPlugin`` options with
a ``channel_config`` that gives a quarter of the channels a Butterworth band-pass (order 4, 0.01-0.1 at 0.25 GHz) and
leaves the rest on SG 11/2; --verify 1 compares with the same chain on the whole run."""
import argparse
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torch.distributed as dist

from waveformanalysis_b200 import distributed as D
from waveformanalysis_b200 import engine, ops
from waveformanalysis_b200.dtypes import HIT_MERGED_DTYPE, RECORDS_DTYPE, THRESHOLD_HIT_DTYPE

ap = argparse.ArgumentParser()
ap.add_argument("--records-per-rank", type=int, default=1_000_000)
ap.add_argument("--verify", type=int, default=1)
ap.add_argument("--zone-rows", type=int, default=4096)
ap.add_argument("--source", choices=("synth", "v1725", "raw"), default="synth")
ap.add_argument("--files-per-rank", type=int, default=2)
ap.add_argument("--groups-per-rank", type=int, default=2)
ap.add_argument("--mixed-widths", action="store_true", help="--source raw: odd groups have 3/4 of --samples per row")
ap.add_argument("--samples", type=int, default=800)
ap.add_argument("--events", action="store_true", help="also run the sharded df -> df_events -> df_paired leg")
ap.add_argument("--hit-events", action="store_true", help="also build the sharded hit_grouped event table")
ap.add_argument("--peaks", action="store_true", help="also run the sharded filter -> hit -> waveform_width -> s1_s2 leg")
ap.add_argument("--channels", action="store_true", help="--peaks with a polarity map and per-channel filters")
args = ap.parse_args()

D.init_process_group("nccl")
rank, ws, local = D.world()
torch.cuda.set_device(local)
n, L, NCH, SEED = args.records_per_rank, args.samples, 16, 4242
DT_INGEST = 4
THR, WINDOW, GAP = 15.0, 100.0, 50.0


def fused(run):
    res = run.features_hits(threshold=THR, hit_cap=1024)
    torch.cuda.synchronize()
    total = int(res["total"].item())
    out = {"hits": torch.empty((total + 16) * 60, dtype=torch.uint8, device="cuda")}
    res = run.features_hits(threshold=THR, hit_cap=total + 16, out=out)
    torch.cuda.synchronize()
    run.check()
    return res, total


def v1725_file(i: int, n_events: int) -> np.ndarray:
    """Stream of file i: board i, every event fires all 16 channels with L samples; seeded by i alone."""
    rng = np.random.default_rng(1000 + i)
    ev_dt = np.dtype([("hdr", "u1", 16), ("ch", [("hdr", "u1", 12), ("wave", "<i2", L)], 16)])
    a = np.zeros(n_events, ev_dt)
    a["hdr"][:, 4] = a["hdr"][:, 11] = 0xFF
    size = 3 + L // 2
    step = rng.integers(1, 4 * L, n_events)
    step[::5] = 0  # events sharing a timestamp
    t = np.cumsum(step).astype(np.int64)
    ts = t[:, None] + rng.integers(0, 3, (n_events, 16))
    ch = a["ch"]
    ch["hdr"][..., 0], ch["hdr"][..., 1], ch["hdr"][..., 2] = size & 0xFF, (size >> 8) & 0xFF, (size >> 16) & 0x3F
    for b in range(6):
        ch["hdr"][..., 4 + b] = (ts >> (8 * b)) & 0xFF
    ch["hdr"][..., 10], ch["hdr"][..., 11] = 8000 & 0xFF, 8000 >> 8
    block = (8000 + rng.integers(-4, 5, 1 << 20)).astype(np.int16)
    for k in range(0, len(block) - 40, 997):  # negative pulses
        block[k:k + 12] -= 150
    windows = np.lib.stride_tricks.sliding_window_view(block, L)
    for e0 in range(0, n_events, 2048):
        e1 = min(e0 + 2048, n_events)
        ch["wave"][e0:e1] = windows[rng.integers(0, len(windows), (e1 - e0, 16))]
    return a.view(np.uint8)


def v1725_name(i: int) -> str:
    return f"run_b{i}_seg0.bin"


def raw_group(g: int, m: int):
    """Raw rows of group g (timestamps_ps, boards, channels, int16 samples): one channel over the whole run; seeded by g."""
    rng = np.random.default_rng(2000 + g)
    width = L - L // 4 if args.mixed_widths and g % 2 else L
    step = rng.integers(1, 4 * L, m)
    step[::5] = 0  # rows sharing a timestamp
    ts = (np.cumsum(step) + rng.integers(0, 3, m)) * (DT_INGEST * 1000)
    block = (8000 + rng.integers(-4, 5, 1 << 20)).astype(np.int16)
    for k in range(0, len(block) - 40, 997):  # negative pulses
        block[k:k + 12] -= 150
    windows = np.lib.stride_tricks.sliding_window_view(block, width)
    samples = np.empty((m, width), dtype=np.int16)
    for r0 in range(0, m, 1 << 15):
        r1 = min(r0 + (1 << 15), m)
        samples[r0:r1] = windows[rng.integers(0, len(windows), r1 - r0)]
    return ts.astype(np.int64), np.full(m, g // NCH, np.int16), np.full(m, g % NCH, np.int16), samples


def report_ingest(title: str, wall: float, peak: int):
    """Print every rank's ingest line on rank 0: stage times, exchange, merge rate against its algorithmic bytes (read and
    write of the samples and the row, write of the 48 B meta), peak memory, GPU.  Returns (run, n, n_total)."""
    import subprocess

    run = ingest["run"]
    tm = ingest["timings"]
    n_all = ingest["n_total"]
    per_record = 4 * run.pool_len / max(run.n, 1) + 252
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(local)],
                         capture_output=True, text=True).stdout.strip()
    line = (f"rank {rank}: records {run.n} (base {ingest['record_base']}) | " +
            " ".join(f"{k} {1e3 * v:.1f} ms" for k, v in tm.items()) +
            f" | exchange {ingest['exchange_bytes'] / 1e9:.3f} GB received, {ingest['exchange_bytes'] / max(tm['exchange'], 1e-9) / 1e9:.1f} GB/s"
            f" | merge {per_record * run.n / max(tm['merge'], 1e-9) / 1e9:.0f} GB/s of {per_record:.0f} B/record"
            f" | ingest wall {1e3 * wall:.1f} ms, {n_all / wall / 1e6:.1f} M records/s run-wide"
            f" | peak device memory {peak / 1e9:.2f} GB ({peak / max(2 * run.pool_len, 1):.2f} x the shard's sample bytes) | {gpu}")
    lines = D.gather_rows(np.frombuffer(line.encode().ljust(1024)[:1024], dtype="S1024")) if ws > 1 else [line.encode()]
    if rank == 0:
        print(f"{title} records={n_all} samples/record={L}")
        for ln in lines:
            print("  " + ln.decode().strip())
    return run, run.n, n_all


ingest = None
if args.source == "v1725":
    import shutil
    import tempfile

    F = ws * args.files_per_rank
    ev_per_file = max(n // (NCH * args.files_per_rank), 1)
    tmp = tempfile.mkdtemp(prefix=f"v1725_r{rank}_")
    paths = [os.path.join(tmp, v1725_name(i)) for i in range(F)]  # every rank lists every file; it writes its own
    mine = list(range(rank * args.files_per_rank, (rank + 1) * args.files_per_rank))
    for i in mine:
        v1725_file(i, ev_per_file).tofile(paths[i])
    torch.cuda.reset_peak_memory_stats()
    if ws > 1:
        dist.barrier()
    tw = time.perf_counter()
    ingest = D.build_records_sharded_v1725(paths, dt_ns=DT_INGEST, mine=mine)
    torch.cuda.synchronize()
    wall = time.perf_counter() - tw
    peak = torch.cuda.max_memory_allocated()
    shutil.rmtree(tmp, ignore_errors=True)
    run, n, n_all = report_ingest(f"v1725 ingest: world={ws} files={F}", wall, peak)
elif args.source == "raw":
    G = ws * args.groups_per_rank
    rows_per_group = max(n // args.groups_per_rank, 1)
    groups = {g: raw_group(g, rows_per_group) for g in range(rank * args.groups_per_rank, (rank + 1) * args.groups_per_rank)}
    torch.cuda.reset_peak_memory_stats()
    if ws > 1:
        dist.barrier()
    tw = time.perf_counter()
    ingest = D.build_records_sharded(groups, n_groups=G, dt_ns=DT_INGEST)
    torch.cuda.synchronize()
    wall = time.perf_counter() - tw
    peak = torch.cuda.max_memory_allocated()
    del groups
    widths = f"{L} and {L - L // 4}" if args.mixed_widths else f"{L}"
    run, n, n_all = report_ingest(f"raw ingest: world={ws} groups={G} widths={widths}", wall, peak)
else:
    run = engine.DeviceRun.synth(n, L, NCH, seed=SEED, record_base=rank * n, with_rows=args.channels)
res, total = fused(run)
if ws > 1:
    dist.barrier()
torch.cuda.synchronize()
t0 = time.perf_counter()
sh = D.merge_group_sharded((res["hits"][: total * 60], total), D.DeviceRows(THRESHOLD_HIT_DTYPE), time_window_ns=WINDOW, merge_gap_ns=GAP,
                           span_ns=(run.lmax * DT_INGEST if ingest is not None else L * 2.0), zone_rows=args.zone_rows)
torch.cuda.synchronize()
if ws > 1:
    dist.barrier()
t1 = time.perf_counter()
ncl, nev = sh["n_clusters"], sh["n_events"]
ev = sh["event_of_merged"]
# structural checks on every rank
a0 = sh["detail"]["abs_start"][:ncl]
i = [r for r in range(ws) if sh["clusters_per_rank"][r] > 0]
lo = sh["cuts"][i[i.index(rank) - 1]] if rank in i and i.index(rank) > 0 else -np.inf
hi = sh["cuts"][rank] if rank in i and i.index(rank) + 1 < len(i) else np.inf
if ncl:
    assert float(a0.min().item()) >= lo and float(a0.max().item()) < hi, "a cluster starts outside the rank's cuts"
    assert int(ev.min().item()) == sh["event_base"] and int(ev.max().item()) == sh["event_base"] + nev - 1, "event ids are not contiguous"
owned_n = sh["owned"][1]
tot = torch.tensor([total, owned_n, ncl, nev], dtype=torch.int64, device="cuda")
if ws > 1:
    dist.all_reduce(tot)
assert int(tot[0]) == int(tot[1]), "hits were lost or duplicated by the ownership exchange"
msg = (f"world={ws} records/rank={n} hits={int(tot[0])} clusters={int(tot[2])} events={int(tot[3])} zone_rows={sh['zone_rows']} "
       f"gathered_bytes/rank={sh['gathered_bytes']} merge+group wall={1e3 * (t1 - t0):.1f} ms")

EV_COLS = ("t_min", "t_max", "dt_ns", "n_hits", "members", "member_ts", "member_channel", "member_area", "member_height", "keep",
           "delta_t", "area_ch", "height_ch")


def events_leg() -> str:
    """df_sharded + events_sharded on this rank's shard; with --verify the single-GPU chain on rank 0."""
    import subprocess

    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base_mem = torch.cuda.memory_allocated()
    if ws > 1:
        dist.barrier()
    t = time.perf_counter()
    df = D.df_sharded(run, res["features"])
    torch.cuda.synchronize()
    t_df = time.perf_counter() - t
    t = time.perf_counter()
    ev = D.events_sharded(df, time_window_ns=WINDOW, pair_window_ns=WINDOW, n_channels=2, start_channel_slice=6, zone_rows=args.zone_rows)
    torch.cuda.synchronize()
    t_ev = time.perf_counter() - t
    peak = torch.cuda.max_memory_allocated() - base_mem
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(local)],
                         capture_output=True, text=True).stdout.strip()
    line = (f"rank {rank}: df rows {df['n']} owned {ev['owned'][1] - ev['owned'][0]} events {ev['n_events']} (base {ev['event_base']}) | "
            f"df_sharded {1e3 * t_df:.1f} ms | events_sharded {1e3 * t_ev:.1f} ms: " +
            " ".join(f"{k} {1e3 * v:.1f} ms" for k, v in ev["timings"].items()) +
            f" | gathered {ev['gathered_bytes']} B, zone_rows {ev['zone_rows']} | peak device memory of the leg {peak / 1e9:.3f} GB | {gpu}")
    lines = D.gather_rows(np.frombuffer(line.encode().ljust(1024)[:1024], dtype="S1024")) if ws > 1 else [line.encode()]
    if rank == 0:
        print(f"events leg: world={ws} records/rank={n}")
        for ln in lines:
            print("  " + ln.decode().strip())
    out = f"events={int(ev['events_per_rank'].sum())} gathered_bytes/rank={ev['gathered_bytes']}"
    if not args.verify:
        return out
    host = lambda x: x.cpu().numpy()  # noqa: E731
    got_df = {k: D.gather_rows(host(df["cols"][k])) for k in ("timestamp", "record_id", "area", "height", "channel")}
    got_df["index"] = D.gather_rows(host(df["index"]))
    got = {}
    for k in EV_COLS:
        a = np.ascontiguousarray(host(ev[k]))
        rows = a.view(np.dtype((np.void, a.dtype.itemsize * a.shape[1]))).reshape(-1) if a.ndim > 1 else a  # one row per event
        got[k] = D.gather_rows(rows)
    feats = D.gather_rows(res["features"][: n * 36].cpu().numpy().view([("b", "u1", (36,))]))
    return out + (verify_events(got_df, got, feats) if rank == 0 else "")


def verify_events(got_df, got, feats) -> str:
    from waveformanalysis_b200.engine import upload

    n_all = len(feats)
    rid = np.sort(got_df["record_id"])  # the whole run's record ids in row order (shards are contiguous record ranges)
    want = ops.df_columns_device(upload(feats.view(np.uint8).reshape(-1)), n_all, upload(rid))
    for k in ("timestamp", "record_id", "area", "height", "channel"):
        assert want[k].cpu().numpy().tobytes() == got_df[k].tobytes(), f"df.{k} differs"
    assert np.array_equal(want["order"].cpu().numpy(), got_df["index"]), "df index differs"
    ts = want["timestamp"]
    e, n_ev = ops.group_time_window_device(ts, n_all, WINDOW)
    t = ops.event_table_device(ts, e, n_all, n_ev, want["channel"], area=want["area"], height=want["height"])
    t.update(ops.pair_events_device(t["offsets"], n_ev, t["member_ts"], t["member_area"], t["member_height"], t["dt_ns"], WINDOW, 2))
    for k in EV_COLS:
        w = np.ascontiguousarray(t[k].cpu().numpy())
        assert w.tobytes() == np.ascontiguousarray(got[k]).tobytes(), f"events.{k} differs"
    return f" | df, df_events and df_paired columns byte-identical to the single-GPU chain ({n_all} rows, {n_ev} events)"


def gpu_name() -> str:
    import subprocess

    return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(local)],
                          capture_output=True, text=True).stdout.strip()


def hit_events_leg():
    """hit_events_sharded on this rank's merge_group_sharded result; with --verify the gathered hit_grouped frame."""
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base_mem = torch.cuda.memory_allocated()
    if ws > 1:
        dist.barrier()
    t = time.perf_counter()
    hev = D.hit_events_sharded(sh, D.DeviceRows(THRESHOLD_HIT_DTYPE))
    torch.cuda.synchronize()
    t_tab = time.perf_counter() - t
    peak = torch.cuda.max_memory_allocated() - base_mem
    line = (f"rank {rank}: events {hev['n_events']} (base {hev['event_base']}) member rows {int(hev['members'].numel())} | "
            f"hit_events_sharded {1e3 * t_tab:.2f} ms | peak extra device memory {peak / 1e9:.3f} GB | {gpu_name()}")
    lines = D.gather_rows(np.frombuffer(line.encode().ljust(1024)[:1024], dtype="S1024")) if ws > 1 else [line.encode()]
    if rank == 0:
        print(f"hit events leg: world={ws} records/rank={n}")
        for ln in lines:
            print("  " + ln.decode().strip())
    frame = D.gather_hit_grouped_frame(hev) if args.verify else None
    return f"hit events={int(hev['events_per_rank'].sum())}", frame


PEAK_FILTER = {"filter_type": "SG", "sg_window_size": 11, "sg_poly_order": 2}
PEAK_OPTS = {"height": 8.0, "width": 2}
WIDTH_OPTS = {"sampling_rate": 0.25}
S1S2_OPTS = {"s1_width_range": (None, 60.0), "s2_width_range": (40.0, None), "conflict_policy": "prefer_s2"}


# --channels: the same map and filter options on every rank (every board a run of up to 64 files can have)
CH_POLARITY = {(b, c): "positive" if c % 2 == 0 else "unknown" for b in range(64) for c in range(NCH)}
CH_FILTER = {"filter_type": "SG", "sg_window_size": 11, "sg_poly_order": 2, "filter_order": 4, "lowcut": 0.01, "highcut": 0.1, "fs": 0.25}
CH_CONFIG = {"channels": {f"{b}:{c}": {"filter_type": "BW"} for b in range(64) for c in range(0, NCH, 4)}}


def positive_copy(r):
    """A copy of a run with positive pulses, as bench.py's c3 leg makes them: samples and baselines mirrored around the
    14-bit mid-scale, records marked positive (waveform_width keeps only peaks above the row's baseline); with
    --channels the polarity comes from CH_POLARITY instead.  Returns the copy and the seconds of ops.apply_polarity."""
    meta = r.meta.clone()
    m = meta.view(-1, 48)
    base = m[:, 8:16].contiguous().view(torch.float64).view(-1)
    m[:, 8:16] = (16383.0 - base).view(torch.uint8).view(-1, 8)
    rows = r.records_rows
    if not args.channels:
        m[:, 36] = 1  # WFB_POL_POSITIVE
    elif rows is not None:
        rows = rows.clone()
    out = engine.DeviceRun(meta, 16383 - r.pool, r.n, 0, r.lmax, records_rows=rows, pool_base=r.pool_base, row_base=r.row_base)
    out.lmin = r.lmin
    t_pol = 0.0
    if args.channels:
        torch.cuda.synchronize()
        t = time.perf_counter()
        ops.apply_polarity(out, CH_POLARITY)
        torch.cuda.synchronize()
        t_pol = time.perf_counter() - t
    return out, t_pol


def peaks_filter() -> dict:
    return dict(filter_options=CH_FILTER, channel_config=CH_CONFIG, run_id="run") if args.channels else dict(filter_cfg=PEAK_FILTER)


def peaks_rows_host(x: dict):
    from waveformanalysis_b200.dtypes import HIT_DTYPE, S1_S2_CLASSIFIER_DTYPE, WAVEFORM_WIDTH_DTYPE

    return tuple(x[k][: x["n_" + k] * dt.itemsize].cpu().numpy().tobytes()
                 for k, dt in (("hits", HIT_DTYPE), ("widths", WAVEFORM_WIDTH_DTYPE), ("labels", S1_S2_CLASSIFIER_DTYPE)))


def peaks_leg() -> str:
    """filter -> hit -> waveform_width -> s1_s2 on this rank's shard (positive copy) with distributed.peaks_sharded; with
    --verify rank 0 runs the same chain on the whole run (the rank-order concatenation of the shards) on its GPU."""
    positive_copy(run)  # warm-up: the first launch of the polarity kernel loads the module
    prun, t_pol = positive_copy(run)
    feats = prun.features_hits(hits=False)["features"]
    if args.channels:  # warm-up: the first Butterworth design imports scipy.signal
        ops.filter_run_device(prun, **peaks_filter())
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base_mem = torch.cuda.memory_allocated()
    if ws > 1:
        dist.barrier()
    t = time.perf_counter()
    ph = D.peaks_sharded(prun, features=feats, peak_opts=PEAK_OPTS, width_opts=WIDTH_OPTS, s1s2_opts=S1S2_OPTS, **peaks_filter())
    torch.cuda.synchronize()
    wall = time.perf_counter() - t
    peak = torch.cuda.max_memory_allocated() - base_mem
    line = (f"rank {rank}: records {prun.n} hits {ph['n_hits']} widths {ph['n_widths']} labels {ph['n_labels']} (bases {ph['hit_base']} / "
            f"{ph['width_base']} / {ph['label_base']}) | " + (f"polarity {1e3 * t_pol:.2f} ms " if args.channels else "") + " ".join(f"{k} {1e3 * v:.1f} ms" for k, v in ph["timings"].items()) +
            f" | leg wall {1e3 * wall:.1f} ms | peak extra device memory {peak / 1e9:.3f} GB "
            f"({peak / max(2 * prun.pool_len, 1):.2f} x the shard's 16-bit sample bytes) | {gpu_name()}")
    lines = D.gather_rows(np.frombuffer(line.encode().ljust(1024)[:1024], dtype="S1024")) if ws > 1 else [line.encode()]
    if rank == 0:
        what = ("polarity map (even channels positive, odd unknown), filter per channel (BW order 4 on a quarter, SG 11/2 on the rest)"
                if args.channels else "filter SG 11/2")
        print(f"peaks leg: world={ws} records/rank={n} samples/record={L} {what}, hit height 8 width 2, waveform_width 0.25 GHz")
        for ln in lines:
            print("  " + ln.decode().strip())
    out = f"peaks: hits={ph['n_hits_total']} widths={ph['n_widths_total']} labels={ph['n_labels_total']}"
    if not args.verify:
        return out
    got_sg = D.gather_rows(ph["filtered"].cpu().numpy())
    got = D.gather_peak_rows(ph)
    if ingest is not None:
        recs_all = D.gather_rows(run.records_rows[: run.n * 102].cpu().numpy().view(RECORDS_DTYPE))
        pool_all = D.gather_rows(run.pool.cpu().numpy().view([("s", "<u2")]))["s"]
    del ph, prun, feats
    if rank != 0:
        return out
    torch.cuda.empty_cache()
    whole = engine.DeviceRun.from_host(recs_all, pool_all) if ingest is not None else engine.DeviceRun.synth(n * ws, L, NCH, seed=SEED)
    whole, _ = positive_copy(whole)
    want = D.peaks_local(whole, features=whole.features_hits(hits=False)["features"], peak_opts=PEAK_OPTS, width_opts=WIDTH_OPTS,
                         s1s2_opts=S1S2_OPTS, **peaks_filter())
    assert want["filtered"].cpu().numpy().tobytes() == got_sg.tobytes(), "filtered pool differs"
    for name, g, w in zip(("hit", "waveform_width", "s1_s2"), got, peaks_rows_host(want)):
        assert g.tobytes() == w, f"{name} rows differ"
    labels = got[2]["label"]
    return out + (f" | filtered pool, hit, waveform_width and s1_s2 rows byte-identical to the single-GPU chain on the whole run "
                  f"({whole.n} records; labels S1 {int((labels == 1).sum())}, S2 {int((labels == 2).sum())}, unknown {int((labels == 0).sum())})")


def frames_equal(got, want) -> bool:
    if list(got.columns) != list(want.columns) or len(got) != len(want) or not got.index.equals(want.index):
        return False
    for c in want.columns:
        if got[c].dtype != want[c].dtype:
            return False
        if want[c].dtype == object:
            if not all(a.dtype == b.dtype and np.array_equal(a, b) for a, b in zip(got[c], want[c])):
                return False
        elif not np.array_equal(got[c].to_numpy(), want[c].to_numpy()):
            return False
    return True


if args.events:
    msg += " | " + events_leg()
if args.peaks:
    msg += " | " + peaks_leg()
hit_frame = None
if args.hit_events:
    out, hit_frame = hit_events_leg()
    msg += " | " + out
if args.verify:
    feats_l = res["features"][: n * 36].cpu().numpy()
    hits_l = res["hits"][: total * 60].cpu().numpy().view(THRESHOLD_HIT_DTYPE)
    merged_l = sh["merged"][: ncl * 72].cpu().numpy().view(HIT_MERGED_DTYPE)
    ev_l = ev.cpu().numpy().view([("e", "i8")])
    feats = D.gather_rows(feats_l.view([("b", "u1", (36,))]))
    hits = D.gather_rows(hits_l)
    merged = D.gather_rows(merged_l)
    evs = D.gather_rows(ev_l)["e"]
    if ingest is not None:
        recs_all = D.gather_rows(run.records_rows[: n * 102].cpu().numpy().view(RECORDS_DTYPE))
        pool_all = D.gather_rows(run.pool.cpu().numpy().view([("s", "<u2")]))["s"]
    if rank == 0:
        del run, res, sh
        torch.cuda.empty_cache()
        if ingest is not None:
            if args.source == "v1725":
                want_rec, want_pool = ops.build_records_from_v1725([v1725_file(i, ev_per_file) for i in range(F)],
                                                                   [v1725_name(i) for i in range(F)], DT_INGEST)
            else:
                gs = [raw_group(g, rows_per_group) for g in range(G)]
                ts, b, c = (np.concatenate([x[k] for x in gs]) for k in range(3))
                if len({x[3].shape[1] for x in gs}) > 1:
                    want_rec, want_pool = ops.build_records_ragged(ts, b, c, [x[3] for x in gs], dt_ns=DT_INGEST)
                else:
                    want_rec, want_pool = ops.build_records(ts, b, c, np.vstack([x[3] for x in gs]), dt_ns=DT_INGEST)
                del gs, ts, b, c
            assert recs_all.tobytes() == want_rec.tobytes(), "records differ"
            assert np.array_equal(pool_all, want_pool), "wave_pool differs"
            full = engine.DeviceRun.from_host(want_rec, want_pool)
            del want_pool, pool_all
        else:
            full = engine.DeviceRun.synth(n * ws, L, NCH, seed=SEED)
        n_all = full.n
        fres, ftotal = fused(full)
        assert np.array_equal(feats.view(np.uint8).reshape(-1), fres["features"][: n_all * 36].cpu().numpy()), "features differ"
        assert np.array_equal(hits.view(np.uint8).reshape(-1), fres["hits"][: ftotal * 60].cpu().numpy()), "hit rows differ"
        m = ops.hit_merge_device(fres["hits"][: ftotal * 60], ftotal, merge_gap_ns=GAP)
        g = ops.group_rows_device(m["merged"], m["n_clusters"], 72, WINDOW, abs_start=m["abs_start"], abs_end=m["abs_end"])
        want_m = m["merged"][: m["n_clusters"] * 72].cpu().numpy().view(HIT_MERGED_DTYPE)
        want_ev = g["event_of_row"][: m["n_clusters"]].cpu().numpy()
        got_m, got_ev = D.assemble_merged(merged, evs)
        assert len(got_m) == len(want_m), (len(got_m), len(want_m))
        for f in want_m.dtype.names:
            if f == "component_offset":
                continue
            assert np.array_equal(got_m[f], want_m[f], equal_nan=want_m[f].dtype.kind == "f"), f"hit_merged.{f} differs"
        assert np.array_equal(got_ev, want_ev), "event ids differ"
        assert g["n_events"] == int(tot[3])
        if hit_frame is not None:
            from waveformanalysis_b200.dtypes import HIT_MERGED_COMPONENTS_DTYPE
            from waveformanalysis_b200.plugins.grouping import hit_grouped_frame, hit_member_columns

            comps = np.zeros(ftotal, dtype=HIT_MERGED_COMPONENTS_DTYPE)
            comps["merged_index"] = m["cluster_index"][:ftotal].cpu().numpy()
            comps["hit_index"] = m["order"][:ftotal].cpu().numpy()
            table = ops.group_hit_windows(want_m, WINDOW, comps, hits)
            assert frames_equal(hit_frame, hit_grouped_frame(table, hit_member_columns(want_m[table["members"]]))), "hit_grouped differs"
            msg += f" | hit_grouped frame equal to ops.group_hit_windows on the single-GPU hit_merged ({len(hit_frame)} events)"
        merged_over = int((want_m["component_count"] > 1).sum())
        what = "records, pool, " if ingest is not None else ""
        msg += f" | {what}features, hits, merged rows and event ids byte-identical to the single-GPU run ({n_all} records, {merged_over} clusters of several hits)"
if rank == 0:
    print("dist_check OK:", msg, f"backend={dist.get_backend() if ws > 1 else 'single'}")
if ws > 1:
    dist.barrier()
    dist.destroy_process_group()
