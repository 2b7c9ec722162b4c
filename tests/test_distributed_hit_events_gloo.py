"""CPU, 2 / 3 / 4 gloo ranks: the hit_grouped event table of a time-sharded run (distributed.hit_events_sharded after
merge_group_sharded, HostRows backend: the compute is the oracle's) and the gathered frame
(distributed.gather_hit_grouped_frame) against the oracle's group_hit_windows of the whole run.

Besides equality, every case pins the two facts that make the rank-order concatenation exact: every event's members
lie on one rank, and a rank's merged rows keep their global (board, channel)-major relative order."""

import os
import socket
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
W_NS = 100.0
CASES = ("base", "grow", "empty", "one_event", "ties")


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _case(name, hits, n_rec, world_size):
    """(hits, record bounds of the ranks, time window, zone rows) of one case."""
    from waveformanalysis_b200 import distributed as D

    b = D.shard_bounds(n_rec, world_size)
    if name == "empty":  # rank 1 holds no records: rank 0 takes its range
        b[1] = b[2]
    if name == "one_event":  # one event over the whole run: only one rank may hold rows, the others are empty
        b = np.full(world_size + 1, n_rec, dtype=np.int64)
        b[: world_size // 2 + 1] = 0
        return hits, b, 1e12, 64
    if name == "ties":  # every third hit twice, tied on all six keys (heights differ so that the order shows)
        dup = hits[::3].copy()
        dup["height"] += 1.0
        both = np.concatenate([hits, dup])
        o = np.argsort(np.r_[np.arange(len(hits)), np.arange(0, len(hits), 3)], kind="stable")
        return both[o], b, W_NS, 64
    return hits, b, W_NS, (4 if name == "grow" else 64)


def _worker(rank, world_size, port, merge_gap, q):
    sys.path.insert(0, ROOT)
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world_size), LOCAL_RANK=str(rank), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    import torch.distributed as dist

    from oracle import np_oracle as O
    from waveformanalysis_b200 import distributed as D
    from waveformanalysis_b200.plugins.grouping import hit_grouped_frame, hit_member_columns
    from waveformanalysis_b200.synth import make_raw_run, records_from_raw

    dist.init_process_group("gloo", rank=rank, world_size=world_size)
    raw = make_raw_run(6, 120, 400, seed=77, coincidence_fraction=0.6)
    rec, pool = records_from_raw(raw)
    hits0 = O.threshold_hits(rec, pool, threshold=12.0)
    out = []
    for name in CASES:
        hits, b, w, zone_rows = _case(name, hits0, len(rec), world_size)
        mine = hits[(hits["record_id"] >= b[rank]) & (hits["record_id"] < b[rank + 1])]
        backend = D.HostRows(O.hit_merge, O.group_hit_windows)
        sh = D.merge_group_sharded(mine, backend, time_window_ns=w, merge_gap_ns=merge_gap, span_ns=400 * 2.0, zone_rows=zone_rows)
        keep = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in sh.items() if k in ("merged", "event_of_merged", "n_events")}
        ev = D.hit_events_sharded(sh, backend)
        unchanged = all(np.array_equal(sh[k], v) if isinstance(v, np.ndarray) else sh[k] == v for k, v in keep.items())
        frame = D.gather_hit_grouped_frame(ev)
        # the tables and the rows they index, gathered in rank order
        tab = np.zeros(ev["n_events"], dtype=[("t_min", "i8"), ("t_max", "i8"), ("dt_ns", "f8"), ("n_hits", "i8"), ("event_id", "i8")])
        for k in tab.dtype.names:
            tab[k] = ev[k]
        tab = D.gather_rows(tab)
        mem = D.gather_rows(np.asarray(ev["members"], dtype=np.int64).view([("m", "i8")]))["m"]
        merged = D.gather_rows(sh["merged"])
        ncl = D.gather_rows(np.array([len(sh["merged"])], dtype=[("n", "i8")]))["n"]
        ok, why = unchanged, "" if unchanged else "merge_group_sharded's result changed"
        if rank == 0 and ok:
            ok, why = _compare(O, hit_grouped_frame, hit_member_columns, hits, merge_gap, w, tab, mem, merged, ncl, ev["events_per_rank"],
                               frame, name, sh["zone_rows"], zone_rows)
        out.append((name, bool(ok), why))
    q.put((rank, out))
    dist.destroy_process_group()


def _compare(O, hit_grouped_frame, hit_member_columns, hits, merge_gap, w, tab, mem, merged, ncl, events_per_rank, frame, name, k_used,
             k0):
    import pandas as pd

    _, want_m, want_c = O.hit_merge(hits, merge_gap_ns=merge_gap, max_total_width_ns=10000.0)
    want = O.group_hit_windows(want_m, w, component_rows=want_c, component_hits=hits)
    # global position of every rank's merged row: the channel-major assembly is a stable sort of the rank-order rows
    key = merged["board"].astype(np.int64) * 65536 + (merged["channel"].astype(np.int64) + 32768)
    pos = np.empty(len(merged), dtype=np.int64)
    pos[np.argsort(key, kind="stable")] = np.arange(len(merged))
    starts = np.r_[0, np.cumsum(ncl)]
    for r in range(len(ncl)):
        if not np.all(np.diff(pos[starts[r]:starts[r + 1]]) > 0):
            return False, f"rank {r}'s merged rows are not in their global relative order"
    rank_of_row = np.empty(len(merged), dtype=np.int64)
    rank_of_row[pos] = np.repeat(np.arange(len(ncl)), ncl)
    off = want["offsets"]
    owner = rank_of_row[want["members"]]
    if len(off) > 1 and not np.array_equal(np.minimum.reduceat(owner, off[:-1]), np.maximum.reduceat(owner, off[:-1])):
        return False, "an event has members on two ranks"
    # the rank-order concatenation of the tables is the whole-run table
    for k in ("t_min", "t_max", "dt_ns", "n_hits", "event_id"):
        if tab[k].tobytes() != np.asarray(want[k]).tobytes():
            return False, f"table.{k}"
    # every rank's members index its own merged rows: through their global positions they are the whole-run members
    ev_at = np.r_[0, np.cumsum(events_per_rank)]
    mem_at = np.r_[0, np.cumsum(tab["n_hits"])][ev_at]
    glob = np.concatenate([pos[starts[r]:starts[r + 1]][mem[mem_at[r]:mem_at[r + 1]]] for r in range(len(ncl))])
    if not np.array_equal(glob, want["members"]):
        return False, "members"
    want_frame = hit_grouped_frame(want, hit_member_columns(want_m[want["members"]])) if len(want_m) else pd.DataFrame()
    why = _frame_diff(frame, want_frame)
    if why:
        return False, why
    if name == "grow" and not k_used > k0:
        return False, "the zones did not grow"
    if name == "one_event" and len(want["t_min"]) != 1:
        return False, "the run is not one event"
    if name == "ties" and merge_gap == 0:
        a0 = O.hit_abs_windows(want_m, "sample_start", "sample_end")[0]
        keys = np.stack([want_m[f].astype(np.int64) for f in ("board", "channel", "dt", "timestamp", "record_id")] + [a0.view(np.int64)])
        if np.unique(keys, axis=1).shape[1] == len(want_m):
            return False, "no ties"
    return True, ""


def _frame_diff(got, want):
    if list(got.columns) != list(want.columns) or len(got) != len(want) or not got.index.equals(want.index):
        return "frame shape"
    for c in want.columns:
        if got[c].dtype != want[c].dtype:
            return f"frame dtype {c}"
        if want[c].dtype == object:
            if not all(a.dtype == b.dtype and np.array_equal(a, b) for a, b in zip(got[c], want[c])):
                return f"frame.{c}"
        elif not np.array_equal(got[c].to_numpy(), want[c].to_numpy()):
            return f"frame.{c}"
    return ""


@pytest.mark.parametrize("merge_gap", [0.0, 50.0])
@pytest.mark.parametrize("world_size", [2, 3, 4])
def test_hit_events_sharded(world_size, merge_gap):
    import torch.multiprocessing as mp

    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world_size, port, merge_gap, q)) for r in range(world_size)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=600) for _ in procs)
    for p in procs:
        p.join(timeout=60)
    bad = [(r, c) for r, cases in res for c in cases if not c[1]]
    assert not bad, bad
