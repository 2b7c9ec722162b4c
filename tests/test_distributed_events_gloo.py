"""CPU: time-sharded df -> df_events -> df_paired (distributed.df_sharded / events_sharded / gather_event_frames) over
2, 3 and 4 gloo ranks with the host backend (the oracle's df_columns, group_time_window and pair_events), and the cut
plan on its own.  On GPUs the same plan / exchange code runs over NCCL with the device kernels
(tools/dist_check.py --events)."""

import os
import socket
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
W_NS = 100.0  # grouping window
PAIR_NS = 80.0  # df_paired window
NCH, START = 3, 6


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def make_run(case: str, n: int = 3000, seed: int = 0):
    """BASIC_FEATURES rows of a time-sorted run (gaps > W now and then, repeated timestamps, negative channels) and
    the RECORDS rows' record_id; returns (features, record_id)."""
    from waveformanalysis_b200.dtypes import BASIC_FEATURES_DTYPE

    rng = np.random.default_rng(seed)
    step = rng.integers(0, 40_000, n)
    step[rng.random(n) < 0.08] = 250_000  # gaps wider than W
    step[rng.random(n) < 0.1] = 0  # equal timestamps
    if case == "no_gaps":
        step = rng.integers(0, 30, n)  # the whole run within W: one segment
    elif case == "sparse_gaps":
        step = rng.integers(0, 40_000, n)
        step[111::500] = 250_000  # a gap every 500 rows, none next to a shard boundary: zones of 2 rows must grow
    ts = 10**9 + np.cumsum(step).astype(np.int64)
    f = np.zeros(n, dtype=BASIC_FEATURES_DTYPE)
    f["timestamp"] = ts
    f["channel"] = rng.integers(-3, 12, n)
    f["board"] = rng.integers(0, 2, n)
    f["area"] = rng.normal(100, 30, n).astype(np.float32)
    f["height"] = rng.normal(40, 9, n).astype(np.float32)
    f["amp"] = rng.normal(20, 3, n).astype(np.float32)
    f["max_abs_diff"] = rng.normal(5, 1, n).astype(np.float32)
    return f, np.arange(n, dtype=np.int64) * 3 + 7


def shard_sizes(case: str, n: int, P: int):
    if case == "empty_rank":
        b = (np.arange(P) * n) // (P - 1)
        sizes = np.diff(np.r_[b, n]).tolist()
        return sizes[:1] + [0] + sizes[1:-1] + [n - sum(sizes[:-1])] if P > 2 else [n, 0]
    b = (np.arange(P + 1) * n) // P
    return np.diff(b).tolist()


def equal_ts_at_boundaries(f, sizes):
    """Repeat the timestamp across every shard boundary (rows on both sides share it)."""
    f = f.copy()
    edges = np.cumsum(sizes)[:-1]
    for e in edges:
        if 2 <= e <= len(f) - 3:
            f["timestamp"][e - 2:e + 3] = f["timestamp"][e - 2]
    return f


def reference(f, rid):
    """The single-process chain on the whole run: df columns, event table, pair_events."""
    from oracle import np_oracle as O

    df = O.df_columns(f, record_id=rid)
    ev = O.group_time_window(df["timestamp"], df["channel"], W_NS)
    m = ev["members"]
    p = O.pair_events(ev["offsets"], df["timestamp"][m], df["area"][m], df["height"][m], ev["dt_ns"], PAIR_NS, NCH)
    return df, ev, p


# ---- the cut plan on its own ----------------------------------------------------------------------------------------


def _zones(ts, sizes, k):
    from waveformanalysis_b200 import distributed as D

    heads, tails, wholes, b = [], [], [], 0
    for s in sizes:
        z = D._pack_zone(ts[b:b + s], np.zeros(s, np.float32), np.zeros(s, np.float32), np.zeros(s, np.int16))
        kh = min(k, s)
        kt = min(k, s - kh)
        heads.append(z[:kh])
        tails.append(z[s - kt:])
        wholes.append(kh + kt == s)
        b += s
    return heads, tails, wholes


def _plan(ts, sizes, k):
    from waveformanalysis_b200 import distributed as D

    while True:
        heads, tails, wholes = _zones(ts, sizes, k)
        bounds, ok = D.plan_event_cuts(heads, tails, wholes, sizes, W_NS * 1e3)
        if ok:
            return bounds, k
        assert not all(wholes)
        k *= 2


def _check_bounds(ts, sizes, bounds):
    """Owned ranges tile [0, n) in rank order and every non-empty range starts at a segment start."""
    from waveformanalysis_b200 import distributed as D

    n = len(ts)
    starts = set(D.segment_starts(ts, W_NS * 1e3).tolist()) | {0}
    owned = [(int(lo), int(hi)) for lo, hi in bounds if hi > lo]
    assert owned[0][0] == 0 and owned[-1][1] == n
    for (a0, a1), (b0, b1) in zip(owned[:-1], owned[1:]):
        assert a1 == b0
    assert all(lo in starts for lo, _ in owned)
    assert all(lo == hi for (lo, hi), s in zip(bounds, sizes) if s == 0)


@pytest.mark.parametrize("case", ["normal", "empty_rank", "equal_ts", "sparse_gaps", "no_gaps"])
@pytest.mark.parametrize("P", [2, 3, 4, 8])
def test_plan_event_cuts(case, P):
    f, _ = make_run(case, seed=P)
    sizes = shard_sizes(case, len(f), P)
    if case == "equal_ts":
        f = equal_ts_at_boundaries(f, sizes)
    ts = f["timestamp"]
    bounds, k = _plan(ts, sizes, 2 if case in ("sparse_gaps", "no_gaps") else 64)
    _check_bounds(ts, sizes, bounds)
    owners = sum(hi > lo for lo, hi in bounds)
    if case == "no_gaps":
        assert owners == 1 and bounds[0].tolist() == [0, len(ts)]  # boundaries dropped: rank 0 owns the run
    elif case == "sparse_gaps":
        assert k > 2  # the zones grew until they held a gap
    else:
        assert owners == sum(s > 0 for s in sizes)


def test_plan_event_cuts_picks_the_start_nearest_the_boundary():
    from waveformanalysis_b200 import distributed as D

    ts = np.r_[np.arange(6) * 10, 10**6 + np.arange(6) * 10, 2 * 10**6 + np.arange(8) * 10].astype(np.int64)  # segments start at 6, 12
    heads, tails, wholes = _zones(ts, [10, 10], 5)
    bounds, ok = D.plan_event_cuts(heads, tails, wholes, [10, 10], W_NS * 1e3)
    assert ok and bounds.tolist() == [[0, 12], [12, 20]]
    heads, tails, wholes = _zones(ts, [7, 13], 5)
    bounds, ok = D.plan_event_cuts(heads, tails, wholes, [7, 13], W_NS * 1e3)
    assert ok and bounds.tolist() == [[0, 6], [6, 20]]


def test_check_time_order():
    from waveformanalysis_b200 import distributed as D

    D.check_time_order(np.array([[3, 0, 10], [0, 0, 0], [2, 10, 11]]))  # equal timestamps across a boundary: fine
    with pytest.raises(ValueError, match="not in time order"):
        D.check_time_order(np.array([[3, 0, 10], [0, 0, 0], [2, 9, 11]]))


# ---- the whole path over gloo ---------------------------------------------------------------------------------------


def _worker(rank, world_size, port, f, rid, sizes, zone_rows, q):
    sys.path.insert(0, ROOT)
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world_size), LOCAL_RANK=str(rank), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    import torch.distributed as dist

    from oracle import np_oracle as O
    from waveformanalysis_b200 import distributed as D

    dist.init_process_group("gloo", rank=rank, world_size=world_size)
    try:
        lo = int(sum(sizes[:rank]))
        hi = lo + sizes[rank]
        be = D.HostEvents(O.df_columns, O.group_time_window, O.pair_events)
        rec = np.zeros(hi - lo, dtype=[("record_id", "<i8")])
        rec["record_id"] = rid[lo:hi]
        df = D.df_sharded(rec, f[lo:hi], backend=be)
        ev = D.events_sharded(df, time_window_ns=W_NS, pair_window_ns=PAIR_NS, n_channels=NCH, start_channel_slice=START,
                              backend=be, zone_rows=zone_rows)
        frames = D.gather_event_frames(df, ev)
        q.put((rank, "ok", df, {k: v for k, v in ev.items()}, frames if rank == 0 else None))
    except ValueError as e:
        q.put((rank, "ValueError", str(e)))
    finally:
        dist.destroy_process_group()


def _run_ranks(world_size, f, rid, sizes, zone_rows, timeout=240):
    import torch.multiprocessing as mp

    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world_size, port, f, rid, sizes, zone_rows, q)) for r in range(world_size)]
    for p in procs:
        p.start()
    res = sorted((q.get(timeout=timeout) for _ in procs), key=lambda r: r[0])
    for p in procs:
        p.join(timeout=60)
    return res


def _expected_frames(df, ev, p):
    from waveformanalysis_b200.plugins.dataframe import df_frame, paired_frame
    from waveformanalysis_b200.plugins.grouping import events_frame

    m = ev["members"]
    e = events_frame(ev, df["channel"][m], df["area"][m], df["height"][m], df["timestamp"][m])
    return df_frame(df, df["order"], False), e, paired_frame(e, ev["offsets"], p, NCH, START)


@pytest.mark.parametrize("case,zone_rows", [("normal", 4096), ("empty_rank", 64), ("equal_ts", 64), ("sparse_gaps", 2), ("no_gaps", 16)])
@pytest.mark.parametrize("world_size", [2, 3, 4])
def test_sharded_events_equal_the_single_run(case, zone_rows, world_size):
    import pandas as pd

    f, rid = make_run(case, seed=world_size)
    sizes = shard_sizes(case, len(f), world_size)
    if case == "equal_ts":
        f = equal_ts_at_boundaries(f, sizes)
    want_df, want_ev, want_p = reference(f, rid)
    res = _run_ranks(world_size, f, rid, sizes, zone_rows)
    assert all(r[1] == "ok" for r in res), res
    dfs, evs = [r[2] for r in res], [r[3] for r in res]
    for k in ("timestamp", "record_id", "area", "height", "amp", "max_abs_diff", "board", "channel"):
        assert np.concatenate([d["cols"][k] for d in dfs]).tobytes() == want_df[k].tobytes(), k
    assert np.array_equal(np.concatenate([d["index"] for d in dfs]), want_df["order"])
    cat = lambda k: np.concatenate([e[k] for e in evs])  # noqa: E731
    for k in ("t_min", "t_max", "dt_ns", "n_hits", "members", "event_id"):
        want = want_ev[k] if k != "event_id" else np.arange(len(want_ev["t_min"]))
        assert cat(k).tobytes() == np.asarray(want).astype(cat(k).dtype).tobytes(), k
    assert np.array_equal(np.r_[0, np.cumsum(cat("n_hits"))], want_ev["offsets"])
    m = want_ev["members"]
    for k, col in (("member_ts", "timestamp"), ("member_channel", "channel"), ("member_area", "area"), ("member_height", "height")):
        assert cat(k).tobytes() == want_df[col][m].tobytes(), k
    assert np.array_equal(cat("keep"), want_p["keep"]) and np.array_equal(cat("delta_t"), want_p["delta_t"])
    assert np.array_equal(cat("area_ch"), want_p["area_ch"], equal_nan=True)
    assert np.array_equal(cat("height_ch"), want_p["height_ch"], equal_nan=True)
    assert [int(x) for x in evs[0]["events_per_rank"]] == [len(e["t_min"]) for e in evs]
    assert all(e["gathered_bytes"] > 0 for e in evs)
    owners = sum(e["owned"][1] > e["owned"][0] for e in evs)
    if case == "no_gaps":
        assert owners == 1 and evs[0]["zone_rows"] >= len(f) // world_size // 2
    if case == "sparse_gaps":
        assert evs[0]["zone_rows"] > 2
    got = res[0][4]
    want = _expected_frames(want_df, want_ev, want_p)
    pd.testing.assert_frame_equal(got[0], want[0])
    for g, w in zip(got[1:], want[1:]):
        assert list(g.columns) == list(w.columns) and g.index.equals(w.index)
        for c in w.columns:
            assert g[c].dtype == w[c].dtype, c
            if w[c].dtype == object:
                assert all(a.dtype == b.dtype and np.array_equal(a, b) for a, b in zip(g[c], w[c])), c
            else:
                assert np.array_equal(g[c].to_numpy(), w[c].to_numpy(), equal_nan=w[c].dtype.kind == "f"), c


def test_shards_out_of_time_order_raise_on_every_rank():
    f, rid = make_run("normal", seed=9)
    n = len(f)
    half = n // 2
    swapped = np.r_[f[half:], f[:half]]  # rank 0 holds the later half
    res = _run_ranks(2, swapped, np.r_[rid[half:], rid[:half]], [n - half, half], 4096, timeout=120)
    assert [r[1] for r in res] == ["ValueError", "ValueError"], res
    assert all("not in time order" in r[2] for r in res)


def test_single_process_without_a_process_group():
    from oracle import np_oracle as O
    from waveformanalysis_b200 import distributed as D

    f, rid = make_run("normal", seed=3)
    want_df, want_ev, want_p = reference(f, rid)
    be = D.HostEvents(O.df_columns, O.group_time_window, O.pair_events)
    rec = np.zeros(len(f), dtype=[("record_id", "<i8")])
    rec["record_id"] = rid
    df = D.df_sharded(rec, f, backend=be)
    ev = D.events_sharded(df, time_window_ns=W_NS, pair_window_ns=PAIR_NS, n_channels=NCH, start_channel_slice=START, backend=be)
    assert ev["t_min"].tobytes() == want_ev["t_min"].tobytes() and ev["members"].tobytes() == want_ev["members"].tobytes()
    assert ev["gathered_bytes"] == 0 and ev["owned"] == (0, len(f))
