"""Multi-GPU execution of the hot path: one process per GPU (torchrun), time-chunk sharding of the
time-sorted records, and ONE all-gather of the hit grouping columns for cross-channel event
grouping (SURVEY.md 8(e)).

* Records are independent units for baseline / filter / hits / features / widths, so a rank simply
  owns a contiguous slice [lo, hi) of the time-sorted record array - a time shard - and no
  collective is needed on that path (weak or strong scaling with zero data-path communication).
* Event grouping needs every hit's absolute window.  Hits are tiny next to samples (36 B of
  grouping columns per hit against 2*L B of samples per record), so every rank all-gathers the
  columns (counts first, then padded payloads) over NCCL / NVLink and computes the global
  boundary flags and event ids redundantly on its own GPU; the result is identical to the
  single-GPU one because ranks concatenate in record order.  This replaces the halo-and-clip
  scheme of the reference's StreamingPlugin (core/plugins/core/streaming.py:318-324, 592-664)
  with an exact global pass.
"""

from __future__ import annotations

import os

import numpy as np

GROUP_COLUMNS = (("timestamp", np.int64), ("position", np.int64), ("start", np.int32), ("end", np.int32), ("dt", np.int32),
                 ("record_id", np.int64), ("board", np.int16), ("channel", np.int16))


def world():
    """(rank, world_size, local_rank) from the torchrun environment."""
    return int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))


def shard_bounds(n: int, world_size: int) -> np.ndarray:
    """Boundaries of equal-count contiguous shards: rank r owns [b[r], b[r+1])."""
    return (np.arange(world_size + 1, dtype=np.int64) * int(n)) // int(world_size)


def shard_slice(records: np.ndarray, pool: np.ndarray, rank: int, world_size: int):
    """The rank's time shard of a time-sorted run: (records[lo:hi], pool view covering them, lo)."""
    b = shard_bounds(len(records), world_size)
    lo, hi = int(b[rank]), int(b[rank + 1])
    return records[lo:hi], pool, lo


def init_process_group(backend: str | None = None):
    import torch
    import torch.distributed as dist

    rank, ws, local = world()
    if ws == 1 or dist.is_initialized():
        return
    if backend is None:
        backend = "nccl" if torch.cuda.is_available() else "gloo"
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    if backend == "nccl":
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    else:
        dist.init_process_group(backend)


def _device_for_collectives():
    import torch
    import torch.distributed as dist

    return torch.device("cuda", torch.cuda.current_device()) if dist.get_backend() == "nccl" else torch.device("cpu")


def allgather_columns(columns: dict) -> dict:
    """All-gather variable-length 1-D numpy columns (same length on a rank) in rank order.

    The columns are packed into one row-structured byte buffer, so the exchange is one tiny
    all_gather of the per-rank counts plus ONE all_gather of the payload padded to the maximum
    count.  Returns the concatenated columns plus ``counts`` (per-rank lengths)."""
    import torch
    import torch.distributed as dist

    names = list(columns)
    n_local = len(columns[names[0]]) if names else 0
    if not dist.is_available() or not dist.is_initialized() or dist.get_world_size() == 1:
        out = {k: np.asarray(v) for k, v in columns.items()}
        out["counts"] = np.array([n_local], dtype=np.int64)
        return out
    ws = dist.get_world_size()
    dev = _device_for_collectives()
    row_dtype = np.dtype([(k, np.asarray(columns[k]).dtype) for k in names])
    rows = np.zeros(n_local, dtype=row_dtype)
    for k in names:
        rows[k] = columns[k]
    cnt = torch.tensor([n_local], dtype=torch.int64, device=dev)
    counts_t = [torch.zeros(1, dtype=torch.int64, device=dev) for _ in range(ws)]
    dist.all_gather(counts_t, cnt)
    counts = np.array([int(c.item()) for c in counts_t], dtype=np.int64)
    nmax = max(int(counts.max()), 1)
    t = torch.zeros(nmax * row_dtype.itemsize, dtype=torch.uint8, device=dev)
    if n_local:
        t[: n_local * row_dtype.itemsize] = torch.from_numpy(rows.view(np.uint8).reshape(-1)).to(dev)
    parts = [torch.empty_like(t) for _ in range(ws)]
    dist.all_gather(parts, t)
    gathered = np.concatenate([parts[r][: int(counts[r]) * row_dtype.itemsize].cpu().numpy() for r in range(ws)]).view(row_dtype)
    out = {k: np.ascontiguousarray(gathered[k]) for k in names}
    out["counts"] = counts
    return out


def hit_group_columns(hits: np.ndarray) -> dict:
    names = hits.dtype.names
    sn, en = ("sample_start", "sample_end") if "sample_start" in names else ("edge_start", "edge_end")
    return {
        "timestamp": hits["timestamp"].astype(np.int64), "position": hits["position"].astype(np.int64),
        "start": hits[sn].astype(np.int32), "end": hits[en].astype(np.int32), "dt": hits["dt"].astype(np.int32),
        "record_id": hits["record_id"].astype(np.int64), "board": hits["board"].astype(np.int16),
        "channel": hits["channel"].astype(np.int16),
    }


def columns_as_hits(cols: dict) -> np.ndarray:
    """Gathered columns -> a minimal structured array accepted by ops.group_hit_windows."""
    n = len(cols["timestamp"])
    h = np.zeros(n, dtype=[("timestamp", "i8"), ("position", "i8"), ("edge_start", "i4"), ("edge_end", "i4"), ("dt", "i4"),
                           ("record_id", "i8"), ("board", "i2"), ("channel", "i2")])
    h["timestamp"], h["position"] = cols["timestamp"], cols["position"]
    h["edge_start"], h["edge_end"], h["dt"] = cols["start"], cols["end"], cols["dt"]
    h["record_id"], h["board"], h["channel"] = cols["record_id"], cols["board"], cols["channel"]
    return h


def group_hits_distributed(local_hits: np.ndarray, time_window_ns: float, group_fn=None) -> dict:
    """Globally consistent event grouping of per-rank hit rows.

    Every rank gathers all ranks' grouping columns, groups the global set (``group_fn`` defaults to
    the device implementation ``ops.group_hit_windows``) and returns the global event table plus
    ``local_event_of_hit`` (event id of each of its own hits) and ``hit_offset`` (index of its first
    hit in the global order)."""
    if group_fn is None:
        from . import ops

        group_fn = ops.group_hit_windows
    cols = allgather_columns(hit_group_columns(local_hits))
    counts = cols.pop("counts")
    rank = world()[0] if len(counts) > 1 else 0
    ev = group_fn(columns_as_hits(cols), time_window_ns)
    start = int(counts[:rank].sum())
    ev["hit_offset"] = start
    ev["local_event_of_hit"] = ev["event_of_hit"][start : start + int(counts[rank])]
    ev["counts"] = counts
    return ev


def process_shard(records: np.ndarray, pool: np.ndarray, **kw) -> dict:
    """Run the fused pass on this rank's time shard of a time-sorted run.  ``event_index`` and the
    padded matrix width are those of the whole run, so concatenating the ranks' rows in rank order
    reproduces the single-GPU output byte for byte."""
    from . import engine

    rank, ws, _ = world()
    sub, pool, lo = shard_slice(records, pool, rank, ws)
    lmax = int(records["event_length"].max()) if len(records) else 0
    out = engine.process_host(sub, pool, row_base=lo, lmax=lmax, **kw)
    out["row_base"] = lo
    return out


def gather_rows(rows: np.ndarray) -> np.ndarray:
    """Concatenate every rank's structured rows in rank order (all ranks get the result)."""
    import torch
    import torch.distributed as dist

    if not dist.is_available() or not dist.is_initialized() or dist.get_world_size() == 1:
        return rows
    ws = dist.get_world_size()
    dev = _device_for_collectives()
    item = rows.dtype.itemsize
    cnt = torch.tensor([len(rows)], dtype=torch.int64, device=dev)
    counts_t = [torch.zeros(1, dtype=torch.int64, device=dev) for _ in range(ws)]
    dist.all_gather(counts_t, cnt)
    counts = [int(c.item()) for c in counts_t]
    nmax = max(max(counts), 1)
    t = torch.zeros(nmax * item, dtype=torch.uint8, device=dev)
    if len(rows):
        t[: len(rows) * item] = torch.from_numpy(np.ascontiguousarray(rows).view(np.uint8).reshape(-1)).to(dev)
    parts = [torch.empty_like(t) for _ in range(ws)]
    dist.all_gather(parts, t)
    return np.concatenate([parts[r][: counts[r] * item].cpu().numpy() for r in range(ws)]).view(rows.dtype)


# ------------------------------------------------------------------------------------------------
# Time-sharded hit_merge -> hit_grouped that SCALES: boundary zones instead of a global gather
# ------------------------------------------------------------------------------------------------
# Every rank holds the hit rows of its time shard (record order).  Event grouping and same-channel hit merging only
# couple hits that are closer than G = max(time_window_ns, merge_gap_ns).  So the ranks agree on CUT TIMES that lie in
# gaps of the global hit stream wider than G, one per shard boundary; a rank then owns the hits whose window starts
# between its two cuts, and no merge chain or event crosses a cut: hit_merge and the grouping run locally on the
# device, and only two counts per rank are exchanged to number clusters and events globally.
#
# What travels: the first and the last K hit rows of every rank (the BOUNDARY ZONES, K = 4096 rows by default, 60 B
# each) in ONE all_gather, plus one all_gather of 16 bytes per rank - O(ranks * K), independent of the run length.
# The zones serve two purposes: every rank derives the same cut for every boundary from them, and a rank imports the
# neighbour's zone rows that fall on its side of the cut (this is the halo of core/plugins/core/streaming.py:318-324,
# 611-632, with the clip to the main range of :380-445 replaced by exact ownership).
#
# Soundness of a cut C at the boundary between ranks r and r + 1 (rows are in record order, records in time order):
#   * rows of r that are NOT in its tail zone belong to records that start no later than the record of the first
#     tail-zone row, so their windows end before lo = that record's start + the longest record span; C > lo + G.
#   * rows of r + 1 that are NOT in its head zone belong to records that start no earlier than the record of the last
#     head-zone row: their windows start at or after hi = that record's start; C <= hi.
#   * C is the window start of a zone row with every earlier zone window ending more than G before it.
# If no such cut exists the zones are doubled; zones that cover whole shards always work (then the exchange is the
# old global gather).


def _rows_windows(rows: np.ndarray):
    """abs_start / abs_end (event_grouping.py:365-367) and the start of the record of packed hit rows, on the host."""
    sn, en = ("sample_start", "sample_end") if "sample_start" in rows.dtype.names else ("edge_start", "edge_end")
    dt_ps = rows["dt"].astype(np.float64) * 1e3
    ts, pos = rows["timestamp"].astype(np.float64), rows["position"].astype(np.float64)
    a0 = ts + (rows[sn].astype(np.float64) - pos) * dt_ps
    a1 = ts + (rows[en].astype(np.float64) - pos) * dt_ps
    return a0, a1, ts - pos * dt_ps


def plan_cuts(heads: list, tails: list, whole: list, gap_ps: float, span_ps: float):
    """Cut times for the boundaries between consecutive NON-EMPTY ranks.  heads[r] / tails[r]: the first / last zone
    rows of rank r (numpy, packed hit rows, disjoint), whole[r]: the two zones are the whole shard.  Returns (cuts, ok):
    cuts[r] is the cut between rank r and the next non-empty rank (None for empty ranks and the last one); ok is False
    when some boundary has no admissible gap inside the zones (the caller grows the zones)."""
    R = len(heads)
    cuts: list = [None] * R
    live = [r for r in range(R) if len(heads[r]) or len(tails[r])]
    for a, b in zip(live[:-1], live[1:]):
        end_a = np.concatenate([heads[a], tails[a]]) if whole[a] else tails[a]
        start_b = np.concatenate([heads[b], tails[b]]) if whole[b] else heads[b]
        ta0, ta1, trec = _rows_windows(end_a)
        ha0, ha1, hrec = _rows_windows(start_b)
        lo = -np.inf if whole[a] else float(trec[0]) + span_ps + gap_ps
        hi = np.inf if whole[b] else float(hrec[-1])
        s0 = np.concatenate([ta0, ha0])
        s1 = np.concatenate([ta1, ha1])
        o = np.argsort(s0, kind="stable")
        s0, s1 = s0[o], s1[o]
        reach = np.maximum.accumulate(s1)
        ok_i = np.flatnonzero((s0[1:] > reach[:-1] + gap_ps) & (s0[1:] > lo) & (s0[1:] <= hi)) + 1
        if len(ok_i) == 0:
            return cuts, False
        # the admissible gap nearest to the nominal boundary (the first window of the next shard)
        nominal = float(ha0.min())
        cuts[a] = float(s0[ok_i[np.argmin(np.abs(s0[ok_i] - nominal))]])
    return cuts, True


def _allgather_zones(head: np.ndarray, tail: np.ndarray, k: int, whole: bool, n_local: int):
    """ONE all_gather of every rank's zones (2k rows, padded) with a 4 x int64 header (rows in head, rows in tail, zone
    covers the shard, local row count).  Returns per-rank lists."""
    import torch
    import torch.distributed as dist

    item = head.dtype.itemsize
    if not dist.is_available() or not dist.is_initialized() or dist.get_world_size() == 1:
        return [head], [tail], [whole], [n_local], 0
    ws = dist.get_world_size()
    dev = _device_for_collectives()
    buf = np.zeros(32 + 2 * k * item, dtype=np.uint8)
    buf[:32].view(np.int64)[:] = (len(head), len(tail), int(whole), n_local)
    buf[32:32 + len(head) * item] = head.view(np.uint8).reshape(-1)
    buf[32 + k * item:32 + k * item + len(tail) * item] = tail.view(np.uint8).reshape(-1)
    t = torch.from_numpy(buf).to(dev)
    parts = [torch.empty_like(t) for _ in range(ws)]
    dist.all_gather(parts, t)
    heads, tails, wholes, counts = [], [], [], []
    for p in parts:
        b = p.cpu().numpy()
        nh, nt, w, nl = (int(x) for x in b[:32].view(np.int64))
        heads.append(b[32:32 + nh * item].view(head.dtype).copy())
        tails.append(b[32 + k * item:32 + k * item + nt * item].view(head.dtype).copy())
        wholes.append(bool(w))
        counts.append(nl)
    return heads, tails, wholes, counts, int(t.numel()) * ws


def _allgather_i64(vals) -> np.ndarray:
    import torch
    import torch.distributed as dist

    v = np.asarray(vals, dtype=np.int64)
    if not dist.is_available() or not dist.is_initialized() or dist.get_world_size() == 1:
        return v[None, :]
    dev = _device_for_collectives()
    t = torch.from_numpy(v).to(dev)
    parts = [torch.empty_like(t) for _ in range(dist.get_world_size())]
    dist.all_gather(parts, t)
    return np.stack([p.cpu().numpy() for p in parts])


class HostRows:
    """Backend for hit rows held as numpy arrays (CPU tests: the compute is the oracle's)."""

    def __init__(self, merge_fn, group_fn):
        self.merge_fn, self.group_fn = merge_fn, group_fn

    def count(self, rows):
        return len(rows)

    def head_tail(self, rows, k):
        n = len(rows)
        kh = min(k, n)
        kt = min(k, n - kh)
        return rows[:kh].copy(), rows[n - kt:].copy()

    def assemble(self, rows, k_head, k_tail, first: np.ndarray, last: np.ndarray):
        return np.concatenate([first, rows[k_head:len(rows) - k_tail], last])

    def merge_and_group(self, owned, merge_gap_ns, max_total_width_ns, time_window_ns):
        clusters, merged, comps = self.merge_fn(owned, merge_gap_ns=merge_gap_ns, max_total_width_ns=max_total_width_ns)
        ev = self.group_fn(merged, time_window_ns, component_rows=comps, component_hits=owned)
        return dict(merged=merged, event_of_merged=np.asarray(ev["event_of_hit"], dtype=np.int64), n_events=len(ev["t_min"]),
                    n_clusters=len(merged), grouping=ev)

    def hit_events(self, sh):
        ev = sh["grouping"]
        m = np.asarray(ev["members"], dtype=np.int64)
        res = {k: np.asarray(ev[k]) for k in ("t_min", "t_max", "dt_ns", "n_hits", "offsets")}
        res.update(members=m, member_rows=sh["merged"][m])
        return res

    def iota(self, n, base):
        return np.arange(n, dtype=np.int64) + base


class DeviceRows:
    """Backend for hit rows that stay on the device (uint8 tensor of packed 60-byte rows + row count)."""

    def __init__(self, dtype):
        self.dtype = dtype

    def count(self, rows):
        return int(rows[1])

    def head_tail(self, rows, k):
        t, n = rows
        item = self.dtype.itemsize
        kh = min(k, n)
        kt = min(k, n - kh)
        head = t[: kh * item].cpu().numpy().view(self.dtype)
        tail = t[(n - kt) * item: n * item].cpu().numpy().view(self.dtype)
        return head, tail

    def assemble(self, rows, k_head, k_tail, first: np.ndarray, last: np.ndarray):
        import torch

        from .engine import upload

        t, n = rows
        item = self.dtype.itemsize
        parts = []
        if len(first):
            parts.append(upload(first))
        parts.append(t[k_head * item:(n - k_tail) * item])
        if len(last):
            parts.append(upload(last))
        out = torch.cat(parts) if len(parts) > 1 else parts[0]
        return out, len(first) + (n - k_head - k_tail) + len(last)

    def merge_and_group(self, owned, merge_gap_ns, max_total_width_ns, time_window_ns):
        from . import ops

        t, n = owned
        m = ops.hit_merge_device(t, n, merge_gap_ns=merge_gap_ns, max_total_width_ns=max_total_width_ns)
        g = ops.group_rows_device(m["merged"], m["n_clusters"], 72, time_window_ns, abs_start=m["abs_start"], abs_end=m["abs_end"])
        return dict(merged=m["merged"], event_of_merged=g["event_of_row"], n_events=g["n_events"], n_clusters=m["n_clusters"], detail=m,
                    grouping=g)

    def hit_events(self, sh):
        from . import ops

        return ops.hit_event_table_device(sh["merged"], sh["n_clusters"], 72, sh["grouping"])

    def iota(self, n, base):
        import torch

        return torch.arange(n, dtype=torch.int64, device="cuda") + base


def merge_group_sharded(rows, backend, *, time_window_ns: float, merge_gap_ns: float = 0.0, max_total_width_ns: float = 10000.0,
                        span_ns: float, zone_rows: int = 4096) -> dict:
    """hit_merge -> hit_grouped of a time-sharded run without gathering the hits.

    ``rows``: this rank's packed hit_threshold rows in record order (a numpy array with ``HostRows``, a
    (uint8 device tensor, count) pair with ``DeviceRows``); ``span_ns``: the longest record of the run in ns.
    Returns the rank's ``merged`` rows (clusters whose window starts between the rank's cuts, in the reference's
    channel-major order), ``event_of_merged`` with GLOBAL event ids, ``cluster_base`` / ``event_base`` (the rank's
    offsets in the global numbering), the counts of every rank, the cuts, and ``gathered_bytes`` (what this rank
    received in the collectives)."""
    rank, ws, _ = world()
    gap_ps = max(float(time_window_ns), float(merge_gap_ns), 0.0) * 1e3
    n = backend.count(rows)
    k = max(int(zone_rows), 1)
    gathered = 0
    while True:
        head, tail = backend.head_tail(rows, k)
        whole = len(head) + len(tail) == n
        heads, tails, wholes, counts, nbytes = _allgather_zones(head, tail, k, whole, n)
        gathered += nbytes
        cuts, ok = plan_cuts(heads, tails, wholes, gap_ps, float(span_ns) * 1e3)
        if ok or all(wholes):
            break
        k *= 2
    if not ok:
        raise RuntimeError("no gap wider than the grouping window between two time shards: the run cannot be cut here")
    R = len(heads)
    me = rank if R > 1 else 0
    owned = owned_hit_rows(backend, rows, me, heads, tails, counts, cuts)
    res = backend.merge_and_group(owned, merge_gap_ns, max_total_width_ns, time_window_ns)
    table = _allgather_i64([res["n_clusters"], res["n_events"]])
    gathered += table.nbytes
    res["cluster_base"] = int(table[:rank, 0].sum())
    res["event_base"] = int(table[:rank, 1].sum())
    res["event_of_merged"] = res["event_of_merged"][: res["n_clusters"]] + res["event_base"]
    res["clusters_per_rank"], res["events_per_rank"] = table[:, 0].copy(), table[:, 1].copy()
    res["cuts"], res["gathered_bytes"], res["zone_rows"], res["owned"] = cuts, gathered, k, owned
    return res


def owned_hit_rows(backend, rows, me: int, heads, tails, counts, cuts):
    """The hit rows rank ``me`` owns in merge_group_sharded, given every rank's zones, row counts and the cuts: lower
    ranks' zone rows, the rank's own rows and upper ranks' zone rows whose window starts between its two cuts, in global
    record order (``rows``: the rank's rows as the backend holds them)."""
    R, n = len(heads), int(counts[me])
    head, tail = heads[me], tails[me]
    live = [r for r in range(R) if counts[r] > 0]
    lo_cut, hi_cut = -np.inf, np.inf
    if me in live:
        i = live.index(me)
        lo_cut = cuts[live[i - 1]] if i > 0 else -np.inf
        hi_cut = cuts[me] if i + 1 < len(live) else np.inf
    elif live:  # an empty shard owns nothing
        lo_cut = hi_cut = np.inf

    def inside(r):
        a0 = _rows_windows(r)[0]
        return r[(a0 >= lo_cut) & (a0 < hi_cut)]

    # rows of other ranks' zones that start between my cuts (in global record order: lower ranks first), my own zone rows
    # that do; rows outside the zones never change owner
    lower = [inside(z) for q in range(me) for z in (heads[q], tails[q])]
    upper = [inside(z) for q in range(me + 1, R) for z in (heads[q], tails[q])]
    first = np.concatenate(lower + [inside(head)]) if n or lower else head[:0]
    last = np.concatenate([inside(tail)] + upper) if n or upper else head[:0]
    return backend.assemble(rows, len(head), len(tail), first, last)


def hit_events_sharded(sh: dict, backend) -> dict:
    """hit_grouped's event table of a time-sharded run: every rank tabulates the events it owns after
    ``merge_group_sharded`` (``sh``, left unchanged) with the same ``backend`` - ``wfb_hit_event_table`` on its device with
    ``DeviceRows``, the grouping function's own table with ``HostRows``.  No collective: every event lies on one rank, and
    ``sh["event_base"]`` (already gathered) numbers them globally.

    Returns ``event_id`` (global), ``t_min``, ``t_max``, ``dt_ns``, ``n_hits``, the CSR ``offsets``, ``members`` (indices
    into the rank's ``sh["merged"]`` rows), ``member_rows`` (those rows in member order: HIT_MERGED rows, packed on the
    device with ``DeviceRows``), ``n_events``, ``event_base`` and ``events_per_rank``.  Concatenated in rank order, the
    tables equal the single-GPU table of the whole run: a rank's merged rows keep their global relative order, so ties
    resolve alike."""
    res = dict(backend.hit_events(sh))
    n_ev, base = int(sh["n_events"]), int(sh["event_base"])
    res.update(event_id=backend.iota(n_ev, base), n_events=n_ev, event_base=base, events_per_rank=np.asarray(sh["events_per_rank"]).copy())
    return res


def gather_hit_grouped_frame(ev_sh: dict):
    """The hit_grouped DataFrame of the WHOLE run on every rank (``hit_events_sharded``'s result), equal to what
    B200HitGroupedPlugin returns for the run.  Every rank receives every event and member row, so this holds the whole
    run in each process (like ``gather_rows``): it is for checks and small runs."""
    import pandas as pd

    from .dtypes import HIT_MERGED_DTYPE
    from .plugins.grouping import HIT_GROUPED_COLUMNS, hit_grouped_frame, hit_member_columns

    n_ev = int(ev_sh["n_events"])
    ev_rows = np.zeros(n_ev, dtype=[("event_id", "<i8"), ("t_min", "<i8"), ("t_max", "<i8"), ("dt_ns", "<f8"), ("n_hits", "<i8")])
    for k in ev_rows.dtype.names:
        ev_rows[k] = _host(ev_sh[k])
    ev_rows = gather_rows(ev_rows)
    m = len(_host(ev_sh["members"]))
    mem = np.ascontiguousarray(_host(ev_sh["member_rows"])).view(np.uint8).reshape(-1)[: m * HIT_MERGED_DTYPE.itemsize]
    mem = gather_rows(mem.view(HIT_MERGED_DTYPE))
    if len(ev_rows) == 0:
        return pd.DataFrame(columns=HIT_GROUPED_COLUMNS)
    table = {k: np.ascontiguousarray(ev_rows[k]) for k in ("event_id", "t_min", "t_max", "dt_ns", "n_hits")}
    table["offsets"] = np.r_[0, np.cumsum(ev_rows["n_hits"])].astype(np.int64)
    return hit_grouped_frame(table, hit_member_columns(mem))


def assemble_merged(merged_all: np.ndarray, event_of_merged_all: np.ndarray):
    """Rank-order concatenation of the ranks' hit_merged rows -> the single-process order: the reference orders the
    merged rows by (board, channel) first and by window start inside a channel (hit_merge.py:125-140), and the ranks'
    pieces of one channel follow each other in time, so a STABLE sort by (board, channel) is all it takes."""
    key = merged_all["board"].astype(np.int64) * 65536 + (merged_all["channel"].astype(np.int64) + 32768)
    o = np.argsort(key, kind="stable")
    return merged_all[o], np.asarray(event_of_merged_all)[o]


# ------------------------------------------------------------------------------------------------
# Time shards built straight from V1725 files: per-rank build, sample-sort exchange, merge
# ------------------------------------------------------------------------------------------------
# The single-GPU order of a V1725 run is lexsort((seq, channel, board, pid = 0, timestamp)) over all files, seq = the
# waveform's index in the concatenation of all files in list order.  The key (timestamp, board, channel, seq) is
# unique, so the order is exact whichever rank reads which file:
#   1. every rank scans and builds only its own files, each row's record_id holding the global seq (the ranks learn
#      the per-file waveform counts from one all-gather);
#   2. every rank samples s = 256 x world_size keys of its sorted rows; all ranks pick the same world_size - 1
#      splitters at the weighted quantiles of the gathered samples (plan_splitters);
#   3. a lower-bound search cuts the local rows at the splitters: each destination's part is one contiguous row range
#      and one contiguous sample range (the local wave_offsets are a running sum);
#   4. all_to_all_single of the counts, then of the rows (102 B each) and of the samples (2 B each);
#   5. one all-gather of the received counts gives the shard's global record and sample bases;
#   6. the received runs (sorted, in source-rank order) are merged by rank and renumbered for the shard's place.
# Every rank sends (P - 1) / P of its rows and samples on average: (P - 1) / P x (2 L + 102) bytes per record.
#
# Raw rows (build_records_sharded: VX2730 CSV groups, anything a format_reader parses, raw_arrays) take the same
# steps 2-6.  Their single-GPU order is the same lexsort over the groups concatenated in group-index order, and both
# single-GPU builders break ties by input position, so seq = a row's index in that concatenation gives the same key.

SPLITTER_SAMPLES_PER_RANK = 256  # s = SPLITTER_SAMPLES_PER_RANK x world_size samples per rank


def key_order(keys: np.ndarray, tie: np.ndarray | None = None) -> np.ndarray:
    """The host restatement of the records order: indices that sort ``keys`` (int64 rows of timestamp, board, channel,
    seq) ascending; ``tie`` (optional) breaks ties between equal keys, then the input order (stable)."""
    k = np.asarray(keys, dtype=np.int64).reshape(-1, 4)
    cols = (k[:, 3], k[:, 2], k[:, 1], k[:, 0])
    return np.lexsort(((tie,) if tie is not None else ()) + cols)


def record_keys(rec: np.ndarray) -> np.ndarray:
    """(n, 4) int64 keys of RECORDS rows whose record_id holds seq."""
    return np.stack([rec["timestamp"].astype(np.int64), rec["board"].astype(np.int64), rec["channel"].astype(np.int64),
                     rec["record_id"].astype(np.int64)], axis=1).reshape(-1, 4)


def lower_bounds(sorted_keys: np.ndarray, queries: np.ndarray) -> np.ndarray:
    """For every key of ``queries`` (ascending) the number of ``sorted_keys`` that are smaller."""
    q = np.asarray(queries, dtype=np.int64).reshape(-1, 4)
    both = np.concatenate([q, np.asarray(sorted_keys, dtype=np.int64).reshape(-1, 4)])
    o = key_order(both, tie=np.r_[np.zeros(len(q), np.int8), np.ones(len(both) - len(q), np.int8)])
    place = np.empty(len(both), dtype=np.int64)
    place[o] = np.arange(len(both))
    return place[: len(q)] - np.arange(len(q))


def splitter_samples(n: int, s: int):
    """Positions of the (at most ``s``) sampled rows of ``n`` sorted rows and their weights: sample i stands for the
    rows from its position up to the next sample's."""
    k = min(int(n), int(s))
    pos = (np.arange(k + 1, dtype=np.int64) * int(n)) // max(k, 1)
    return pos[:k], np.diff(pos)


def plan_splitters(keys: np.ndarray, weights: np.ndarray, n_shards: int) -> np.ndarray:
    """The ``n_shards - 1`` splitters (int64 rows of timestamp, board, channel, seq) that cut the run into shards of
    about equal counts, from the samples of every rank (``keys`` with their ``weights``, any order): splitter j is the
    first sample (in key order) with at least j / n_shards of the total weight before it; past the last sample it is
    a key above every record.  Every rank passes the same gathered samples and gets the same splitters."""
    k = np.asarray(keys, dtype=np.int64).reshape(-1, 4)
    w = np.asarray(weights, dtype=np.int64)
    o = key_order(k)
    k, w = k[o], w[o]
    before = (np.cumsum(w) - w) * int(n_shards)
    total = int(w.sum())
    out = np.full((max(int(n_shards) - 1, 0), 4), np.iinfo(np.int64).max, dtype=np.int64)
    for j in range(1, int(n_shards)):
        m = int(np.searchsorted(before, j * total, side="left"))
        if m < len(k):
            out[j - 1] = k[m]
    return out


def default_file_owners(sizes, world_size: int) -> np.ndarray:
    """Owner rank of every file: contiguous blocks of the list balanced by size (a file goes to the rank whose equal
    share of the total bytes holds the file's middle byte)."""
    sz = np.asarray(sizes, dtype=np.float64)
    P = int(world_size)
    if len(sz) == 0:
        return np.zeros(0, dtype=np.int64)
    total = float(sz.sum())
    if total <= 0:
        return (np.arange(len(sz), dtype=np.int64) * P) // len(sz)
    mid = np.cumsum(sz) - sz / 2
    return np.minimum((mid * P / total).astype(np.int64), P - 1)


def _dist():
    import torch.distributed as dist

    if dist.is_available() and dist.is_initialized():
        return dist, dist.get_rank(), dist.get_world_size()
    return None, 0, 1


def _allreduce_max(v: int) -> int:
    import torch

    dist, _, ws = _dist()
    if ws == 1:
        return int(v)
    t = torch.tensor([int(v)], dtype=torch.int64, device=_device_for_collectives())
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return int(t.item())


def _exchange(rows, pool, row_counts, sample_counts, backend):
    """all_to_all_single of the per-destination counts, then of the row bytes and the sample bytes (uneven splits).
    Returns the received (rows, pool) byte tensors and the per-source (rows, samples) counts."""
    import torch

    dist, _, P = _dist()
    if P == 1:
        return rows, pool, np.stack([row_counts, sample_counts], axis=1)
    dev = _device_for_collectives()
    c = torch.from_numpy(np.stack([row_counts, sample_counts], axis=1).reshape(-1).astype(np.int64)).to(dev)
    rc = torch.empty_like(c)
    dist.all_to_all_single(rc, c)
    recv = rc.cpu().numpy().reshape(P, 2)
    out_rows = backend.empty_bytes(int(recv[:, 0].sum()) * 102)
    dist.all_to_all_single(out_rows, rows, output_split_sizes=(recv[:, 0] * 102).tolist(), input_split_sizes=(row_counts * 102).tolist())
    out_pool = backend.empty_bytes(int(recv[:, 1].sum()) * 2)
    dist.all_to_all_single(out_pool, pool, output_split_sizes=(recv[:, 1] * 2).tolist(), input_split_sizes=(sample_counts * 2).tolist())
    return out_rows, out_pool, recv


class HostRecords:
    """Backend for the records of a rank held as numpy arrays (CPU tests over gloo): the oracle's scan (V1725 files)
    and baseline mean (raw rows), the host key order for the local sort and the merge."""

    def __init__(self, scan_fn=None, baseline_fn=None):
        self.scan_fn = scan_fn
        self.baseline_fn = baseline_fn

    def sync(self):
        pass

    def scan(self, blob):
        s = dict(self.scan_fn(blob))
        s["bytes"] = blob
        return s

    def upload(self, scans, names):
        return scans, names

    def build(self, up, dt_ns: int, seq: np.ndarray):
        from . import ops
        from .dtypes import RECORDS_DTYPE

        scans, names = up
        n = len(seq)
        rec = np.zeros(n, dtype=RECORDS_DTYPE)
        if n == 0:
            return rec, np.zeros(0, dtype=np.uint16)
        cat = {k: np.concatenate([s[k] for s in scans]) for k in ("payload_offset", "n_samples", "channel", "timestamp", "baseline", "trunc")}
        board = np.concatenate([np.full(len(s["channel"]), ops.v1725_board_from_name(nm), dtype=np.int16) for s, nm in zip(scans, names)])
        waves = [np.frombuffer(s["bytes"], dtype=np.uint8)[o:o + 2 * m].view(np.uint16)
                 for s in scans for o, m in zip(s["payload_offset"].tolist(), s["n_samples"].tolist())]
        ts = cat["timestamp"] * np.int64(int(dt_ns) * 1000)
        order = key_order(np.stack([ts, board.astype(np.int64), cat["channel"].astype(np.int64), seq], axis=1))
        rec["timestamp"], rec["board"], rec["channel"] = ts[order], board[order], cat["channel"][order]
        rec["baseline"] = cat["baseline"][order].astype(np.float64)
        rec["baseline_upstream"] = np.nan
        rec["polarity"] = "unknown"
        rec["record_id"] = seq[order]
        rec["dt"] = int(dt_ns)
        rec["flags"] = cat["trunc"][order]
        lens = cat["n_samples"][order].astype(np.int64)
        rec["event_length"] = lens
        rec["wave_offset"] = np.cumsum(lens) - lens
        rec["time"] = rec["timestamp"] // 1000
        return rec, np.concatenate([waves[i] for i in order.tolist()]).astype(np.uint16, copy=False)

    def upload_raw(self, ts, board, channel, blocks):
        return ts, board, channel, blocks

    def build_raw(self, up, dt_ns: int, baseline_window, epoch_ns, seq: np.ndarray):
        """The oracle's build_records over raw rows of any widths, ordered by (timestamp, board, channel, seq)."""
        from .dtypes import RECORDS_DTYPE

        ts, board, channel, blocks = up
        n = len(seq)
        rec = np.zeros(n, dtype=RECORDS_DTYPE)
        if n == 0:
            return rec, np.zeros(0, dtype=np.uint16)
        lens = np.concatenate([np.full(len(b), b.shape[1], dtype=np.int64) for b in blocks])
        baseline = np.concatenate([self.baseline_fn(b.view(np.int16), *baseline_window) for b in blocks])
        samples = np.concatenate([b.reshape(-1).view(np.uint16) for b in blocks])
        order = key_order(np.stack([ts, board.astype(np.int64), channel.astype(np.int64), seq], axis=1))
        rec["timestamp"], rec["board"], rec["channel"] = ts[order], board[order], channel[order]
        rec["baseline"] = baseline[order]
        rec["baseline_upstream"] = np.nan
        rec["polarity"] = "unknown"
        rec["record_id"] = seq[order]
        rec["dt"] = int(dt_ns)
        out_lens = lens[order]
        out_start = np.cumsum(out_lens) - out_lens
        rec["event_length"] = out_lens
        rec["wave_offset"] = out_start
        rec["time"] = rec["timestamp"] // 1000 + (0 if epoch_ns is None else int(epoch_ns))
        in_start = (np.cumsum(lens) - lens)[order]
        return rec, samples[np.arange(int(out_lens.sum()), dtype=np.int64) + np.repeat(in_start - out_start, out_lens)]

    def count(self, local):
        return len(local[0])

    def n_samples(self, local):
        return len(local[1])

    def rows_at(self, local, idx):
        return local[0][np.asarray(idx, dtype=np.int64)]

    def split_points(self, local, splitters):
        return lower_bounds(record_keys(local[0]), splitters)

    def send_buffers(self, local):
        import torch

        return (torch.from_numpy(np.ascontiguousarray(local[0]).view(np.uint8).reshape(-1)),
                torch.from_numpy(np.ascontiguousarray(local[1]).view(np.uint8).reshape(-1)))

    def empty_bytes(self, nbytes: int):
        import torch

        return torch.empty(int(nbytes), dtype=torch.uint8)

    def merge(self, rows, pool, run_offsets, record_base: int, pool_base: int):
        from .dtypes import RECORDS_DTYPE

        rec = rows.numpy().view(RECORDS_DTYPE)
        samples = pool.numpy().view(np.uint16)
        keys = record_keys(rec)
        for a, b in zip(run_offsets[:-1], run_offsets[1:]):
            k = keys[a:b]
            if not (np.array_equal(key_order(k), np.arange(len(k))) and not np.any(np.all(k[1:] == k[:-1], axis=1))):
                raise ValueError("wfb_merge_record_runs: a run is not strictly increasing in (timestamp, board, channel, record_id)")
        order = key_order(keys)
        lens = rec["event_length"].astype(np.int64)
        out = rec[order].copy()
        out_lens = lens[order]
        out_start = np.cumsum(out_lens) - out_lens
        out["record_id"] = int(record_base) + np.arange(len(out), dtype=np.int64)
        out["wave_offset"] = int(pool_base) + out_start
        in_start = (np.cumsum(lens) - lens)[order]
        idx = np.arange(int(out_lens.sum()), dtype=np.int64) + np.repeat(in_start - out_start, out_lens)
        return out, samples[idx]

    def lmax(self, shard):
        return int(shard[0]["event_length"].max()) if len(shard[0]) else 0

    def run(self, shard, lmax: int, record_base: int, pool_base: int):
        from types import SimpleNamespace

        return SimpleNamespace(records=shard[0], pool=shard[1], n=len(shard[0]), lmax=lmax, pool_base=pool_base, row_base=record_base)

    def apply_polarity(self, run, polarity):
        """The numpy assignment of plugins.records._apply_polarity."""
        from .ops import polarity_entries

        rec = run.records
        for b, c, v in polarity_entries(polarity):
            if v != "unknown":
                rec["polarity"][(rec["board"] == b) & (rec["channel"] == c)] = v


class DeviceRecords:
    """Backend for the records of a rank on its GPU: libwfb200's scan, build (with seq), split points and merge."""

    def sync(self):
        import torch

        torch.cuda.synchronize()

    def scan(self, blob):
        from . import ops

        return ops.v1725_scan(blob)

    def upload(self, scans, names):
        from . import ops

        return ops.v1725_upload(scans, names)

    def build(self, up, dt_ns: int, seq: np.ndarray):
        from . import ops

        rows, pool, _ = ops.build_records_v1725_device(up, dt_ns, seq=seq)
        return rows, pool, up["n"]

    def upload_raw(self, ts, board, channel, blocks):
        from . import ops

        return ops.raw_upload(ts, board, channel, blocks)

    def build_raw(self, up, dt_ns: int, baseline_window, epoch_ns, seq: np.ndarray):
        from . import ops

        rows, pool, _ = ops.build_records_ragged_device(up, dt_ns=dt_ns, baseline_window=baseline_window, epoch_ns=epoch_ns, seq=seq)
        return rows, pool, up["n"]

    def count(self, local):
        return local[2]

    def n_samples(self, local):
        return int(local[1].numel())

    def rows_at(self, local, idx):
        import torch

        from .dtypes import RECORDS_DTYPE

        rows, _, n = local
        i = torch.as_tensor(np.asarray(idx, dtype=np.int64), device=rows.device)
        return rows[: n * 102].view(n, 102).index_select(0, i).cpu().numpy().reshape(-1).view(RECORDS_DTYPE)

    def split_points(self, local, splitters):
        from . import ops

        return ops.record_split_points(local[0], local[2], splitters)

    def send_buffers(self, local):
        import torch

        rows, pool, n = local
        return rows[: n * 102], pool.view(torch.uint8)

    def empty_bytes(self, nbytes: int):
        import torch

        return torch.empty(int(nbytes), dtype=torch.uint8, device="cuda")

    def merge(self, rows, pool, run_offsets, record_base: int, pool_base: int):
        import torch

        from . import ops

        rows_o, pool_o, meta = ops.merge_record_runs(rows, pool.view(torch.int16), run_offsets, record_base=record_base, pool_base=pool_base)
        return rows_o, pool_o, meta, int(run_offsets[-1])

    def lmax(self, shard):
        import ctypes as C

        import torch

        from . import _lib
        from .engine import _ptr, _stream

        stats = np.zeros(3, dtype=np.int32)
        scratch = torch.empty(4, dtype=torch.int32, device="cuda")
        _lib.check(_lib.load().wfb_meta_stats(_ptr(shard[2]), shard[3], _ptr(scratch), C.c_void_p(stats.ctypes.data), _stream()),
                   "wfb_meta_stats")
        return max(int(stats[0]), 0)

    def run(self, shard, lmax: int, record_base: int, pool_base: int):
        from .engine import DeviceRun

        rows, pool, meta, n = shard
        return DeviceRun(meta, pool, n, 0, lmax, records_rows=rows, pool_base=pool_base, row_base=record_base)

    def apply_polarity(self, run, polarity):
        from . import ops

        ops.apply_polarity(run, polarity)


def build_records_sharded_v1725(paths, *, dt_ns: int, mine=None, backend=None, polarity: dict | None = None) -> dict:
    """This rank's time shard of the V1725 run made of ``paths`` (the full ordered file list, the same on every rank;
    file names give the board id), without any process holding the whole run.

    ``mine``: the indices of the files this rank reads (node-local disks); by default every rank reads a contiguous
    block of the list balanced by file size, which needs every file's size on every rank.  A file claimed by no rank
    or by two ranks raises ValueError on every rank; a file that cannot be read raises on every rank too.

    Returns ``run`` (an ``engine.DeviceRun`` of rows [record_base, record_base + n) of the single-GPU build with its
    pool slice, the run-wide longest record as ``lmax``: ``run.features_hits`` gives global event indices and
    ``merge_group_sharded`` takes its hits unchanged), ``record_base``, ``n_total``, ``records_per_rank``,
    ``exchange_bytes`` (row and sample bytes this rank received from the other ranks) and ``timings`` (seconds per
    stage, each ended by a device synchronize).

    ``polarity``: {(board, channel): "positive" | "negative" | "unknown"}, applied to the shard's records as
    ``plugins.records`` applies the channel metadata to a single-GPU build (``ops.apply_polarity``).  It must be the
    same on every rank; maps that differ, or an invalid map on any rank, raise ValueError on every rank."""
    import time

    backend = backend if backend is not None else DeviceRecords()
    dist, rank, P = _dist()
    paths = [str(p) for p in paths]
    F = len(paths)
    T: dict = {}
    err = None
    pol_err, pol_digest = _polarity_digest(polarity)

    if mine is None:
        sizes = []
        for p in paths:
            try:
                sizes.append(os.path.getsize(p))
            except OSError as e:
                err = err or e
                sizes.append(0)
        mine = np.flatnonzero(default_file_owners(sizes, P) == rank)
    mine = np.asarray(mine, dtype=np.int64).reshape(-1)

    # ownership, checked on the gathered claims so that every rank raises
    claims = allgather_columns({"file": mine})["file"]
    claimed = np.bincount(claims[(claims >= 0) & (claims < F)], minlength=F)
    if len(claims) != int(claimed.sum()) or np.any(claimed != 1):
        bad = sorted(set(np.flatnonzero(claimed != 1).tolist()) | set(claims[(claims < 0) | (claims >= F)].tolist()))
        raise ValueError(f"every file must be read by exactly one rank: files {bad[:10]} are claimed by none, by several ranks or do not exist")

    # read + scan the own files in list order (a rank's files are a subsequence of the list: local order = global order)
    own = sorted(set(mine.tolist()))
    t = time.perf_counter()
    blobs, scans = [], []
    try:
        if err is None:
            for f in own:
                blobs.append(np.fromfile(paths[f], dtype=np.uint8))
            T["read"] = time.perf_counter() - t
            t = time.perf_counter()
            scans = [backend.scan(b) for b in blobs]
            T["scan"] = time.perf_counter() - t
    except (OSError, ValueError) as e:
        err = e
    status = np.zeros(F + 3, dtype=np.int64)
    status[:3] = [int(err is not None), int(pol_err is not None), pol_digest]
    for f, s in zip(own, scans):
        status[3 + f] = len(s["channel"])
    table = _allgather_i64(status)
    if table[:, 0].any():
        if err is not None:
            raise err
        raise RuntimeError(f"ranks {np.flatnonzero(table[:, 0]).tolist()} could not read their V1725 files")
    _check_polarity(table[:, 1], table[:, 2], pol_err)
    counts = table[:, 3:].sum(axis=0)
    seq_base = np.cumsum(counts) - counts
    seq = np.concatenate([seq_base[f] + np.arange(counts[f], dtype=np.int64) for f in own] or [np.zeros(0, np.int64)])

    # 1. local build
    t = time.perf_counter()
    up = backend.upload(scans, [paths[f] for f in own])
    del blobs, scans
    backend.sync()
    T["h2d"] = time.perf_counter() - t
    t = time.perf_counter()
    built = [backend.build(up, int(dt_ns), seq)]
    del up  # the stream bytes
    backend.sync()
    T["build"] = time.perf_counter() - t
    return _time_shard(built, backend, T, polarity)


def _polarity_digest(polarity) -> tuple:
    """(the ValueError of an invalid map or None, digest of the validated map)."""
    from .ops import polarity_entries

    try:
        return None, _digest(polarity_entries(polarity))
    except ValueError as e:
        return e, 0


def _check_polarity(bad, digests, own_err) -> None:
    """Raise on every rank when a rank's polarity map is invalid or the maps differ (gathered flag / digest columns)."""
    if np.any(bad):
        if own_err is not None:
            raise own_err
        raise ValueError(f"ranks {np.flatnonzero(bad).tolist()} were given an invalid polarity map")
    if np.any(digests != digests[0]):
        raise ValueError("polarity must be the same on every rank")


def _time_shard(built: list, backend, T: dict, polarity: dict | None = None) -> dict:
    """Stages 2-6 of the distributed time sort on a rank's locally built rows (record_id = global seq, sorted by
    (timestamp, board, channel, seq)): splitters, split points, exchange, global bases, merge, run-wide lmax, then the
    polarity map (validated by the caller) on the merged records.  ``built`` holds the local build and is emptied, so
    that the rows are freed once they are sent; ``T`` gets the stage timings.  Returns the dict of
    build_records_sharded_v1725."""
    import time

    _, rank, P = _dist()
    local = built.pop()

    # 2. splitters, 3. split points
    t = time.perf_counter()
    n_local = backend.count(local)
    pos, w = splitter_samples(n_local, SPLITTER_SAMPLES_PER_RANK * P)
    k = record_keys(backend.rows_at(local, pos))
    g = allgather_columns({"ts": k[:, 0], "board": k[:, 1], "channel": k[:, 2], "seq": k[:, 3], "w": w})
    splitters = plan_splitters(np.stack([g["ts"], g["board"], g["channel"], g["seq"]], axis=1), g["w"], P)
    cuts = np.r_[0, np.asarray(backend.split_points(local, splitters), dtype=np.int64), n_local]
    inner = cuts[:-1][cuts[:-1] < n_local]
    offs = np.r_[backend.rows_at(local, inner)["wave_offset"].astype(np.int64), np.full(P + 1 - len(inner), backend.n_samples(local))]
    row_counts, sample_counts = np.diff(cuts), np.diff(offs)
    T["splitters"] = time.perf_counter() - t

    # 4. exchange
    t = time.perf_counter()
    send_rows, send_pool = backend.send_buffers(local)
    rows, pool, recv = _exchange(send_rows, send_pool, row_counts, sample_counts, backend)
    del local, send_rows, send_pool
    backend.sync()
    T["exchange"] = time.perf_counter() - t
    others = np.arange(P) != rank
    exchange_bytes = int((recv[others, 0] * 102 + recv[others, 1] * 2).sum())

    # 5. global bases, 6. merge
    n_recv, s_recv = int(recv[:, 0].sum()), int(recv[:, 1].sum())
    bases = _allgather_i64([n_recv, s_recv])
    record_base, pool_base = int(bases[:rank, 0].sum()), int(bases[:rank, 1].sum())
    t = time.perf_counter()
    shard = backend.merge(rows, pool, np.r_[0, np.cumsum(recv[:, 0])], record_base, pool_base)
    del rows, pool
    backend.sync()
    T["merge"] = time.perf_counter() - t
    lmax = _allreduce_max(backend.lmax(shard))
    run = backend.run(shard, lmax, record_base, pool_base)
    if polarity:
        t = time.perf_counter()
        backend.apply_polarity(run, polarity)
        backend.sync()
        T["polarity"] = time.perf_counter() - t
    return dict(run=run, record_base=record_base, pool_base=pool_base,
                n_total=int(bases[:, 0].sum()), records_per_rank=bases[:, 0].copy(), exchange_bytes=exchange_bytes, timings=T)


def _check_group(g: int, cols) -> tuple:
    """One raw row group -> (timestamps_ps int64, boards int16, channels int16, samples 2-D int16 / uint16); ValueError
    when the columns do not describe the same rows."""
    try:
        ts, board, channel, samples = cols
    except (TypeError, ValueError):
        raise ValueError(f"group {g}: expected (timestamps_ps, boards, channels, samples)") from None
    samples = np.asarray(samples)
    if samples.ndim != 2 or samples.dtype not in (np.int16, np.uint16):
        raise ValueError(f"group {g}: samples must be a 2-D int16 array, got {samples.dtype} {samples.shape}")
    out = (np.asarray(ts, dtype=np.int64).reshape(-1), np.asarray(board, dtype=np.int16).reshape(-1),
           np.asarray(channel, dtype=np.int16).reshape(-1), samples)
    if not len(out[0]) == len(out[1]) == len(out[2]) == len(samples):
        raise ValueError(f"group {g}: {len(out[0])} timestamps, {len(out[1])} boards, {len(out[2])} channels and {len(samples)} "
                         "sample rows")
    return out


def build_records_sharded(groups, *, n_groups: int, dt_ns: int, baseline_window=(0, 40), epoch_ns: int | None = None,
                          backend=None, polarity: dict | None = None) -> dict:
    """This rank's time shard of a run made of ``n_groups`` groups of raw rows, without any process holding the whole
    run: the result of ``ops.build_records`` / ``ops.build_records_ragged`` (as ``plugins.records.build_bundle`` picks
    them) on all groups concatenated in group-index order.

    ``groups`` maps a global group index to ``(timestamps_ps, boards, channels, samples)`` (``samples`` a 2-D int16
    array, one row per waveform) for the groups THIS rank read, e.g. one per-channel file group parsed by the
    reference's ``format_reader``.  Groups may have different widths.  A group index outside [0, n_groups), a group
    claimed by no rank or by two ranks, a group whose columns differ in length, and ``n_groups``, ``dt_ns``,
    ``baseline_window`` or ``epoch_ns`` differing between ranks raise ValueError on every rank.

    Each row's seq is its index in the concatenation of all groups; every rank builds its own rows with record_id =
    seq (``wfb_build_records_ragged_seq``), which orders them by (timestamp, board, channel, seq), the single-GPU
    order, and the distributed time sort of build_records_sharded_v1725 does the rest.  Returns the same dict;
    ``timings`` has h2d, build, splitters, exchange and merge (and polarity).  ``polarity`` as in
    build_records_sharded_v1725."""
    import time

    backend = backend if backend is not None else DeviceRecords()
    T: dict = {}
    err = None
    pol_err, pol_digest = _polarity_digest(polarity)
    own: list = []
    cols: list = []
    params = np.zeros(6, dtype=np.int64)
    try:
        bl0, bl1 = (int(x) for x in baseline_window)
        params[:] = [int(n_groups), int(dt_ns), bl0, bl1, epoch_ns is None, 0 if epoch_ns is None else int(epoch_ns)]
        if int(dt_ns) <= 0 or int(n_groups) < 0:
            raise ValueError(f"dt_ns must be positive and n_groups non-negative, got {dt_ns} and {n_groups}")
        items = sorted((int(g), c) for g, c in dict(groups).items())
        own = [g for g, _ in items]
        cols = [_check_group(g, c) for g, c in items]
    except (TypeError, ValueError) as e:
        err, own, cols = e, [], []

    # parameters and local errors first (fixed size, so a rank with different arguments cannot stall the gather)
    table = _allgather_i64(np.r_[int(err is not None), params, int(pol_err is not None), pol_digest])
    if table[:, 0].any():
        if err is not None:
            raise err
        raise ValueError(f"ranks {np.flatnonzero(table[:, 0]).tolist()} were given malformed row groups or arguments")
    if np.any(table[:, 1:7] != table[:1, 1:7]):
        raise ValueError("n_groups, dt_ns, baseline_window and epoch_ns must be the same on every rank")
    _check_polarity(table[:, 7], table[:, 8], pol_err)

    # ownership, checked on the gathered claims so that every rank raises
    G = int(n_groups)
    g = allgather_columns({"group": np.asarray(own, dtype=np.int64), "rows": np.array([len(c[0]) for c in cols], dtype=np.int64)})
    claims = g["group"]
    inside = (claims >= 0) & (claims < G)
    claimed = np.bincount(claims[inside], minlength=G)
    if not inside.all() or np.any(claimed != 1):
        bad = sorted(set(np.flatnonzero(claimed != 1).tolist()) | set(claims[~inside].tolist()))
        raise ValueError(f"every group must be read by exactly one rank: groups {bad[:10]} are claimed by none, by several ranks "
                         f"or are outside [0, {G})")
    counts = np.zeros(G, dtype=np.int64)
    counts[claims] = g["rows"]
    seq_base = np.cumsum(counts) - counts
    seq = np.concatenate([seq_base[f] + np.arange(counts[f], dtype=np.int64) for f in own] or [np.zeros(0, np.int64)])

    # 1. local build (the rank's groups in increasing index: its input order is the global order restricted to them)
    t = time.perf_counter()
    ts, board, channel = (np.concatenate([c[k] for c in cols] or [np.zeros(0, dt)]) for k, dt in enumerate((np.int64, np.int16, np.int16)))
    up = backend.upload_raw(ts, board, channel, [c[3] for c in cols])
    del cols, ts, board, channel
    backend.sync()
    T["h2d"] = time.perf_counter() - t
    t = time.perf_counter()
    built = [backend.build_raw(up, int(dt_ns), (int(params[2]), int(params[3])), epoch_ns, seq)]
    del up
    backend.sync()
    T["build"] = time.perf_counter() - t
    return _time_shard(built, backend, T, polarity)


# ------------------------------------------------------------------------------------------------
# Time-sharded df -> df_events -> df_paired: anchored windows cut at segment starts
# ------------------------------------------------------------------------------------------------
# The `df` rows of a rank are its time shard sorted by timestamp; concatenated in rank order they are the single-run
# `df` when the shards are in time order (df_sharded checks that on gathered first / last timestamps).
#
# df_events groups the time-sorted rows into anchored windows (event_grouping.py:477-510).  A SEGMENT starts wherever
# (double)ts[i] > (double)ts[i - 1] + W (k4_segment_flags_kernel): every segment start is an anchor whatever came
# before it, and the anchors inside a segment depend on that segment alone.  So a cut at a segment start splits the
# run into parts that group independently, and two counts per rank number the events globally.
#
# What travels: the first and the last K df rows of every rank (timestamp, area, height, channel: 24 B per row,
# K = 4096 by default) in ONE all_gather, plus one all_gather of 8 bytes per rank.  The zones of two neighbouring
# non-empty ranks are consecutive in the global order, so every rank finds the same segment starts in
# tail[r] ++ head[next] and picks the one nearest to the nominal boundary.  Without one the zones are doubled; when
# both zones already hold their whole shards the boundary is dropped: the rank after it owns nothing and its rows
# (all of them in the gathered zones) go to the owner before it.  A run without gaps is therefore legal: one segment
# spanning all ranks ends up with one owner.

EVENT_ZONE_DTYPE = np.dtype({"names": ["timestamp", "area", "height", "channel"], "formats": ["<i8", "<f4", "<f4", "<i2"],
                             "offsets": [0, 8, 12, 16], "itemsize": 24})


def check_time_order(table: np.ndarray) -> None:
    """``table``: one row (rows, first timestamp, last timestamp) per rank.  Raises ValueError when a non-empty
    rank ends after the next non-empty rank starts (the same on every rank: the table is gathered)."""
    t = np.asarray(table, dtype=np.int64).reshape(-1, 3)
    live = np.flatnonzero(t[:, 0] > 0)
    for a, b in zip(live[:-1], live[1:]):
        if t[a, 2] > t[b, 1]:
            raise ValueError(f"the df shards are not in time order: rank {a} ends at timestamp {t[a, 2]}, after rank {b} starts "
                             f"at {t[b, 1]}; concatenated in rank order they would not be the run's df")


def segment_starts(ts: np.ndarray, w_ps: float) -> np.ndarray:
    """Positions i >= 1 of consecutive time-sorted rows where a segment starts: the kernel's float64 test
    (double)ts[i] > (double)ts[i - 1] + W."""
    t = np.asarray(ts, dtype=np.int64).astype(np.float64)
    return np.flatnonzero(t[1:] > t[:-1] + float(w_ps)) + 1


def plan_event_cuts(heads: list, tails: list, wholes: list, counts, w_ps: float):
    """The global df rows every rank owns for df_events.  heads[r] / tails[r]: the first / last zone rows of rank r
    (EVENT_ZONE_DTYPE, disjoint), wholes[r]: the two zones are the whole shard, counts[r]: its rows, w_ps: the window
    in ps.  Returns (bounds, ok): bounds[r] = [lo, hi) of global rows owned by rank r (lo == hi: nothing); ok is False
    when a boundary has no segment start inside zones that do not cover both shards yet (the caller doubles them)."""
    counts = np.asarray(counts, dtype=np.int64)
    R = len(counts)
    base = np.r_[0, np.cumsum(counts)]
    live = [r for r in range(R) if counts[r] > 0]
    cuts: list = []  # cut between live[i] and live[i + 1]: a global row, or None (boundary dropped)
    for a, b in zip(live[:-1], live[1:]):
        za = np.concatenate([heads[a], tails[a]]) if wholes[a] else tails[a]
        zb = np.concatenate([heads[b], tails[b]]) if wholes[b] else heads[b]
        s = segment_starts(np.concatenate([za["timestamp"], zb["timestamp"]]), w_ps)
        if len(s) == 0:
            if wholes[a] and wholes[b]:
                cuts.append(None)
                continue
            return None, False
        g = int(base[a + 1]) - len(za) + s  # global rows of the candidates
        cuts.append(int(g[np.argmin(np.abs(g - base[b]))]))
    bounds = np.stack([base[:-1], base[:-1]], axis=1)
    for i, r in enumerate(live):
        lo = 0 if i == 0 else cuts[i - 1]
        if lo is None:
            continue
        hi = next((c for c in cuts[i:] if c is not None), int(base[-1]))
        bounds[r] = (lo, hi)
    return bounds, True


def _zone_rows_in(heads, tails, counts, ranks, lo: int, hi: int) -> np.ndarray:
    """The zone rows of ``ranks`` (ascending) at global rows [lo, hi), in global order; every such row must be in the
    zones (the cut plan guarantees it)."""
    base = np.r_[0, np.cumsum(np.asarray(counts, dtype=np.int64))]
    parts = []
    for q in ranks:
        b, n = int(base[q]), int(counts[q])
        hq, tq = heads[q], tails[q]
        pos = np.r_[b + np.arange(len(hq)), b + n - len(tq) + np.arange(len(tq))]
        sel = (pos >= lo) & (pos < hi)
        want = max(min(hi, b + n) - max(lo, b), 0)
        if int(sel.sum()) != want:
            raise RuntimeError(f"events_sharded: rank {q} has owned rows outside its gathered zones")
        parts.append(np.concatenate([hq, tq])[sel])
    return np.concatenate(parts) if parts else np.zeros(0, dtype=EVENT_ZONE_DTYPE)


def _pack_zone(ts, area, height, channel) -> np.ndarray:
    z = np.zeros(len(ts), dtype=EVENT_ZONE_DTYPE)
    z["timestamp"], z["area"], z["height"], z["channel"] = ts, area, height, channel
    return z


class HostEvents:
    """Backend for df columns held as numpy arrays (CPU tests: the compute is the oracle's ``df_columns``,
    ``group_time_window`` and ``pair_events``).  ``run`` is the shard's RECORDS rows, ``features`` its
    BASIC_FEATURES rows."""

    def __init__(self, df_fn, group_fn, pair_fn):
        self.df_fn, self.group_fn, self.pair_fn = df_fn, group_fn, pair_fn

    def df_local(self, run, features, gains):
        cols = dict(self.df_fn(features, record_id=np.asarray(run["record_id"], dtype=np.int64), gains=gains))
        return cols, np.asarray(cols.pop("order"), dtype=np.int64), len(features)

    def ts_ends(self, cols, n):
        return (int(cols["timestamp"][0]), int(cols["timestamp"][n - 1])) if n else (0, 0)

    def zone(self, cols, a, b):
        return _pack_zone(cols["timestamp"][a:b], cols["area"][a:b], cols["height"][a:b], cols["channel"][a:b])

    def assemble(self, cols, l0, l1, first, last):
        return {k: np.concatenate([first[k], np.asarray(cols[k][l0:l1]), last[k]]) for k in EVENT_ZONE_DTYPE.names}

    def iota(self, n, base):
        return np.arange(n, dtype=np.int64) + base

    def sync(self):
        pass

    def events(self, owned, time_window_ns, pair_window_ns, n_channels, timings=None):
        ev = self.group_fn(owned["timestamp"], owned["channel"], time_window_ns)
        m = np.asarray(ev["members"], dtype=np.int64)
        res = dict(t_min=ev["t_min"], t_max=ev["t_max"], dt_ns=ev["dt_ns"], n_hits=np.asarray(ev["n_hits"], dtype=np.int64),
                   offsets=np.asarray(ev["offsets"], dtype=np.int64), members=m, member_ts=owned["timestamp"][m],
                   member_channel=owned["channel"][m], member_area=owned["area"][m], member_height=owned["height"][m])
        p = self.pair_fn(res["offsets"], res["member_ts"], res["member_area"], res["member_height"], res["dt_ns"], pair_window_ns, n_channels)
        res.update(keep=np.asarray(p["keep"], dtype=bool), delta_t=p["delta_t"], area_ch=p["area_ch"], height_ch=p["height_ch"],
                   n_events=len(res["t_min"]))
        return res


class DeviceEvents:
    """Backend for df columns that stay on the device: ``run`` is a ``DeviceRun``, ``features`` its BASIC_FEATURES rows
    from ``DeviceRun.features_hits`` (uint8 tensor, 36 B per row); record_id is the rows' ``wfb_rec_meta.record_id``."""

    def df_local(self, run, features, gains):
        import torch

        from . import ops

        n = run.n
        rid = run.meta[: n * 48].view(n, 48)[:, 40:48].contiguous().view(-1).view(torch.int64) if n else None  # wfb_rec_meta.record_id
        cols = ops.df_columns_device(features[: n * 36] if n else None, n, rid, gains)
        return cols, cols.pop("order"), n

    def ts_ends(self, cols, n):
        if not n:
            return 0, 0
        t = cols["timestamp"][[0, n - 1]].cpu().numpy()
        return int(t[0]), int(t[1])

    def zone(self, cols, a, b):
        return _pack_zone(*(cols[k][a:b].cpu().numpy() for k in ("timestamp", "area", "height", "channel")))

    def assemble(self, cols, l0, l1, first, last):
        import torch

        from .engine import upload

        out = {}
        for k in EVENT_ZONE_DTYPE.names:
            parts = [upload(np.ascontiguousarray(z[k])) for z in (first,) if len(z)]
            parts.append(cols[k][l0:max(l0, l1)])
            parts += [upload(np.ascontiguousarray(z[k])) for z in (last,) if len(z)]
            out[k] = torch.cat(parts) if len(parts) > 1 else parts[0]
        return out

    def iota(self, n, base):
        import torch

        return torch.arange(n, dtype=torch.int64, device="cuda") + base

    def sync(self):
        import torch

        torch.cuda.synchronize()

    def events(self, owned, time_window_ns, pair_window_ns, n_channels, timings=None):
        import time

        from . import ops

        T = timings if timings is not None else {}
        ts = owned["timestamp"]
        n = int(ts.numel())
        t = time.perf_counter()
        ev, n_ev = ops.group_time_window_device(ts, n, time_window_ns)
        self.sync()
        T["group"], t = time.perf_counter() - t, time.perf_counter()
        res = ops.event_table_device(ts, ev, n, n_ev, owned["channel"], area=owned["area"], height=owned["height"])
        self.sync()
        T["event_table"], t = time.perf_counter() - t, time.perf_counter()
        res.update(ops.pair_events_device(res["offsets"], n_ev, res["member_ts"], res["member_area"], res["member_height"], res["dt_ns"],
                                          pair_window_ns, n_channels))
        self.sync()
        T["pair"] = time.perf_counter() - t
        res["n_events"] = n_ev
        return res


def df_sharded(run, features, *, gains: dict | None = None, backend=None) -> dict:
    """This rank's part of the run's `df`: ``wfb_df_columns`` on the rank's feature rows, left where they are (device
    tensors with ``DeviceEvents``, the default).  ``run`` / ``features``: the rank's time shard and its basic_features
    rows (``DeviceRun`` + ``features_hits()["features"]``); record_id is the rows' record_id, global for the shards of
    ``build_records_sharded_v1725`` and ``DeviceRun.synth(record_base=...)``.

    The shards must be in time order: every rank gathers every non-empty rank's first and last timestamp and raises
    ValueError (every rank alike) when one ends after the next one starts.  Returns ``cols`` (timestamp, record_id,
    area, height, amp, max_abs_diff, board, channel [, area_pe, height_pe]; timestamp-sorted), ``index`` (row_base +
    the local sort order: the DataFrame index), ``n``, ``row_base``, ``rows_per_rank`` and ``with_pe``."""
    backend = backend if backend is not None else DeviceEvents()
    _, rank, _ = _dist()
    cols, order, n = backend.df_local(run, features, gains)
    first, last = backend.ts_ends(cols, n)
    table = _allgather_i64([n, first, last])
    check_time_order(table)
    me = rank if len(table) > 1 else 0
    row_base = int(table[:me, 0].sum())
    return dict(cols=cols, index=order + row_base, n=n, row_base=row_base, rows_per_rank=table[:, 0].copy(), with_pe=gains is not None)


def events_sharded(df: dict, *, time_window_ns: float = 100.0, pair_window_ns: float = 100.0, n_channels: int = 2,
                   start_channel_slice: int = 6, backend=None, zone_rows: int = 4096) -> dict:
    """df_events + df_paired of a time-sharded `df` (``df_sharded``'s result) without gathering the rows.

    Every rank exchanges its boundary zones (``zone_rows`` rows per end, doubled while a boundary has no segment
    start in them), owns the global rows between its two cuts (assembled on its device: gathered zone rows, then the
    untouched middle of its shard), groups them (``wfb_group_time_window``), builds the event table
    (``wfb_event_table``) and pairs the events (``wfb_pair_events``, ``pair_window_ns``).  Returns the rank's events
    with GLOBAL ids (``event_id``, ``t_min``, ``t_max``, ``dt_ns``, ``n_hits``), the CSR ``offsets`` with ``members``
    (global df rows) and the member-ordered ``member_ts`` / ``member_channel`` / ``member_area`` / ``member_height``,
    ``keep`` / ``delta_t`` / ``area_ch`` / ``height_ch``, ``event_base``, ``events_per_rank``, ``bounds`` (every rank's
    owned [lo, hi)), ``zone_rows``, ``gathered_bytes`` (what this rank received in the collectives) and ``timings``
    (seconds per stage, each ended by a device synchronize)."""
    import time

    backend = backend if backend is not None else DeviceEvents()
    _, rank, _ = _dist()
    cols, n = df["cols"], int(df["n"])
    w_ps = float(time_window_ns) * 1e3
    k = max(int(zone_rows), 1)
    gathered = 0
    T: dict = {}
    t = time.perf_counter()
    while True:
        head, tail, whole = event_zones(backend, cols, n, k)
        heads, tails, wholes, counts, nbytes = _allgather_zones(head, tail, k, whole, n)
        gathered += nbytes
        bounds, ok = plan_event_cuts(heads, tails, wholes, counts, w_ps)
        if ok:
            break
        k *= 2
    R = len(heads)
    me = rank if R > 1 else 0
    T["zones"] = time.perf_counter() - t
    res = owned_events(backend, cols, me, heads, tails, counts, bounds, time_window_ns=time_window_ns, pair_window_ns=pair_window_ns,
                       n_channels=n_channels, timings=T)
    table = _allgather_i64([res["n_events"]])
    gathered += table.nbytes if R > 1 else 0
    res["event_base"] = int(table[:me, 0].sum())
    res["event_id"] = backend.iota(res["n_events"], res["event_base"])
    res.update(events_per_rank=table[:, 0].copy(), bounds=bounds, zone_rows=k, gathered_bytes=gathered, n_channels=int(n_channels),
               start_channel_slice=int(start_channel_slice), pair_window_ns=float(pair_window_ns), timings=T)
    return res


def event_zones(backend, cols, n: int, k: int):
    """The first and the last (at most) ``k`` df rows of a rank as EVENT_ZONE_DTYPE rows, disjoint, and whether they
    are the whole shard."""
    kh = min(k, n)
    kt = min(k, n - kh)
    return backend.zone(cols, 0, kh), backend.zone(cols, n - kt, n), kh + kt == n


def owned_events(backend, cols, me: int, heads, tails, counts, bounds, *, time_window_ns: float, pair_window_ns: float,
                 n_channels: int, timings: dict | None = None) -> dict:
    """The local part of events_sharded on rank ``me``, given every rank's zones and the plan: assemble the owned rows
    (lower ranks' zone rows, the rank's own rows between the cuts, upper ranks' zone rows), group them, build the event
    table and pair the events.  ``members`` are global df rows; ``owned`` is the rank's [lo, hi)."""
    R = len(counts)
    lo, hi = (int(x) for x in bounds[me])
    base, n = int(sum(counts[:me])), int(counts[me])
    l0, l1 = min(max(lo - base, 0), n), min(max(hi - base, 0), n)
    first = _zone_rows_in(heads, tails, counts, range(me), lo, hi)
    last = _zone_rows_in(heads, tails, counts, range(me + 1, R), lo, hi)
    import time

    t = time.perf_counter()
    owned = backend.assemble(cols, l0, l1, first, last)
    backend.sync()
    if timings is not None:
        timings["assemble"] = time.perf_counter() - t
    res = backend.events(owned, float(time_window_ns), float(pair_window_ns), int(n_channels), timings)
    res["members"] = res["members"] + lo
    res["owned"] = (lo, hi)
    return res


def _host(x) -> np.ndarray:
    return x.cpu().numpy() if hasattr(x, "cpu") else np.asarray(x)


def gather_event_frames(df_sh: dict, ev_sh: dict):
    """(df, df_events, df_paired) of the WHOLE run on every rank, equal to what B200DataFramePlugin,
    B200GroupedEventsPlugin and B200PairedEventsPlugin return for the run.  Every rank receives every row, member and
    event, so this holds the whole run in each process (like ``gather_rows``): it is for checks and small runs, the
    sharded results themselves stay distributed."""
    import pandas as pd

    from .plugins.dataframe import DF_COLUMNS, df_frame, pair_events_frame, paired_frame
    from .plugins.grouping import DF_EVENTS_COLUMNS, events_frame

    cols, with_pe = df_sh["cols"], bool(df_sh["with_pe"])
    names = list(DF_COLUMNS) + (["area_pe", "height_pe"] if with_pe else [])
    host = {k: _host(cols[k]) for k in names}
    rows = np.zeros(int(df_sh["n"]), dtype=[("index", "<i8")] + [(k, host[k].dtype) for k in names])
    rows["index"] = _host(df_sh["index"])
    for k in names:
        rows[k] = host[k]
    rows = gather_rows(rows)
    df = df_frame({k: rows[k] for k in names}, rows["index"], with_pe)

    nc, start = ev_sh["n_channels"], ev_sh["start_channel_slice"]
    n_ev = int(ev_sh["n_events"])
    ev_rows = np.zeros(n_ev, dtype=[("event_id", "<i8"), ("t_min", "<i8"), ("t_max", "<i8"), ("dt_ns", "<f8"), ("n_hits", "<i8"),
                                    ("keep", "u1"), ("delta_t", "<f8"), ("area_ch", "<f4", (nc,)), ("height_ch", "<f4", (nc,))])
    for k in ev_rows.dtype.names:
        ev_rows[k] = _host(ev_sh[k]).reshape(ev_rows[k].shape)
    ev_rows = gather_rows(ev_rows)
    m = len(_host(ev_sh["member_ts"]))
    mem = np.zeros(m, dtype=[("ts", "<i8"), ("channel", "<i2"), ("area", "<f4"), ("height", "<f4")])
    mem["ts"], mem["channel"] = _host(ev_sh["member_ts"]), _host(ev_sh["member_channel"])
    mem["area"], mem["height"] = _host(ev_sh["member_area"]), _host(ev_sh["member_height"])
    mem = gather_rows(mem)

    if len(df) == 0:
        df_events = pd.DataFrame(columns=DF_EVENTS_COLUMNS)
        return df, df_events, pair_events_frame(df_events, nc, start, ev_sh["pair_window_ns"])
    offsets = np.r_[0, np.cumsum(ev_rows["n_hits"])].astype(np.int64)
    table = {k: np.ascontiguousarray(ev_rows[k]) for k in ("event_id", "t_min", "t_max", "dt_ns", "n_hits")}
    table["offsets"] = offsets
    df_events = events_frame(table, np.ascontiguousarray(mem["channel"]), np.ascontiguousarray(mem["area"]),
                             np.ascontiguousarray(mem["height"]), np.ascontiguousarray(mem["ts"]))
    out = dict(keep=ev_rows["keep"].astype(bool), delta_t=np.ascontiguousarray(ev_rows["delta_t"]),
               area_ch=np.ascontiguousarray(ev_rows["area_ch"]).reshape(-1, nc), height_ch=np.ascontiguousarray(ev_rows["height_ch"]).reshape(-1, nc))
    return df, df_events, paired_frame(df_events, offsets, out, nc, start)


# ------------------------------------------------------------------------------------------------
# Time-sharded wave_pool_filtered -> hit -> waveform_width -> s1_s2: per-record rows, no boundary zones
# ------------------------------------------------------------------------------------------------
# Every row of this branch depends on one record only: the filtered samples of a record, its find_peaks rows, the
# width of each of its peaks and that width's label (with the record's own basic_features row).  So a rank runs the
# chain on its time shard alone and the rank-order concatenation of the shards' rows is the single-GPU result.  The
# only collective is ONE fixed-size all_gather per rank: an error flag, a digest of the options and the three row
# counts, which number every rank's rows globally.


def _sync():
    import torch

    torch.cuda.current_stream().synchronize()


def peaks_local(run, *, filter_cfg: dict | None = None, features=None, peak_opts: dict | None = None, width_opts: dict | None = None,
                s1s2_opts: dict | None = None, filter_options: dict | None = None, channel_config=None, run_id: str | None = None) -> dict:
    """The filter -> hit -> waveform_width -> s1_s2 chain on ONE time shard (a ``DeviceRun`` with its own records and
    pool slice, ``pool_base`` / ``row_base`` set), with no collective.  Everything stays on the device.

    1. ``filter_cfg`` (one configuration for every record) or ``filter_options`` with ``channel_config`` and ``run_id``
       (``B200WavePoolFilteredPlugin``'s options, resolved for each channel of the shard as the plugin resolves
       them) filters the shard into a float32 pool through ``ops.filter_run_device``; neither keeps the raw 16-bit
       pool (the ``use_filtered=False`` route).  Both is a ValueError.
    2. ``ops.find_peaks_device`` on those samples (``WFB_WAVE_REC_F32`` / ``WFB_WAVE_REC_U16``) with ``peak_opts``
       (``find_peaks_launch``'s options): the `hit` rows of ``B200HitFinderPlugin(wave_source="records")``.
    3. ``ops.waveform_width_run`` on the same samples with ``width_opts`` (sampling_rate, rise_low, rise_high,
       fall_high, fall_low, interpolation): ``B200WaveformWidthPlugin`` on the shard's st_waveforms / filtered rows.
    4. With ``features`` (the shard's packed basic_features rows, as ``run.features_hits()["features"]`` returns
       them): ``ops.s1s2_classify_device`` with ``feat_row_base = run.row_base`` and ``s1s2_opts`` (width_unit,
       normalised ranges, conflict_policy).

    Returns ``filtered`` (float32 device pool or None), ``hits`` / ``widths`` / ``labels`` (packed rows as device
    uint8 tensors; ``labels`` None without features) with ``n_hits`` / ``n_widths`` / ``n_labels``, and ``timings``
    (seconds per stage, each ended by a device synchronize)."""
    import time

    from . import _lib, ops
    from .engine import DeviceRun

    if filter_cfg is not None and filter_options is not None:
        raise ValueError("peaks_local takes filter_cfg or filter_options, not both")
    T: dict = {}
    t = time.perf_counter()
    src, filtered = run, None
    if filter_cfg is not None or filter_options is not None:
        filtered = ops.filter_run_device(run, filter_cfg, filter_options=filter_options, channel_config=channel_config, run_id=run_id)
        src = DeviceRun(run.meta, filtered, run.n, 1, run.lmax, records_rows=run.records_rows, pool_base=run.pool_base, row_base=run.row_base)
        _sync()
        T["filter"] = time.perf_counter() - t
    t = time.perf_counter()
    if run.n and run.lmax > 0:
        kind = _lib.WAVE_REC_F32 if src.pool_is_f32 else _lib.WAVE_REC_U16
        hits, n_hits = ops.find_peaks_device(src, kind, src.lmax, **(peak_opts or {}))
    else:
        hits, n_hits = ops._empty(0), 0
    _sync()
    T["hit"] = time.perf_counter() - t
    t = time.perf_counter()
    widths, n_widths = ops.waveform_width_run(src, hits, n_hits, **(width_opts or {}))
    _sync()
    T["width"] = time.perf_counter() - t
    labels, n_labels = None, 0
    if features is not None:
        t = time.perf_counter()
        labels = ops.s1s2_classify_device(widths, n_widths, features, run.n, feat_row_base=run.row_base, **(s1s2_opts or {}))
        n_labels = n_widths
        _sync()
        T["s1_s2"] = time.perf_counter() - t
    return dict(filtered=filtered, hits=hits, n_hits=int(n_hits), widths=widths, n_widths=int(n_widths), labels=labels, n_labels=int(n_labels),
                timings=T)


def _canonical(x):
    """A JSON-able form of an options tree that equal options share: mappings become key-sorted [key, value] pairs,
    channel keys (HardwareChannel-like objects, (board, channel) pairs, "board:channel" strings) one form, arrays and
    tuples lists."""
    import json
    from collections.abc import Mapping

    from .channel_config import parse_channel_ref

    if isinstance(x, Mapping):
        items = []
        for k, v in x.items():
            ref = parse_channel_ref(k) if not isinstance(k, (int, float)) else None
            items.append([["channel", *ref] if ref is not None else _canonical(k), _canonical(v)])
        return ["map", sorted(items, key=lambda kv: json.dumps(kv[0]))]
    if isinstance(x, (str, bool, int, float)) or x is None:
        return x
    if isinstance(x, (list, tuple)):
        return [_canonical(v) for v in x]
    if isinstance(x, (np.ndarray, np.generic)):
        return np.asarray(x).tolist()
    return repr(x)


def _digest(x) -> int:
    """64-bit digest of ``_canonical(x)``: equal on every process for equal options."""
    import hashlib
    import json

    blob = json.dumps(_canonical(x))
    return int(np.frombuffer(hashlib.blake2b(blob.encode(), digest_size=8).digest(), dtype="<i8")[0])


def peaks_options_digest(filter_cfg, with_features: bool, peak_opts, width_opts, s1s2_opts, *, filter_options=None, channel_config=None,
                         run_id=None) -> int:
    """64-bit digest of the options of the peaks leg, equal on every process for equal options."""
    return _digest([filter_cfg, bool(with_features), peak_opts or {}, width_opts or {}, s1s2_opts or {}, filter_options, channel_config,
                    run_id])


def peaks_sharded(run, *, filter_cfg: dict | None = None, features=None, peak_opts: dict | None = None, width_opts: dict | None = None,
                  s1s2_opts: dict | None = None, filter_options: dict | None = None, channel_config=None, run_id: str | None = None,
                  local_fn=None) -> dict:
    """``peaks_local`` on this rank's time shard plus ONE fixed-size all_gather (error flag, options digest, the three
    row counts).  Options that differ between ranks, or an error on any rank, raise ValueError on every rank (the
    rank that failed raises its own error).  With ``filter_options`` / ``channel_config`` each rank resolves the
    filters of its own channels; the resolution depends on (run_id, board, channel) only, so the ranks agree.

    Returns ``peaks_local``'s result plus ``hit_base`` / ``width_base`` / ``label_base`` (global index of the rank's
    first row), ``hits_per_rank`` / ``widths_per_rank`` / ``labels_per_rank`` and the totals ``n_hits_total`` /
    ``n_widths_total`` / ``n_labels_total``.  ``local_fn`` replaces ``peaks_local`` (tests of the collective)."""
    local_fn = local_fn if local_fn is not None else peaks_local
    _, rank, _ = _dist()
    err, res, digest = None, {}, 0
    try:
        digest = peaks_options_digest(filter_cfg, features is not None, peak_opts, width_opts, s1s2_opts, filter_options=filter_options,
                                      channel_config=channel_config, run_id=run_id)
        res = local_fn(run, filter_cfg=filter_cfg, features=features, peak_opts=peak_opts, width_opts=width_opts, s1s2_opts=s1s2_opts,
                       filter_options=filter_options, channel_config=channel_config, run_id=run_id)
        counts = [int(res["n_hits"]), int(res["n_widths"]), int(res["n_labels"])]
    except Exception as e:  # noqa: BLE001 - every rank must reach the gather, the error is raised after it
        err, counts = e, [0, 0, 0]
    table = _allgather_i64([int(err is not None), digest, *counts])
    if table[:, 0].any():
        if err is not None:
            raise err
        raise ValueError(f"the peaks leg failed on ranks {np.flatnonzero(table[:, 0]).tolist()}")
    if np.any(table[:, 1] != table[0, 1]):
        raise ValueError("filter_cfg, filter_options, channel_config, run_id, features (given or not), peak_opts, width_opts and s1s2_opts "
                         "must be the same on every rank")
    me = rank if len(table) > 1 else 0
    res = dict(res)
    for j, k in enumerate(("hit", "width", "label")):
        res[f"{k}_base"] = int(table[:me, 2 + j].sum())
        res[f"{k}s_per_rank"] = table[:, 2 + j].copy()
        res[f"n_{k}s_total"] = int(table[:, 2 + j].sum())
    return res


def gather_peak_rows(sh: dict):
    """(hit, waveform_width, s1_s2) rows of the WHOLE run on every rank, as HIT_DTYPE, WAVEFORM_WIDTH_DTYPE and
    S1_S2_CLASSIFIER_DTYPE arrays (s1_s2 None when the leg ran without features).  Every rank receives every row,
    like ``gather_rows``: for checks and small runs."""
    from .dtypes import HIT_DTYPE, S1_S2_CLASSIFIER_DTYPE, WAVEFORM_WIDTH_DTYPE

    def rows(t, n, dt):
        n = int(n)
        return _host(t[: n * dt.itemsize]).view(dt) if n else np.zeros(0, dtype=dt)

    hits = gather_rows(rows(sh["hits"], sh["n_hits"], HIT_DTYPE))
    widths = gather_rows(rows(sh["widths"], sh["n_widths"], WAVEFORM_WIDTH_DTYPE))
    labels = None if sh["labels"] is None else gather_rows(rows(sh["labels"], sh["n_labels"], S1_S2_CLASSIFIER_DTYPE))
    return hits, widths, labels


def channel_rules(run, channel_config, *, run_id: str | None, threshold: float, fixed_baseline: float | None = None) -> np.ndarray:
    """The wfb_chan_rule array for ``run.features_hits(threshold=threshold, rules=...)`` on a time shard: the
    ``threshold`` and ``fixed_baseline`` of each channel of the shard resolved from ``channel_config`` the way
    ``B200ThresholdHitPlugin`` and ``B200BasicFeaturesPlugin`` resolve them for ``run_id`` (a rule only for a channel
    whose threshold differs from ``threshold`` or that has a fixed baseline)."""
    from .channel_config import resolve_channel_values
    from .engine import make_rules
    from .ops import shard_channels

    base = {"threshold": threshold, "fixed_baseline": fixed_baseline}
    thr, fixed = {}, {}
    for b, c in shard_channels(run):
        v = resolve_channel_values(channel_config, run_id, b, c, base)
        if float(v["threshold"]) != float(threshold):
            thr[(b, c)] = float(v["threshold"])
        if v.get("fixed_baseline") is not None:
            fixed[(b, c)] = float(v["fixed_baseline"])
    return make_rules(thr, fixed)
