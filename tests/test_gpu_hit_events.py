"""GPU: the device hit_grouped event table (wfb_hit_event_table behind ops.group_hit_windows and
ops.hit_event_table_device) against the oracle, and the time-sharded hit_merge -> hit_grouped table with P ranks
simulated on one GPU (the zone / cut / owned-row code of distributed.merge_group_sharded with the device backend, then
distributed.hit_events_sharded), compared with B200HitGroupedPlugin over the whole run."""

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

W_NS = 100.0
TABLE_KEYS = ("event_id", "t_min", "t_max", "dt_ns", "n_hits", "offsets", "members", "event_of_hit")


def _check_table(got, want, keys=TABLE_KEYS):
    for k in keys:
        g, w = np.asarray(got[k]), np.asarray(want[k])
        assert g.dtype == w.dtype, k
        assert np.array_equal(g, w), k


def _hits(sizes, seed, *, t0=10**9, shuffle=True):
    """THRESHOLD_HIT rows forming events of exactly ``sizes`` members at W_NS (every member within 50 ns of the event's
    first, 1 us between events), with few boards / channels / dts so that the member keys repeat."""
    from waveformanalysis_b200.dtypes import THRESHOLD_HIT_DTYPE

    rng = np.random.default_rng(seed)
    n = int(sum(sizes))
    ts = np.concatenate([t0 + i * 10**6 + rng.integers(0, 50_000, m) for i, m in enumerate(sizes)]) if n else np.zeros(0, np.int64)
    h = np.zeros(n, dtype=THRESHOLD_HIT_DTYPE)
    h["timestamp"] = ts
    h["position"] = rng.integers(4, 100, n)
    h["edge_start"] = h["position"] - rng.integers(0, 5, n)
    h["edge_end"] = h["position"] + rng.integers(1, 8, n)
    h["dt"] = rng.choice([2, 4], n)
    h["board"] = rng.integers(0, 3, n)
    h["channel"] = rng.integers(-2, 4, n)
    h["record_id"] = rng.integers(0, 50, n)
    h["height"] = rng.normal(size=n)
    if shuffle:
        h = h[rng.permutation(n)]
    return h


@pytest.mark.parametrize("sizes", [[1], [31], [32], [33], [1000], [5000], [1, 31, 32, 33, 1000, 5000, 2, 64, 1]])
@pytest.mark.parametrize("w", [W_NS, 0.0])
def test_hit_event_table_sizes(sizes, w):
    from oracle import np_oracle as O
    from waveformanalysis_b200 import ops

    h = _hits(sizes, seed=len(sizes) + sum(sizes))
    got, want = ops.group_hit_windows(h, w), O.group_hit_windows(h, w)
    if w == W_NS:
        assert np.array_equal(got["n_hits"], np.asarray(sizes, dtype=np.int64))
    _check_table(got, want)


def test_hit_event_table_ties_and_negative_windows():
    """Members tied on all six keys keep their input order; windows before time zero."""
    from oracle import np_oracle as O
    from waveformanalysis_b200 import ops

    for m in (20, 32, 33, 3000):
        h = _hits([m], seed=m)
        for f in ("position", "edge_start", "edge_end", "dt", "board", "channel", "record_id", "timestamp"):
            h[f] = h[f][0]
        h["height"] = np.arange(m)  # the input order, visible in the members
        got = ops.group_hit_windows(h, W_NS)
        assert got["members"].tolist() == list(range(m))
        _check_table(got, O.group_hit_windows(h, W_NS))
    mixed = _hits([40, 7, 40], seed=3, t0=-10**10)
    mixed = np.concatenate([mixed, mixed[::2]])  # exact duplicates among distinct rows
    assert (O.hit_abs_windows(mixed)[1] < 0).all()
    for w in (W_NS, 0.0):
        _check_table(ops.group_hit_windows(mixed, w), O.group_hit_windows(mixed, w))


def _table_of_windows(h, a0, a1, w):
    """The oracle's grouping and table (np_oracle.group_hit_windows) for given absolute windows."""
    ts, dtv, rid = h["timestamp"].astype(np.int64), h["dt"].astype(np.int32), h["record_id"].astype(np.int64)
    order = np.lexsort((rid, ts, dtv, a0))
    pm = np.maximum.accumulate(a1[order])
    new = np.r_[True, a0[order][1:] > pm[:-1] + w * 1e3]
    ev = np.empty(len(h), dtype=np.int64)
    ev[order] = np.cumsum(new) - 1
    n_ev = int(ev.max()) + 1
    members = np.lexsort((rid, ts, a0, dtv, h["channel"].astype(np.int16), h["board"].astype(np.int16), ev))
    tmin, tmax = np.full(n_ev, np.inf), np.full(n_ev, -np.inf)
    np.minimum.at(tmin, ev, a0)
    np.maximum.at(tmax, ev, a1)
    t_min, t_max = tmin.astype(np.int64), tmax.astype(np.int64)
    return dict(t_min=t_min, t_max=t_max, dt_ns=(t_max - t_min) / 1e3, n_hits=np.bincount(ev).astype(np.int64),
                offsets=np.r_[0, np.cumsum(np.bincount(ev))].astype(np.int64), members=members.astype(np.int64))


def test_hit_event_table_device_truncates_toward_zero():
    """Fractional windows on both sides of zero: t_min / t_max are truncated toward zero like numpy's astype; the packed
    member rows are the rows in member order."""
    from waveformanalysis_b200 import ops
    from waveformanalysis_b200.engine import upload

    h = _hits([3, 40, 1, 33, 5], seed=9, t0=-2_500_000)
    rng = np.random.default_rng(4)
    a0 = h["timestamp"].astype(np.float64) + rng.uniform(-3000.0, 0.0, len(h))
    a0[::4] = -rng.uniform(0.1, 0.9, len(a0[::4]))  # in (-1, 0): truncates to 0, floor would give -1
    a1 = a0 + rng.uniform(0.0, 9000.0, len(h))
    d_rows = upload(h)
    for w in (W_NS, 0.0, 2000.0):
        g = ops.group_rows_device(d_rows, len(h), 60, w, abs_start=upload(a0), abs_end=upload(a1))
        t = ops.hit_event_table_device(d_rows, len(h), 60, g)
        want = _table_of_windows(h, a0, a1, w)
        _check_table({k: t[k].cpu().numpy() for k in want}, want, keys=tuple(want))
        m = want["members"]
        assert t["member_rows"].cpu().numpy().tobytes() == h[m].tobytes()
    assert (_table_of_windows(h, a0, a1, W_NS)["t_min"] == 0).any()


def test_hit_event_table_empty():
    import torch

    from waveformanalysis_b200 import ops
    from waveformanalysis_b200.dtypes import HIT_MERGED_DTYPE

    got = ops.group_hit_windows(np.zeros(0, dtype=HIT_MERGED_DTYPE), W_NS)
    assert got["offsets"].tolist() == [0] and len(got["members"]) == 0
    rows = torch.empty(16, dtype=torch.uint8, device="cuda")
    t = ops.hit_event_table_device(rows, 0, 72, ops.group_rows_device(rows, 0, 72, W_NS))
    assert t["offsets"].cpu().numpy().tolist() == [0] and t["members"].numel() == 0 and t["member_rows"].numel() == 0


def test_hit_event_table_cross_record_rows():
    """hit_merged rows merged across records (sample_start = -1 at merge_gap_ns = 50) take their windows from their
    components."""
    from oracle import np_oracle as O
    from waveformanalysis_b200 import ops
    from waveformanalysis_b200.synth import make_v1725_blob

    blobs = [make_v1725_blob(n_events=300, seed=21, tie_every=3, lengths=(32, 200)), make_v1725_blob(n_events=200, seed=23, tie_every=2)]
    rec, pool = O.build_records_from_v1725(blobs, ["run_b0_seg0.bin", "run_b1_seg0.bin"], 4)
    h = O.threshold_hits(rec, pool, threshold=10.0)
    _, mg, cp = O.hit_merge(h, merge_gap_ns=50.0)
    assert (mg["sample_start"] < 0).sum() > 50
    for w in (W_NS, 0.0, 3000.0):
        _check_table(ops.group_hit_windows(mg, w, cp, h), O.group_hit_windows(mg, w, cp, h))


def test_hit_event_table_random_million():
    from oracle import np_oracle as O
    from waveformanalysis_b200 import ops
    from waveformanalysis_b200.dtypes import HIT_MERGED_DTYPE

    rng = np.random.default_rng(17)
    n = 1_000_000
    h = np.zeros(n, dtype=HIT_MERGED_DTYPE)
    h["timestamp"] = rng.integers(0, n * 400_000, n)
    h["timestamp"][rng.integers(0, n, n // 20)] = h["timestamp"][rng.integers(0, n, n // 20)]  # repeated timestamps
    h["position"] = rng.integers(10, 200, n)
    h["sample_start"] = h["position"] - rng.integers(0, 10, n)
    h["sample_end"] = h["position"] + rng.integers(1, 20, n)
    h["dt"] = rng.choice([2, 4], n)
    h["board"], h["channel"] = rng.integers(0, 4, n), rng.integers(0, 16, n)
    h["record_id"] = rng.integers(0, n // 4, n)
    for w in (W_NS, 3000.0):  # events of a few members, then mostly more than 32
        want = O.group_hit_windows(h, w)
        _check_table(ops.group_hit_windows(h, w), want)
    assert (want["n_hits"] > 32).mean() > 0.3 and want["n_hits"].max() > 100


# ---- sharded hit_merge -> hit_grouped table, P ranks simulated on one GPU --------------------------------------------------


def simulate(shards, *, span_ns, gap=50.0, w=W_NS, zone_rows=64):
    """What merge_group_sharded + hit_events_sharded compute on P ranks, with the gathers done in-process; returns the
    rank-order concatenation as ONE rank's result (so gather_hit_grouped_frame, without a process group, builds the
    frame) and the per-rank results."""
    import torch

    from waveformanalysis_b200 import distributed as D
    from waveformanalysis_b200.dtypes import THRESHOLD_HIT_DTYPE

    be = D.DeviceRows(THRESHOLD_HIT_DTYPE)
    counts = [n for _, n in shards]
    k = zone_rows
    while True:
        z = [be.head_tail(rows, k) for rows in shards]
        heads, tails = [a for a, _ in z], [b for _, b in z]
        wholes = [len(a) + len(b) == n for (a, b), n in zip(z, counts)]
        cuts, ok = D.plan_cuts(heads, tails, wholes, max(w, gap) * 1e3, span_ns * 1e3)
        if ok or all(wholes):
            break
        k *= 2
    assert ok
    shs = [be.merge_and_group(D.owned_hit_rows(be, rows, me, heads, tails, counts, cuts), gap, 10000.0, w) for me, rows in enumerate(shards)]
    per_rank = np.array([sh["n_events"] for sh in shs], dtype=np.int64)
    evs = []
    for me, sh in enumerate(shs):
        sh.update(event_base=int(per_rank[:me].sum()), events_per_rank=per_rank)
        evs.append(D.hit_events_sharded(sh, be))
    ev = {k_: torch.cat([e[k_] for e in evs]) for k_ in ("event_id", "t_min", "t_max", "dt_ns", "n_hits", "members", "member_rows")}
    ev["n_events"] = int(per_rank.sum())
    return ev, evs


def _device_hits(run, threshold):
    """The run's threshold hit rows on the device: one pass counts them, the second writes them into a buffer that fits."""
    import torch

    total = int(run.features_hits(threshold=threshold, features=False, hit_cap=1024)["total"].item())
    out = {"hits": torch.empty((total + 16) * 60, dtype=torch.uint8, device="cuda")}
    run.features_hits(threshold=threshold, features=False, hit_cap=total + 16, out=out)
    run.check()
    return out["hits"][: total * 60], total


def whole_run_frame(hits, gap=50.0, w=W_NS):
    from fakes import Ctx

    from waveformanalysis_b200 import ops
    from waveformanalysis_b200 import plugins as P

    _, merged, comps = ops.hit_merge(hits, merge_gap_ns=gap)
    ctx = Ctx({"time_window_ns": w}, {"hit_merged": merged, "hit_merged_components": comps, "hit_threshold": hits})
    return P.B200HitGroupedPlugin().compute(ctx, "run"), merged, comps


def assert_frame_equal(got, want):
    assert list(got.columns) == list(want.columns) and got.index.equals(want.index) and len(got) == len(want)
    for c in want.columns:
        assert got[c].dtype == want[c].dtype, c
        if want[c].dtype == object:
            assert all(a.dtype == b.dtype and np.array_equal(a, b) for a, b in zip(got[c], want[c])), c
        else:
            assert np.array_equal(got[c].to_numpy(), want[c].to_numpy()), c


def _check_sharded(shards, hits, span_ns, P):
    from waveformanalysis_b200 import distributed as D
    from waveformanalysis_b200 import ops

    ev, evs = simulate(shards, span_ns=span_ns)
    want, merged, comps = whole_run_frame(hits)
    assert len(want) > 100 and (want["n_hits"] > 1).any()
    assert_frame_equal(D.gather_hit_grouped_frame(ev), want)
    # the rank-order concatenation of the tables is the single-GPU table byte for byte
    table = ops.group_hit_windows(merged, W_NS, comps, hits)
    for k in ("event_id", "t_min", "t_max", "dt_ns", "n_hits"):
        assert ev[k].cpu().numpy().tobytes() == table[k].tobytes(), k
    return evs


@pytest.mark.parametrize("P", [1, 2, 3, 8])
def test_sharded_hit_events_from_synth_shards(P):
    from waveformanalysis_b200.dtypes import THRESHOLD_HIT_DTYPE
    from waveformanalysis_b200.engine import DeviceRun

    N, L, NCH, SEED = 24_000, 128, 16, 77
    full = DeviceRun.synth(N, L, NCH, seed=SEED)
    d_hits, total = _device_hits(full, 15.0)
    hits = d_hits.cpu().numpy().view(THRESHOLD_HIT_DTYPE)
    b = (np.arange(P + 1) * N) // P
    b[1:-1] += np.random.default_rng(P).integers(-50, 50, P - 1)  # uneven shards
    shards = [_device_hits(DeviceRun.synth(int(b[r + 1] - b[r]), L, NCH, seed=SEED, record_base=int(b[r])), 15.0) for r in range(P)]
    assert sum(n for _, n in shards) == total
    evs = _check_sharded(shards, hits, L * 2.0, P)
    assert all(e["n_events"] > 0 for e in evs)


@pytest.mark.parametrize("P", [1, 2, 3, 8])
def test_sharded_hit_events_from_v1725_shards(P):
    from waveformanalysis_b200 import ops
    from waveformanalysis_b200.dtypes import THRESHOLD_HIT_DTYPE
    from waveformanalysis_b200.engine import DeviceRun
    from waveformanalysis_b200.synth import make_v1725_blob

    blobs = {"run_b0_seg0.bin": make_v1725_blob(n_events=300, seed=21, tie_every=3, lengths=(32, 200)),
             "run_b1_seg0.bin": make_v1725_blob(n_events=250, seed=22, lengths=(64, 128)),
             "run_b2_seg0.bin": make_v1725_blob(n_events=200, seed=23, tie_every=2, t0=40_000)}
    rec, pool = ops.build_records_from_v1725(list(blobs.values()), list(blobs), 4)
    full = DeviceRun.from_host(rec, pool)
    d_hits, total = _device_hits(full, 10.0)
    hits = d_hits.cpu().numpy().view(THRESHOLD_HIT_DTYPE)
    b = (np.arange(P + 1) * len(rec)) // P
    shards = []
    for r in range(P):
        run = DeviceRun.from_host(rec[b[r]:b[r + 1]], pool, row_base=int(b[r]))
        run.lmax = full.lmax
        shards.append(_device_hits(run, 10.0))
    assert sum(n for _, n in shards) == total
    _, merged, _ = ops.hit_merge(hits, merge_gap_ns=50.0)
    assert (merged["sample_start"] < 0).any()
    _check_sharded(shards, hits, full.lmax * 4.0, P)
