"""GPU: the device event table (wfb_event_table behind ops.group_time_window) against the oracle, and the time-sharded
df -> df_events -> df_paired path with P ranks simulated on one GPU (the plan / zone / owned-row code of
distributed.events_sharded with the device backend), compared with the three B200 plugins run over the whole run."""

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

W_NS = 100.0


def _check_table(got, want):
    for k in ("event_id", "t_min", "t_max", "dt_ns", "n_hits", "offsets", "members"):
        assert got[k].dtype == want[k].dtype, k
        assert np.array_equal(got[k], want[k]), k


def _clustered(sizes, seed, shuffle=True, ch_range=(-5, 6)):
    """Events of exactly ``sizes`` members (every member within W of the first, gaps > W between events), random
    channels with repeats, rows in shuffled input order."""
    rng = np.random.default_rng(seed)
    ts, t0 = [], 10**9
    for m in sizes:
        ts.append(t0 + np.sort(rng.integers(0, int(W_NS * 1e3) + 1, m)))
        t0 += int(W_NS * 1e3) * 3 + int(rng.integers(1, 1000))
    ts = np.concatenate(ts).astype(np.int64) if sizes else np.zeros(0, np.int64)
    ch = rng.integers(*ch_range, len(ts)).astype(np.int16)
    if shuffle:
        p = rng.permutation(len(ts))
        ts, ch = ts[p], ch[p]
    return ts, ch


@pytest.mark.parametrize("sizes", [[], [1], [31], [32], [33], [5000], [1, 31, 32, 33, 5000, 2, 64, 1, 100]])
def test_event_table_sizes(sizes):
    from oracle import np_oracle as O
    from waveformanalysis_b200 import ops

    ts, ch = _clustered(sizes, seed=len(sizes) + sum(sizes))
    got, want = ops.group_time_window(ts, ch, W_NS), O.group_time_window(ts, ch, W_NS)
    assert len(got["t_min"]) == len(sizes) and np.array_equal(got["n_hits"], np.asarray(sizes, dtype=np.int64))
    _check_table(got, want)


def test_event_table_ties_and_one_giant_event():
    """Every timestamp equal (one event of the whole run, members by channel then input row), and a run within W."""
    from oracle import np_oracle as O
    from waveformanalysis_b200 import ops

    rng = np.random.default_rng(2)
    for ts in (np.full(20_000, 5_000, np.int64), np.sort(rng.integers(0, 90_000, 50_000)).astype(np.int64)):
        ch = rng.integers(-32768, 32767, len(ts)).astype(np.int16)
        ch[::7] = 3  # repeated channels
        _check_table(ops.group_time_window(ts, ch, W_NS), O.group_time_window(ts, ch, W_NS))


def _host_table(ts, ch):
    """The event table by a host lexsort over the device's event ids (the oracle's per-event loop is too slow at 1 M
    rows): members by (event, channel, sorted position), t_min / t_max of the first / last member."""
    from waveformanalysis_b200 import ops
    from waveformanalysis_b200.engine import upload

    n = len(ts)
    order = np.argsort(ts, kind="stable")
    ev, n_ev = ops.group_time_window_device(upload(ts[order]), n, W_NS)
    ev = ev.cpu().numpy()
    members = order[np.lexsort((np.arange(n), ch[order], ev))]
    counts = np.bincount(ev, minlength=n_ev)
    offsets = np.r_[0, np.cumsum(counts)].astype(np.int64)
    t_min, t_max = ts[members][offsets[:-1]], ts[members][offsets[1:] - 1]
    return dict(event_id=np.arange(n_ev, dtype=np.int64), t_min=t_min, t_max=t_max, dt_ns=(t_max - t_min) / 1e3,
                n_hits=counts.astype(np.int64), offsets=offsets, members=members.astype(np.int64))


def test_event_table_random_million():
    from waveformanalysis_b200 import ops

    rng = np.random.default_rng(7)
    n = 1_000_000
    ts = rng.integers(0, n * 60_000, n).astype(np.int64)  # ~1.7 members per event, events up to a few dozen
    ts[rng.integers(0, n, n // 20)] = ts[rng.integers(0, n, n // 20)]  # repeated timestamps
    ch = rng.integers(-4, 16, n).astype(np.int16)
    want = _host_table(ts, ch)
    assert want["n_hits"].max() > 8
    _check_table(ops.group_time_window(ts, ch, W_NS), want)
    dense = rng.integers(0, n * 2_000, n).astype(np.int64)  # events of ~50 members: the radix-sorted path
    want = _host_table(dense, ch)
    assert (want["n_hits"] > 32).mean() > 0.5
    _check_table(ops.group_time_window(dense, ch, W_NS), want)


def test_event_table_member_columns():
    """wfb_event_table's member-ordered columns equal the inputs gathered through the members."""
    import torch

    from waveformanalysis_b200 import ops
    from waveformanalysis_b200.engine import upload

    ts, ch = _clustered([3, 40, 1, 32, 33, 7], seed=5, shuffle=False)
    rng = np.random.default_rng(1)
    area, height = rng.normal(size=len(ts)).astype(np.float32), rng.normal(size=len(ts)).astype(np.float32)
    d_ts = upload(ts)
    ev, n_ev = ops.group_time_window_device(d_ts, len(ts), W_NS)
    t = ops.event_table_device(d_ts, ev, len(ts), n_ev, upload(ch), area=upload(area), height=upload(height))
    m = t["members"].cpu().numpy()
    assert np.array_equal(t["member_ts"].cpu().numpy(), ts[m]) and np.array_equal(t["member_channel"].cpu().numpy(), ch[m])
    assert np.array_equal(t["member_area"].cpu().numpy(), area[m]) and np.array_equal(t["member_height"].cpu().numpy(), height[m])
    e = ops.event_table_device(d_ts[:0], ev[:0], 0, 0, upload(ch)[:0])
    assert e["offsets"].cpu().numpy().tolist() == [0] and e["members"].numel() == 0
    assert isinstance(e["member_ts"], torch.Tensor)


def test_group_time_window_rejects_wide_channels():
    from waveformanalysis_b200 import ops

    with pytest.raises(ValueError, match="int16"):
        ops.group_time_window(np.arange(3, dtype=np.int64), np.array([0, 1, 70_000]), W_NS)


# ---- sharded df -> df_events -> df_paired, P ranks simulated on one GPU ---------------------------------------------------


def simulate(shards, *, gains=None, zone_rows=64, nch=3, start=6, pair_ns=80.0, w_ns=W_NS):
    """What df_sharded + events_sharded compute on P ranks, with the gathers done in-process; returns the rank-order
    concatenation as ONE rank's df / events dicts (so gather_event_frames, without a process group, builds the frames)."""
    from waveformanalysis_b200 import distributed as D

    be = D.DeviceEvents()
    loc = [be.df_local(run, feat, gains) for run, feat in shards]
    table = np.array([[n, *be.ts_ends(c, n)] for c, _, n in loc], dtype=np.int64)
    D.check_time_order(table)
    counts = table[:, 0]
    k = zone_rows
    while True:
        z = [D.event_zones(be, c, n, k) for c, _, n in loc]
        bounds, ok = D.plan_event_cuts([h for h, _, _ in z], [t for _, t, _ in z], [w for _, _, w in z], counts, w_ns * 1e3)
        if ok:
            break
        k *= 2
    heads, tails = [h for h, _, _ in z], [t for _, t, _ in z]
    evs = [D.owned_events(be, c, me, heads, tails, counts, bounds, time_window_ns=w_ns, pair_window_ns=pair_ns, n_channels=nch)
           for me, (c, _, _) in enumerate(loc)]
    import torch

    cat = lambda xs: torch.cat(xs) if xs else xs  # noqa: E731
    names = list(loc[0][0])
    df = dict(cols={k_: cat([c[k_] for c, _, _ in loc]) for k_ in names}, n=int(counts.sum()), with_pe=gains is not None,
              index=cat([o + int(counts[:r].sum()) for r, (_, o, _) in enumerate(loc)]))
    ev = {k_: cat([e[k_] for e in evs]) for k_ in ("t_min", "t_max", "dt_ns", "n_hits", "members", "member_ts", "member_channel",
                                                   "member_area", "member_height", "keep", "delta_t", "area_ch", "height_ch")}
    n_ev = sum(e["n_events"] for e in evs)
    ev.update(n_events=n_ev, event_id=torch.arange(n_ev, dtype=torch.int64, device="cuda"), n_channels=nch, start_channel_slice=start,
              pair_window_ns=pair_ns)
    return df, ev, bounds, k


def whole_run_frames(records, features, *, gains=None, nch=3, start=6, pair_ns=80.0, w_ns=W_NS):
    from fakes import Ctx

    from waveformanalysis_b200 import plugins as P

    conf = {"wave_source": "records"}
    if gains is not None:
        conf["gain_adc_per_pe"] = {f"{b}:{c}": g for (b, c), g in gains.items()}
    df = P.B200DataFramePlugin().compute(Ctx(conf, {"records": records, "basic_features": features}), "run")
    ev = P.B200GroupedEventsPlugin().compute(Ctx({"time_window_ns": w_ns}, {"df": df}), "run")
    paired = P.B200PairedEventsPlugin().compute(Ctx({"n_channels": nch, "start_channel_slice": start, "time_window_ns": pair_ns},
                                                    {"df_events": ev}), "run")
    return df, ev, paired


def assert_frames_equal(got, want):
    import pandas as pd

    pd.testing.assert_frame_equal(got[0], want[0])
    for g, w in zip(got[1:], want[1:]):
        assert list(g.columns) == list(w.columns) and g.index.equals(w.index) and len(g) == len(w)
        for c in w.columns:
            assert g[c].dtype == w[c].dtype, c
            if w[c].dtype == object:
                assert all(a.dtype == b.dtype and np.array_equal(a, b) for a, b in zip(g[c], w[c])), c
            else:
                assert np.array_equal(g[c].to_numpy(), w[c].to_numpy(), equal_nan=w[c].dtype.kind == "f"), c


def _features(run):
    res = run.features_hits(hits=False)
    run.check()
    return res["features"]


@pytest.mark.parametrize("P", [1, 2, 3, 8])
def test_sharded_events_from_synth_shards(P):
    from waveformanalysis_b200 import distributed as D
    from waveformanalysis_b200.dtypes import BASIC_FEATURES_DTYPE
    from waveformanalysis_b200.engine import DeviceRun

    N, L, NCH, SEED = 24_000, 128, 16, 77
    full = DeviceRun.synth(N, L, NCH, seed=SEED, with_rows=True)
    rec = full.records_to_host()
    feats = _features(full)[: N * 36].cpu().numpy().view(BASIC_FEATURES_DTYPE)
    b = (np.arange(P + 1) * N) // P
    b[1:-1] += np.random.default_rng(P).integers(-50, 50, P - 1)  # uneven shards
    shards = []
    for r in range(P):
        run = DeviceRun.synth(int(b[r + 1] - b[r]), L, NCH, seed=SEED, record_base=int(b[r]))
        shards.append((run, _features(run)))
    gains = {(0, c): 1.5 + c for c in range(0, NCH, 2)}
    w = 4000.0  # records ~3 us apart: events of one or two records, gaps wider than W now and then
    df, ev, bounds, _ = simulate(shards, gains=gains, w_ns=w, pair_ns=3000.0)
    assert sum(hi > lo for lo, hi in bounds) == P
    got = D.gather_event_frames(df, ev)
    assert_frames_equal(got, whole_run_frames(rec, feats, gains=gains, w_ns=w, pair_ns=3000.0))
    assert len(got[1]) > 1000 and (got[1]["n_hits"] > 1).any() and 0 < len(got[2]) < len(got[1])


@pytest.mark.parametrize("P", [1, 2, 3, 8])
def test_sharded_events_from_v1725_shards(P):
    from waveformanalysis_b200 import distributed as D
    from waveformanalysis_b200 import ops
    from waveformanalysis_b200.dtypes import BASIC_FEATURES_DTYPE
    from waveformanalysis_b200.engine import DeviceRun
    from waveformanalysis_b200.synth import make_v1725_blob

    blobs = {"run_b0_seg0.bin": make_v1725_blob(n_events=300, seed=21, tie_every=3, lengths=(32, 200)),
             "run_b1_seg0.bin": make_v1725_blob(n_events=250, seed=22, lengths=(64, 128)),
             "run_b2_seg0.bin": make_v1725_blob(n_events=200, seed=23, tie_every=2, t0=40_000)}
    rec, pool = ops.build_records_from_v1725(list(blobs.values()), list(blobs), 4)
    full = DeviceRun.from_host(rec, pool)
    feats = _features(full)[: len(rec) * 36].cpu().numpy().view(BASIC_FEATURES_DTYPE)
    b = (np.arange(P + 1) * len(rec)) // P
    shards = []
    for r in range(P):
        run = DeviceRun.from_host(rec[b[r]:b[r + 1]], pool, row_base=int(b[r]))
        run.lmax = full.lmax
        shards.append((run, _features(run)))
    df, ev, _, _ = simulate(shards, zone_rows=8)
    assert_frames_equal(D.gather_event_frames(df, ev), whole_run_frames(rec, feats))


def test_sharded_events_single_segment_and_time_order():
    """All rows within W: the boundaries are dropped and rank 0 owns the run; shards out of time order raise."""
    from types import SimpleNamespace

    from waveformanalysis_b200 import distributed as D
    from waveformanalysis_b200.dtypes import BASIC_FEATURES_DTYPE
    from waveformanalysis_b200.engine import DeviceRun, upload

    N, L = 3000, 64
    full = DeviceRun.synth(N, L, 4, seed=5, with_rows=True)
    rec = full.records_to_host()
    feats = _features(full)[: N * 36].cpu().numpy().view(BASIC_FEATURES_DTYPE).copy()
    feats["timestamp"] = 10**9 + np.sort(np.random.default_rng(0).integers(0, 50_000, N))
    rec["timestamp"] = feats["timestamp"]
    b = [0, 1000, 1000, 2000, N]  # an empty rank too
    shards = []
    for r in range(4):
        if b[r + 1] == b[r]:
            shards.append((SimpleNamespace(n=0, meta=None), None))
            continue
        run = DeviceRun.from_host(rec[b[r]:b[r + 1]], np.zeros(N * L, np.uint16), row_base=b[r])
        shards.append((run, upload(feats[b[r]:b[r + 1]])))
    df, ev, bounds, k = simulate(shards, zone_rows=16)
    assert bounds[0].tolist() == [0, N] and all(hi == lo for lo, hi in bounds[1:]) and k >= 500
    assert_frames_equal(D.gather_event_frames(df, ev), whole_run_frames(rec, feats))
    with pytest.raises(ValueError, match="not in time order"):
        simulate([shards[3], shards[0]])
