"""GPU: the kernels behind distributed.build_records_sharded on raw digitizer rows, with P sources simulated on one GPU:
the ragged build with a global seq as record_id, split points at planned splitters and the merge of every destination's
runs, checked byte for byte against the single-GPU builders of all groups (ops.build_records for one width,
ops.build_records_ragged for several), and the records plugin on seeded raw_arrays against the sharded build."""

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

DT_NS = 2


def _groups(widths, seed=5, rows=(150, 400)):
    """Per-channel groups of raw rows (timestamps_ps, boards, channels, int16 samples): every group spans the whole run in
    time, timestamps repeat inside and across groups, and a third of the rows carry a negative pulse."""
    rng = np.random.default_rng(seed)
    out = []
    for g, w in enumerate(widths):
        n = int(rng.integers(*rows)) if g != 2 else 0  # group 2 is empty
        ts = rng.integers(-2_000, 400_000, n) * 1000
        ts[::5] = 7_000_000
        s = (8000 + rng.integers(-4, 5, (n, w))).astype(np.int16)
        for i in range(0, n, 3):
            p = int(rng.integers(0, max(w - 12, 1)))
            s[i, p:p + 12] -= 150
        out.append((ts.astype(np.int64), np.full(n, g // 4, np.int16), np.full(n, g % 3, np.int16), s))
    return out


FIXED = [160] * 8
MIXED = [160, 96, 160, 24, 400, 160, 37, 96]


def _cat(groups, k):
    return np.concatenate([g[k] for g in groups])


def _single(groups, **kw):
    from waveformanalysis_b200 import ops

    ts, b, c = (_cat(groups, k) for k in range(3))
    if len({g[3].shape[1] for g in groups}) == 1:
        return ops.build_records(ts, b, c, np.vstack([g[3] for g in groups]), dt_ns=DT_NS, **kw)
    return ops.build_records_ragged(ts, b, c, [g[3] for g in groups], dt_ns=DT_NS, **kw)


def _host_rows(rows, n):
    from waveformanalysis_b200.dtypes import RECORDS_DTYPE

    return rows[: n * 102].cpu().numpy().view(RECORDS_DTYPE)


def _unpack(rows_np):
    import torch

    from waveformanalysis_b200 import _lib
    from waveformanalysis_b200.engine import _ptr, _stream, upload

    n = len(rows_np)
    meta = torch.empty(max(n, 1) * 48, dtype=torch.uint8, device="cuda")
    _lib.check(_lib.load().wfb_records_unpack(_ptr(upload(rows_np)), n, _ptr(meta), _stream()), "wfb_records_unpack")
    return meta[: n * 48].cpu().numpy()


@pytest.mark.parametrize("width", [24, 37, 800])
def test_single_block_ragged_build_equals_the_fixed_build(width):
    """One sample block through wfb_build_records_ragged gives the bytes of wfb_build_records: rows, pool and meta.  So
    the sharded build takes every width through the ragged entry point."""
    from waveformanalysis_b200 import ops

    g = _groups([width] * 5, seed=width)
    ts, b, c = (_cat(g, k) for k in range(3))
    s = np.vstack([x[3] for x in g])
    for kw in ({}, {"baseline_window": (3, 30), "epoch_ns": 1_700_000_000_000_000_000}):
        want_rec, want_pool = ops.build_records(ts, b, c, s, dt_ns=DT_NS, **kw)
        up = ops.raw_upload(ts, b, c, [s])
        rows, pool, meta = ops.build_records_ragged_device(up, dt_ns=DT_NS, meta=True, **kw)
        n = up["n"]
        assert rows[: n * 102].cpu().numpy().tobytes() == want_rec.tobytes()
        assert np.array_equal(pool.cpu().numpy().view(np.uint16), want_pool)
        assert np.array_equal(meta[: n * 48].cpu().numpy(), _unpack(want_rec))


def test_seq_build_differs_only_in_record_id():
    from waveformanalysis_b200 import distributed as D
    from waveformanalysis_b200 import ops

    g = _groups(MIXED)
    ts, b, c = (_cat(g, k) for k in range(3))
    up = ops.raw_upload(ts, b, c, [x[3] for x in g])
    n = up["n"]
    seq = 1000 + 3 * np.arange(n, dtype=np.int64)
    plain, _, m0 = ops.build_records_ragged_device(up, dt_ns=DT_NS, meta=True)
    with_seq, _, m1 = ops.build_records_ragged_device(up, dt_ns=DT_NS, meta=True, seq=seq)
    plain, with_seq = _host_rows(plain, n), _host_rows(with_seq, n)
    for f in plain.dtype.names:
        if f != "record_id":
            assert plain[f].tobytes() == with_seq[f].tobytes(), f
    assert np.array_equal(plain["record_id"], np.arange(n))
    order = D.key_order(np.stack([ts, b, c, np.arange(n)], axis=1))
    assert np.array_equal(with_seq["record_id"], seq[order])
    assert np.array_equal(m1[: n * 48].cpu().numpy(), _unpack(with_seq))
    with pytest.raises(ValueError):
        ops.build_records_ragged_device(up, dt_ns=DT_NS, seq=seq[:-1])


def _local(groups, owned, counts):
    """One source: its groups (ascending indices) built on the device with record_id = global seq."""
    from waveformanalysis_b200 import ops

    seq_base = np.cumsum(counts) - counts
    mine = [groups[f] for f in owned]
    cols = [np.concatenate([x[k] for x in mine] or [np.zeros(0, dt)]) for k, dt in enumerate((np.int64, np.int16, np.int16))]
    up = ops.raw_upload(*cols, [x[3] for x in mine])
    s = np.concatenate([seq_base[f] + np.arange(counts[f]) for f in owned] or [np.zeros(0, np.int64)]).astype(np.int64)
    rows, pool, _ = ops.build_records_ragged_device(up, dt_ns=DT_NS, seq=s)
    return rows, pool, up["n"]


_FULL = {}


def _check_fused(want_rec, want_pool, lo, m, pb, meta, pool, rows, lmax):
    """features_hits of the merged shard as a DeviceRun == the single-GPU rows of its records."""
    from waveformanalysis_b200 import engine

    key = (len(want_rec), len(want_pool))
    if key not in _FULL:
        _FULL.clear()
        _FULL[key] = engine.DeviceRun.from_host(want_rec, want_pool).run_to_host(threshold=15.0)
    full = _FULL[key]
    run = engine.DeviceRun(meta, pool, m, 0, lmax, records_rows=rows, pool_base=pb, row_base=lo)
    got = run.run_to_host(threshold=15.0)
    assert got["features"].tobytes() == full["features"][lo:lo + m].tobytes()
    fh = full["hits"][(full["hits"]["record_id"] >= lo) & (full["hits"]["record_id"] < lo + m)]
    assert len(fh) > 0 and got["hits"].tobytes() == fh.tobytes()


@pytest.mark.parametrize("widths", [FIXED, MIXED], ids=["fixed", "mixed"])
@pytest.mark.parametrize("P", [1, 2, 3, 8])
def test_split_and_merge_equal_the_single_build(P, widths):
    import torch

    from waveformanalysis_b200 import distributed as D
    from waveformanalysis_b200 import ops

    groups = _groups(widths)
    counts = np.array([len(g[0]) for g in groups], dtype=np.int64)
    want_rec, want_pool = _single(groups)
    sources = [[f for f in range(len(groups)) if f % P == p] for p in range(P)]  # not contiguous; P = 8: group 2 empty
    locs = [_local(groups, fs, counts) for fs in sources]
    host = [_host_rows(r, n) for r, _, n in locs]
    s = D.SPLITTER_SAMPLES_PER_RANK * P
    ks, ws = [], []
    for h in host:
        pos, w = D.splitter_samples(len(h), s)
        ks.append(D.record_keys(h[pos]))
        ws.append(w)
    spl = D.plan_splitters(np.concatenate(ks), np.concatenate(ws), P)
    if P > 1:  # one splitter inside the run of rows at the repeated timestamp
        all_keys = D.record_keys(np.concatenate(host))
        all_keys = all_keys[D.key_order(all_keys)]
        tie = np.flatnonzero(all_keys[:, 0] == 7_000_000)
        spl[0] = all_keys[tie[len(tie) // 2]]
        spl = spl[D.key_order(spl)]
    cuts = []
    for (rows, _, n), h in zip(locs, host):
        c = ops.record_split_points(rows, n, spl)
        assert np.array_equal(c, D.lower_bounds(D.record_keys(h), spl))
        cuts.append(np.r_[0, c, n])
    lmax = int(want_rec["event_length"].max())
    lo = pb = 0
    for d in range(P):
        parts_r, parts_p, run_off = [], [], [0]
        for (rows, pool, n), h, c in zip(locs, host, cuts):
            a, b = int(c[d]), int(c[d + 1])
            pa = int(h["wave_offset"][a]) if a < n else int(pool.numel())
            pz = int(h["wave_offset"][b]) if b < n else int(pool.numel())
            parts_r.append(rows[a * 102: b * 102])
            parts_p.append(pool[pa:pz])
            run_off.append(run_off[-1] + b - a)
        m = run_off[-1]
        out_rows, out_pool, meta = ops.merge_record_runs(torch.cat(parts_r), torch.cat(parts_p), np.array(run_off), record_base=lo,
                                                         pool_base=pb)
        assert out_rows[: m * 102].cpu().numpy().tobytes() == want_rec[lo:lo + m].tobytes(), d
        np_pool = out_pool.cpu().numpy().view(np.uint16)
        assert np.array_equal(np_pool, want_pool[pb:pb + len(np_pool)])
        assert np.array_equal(meta[: m * 48].cpu().numpy(), _unpack(want_rec[lo:lo + m]))
        if m:
            _check_fused(want_rec, want_pool, lo, m, pb, meta, out_pool, out_rows, lmax)
        lo += m
        pb += len(np_pool)
    assert lo == len(want_rec) and pb == len(want_pool)


@pytest.mark.parametrize("widths", [FIXED, MIXED], ids=["fixed", "mixed"])
def test_records_plugin_equals_the_sharded_build(widths):
    """B200RecordsPlugin / B200WavePoolPlugin on seeded raw_arrays (VX2730 columns: board, channel, timestamp at 0..2,
    samples from column 7) == distributed.build_records_sharded of the same groups (one process, device backend)."""
    from fakes import Ctx

    from waveformanalysis_b200 import distributed as D
    from waveformanalysis_b200.plugins.records import B200RecordsPlugin, B200WavePoolPlugin

    groups = _groups(widths, seed=9)
    raws = []
    for ts, b, c, s in groups:
        arr = np.zeros((len(ts), 7 + s.shape[1]), dtype=np.int64)
        arr[:, 0], arr[:, 1], arr[:, 2], arr[:, 7:] = b, c, ts, s
        raws.append(arr)
    ctx = Ctx({"dt": DT_NS}, {"raw_arrays": raws})
    rec = B200RecordsPlugin().compute(ctx, "run")
    pool = B200WavePoolPlugin().compute(ctx, "run")
    res = D.build_records_sharded(dict(enumerate(groups)), n_groups=len(groups), dt_ns=DT_NS)
    run = res["run"]
    assert res["n_total"] == len(rec) and run.lmax == int(rec["event_length"].max())
    assert run.records_rows[: run.n * 102].cpu().numpy().tobytes() == rec.tobytes()
    assert np.array_equal(run.pool.cpu().numpy().view(np.uint16), pool)
    assert np.array_equal(run.meta[: run.n * 48].cpu().numpy(), _unpack(rec))
