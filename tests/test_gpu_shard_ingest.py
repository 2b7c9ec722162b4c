"""GPU: the kernels behind distributed.build_records_sharded_v1725, with P sources simulated on one GPU: the V1725
build with a global seq as record_id, split points at planned splitters, and the merge of every destination's runs,
checked byte for byte against the single-GPU build of all files."""

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

DT_NS = 4


def _blobs():
    from waveformanalysis_b200.synth import make_v1725_blob

    return {
        "run_b0_seg0.bin": make_v1725_blob(n_events=120, seed=11, tie_every=3, lengths=(32, 400)),
        "run_b1_seg0.bin": make_v1725_blob(n_events=100, seed=12, lengths=(64, 256)),
        "run_b1_seg1.bin": make_v1725_blob(n_events=100, seed=12, lengths=(64, 256)),  # equal keys up to seq
        "run_b2_seg0.bin": make_v1725_blob(n_events=80, seed=13, tie_every=2, t0=150_000),
        "run_b3_seg0.bin": make_v1725_blob(n_events=1, seed=14)[:30],  # no complete waveform
        "run_b5_seg0.bin": make_v1725_blob(n_events=2, seed=15, n_channels=2, lengths=(70_000, 70_010), t0=400),  # > 65 k samples
        "run_b0_seg1.bin": make_v1725_blob(n_events=90, seed=16, t0=300_000, lengths=(16, 800)),
        "run_b4_seg0.bin": make_v1725_blob(n_events=60, seed=17, n_channels=4, t0=60_000),
    }


def _local(names, blobs, files, counts, seq=True):
    """One source: its files (ascending list indices) built on the device with record_id = global seq."""
    from waveformanalysis_b200 import ops

    seq_base = np.cumsum(counts) - counts
    scans = [ops.v1725_scan(blobs[names[f]]) for f in files]
    up = ops.v1725_upload(scans, [names[f] for f in files])
    s = np.concatenate([seq_base[f] + np.arange(counts[f]) for f in files] or [np.zeros(0, np.int64)]).astype(np.int64)
    rows, pool, _ = ops.build_records_v1725_device(up, DT_NS, seq=s if seq else None)
    return rows, pool, up["n"]


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


def _counts(names, blobs):
    from waveformanalysis_b200 import ops

    return np.array([len(ops.v1725_scan(blobs[n])["channel"]) for n in names], dtype=np.int64)


def test_seq_build_differs_only_in_record_id():
    from waveformanalysis_b200 import distributed as D
    from waveformanalysis_b200 import ops

    blobs = _blobs()
    names = list(blobs)
    files = [0, 1, 2, 3, 6]
    scans = [ops.v1725_scan(blobs[names[f]]) for f in files]
    up = ops.v1725_upload(scans, [names[f] for f in files])
    n = up["n"]
    seq = 1000 + 3 * np.arange(n, dtype=np.int64)
    plain = _host_rows(ops.build_records_v1725_device(up, DT_NS)[0], n)
    with_seq = _host_rows(ops.build_records_v1725_device(up, DT_NS, seq=seq)[0], n)
    for f in plain.dtype.names:
        if f != "record_id":
            assert plain[f].tobytes() == with_seq[f].tobytes(), f
    assert np.array_equal(plain["record_id"], np.arange(n))
    board = np.concatenate([np.full(len(s["channel"]), ops.v1725_board_from_name(names[f])) for s, f in zip(scans, files)])
    ts = np.concatenate([s["timestamp"] for s in scans]) * DT_NS * 1000
    ch = np.concatenate([s["channel"] for s in scans])
    order = D.key_order(np.stack([ts, board, ch, np.arange(n)], axis=1))
    assert np.array_equal(with_seq["record_id"], seq[order])


@pytest.mark.parametrize("P", [1, 2, 3, 8])
def test_split_and_merge_equal_the_single_build(P):
    import torch

    from waveformanalysis_b200 import distributed as D
    from waveformanalysis_b200 import ops
    from waveformanalysis_b200.dtypes import RECORDS_DTYPE

    blobs = _blobs()
    names = list(blobs)
    counts = _counts(names, blobs)
    want_rec, want_pool = ops.build_records_from_v1725([blobs[n] for n in names], names, DT_NS)
    sources = [[f for f in range(len(names)) if f % P == p] for p in range(P)]  # not contiguous; P = 8: some sources empty
    locs = [_local(names, blobs, fs, counts) for fs in sources]
    host = [_host_rows(r, n) for r, _, n in locs]
    # splitters at the planned quantiles; one of them inside a run of equal timestamps
    s = D.SPLITTER_SAMPLES_PER_RANK * P
    ks, ws = [], []
    for h in host:
        pos, w = D.splitter_samples(len(h), s)
        ks.append(D.record_keys(h[pos]))
        ws.append(w)
    spl = D.plan_splitters(np.concatenate(ks), np.concatenate(ws), P)
    if P > 1:
        all_keys = D.record_keys(np.concatenate(host))
        all_keys = all_keys[D.key_order(all_keys)]
        tie = np.flatnonzero((all_keys[1:-1, 0] == all_keys[:-2, 0]) & (all_keys[1:-1, 0] == all_keys[2:, 0]))
        spl[0] = all_keys[1 + tie[len(tie) // 2]]
        spl = spl[D.key_order(spl)]
    cuts = []
    for (rows, _, n), h in zip(locs, host):
        c = ops.record_split_points(rows, n, spl)
        assert np.array_equal(c, D.lower_bounds(D.record_keys(h), spl))
        cuts.append(np.r_[0, c, n])
    lmax = int(want_rec["event_length"].max())
    lo = pb = 0
    shards_without_longest = 0
    for d in range(P):
        parts_r, parts_p, run_off = [], [], [0]
        for (rows, pool, n), h, c in zip(locs, host, cuts):
            a, b = int(c[d]), int(c[d + 1])
            pa = int(h["wave_offset"][a]) if a < n else int(pool.numel())
            pz = int(h["wave_offset"][b]) if b < n else int(pool.numel())
            parts_r.append(rows[a * 102: b * 102])
            parts_p.append(pool[pa:pz])
            run_off.append(run_off[-1] + b - a)
        rows_in, pool_in = torch.cat(parts_r), torch.cat(parts_p)
        m = run_off[-1]
        out_rows, out_pool, meta = ops.merge_record_runs(rows_in, pool_in, np.array(run_off), record_base=lo, pool_base=pb)
        got = out_rows[: m * 102].cpu().numpy()
        assert got.tobytes() == want_rec[lo:lo + m].tobytes(), d
        np_pool = out_pool.cpu().numpy().view(np.uint16)
        assert np.array_equal(np_pool, want_pool[pb:pb + len(np_pool)])
        assert np.array_equal(meta[: m * 48].cpu().numpy(), _unpack(want_rec[lo:lo + m]))
        if m:
            shard_rec = got.view(RECORDS_DTYPE)
            shards_without_longest += int(shard_rec["event_length"].max()) < lmax
            _check_fused(want_rec, want_pool, lo, m, pb, meta, out_pool, out_rows, lmax)
        lo += m
        pb += len(np_pool)
    assert lo == len(want_rec) and pb == len(want_pool)
    if P > 1:
        assert shards_without_longest >= 1


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


def test_merge_rejects_an_unsorted_run():
    from waveformanalysis_b200 import ops

    blobs = _blobs()
    names = list(blobs)
    counts = _counts(names, blobs)
    rows, pool, n = _local(names, blobs, [0, 1], counts)
    h = _host_rows(rows, n)
    swapped = h.copy()
    swapped[[3, 4]] = h[[4, 3]]
    from waveformanalysis_b200.engine import upload

    with pytest.raises(ValueError, match="strictly increasing"):
        ops.merge_record_runs(upload(swapped), pool, np.array([0, 10, n]), record_base=0, pool_base=0)
    # equal neighbours are not strictly increasing either
    dup = h.copy()
    dup[5] = h[4]
    with pytest.raises(ValueError, match="strictly increasing"):
        ops.merge_record_runs(upload(dup), pool, np.array([0, n]), record_base=0, pool_base=0)


def test_sharded_build_single_process_equals_the_single_build(tmp_path):
    from waveformanalysis_b200 import distributed as D
    from waveformanalysis_b200 import ops

    blobs = _blobs()
    paths = []
    for name, b in blobs.items():
        p = tmp_path / name
        p.write_bytes(b)
        paths.append(str(p))
    want_rec, want_pool = ops.build_records_from_v1725(list(blobs.values()), paths, DT_NS)
    res = D.build_records_sharded_v1725(paths, dt_ns=DT_NS)
    run = res["run"]
    assert run.records_rows[: run.n * 102].cpu().numpy().tobytes() == want_rec.tobytes()
    assert np.array_equal(run.pool.cpu().numpy().view(np.uint16), want_pool)
    assert run.lmax == int(want_rec["event_length"].max()) and res["n_total"] == len(want_rec) and res["record_base"] == 0
    assert np.array_equal(run.meta[: run.n * 48].cpu().numpy(), _unpack(want_rec))
