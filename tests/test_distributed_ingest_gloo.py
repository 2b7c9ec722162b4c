"""CPU: time shards built straight from V1725 files (distributed.build_records_sharded_v1725) over 2, 3 and 4 gloo
ranks with the host backend (the oracle's scan, the host key order), the splitter plan and the default file
assignment.  On GPUs the same plan / exchange code runs over NCCL with the device kernels (tools/dist_check.py
--source v1725)."""

import os
import socket
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DT_NS = 4


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


# ---- splitter plan -----------------------------------------------------------------------------------------------------


def _shard_sizes(local_keys, P):
    """Plan the splitters from every rank's samples the way build_records_sharded_v1725 does and count the shards."""
    from waveformanalysis_b200 import distributed as D

    s = D.SPLITTER_SAMPLES_PER_RANK * P
    sorted_keys = [k[D.key_order(k)] for k in local_keys]
    ks, ws = [], []
    for k in sorted_keys:
        pos, w = D.splitter_samples(len(k), s)
        ks.append(k[pos])
        ws.append(w)
    spl = D.plan_splitters(np.concatenate(ks), np.concatenate(ws), P)
    assert spl.shape == (P - 1, 4)
    cuts = sum(np.r_[0, D.lower_bounds(k, spl), len(k)] for k in sorted_keys)
    return np.diff(cuts), s


def _keys(ts, board=0, channel=None, seq0=0):
    n = len(ts)
    ch = np.arange(n) % 16 if channel is None else np.full(n, channel)
    return np.stack([np.asarray(ts, np.int64), np.full(n, board), ch, seq0 + np.arange(n)], axis=1).astype(np.int64)


@pytest.mark.parametrize("case", ["uniform", "skewed", "equal_ts", "empty_ranks", "tiny"])
@pytest.mark.parametrize("P", [2, 3, 8])
def test_plan_splitters_balances_the_shards(case, P):
    rng = np.random.default_rng(P * 100 + len(case))
    N = 200_000
    if case == "uniform":
        sizes = [N // P] * P
    elif case == "skewed":  # one rank holds 90 % of the records
        sizes = [int(0.9 * N)] + [int(0.1 * N) // (P - 1)] * (P - 1)
    elif case == "empty_ranks":
        sizes = [N // 2, N - N // 2] + [0] * (P - 2) if P > 2 else [N, 0]
    elif case == "tiny":  # fewer records than shards
        sizes = [P - 1] + [0] * (P - 1)
    else:
        sizes = [N // P] * P
    local, seq0 = [], 0
    for r, n in enumerate(sizes):
        ts = np.full(n, 7_000) if case == "equal_ts" else rng.integers(0, 10**9, n)
        local.append(_keys(ts, board=r % 3, seq0=seq0))
        seq0 += n
    counts, s = _shard_sizes(local, P)
    n_all = sum(sizes)
    assert counts.sum() == n_all
    assert np.all(np.abs(counts - n_all / P) <= 4 * n_all / s + 2 * P), (counts, n_all / P)


def test_lower_bounds_match_searchsorted():
    from waveformanalysis_b200 import distributed as D

    rng = np.random.default_rng(3)
    ts = np.sort(rng.integers(0, 50, 1000))  # many equal timestamps: board, channel and seq decide
    k = _keys(ts)
    k = k[D.key_order(k)]
    q = k[rng.integers(0, len(k), 40)]
    q[::3, 3] += 1  # keys between two records
    q = q[D.key_order(q)]
    flat = lambda a: (a[:, 0] * 1000 + a[:, 1] * 100 + a[:, 2]) * 10_000 + a[:, 3]  # noqa: E731  (exact at these sizes)
    assert np.array_equal(D.lower_bounds(k, q), np.searchsorted(flat(k), flat(q), side="left"))


def test_default_file_owners_are_contiguous_blocks():
    from waveformanalysis_b200 import distributed as D

    rng = np.random.default_rng(0)
    for sizes in ([], [5], [0, 0, 0], [10, 1, 1, 1, 1, 30, 2], rng.integers(0, 1000, 37).tolist(), [1] * 16):
        for P in (1, 2, 3, 4, 8):
            own = D.default_file_owners(sizes, P)
            assert len(own) == len(sizes)
            assert np.all((own >= 0) & (own < P)) and np.all(np.diff(own) >= 0)  # every index once, contiguous blocks
    own = D.default_file_owners([100, 100, 100, 100], 2)
    assert own.tolist() == [0, 0, 1, 1]


# ---- multi-rank build over gloo -------------------------------------------------------------------------------------------


def _write_files(tmp):
    from waveformanalysis_b200.synth import make_v1725_blob

    blobs = {
        "run_b0_seg0.bin": make_v1725_blob(n_events=40, seed=1, tie_every=3, lengths=(32, 200)),
        "run_b1_seg0.bin": make_v1725_blob(n_events=40, seed=2, lengths=(32, 96)),  # overlaps board 0 in time
        "run_b1_seg1.bin": make_v1725_blob(n_events=40, seed=2, lengths=(32, 96)),  # seg0's timestamps again: seq decides
        "run_b2_seg0.bin": make_v1725_blob(n_events=30, seed=3, tie_every=2, t0=50_000),
        "run_b3_seg0.bin": make_v1725_blob(n_events=1, seed=7)[:30],  # no complete waveform
        "run_b0_seg1.bin": make_v1725_blob(n_events=40, seed=5, t0=100_000, lengths=(16, 300)),
        "run_b4_seg0.bin": make_v1725_blob(n_events=25, seed=6, n_channels=4, t0=20_000),
    }
    paths = []
    for name, b in blobs.items():
        p = os.path.join(str(tmp), name)
        with open(p, "wb") as f:
            f.write(b)
        paths.append(p)
    return paths


def _ingest_worker(rank, world_size, port, paths, mine, q):
    sys.path.insert(0, ROOT)
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world_size), LOCAL_RANK=str(rank), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    import torch.distributed as dist

    from oracle import np_oracle as O
    from waveformanalysis_b200 import distributed as D

    dist.init_process_group("gloo", rank=rank, world_size=world_size)
    try:
        res = D.build_records_sharded_v1725(paths, dt_ns=DT_NS, mine=None if mine is None else mine[rank],
                                            backend=D.HostRecords(O.v1725_scan))
        run = res["run"]
        q.put((rank, "ok", run.records.tobytes(), run.pool.tobytes(), res["record_base"], run.pool_base, run.lmax, res["n_total"],
               res["records_per_rank"].tolist()))
    except ValueError as e:
        q.put((rank, "ValueError", str(e)))
    finally:
        dist.destroy_process_group()


def _run_ranks(world_size, paths, mine, timeout=240):
    import torch.multiprocessing as mp

    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_ingest_worker, args=(r, world_size, port, paths, mine, q)) for r in range(world_size)]
    for p in procs:
        p.start()
    res = sorted((q.get(timeout=timeout) for _ in procs), key=lambda r: r[0])
    for p in procs:
        p.join(timeout=60)
    return res


@pytest.mark.parametrize("world_size,mine", [
    (2, None),  # contiguous blocks by size
    (3, [[0, 2, 5], [1, 6], [3, 4]]),  # not contiguous; the two board-1 segments with equal timestamps on different ranks
    (4, [[2, 6], [], [0, 4, 5], [1, 3]]),  # rank 1 reads nothing
])
def test_sharded_v1725_build_equals_the_single_build(world_size, mine, tmp_path):
    from oracle import np_oracle as O
    from waveformanalysis_b200.dtypes import RECORDS_DTYPE

    paths = _write_files(tmp_path)
    want_rec, want_pool = O.build_records_from_v1725([open(p, "rb").read() for p in paths], paths, DT_NS)
    assert len(want_rec) > 1000 and np.any(np.diff(want_rec["timestamp"]) == 0)
    res = _run_ranks(world_size, paths, mine)
    assert all(r[1] == "ok" for r in res), res
    recs = [np.frombuffer(r[2], dtype=RECORDS_DTYPE) for r in res]
    assert np.concatenate(recs).tobytes() == want_rec.tobytes()
    rb = pb = 0
    for r, rec in zip(res, recs):
        pool = np.frombuffer(r[3], dtype=np.uint16)
        assert r[4] == rb and r[5] == pb, (r[0], r[4], rb, r[5], pb)
        assert np.array_equal(pool, want_pool[pb:pb + len(pool)])
        assert r[6] == int(want_rec["event_length"].max())
        assert r[7] == len(want_rec) and r[8] == [len(x) for x in recs]
        rb += len(rec)
        pb += len(pool)
    assert pb == len(want_pool)
    assert sum(len(x) > 0 for x in recs) >= 2


@pytest.mark.parametrize("mine", [[[0, 1, 2, 3], [3, 4, 5, 6]], [[0, 1, 2], [4, 5, 6]]], ids=["claimed_twice", "not_claimed"])
def test_bad_ownership_raises_on_every_rank(mine, tmp_path):
    paths = _write_files(tmp_path)
    res = _run_ranks(2, paths, mine, timeout=120)
    assert [r[1] for r in res] == ["ValueError", "ValueError"], res


def test_single_process_without_a_process_group(tmp_path):
    from oracle import np_oracle as O
    from waveformanalysis_b200 import distributed as D

    paths = _write_files(tmp_path)
    want_rec, want_pool = O.build_records_from_v1725([open(p, "rb").read() for p in paths], paths, DT_NS)
    res = D.build_records_sharded_v1725(paths, dt_ns=DT_NS, backend=D.HostRecords(O.v1725_scan))
    assert res["run"].records.tobytes() == want_rec.tobytes() and np.array_equal(res["run"].pool, want_pool)
    assert res["record_base"] == 0 and res["n_total"] == len(want_rec) and res["exchange_bytes"] == 0


def test_merge_rejects_an_unsorted_run():
    import torch

    from oracle import np_oracle as O
    from waveformanalysis_b200 import distributed as D
    from waveformanalysis_b200.synth import make_v1725_blob

    rec, pool = O.build_records_from_v1725([make_v1725_blob(n_events=5, seed=1)], ["x_b0.bin"], DT_NS)
    rows = torch.from_numpy(rec[::-1].copy().view(np.uint8).reshape(-1))
    with pytest.raises(ValueError, match="strictly increasing"):
        D.HostRecords(O.v1725_scan).merge(rows, torch.from_numpy(pool.view(np.uint8)), np.array([0, len(rec)]), 0, 0)
