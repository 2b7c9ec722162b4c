"""CPU: time shards built from raw digitizer rows (distributed.build_records_sharded) over 2, 3 and 4 gloo ranks with the
host backend (the oracle's baseline mean, the host key order), checked against the oracle's single build of all groups.
One process group per world size runs every case in turn, so the error cases also show that no rank is left waiting in
a collective.  On GPUs the same code runs over NCCL with the device kernels (tools/dist_check.py --source raw)."""

import os
import socket
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DT_NS = 2
EPOCH_NS = 1_700_000_000_123_456_789


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _group(rng, n, width, board, channel, *, ts=None, span=10**9):
    """One per-channel group: rows over the whole run in time (unsorted, with repeats), int16 samples of both signs."""
    if ts is None:
        ts = rng.integers(-span // 50, span, n) // 1000 * 1000
        ts[::4] = ts[:1]  # equal timestamps inside the group
    samples = rng.integers(-3000, 3000, (n, width)).astype(np.int16)
    return (np.asarray(ts, np.int64), np.full(n, board, np.int16), np.full(n, channel, np.int16), samples)


def case_groups(case: str):
    """(groups, kwargs) of a case: the groups of the whole run, in group-index order."""
    rng = np.random.default_rng(sum(map(ord, case)))
    kw = dict(dt_ns=DT_NS)
    if case == "uniform":
        g = [_group(rng, n, 48, b, c) for n, b, c in ((90, 0, 0), (70, 0, 1), (110, 1, 0), (60, 1, 1), (80, 0, 0), (50, 2, 3))]
        g[4] = (g[0][0][:80].copy(),) + g[4][1:]  # board 0 channel 0 again with group 0's timestamps: only seq orders them
        kw.update(baseline_window=(5, 30), epoch_ns=EPOCH_NS)
    elif case == "mixed":
        g = [_group(rng, n, w, b, c) for n, w, b, c in ((90, 32, 0, 0), (70, 80, 0, 1), (110, 48, 1, 0), (60, 16, 1, 1), (40, 80, 0, 0))]
    elif case == "equal_ts":  # every row at one timestamp: board, channel and seq decide
        g = [_group(rng, n, w, b, c, ts=np.full(n, 123_000)) for n, w, b, c in ((30, 40, 1, 1), (25, 40, 0, 1), (35, 40, 1, 1), (20, 40, 0, 0))]
    elif case == "empty_groups":
        g = [_group(rng, n, w, 0, c) for n, w, c in ((0, 64, 0), (50, 24, 1), (0, 24, 2), (70, 24, 3), (0, 8, 4), (40, 24, 5))]
    elif case == "n_lt_p":  # fewer rows than ranks
        g = [_group(rng, n, 24, 0, c) for n, c in ((1, 0), (0, 1), (1, 2))]
    else:
        raise KeyError(case)
    return g, kw


# case -> which groups every rank claims, as a function of the world size P and the group count G
OWNERS = {
    "uniform": lambda P, G: [list(range(r * G // P, (r + 1) * G // P)) for r in range(P)],  # contiguous blocks
    "mixed": lambda P, G: [[g for g in range(G) if g % P == r] for r in range(P)],
    "no_group_rank": lambda P, G: [[g for g in range(G) if g % (P - 1) == r - (r > 1)] if r != 1 else [] for r in range(P)],
    "non_contiguous": lambda P, G: [[0, 2]] + [[g for g in range(G) if g not in (0, 2) and g % (P - 1) == r - 1] for r in range(1, P)],
    "equal_ts": lambda P, G: [[g for g in range(G) if (G - 1 - g) % P == r] for r in range(P)],
    "empty_groups": lambda P, G: [[g for g in range(G) if g % P == r] for r in range(P)],
    "n_lt_p": lambda P, G: [[g for g in range(G) if g % P == r] for r in range(P)],
}
DATA = {"no_group_rank": "uniform", "non_contiguous": "mixed"}  # cases that reuse another case's groups
ERRORS = ("claimed_twice", "not_claimed", "out_of_range", "dt_mismatch", "malformed")


def run_case(case: str, rank: int, P: int):
    """build_records_sharded on this rank for a case -> a picklable result."""
    from oracle import np_oracle as O
    from waveformanalysis_b200 import distributed as D

    backend = D.HostRecords(baseline_fn=O.baseline_mean)
    if case in ERRORS:
        g, kw = case_groups("mixed")
        G = len(g)
        mine = OWNERS["mixed"](P, G)[rank]
        if case == "claimed_twice" and rank == P - 1:
            mine = mine + [0]
        elif case == "not_claimed":
            mine = [x for x in mine if x != G - 1]
        elif case == "out_of_range" and rank == 0:
            mine = mine + [G]
        elif case == "dt_mismatch" and rank == 1:
            kw = dict(kw, dt_ns=DT_NS + 1)
        groups = {x: (g[x] if x < G else g[0]) for x in mine}
        if case == "malformed" and rank == P - 1:
            ts, b, c, s = groups[mine[0]]
            groups[mine[0]] = (ts[:-1], b, c, s)
    else:
        g, kw = case_groups(DATA.get(case, case))
        G = len(g)
        groups = {x: g[x] for x in OWNERS[case](P, G)[rank]}
    try:
        res = D.build_records_sharded(groups, n_groups=G, backend=backend, **kw)
    except ValueError as e:
        return ("ValueError", str(e))
    run = res["run"]
    return ("ok", run.records.tobytes(), run.pool.tobytes(), res["record_base"], run.pool_base, run.lmax, res["n_total"],
            res["records_per_rank"].tolist(), res["exchange_bytes"])


CASES = list(OWNERS) + list(ERRORS)


def _worker(rank, world_size, port, q):
    sys.path.insert(0, ROOT)
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world_size), LOCAL_RANK=str(rank), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    import torch.distributed as dist

    dist.init_process_group("gloo", rank=rank, world_size=world_size)
    try:
        for i, case in enumerate(CASES):
            try:
                q.put((case, rank, run_case(case, rank, world_size)))
            except Exception as e:  # report instead of leaving the test waiting; the group is unusable after this
                for c in CASES[i:]:
                    q.put((c, rank, ("error", repr(e))))
                break
    finally:
        dist.destroy_process_group()


@pytest.fixture(scope="module", params=[2, 3, 4], ids=lambda P: f"P{P}")
def ranks(request):
    """{case: [result of rank 0, ..., rank P - 1]} for one world size."""
    import torch.multiprocessing as mp

    P = request.param
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, P, port, q)) for r in range(P)]
    for p in procs:
        p.start()
    out: dict = {c: [None] * P for c in CASES}
    try:
        for _ in range(P * len(CASES)):
            case, rank, res = q.get(timeout=300)
            out[case][rank] = res
    finally:
        for p in procs:
            p.join(timeout=60)
    return P, out


def want_build(case: str):
    from oracle import np_oracle as O

    g, kw = case_groups(DATA.get(case, case))
    ts, b, c = (np.concatenate([x[k] for x in g]) for k in range(3))
    if len({x[3].shape[1] for x in g}) == 1:
        return O.build_records(ts, b, c, np.vstack([x[3] for x in g]), **kw)
    return O.build_records_ragged(ts, b, c, [x[3] for x in g], **kw)


@pytest.mark.parametrize("case", list(OWNERS))
def test_sharded_raw_build_equals_the_single_build(ranks, case):
    from waveformanalysis_b200.dtypes import RECORDS_DTYPE

    P, out = ranks
    want_rec, want_pool = want_build(case)
    res = out[case]
    assert all(r[0] == "ok" for r in res), res
    recs = [np.frombuffer(r[1], dtype=RECORDS_DTYPE) for r in res]
    assert np.concatenate(recs).tobytes() == want_rec.tobytes()
    rb = pb = 0
    for r, rec in zip(res, recs):
        pool = np.frombuffer(r[2], dtype=np.uint16)
        assert r[3] == rb and r[4] == pb
        assert np.array_equal(pool, want_pool[pb:pb + len(pool)])
        assert r[5] == (int(want_rec["event_length"].max()) if len(want_rec) else 0)
        assert r[6] == len(want_rec) and r[7] == [len(x) for x in recs]
        rb += len(rec)
        pb += len(pool)
    assert pb == len(want_pool)
    if len(want_rec) >= P:
        assert sum(len(x) > 0 for x in recs) >= 2
        assert sum(r[8] for r in res) > 0  # rows crossed the exchange


def test_the_cases_cover_what_they_name():
    """The properties the case names promise, on the data and the ownership the ranks use."""
    for P in (2, 3, 4):
        for case, owners in OWNERS.items():
            g, _ = case_groups(DATA.get(case, case))
            claims = sorted(x for o in owners(P, len(g)) for x in o)
            assert claims == list(range(len(g))), (case, P)
        assert OWNERS["no_group_rank"](P, 6)[1] == []
        assert OWNERS["non_contiguous"](P, 5)[0] == [0, 2]
    widths = {x[3].shape[1] for x in case_groups("mixed")[0]}
    assert len(widths) > 1 and len({x[3].shape[1] for x in case_groups("uniform")[0]}) == 1
    assert len(np.unique(np.concatenate([x[0] for x in case_groups("equal_ts")[0]]))) == 1
    assert any(len(x[0]) == 0 for x in case_groups("empty_groups")[0])
    assert sum(len(x[0]) for x in case_groups("n_lt_p")[0]) < 3


@pytest.mark.parametrize("case", ERRORS)
def test_bad_groups_raise_on_every_rank(ranks, case):
    P, out = ranks
    assert [r[0] for r in out[case]] == ["ValueError"] * P, out[case]


def test_single_process_without_a_process_group():
    from oracle import np_oracle as O
    from waveformanalysis_b200 import distributed as D

    for case in ("uniform", "mixed", "empty_groups"):
        g, kw = case_groups(case)
        want_rec, want_pool = want_build(case)
        res = D.build_records_sharded(dict(enumerate(g)), n_groups=len(g), backend=D.HostRecords(baseline_fn=O.baseline_mean), **kw)
        assert res["run"].records.tobytes() == want_rec.tobytes() and np.array_equal(res["run"].pool, want_pool), case
        assert res["record_base"] == 0 and res["n_total"] == len(want_rec) and res["exchange_bytes"] == 0
        assert set(res["timings"]) == {"h2d", "build", "splitters", "exchange", "merge"}
