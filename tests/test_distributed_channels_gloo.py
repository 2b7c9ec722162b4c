"""CPU: channel maps and per-channel options on time shards over 2 and 3 gloo ranks.  A sharded build from raw rows
with a polarity map (host backend) equals the oracle's single build with the numpy assignment of
plugins.records._apply_polarity; polarity maps, channel_config or filter_options that differ between ranks, and an
invalid polarity value on one rank, raise ValueError on every rank.  One process group per world size runs every case
in turn, so the error cases also show that no rank is left waiting in a collective."""

import os
import socket
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))

from test_distributed_ingest_raw_gloo import OWNERS, case_groups  # noqa: E402

POLARITY = {(0, 0): "positive", (0, 1): "negative", (1, 0): "unknown", (1, 1): "positive", (2, 3): "negative", (9, -4): "positive"}
FOPTS = {"filter_type": "SG", "sg_window_size": 11, "sg_poly_order": 2}
CC = {"channels": {(0, 1): {"filter_type": "BW", "lowcut": 0.01, "highcut": 0.1, "fs": 0.25}, "1:0": {"sg_window_size": 21}}}
PEAKS = dict(peak_opts={"height": 8.0, "width": 2}, width_opts={"sampling_rate": 0.25})


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def want_polarity(rec, polarity):
    rec = rec.copy()
    for (b, c), v in polarity.items():
        if v != "unknown":
            rec["polarity"][(rec["board"] == b) & (rec["channel"] == c)] = v
    return rec


def _fake_local(run, **_kw):
    return dict(hits=None, n_hits=0, widths=None, n_widths=0, labels=None, n_labels=0)


def run_case(case: str, rank: int, P: int):
    from oracle import np_oracle as O
    from waveformanalysis_b200 import distributed as D

    last = rank == P - 1
    if case.startswith("build"):
        g, kw = case_groups("mixed")
        groups = {x: g[x] for x in OWNERS["mixed"](P, len(g))[rank]}
        pol = dict(POLARITY)
        if case == "build_mismatch" and last:
            pol[(0, 0)] = "negative"
        elif case == "build_invalid" and rank == 0:
            pol[(0, 0)] = "rawpos"
        try:
            res = D.build_records_sharded(groups, n_groups=len(g), backend=D.HostRecords(baseline_fn=O.baseline_mean), polarity=pol, **kw)
        except ValueError as e:
            return ("ValueError", str(e))
        return ("ok", res["run"].records.tobytes(), "polarity" in res["timings"])
    opts = dict(filter_options=dict(FOPTS), channel_config=CC, run_id="run", **PEAKS)
    if case == "peaks_options" and last:
        opts["filter_options"]["sg_window_size"] = 13
    elif case == "peaks_channel_config" and last:
        opts["channel_config"] = {"channels": {(0, 1): {"filter_type": "SG"}}}
    elif case == "peaks_run_id" and last:
        opts["run_id"] = "other"
    try:
        D.peaks_sharded(None, local_fn=_fake_local, **opts)
    except ValueError as e:
        return ("ValueError", str(e))
    return ("ok",)


CASES = ["build_ok", "build_mismatch", "build_invalid", "peaks_ok", "peaks_options", "peaks_channel_config", "peaks_run_id"]


def _worker(rank, world_size, port, q):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
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


@pytest.fixture(scope="module", params=[2, 3], ids=lambda P: f"P{P}")
def ranks(request):
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


def test_sharded_build_with_polarity_equals_the_single_build(ranks):
    from oracle import np_oracle as O
    from waveformanalysis_b200.dtypes import RECORDS_DTYPE

    _, out = ranks
    res = out["build_ok"]
    assert all(r[0] == "ok" for r in res), res
    g, kw = case_groups("mixed")
    ts, b, c = (np.concatenate([x[k] for x in g]) for k in range(3))
    rec, _ = O.build_records_ragged(ts, b, c, [x[3] for x in g], **kw)
    want = want_polarity(rec, POLARITY)
    assert set(want["polarity"].tolist()) == {"positive", "negative", "unknown"}
    assert b"".join(r[1] for r in res) == want.tobytes()
    assert all(r[2] for r in res)
    assert np.frombuffer(b"".join(r[1] for r in res), dtype=RECORDS_DTYPE).shape == (len(rec),)


@pytest.mark.parametrize("case,msg", [("build_mismatch", "same on every rank"), ("build_invalid", "polarity"),
                                      ("peaks_options", "same on every rank"), ("peaks_channel_config", "same on every rank"),
                                      ("peaks_run_id", "same on every rank")])
def test_differing_or_invalid_arguments_raise_on_every_rank(ranks, case, msg):
    _, out = ranks
    res = out[case]
    assert all(r[0] == "ValueError" for r in res), res
    assert all(msg in r[1] for r in res), res


def test_equal_arguments_pass(ranks):
    _, out = ranks
    assert all(r == ("ok",) for r in out["peaks_ok"]), out["peaks_ok"]


def test_polarity_entries_check_values():
    from waveformanalysis_b200 import ops

    assert ops.polarity_entries({(0, -1): "negative", (0, 1): "positive", (1, 0): "unknown"}) == [(0, -1, "negative"), (0, 1, "positive"),
                                                                                                  (1, 0, "unknown")]
    for bad in ({(0, 1): "rawpos"}, {(0, 1): "POSITIVE"}, {(0, 1): None}, {"0:1": "positive"}, {(0, 1, 2): "positive"}):
        with pytest.raises(ValueError):
            ops.polarity_entries(bad)
    t = ops.polarity_table({(0, 1): "positive", (0, -1): "negative", (1, 0): "unknown", (70000, 0): "positive"})
    assert t["key"].tolist() == [1, 65535]  # unknown and out-of-range channels are left out; keys sorted as unsigned channels
    img = np.zeros(1, dtype=[("p", "U8")])
    img["p"] = "negative"
    assert t["image"][1].tobytes() == img.tobytes()


class _Channel:
    def __init__(self, board, channel):
        self.board, self.channel = board, channel


def test_channel_keyed_configurations_digest():
    from waveformanalysis_b200 import distributed as D

    def digest(cc):
        return D.peaks_options_digest(None, False, {}, {}, {}, filter_options=FOPTS, channel_config=cc, run_id="run")

    tuple_keyed = {"channels": {(0, 1): {"sg_window_size": 21}, (2, 3): {"filter_type": "BW"}}}
    string_keyed = {"channels": {"0:1": {"sg_window_size": 21}, "2:3": {"filter_type": "BW"}}}
    object_keyed = {"channels": {_Channel(2, 3): {"filter_type": "BW"}, _Channel(0, 1): {"sg_window_size": 21}}}
    assert digest(tuple_keyed) == digest(string_keyed) == digest(object_keyed)
    assert digest(tuple_keyed) != digest({"channels": {(0, 1): {"sg_window_size": 23}, (2, 3): {"filter_type": "BW"}}})
    assert digest(None) != digest(tuple_keyed)
    groups = {"groups": [{"channels": [(0, 1), "0:2"], "config": {"filter_type": "BW"}}]}
    assert digest(groups) == digest({"groups": [{"channels": [[0, 1], "0:2"], "config": {"filter_type": "BW"}}]})
