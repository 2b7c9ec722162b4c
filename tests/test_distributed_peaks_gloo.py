"""CPU: the one collective of the time-sharded peaks leg (distributed.peaks_sharded) over 2 and 3 gloo ranks: the
count / options-digest gather gives every rank its bases and the totals, an empty rank included, and options that
differ between ranks, or an error on one rank, raise ValueError on every rank.  The per-shard chain itself
(peaks_local) runs on the GPU (tests/test_gpu_peaks_sharded.py)."""

import os
import socket
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _fake_local(counts):
    """A stand-in for peaks_local that returns this rank's row counts (or raises when they are None)."""

    def local(run, **_kw):
        if counts is None:
            raise ValueError("shard failed")
        n_hits, n_widths, n_labels = counts
        return dict(hits=np.zeros(0, np.uint8), n_hits=n_hits, widths=np.zeros(0, np.uint8), n_widths=n_widths, labels=None, n_labels=n_labels)

    return local


def _worker(rank, world_size, port, counts, opts, q):
    sys.path.insert(0, ROOT)
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world_size), LOCAL_RANK=str(rank), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    import torch.distributed as dist

    from waveformanalysis_b200 import distributed as D

    dist.init_process_group("gloo", rank=rank, world_size=world_size)
    try:
        sh = D.peaks_sharded(None, local_fn=_fake_local(counts[rank]), **opts[rank])
        q.put((rank, "ok", {k: v for k, v in sh.items() if k.endswith(("_base", "_per_rank", "_total"))}))
    except ValueError as e:
        q.put((rank, "ValueError", str(e)))
    finally:
        dist.destroy_process_group()


def _run_ranks(counts, opts, timeout=240):
    import torch.multiprocessing as mp

    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, len(counts), port, counts, opts, q)) for r in range(len(counts))]
    for p in procs:
        p.start()
    res = sorted((q.get(timeout=timeout) for _ in procs), key=lambda r: r[0])
    for p in procs:
        p.join(timeout=60)
    return res


OPTS = dict(filter_cfg={"filter_type": "SG", "sg_window_size": 11, "sg_poly_order": 2}, peak_opts={"height": 8.0, "width": 2},
            width_opts={"sampling_rate": 0.25}, s1s2_opts={"s1_width_range": (None, 40.0), "conflict_policy": "prefer_s1"})


@pytest.mark.parametrize("counts", [[(5, 4, 4), (7, 6, 6)], [(5, 4, 4), (0, 0, 0), (9, 3, 3)], [(0, 0, 0), (2, 1, 1), (0, 0, 0)]])
def test_bases_and_totals(counts):
    res = _run_ranks(counts, [OPTS] * len(counts))
    assert all(r[1] == "ok" for r in res), res
    c = np.array(counts)
    for rank, _, sh in res:
        for j, k in enumerate(("hit", "width", "label")):
            assert sh[f"{k}_base"] == int(c[:rank, j].sum())
            assert sh[f"{k}s_per_rank"].tolist() == c[:, j].tolist()
            assert sh[f"n_{k}s_total"] == int(c[:, j].sum())


@pytest.mark.parametrize("change", ["peak_opts", "filter_cfg", "s1s2_opts"])
def test_mismatched_options_raise_on_every_rank(change):
    other = dict(OPTS)
    other[change] = {"peak_opts": {"height": 9.0, "width": 2}, "filter_cfg": None, "s1s2_opts": {"conflict_policy": "prefer_s2"}}[change]
    res = _run_ranks([(1, 1, 1), (2, 2, 2), (3, 3, 3)], [OPTS, OPTS, other])
    assert [r[1] for r in res] == ["ValueError"] * 3, res
    assert all("same on every rank" in r[2] for r in res)


def test_an_error_on_one_rank_raises_on_every_rank():
    res = _run_ranks([(1, 1, 1), None], [OPTS, OPTS])
    assert [r[1] for r in res] == ["ValueError", "ValueError"], res
    assert res[1][2] == "shard failed" and "ranks [1]" in res[0][2]


def test_options_digest_is_stable():
    from waveformanalysis_b200 import distributed as D

    a = D.peaks_options_digest(OPTS["filter_cfg"], True, OPTS["peak_opts"], OPTS["width_opts"], OPTS["s1s2_opts"])
    assert a == D.peaks_options_digest(dict(OPTS["filter_cfg"]), True, dict(OPTS["peak_opts"]), OPTS["width_opts"], OPTS["s1s2_opts"])
    assert a != D.peaks_options_digest(OPTS["filter_cfg"], False, OPTS["peak_opts"], OPTS["width_opts"], OPTS["s1s2_opts"])


def test_single_process_without_a_process_group():
    from waveformanalysis_b200 import distributed as D

    sh = D.peaks_sharded(None, local_fn=_fake_local((4, 3, 0)), **OPTS)
    assert sh["hit_base"] == 0 and sh["n_hits_total"] == 4 and sh["n_widths_total"] == 3 and sh["hits_per_rank"].tolist() == [4]
