"""GPU: detectors whose channels are not configured alike, on time shards simulated on one GPU (uneven bounds, one
empty shard from P = 3 on): polarity from a channel map (ops.apply_polarity, the sharded builders' ``polarity``),
per-channel filters (ops.filter_run_device / distributed.peaks_local with ``filter_options`` and ``channel_config``)
and per-channel thresholds / fixed baselines (distributed.channel_rules), checked byte for byte against the single-GPU
plugins on the whole run; and one Butterworth configuration shared by every channel running the uniform kernel."""

import numpy as np
import pytest

from conftest import ATOL, RTOL
from fakes import Ctx
from test_gpu_peaks_sharded import PEAKS, WIDTH, cat_rows, make_shards, same_bytes, shard_bounds
from test_gpu_r2 import filtered_rows, st_from_records

pytestmark = pytest.mark.gpu

PARTS = [1, 2, 3, 8]
# mixed values, "unknown" entries, channels no record has, negative channel numbers
POLARITY = {**{(b, c): ("positive", "negative", "unknown")[(b + c) % 3] for b in range(3) for c in range(-3, 13)},
            (5, 1): "positive", (0, 40): "negative", (7, -2): "unknown"}
FOPTS = {"filter_type": "SG", "sg_window_size": 11, "sg_poly_order": 2, "lowcut": 0.01, "highcut": 0.1, "fs": 0.25, "filter_order": 4}
THR = 12.0


def channel_config():
    """A quarter of the channels BW order 4, some SG 41/3 (longer than the short records), some SG 5/4 (identity on
    records of at most 4 samples), the rest on the options; thresholds and fixed baselines on some channels.  Keys in
    all three forms the reference accepts."""
    ch = {}
    for b in range(3):
        for c in range(-3, 13):
            v = {}
            if c % 4 == 0:
                v["filter_type"] = "BW"
            elif c % 4 == 1:
                v.update(sg_window_size=41, sg_poly_order=3)
            elif (b + c) % 3 == 0:
                v.update(sg_window_size=5, sg_poly_order=4)
            if c % 3 == 1:
                v["threshold"] = 25.0
            if c % 5 == 2:
                v["fixed_baseline"] = 16383.0 - 8000.0 - 10.0 * (c % 16)
            if v:
                ch[(b, c) if c % 2 else f"{b}:{c}"] = v
    return {"channels": ch}


def want_polarity(rec, polarity):
    """plugins.records._apply_polarity's numpy assignment."""
    rec = rec.copy()
    for (b, c), v in polarity.items():
        if v != "unknown":
            rec["polarity"][(rec["board"] == b) & (rec["channel"] == c)] = v
    return rec


def channel_run(n=2400, L=400, seed=3):
    """Host records + pool of a seeded device run with positive pulses (samples and baselines mirrored around the
    14-bit mid-scale), boards 0-2 and channels -3..12."""
    from waveformanalysis_b200.dtypes import RECORDS_DTYPE
    from waveformanalysis_b200.engine import DeviceRun

    r = DeviceRun.synth(n, L, 16, dt_ns=4, seed=seed, with_rows=True)
    rec = r.records_rows.cpu().numpy().view(RECORDS_DTYPE).copy()
    pool = r.pool.cpu().numpy().view(np.uint16)
    rec["board"] = np.random.default_rng(seed).integers(0, 3, n)
    rec["channel"] -= 3
    rec["baseline"] = 16383.0 - rec["baseline"]
    return rec, (16383 - pool.astype(np.int64)).astype(np.uint16)


def ragged(rec, pool, seed=5, lo=2, hi=400):
    """Every record cut to a random length (it keeps its first samples), in a pool without gaps."""
    lens = np.random.default_rng(seed).integers(lo, hi + 1, len(rec)).astype(np.int32)
    out = rec.copy()
    out["event_length"] = lens
    out["wave_offset"] = np.r_[0, np.cumsum(lens)[:-1]]
    return out, np.concatenate([pool[o:o + k] for o, k in zip(rec["wave_offset"], lens)])


def meta_bytes(run):
    return run.meta[: run.n * 48].cpu().numpy().tobytes()


def rows_bytes(run):
    return run.records_rows[: run.n * 102].cpu().numpy().tobytes()


def check_polarity_shards(rec, pool, polarity, Pn, seed=0, clamp=None):
    from waveformanalysis_b200 import ops
    from waveformanalysis_b200.engine import DeviceRun

    want = want_polarity(rec, polarity)
    b = shard_bounds(len(rec), Pn, seed=seed)
    shards = make_shards(rec, pool, b)
    if clamp is not None:  # the same shards with an edge clamp in wfb_rec_meta.pad_
        for s, lo, hi in zip(shards, b[:-1], b[1:]):
            s2 = DeviceRun.from_host(rec[lo:hi], pool[s.pool_base:s.pool_base + s.pool_len], pool_base=s.pool_base, row_base=lo,
                                     clamp_lengths=clamp[lo:hi])
            s.meta, s.records_rows = s2.meta, s2.records_rows
    for s in shards:
        ops.apply_polarity(s, polarity)
    assert b"".join(rows_bytes(s) for s in shards) == want.tobytes()
    for s, lo, hi in zip(shards, b[:-1], b[1:]):
        ref = DeviceRun.from_host(want[lo:hi], pool[s.pool_base:s.pool_base + s.pool_len], clamp_lengths=None if clamp is None else clamp[lo:hi])
        assert meta_bytes(s) == meta_bytes(ref)
    return want


# ---- polarity ---------------------------------------------------------------------------------------------------------


@pytest.mark.parametrize("Pn", PARTS)
def test_polarity_on_shards(Pn):
    rec, pool = channel_run()
    want = check_polarity_shards(rec, pool, POLARITY, Pn, seed=Pn)
    pol = want["polarity"]
    assert {"positive", "negative", "unknown"} <= set(pol.tolist()) and (rec["channel"] < 0).any()


def test_polarity_ragged_shards():
    rec, pool = ragged(*channel_run(n=900))
    check_polarity_shards(rec, pool, POLARITY, 3, seed=7)


@pytest.mark.parametrize("size", [1, 4096])
def test_polarity_table_sizes(size):
    rec, pool = channel_run(n=1500)
    if size == 1:
        pol = {(1, 2): "negative"}
    else:
        pol = {(b, c): ("positive", "negative")[(b * 16 + c) % 2] for b in range(256) for c in range(-3, 13)}
        assert len(pol) == 4096
    check_polarity_shards(rec, pool, pol, 3, seed=size)


def test_polarity_keeps_the_edge_clamp():
    """A run from structured rows whose hit edges are clamped (wfb_meta_set_clamp): the clamp in pad_ survives."""
    rec, pool = channel_run(n=800, L=200)
    clamp = np.random.default_rng(1).integers(-1, 200, len(rec)).astype(np.int32)
    check_polarity_shards(rec, pool, POLARITY, 2, seed=9, clamp=clamp)


def test_polarity_values_are_checked():
    from waveformanalysis_b200 import ops

    rec, pool = channel_run(n=64)
    run = make_shards(rec, pool, [0, len(rec)])[0]
    for bad in ({(0, 1): "rawpos"}, {(0, 1): "Positive"}, {(0, 1): 1}, {0: "positive"}):
        with pytest.raises(ValueError):
            ops.apply_polarity(run, bad)
    assert rows_bytes(run) == rec.tobytes()


def test_sharded_v1725_build_with_polarity(tmp_path):
    from test_gpu_shard_ingest import DT_NS, _blobs

    from waveformanalysis_b200 import distributed as D, ops
    from waveformanalysis_b200.engine import DeviceRun

    blobs = _blobs()
    paths = []
    for name, b in blobs.items():
        (tmp_path / name).write_bytes(b)
        paths.append(str(tmp_path / name))
    rec, pool = ops.build_records_from_v1725(list(blobs.values()), paths, DT_NS)
    pol = {(b, c): ("positive", "negative", "unknown")[(b + c) % 3] for b in range(6) for c in range(16)}
    want = want_polarity(rec, pol)
    res = D.build_records_sharded_v1725(paths, dt_ns=DT_NS, polarity=pol)
    assert rows_bytes(res["run"]) == want.tobytes() and "polarity" in res["timings"]
    assert meta_bytes(res["run"]) == meta_bytes(DeviceRun.from_host(want, pool))


def test_sharded_raw_build_with_polarity():
    from test_gpu_shard_ingest_raw import DT_NS, MIXED, _groups

    from waveformanalysis_b200 import distributed as D
    from waveformanalysis_b200.engine import DeviceRun

    groups = _groups(MIXED, seed=9)
    pol = {(b, c): ("negative", "positive", "unknown")[(b + c) % 3] for b in range(2) for c in range(3)}
    plain = D.build_records_sharded(dict(enumerate(groups)), n_groups=len(groups), dt_ns=DT_NS)["run"]
    rec = plain.records_to_host()[: plain.n]
    want = want_polarity(rec, pol)
    assert (want["polarity"] != rec["polarity"]).any()
    run = D.build_records_sharded(dict(enumerate(groups)), n_groups=len(groups), dt_ns=DT_NS, polarity=pol)["run"]
    assert rows_bytes(run) == want.tobytes()
    assert meta_bytes(run) == meta_bytes(DeviceRun.from_host(want, plain.pool.cpu().numpy().view(np.uint16)))


# ---- per-channel filters ----------------------------------------------------------------------------------------------


def plugin_filtered(rec, pool, cc, opts=FOPTS):
    from waveformanalysis_b200.plugins import B200WavePoolFilteredPlugin

    return B200WavePoolFilteredPlugin().compute(Ctx({"wave_pool_filtered": dict(opts, channel_config=cc)}, {"records": rec, "wave_pool": pool}),
                                                "run")


@pytest.mark.parametrize("Pn", PARTS)
def test_per_channel_filters_on_ragged_shards(Pn):
    from waveformanalysis_b200 import ops

    rec, pool = ragged(*channel_run(n=1500), lo=2, hi=300)
    assert (rec["event_length"] < 41).any() and (rec["event_length"] <= 4).any()
    cc = channel_config()
    want = plugin_filtered(rec, pool, cc)
    shards = make_shards(rec, pool, shard_bounds(len(rec), Pn, seed=11))
    got = [ops.filter_run_device(s, filter_options=FOPTS, channel_config=cc, run_id="run").cpu().numpy() for s in shards]
    assert np.concatenate(got).tobytes() == want.tobytes()


def test_per_channel_filters_against_the_oracle():
    from oracle import np_oracle as O
    from waveformanalysis_b200 import ops
    from waveformanalysis_b200.channel_config import unique_channels
    from waveformanalysis_b200.plugins.filtering import channel_filter_configs

    rec, pool = ragged(*channel_run(n=240), lo=2, hi=120, seed=8)
    cc = channel_config()
    configs, default = channel_filter_configs(unique_channels(rec["board"], rec["channel"]), FOPTS, cc, "run")
    assert {c["filter_type"] for c in configs.values()} == {"BW", "SG"}
    shards = make_shards(rec, pool, [0, 100, 100, len(rec)])
    got = np.concatenate([ops.filter_run_device(s, filter_options=FOPTS, channel_config=cc, run_id="run").cpu().numpy() for s in shards])
    want = O.wave_pool_filtered(rec, pool, configs=configs, default=default)
    assert np.allclose(got, want, rtol=RTOL, atol=ATOL)


def test_filter_arguments_are_checked():
    from waveformanalysis_b200 import distributed as D, ops

    rec, pool = channel_run(n=64)
    run = make_shards(rec, pool, [0, len(rec)])[0]
    with pytest.raises(ValueError):
        D.peaks_local(run, filter_cfg={"filter_type": "SG", "sg_window_size": 11, "sg_poly_order": 2}, filter_options=FOPTS)
    with pytest.raises(ValueError, match="unknown filter options"):
        ops.filter_run_device(run, filter_options={"sg_window": 11})
    with pytest.raises(ValueError):
        ops.filter_run_device(run, filter_options=FOPTS, channel_config={"defaults": {"filter_type": "XX"}}, run_id="run")


# ---- the whole chain --------------------------------------------------------------------------------------------------


@pytest.fixture(scope="module")
def chain():
    """The single-GPU plugins on the whole run with the polarity applied to the host records."""
    from waveformanalysis_b200 import plugins as P

    rec, pool = channel_run(n=3000, L=400, seed=21)
    cc = channel_config()
    want = want_polarity(rec, POLARITY)
    data = {"records": want, "wave_pool": pool}
    feats = P.B200BasicFeaturesPlugin().compute(Ctx({"basic_features": {"wave_source": "records", "channel_config": cc}}, data), "run")
    hits_thr = P.B200ThresholdHitPlugin().compute(Ctx({"hit_threshold": {"wave_source": "records", "threshold": THR, "channel_config": cc}}, data),
                                                 "run")
    fpool = plugin_filtered(want, pool, cc)
    hit = P.B200HitFinderPlugin().compute(Ctx({"hit": dict(PEAKS, use_filtered=True, wave_source="records")},
                                              {"records": want, "wave_pool_filtered": fpool}), "run")
    st = st_from_records(want, pool)
    width = P.B200WaveformWidthPlugin().compute(Ctx({"waveform_width": dict(WIDTH, use_filtered=True)},
                                                    {"hit": hit, "filtered_waveforms": filtered_rows(st, fpool), "st_waveforms": st}), "run")
    q = np.quantile(width["total_width"], [0.3, 0.7])
    s1s2 = {"s1_width_range": (None, float(q[1])), "s2_width_range": (float(q[0]), None), "conflict_policy": "prefer_s2"}
    labels = P.B200S1S2ClassifierPlugin().compute(Ctx({"s1_s2": s1s2}, {"waveform_width": width, "basic_features": feats}), "run")
    return dict(rec=rec, pool=pool, cc=cc, feats=feats, hits_thr=hits_thr, fpool=fpool, hit=hit, width=width, labels=labels, s1s2=s1s2)


@pytest.mark.parametrize("Pn", PARTS)
def test_whole_chain_on_shards(chain, Pn):
    from waveformanalysis_b200 import distributed as D, ops
    from waveformanalysis_b200.dtypes import HIT_DTYPE, S1_S2_CLASSIFIER_DTYPE, WAVEFORM_WIDTH_DTYPE

    assert len(chain["hits_thr"]) > 100 and len(chain["width"]) > 100 and {1, 2} <= set(np.unique(chain["labels"]["label"]).tolist())
    shards = make_shards(chain["rec"], chain["pool"], shard_bounds(len(chain["rec"]), Pn, seed=13))
    feats, hits, parts = [], [], []
    for s in shards:
        ops.apply_polarity(s, POLARITY)
        rules = D.channel_rules(s, chain["cc"], run_id="run", threshold=THR)
        out = s.run_to_host(threshold=THR, rules=rules if len(rules) else None)
        feats.append(out["features"])
        hits.append(out["hits"])
        f_dev = s.features_hits(hits=False, rules=rules if len(rules) else None)["features"]
        parts.append(D.peaks_local(s, filter_options=FOPTS, channel_config=chain["cc"], run_id="run", features=f_dev, peak_opts=PEAKS,
                                   width_opts=WIDTH, s1s2_opts=chain["s1s2"]))
    same_bytes(np.concatenate(feats), chain["feats"], "basic_features")
    same_bytes(np.concatenate(hits), chain["hits_thr"], "hit_threshold")
    assert np.concatenate([p["filtered"].cpu().numpy() for p in parts]).tobytes() == chain["fpool"].tobytes()
    same_bytes(cat_rows(parts, "hits", HIT_DTYPE), chain["hit"], "hit")
    same_bytes(cat_rows(parts, "widths", WAVEFORM_WIDTH_DTYPE), chain["width"], "waveform_width")
    same_bytes(cat_rows(parts, "labels", S1_S2_CLASSIFIER_DTYPE), chain["labels"], "s1_s2")


def test_channel_rules_follow_the_plugins(chain):
    from waveformanalysis_b200 import distributed as D, ops

    run = make_shards(chain["rec"], chain["pool"], [0, len(chain["rec"])])[0]
    rules = D.channel_rules(run, chain["cc"], run_id="run", threshold=THR)
    assert len(rules) and set(rules["has_threshold"].tolist()) == {0, 1} and set(rules["has_fixed_baseline"].tolist()) == {0, 1}
    assert len(D.channel_rules(run, None, run_id="run", threshold=THR)) == 0
    fixed = D.channel_rules(run, None, run_id="run", threshold=THR, fixed_baseline=8000.0)
    assert len(fixed) == len(ops.shard_channels(run)) == 48 and fixed["has_fixed_baseline"].all()


# ---- one Butterworth configuration for every channel ------------------------------------------------------------------


def test_shared_bw_configuration_takes_the_uniform_kernel(monkeypatch):
    import torch
    from torch.profiler import ProfilerActivity, profile

    from waveformanalysis_b200 import ops
    from waveformanalysis_b200.channel_config import unique_channels
    from waveformanalysis_b200.engine import DeviceRun
    from waveformanalysis_b200.plugins.filtering import channel_filter_configs

    run = DeviceRun.synth(4000, 400, 16, dt_ns=4, seed=31, with_rows=True)
    rec = run.records_to_host()[: run.n]
    pool = run.pool_to_host()
    opts = dict(FOPTS, filter_type="BW")
    configs, default = channel_filter_configs(unique_channels(rec["board"], rec["channel"]), opts, None, "run")
    assert len(configs) == 16 and ops.filter_plan(run, configs)["n_cfg"] == 1
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        got = plugin_filtered(rec, pool, None, opts)
        torch.cuda.synchronize()
    names = [e.key for e in prof.key_averages()]
    assert any("bw_fast_kernel" in k and "true>" in k for k in names), [k for k in names if "bw_" in k]
    want = ops.filter_run_device(DeviceRun.from_host(rec, pool), {"filter_type": "BW", "sos": default["sos"]}).cpu().numpy()
    assert got.tobytes() == want.tobytes()
    monkeypatch.setenv("WFB_BW_UNIFORM", "0")  # the multi-configuration kernel gives the same bits
    assert ops.filter_pool(rec, pool, configs=configs, default=default).tobytes() == want.tobytes()
