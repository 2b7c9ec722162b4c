"""GPU: the time-sharded wave_pool_filtered -> hit -> waveform_width -> s1_s2 leg (distributed.peaks_local), with P
shards simulated on one GPU.  Each shard holds its own records slice and its own pool slice
(``DeviceRun.from_host(rec[a:b], pool[o_a:o_b], pool_base=o_a, row_base=a)``, as the sharded ingest leaves them);
the rank-order concatenation of the shards' rows must equal the single-GPU plugin chain on the whole run byte for
byte."""

import os

import numpy as np
import pytest

from conftest import ROOT, assert_rows_match
from fakes import Ctx
from test_gpu_r2 import filtered_rows, st_from_records

pytestmark = pytest.mark.gpu

SG = {"filter_type": "SG", "sg_window_size": 11, "sg_poly_order": 2}
PEAKS = {"height": 8.0, "width": 2}
WIDTH = {"sampling_rate": 0.25}
WIDTH_1050 = {"sampling_rate": 0.25, "rise_low": 0.1, "rise_high": 0.5, "fall_high": 0.5, "fall_low": 0.1}
FLOATS_HIT = ("height", "integral", "edge_start", "edge_end")
FLOATS_WIDTH = ("rise_time", "fall_time", "total_width", "rise_time_samples", "fall_time_samples", "total_width_samples", "peak_height")


@pytest.fixture(scope="module")
def G():
    return np.load(os.path.join(ROOT, "tests", "golden", "r2_golden.npz"), allow_pickle=False)


@pytest.fixture(scope="module")
def P():
    from waveformanalysis_b200 import plugins

    return plugins


def run(plugin, data, config=None):
    return plugin.compute(Ctx(config, data), "run")


def shard_bounds(n: int, P: int, seed: int = 0) -> list:
    """Uneven bounds of P shards; with P >= 3 one shard (the second) is empty."""
    if P == 1:
        return [0, n]
    rng = np.random.default_rng(seed + P)
    cuts = np.sort(rng.choice(np.arange(1, n), size=P - 1, replace=False))
    if P >= 3:
        cuts[1] = cuts[0]
    return [0, *cuts.tolist(), n]


def make_shards(rec, pool, bounds):
    from waveformanalysis_b200.engine import DeviceRun

    out = []
    for a, b in zip(bounds[:-1], bounds[1:]):
        o_a = int(rec["wave_offset"][a]) if a < len(rec) else len(pool)
        o_b = int(rec["wave_offset"][b - 1]) + int(rec["event_length"][b - 1]) if b > a else o_a
        out.append(DeviceRun.from_host(rec[a:b], pool[o_a:o_b], pool_base=o_a, row_base=a))
    return out


def host_rows(t, n, dt):
    return t[: int(n) * dt.itemsize].cpu().numpy().view(dt).copy() if n else np.zeros(0, dtype=dt)


def cat_rows(parts, key, dt):
    return np.concatenate([host_rows(p[key], p["n_" + key], dt) for p in parts])


def same_bytes(got, want, what):
    assert got.dtype == want.dtype and len(got) == len(want), (what, got.dtype, want.dtype, len(got), len(want))
    assert got.tobytes() == want.tobytes(), what


def exact(got, want, what, floats):
    assert_rows_match(got, want, what=what, float_exact=floats)


def positive(rec, pool):
    """Positive pulses: mirror the 14-bit samples and the baselines around mid-scale, mark the records positive."""
    rec = rec.copy()
    rec["baseline"] = 16383.0 - rec["baseline"]
    rec["polarity"] = "positive"
    return rec, (16383 - pool.astype(np.int64)).astype(np.uint16)


def shard_features(shards):
    return [s.features_hits(hits=False)["features"] for s in shards]


# ---- c3: the reference's config-3 chain ----------------------------------------------------------------------------


@pytest.mark.parametrize("Pn", [1, 2, 3, 8])
def test_c3_golden_from_sg(P, G, Pn):
    """Starting from the reference's filtered pool, the shards reproduce c3_hit_records, c3_width and c3_width_1050."""
    from waveformanalysis_b200 import distributed as D, ops
    from waveformanalysis_b200.dtypes import HIT_DTYPE, WAVEFORM_WIDTH_DTYPE

    r, sg = G["c3_records"], G["c3_sg"]
    shards = make_shards(r, sg, shard_bounds(len(r), Pn))
    parts = [D.peaks_local(s, peak_opts=PEAKS, width_opts=WIDTH) for s in shards]
    hits = cat_rows(parts, "hits", HIT_DTYPE)
    widths = cat_rows(parts, "widths", WAVEFORM_WIDTH_DTYPE)
    w1050 = np.concatenate([host_rows(*ops.waveform_width_run(s, p["hits"], p["n_hits"], **WIDTH_1050), WAVEFORM_WIDTH_DTYPE)
                            for s, p in zip(shards, parts)])
    exact(hits, G["c3_hit_records"], "c3_hit_records", FLOATS_HIT)
    exact(widths, G["c3_width"], "c3_width", FLOATS_WIDTH)
    exact(w1050, G["c3_width_1050"], "c3_width_1050", FLOATS_WIDTH)
    st = st_from_records(r, G["c3_pool"])
    want_h = run(P.B200HitFinderPlugin(), {"records": r, "wave_pool_filtered": sg}, dict(PEAKS, use_filtered=True, wave_source="records"))
    data = {"hit": want_h, "filtered_waveforms": filtered_rows(st, sg), "st_waveforms": st}
    same_bytes(hits, want_h, "hit")
    same_bytes(widths, run(P.B200WaveformWidthPlugin(), data, dict(WIDTH, use_filtered=True)), "waveform_width")
    same_bytes(w1050, run(P.B200WaveformWidthPlugin(), data, dict(WIDTH_1050, use_filtered=True)), "waveform_width 10/50")


@pytest.mark.parametrize("Pn", [1, 2, 3, 8])
def test_c3_device_sg_chain_with_s1s2(P, G, Pn):
    """From the raw pool with the device SG filter: filtered pool, hit, waveform_width and s1_s2 equal the single-GPU
    plugin chain on the whole run byte for byte."""
    from waveformanalysis_b200 import distributed as D, ops
    from waveformanalysis_b200.dtypes import HIT_DTYPE, S1_S2_CLASSIFIER_DTYPE, WAVEFORM_WIDTH_DTYPE
    from waveformanalysis_b200.engine import DeviceRun

    r, p = G["c3_records"], G["c3_pool"]
    whole_sg = ops.filter_run_device(DeviceRun.from_host(r, p), SG).cpu().numpy()
    st = st_from_records(r, p)
    want_h = run(P.B200HitFinderPlugin(), {"records": r, "wave_pool_filtered": whole_sg}, dict(PEAKS, use_filtered=True, wave_source="records"))
    want_w = run(P.B200WaveformWidthPlugin(), {"hit": want_h, "filtered_waveforms": filtered_rows(st, whole_sg), "st_waveforms": st},
                 dict(WIDTH, use_filtered=True))
    feats = run(P.B200BasicFeaturesPlugin(), {"records": r, "wave_pool": p}, {"wave_source": "records"})
    q = np.quantile(want_w["total_width"], [0.3, 0.7])
    s1s2 = {"s1_width_range": (None, float(q[1])), "s2_width_range": (float(q[0]), None), "conflict_policy": "prefer_s2"}
    want_l = run(P.B200S1S2ClassifierPlugin(), {"waveform_width": want_w, "basic_features": feats}, s1s2)
    assert {1, 2} <= set(np.unique(want_l["label"]).tolist()), "both width ranges select rows"

    shards = make_shards(r, p, shard_bounds(len(r), Pn, seed=1))
    fs = shard_features(shards)
    parts = [D.peaks_local(s, filter_cfg=SG, features=f, peak_opts=PEAKS, width_opts=WIDTH, s1s2_opts=s1s2) for s, f in zip(shards, fs)]
    got_f = np.concatenate([host_rows(f, s.n, feats.dtype) for f, s in zip(fs, shards)])
    assert np.array_equal(got_f["height"], feats["height"]) and np.array_equal(got_f["area"], feats["area"])
    assert np.concatenate([x["filtered"].cpu().numpy() for x in parts]).tobytes() == whole_sg.tobytes()
    same_bytes(cat_rows(parts, "hits", HIT_DTYPE), want_h, "hit")
    same_bytes(cat_rows(parts, "widths", WAVEFORM_WIDTH_DTYPE), want_w, "waveform_width")
    same_bytes(cat_rows(parts, "labels", S1_S2_CLASSIFIER_DTYPE), want_l, "s1_s2")


@pytest.mark.parametrize("Pn", [2, 3])
def test_raw_16bit_route(P, G, Pn):
    """filter_cfg=None: hit on the raw pool (use_filtered=False) and widths on the st_waveforms rows."""
    from waveformanalysis_b200 import distributed as D
    from waveformanalysis_b200.dtypes import HIT_DTYPE, WAVEFORM_WIDTH_DTYPE

    r, p = G["c3_records"], G["c3_pool"]
    st = st_from_records(r, p)
    opts = {"height": 12.0, "width": 2}
    want_h = run(P.B200HitFinderPlugin(), {"records": r, "wave_pool": p}, dict(opts, use_filtered=False, wave_source="records"))
    want_w = run(P.B200WaveformWidthPlugin(), {"hit": want_h, "st_waveforms": st}, dict(WIDTH, use_filtered=False))
    assert len(want_w) > 0
    parts = [D.peaks_local(s, peak_opts=opts, width_opts=WIDTH) for s in make_shards(r, p, shard_bounds(len(r), Pn, seed=2))]
    assert all(x["filtered"] is None and x["labels"] is None for x in parts)
    same_bytes(cat_rows(parts, "hits", HIT_DTYPE), want_h, "hit")
    same_bytes(cat_rows(parts, "widths", WAVEFORM_WIDTH_DTYPE), want_w, "waveform_width")


# ---- synthetic shards of one run (DeviceRun.synth with record_base) --------------------------------------------------


def _positive_run(run):
    run.pool.copy_(16383 - run.pool)
    meta = run.meta.view(-1, 48)
    base = meta[:, 8:16].contiguous().view(torch_f64()).view(-1)
    meta[:, 8:16] = (16383.0 - base).view(meta.dtype).view(-1, 8)
    meta[:, 36] = 1  # WFB_POL_POSITIVE
    return run


def torch_f64():
    import torch

    return torch.float64


@pytest.mark.parametrize("filt", ["SG", "BW"])
@pytest.mark.parametrize("Pn", [2, 3, 8])
def test_synth_shards_equal_the_whole_run(filt, Pn):
    from waveformanalysis_b200 import distributed as D, ops
    from waveformanalysis_b200.dtypes import HIT_DTYPE, WAVEFORM_WIDTH_DTYPE
    from waveformanalysis_b200.engine import DeviceRun

    N, L, seed = 3000, 400, 77
    cfg = SG if filt == "SG" else {"filter_type": "BW", "sos": ops.butter_bandpass_sos(4, 0.01, 0.1, 0.25)}
    whole = _positive_run(DeviceRun.synth(N, L, 16, dt_ns=4, seed=seed))
    want = D.peaks_local(whole, filter_cfg=cfg, peak_opts=PEAKS, width_opts=WIDTH)
    assert want["n_widths"] > 100
    b = shard_bounds(N, Pn, seed=3)
    parts = [D.peaks_local(_positive_run(DeviceRun.synth(hi - lo, L, 16, dt_ns=4, seed=seed, record_base=lo)), filter_cfg=cfg, peak_opts=PEAKS,
                           width_opts=WIDTH) for lo, hi in zip(b[:-1], b[1:])]
    assert np.concatenate([x["filtered"].cpu().numpy() for x in parts]).tobytes() == want["filtered"].cpu().numpy().tobytes()
    same_bytes(cat_rows(parts, "hits", HIT_DTYPE), host_rows(want["hits"], want["n_hits"], HIT_DTYPE), "hit")
    same_bytes(cat_rows(parts, "widths", WAVEFORM_WIDTH_DTYPE), host_rows(want["widths"], want["n_widths"], WAVEFORM_WIDTH_DTYPE), "width")


# ---- ragged records: V1725 shards with mixed waveform sizes -----------------------------------------------------------


def _ragged_run(G):
    """The c3 records cut to random lengths of 8 to 800 samples (each keeps its first event_length samples) in a pool
    without gaps: V1725-like records of mixed waveform sizes with positive pulses."""
    r, p = G["c3_records"], G["c3_pool"]
    lens = np.random.default_rng(5).integers(8, 801, len(r)).astype(np.int32)
    rec = r.copy()
    rec["event_length"] = lens
    rec["wave_offset"] = np.r_[0, np.cumsum(lens)[:-1]]
    return rec, np.concatenate([p[o:o + n] for o, n in zip(r["wave_offset"], lens)])


@pytest.mark.parametrize("Pn", [1, 3, 8])
def test_ragged_shards_against_the_oracle(G, Pn):
    from oracle import np_oracle as O
    from waveformanalysis_b200 import distributed as D, ops
    from waveformanalysis_b200.dtypes import HIT_DTYPE, WAVEFORM_WIDTH_DTYPE
    from waveformanalysis_b200.engine import DeviceRun

    rec, pool = _ragged_run(G)
    assert len(np.unique(rec["event_length"])) > 10
    opts = {"height": 12.0, "width": 2}
    shards = make_shards(rec, pool, shard_bounds(len(rec), Pn, seed=4))
    whole_sg = ops.filter_run_device(DeviceRun.from_host(rec, pool), SG).cpu().numpy()
    for filt in (None, SG):
        parts = [D.peaks_local(s, filter_cfg=filt, peak_opts=opts, width_opts=WIDTH) for s in shards]
        hits = cat_rows(parts, "hits", HIT_DTYPE)
        src = pool if filt is None else whole_sg
        same_bytes(hits, ops.find_peaks_records(rec, src, **opts), f"hit {filt}")
        if filt is not None:
            assert np.concatenate([x["filtered"].cpu().numpy() for x in parts]).tobytes() == whole_sg.tobytes()
        waves = [src[o:o + n].view(np.int16) if filt is None else src[o:o + n] for o, n in zip(rec["wave_offset"], rec["event_length"])]
        want = O.waveform_width(hits, rec["record_id"], waves, **WIDTH)
        got = cat_rows(parts, "widths", WAVEFORM_WIDTH_DTYPE)
        assert len(want) > 0
        if filt is None:
            exact(got, want, "ragged widths int16", FLOATS_WIDTH)
        else:
            assert_rows_match(got, want, what="ragged widths float32")


# ---- edge cases -------------------------------------------------------------------------------------------------------


def test_shards_without_peaks_or_without_width_rows(P, G):
    """Shard 1 is flat (no peaks); in shard 2 every record rises over samples 5-9 to a plateau that ends at sample 50:
    one peak at the rising edge, below the mean of the first 50 samples, so no width row."""
    from waveformanalysis_b200 import distributed as D
    from waveformanalysis_b200.dtypes import HIT_DTYPE, WAVEFORM_WIDTH_DTYPE

    r, p = G["c3_records"].copy(), G["c3_pool"].copy()
    b = [0, 100, 200, len(r)]
    L = int(r["event_length"][0])
    r["baseline"][b[1]:] = np.rint(r["baseline"][b[1]:])
    rows = p.reshape(len(r), L)
    rows[b[1]:] = r["baseline"][b[1]:, None].astype(np.uint16)
    rows[b[2]:, 5:10] += np.array([40, 80, 120, 160, 200], dtype=np.uint16)
    rows[b[2]:, 10:50] += 200
    opts = {"height": 12.0, "width": 2}
    st = st_from_records(r, p)
    want_h = run(P.B200HitFinderPlugin(), {"records": r, "wave_pool": p}, dict(opts, use_filtered=False, wave_source="records"))
    want_w = run(P.B200WaveformWidthPlugin(), {"hit": want_h, "st_waveforms": st}, dict(WIDTH, use_filtered=False))
    parts = [D.peaks_local(s, peak_opts=opts, width_opts=WIDTH) for s in make_shards(r, p, b)]
    assert parts[0]["n_widths"] > 0 and parts[1]["n_hits"] == 0 and parts[2]["n_hits"] > 0 and parts[2]["n_widths"] == 0
    same_bytes(cat_rows(parts, "hits", HIT_DTYPE), want_h, "hit")
    same_bytes(cat_rows(parts, "widths", WAVEFORM_WIDTH_DTYPE), want_w, "waveform_width")


def test_hit_buffer_that_must_grow(G):
    from waveformanalysis_b200 import _lib, ops
    from waveformanalysis_b200.dtypes import HIT_DTYPE

    r, sg = G["c3_records"], G["c3_sg"]
    shard = make_shards(r, sg, [0, 150, len(r)])[1]
    assert shard.pool_base > 0
    job = ops.find_peaks_launch(shard, _lib.WAVE_REC_F32, shard.lmax, cap=1, **PEAKS)
    rows, n = ops.find_peaks_finish(job)
    assert n > 1 and rows.numel() >= n * HIT_DTYPE.itemsize
    want = ops.find_peaks_records(r, sg, **PEAKS)
    same_bytes(host_rows(rows, n, HIT_DTYPE), want[want["record_id"] >= 150], "grown buffer")


def test_hits_without_a_record_in_the_run_give_no_width_row(G):
    import torch

    from waveformanalysis_b200 import _lib, ops
    from waveformanalysis_b200.dtypes import HIT_DTYPE, WAVEFORM_WIDTH_DTYPE
    from waveformanalysis_b200.engine import DeviceRun

    r, sg = G["c3_records"], G["c3_sg"]
    shard = make_shards(r, sg, [0, 100, 250, len(r)])[1]
    hits = host_rows(*ops.find_peaks_device(shard, _lib.WAVE_REC_F32, shard.lmax, **PEAKS), HIT_DTYPE)
    want = host_rows(*ops.waveform_width_run(shard, torch.from_numpy(hits.view(np.uint8).copy()).cuda(), len(hits), **WIDTH), WAVEFORM_WIDTH_DTYPE)
    assert len(want) > 10
    bad = hits.copy()
    drop = np.zeros(len(hits), dtype=bool)
    drop[::3] = True
    bad["record_id"][0::6] = 99  # below row_base
    bad["record_id"][3::6] = 250 + np.arange(len(bad["record_id"][3::6]))  # at or past row_base + n
    got = host_rows(*ops.waveform_width_run(shard, torch.from_numpy(bad.view(np.uint8).copy()).cuda(), len(bad), **WIDTH), WAVEFORM_WIDTH_DTYPE)
    want_kept = host_rows(*ops.waveform_width_run(shard, torch.from_numpy(hits[~drop].view(np.uint8).copy()).cuda(), int((~drop).sum()), **WIDTH),
                          WAVEFORM_WIDTH_DTYPE)
    same_bytes(got, want_kept, "hits outside the run dropped")
    # a row in range whose record holds another record_id: no row either
    r2 = r[100:250].copy()
    r2["record_id"] += 10_000
    other = DeviceRun.from_host(r2, sg[100 * 800:250 * 800], pool_base=100 * 800, row_base=100)
    _, n = ops.waveform_width_run(other, torch.from_numpy(hits.view(np.uint8).copy()).cuda(), len(hits), **WIDTH)
    assert n == 0


def test_aos_wave_kind_with_a_pool_base_raises(G):
    from waveformanalysis_b200 import _lib, ops

    r, sg = G["c3_records"], G["c3_sg"]
    shard = make_shards(r, sg, [0, 100, len(r)])[1]
    with pytest.raises(ValueError, match="pool_base"):
        ops.find_peaks_device(shard, _lib.WAVE_AOS_F32, shard.lmax, **PEAKS)
