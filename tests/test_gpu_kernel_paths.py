"""The filter, width and find_peaks kernels against the numpy oracle on every dispatch path they select.

wfb_filter_pool, wfb_width_integral, wfb_waveform_width and wfb_find_peaks pick specialised code by record length,
16-byte alignment, section count, sample type and shared-memory fit.  Each case below is a seeded, hand-built run that
names the path it is meant to reach; the bars are the suite's: bit-exact where the kernel restates the reference's
arithmetic (WFB_BW_EXACT=1, the SG interior, width_integral, waveform_width on int16 rows, find_peaks positions and
edges), RTOL / ATOL where it evaluates the same formula differently (SG edges, the fast Butterworth kernel, float32
waveform_width rows)."""

import numpy as np
import pytest

from conftest import ATOL, RTOL, assert_rows_match

pytestmark = pytest.mark.gpu

FX_PEAKS = ("height", "edge_start", "edge_end")
FX_WW = ("rise_time", "fall_time", "total_width", "rise_time_samples", "fall_time_samples", "total_width_samples", "peak_height")
BANDS = ((0.01, 0.1, 0.5), (0.02, 0.2, 1.0), (0.05, 0.06, 0.5), (0.001, 0.45, 1.0))


@pytest.fixture(scope="module")
def ops():
    from waveformanalysis_b200 import ops

    return ops


@pytest.fixture(scope="module")
def O():
    from oracle import np_oracle

    return np_oracle


def make_records(lens, offs, *, board=0, channel=0, polarity="unknown", baseline=8000.0):
    from waveformanalysis_b200.dtypes import RECORDS_DTYPE

    n = len(lens)
    rec = np.zeros(n, dtype=RECORDS_DTYPE)
    rec["wave_offset"] = offs
    rec["event_length"] = lens
    rec["timestamp"] = np.arange(n, dtype=np.int64) * 10**6
    rec["dt"] = 2
    rec["board"] = board
    rec["channel"] = channel
    rec["record_id"] = np.arange(n)
    rec["baseline"] = baseline
    rec["baseline_upstream"] = np.nan
    rec["polarity"] = polarity
    return rec


def layout(lens, residues, gap=0):
    """Record offsets in a pool: record i starts at an element index = residues[i] (mod 8) and at least ``gap``
    elements behind the previous record (16-bit pools: residue 0 is a 16-byte aligned record)."""
    offs = np.zeros(len(lens), dtype=np.int64)
    cur = gap
    for i, (L, r) in enumerate(zip(lens, residues)):
        cur += (int(r) - cur) % 8
        offs[i] = cur
        cur += int(L) + gap
    return offs, cur + gap


def pulse_pool(rng, rec, pool_len, dtype, *, junk=12345):
    """Baseline 8000 + noise + one negative pulse per record; the gaps between records hold ``junk``."""
    pool = np.full(pool_len, junk, dtype=np.float64)
    for o, L in zip(rec["wave_offset"].tolist(), rec["event_length"].tolist()):
        t = np.arange(L)
        at = rng.integers(0, max(L, 1))
        pool[o:o + L] = 8000 + rng.normal(0, 3, L) - rng.uniform(20, 3000) * np.exp(-np.abs(t - at) / 5.0)
    if dtype == np.float32:
        return (pool + rng.uniform(-0.5, 0.5, pool_len)).astype(np.float32)
    return np.clip(np.round(pool), 0, 16383).astype(dtype)


def covered(rec, pool_len):
    m = np.zeros(pool_len, dtype=bool)
    for o, L in zip(rec["wave_offset"].tolist(), rec["event_length"].tolist()):
        m[o:o + max(L, 0)] = True
    return m


def check_filtered(got, want, rec, *, exact_mask=None, what=""):
    """Positions no record points at are exactly 0; ``exact_mask`` positions are bit-exact; the rest within the bar."""
    assert got.dtype == np.float32 and got.shape == want.shape, what
    cov = covered(rec, len(want))
    assert not np.any(got[~cov]), f"{what}: {np.count_nonzero(got[~cov])} nonzero samples outside the records"
    ok = np.isclose(got, want, rtol=RTOL, atol=ATOL, equal_nan=True)
    if not ok.all():
        bad = np.flatnonzero(~ok)
        raise AssertionError(f"{what}: {bad.size} samples out of tolerance, first at {bad[:5]}: got {got[bad[:5]]} want {want[bad[:5]]}")
    if exact_mask is not None:
        g, w = got[exact_mask], want[exact_mask]
        same = (g == w) | (np.isnan(g) & np.isnan(w))
        if not same.all():
            bad = np.flatnonzero(exact_mask)[~same]
            raise AssertionError(f"{what}: {bad.size} samples not bit-exact, first at {bad[:5]}: got {got[bad[:5]]} want {want[bad[:5]]}")


def sg_interior_mask(O, rec, pool_len, window_of):
    """Samples every record computes with the SG taps (not the edge fit): bit-exact against the oracle.  Records whose
    effective window is <= poly are copies, bit-exact as a whole."""
    m = np.zeros(pool_len, dtype=bool)
    for i, (o, L) in enumerate(zip(rec["wave_offset"].tolist(), rec["event_length"].tolist())):
        w0, poly = window_of(i)
        w = O.effective_sg_window(L, w0, poly)
        h = 0 if w is None else w // 2
        m[o + h:o + L - h] = True
    return m


# ---------------------------------------------------------------------------------------------------------------------
# wfb_filter_pool: Butterworth
# ---------------------------------------------------------------------------------------------------------------------
BW_LENGTHS = (15, 16, 17, 31, 32, 33, 47, 48, 49, 127, 128, 129, 255, 256, 257)


def bw_run(rng, O, sos, dtype, *, nan_record=None):
    """Every length of BW_LENGTHS plus padlen and padlen + 1 (the longest record copied / the shortest filtered), each
    at all eight start residues: the 16-sample vector forward loop runs only on 16-byte aligned uint16 records with
    L >= 16, the float4 stores of the backward loop only where y + o - 15 is 16-byte aligned.  Gaps of 3 between
    records."""
    pad = O.bw_padlen(sos)
    lens = np.repeat(np.array(sorted(set(BW_LENGTHS + (pad, pad + 1))), dtype=np.int32), 8)
    res = np.tile(np.arange(8), len(lens) // 8)
    offs, total = layout(lens, res, gap=3)
    rec = make_records(lens, offs)
    pool = pulse_pool(rng, rec, total, dtype)
    if nan_record is not None:  # a NaN sample reaches nothing outside its own record
        o, L = int(offs[nan_record]), int(lens[nan_record])
        pool[o + L // 2] = np.nan
    return rec, pool


# order -> kernel: 2 and 4 sections in one configuration -> the uniform kernel (coefficients as kernel parameters);
# 1 and 3 -> the non-uniform MAXS = 4 instance; 5 and 8 -> MAXS = 8; 9 and 16 -> MAXS = 16 (WFB_MAX_SOS_SECTIONS)
@pytest.mark.parametrize("order", [1, 2, 3, 4, 5, 8, 9, 16])
@pytest.mark.parametrize("dtype", [np.uint16, np.float32], ids=["u16", "f32"])
@pytest.mark.parametrize("mode", ["fast", "exact"])
def test_bw_single_config(ops, O, order, dtype, mode, monkeypatch):
    if mode == "exact":
        monkeypatch.setenv("WFB_BW_EXACT", "1")
    rng = np.random.default_rng(order * 10 + (dtype == np.float32))
    lo, hi, fs = BANDS[order % len(BANDS)]
    sos = ops.butter_bandpass_sos(order, lo, hi, fs)
    rec, pool = bw_run(rng, O, sos, dtype, nan_record=37 if dtype == np.float32 else None)
    cfg = {"filter_type": "BW", "sos": sos}
    got = ops.filter_pool(rec, pool, configs={}, default=cfg)
    want = O.wave_pool_filtered(rec, pool, configs={}, default=cfg)
    check_filtered(got, want, rec, exact_mask=covered(rec, len(pool)) if mode == "exact" else None, what=f"BW order {order} {mode}")


@pytest.mark.parametrize("order", [2, 4])
@pytest.mark.parametrize("dtype", [np.uint16, np.float32], ids=["u16", "f32"])
def test_bw_uniform_disabled(ops, O, order, dtype, monkeypatch):
    """WFB_BW_UNIFORM=0: a single 2- or 4-section configuration through the non-uniform kernel."""
    monkeypatch.setenv("WFB_BW_UNIFORM", "0")
    rng = np.random.default_rng(500 + order)
    sos = ops.butter_bandpass_sos(order, 0.02, 0.2, 1.0)
    rec, pool = bw_run(rng, O, sos, dtype)
    cfg = {"filter_type": "BW", "sos": sos}
    check_filtered(ops.filter_pool(rec, pool, configs={}, default=cfg), O.wave_pool_filtered(rec, pool, configs={}, default=cfg), rec,
                   what=f"BW order {order} non-uniform")


def test_bw_grid_stride(ops, O, monkeypatch):
    """More records than resident threads (SMs x 2048): every thread filters records rec, rec + n_threads, ... and
    reuses its scratch rows.  Fixed-length 16-byte aligned uint16 records: the uniform kernel's vector loops."""
    import torch

    sms = torch.cuda.get_device_properties(0).multi_processor_count
    n, L = int(1.5 * sms * 2048) + 37, 48
    rng = np.random.default_rng(7)
    rec = make_records(np.full(n, L, np.int32), np.arange(n, dtype=np.int64) * L)
    t = np.arange(L)
    at = rng.integers(0, L, size=(n, 1))
    pool = np.clip(np.round(8000 + rng.normal(0, 3, (n, L)) - rng.uniform(20, 3000, (n, 1)) * np.exp(-np.abs(t - at) / 5.0)), 0, 16383)
    pool = pool.astype(np.uint16).reshape(-1)
    sos = ops.butter_bandpass_sos(2, 0.01, 0.1, 0.5)
    cfg = {"filter_type": "BW", "sos": sos}
    want = O.bw_filter_rows(pool.reshape(n, L).astype(np.float32), sos).reshape(-1)
    check_filtered(ops.filter_pool(rec, pool, configs={}, default=cfg), want, rec, what="BW grid stride, fast")
    monkeypatch.setenv("WFB_BW_EXACT", "1")
    check_filtered(ops.filter_pool(rec, pool, configs={}, default=cfg), want, rec, exact_mask=np.ones(n * L, bool), what="BW grid stride, exact")


# ---------------------------------------------------------------------------------------------------------------------
# wfb_filter_pool: Savitzky-Golay
# ---------------------------------------------------------------------------------------------------------------------
SG_LENGTHS = (1, 2, 3, 4, 5, 7, 8, 9, 15, 16, 17, 31, 32, 33, 47, 48, 49, 100, 255, 256, 257)


# h = window // 2: h 1..8 on 16-byte aligned uint16 records with L >= 32 take the sg_block8 fast interior, h >= 9, other
# residues, float32 pools and shorter records the scalar loop; even windows are forced odd; window <= poly is a copy
@pytest.mark.parametrize("window,poly", [(3, 1), (5, 2), (11, 2), (17, 3), (19, 2), (21, 4), (31, 3), (10, 2), (4, 3)])
@pytest.mark.parametrize("dtype", [np.uint16, np.float32], ids=["u16", "f32"])
def test_sg_single_config(ops, O, window, poly, dtype):
    rng = np.random.default_rng(window * 10 + poly)
    lens = np.repeat(np.array(SG_LENGTHS, dtype=np.int32), 8)
    offs, total = layout(lens, np.tile(np.arange(8), len(SG_LENGTHS)), gap=2)
    rec = make_records(lens, offs)
    pool = pulse_pool(rng, rec, total, dtype)
    if dtype == np.float32:
        pool[int(offs[-20]) + 100] = np.nan
    cfg = {"filter_type": "SG", "sg_window_size": window, "sg_poly_order": poly}
    got = ops.filter_pool(rec, pool, configs={}, default=cfg)
    want = O.wave_pool_filtered(rec, pool, configs={}, default=cfg)
    check_filtered(got, want, rec, exact_mask=sg_interior_mask(O, rec, total, lambda i: (window, poly)), what=f"SG {window}/{poly}")


# ---------------------------------------------------------------------------------------------------------------------
# wfb_filter_pool: per-channel configurations in one call
# ---------------------------------------------------------------------------------------------------------------------
def mixed_configs(ops):
    bw = lambda order, band: {"filter_type": "BW", "sos": ops.butter_bandpass_sos(order, *BANDS[band])}  # noqa: E731
    sg = lambda w, p: {"filter_type": "SG", "sg_window_size": w, "sg_poly_order": p}  # noqa: E731
    return {(0, 0): sg(3, 1), (0, 1): sg(5, 2), (0, 2): sg(17, 3), (0, 3): sg(31, 3), (0, 4): sg(10, 2), (0, 5): sg(4, 3),
            (0, 6): bw(1, 0), (0, 7): bw(2, 1), (1, 0): bw(4, 2), (1, 1): bw(9, 3), (1, 2): sg(21, 4), (1, 3): bw(5, 0)}


@pytest.mark.parametrize("dtype", [np.uint16, np.float32], ids=["u16", "f32"])
@pytest.mark.parametrize("mode", ["fast", "exact"])
def test_filter_mixed_channels(ops, O, dtype, mode, monkeypatch):
    """SG windows 3-31 and BW orders 1-9 per (board, channel) in one call, plus channels on the default: every BW record
    runs in the largest compiled instance (MAXS = 16 for the 9-section channel), every SG record with its own table."""
    if mode == "exact":
        monkeypatch.setenv("WFB_BW_EXACT", "1")
    rng = np.random.default_rng(11 + (dtype == np.float32))
    configs = mixed_configs(ops)
    default = {"filter_type": "SG", "sg_window_size": 11, "sg_poly_order": 2}
    keys = list(configs) + [(2, 0), (2, 1)]
    n = 600
    lens = rng.choice(np.array(SG_LENGTHS + (60, 61, 62, 63, 64, 65, 66, 67, 70, 150, 800)), size=n).astype(np.int32)
    offs, total = layout(lens, rng.integers(0, 8, size=n), gap=1)
    which = rng.integers(0, len(keys), size=n)
    rec = make_records(lens, offs, board=[keys[k][0] for k in which], channel=[keys[k][1] for k in which])
    pool = pulse_pool(rng, rec, total, dtype)
    got = ops.filter_pool(rec, pool, configs=configs, default=default)
    want = O.wave_pool_filtered(rec, pool, configs=configs, default=default)

    def window_of(i):
        c = configs.get(keys[which[i]], default)
        return (c["sg_window_size"], c["sg_poly_order"]) if c["filter_type"] == "SG" else (0, 0)

    exact = sg_interior_mask(O, rec, total, window_of)
    is_bw = np.array([configs.get(keys[k], default)["filter_type"] == "BW" for k in which])
    bw_mask = covered(rec[is_bw], total)
    exact = (exact & ~bw_mask) | (bw_mask if mode == "exact" else False)
    check_filtered(got, want, rec, exact_mask=exact, what=f"mixed {mode}")


# ---------------------------------------------------------------------------------------------------------------------
# ops.filter_run_device on a ragged device-resident run
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("window,poly,dtype", [(11, 2, np.uint16), (7, 3, np.uint16), (9, 2, np.float32)], ids=["11-2-u16", "7-3-u16", "9-2-f32"])
def test_filter_run_device_ragged(ops, O, window, poly, dtype):
    """Records shorter than the window are filtered with their own effective window min(window, L) (forced odd), and
    left unchanged where that is <= poly - not with the taps of the longest record's window."""
    from waveformanalysis_b200 import engine

    rng = np.random.default_rng(window + poly)
    lens = np.array(list(range(1, 16)) * 3 + [40, 800, 33, 7, 800], dtype=np.int32)
    rng.shuffle(lens)
    offs, total = layout(lens, rng.integers(0, 8, size=len(lens)), gap=1)
    rec = make_records(lens, offs)
    pool = pulse_pool(rng, rec, total, dtype)
    cfg = {"filter_type": "SG", "sg_window_size": window, "sg_poly_order": poly}
    run = engine.DeviceRun.from_host(rec, pool, explicit_dt=1)
    got = ops.filter_run_device(run, cfg).cpu().numpy()
    want = O.wave_pool_filtered(rec, pool, configs={}, default=cfg)
    check_filtered(got, want, rec, exact_mask=sg_interior_mask(O, rec, total, lambda i: (window, poly)), what=f"filter_run_device {window}/{poly}")


def test_filter_run_device_fixed_length(ops, O):
    """A device-synthesised fixed-length run (the benchmark's input): one table for every record."""
    from waveformanalysis_b200 import engine
    from waveformanalysis_b200.dtypes import RECORDS_DTYPE

    n, L = 300, 800
    run = engine.DeviceRun.synth(n, L, 8, seed=5, with_rows=True)
    assert run.lmin == L
    rec = run.records_rows.cpu().numpy().view(RECORDS_DTYPE)
    pool = run.pool.cpu().numpy().view(np.uint16)
    for cfg in ({"filter_type": "SG", "sg_window_size": 11, "sg_poly_order": 2},
                {"filter_type": "BW", "sos": ops.butter_bandpass_sos(4, 0.01, 0.1, 0.25)}):
        got = ops.filter_run_device(run, cfg).cpu().numpy()
        want = O.wave_pool_filtered(rec, pool, configs={}, default=cfg)
        exact = sg_interior_mask(O, rec, n * L, lambda i: (11, 2)) if cfg["filter_type"] == "SG" else None
        check_filtered(got, want, rec, exact_mask=exact, what=f"synth {cfg['filter_type']}")


# ---------------------------------------------------------------------------------------------------------------------
# wfb_width_integral
# ---------------------------------------------------------------------------------------------------------------------
# numpy's pairwise sum: blocks of <= 128 with eight accumulators, recursion at 128 / 256 / > 1000 (halves rounded to 8)
WI_LENGTHS = (0, 1, 2, 7, 8, 9, 15, 16, 17, 127, 128, 129, 255, 256, 257, 1000, 1031, 2053)


@pytest.mark.parametrize("kind", ["u16", "i16", "f32"])
def test_width_integral_paths(ops, O, kind):
    """Every length at all eight residues and three polarities: the uint16 / int16 fast path (L >= 8, 16-byte aligned
    start) and the scalar path everywhere else; records entirely below the baseline (q = 0), NaN / inf samples and NaN
    baselines (q not finite), cumulative sums that land exactly on the quantile targets, and q_high so close to 1 that the cumulative sum never reaches it (searchsorted -> L).
    Every field bit-exact."""
    from waveformanalysis_b200.dtypes import WAVEFORM_WIDTH_INTEGRAL_DTYPE

    rng = np.random.default_rng({"u16": 1, "i16": 2, "f32": 3}[kind])
    lens = np.repeat(np.array(WI_LENGTHS, dtype=np.int32), 24)
    res = np.tile(np.repeat(np.arange(8), 3), len(WI_LENGTHS))
    pols = np.tile(np.array(["unknown", "negative", "positive"]), len(lens) // 3)
    offs, total = layout(lens, res, gap=1)
    base = -3000.0 if kind == "i16" else 8000.0
    rec = make_records(lens, offs, polarity=pols, baseline=base + rng.choice([0.0, 0.25, -0.5, 0.999], size=len(lens)))
    pool = np.full(total, base, dtype=np.float64)
    for i, (o, L) in enumerate(zip(offs.tolist(), lens.tolist())):
        sign = -1.0 if pols[i] != "positive" else 1.0
        t = np.arange(L)
        pool[o:o + L] = base + rng.normal(0, 2, L) + sign * rng.uniform(5, 2000) * np.exp(-np.abs(t - rng.integers(0, max(L, 1))) / 20.0)
    if kind == "f32":
        pool = (pool + rng.uniform(-0.5, 0.5, total)).astype(np.float32)
    else:
        pool = np.clip(np.round(pool), -32768 if kind == "i16" else 0, 32767 if kind == "i16" else 65535)
        pool = pool.astype(np.int16 if kind == "i16" else np.uint16)
    below = (lens > 0) & (np.arange(len(lens)) % 24 == 5)  # all charge on the wrong side of the baseline: q = 0
    for i in np.flatnonzero(below):
        o, L = int(offs[i]), int(lens[i])
        pool[o:o + L] = base + (50 if pols[i] != "positive" else -50)
    flat = np.flatnonzero((lens % 4 == 0) & (lens > 0) & np.isin(np.arange(len(lens)) % 24, (0, 1, 2, 12, 13, 14)))
    for i in flat:  # unit charge per sample: the cumulative sum lands exactly on q_low * q and q_high * q at 0.25 / 0.75
        o, L = int(offs[i]), int(lens[i])
        pool[o:o + L] = base + (-1 if pols[i] != "positive" else 1)
    rec["baseline"][flat] = base
    rec["baseline"][np.flatnonzero(lens > 8)[7::40]] = np.nan
    if kind == "f32":
        big = np.flatnonzero(lens > 8)
        pool[offs[big[3::40]] + 4] = np.nan
        pool[offs[big[11::40]] + 2] = np.inf
        pool[offs[big[19::40]] + 1] = -np.inf
        # unit charge first, then tiny charges: np.cumsum stays at 1 where the pairwise total grows past it, so with
        # q_high = 1 - 2^-53 the cumulative sum never reaches q_high * q
        tiny = int(np.flatnonzero((lens == 257) & (pols == "unknown"))[0])
        rec["baseline"][tiny] = 0.0
        pool[offs[tiny]] = -1.0
        pool[offs[tiny] + 1:offs[tiny] + 257] = -1e-16
    signed = kind == "i16"
    fx = WAVEFORM_WIDTH_INTEGRAL_DTYPE.names
    dev_pool = pool.view(np.uint16) if signed else pool  # int16 samples travel as 16-bit words, read back as signed
    for q_low, q_high, dt in ((0.1, 0.9, None), (0.25, 0.75, 2.0), (1e-9, float(np.nextafter(1.0, 0.0)), 4.0)):
        got = ops.width_integral(rec, dev_pool, q_low=q_low, q_high=q_high, dt=dt, signed_samples=signed)
        want = O.width_integral(rec, pool, q_low=q_low, q_high=q_high, dt=dt)
        assert_rows_match(got, want, float_exact=fx, what=f"width_integral {kind} q {q_low}/{q_high}")
        if q_high > 0.99 and kind == "f32":
            assert want["t_high_samples"][tiny] == 257, "the cumulative sum reached q_high * q"
    assert np.any(want["q_total"] == 0) and np.any(np.isnan(want["q_total"]))


# ---------------------------------------------------------------------------------------------------------------------
# wfb_waveform_width
# ---------------------------------------------------------------------------------------------------------------------
def width_rows(rng, L, n, dtype):
    """Rows with a constant baseline and one triangular pulse whose edges start next to the 32- and 128-sample groups
    of the warp scan (the falling edge is scanned from the peak position)."""
    waves = np.zeros((n, L), dtype=np.float64) + 1000.0
    peaks = np.zeros(n, dtype=np.int64)
    starts = [s for s in (0, 1, 30, 31, 32, 33, 50, 126, 127, 128, 129, 130, 160, 161) if s < L] or [0]
    for i in range(n):
        a = int(rng.choice(starts))
        r = int(rng.integers(1, 40))
        p = min(a + r, L - 1)
        f = int(rng.choice([1, 2, 31, 32, 33, 127, 128, 129, 200]))
        amp = float(rng.choice([10.0, 100.0, 1000.0, 3.0]))
        t = np.arange(L)
        up = np.clip((t - a) / max(p - a, 1), 0, 1)
        down = np.clip(1 - (t - p) / f, 0, 1)
        waves[i] += amp * np.where(t <= p, up, down)
        if rng.random() < 0.3:
            waves[i] += rng.normal(0, 1, L)
        peaks[i] = p
    if dtype == np.int16:
        return np.round(waves).astype(np.int16), peaks
    return waves.astype(np.float32), peaks


@pytest.mark.parametrize("dtype", [np.int16, np.float32], ids=["i16", "f32"])
@pytest.mark.parametrize("L", [1, 5, 7, 8, 9, 31, 49, 50, 51, 160, 300])
def test_waveform_width_paths(ops, O, dtype, L):
    """Rows shorter than the 50-sample baseline and than 8 (numpy_mean_f32_warp's branches), crossings at the scan's
    32 / 128-sample group edges, thresholds equal to a sample (integer pulses of 10 / 100 / 1000), fractions 0 and 1,
    positions 0, L - 1 and negative (numpy wraps the index but the falling edge adds the raw position), positions past
    the row (dropped), unknown and duplicate record ids (the first row wins).  int16 rows bit-exact, float32 rows within
    the bar."""
    from waveformanalysis_b200.dtypes import HIT_DTYPE

    rng = np.random.default_rng(L * 3 + (dtype == np.float32))
    n = 40
    waves, peaks = width_rows(rng, L, n, dtype)
    rids = np.arange(n, dtype=np.int64) + 100
    rids[5] = rids[4]  # duplicate id: row 4 wins
    hits = np.zeros(4 * n + 6, dtype=HIT_DTYPE)
    pos = np.concatenate([peaks, peaks - 1, rng.integers(-L, L, size=n), rng.integers(0, max(L, 1), size=n), [0, L - 1, -1, -L, L, L + 3]])
    hits["position"] = pos
    hits["record_id"] = np.concatenate([rids, rids, rids, rids, rids[:6]])
    hits["record_id"][7] = 10**6  # no such row
    hits["timestamp"] = np.arange(len(hits)) * 1000 + 5
    hits["board"] = np.arange(len(hits)) % 3
    hits["channel"] = np.arange(len(hits)) % 7
    fx = FX_WW if dtype == np.int16 else ()
    for kw in ({}, {"rise_low": 0.0, "rise_high": 1.0, "fall_high": 1.0, "fall_low": 0.0}, {"rise_low": 0.5, "rise_high": 0.5, "fall_high": 0.5,
               "fall_low": 0.5, "sampling_rate": 0.25}, {"interpolation": False, "sampling_rate": 0.3}):
        got = ops.waveform_width(hits, rids, waves, **kw)
        want = O.waveform_width(hits, rids, waves, **kw)
        assert_rows_match(got, want, float_exact=fx, what=f"waveform_width L {L} {kw}")


def test_waveform_width_f32_special_values(ops, O):
    """float32 rows: a NaN peak value is kept (NaN <= 0 is False) with zero widths; a NaN in the baseline window makes
    every value NaN; amplitudes so small that |dy| < 1e-10 takes the plateau branch of the interpolation."""
    from waveformanalysis_b200.dtypes import HIT_DTYPE

    L = 200
    waves = np.zeros((4, L), dtype=np.float32)
    t = np.arange(L)
    waves[0] = 50 * np.exp(-np.abs(t - 100) / 8.0)
    waves[0, 100] = np.nan
    waves[1] = 50 * np.exp(-np.abs(t - 100) / 8.0)
    waves[1, 3] = np.nan
    waves[2] = (1e-11 * np.exp(-np.abs(t - 120) / 3.0)).astype(np.float32)
    waves[3] = np.where(np.abs(t - 90) < 20, 1e-12, 0).astype(np.float32)
    hits = np.zeros(5, dtype=HIT_DTYPE)
    hits["position"] = [100, 100, 120, 90, 95]
    hits["record_id"] = [0, 1, 2, 3, 3]
    hits["channel"] = 1
    got = ops.waveform_width(hits, np.arange(4), waves)
    want = O.waveform_width(hits, np.arange(4), waves)
    assert len(want) == 5 and np.isnan(want["peak_height"][:2]).all()
    assert_rows_match(got, want, what="waveform_width f32 special")


# ---------------------------------------------------------------------------------------------------------------------
# wfb_find_peaks
# ---------------------------------------------------------------------------------------------------------------------
def peak_records(rng, lens, n_pulses, *, spacing=None):
    """uint16 records with well separated negative Gaussian pulses (clean: one derivative peak per pulse)."""
    lens = np.asarray(lens, dtype=np.int32)
    offs = np.concatenate([[0], np.cumsum(lens[:-1])]).astype(np.int64)
    pool = np.zeros(int(lens.sum()), dtype=np.float64)
    for o, L, k in zip(offs.tolist(), lens.tolist(), n_pulses):
        t = np.arange(L)
        w = np.full(L, 9000.0)
        step = spacing or max(L // (k + 1), 1)
        for j in range(k):
            w -= rng.uniform(300, 2000) * np.exp(-0.5 * ((t - step * (j + 1)) / 3.0) ** 2)
        pool[o:o + L] = w
    rec = make_records(lens, offs, baseline=9000.0)
    rec["channel"] = np.arange(len(lens)) % 4
    return rec, np.round(pool).astype(np.uint16)


def records_waves(rec, pool):
    """-RecordsView.signals() in float64 for unknown / negative polarity records."""
    out = []
    for o, L, b in zip(rec["wave_offset"].tolist(), rec["event_length"].tolist(), rec["baseline"].tolist()):
        out.append(-(pool[o:o + L].astype(np.float32) - np.float32(b)).astype(np.float64))
    return out


def aos_rows(rec, pool, dtype):
    from waveformanalysis_b200.dtypes import create_record_dtype

    L = int(rec["event_length"].max())
    st_dt = create_record_dtype(L)
    if dtype == np.float32:
        st_dt = np.dtype([(nm, (np.float32, (L,)) if nm == "wave" else st_dt.fields[nm][0]) for nm in st_dt.names])
    st = np.zeros(len(rec), dtype=st_dt)
    for f in ("baseline", "timestamp", "record_id", "dt", "board", "channel"):
        st[f] = rec[f]
    st["event_length"] = L
    st["polarity"] = "unknown"
    st["wave"] = 9000
    for i, (o, n) in enumerate(zip(rec["wave_offset"].tolist(), rec["event_length"].tolist())):
        st["wave"][i, :n] = pool[o:o + n]
    return st


# Shared-memory layout of wfb_find_peaks (hit_peaks.cu): lcap = (lmax + 1) & ~1 and one warp stages
# per_warp = round_up_16(8 lcap + 5 (lcap / 2 + 2)) ~ 10.5 lcap + 10 bytes; the block takes 4, 2 or 1 warps while
# nwarps * per_warp <= 200 KiB, else the records stage in global memory:
#   lmax 4874: per_warp 51200 -> 4 warps;   4875 (lcap 4876): 51216 -> 2 warps
#   lmax 9750: per_warp 102400 -> 2 warps;  9751 (lcap 9752): 102416 -> 1 warp
#   lmax 19502: per_warp 204784 -> 1 warp;  19503 (lcap 19504): 204816 -> global staging
@pytest.mark.parametrize("lmax", [4874, 4875, 9750, 9751, 19502, 19503])
def test_find_peaks_shared_memory_layouts(ops, O, lmax):
    rng = np.random.default_rng(lmax)
    rec, pool = peak_records(rng, [lmax, lmax - 1, 333, lmax], [30, 3, 7, 9])
    kw = dict(height=12.0, width=2)
    want = O.hit_find_peaks(records_waves(rec, pool), rec, source="records", **kw)
    assert len(want) >= 40
    assert_rows_match(ops.find_peaks_records(rec, pool, **kw), want, what=f"records lmax {lmax}", float_exact=FX_PEAKS)
    st = aos_rows(rec[[0, 3]], pool, np.int16)
    want = O.hit_find_peaks(list(st["wave"]), st, source="aos", **kw)
    assert_rows_match(ops.find_peaks_waveforms(st, **kw), want, what=f"aos lmax {lmax}", float_exact=FX_PEAKS)


@pytest.mark.parametrize("source", ["rec_u16", "rec_f32", "aos_i16", "aos_f32"])
def test_find_peaks_cache_split(ops, O, source):
    """Records with 0..5, exactly 6 (the counting pass caches kPeakCache = 6 peaks: emitted by peaks_emit_cached_kernel),
    exactly 7 and many peaks (re-emitted by the second find_peaks_kernel pass), interleaved."""
    rng = np.random.default_rng(61)
    counts = [6, 7, 0, 1, 5, 6, 40, 7, 6, 2, 13, 6, 7]
    rec, pool = peak_records(rng, [600] * len(counts), counts)
    kw = dict(height=12.0, width=2)
    if source.startswith("rec"):
        p = pool.astype(np.float32) + np.float32(0.25) if source == "rec_f32" else pool
        want = O.hit_find_peaks(records_waves(rec, p), rec, source="records", **kw)
        got = ops.find_peaks_records(rec, p, **kw)
    else:
        st = aos_rows(rec, pool, np.float32 if source == "aos_f32" else np.int16)
        want = O.hit_find_peaks(list(st["wave"]), st, source="aos", **kw)
        got = ops.find_peaks_waveforms(st, **kw)
    per_record = np.bincount(want["record_id"], minlength=len(counts))
    assert per_record.tolist() == counts, "the records do not have the intended peak counts"
    assert_rows_match(got, want, what=f"cache split {source}", float_exact=FX_PEAKS)
