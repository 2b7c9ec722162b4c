"""Host-array front ends of the remaining C-ABI entry points: records builder (K1),
wave_pool_filtered, waveform_width, waveform_width_integral, hit merging and event grouping (K4).

Every function takes / returns host numpy arrays in the reference's dtypes and does its
arithmetic on the device through libwfb200.so; torch tensors only own device memory.
"""

from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from .dtypes import (
    THRESHOLD_HIT_DTYPE,
    HIT_MERGE_CLUSTERS_DTYPE,
    HIT_MERGED_COMPONENTS_DTYPE,
    HIT_MERGED_DTYPE,
    RECORDS_DTYPE,
    WAVEFORM_WIDTH_DTYPE,
    WAVEFORM_WIDTH_INTEGRAL_DTYPE,
)
from .engine import DeviceRun, _ptr, _stream, _torch, check_pool, packed_records, upload

# --------------------------------------------------------------------------------------------
# small helpers
# --------------------------------------------------------------------------------------------


def _dev(a: np.ndarray):
    return upload(a)


def _empty(nbytes: int):
    return _torch().empty(max(int(nbytes), 16), dtype=_torch().uint8, device="cuda")


# --------------------------------------------------------------------------------------------
# K1: records builder
# --------------------------------------------------------------------------------------------
def build_records_ragged(timestamps_ps, boards, channels, sample_blocks, *, dt_ns: int, baseline_window=(0, 40), baselines=None,
                         epoch_ns: int | None = None):
    """Like build_records for parts of different waveform widths: ``sample_blocks`` is a list of int16
    matrices (n_k, L_k) whose rows follow each other in the order of the per-record columns."""
    up = raw_upload(timestamps_ps, boards, channels, sample_blocks, baselines=baselines)
    n = up["n"]
    if n == 0:
        return np.zeros(0, dtype=RECORDS_DTYPE), np.zeros(0, dtype=np.uint16)
    rows, pool, _ = build_records_ragged_device(up, dt_ns=dt_ns, baseline_window=baseline_window, epoch_ns=epoch_ns)
    rec = rows[: n * 102].cpu().numpy().view(RECORDS_DTYPE)
    return rec, pool.cpu().numpy().view(np.uint16)


def raw_upload(timestamps_ps, boards, channels, sample_blocks, *, baselines=None) -> dict:
    """Raw rows on the device for build_records_ragged_device: the int16 / uint16 matrices of ``sample_blocks`` at
    16-byte aligned bases of ONE device buffer, every row's byte offset and length, and the per-row columns (which
    follow the blocks' rows in order)."""
    torch = _torch()
    blocks = [np.ascontiguousarray(b) for b in sample_blocks]
    for b in blocks:
        if b.dtype not in (np.int16, np.uint16) or b.ndim != 2:
            raise ValueError(f"sample blocks must be 2-D int16 arrays, got {b.dtype} {b.shape}")
    n = sum(len(b) for b in blocks)
    offs, lens, cursor = [np.zeros(0, np.int64)], [np.zeros(0, np.int32)], 0
    for b in blocks:
        offs.append(cursor + np.arange(len(b), dtype=np.int64) * (b.shape[1] * 2))
        lens.append(np.full(len(b), b.shape[1], dtype=np.int32))
        cursor += (b.nbytes + 15) & ~15
    d_blob = torch.empty(cursor + 16, dtype=torch.uint8, device="cuda")
    base = 0
    for b in blocks:
        if b.nbytes:
            d_blob[base:base + b.nbytes].copy_(upload(b.reshape(-1).view(np.uint8)))
        base += (b.nbytes + 15) & ~15
    ln = np.concatenate(lens)
    cols = {"timestamp": (timestamps_ps, np.int64), "board": (boards, np.int16), "channel": (channels, np.int16)}
    if baselines is not None:
        cols["baseline"] = (baselines, np.float64)
    up = {k: np.asarray(v, dtype=t).reshape(-1) for k, (v, t) in cols.items()}
    for k, v in up.items():
        if len(v) != n:
            raise ValueError(f"{k} has {len(v)} entries for {n} sample rows")
    up = {k: _dev(v) for k, v in up.items()}
    up.update(blob=d_blob, blob_bytes=cursor, sample_offset=_dev(np.concatenate(offs)), n_samples=_dev(ln), n=n,
              total=int(ln.astype(np.int64).sum()))
    return up


def build_records_ragged_device(up: dict, *, dt_ns: int, baseline_window=(0, 40), epoch_ns: int | None = None,
                                seq: np.ndarray | None = None, meta: bool = False):
    """wfb_build_records_ragged (``seq`` given: wfb_build_records_ragged_seq, record_id = seq) on the output of
    raw_upload -> device (rows uint8 [n * 102], pool int16 [total] with a 16-sample tail, meta uint8 [n * 48] or None)."""
    lib = _lib.load()
    torch = _torch()
    n, total = up["n"], up["total"]
    rows = _empty(n * 102)
    pool = torch.empty(total + 16, dtype=torch.int16, device="cuda")[:total]
    d_meta = torch.empty(max(n, 1) * 48, dtype=torch.uint8, device="cuda") if meta else None
    if n == 0:
        return rows, pool, d_meta
    ws = _empty(lib.wfb_build_records_v1725_workspace_bytes(n))
    cols = (_ptr(up["blob"]), up["blob_bytes"], _ptr(up["sample_offset"]), _ptr(up["n_samples"]), _ptr(up["timestamp"]), _ptr(up["board"]),
            _ptr(up["channel"]), _ptr(up.get("baseline")))
    tail = (n, int(dt_ns), int(baseline_window[0]), int(baseline_window[1]), int(epoch_ns or 0), _ptr(rows), _ptr(pool), total, _ptr(d_meta),
            _ptr(ws), ws.numel(), _stream())
    if seq is None:
        _lib.check(lib.wfb_build_records_ragged(*cols, *tail), "wfb_build_records_ragged")
    else:
        d_seq = _dev(np.ascontiguousarray(seq, dtype=np.int64))
        if len(d_seq) != n:
            raise ValueError(f"seq has {len(d_seq)} entries for {n} rows")
        _lib.check(lib.wfb_build_records_ragged_seq(*cols, _ptr(d_seq), *tail), "wfb_build_records_ragged_seq")
    return rows, pool, d_meta




def build_records(timestamps_ps, boards, channels, samples, *, dt_ns: int, baseline_window=(0, 40),
                  baselines=None, epoch_ns: int | None = None, return_device: bool = False):
    """raw rows (per-channel file order) -> (records[RECORDS_DTYPE], wave_pool[uint16]) in the
    reference's global order (records_builder.py:115-120, 212-302, 341-426)."""
    lib = _lib.load()
    torch = _torch()
    samples = np.ascontiguousarray(samples)
    if samples.dtype not in (np.int16, np.uint16):
        raise ValueError(f"samples must be int16, got {samples.dtype}")
    n, L = samples.shape
    if n == 0:
        return np.zeros(0, dtype=RECORDS_DTYPE), np.zeros(0, dtype=np.uint16)
    d_s = upload(samples.reshape(-1), tail=16)
    d_ts = _dev(np.asarray(timestamps_ps, dtype=np.int64))
    d_b = _dev(np.asarray(boards, dtype=np.int16))
    d_c = _dev(np.asarray(channels, dtype=np.int16))
    d_bl = _dev(np.asarray(baselines, dtype=np.float64)) if baselines is not None else None
    rows = _empty(n * 102)
    pool = torch.empty(n * L + 16, dtype=torch.int16, device="cuda")[: n * L]
    ws = _empty(lib.wfb_build_records_workspace_bytes(n))
    _lib.check(lib.wfb_build_records(_ptr(d_s), _ptr(d_ts), _ptr(d_b), _ptr(d_c), _ptr(d_bl), n, L, int(baseline_window[0]),
                                     int(baseline_window[1]), int(dt_ns), int(epoch_ns or 0), _ptr(rows), _ptr(pool), C.c_void_p(0),
                                     _ptr(ws), ws.numel(), _stream()), "wfb_build_records")
    rec = rows[: n * 102].cpu().numpy().view(RECORDS_DTYPE)
    if return_device:
        return rec, pool.cpu().numpy().view(np.uint16), pool
    return rec, pool.cpu().numpy().view(np.uint16)


def sort_pairs(keys: np.ndarray, vals: np.ndarray):
    lib = _lib.load()
    torch = _torch()
    n = len(keys)
    dk, dv = _dev(np.asarray(keys, np.int64)), _dev(np.asarray(vals, np.int64))
    ok, ov = torch.empty_like(dk), torch.empty_like(dv)
    ws = _empty(lib.wfb_sort_workspace_bytes(n))
    _lib.check(lib.wfb_sort_pairs_i64(_ptr(dk), _ptr(dv), _ptr(ok), _ptr(ov), n, _ptr(ws), ws.numel(), _stream()), "wfb_sort_pairs_i64")
    return ok.cpu().numpy(), ov.cpu().numpy()


# --------------------------------------------------------------------------------------------
# wave_pool_filtered
# --------------------------------------------------------------------------------------------


def sg_tables(window: int, poly: int) -> np.ndarray:
    """[taps (w) | projector rows for outputs 0..h-1 (h*w) | rows for outputs L-h..L-1 (h*w)].

    Host-side filter design, the analogue of scipy.signal.savgol_coeffs and the polynomial edge
    fit of savgol_filter(mode='interp') (filtering.py:226-241): least-squares solve, done once per
    distinct window."""
    h = window // 2
    x = np.arange(-h, window - h, dtype=float)[::-1]
    A = x ** np.arange(poly + 1).reshape(-1, 1)
    y = np.zeros(poly + 1)
    y[0] = 1.0
    c, *_ = np.linalg.lstsq(A, y, rcond=None)
    taps = c[::-1].copy()  # y[k] = sum_j taps[j] * x[k-h+j]
    V = np.vander(np.arange(window, dtype=float), poly + 1)
    P = V @ np.linalg.pinv(V)
    return np.concatenate([taps, P[:h].reshape(-1), P[window - h:].reshape(-1)])


def butter_bandpass_sos(order: int, lowcut: float, highcut: float, fs: float) -> np.ndarray:
    """Filter design is host-side configuration exactly as in the reference
    (filtering.py:101: scipy.signal.butter(..., output='sos'))."""
    from scipy.signal import butter

    return butter(int(order), [float(lowcut), float(highcut)], btype="band", output="sos", fs=float(fs))


def sos_zi(sos: np.ndarray) -> np.ndarray:
    """Steady-state DF2T state per section (scipy.signal.sosfilt_zi, scipy 1.18 formula):
    y_inf = sum(b)/sum(a); zi = reversed cumulative sum of (b - y_inf*a) without its first entry,
    scaled by the DC gain of the sections before."""
    sos = np.asarray(sos, dtype=np.float64)
    zi = np.zeros((sos.shape[0], 2))
    scale = 1.0
    for s in range(sos.shape[0]):
        b, a = sos[s, :3], sos[s, 3:]
        if a[0] != 1:
            b, a = b / a[0], a / a[0]
        y_inf = np.sum(b) / np.sum(a)
        v = b - y_inf * a
        zi[s, 1] = scale * v[2]
        zi[s, 0] = scale * (v[2] + v[1])
        scale *= np.sum(sos[s, :3]) / np.sum(sos[s, 3:])
    return zi


# --------------------------------------------------------------------------------------------
# per-channel tables: channel keys, polarity, filter plan
# --------------------------------------------------------------------------------------------
POLARITY_VALUES = ("positive", "negative", "unknown")
POLARITY_ENTRY_DTYPE = np.dtype([("key", "<i4"), ("image", "<u4", 8)])  # wfb_polarity_entry
assert POLARITY_ENTRY_DTYPE.itemsize == 36


def channel_key(board: int, channel: int) -> int:
    """The key the device tables are sorted by (channel_config.unique_channels' order)."""
    return int(board) * 65536 + (int(channel) & 0xFFFF)


def _in_i16(*v) -> bool:
    return all(-32768 <= int(x) <= 32767 for x in v)


def shard_channels(run: DeviceRun) -> list[tuple[int, int]]:
    """The distinct (board, channel) pairs of a device run's records, sorted (``channel_config.unique_channels``)."""
    torch = _torch()
    n = run.n
    if n == 0:
        return []
    bc = run.meta[: n * 48].view(n, 48)[:, 32:36].contiguous().view(torch.int16).view(n, 2).long()  # wfb_rec_meta board, channel
    keys = torch.unique(bc[:, 0] * 65536 + (bc[:, 1] & 0xFFFF)).cpu().numpy()
    return sorted((int(k) >> 16, ((int(k) & 0xFFFF) ^ 0x8000) - 0x8000) for k in keys.tolist())


def polarity_entries(polarity: dict | None) -> list[tuple[int, int, str]]:
    """The sorted (board, channel, value) entries of a polarity map {(board, channel): "positive" | "negative" |
    "unknown"}.  Any other value, a key that is not a pair of integers, or one channel given two values raise
    ValueError."""
    out: dict[tuple[int, int], str] = {}
    for k, v in dict(polarity or {}).items():
        try:
            b, c = (int(x) for x in k)
        except (TypeError, ValueError):
            raise ValueError(f"polarity keys are (board, channel) pairs, got {k!r}") from None
        if not isinstance(v, str) or v not in POLARITY_VALUES:
            raise ValueError(f"polarity of channel {(b, c)} must be one of {POLARITY_VALUES}, got {v!r}")
        if out.setdefault((b, c), v) != v:
            raise ValueError(f"channel {(b, c)} is given two polarities")
    return sorted((b, c, v) for (b, c), v in out.items())


def polarity_table(polarity: dict | None) -> np.ndarray:
    """wfb_polarity_entry rows of a polarity map: its "positive" / "negative" channels sorted by key, each with the
    UTF-32 image numpy stores for that string in a RECORDS_DTYPE polarity field.  "unknown" entries and channels
    outside the int16 range of records' board / channel match no record change and are left out."""
    ent = [(channel_key(b, c), v) for b, c, v in polarity_entries(polarity) if v != "unknown" and _in_i16(b, c)]
    ent.sort()
    table = np.zeros(len(ent), dtype=POLARITY_ENTRY_DTYPE)
    for i, (k, v) in enumerate(ent):
        table[i]["key"] = k
        table[i]["image"] = np.array([v], dtype="U8").view(np.uint32)
    if len(table) > _lib.MAX_CHANNEL_KEYS:
        raise ValueError(f"a polarity map sets at most {_lib.MAX_CHANNEL_KEYS} channels, got {len(table)}")
    return table


def apply_polarity(run: DeviceRun, polarity: dict | None) -> None:
    """records["polarity"] of a device run from a channel map, as plugins.records._apply_polarity sets it on host
    records: every record of a "positive" / "negative" channel gets that value in ``run.records_rows`` (when the run
    has them) and the matching code in ``run.meta``; records of other channels and of "unknown" channels keep theirs.
    In place, on the current stream."""
    table = polarity_table(polarity)
    if run.n == 0 or len(table) == 0:
        return
    _lib.check(_lib.load().wfb_apply_polarity(_ptr(run.meta), _ptr(run.records_rows), run.n, _ptr(upload(table)), len(table), _stream()),
               "wfb_apply_polarity")


def _filter_cfg_struct(cfg: dict) -> "_lib.FilterCfg":
    c = _lib.FilterCfg()
    if cfg["filter_type"] == "BW":
        sos = np.asarray(cfg["sos"], dtype=np.float64)
        if sos.shape[0] > _lib.MAX_SOS_SECTIONS:
            raise ValueError(f"filter_order too high: {sos.shape[0]} sections > {_lib.MAX_SOS_SECTIONS}")
        zi = sos_zi(sos)
        c.type, c.n_sections = 1, sos.shape[0]
        for s in range(sos.shape[0]):
            for j in range(6):
                c.sos[s][j] = sos[s, j]
            c.zi[s][0], c.zi[s][1] = zi[s, 0], zi[s, 1]
    else:
        c.type, c.sg_window, c.sg_poly = 0, int(cfg["sg_window_size"]), int(cfg["sg_poly_order"])
    return c


def filter_plan(run: DeviceRun, configs: dict, default: dict | None = None, *, lengths: np.ndarray | None = None) -> dict:
    """The per-record arguments of wfb_filter_pool, planned on the device by wfb_filter_plan.

    ``configs[(board, channel)]`` / ``default``: configurations as ``filter_pool`` takes them.  Without ``default``,
    ``configs`` must hold every channel of the run.  One wfb_filter_cfg per DISTINCT configuration (so channels that
    share one Butterworth filter take the uniform kernel), one Savitzky-Golay table per effective (window, poly); for
    every SG configuration a table offset per record length 0 .. min(window, lmax).  ``lengths``: the record lengths
    that occur (host records); otherwise those of [run.lmin, lmax], or of 0 .. lmax, get a table."""
    torch = _torch()
    distinct: list[dict] = []
    at: dict = {}

    def index(cfg: dict) -> int:
        ident = (("BW", np.asarray(cfg["sos"], dtype=np.float64).tobytes()) if cfg["filter_type"] == "BW"
                 else ("SG", int(cfg["sg_window_size"]), int(cfg["sg_poly_order"])))
        if ident not in at:
            at[ident] = len(distinct)
            distinct.append(cfg)
        return at[ident]

    keyed = sorted((channel_key(b, c), index(cfg)) for (b, c), cfg in configs.items() if _in_i16(b, c))
    default_cfg = index(default) if default is not None else 0
    if not distinct:
        raise ValueError("filter_plan: no filter configuration")
    if len(keyed) > _lib.MAX_CHANNEL_KEYS:
        raise ValueError(f"at most {_lib.MAX_CHANNEL_KEYS} per-channel filter configurations, got {len(keyed)}")
    lmax = max(run.lmax, 0)
    present = None
    if lengths is not None:
        present = np.unique(np.clip(np.asarray(lengths, dtype=np.int64), 0, lmax))
    tables, table_at, cursor = [], {}, 0
    lut_parts, lut_off, wcaps, lut_len = [], [], [], 0
    for cfg in distinct:
        if cfg["filter_type"] == "BW":
            lut_off.append(-1)
            wcaps.append(0)
            continue
        w0, poly = int(cfg["sg_window_size"]), int(cfg["sg_poly_order"])
        wcap = min(w0, lmax)
        need = np.zeros(wcap + 1, dtype=bool)
        if present is not None:
            need[np.minimum(present, wcap)] = True
        else:
            need[min(run.lmin or 0, wcap):] = True
        lut = np.full(wcap + 1, -1, dtype=np.int32)
        for L in np.flatnonzero(need).tolist():
            w = min(w0, L)
            w -= (w % 2 == 0)
            if w <= poly or w <= 0:
                continue  # identity (filtering.py:193-194, 231-232)
            if (w, poly) not in table_at:
                tables.append(sg_tables(w, poly))
                table_at[(w, poly)] = cursor
                cursor += len(tables[-1])
            lut[L] = table_at[(w, poly)]
        lut_parts.append(lut)
        lut_off.append(lut_len)
        wcaps.append(wcap)
        lut_len += len(lut)
    n = run.n
    cfgs = (_lib.FilterCfg * len(distinct))(*[_filter_cfg_struct(c) for c in distinct])
    plan = dict(
        n_cfg=len(distinct), configs=distinct, has_bw=any(c["filter_type"] == "BW" for c in distinct),
        d_cfg=upload(np.frombuffer(bytes(cfgs), dtype=np.uint8).copy()),
        d_tab=upload(np.concatenate(tables) if tables else np.zeros(1)),
        d_idx=torch.empty(max(n, 1), dtype=torch.int32, device="cuda"),
        d_toff=torch.empty(max(n, 1), dtype=torch.int32, device="cuda"),
    )
    keys = np.array([k for k, _ in keyed] or [0], dtype=np.int32)
    cfg_of_key = np.array([c for _, c in keyed] or [0], dtype=np.int32)
    d_keys, d_cok = upload(keys), upload(cfg_of_key)
    d_lut = upload(np.concatenate(lut_parts) if lut_parts else np.full(1, -1, np.int32))
    d_off, d_wcap = upload(np.array(lut_off, dtype=np.int32)), upload(np.array(wcaps, dtype=np.int32))
    _lib.check(_lib.load().wfb_filter_plan(_ptr(run.meta), n, _ptr(d_keys), _ptr(d_cok), len(keyed), default_cfg, _ptr(d_lut), _ptr(d_off),
                                           _ptr(d_wcap), _ptr(plan["d_idx"]), _ptr(plan["d_toff"]), _stream()), "wfb_filter_plan")
    return plan


def _filter_launch(run: DeviceRun, plan: dict, pool_len: int, lmax: int):
    """wfb_filter_pool on a planned run -> the float32 pool (device tensor)."""
    lib = _lib.load()
    torch = _torch()
    d_out = torch.empty(pool_len + 16, dtype=torch.float32, device="cuda")[:pool_len]
    ws = _empty(lib.wfb_filter_workspace_bytes(run.n, lmax)) if plan["has_bw"] else None
    _lib.check(lib.wfb_filter_pool(_ptr(run.pool), run.pool_is_f32, pool_len, _ptr(run.meta), run.n, _ptr(plan["d_cfg"]), plan["n_cfg"],
                                   _ptr(plan["d_idx"]), _ptr(plan["d_tab"]), _ptr(plan["d_toff"]), _ptr(d_out), run.pool_base, _ptr(ws),
                                   0 if ws is None else ws.numel(), lmax, _stream()), "wfb_filter_pool")
    return d_out


def filter_pool(records: np.ndarray, pool: np.ndarray, *, configs: dict, default: dict, run: DeviceRun | None = None,
                return_device: bool = False):
    """uint16 wave_pool -> float32 wave_pool_filtered (records.py:368-438).

    ``default`` / ``configs[(board, channel)]``: {"filter_type": "SG", "sg_window_size", "sg_poly_order"} or
    {"filter_type": "BW", "sos": ndarray (n_sections, 6)}.
    """
    from .channel_config import unique_channels

    pool_h, is_f32 = check_pool(pool)
    out = np.zeros(len(pool_h), dtype=np.float32)
    rec = packed_records(records, explicit_dt=1)
    n = len(rec)
    if n == 0 or len(pool_h) == 0:
        return (out, None) if return_device else out
    if run is None:
        run = DeviceRun.from_host(rec, pool_h)
    lens = rec["event_length"]
    per_channel = {bc: configs.get(bc, default) for bc in unique_channels(rec["board"], rec["channel"])}
    plan = filter_plan(run, per_channel, lengths=np.unique(lens))
    d_out = _filter_launch(run, plan, len(pool_h), max(int(lens.max()), 1))
    host = d_out.cpu().numpy()
    if return_device:  # the filtered pool stays in HBM for the next plugin (same records metadata, float32 samples)
        return host, DeviceRun(run.meta, d_out, n, 1, run.lmax, records_rows=run.records_rows, pool_base=run.pool_base, row_base=run.row_base)
    return host

# --------------------------------------------------------------------------------------------
# waveform_width / waveform_width_integral
# --------------------------------------------------------------------------------------------


def waveform_width(hits: np.ndarray, wave_record_ids: np.ndarray, waves: np.ndarray, *, sampling_rate=None, rise_low=0.1,
                   rise_high=0.9, fall_high=0.9, fall_low=0.1, interpolation=True) -> np.ndarray:
    """Per-hit rise / fall / total widths (waveform_width.py:97-194).  ``waves`` is the (n, L)
    int16 (st_waveforms) or float32 (filtered_waveforms) sample matrix (may be a strided view of
    the structured array's ``wave`` field); ``wave_record_ids[i]`` the record_id of row i."""
    lib = _lib.load()
    torch = _torch()
    if sampling_rate is None:
        sampling_rate = 0.5
    nh = len(hits)
    if nh == 0 or len(waves) == 0:
        return np.zeros(0, dtype=WAVEFORM_WIDTH_DTYPE)
    if waves.dtype == np.int16:
        is_f32 = 0
    elif waves.dtype == np.float32:
        is_f32 = 1
    else:
        raise ValueError(f"waveform samples must be int16 or float32, got {waves.dtype}")
    n_w, L = waves.shape
    # first row whose record_id matches (np.flatnonzero(...)[0], waveform_width.py:165-168)
    rids = np.asarray(wave_record_ids, dtype=np.int64)
    uniq, first = np.unique(rids, return_index=True)
    h_rid = hits["record_id"].astype(np.int64)
    loc = np.searchsorted(uniq, h_rid)
    loc_c = np.minimum(loc, len(uniq) - 1)
    hit_row = np.where(uniq[loc_c] == h_rid, first[loc_c], -1).astype(np.int64)
    d_w = _dev(np.ascontiguousarray(waves).reshape(-1))
    p = _lib.WidthParams(float(rise_low), float(rise_high), float(fall_high), float(fall_low), float(sampling_rate),
                         1 if interpolation else 0, is_f32)
    names = hits.dtype.names
    d_row, d_pos = _dev(hit_row), _dev(hits["position"].astype(np.int64))
    d_ts, d_rid = _dev(hits["timestamp"].astype(np.int64)), _dev(h_rid)
    d_b = _dev(hits["board"].astype(np.int16)) if "board" in names else None
    d_c = _dev(hits["channel"].astype(np.int16))
    out = _empty(nh * 56)
    valid = _empty(nh)
    _lib.check(lib.wfb_waveform_width(_ptr(d_w), n_w, L, L, _ptr(d_row), _ptr(d_pos), _ptr(d_ts), _ptr(d_b), _ptr(d_c), _ptr(d_rid), nh,
                                      C.byref(p), _ptr(out), _ptr(valid), _stream()), "wfb_waveform_width")
    rows = out[: nh * 56].cpu().numpy().view(WAVEFORM_WIDTH_DTYPE)
    keep = valid[:nh].cpu().numpy().astype(bool)
    return rows[keep].copy()


def waveform_width_run(run: DeviceRun, d_hits, n_hits: int, *, sampling_rate=None, rise_low=0.1, rise_high=0.9, fall_high=0.9,
                       fall_low=0.1, interpolation=True):
    """``waveform_width`` for packed HIT_DTYPE rows that live on the device (``d_hits``, uint8 tensor) against a
    device-resident run, a time shard included: a hit's waveform is run row ``record_id - run.row_base`` when that row
    holds the record, its samples the record's own event_length samples (float32 pool: the filtered_waveforms rows,
    16-bit pool: the st_waveforms rows read as int16).  Returns (WAVEFORM_WIDTH rows as a device uint8 tensor in hit
    order, row count); only the count crosses PCIe."""
    lib = _lib.load()
    torch = _torch()
    n_hits = int(n_hits)
    p = _lib.WidthParams(float(rise_low), float(rise_high), float(fall_high), float(fall_low), float(0.5 if sampling_rate is None else sampling_rate),
                         1 if interpolation else 0, int(run.pool_is_f32))
    out = _empty(n_hits * WAVEFORM_WIDTH_DTYPE.itemsize)
    count = torch.zeros(1, dtype=torch.int64, device="cuda")
    ws = _empty(lib.wfb_waveform_width_run_workspace_bytes(n_hits))
    _lib.check(lib.wfb_waveform_width_run(_ptr(run.pool), run.pool_is_f32, run.pool_len, _ptr(run.meta), run.n, run.pool_base, run.row_base,
                                          _ptr(d_hits) if n_hits else None, n_hits, C.byref(p), _ptr(out), _ptr(count), _ptr(ws), ws.numel(),
                                          _stream()), "wfb_waveform_width_run")
    return out, int(count.item())


def width_integral(records: np.ndarray, pool: np.ndarray, *, q_low=0.10, q_high=0.90, sampling_rate=0.5, dt=None,
                   run: DeviceRun | None = None, signed_samples: bool = False) -> np.ndarray:
    """Per-record cumulative-charge quantile widths (waveform_width_integral.py:83-231).  ``signed_samples``: the
    16-bit pool holds int16 values (structured st_waveforms rows used in place)."""
    lib = _lib.load()
    if dt is None:
        if sampling_rate <= 0:
            raise ValueError(f"sampling_rate ({sampling_rate}) must be > 0")
        dt = 1.0 / float(sampling_rate)
    if q_low <= 0 or q_high >= 1 or q_low >= q_high:
        raise ValueError(f"q_low/q_high invalid: q_low={q_low}, q_high={q_high}")
    n = len(records)
    if n == 0:
        return np.zeros(0, dtype=WAVEFORM_WIDTH_INTEGRAL_DTYPE)
    if run is None:
        run = DeviceRun.from_host(records, pool, explicit_dt=1)
    out = _empty(n * 52)
    kind = 2 if (signed_samples and not run.pool_is_f32) else run.pool_is_f32
    _lib.check(lib.wfb_width_integral(_ptr(run.pool), kind, run.pool_len, _ptr(run.meta), n, float(q_low), float(q_high),
                                      float(dt), run.pool_base, run.row_base, _ptr(out), _stream()), "wfb_width_integral")
    return out[: n * 52].cpu().numpy().view(WAVEFORM_WIDTH_INTEGRAL_DTYPE)


# --------------------------------------------------------------------------------------------
# K4: grouping
# --------------------------------------------------------------------------------------------


def group_hit_windows(hits: np.ndarray, time_window_ns: float, component_rows=None, component_hits=None) -> dict:
    """Chain clustering of absolute hit windows (event_grouping.py:287-471).  Rows merged across records
    (sample window -1) take their window from the component hits (``hit_merged_components`` rows +
    ``hit_threshold``), a small host reduction; everything after the windows runs on the device: the sort,
    running maximum, boundary flags and event ids (wfb_group_hit_windows / wfb_group_abs_windows), then the
    event table (wfb_hit_event_table: member order, t_min / t_max / dt/ns / n_hits).  Returns the same dict
    as the oracle, plus ``order``."""
    lib = _lib.load()
    torch = _torch()
    if time_window_ns < 0:
        raise ValueError("time_window_ns must be >= 0")
    names = hits.dtype.names
    sn, en = ("sample_start", "sample_end") if "sample_start" in names else ("edge_start", "edge_end")
    nh = len(hits)
    if nh == 0:
        z = np.zeros(0, dtype=np.int64)
        return dict(event_id=z, t_min=z, t_max=z, dt_ns=np.zeros(0), n_hits=z, offsets=np.zeros(1, np.int64), members=z, event_of_hit=z)
    d_ts = _dev(hits["timestamp"].astype(np.int64))
    d_dt, d_rid = _dev(hits["dt"].astype(np.int32)), _dev(hits["record_id"].astype(np.int64))
    order = torch.empty(nh, dtype=torch.int64, device="cuda")
    ev = torch.empty(nh, dtype=torch.int64, device="cuda")
    n_ev = torch.zeros(1, dtype=torch.int64, device="cuda")
    ws = _empty(lib.wfb_group_workspace_bytes(nh))
    bad = np.flatnonzero((hits[sn] < 0) | (hits[en] < 0))
    if len(bad):
        if component_rows is None or component_hits is None:
            raise ValueError("component_rows and component_hits are required when hit windows contain invalid edges")
        dt_ps = hits["dt"].astype(np.float64) * 1e3
        pos = hits["position"].astype(np.float64)
        h0 = hits["timestamp"].astype(np.float64) + (hits[sn].astype(np.int32) - pos) * dt_ps
        h1 = hits["timestamp"].astype(np.float64) + (hits[en].astype(np.int32) - pos) * dt_ps
        cdt = component_hits["dt"].astype(np.float64) * 1e3
        cpos = component_hits["position"].astype(np.float64)
        c0 = component_hits["timestamp"].astype(np.float64) + (component_hits["edge_start"].astype(np.int32) - cpos) * cdt
        c1 = component_hits["timestamp"].astype(np.float64) + (component_hits["edge_end"].astype(np.int32) - cpos) * cdt
        idx = component_rows["hit_index"].astype(np.int64)
        for m in bad.tolist():  # a handful of rows: clusters that straddle two records
            o, c = int(hits["component_offset"][m]), int(hits["component_count"][m])
            if c <= 0:
                raise ValueError(f"missing hit_merged_components rows for hit_merged index {m}")
            h0[m] = c0[idx[o:o + c]].min()
            h1[m] = c1[idx[o:o + c]].max()
        a0, a1 = _dev(h0), _dev(h1)
        _lib.check(lib.wfb_group_abs_windows(_ptr(d_ts), _ptr(a0), _ptr(a1), _ptr(d_dt), _ptr(d_rid), nh, float(time_window_ns), _ptr(order),
                                             _ptr(ev), _ptr(n_ev), _ptr(ws), ws.numel(), _stream()), "wfb_group_abs_windows")
    else:
        d_pos = _dev(hits["position"].astype(np.int64))
        d_s, d_e = _dev(hits[sn].astype(np.int32)), _dev(hits[en].astype(np.int32))
        a0 = torch.empty(nh, dtype=torch.float64, device="cuda")
        a1 = torch.empty(nh, dtype=torch.float64, device="cuda")
        _lib.check(lib.wfb_group_hit_windows(_ptr(d_ts), _ptr(d_pos), _ptr(d_s), _ptr(d_e), _ptr(d_dt), _ptr(d_rid), nh, float(time_window_ns),
                                             _ptr(order), _ptr(ev), _ptr(a0), _ptr(a1), _ptr(n_ev), _ptr(ws), ws.numel(), _stream()),
                   "wfb_group_hit_windows")
    n_events = int(n_ev.item())
    t = _hit_event_table(order, ev, nh, n_events, _dev(hits["board"].astype(np.int16)), _dev(hits["channel"].astype(np.int16)), d_dt, a0, a1)
    host = {k: t[k].cpu().numpy() for k in ("offsets", "members", "t_min", "t_max", "dt_ns", "n_hits")}
    return dict(event_id=np.arange(n_events, dtype=np.int64), t_min=host["t_min"], t_max=host["t_max"], dt_ns=host["dt_ns"],
                n_hits=host["n_hits"], offsets=host["offsets"], members=host["members"], event_of_hit=ev.cpu().numpy(),
                order=order.cpu().numpy())


def _hit_event_table(d_order, d_event_id, n: int, n_events: int, d_board, d_channel, d_dt, d_abs_start, d_abs_end, *, rows=None,
                     row_bytes: int = 0) -> dict:
    """wfb_hit_event_table on device columns indexed by input row (``order`` / ``event_id`` as the grouping wrote them):
    device tensors ``offsets``, ``members``, ``t_min``, ``t_max``, ``dt_ns``, ``n_hits`` and - when ``rows`` (packed rows
    of ``row_bytes``) is given - ``member_rows`` (uint8, the rows in member order)."""
    lib = _lib.load()
    torch = _torch()
    n, n_events = int(n), int(n_events)
    dev = "cuda"
    out = dict(offsets=torch.zeros(n_events + 1, dtype=torch.int64, device=dev), members=torch.empty(n, dtype=torch.int64, device=dev),
               t_min=torch.empty(n_events, dtype=torch.int64, device=dev), t_max=torch.empty(n_events, dtype=torch.int64, device=dev),
               dt_ns=torch.empty(n_events, dtype=torch.float64, device=dev), n_hits=torch.empty(n_events, dtype=torch.int64, device=dev))
    if rows is not None:
        out["member_rows"] = torch.empty(n * int(row_bytes), dtype=torch.uint8, device=dev)
    if n == 0:
        return out
    ws = _empty(lib.wfb_hit_event_table_workspace_bytes(n))
    _lib.check(lib.wfb_hit_event_table(_ptr(d_order), _ptr(d_event_id), n, n_events, _ptr(d_board), _ptr(d_channel), _ptr(d_dt),
                                       _ptr(d_abs_start), _ptr(d_abs_end), _ptr(rows), int(row_bytes), _ptr(out["offsets"]), _ptr(out["members"]),
                                       _ptr(out["t_min"]), _ptr(out["t_max"]), _ptr(out["dt_ns"]), _ptr(out["n_hits"]), _ptr(out.get("member_rows")),
                                       _ptr(ws), ws.numel(), _stream()), "wfb_hit_event_table")
    return out


def group_time_window(timestamps: np.ndarray, channels: np.ndarray, time_window_ns: float) -> dict:
    """Anchored fixed-window clustering (event_grouping.py:99-283, 477-510) on the device: stable time sort, anchor
    search, event ids and the event table (members stably ordered by channel, t_min / t_max / dt/ns / n_hits).
    ``channels`` must fit int16 (the project's channel dtype)."""
    torch = _torch()
    ts_in = np.asarray(timestamps, dtype=np.int64)
    n = len(ts_in)
    if n == 0:
        z = np.zeros(0, dtype=np.int64)
        return dict(event_id=z, t_min=z, t_max=z, dt_ns=np.zeros(0), n_hits=z, offsets=np.zeros(1, np.int64), members=z)
    ch_in = np.asarray(channels)
    ch16 = ch_in.astype(np.int16)
    if len(ch16) != n or not np.array_equal(ch16, ch_in):
        raise ValueError("group_time_window: channels must be int16 values, one per timestamp")
    lib = _lib.load()
    d_ts = _dev(ts_in)
    d_sorted, d_order = torch.empty_like(d_ts), torch.empty_like(d_ts)
    ws = _empty(lib.wfb_sort_workspace_bytes(n))
    _lib.check(lib.wfb_sort_pairs_i64(_ptr(d_ts), _ptr(torch.arange(n, dtype=torch.int64, device="cuda")), _ptr(d_sorted), _ptr(d_order),
                                      n, _ptr(ws), ws.numel(), _stream()), "wfb_sort_pairs_i64")
    ev, n_events = group_time_window_device(d_sorted, n, time_window_ns)
    t = event_table_device(d_sorted, ev, n, n_events, _dev(ch16), order=d_order)
    host = {k: t[k].cpu().numpy() for k in ("offsets", "members", "t_min", "t_max", "dt_ns", "n_hits")}
    return dict(event_id=np.arange(n_events, dtype=np.int64), t_min=host["t_min"], t_max=host["t_max"], dt_ns=host["dt_ns"],
                n_hits=host["n_hits"], offsets=host["offsets"], members=host["members"])


def group_time_window_device(d_ts_sorted, n: int, time_window_ns: float):
    """wfb_group_time_window on time-sorted int64 timestamps already on the device: (event ids int64[n] tensor,
    number of events)."""
    lib = _lib.load()
    torch = _torch()
    n = int(n)
    ev = torch.empty(max(n, 1), dtype=torch.int64, device="cuda")
    if n == 0:
        return ev[:0], 0
    n_ev = torch.zeros(1, dtype=torch.int64, device="cuda")
    ws = _empty(lib.wfb_group_workspace_bytes(n))
    _lib.check(lib.wfb_group_time_window(_ptr(d_ts_sorted), n, float(time_window_ns), _ptr(ev), _ptr(n_ev), _ptr(ws), ws.numel(), _stream()),
               "wfb_group_time_window")
    return ev[:n], int(n_ev.item())


def event_table_device(d_ts_sorted, d_event_id, n: int, n_events: int, d_channel, *, order=None, area=None, height=None) -> dict:
    """wfb_event_table: the CSR event table of wfb_group_time_window's events, all device tensors: ``offsets``,
    ``members`` (input rows), ``t_min``, ``t_max``, ``dt_ns``, ``n_hits`` and the member-ordered ``member_ts``,
    ``member_channel`` and - when ``area`` / ``height`` (float32, by input row) are given - ``member_area`` /
    ``member_height``.  ``order``: sorted position -> input row (None: the rows are the sorted rows)."""
    lib = _lib.load()
    torch = _torch()
    n, n_events = int(n), int(n_events)
    dev = "cuda"
    out = dict(offsets=torch.zeros(n_events + 1, dtype=torch.int64, device=dev), members=torch.empty(n, dtype=torch.int64, device=dev),
               t_min=torch.empty(n_events, dtype=torch.int64, device=dev), t_max=torch.empty(n_events, dtype=torch.int64, device=dev),
               dt_ns=torch.empty(n_events, dtype=torch.float64, device=dev), n_hits=torch.empty(n_events, dtype=torch.int64, device=dev),
               member_ts=torch.empty(n, dtype=torch.int64, device=dev), member_channel=torch.empty(n, dtype=torch.int16, device=dev))
    if area is not None:
        out["member_area"] = torch.empty(n, dtype=torch.float32, device=dev)
    if height is not None:
        out["member_height"] = torch.empty(n, dtype=torch.float32, device=dev)
    if n == 0:
        return out
    ws = _empty(lib.wfb_event_table_workspace_bytes(n))
    _lib.check(lib.wfb_event_table(_ptr(d_ts_sorted), _ptr(d_event_id), n, n_events, _ptr(d_channel), _ptr(order), _ptr(area), _ptr(height),
                                   _ptr(out["offsets"]), _ptr(out["members"]), _ptr(out["t_min"]), _ptr(out["t_max"]), _ptr(out["dt_ns"]),
                                   _ptr(out["n_hits"]), _ptr(out["member_ts"]), _ptr(out["member_channel"]), _ptr(out.get("member_area")),
                                   _ptr(out.get("member_height")), _ptr(ws), ws.numel(), _stream()), "wfb_event_table")
    return out


# --------------------------------------------------------------------------------------------
# hit_merge (hit_merge.py:115-181, 256-322): ordering on the device, chain on the host-free path
# --------------------------------------------------------------------------------------------


def hit_merge_default(hits: np.ndarray):
    """merge_gap_ns <= 0 (the default): every hit is its own cluster, rows regrouped by
    (board, channel) and ordered by absolute window start (stable).  Device sorts."""
    nh = len(hits)
    if nh == 0:
        return (np.zeros(0, dtype=HIT_MERGE_CLUSTERS_DTYPE), np.zeros(0, dtype=HIT_MERGED_DTYPE),
                np.zeros(0, dtype=HIT_MERGED_COMPONENTS_DTYPE))
    ts = hits["timestamp"].astype(np.float64)
    a0 = ts + (hits["edge_start"].astype(np.float64) - hits["position"].astype(np.float64)) * (hits["dt"].astype(np.float64) * 1e3)
    # float64 keys -> order-preserving int64 (abs_start >= 0 for real data; general mapping kept)
    bits = a0.view(np.int64)
    keys = np.where(bits >= 0, bits, np.int64(-(2**63)) - bits - 1 + 0)  # negative floats reversed
    _, o1 = sort_pairs(keys, np.arange(nh, dtype=np.int64))
    ck = hits["board"].astype(np.int64)[o1] * 65536 + (hits["channel"].astype(np.int64)[o1] + 32768)
    _, order = sort_pairs(ck, o1)
    clusters = np.zeros(nh, dtype=HIT_MERGE_CLUSTERS_DTYPE)
    clusters["cluster_index"] = np.arange(nh)
    clusters["hit_index"] = order
    merged = np.zeros(nh, dtype=HIT_MERGED_DTYPE)
    h = hits[order]
    for f_out, f_in in (("position", "position"), ("height", "height"), ("integral", "integral"), ("sample_start", "edge_start"),
                        ("sample_end", "edge_end"), ("width", "width"), ("dt", "dt"), ("rise_time", "rise_time"),
                        ("fall_time", "fall_time"), ("timestamp", "timestamp"), ("board", "board"), ("channel", "channel"),
                        ("record_id", "record_id")):
        merged[f_out] = h[f_in]
    merged["component_offset"] = np.arange(nh)
    merged["component_count"] = 1
    comps = np.zeros(nh, dtype=HIT_MERGED_COMPONENTS_DTYPE)
    comps["merged_index"] = np.arange(nh)
    comps["hit_index"] = order
    return clusters, merged, comps


def hit_merge(hits: np.ndarray, *, merge_gap_ns: float = 0.0, max_total_width_ns: float = 10000.0):
    """hit_merge_clusters / hit_merged / hit_merged_components for any merge_gap_ns
    (hit_merge.py:115-181, 256-322): sort, certain-break flags, per-piece greedy replay and the
    merged rows all run on the device (wfb_hit_merge)."""
    nh = len(hits)
    if nh == 0:
        return (np.zeros(0, dtype=HIT_MERGE_CLUSTERS_DTYPE), np.zeros(0, dtype=HIT_MERGED_DTYPE),
                np.zeros(0, dtype=HIT_MERGED_COMPONENTS_DTYPE))
    if hits.dtype != THRESHOLD_HIT_DTYPE:
        raise ValueError("hit_merge expects THRESHOLD_HIT_DTYPE rows")
    lib = _lib.load()
    torch = _torch()
    d_hits = upload(hits)
    d_order = torch.empty(nh, dtype=torch.int64, device="cuda")
    d_cidx = torch.empty(nh, dtype=torch.int64, device="cuda")
    d_merged = torch.empty(nh * HIT_MERGED_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
    d_ncl = torch.zeros(1, dtype=torch.int64, device="cuda")
    ws = _empty(lib.wfb_hit_merge_workspace_bytes(nh))
    _lib.check(lib.wfb_hit_merge(_ptr(d_hits), nh, float(merge_gap_ns), float(max_total_width_ns), _ptr(d_order), _ptr(d_cidx),
                                 _ptr(d_merged), _ptr(d_ncl), _ptr(ws), ws.numel(), _stream()), "wfb_hit_merge")
    ncl = int(d_ncl.item())
    clusters = np.zeros(nh, dtype=HIT_MERGE_CLUSTERS_DTYPE)
    clusters["cluster_index"] = d_cidx.cpu().numpy()
    clusters["hit_index"] = d_order.cpu().numpy()
    merged = d_merged[: ncl * HIT_MERGED_DTYPE.itemsize].cpu().numpy().view(HIT_MERGED_DTYPE).copy()
    comps = np.zeros(nh, dtype=HIT_MERGED_COMPONENTS_DTYPE)
    comps["merged_index"] = clusters["cluster_index"]
    comps["hit_index"] = clusters["hit_index"]
    return clusters, merged, comps


# --------------------------------------------------------------------------------------------
# CAEN V1725 binary ingest
# --------------------------------------------------------------------------------------------
def v1725_board_from_name(name) -> int:
    """Board id from the file name, 0 when absent (utils/formats/v1725.py:62-67)."""
    import os
    import re

    m = re.search(r"_b(\d+)", os.path.basename(str(name)), flags=re.IGNORECASE)
    return int(m.group(1)) if m else 0


def v1725_scan(blob) -> dict:
    """Header-chain index of one .bin stream (wfb_v1725_scan_host): one entry per waveform."""
    lib = _lib.load()
    buf = np.frombuffer(blob, dtype=np.uint8) if not isinstance(blob, np.ndarray) else np.ascontiguousarray(blob).view(np.uint8).reshape(-1)
    n_rec, n_tot = C.c_int64(0), C.c_int64(0)
    _lib.check(lib.wfb_v1725_scan_host(_hp(buf), len(buf), 0, None, None, None, None, None, None, C.byref(n_rec), C.byref(n_tot)),
               "wfb_v1725_scan_host")
    n = int(n_rec.value)
    cols = dict(payload_offset=np.empty(n, np.int64), n_samples=np.empty(n, np.int32), channel=np.empty(n, np.int16),
                timestamp=np.empty(n, np.int64), baseline=np.empty(n, np.uint16), trunc=np.empty(n, np.uint8))
    if n:
        _lib.check(lib.wfb_v1725_scan_host(_hp(buf), len(buf), n, _hp(cols["payload_offset"]), _hp(cols["n_samples"]), _hp(cols["channel"]),
                                           _hp(cols["timestamp"]), _hp(cols["baseline"]), _hp(cols["trunc"]), C.byref(n_rec), C.byref(n_tot)),
                   "wfb_v1725_scan_host")
    cols["n_samples_total"] = int(n_tot.value)
    cols["bytes"] = buf
    return cols


def _hp(a: np.ndarray | None):
    return C.c_void_p(0) if a is None or a.size == 0 else C.c_void_p(a.ctypes.data)


def build_records_from_v1725(blobs, names, dt_ns: int):
    """V1725 .bin streams (bytes / uint8 arrays, one per file, with their file names for the board id)
    -> (records[RECORDS_DTYPE], wave_pool[uint16]) in the reference's order
    (records_builder.py:798-830 build_records_from_v1725_files)."""
    up = v1725_upload([v1725_scan(b) for b in blobs], names)
    if up["n"] == 0:
        return np.zeros(0, dtype=RECORDS_DTYPE), np.zeros(0, dtype=np.uint16)
    rows, pool, _ = build_records_v1725_device(up, dt_ns)
    rec = rows[: up["n"] * 102].cpu().numpy().view(RECORDS_DTYPE)
    return rec, pool.cpu().numpy().view(np.uint16)


def v1725_upload(scans, names) -> dict:
    """The streams of ``scans`` (v1725_scan of each file, in list order) at 16-byte aligned bases of ONE device buffer
    and their index columns on the device (payload offsets rebased, board ids from ``names``)."""
    lib = _lib.load()
    torch = _torch()
    bases, cursor = [], 0
    for s in scans:
        bases.append(cursor)
        cursor += (len(s["bytes"]) + 15) & ~15
    d_blob = torch.empty(cursor + 16, dtype=torch.uint8, device="cuda")
    for s, base in zip(scans, bases):
        if len(s["bytes"]):
            _lib.check(lib.wfb_memcpy_h2d(C.c_void_p(d_blob.data_ptr() + base), _hp(s["bytes"]), len(s["bytes"]), _stream()), "wfb_memcpy_h2d")
    off = np.concatenate([s["payload_offset"] + base for s, base in zip(scans, bases)] or [np.zeros(0, np.int64)])
    board = np.concatenate([np.full(len(s["channel"]), v1725_board_from_name(nm), dtype=np.int16) for s, nm in zip(scans, names)]
                           or [np.zeros(0, np.int16)])
    up = {k: _dev(np.concatenate([s[k] for s in scans])) for k in ("n_samples", "channel", "timestamp", "baseline", "trunc")} if scans else {}
    up.update(blob=d_blob, blob_bytes=cursor, payload_offset=_dev(off), board=_dev(board), n=len(off),
              total=sum(s["n_samples_total"] for s in scans))
    return up


def build_records_v1725_device(up: dict, dt_ns: int, *, seq: np.ndarray | None = None, meta: bool = False):
    """wfb_build_records_v1725 (``seq`` given: wfb_build_records_v1725_seq, record_id = seq) on the output of
    v1725_upload -> device (rows uint8 [n * 102], pool int16 [total] with a 16-sample tail, meta uint8 [n * 48] or None)."""
    lib = _lib.load()
    torch = _torch()
    n, total = up["n"], up["total"]
    rows = _empty(n * 102)
    pool = torch.empty(total + 16, dtype=torch.int16, device="cuda")[:total]
    d_meta = torch.empty(max(n, 1) * 48, dtype=torch.uint8, device="cuda") if meta else None
    if n == 0:
        return rows, pool, d_meta
    ws = _empty(lib.wfb_build_records_v1725_workspace_bytes(n))
    cols = (_ptr(up["blob"]), up["blob_bytes"], _ptr(up["payload_offset"]), _ptr(up["n_samples"]), _ptr(up["timestamp"]), _ptr(up["board"]),
            _ptr(up["channel"]), _ptr(up["baseline"]), _ptr(up["trunc"]))
    tail = (n, int(dt_ns), _ptr(rows), _ptr(pool), total, _ptr(d_meta), _ptr(ws), ws.numel(), _stream())
    if seq is None:
        _lib.check(lib.wfb_build_records_v1725(*cols, *tail), "wfb_build_records_v1725")
    else:
        d_seq = _dev(np.ascontiguousarray(seq, dtype=np.int64))
        if len(d_seq) != n:
            raise ValueError(f"seq has {len(d_seq)} entries for {n} waveforms")
        _lib.check(lib.wfb_build_records_v1725_seq(*cols, _ptr(d_seq), *tail), "wfb_build_records_v1725_seq")
    return rows, pool, d_meta


def record_split_points(rows, n: int, keys: np.ndarray) -> np.ndarray:
    """wfb_record_split_points: lower bound of every key (int64 rows of timestamp, board, channel, record_id) among
    the first ``n`` sorted RECORDS rows of the device tensor ``rows``."""
    lib = _lib.load()
    k = np.ascontiguousarray(keys, dtype=np.int64).reshape(-1, 4)
    if len(k) == 0:
        return np.zeros(0, dtype=np.int64)
    d_k = _dev(k.reshape(-1))
    out = _torch().empty(len(k), dtype=_torch().int64, device="cuda")
    _lib.check(lib.wfb_record_split_points(_ptr(rows), int(n), _ptr(d_k), len(k), _ptr(out), _stream()), "wfb_record_split_points")
    return out.cpu().numpy()


def merge_record_runs(rows, pool, run_offsets, *, record_base: int, pool_base: int):
    """wfb_merge_record_runs: merge the sorted runs rows[run_offsets[r]:run_offsets[r + 1]] (device RECORDS rows, their
    samples concatenated in the same order in ``pool``) -> device (rows, pool with a 16-sample tail, meta), numbered
    from ``record_base`` / ``pool_base``."""
    lib = _lib.load()
    torch = _torch()
    ro = np.ascontiguousarray(run_offsets, dtype=np.int64)
    n, total = int(ro[-1]), int(pool.numel())
    out_rows = _empty(n * 102)
    out_pool = torch.empty(total + 16, dtype=torch.int16, device="cuda")[:total]
    meta = torch.empty(max(n, 1) * 48, dtype=torch.uint8, device="cuda")
    ws = _empty(lib.wfb_merge_record_runs_workspace_bytes(n, len(ro) - 1))
    _lib.check(lib.wfb_merge_record_runs(_ptr(rows), _ptr(pool), n, _hp(ro), len(ro) - 1, int(record_base), int(pool_base), _ptr(out_rows),
                                         _ptr(out_pool), total, _ptr(meta), _ptr(ws), ws.numel(), _stream()), "wfb_merge_record_runs")
    return out_rows, out_pool, meta


# --------------------------------------------------------------------------------------------
# hit = scipy.signal.find_peaks per record
# --------------------------------------------------------------------------------------------
def _find_peaks(records: np.ndarray, pool: np.ndarray, kind: int, *, use_derivative=True, height=30.0, distance=2, prominence=0.7,
                width=4, threshold=None, height_method="minmax", height_window_extension=4, cumsum_diff=False,
                level_f32: bool = False, run: DeviceRun | None = None) -> np.ndarray:
    from .dtypes import HIT_DTYPE

    lib = _lib.load()
    torch = _torch()
    if height_method not in ("minmax", "diff"):
        raise ValueError(f"不支持的峰高计算方法: {height_method}")  # the reference's message (peak_finding.py:611)
    if distance is not None and distance < 1:
        raise ValueError("`distance` must be greater or equal to 1")  # scipy's check
    n = len(records)
    if n == 0:
        return np.zeros(0, dtype=HIT_DTYPE)
    lmax = int(records["event_length"].max())
    if lmax <= 0:
        return np.zeros(0, dtype=HIT_DTYPE)
    if run is None:
        run = DeviceRun.from_host(records, pool)
    return find_peaks_collect(find_peaks_launch(run, kind, lmax, use_derivative=use_derivative, height=height, distance=distance,
                                                prominence=prominence, width=width, threshold=threshold, height_method=height_method,
                                                height_window_extension=height_window_extension, cumsum_diff=cumsum_diff,
                                                level_f32=level_f32))


def find_peaks_launch(run: DeviceRun, kind: int, lmax: int, *, use_derivative=True, height=30.0, distance=2, prominence=0.7, width=4,
                      threshold=None, height_method="minmax", height_window_extension=4, cumsum_diff=False, level_f32=False,
                      cap: int | None = None) -> dict:
    """Enqueue ``wfb_find_peaks`` for a device-resident run on the current stream; nothing is read back (the streaming
    backend launches chunk k + 1 before it collects chunk k)."""
    lib = _lib.load()
    torch = _torch()
    n = run.n
    p = _lib.PeakParams(wave_kind=kind, use_derivative=int(bool(use_derivative)), height=float(height), prominence=float(prominence),
                        width=float(width), threshold=float(threshold) if threshold is not None else 0.0,
                        has_threshold=int(threshold is not None), distance=int(distance if distance is not None else 1),
                        height_method=0 if height_method == "minmax" else (2 if cumsum_diff else 1),
                        height_window_extension=int(height_window_extension),
                        lmax=int(lmax), level_f32=int(bool(level_f32)), pool_base=run.pool_base)
    ws = _empty(lib.wfb_find_peaks_workspace_bytes(n))
    total = torch.zeros(1, dtype=torch.int64, device="cuda")
    cap = max(1024, 2 * n) if cap is None else int(cap)
    rows = _empty(cap * 48)
    _lib.check(lib.wfb_find_peaks(_ptr(run.pool), run.pool_len, _ptr(run.meta), n, C.byref(p), _ptr(rows), cap, C.c_void_p(0),
                                  _ptr(total), _ptr(ws), ws.numel(), _stream()), "wfb_find_peaks")
    total_h = torch.empty(1, dtype=torch.int64, pin_memory=True)
    total_h.copy_(total, non_blocking=True)
    return dict(run=run, params=p, ws=ws, total=total, total_h=total_h, rows=rows, cap=cap)


def find_peaks_finish(job: dict):
    """Wait for a ``find_peaks_launch`` and return its HIT_DTYPE rows as (device uint8 tensor, row count); launches
    again with a row buffer of the right size when the first one was too small."""
    from .dtypes import HIT_DTYPE

    lib = _lib.load()
    torch = _torch()
    torch.cuda.current_stream().synchronize()
    run, p = job["run"], job["params"]
    nt = int(job["total_h"][0])
    rows, cap = job["rows"], job["cap"]
    while nt > cap:
        cap = nt
        rows = _empty(cap * HIT_DTYPE.itemsize)
        job["total"].zero_()
        _lib.check(lib.wfb_find_peaks(_ptr(run.pool), run.pool_len, _ptr(run.meta), run.n, C.byref(p), _ptr(rows), cap, C.c_void_p(0),
                                      _ptr(job["total"]), _ptr(job["ws"]), job["ws"].numel(), _stream()), "wfb_find_peaks")
        nt = int(job["total"].item())
    return rows, nt


def find_peaks_device(run: DeviceRun, kind: int, lmax: int, **opts):
    """``wfb_find_peaks`` on a device-resident run (a time shard included: the records sources read
    ``wave_offset - run.pool_base``): (packed HIT_DTYPE rows as a device uint8 tensor, row count).  The rows stay on
    the device; ``opts`` as ``find_peaks_launch`` takes them."""
    return find_peaks_finish(find_peaks_launch(run, kind, lmax, **opts))


def find_peaks_collect(job: dict) -> np.ndarray:
    """Wait for a ``find_peaks_launch`` and return its HIT_DTYPE rows on the host."""
    from .dtypes import HIT_DTYPE

    rows, nt = find_peaks_finish(job)
    return rows[: nt * HIT_DTYPE.itemsize].cpu().numpy().view(HIT_DTYPE).copy()


def find_peaks_records(records: np.ndarray, pool: np.ndarray, run: DeviceRun | None = None, **opts) -> np.ndarray:
    """`hit` rows from records + wave_pool / wave_pool_filtered (peak_finding.py:392-444: waveform =
    -RecordsView.signals() in float64, positive-going pulses).  ``run``: the device-resident copy, if there is one."""
    pool_h, is_f32 = check_pool(pool)
    return _find_peaks(packed_records(records, None), pool_h, _lib.WAVE_REC_F32 if is_f32 else _lib.WAVE_REC_U16, run=run, **opts)


def find_peaks_waveforms(data: np.ndarray, *, explicit_dt=None, **opts) -> np.ndarray:
    """`hit` rows from st_waveforms / filtered_waveforms rows used in place (peak_finding.py:326-390:
    negative pulses, detection on -diff(wave) or baseline - wave, rows truncated to event_length)."""
    from .aos import structured_as_records

    names = data.dtype.names or ()
    if "dt" not in names and explicit_dt is None:
        raise ValueError("[hit] st_waveforms is missing required field 'dt'; provide explicit config 'dt'.")
    rec, pool, signed = structured_as_records(data, explicit_dt=explicit_dt)
    if pool.dtype == np.float32:
        kind = _lib.WAVE_AOS_F32
    elif signed:
        kind = _lib.WAVE_AOS_I16
    else:
        kind = _lib.WAVE_AOS_U16  # np.diff / negation of uint16 rows wrap modulo 65536, as in the reference
    L = int(rec["event_length"][0]) if len(rec) else 0
    if "event_length" in names and len(data):
        el = data["event_length"].astype(np.int64)
        rec["event_length"] = np.where((el > 0) & (el < L), el, L)
    level_f32 = False
    if "baseline" not in names and len(data) and not opts.get("use_derivative", True):
        # no baseline field: the level is np.mean of the (truncated) row, in the row's own mean dtype
        # (peak_finding.py:508-511: float64 for integer rows, float32 for float32 rows)
        lens = rec["event_length"].astype(np.int64)
        wave = data["wave"]
        if np.all(lens == L):
            means = wave.mean(axis=1)
        else:
            means = np.array([wave[i, : lens[i]].mean() for i in range(len(data))])
        rec["baseline"] = means.astype(np.float64)
        level_f32 = pool.dtype == np.float32
    rec["polarity"] = "unknown"
    return _find_peaks(rec, pool, kind, level_f32=level_f32, **opts)


def peaks_stream_inputs(st_chunk: np.ndarray, filtered_chunk: np.ndarray, *, explicit_dt=None, event_offset=0, use_derivative=True):
    """Host side of one signal_peaks_stream chunk: (records rows, float32 pool) or None for an empty chunk."""
    from .aos import structured_as_records

    n = min(len(st_chunk), len(filtered_chunk))
    if n == 0:
        return None
    st_chunk, filtered_chunk = st_chunk[:n], filtered_chunk[:n]
    names = st_chunk.dtype.names or ()
    if filtered_chunk.dtype.names and "wave" in filtered_chunk.dtype.names:
        rec, pool, _ = structured_as_records(filtered_chunk, explicit_dt=explicit_dt)
    else:  # plain 2-D array of filtered rows
        rows = np.ascontiguousarray(filtered_chunk, dtype=np.float32)
        pool = rows.reshape(-1)
        rec = np.zeros(n, dtype=RECORDS_DTYPE)
        rec["wave_offset"] = np.arange(n, dtype=np.int64) * rows.shape[1]
        rec["event_length"] = rows.shape[1]
    if pool.dtype != np.float32:
        pool = pool.astype(np.float32)  # the plugin promotes whatever dtype the rows have to float64; float32 rows are exact
    rec["timestamp"] = st_chunk["timestamp"]
    rec["channel"] = st_chunk["channel"]
    rec["board"] = st_chunk["board"] if "board" in names else 0
    if "baseline" in names:
        rec["baseline"] = st_chunk["baseline"]
    elif not use_derivative:  # np.mean of the float64 copy of the row (signal_peaks.py:318-320)
        L = int(rec["event_length"][0])
        offs = rec["wave_offset"].astype(np.int64)
        rows64 = pool[(offs[:, None] + np.arange(L)[None, :])].astype(np.float64)
        rec["baseline"] = rows64.mean(axis=1)
    if "dt" in names:
        rec["dt"] = st_chunk["dt"]
    elif explicit_dt is not None:
        rec["dt"] = int(explicit_dt)
    else:
        raise ValueError("[signal_peaks_stream] st_waveforms is missing required field 'dt'; provide explicit config 'dt'.")
    if np.any(rec["dt"] <= 0):
        raise ValueError("[signal_peaks_stream] dt must be > 0")
    rec["record_id"] = st_chunk["record_id"] if "record_id" in names else int(event_offset) + np.arange(n, dtype=np.int64)
    rec["polarity"] = "unknown"
    return rec, pool


def find_peaks_stream_chunk(st_chunk: np.ndarray, filtered_chunk: np.ndarray, *, explicit_dt=None, event_offset=0, use_derivative=True,
                            height=30.0, distance=2, prominence=0.7, width=4, threshold=None, height_method="diff",
                            minmax_window_expand=2) -> np.ndarray:
    """One chunk of signal_peaks_stream (plugins/builtin/streaming/cpu/signal_peaks.py:234-401): metadata from
    the st_waveforms rows, samples from the filtered rows promoted to float64."""
    from .dtypes import HIT_DTYPE

    inp = peaks_stream_inputs(st_chunk, filtered_chunk, explicit_dt=explicit_dt, event_offset=event_offset, use_derivative=use_derivative)
    if inp is None:
        return np.zeros(0, dtype=HIT_DTYPE)
    rec, pool = inp
    return _find_peaks(rec, pool, _lib.WAVE_AOS_F32_AS_F64, use_derivative=use_derivative, height=height, distance=distance,
                       prominence=prominence, width=width, threshold=threshold, height_method=height_method,
                       height_window_extension=minmax_window_expand, cumsum_diff=True)


# --------------------------------------------------------------------------------------------
# the step after the path: df / s1_s2 / df_paired (dataframe.py:192-311, s1_s2_classifier.py:133-228,
# analyzer.py:66-110)
# --------------------------------------------------------------------------------------------


def df_columns(features: np.ndarray, record_id: np.ndarray | None = None, gains: dict | None = None) -> dict:
    """Columns of the `df` DataFrame in timestamp order (stable) plus ``order`` (the DataFrame index).
    ``gains``: {(board, channel): gain_adc_per_pe > 0} or None (no calibrated columns)."""
    from .dtypes import BASIC_FEATURES_DTYPE

    features = np.ascontiguousarray(features)
    if features.dtype != BASIC_FEATURES_DTYPE:
        raise ValueError("df_columns expects packed BASIC_FEATURES rows")
    n = len(features)
    d_feat = _dev(features) if n else None
    d_rid = _dev(np.asarray(record_id, dtype=np.int64)) if record_id is not None and n else None
    cols = df_columns_device(d_feat, n, d_rid, gains)
    return {k: v.cpu().numpy() for k, v in cols.items()}


def df_columns_device(d_feat, n: int, d_record_id=None, gains: dict | None = None) -> dict:
    """``df_columns`` on packed BASIC_FEATURES rows that live on the device (uint8 tensor, 36 B per row) with an
    optional int64 device ``record_id`` column: the same columns, left on the device."""
    lib = _lib.load()
    torch = _torch()
    n = int(n)
    with_pe = gains is not None
    cols = dict(order=torch.empty(n, dtype=torch.int64, device="cuda"), timestamp=torch.empty(n, dtype=torch.int64, device="cuda"),
                record_id=torch.empty(n, dtype=torch.int64, device="cuda"), area=torch.empty(n, dtype=torch.float32, device="cuda"),
                height=torch.empty(n, dtype=torch.float32, device="cuda"), amp=torch.empty(n, dtype=torch.float32, device="cuda"),
                max_abs_diff=torch.empty(n, dtype=torch.float32, device="cuda"), board=torch.empty(n, dtype=torch.int16, device="cuda"),
                channel=torch.empty(n, dtype=torch.int16, device="cuda"))
    if with_pe:
        cols["area_pe"] = torch.empty(n, dtype=torch.float64, device="cuda")
        cols["height_pe"] = torch.empty(n, dtype=torch.float64, device="cuda")
    if n:
        rules = (_lib.GainRule * max(len(gains or {}), 1))()
        for i, ((b, c), g) in enumerate((gains or {}).items()):
            rules[i].board, rules[i].channel, rules[i].gain = int(b), int(c), float(g)
        ws = _empty(lib.wfb_df_columns_workspace_bytes(n))
        _lib.check(lib.wfb_df_columns(_ptr(d_feat), _ptr(d_record_id) if d_record_id is not None else None, n, rules, len(gains or {}), int(with_pe),
                                      _ptr(cols["order"]), _ptr(cols["timestamp"]), _ptr(cols["record_id"]), _ptr(cols["area"]),
                                      _ptr(cols["height"]), _ptr(cols["amp"]), _ptr(cols["max_abs_diff"]), _ptr(cols["board"]),
                                      _ptr(cols["channel"]), _ptr(cols["area_pe"]) if with_pe else None,
                                      _ptr(cols["height_pe"]) if with_pe else None, _ptr(ws), ws.numel(), _stream()), "wfb_df_columns")
        torch.cuda.current_stream().synchronize()  # `rules` (host) must outlive the staged copy
    return cols


def _range_struct(bounds) -> "_lib.Range":
    r = _lib.Range()
    if bounds is None:
        return r
    lo, hi = bounds
    r.present = 1
    if lo is not None:
        r.has_lo, r.lo = 1, float(lo)
    if hi is not None:
        r.has_hi, r.hi = 1, float(hi)
    return r


def s1s2_classify(widths: np.ndarray, features: np.ndarray, *, width_unit: str = "ns", s1_width_range=None, s2_width_range=None,
                  s1_area_range=None, s2_area_range=None, s1_height_range=None, s2_height_range=None,
                  conflict_policy: str = "unknown") -> np.ndarray:
    """Packed S1_S2_CLASSIFIER rows, one per waveform_width row; ranges are (lo, hi) with None = open,
    already normalised (a (None, None) range is passed as None)."""
    from .dtypes import BASIC_FEATURES_DTYPE, S1_S2_CLASSIFIER_DTYPE, WAVEFORM_WIDTH_DTYPE

    widths = np.ascontiguousarray(widths)
    features = np.ascontiguousarray(features)
    if widths.dtype != WAVEFORM_WIDTH_DTYPE or features.dtype != BASIC_FEATURES_DTYPE:
        raise ValueError("s1s2_classify expects packed WAVEFORM_WIDTH and BASIC_FEATURES rows")
    n = len(widths)
    if n == 0:
        return np.zeros(0, dtype=S1_S2_CLASSIFIER_DTYPE)
    out = s1s2_classify_device(_dev(widths), n, _dev(features) if len(features) else _empty(16), len(features), feat_row_base=0,
                               width_unit=width_unit, s1_width_range=s1_width_range, s2_width_range=s2_width_range,
                               s1_area_range=s1_area_range, s2_area_range=s2_area_range, s1_height_range=s1_height_range,
                               s2_height_range=s2_height_range, conflict_policy=conflict_policy)
    return out.cpu().numpy().view(S1_S2_CLASSIFIER_DTYPE)


def s1s2_classify_device(d_widths, n: int, d_feat, n_feat: int, *, feat_row_base: int = 0, width_unit: str = "ns", s1_width_range=None,
                         s2_width_range=None, s1_area_range=None, s2_area_range=None, s1_height_range=None, s2_height_range=None,
                         conflict_policy: str = "unknown"):
    """``s1s2_classify`` on packed rows that live on the device (uint8 tensors): ``n`` WAVEFORM_WIDTH rows and
    ``n_feat`` BASIC_FEATURES rows, the first of them for record ``feat_row_base`` (a time shard's ``row_base``).
    Returns the S1_S2_CLASSIFIER rows as a device uint8 tensor (45 B per row); the same normalised ranges."""
    from .dtypes import S1_S2_CLASSIFIER_DTYPE

    lib = _lib.load()
    torch = _torch()
    n = int(n)
    p = _lib.S1S2Params()
    p.s1_width, p.s1_area, p.s1_height = _range_struct(s1_width_range), _range_struct(s1_area_range), _range_struct(s1_height_range)
    p.s2_width, p.s2_area, p.s2_height = _range_struct(s2_width_range), _range_struct(s2_area_range), _range_struct(s2_height_range)
    p.width_in_samples = 1 if width_unit == "samples" else 0
    p.conflict_policy = {"unknown": 0, "prefer_s1": 1, "prefer_s2": 2}[conflict_policy]
    p.feat_row_base = int(feat_row_base)
    out = torch.empty(max(n, 1) * S1_S2_CLASSIFIER_DTYPE.itemsize, dtype=torch.uint8, device="cuda")[: n * S1_S2_CLASSIFIER_DTYPE.itemsize]
    _lib.check(lib.wfb_s1s2_classify(_ptr(d_widths) if n else None, n, _ptr(d_feat) if n_feat else None, int(n_feat), C.byref(p), _ptr(out),
                                     _stream()), "wfb_s1s2_classify")
    return out


def pair_events(offsets: np.ndarray, member_ts: np.ndarray, member_area: np.ndarray, member_height: np.ndarray, dt_ns: np.ndarray,
                time_window_ns: float, n_channels: int) -> dict:
    """keep mask, delta_t and the per-channel area / height columns of `df_paired` for CSR events."""
    lib = _lib.load()
    torch = _torch()
    offsets = np.asarray(offsets, dtype=np.int64)
    n_ev = len(offsets) - 1
    nc = int(n_channels)
    if n_ev <= 0:
        return dict(keep=np.zeros(0, bool), delta_t=np.zeros(0), area_ch=np.zeros((0, nc), np.float32), height_ch=np.zeros((0, nc), np.float32))
    d_off, d_ts = _dev(offsets), _dev(np.asarray(member_ts, dtype=np.int64))
    d_a, d_h = _dev(np.asarray(member_area, dtype=np.float32)), _dev(np.asarray(member_height, dtype=np.float32))
    d_dt = _dev(np.asarray(dt_ns, dtype=np.float64))
    out = pair_events_device(d_off, n_ev, d_ts, d_a, d_h, d_dt, time_window_ns, nc)
    return dict(keep=out["keep"].cpu().numpy().astype(bool), delta_t=out["delta_t"].cpu().numpy(),
                area_ch=out["area_ch"].cpu().numpy(), height_ch=out["height_ch"].cpu().numpy())


def pair_events_device(d_offsets, n_events: int, d_member_ts, d_member_area, d_member_height, d_dt_ns, time_window_ns: float,
                       n_channels: int) -> dict:
    """wfb_pair_events on CSR events that live on the device: ``keep`` (uint8), ``delta_t`` and the (n_events,
    n_channels) ``area_ch`` / ``height_ch``, all device tensors."""
    lib = _lib.load()
    torch = _torch()
    n_ev, nc = int(n_events), int(n_channels)
    keep = torch.empty(n_ev, dtype=torch.uint8, device="cuda")
    delta = torch.empty(n_ev, dtype=torch.float64, device="cuda")
    a_ch = torch.empty(max(n_ev * nc, 1), dtype=torch.float32, device="cuda")
    h_ch = torch.empty(max(n_ev * nc, 1), dtype=torch.float32, device="cuda")
    if n_ev:
        _lib.check(lib.wfb_pair_events(_ptr(d_offsets), n_ev, _ptr(d_member_ts), _ptr(d_member_area), _ptr(d_member_height), _ptr(d_dt_ns),
                                       float(time_window_ns), nc, _ptr(keep), _ptr(delta), _ptr(a_ch), _ptr(h_ch), _stream()), "wfb_pair_events")
    return dict(keep=keep, delta_t=delta, area_ch=a_ch[: n_ev * nc].view(n_ev, nc), height_ch=h_ch[: n_ev * nc].view(n_ev, nc))


# --------------------------------------------------------------------------------------------
# device-resident hit_merge -> hit_grouped (time-sharded multi-GPU runs keep the rows in HBM)
# --------------------------------------------------------------------------------------------


def hit_merge_device(d_hits, n: int, *, merge_gap_ns: float = 0.0, max_total_width_ns: float = 10000.0) -> dict:
    """wfb_hit_merge on packed THRESHOLD_HIT rows that already live on the device (uint8 tensor, 60 B per row).
    Returns device tensors: ``order`` / ``cluster_index`` (int64[n]), ``merged`` (uint8, 72 B per cluster), the
    clusters' absolute windows ``abs_start`` / ``abs_end`` (float64) and ``n_clusters`` (int)."""
    lib = _lib.load()
    torch = _torch()
    n = int(n)
    order = torch.empty(max(n, 1), dtype=torch.int64, device="cuda")
    cidx = torch.empty(max(n, 1), dtype=torch.int64, device="cuda")
    merged = torch.empty(max(n, 1) * HIT_MERGED_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
    d_ncl = torch.zeros(1, dtype=torch.int64, device="cuda")
    if n:
        ws = _empty(lib.wfb_hit_merge_workspace_bytes(n))
        _lib.check(lib.wfb_hit_merge(_ptr(d_hits), n, float(merge_gap_ns), float(max_total_width_ns), _ptr(order), _ptr(cidx), _ptr(merged),
                                     _ptr(d_ncl), _ptr(ws), ws.numel(), _stream()), "wfb_hit_merge")
    ncl = int(d_ncl.item())
    a0 = torch.empty(max(ncl, 1), dtype=torch.float64, device="cuda")
    a1 = torch.empty(max(ncl, 1), dtype=torch.float64, device="cuda")
    _lib.check(lib.wfb_merged_abs_windows(_ptr(d_hits), _ptr(order), _ptr(merged), ncl, _ptr(a0), _ptr(a1), _stream()), "wfb_merged_abs_windows")
    return dict(order=order, cluster_index=cidx, merged=merged, abs_start=a0, abs_end=a1, n_clusters=ncl)


def group_rows_device(d_rows, n: int, row_bytes: int, time_window_ns: float, abs_start=None, abs_end=None) -> dict:
    """Chain clustering (event_grouping.py:287-471) of packed hit rows on the device: ``event_of_row`` (int64[n], in row
    order), ``n_events``, the sort ``order`` and the rows' ``dt`` / ``abs_start`` / ``abs_end`` (what
    ``hit_event_table_device`` takes); ``abs_start`` / ``abs_end`` default to the rows' own sample windows."""
    lib = _lib.load()
    torch = _torch()
    n = int(n)
    ev = torch.empty(max(n, 1), dtype=torch.int64, device="cuda")
    if n == 0:
        return dict(event_of_row=ev[:0], n_events=0, order=ev[:0])
    ts = torch.empty(n, dtype=torch.int64, device="cuda")
    dt = torch.empty(n, dtype=torch.int32, device="cuda")
    rid = torch.empty(n, dtype=torch.int64, device="cuda")
    own = abs_start is None
    if own:
        abs_start = torch.empty(n, dtype=torch.float64, device="cuda")
        abs_end = torch.empty(n, dtype=torch.float64, device="cuda")
    _lib.check(lib.wfb_hit_columns(_ptr(d_rows), n, int(row_bytes), _ptr(ts), _ptr(dt), _ptr(rid), _ptr(abs_start) if own else None,
                                   _ptr(abs_end) if own else None, _stream()), "wfb_hit_columns")
    order = torch.empty(n, dtype=torch.int64, device="cuda")
    n_ev = torch.zeros(1, dtype=torch.int64, device="cuda")
    ws = _empty(lib.wfb_group_workspace_bytes(n))
    _lib.check(lib.wfb_group_abs_windows(_ptr(ts), _ptr(abs_start), _ptr(abs_end), _ptr(dt), _ptr(rid), n, float(time_window_ns), _ptr(order),
                                         _ptr(ev), _ptr(n_ev), _ptr(ws), ws.numel(), _stream()), "wfb_group_abs_windows")
    return dict(event_of_row=ev, n_events=int(n_ev.item()), abs_start=abs_start, abs_end=abs_end, order=order, dt=dt)


def hit_event_table_device(d_rows, n: int, row_bytes: int, group: dict) -> dict:
    """wfb_hit_event_table on packed hit rows that stay on the device (uint8 tensor, ``row_bytes`` = 60 or 72 per row) and
    their grouping ``group`` (``group_rows_device``'s result): device tensors ``offsets``, ``members`` (row indices),
    ``t_min``, ``t_max``, ``dt_ns``, ``n_hits`` and ``member_rows`` (the packed rows in member order)."""
    n, rb = int(n), int(row_bytes)
    if n == 0:
        return _hit_event_table(None, None, 0, 0, None, None, None, None, None, rows=d_rows, row_bytes=rb)
    bc = d_rows[: n * rb].view(n, rb)[:, 48:52].contiguous().view(_torch().int16).view(n, 2)  # board, channel
    return _hit_event_table(group["order"], group["event_of_row"], n, group["n_events"], bc[:, 0].contiguous(), bc[:, 1].contiguous(),
                            group["dt"], group["abs_start"], group["abs_end"], rows=d_rows, row_bytes=rb)


def filter_run_device(run: DeviceRun, cfg: dict | None = None, *, filter_options: dict | None = None, channel_config=None,
                      run_id: str | None = None):
    """wfb_filter_pool on a device-resident run (benchmarks, multi-GPU shards): returns the float32 pool as a device
    tensor, nothing crosses PCIe.

    ``cfg`` (as ``filter_pool``'s ``default``): one configuration for every record.  ``filter_options`` (the
    ``B200WavePoolFilteredPlugin`` options named in ``FILTER_OPTION_NAMES``; missing ones take the plugin's defaults)
    with ``channel_config``: every channel of the run resolved the way the plugin resolves it for ``run_id``.  Each
    record gets its configuration and its Savitzky-Golay table (effective window min(window, L), forced odd, left
    unchanged when that is <= poly) from wfb_filter_plan on the device."""
    if (cfg is None) == (filter_options is None):
        raise ValueError("filter_run_device takes one of cfg and filter_options")
    if cfg is not None:
        plan = filter_plan(run, {}, cfg)
    else:
        from .plugins.filtering import channel_filter_configs

        per_channel, default = channel_filter_configs(shard_channels(run), filter_options, channel_config, run_id)
        plan = filter_plan(run, per_channel, None if per_channel else default)
    return _filter_launch(run, plan, run.pool_len, max(run.lmax, 1))

# --------------------------------------------------------------------------------------------
# st_waveforms: structured rows with the dual baseline (waveforms.py:644-799)
# --------------------------------------------------------------------------------------------


def structure_waveforms(timestamps_ps, boards, channels, samples, *, dt_ns: int, wave_length: int | None = None, baseline_window=(0, 40),
                        baselines=None, baseline_upstream=None, record_base: int = 0) -> np.ndarray:
    """Raw rows (input order) -> ``st_waveforms`` rows (``create_record_dtype(wave_length)``): baseline over the sample
    window, the upstream baseline carried along (NaN without one), samples truncated / zero padded to ``wave_length``."""
    from .dtypes import create_record_dtype

    lib = _lib.load()
    samples = np.ascontiguousarray(samples)
    if samples.dtype not in (np.int16, np.uint16) or samples.ndim != 2:
        raise ValueError(f"samples must be a 2-D int16 array, got {samples.dtype} {samples.shape}")
    n, L = samples.shape
    wl = int(L if wave_length is None else wave_length)
    dtype = create_record_dtype(wl)
    if n == 0:
        return np.zeros(0, dtype=dtype)
    d_s = upload(samples.reshape(-1), tail=16)
    d_ts = _dev(np.asarray(timestamps_ps, dtype=np.int64))
    d_b = _dev(np.asarray(boards, dtype=np.int16))
    d_c = _dev(np.asarray(channels, dtype=np.int16))
    d_bl = _dev(np.asarray(baselines, dtype=np.float64)) if baselines is not None else None
    d_up = _dev(np.asarray(baseline_upstream, dtype=np.float64)) if baseline_upstream is not None else None
    rows = _empty(n * dtype.itemsize)
    _lib.check(lib.wfb_structure_waveforms(_ptr(d_s), _ptr(d_ts), _ptr(d_b), _ptr(d_c), _ptr(d_bl), _ptr(d_up), n, L, wl, int(baseline_window[0]),
                                           int(baseline_window[1]), int(dt_ns), int(record_base), _ptr(rows), _stream()), "wfb_structure_waveforms")
    from .engine import to_host

    return to_host(rows[: n * dtype.itemsize]).view(dtype)


def build_records_from_st(st: np.ndarray, *, default_dt_ns: int = 1):
    """records + wave_pool from structured st_waveforms rows (records_builder.py:645-777): time sort and gather on the
    device, ``baseline`` / ``baseline_upstream`` / ``polarity`` of the rows carried into the records (:676-695).  The
    device sort gets the source row index in the baseline slot and hands it back in the sorted rows."""
    names = st.dtype.names or ()
    n = len(st)
    if n == 0:
        return np.zeros(0, dtype=RECORDS_DTYPE), np.zeros(0, dtype=np.uint16)
    L = st["wave"].shape[1]
    lens = np.clip(st["event_length"].astype(np.int64), 0, L) if "event_length" in names else np.full(n, L, dtype=np.int64)
    dts = st["dt"].astype(np.int64) if "dt" in names else np.full(n, int(default_dt_ns), dtype=np.int64)
    if len(np.unique(dts)) != 1:
        raise ValueError("build_records_from_st: rows with different dt are not supported on the device")
    boards = st["board"] if "board" in names else np.zeros(n, np.int16)
    waves = np.ascontiguousarray(st["wave"])
    if waves.dtype == np.int16 and waves.size and int(waves.min()) < 0:
        waves = np.clip(waves, 0, None)  # _clip_wave_to_uint16 (records_builder.py:760-768)
    if np.all(lens == L):
        rec, pool = build_records(st["timestamp"], boards, st["channel"], waves, dt_ns=int(dts[0]), baselines=np.arange(n, dtype=np.float64))
    else:
        raise ValueError("build_records_from_st: rows with event_length shorter than the row are not supported on the device")
    src = rec["baseline"].astype(np.int64)
    rec["baseline"] = st["baseline"][src] if "baseline" in names else 0.0
    rec["baseline_upstream"] = st["baseline_upstream"][src] if "baseline_upstream" in names else np.nan
    rec["polarity"] = st["polarity"][src] if "polarity" in names else "unknown"
    if "record_id" in names and np.all(st["record_id"] >= 0):  # the source ids survive the sort (:742-746)
        rec["record_id"] = st["record_id"][src]
    return rec, pool
