"""Host-side runtime over the C-ABI: device buffers (torch tensors as owners only), parameter
blocks, and the two ways into the fused pass:

  * ``process_host``  - reference-facing: host numpy records + wave_pool in, host rows out
                        (chunked H2D -> kernels -> D2H pipeline inside ``wfb_process_host``).
  * ``DeviceRun``     - device-resident records + pool for repeated passes (bench ``value``,
                        multi-GPU shards, plugin chains that reuse one upload).
"""

from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from .dtypes import (
    BASIC_FEATURES_DTYPE,
    RECORDS_DTYPE,
    THRESHOLD_HIT_DTYPE,
)

CHAN_RULE_DTYPE = np.dtype(
    [
        ("board", "i4"),
        ("channel", "i4"),
        ("threshold", "f8"),
        ("fixed_baseline", "f8"),
        ("has_threshold", "i4"),
        ("has_fixed_baseline", "i4"),
    ]
)
assert CHAN_RULE_DTYPE.itemsize == C.sizeof(_lib.ChanRule)


def _torch():
    import torch

    if not torch.cuda.is_available():
        raise RuntimeError("no CUDA device visible: the B200 plugins have no CPU fallback")
    return torch


def _ptr(t) -> C.c_void_p:
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _stream():
    return C.c_void_p(_torch().cuda.current_stream().cuda_stream)


def _hptr(a: np.ndarray | None) -> C.c_void_p:
    return C.c_void_p(a.ctypes.data) if a is not None else C.c_void_p(0)


_TORCH_DTYPES: dict = {}
PINNED_RESULT_MAX = 8 << 30  # larger results go through a pageable copy


def to_host(t) -> np.ndarray:
    """Device bytes -> a NEW host array for the caller.  Results of a megabyte and more land in pinned memory from
    torch's caching host allocator: a fresh pageable array costs a page fault per 4 KB on first touch (measured:
    1.4 GB of hit rows 640 ms pageable, 27 ms pinned), and the allocator hands a block back as soon as the caller
    (the Context replaces results by memmap views of its cache files) drops the array.  ``WFB_PINNED_RESULTS=0``
    switches to plain pageable arrays."""
    import os

    torch = _torch()
    t = t.contiguous()
    nbytes = t.numel() * t.element_size()
    if nbytes < (1 << 20) or nbytes > PINNED_RESULT_MAX or os.environ.get("WFB_PINNED_RESULTS", "1") == "0":
        return t.cpu().numpy()
    # block sizes rounded up to 8 MB: result sizes vary from call to call (hit counts), exact sizes would seldom find a
    # cached block and cudaHostAlloc costs ~0.3 ms per MB
    quantum = 8 << 20
    try:
        raw = torch.empty(-(-nbytes // quantum) * quantum, dtype=torch.uint8, pin_memory=True)
    except RuntimeError:  # no pinned memory left
        return t.cpu().numpy()
    h = raw[:nbytes].view(t.dtype).view(t.shape)
    h.copy_(t)
    return h.numpy()


def upload(a: np.ndarray, *, tail: int = 0):
    """Host array -> device tensor through ``wfb_memcpy_h2d``.  Takes whatever a Context hands to a plugin - pageable,
    read-only or ``np.memmap`` arrays (core/context_execution.py:241-251) - without ``torch.from_numpy`` (which wants
    writable memory).  uint16 travels as int16, structured / string arrays as bytes; ``tail`` extra elements are
    allocated behind the data (the kernels may read up to the next 16-byte boundary)."""
    torch = _torch()
    a = np.ascontiguousarray(a)
    if a.dtype == np.uint16:
        tdt, count = torch.int16, a.size
    elif a.dtype.names is not None or a.dtype.kind in "USV":
        tdt, count = torch.uint8, a.nbytes
    else:
        key = a.dtype.str
        if key not in _TORCH_DTYPES:
            _TORCH_DTYPES[key] = torch.from_numpy(np.empty(0, dtype=a.dtype)).dtype
        tdt, count = _TORCH_DTYPES[key], a.size
    t = torch.empty(count + int(tail), dtype=tdt, device="cuda")
    if a.nbytes:
        _lib.check(_lib.load().wfb_memcpy_h2d(C.c_void_p(t.data_ptr()), C.c_void_p(a.ctypes.data), a.nbytes, _stream()), "wfb_memcpy_h2d")
    return t[:count] if tail else t


# --------------------------------------------------------------------------------------------
# host-side argument preparation
# --------------------------------------------------------------------------------------------


def packed_records(records: np.ndarray, explicit_dt: int | None = None) -> np.ndarray:
    """Return ``records`` as a C-contiguous RECORDS_DTYPE array (no copy when it already is).

    Arrays with a subset of the fields (as RecordsView accepts, records_view.py:18-23) are
    widened with the defaults the reference plugins use: board/channel 0, polarity 'unknown',
    record_id = arange (basic_features.py:115-129), dt from ``explicit_dt``.
    """
    if records.dtype == RECORDS_DTYPE:
        return np.ascontiguousarray(records)
    names = records.dtype.names
    if names is None:
        raise ValueError("records must be a structured array")
    required = ("wave_offset", "event_length", "timestamp", "baseline")
    missing = [f for f in required if f not in names]
    if missing:
        raise ValueError(f"records missing required fields: {missing}")
    out = np.zeros(len(records), dtype=RECORDS_DTYPE)
    out["baseline_upstream"] = np.nan
    out["polarity"] = "unknown"
    out["record_id"] = np.arange(len(records), dtype=np.int64)
    for f in RECORDS_DTYPE.names:
        if f in names:
            out[f] = records[f]
    if "dt" not in names:
        if explicit_dt is None:
            raise ValueError("records is missing required field 'dt'; provide explicit config 'dt'")
        out["dt"] = int(explicit_dt)
    return out


def check_pool(pool: np.ndarray) -> tuple[np.ndarray, int]:
    if not isinstance(pool, np.ndarray):
        raise ValueError("wave_pool must be a numpy array")
    if pool.dtype == np.uint16:
        return np.ascontiguousarray(pool).reshape(-1), 0
    if pool.dtype == np.float32:
        return np.ascontiguousarray(pool).reshape(-1), 1
    raise ValueError(f"wave_pool dtype must be uint16 or float32, got {pool.dtype}")


def make_rules(thresholds: dict | None = None, fixed_baselines: dict | None = None) -> np.ndarray:
    """(board, channel) -> override tables -> wfb_chan_rule array."""
    keys = sorted(set(thresholds or {}) | set(k for k, v in (fixed_baselines or {}).items() if v is not None))
    rules = np.zeros(len(keys), dtype=CHAN_RULE_DTYPE)
    for i, (b, c) in enumerate(keys):
        rules[i]["board"], rules[i]["channel"] = int(b), int(c)
        if thresholds and (b, c) in thresholds:
            rules[i]["threshold"] = float(thresholds[(b, c)])
            rules[i]["has_threshold"] = 1
        if fixed_baselines and fixed_baselines.get((b, c)) is not None:
            rules[i]["fixed_baseline"] = float(fixed_baselines[(b, c)])
            rules[i]["has_fixed_baseline"] = 1
    return rules


def _slice_arg(v, default):
    if v is None:
        return default
    return int(v)


def make_params(
    *,
    flags: int,
    pool_is_f32: int,
    height_range=(40, 90),
    area_range=(0, None),
    threshold: float = 10.0,
    left_extension: int = 2,
    right_extension: int = 2,
    lmax: int = 0,
    n_rules: int = 0,
    rules_dev: int = 0,
    pool_base: int = 0,
    row_base: int = 0,
    signed_samples: bool = False,
) -> _lib.FHParams:
    p = _lib.FHParams()
    p.flags = int(flags)
    p.pool_is_f32 = int(pool_is_f32)
    p.height_start = _slice_arg(height_range[0], 0)
    p.height_end = _slice_arg(height_range[1], _lib.SLICE_END_NONE)
    p.area_start = _slice_arg(area_range[0], 0)
    p.area_end = _slice_arg(area_range[1], _lib.SLICE_END_NONE)
    p.threshold = float(threshold)
    p.left_extension = max(0, int(left_extension))
    p.right_extension = max(0, int(right_extension))
    p.lmax = int(lmax)
    p.n_rules = int(n_rules)
    p.rules_dev = rules_dev
    p.pool_base = int(pool_base)
    p.row_base = int(row_base)
    p.signed_samples = 1 if signed_samples else 0
    return p


# --------------------------------------------------------------------------------------------
# reference-facing call: host buffers in, host rows out
# --------------------------------------------------------------------------------------------


def process_host(
    records: np.ndarray,
    pool: np.ndarray,
    *,
    features: bool = True,
    hits: bool = True,
    height_range=(40, 90),
    area_range=(0, None),
    threshold: float = 10.0,
    left_extension: int = 2,
    right_extension: int = 2,
    thresholds: dict | None = None,
    fixed_baselines: dict | None = None,
    explicit_dt: int | None = None,
    want_counts: bool = False,
    hit_cap: int | None = None,
    chunk_records: int = 0,
    out_features: np.ndarray | None = None,
    out_hits: np.ndarray | None = None,
    signed_samples: bool = False,
    row_base: int = 0,
    lmax: int | None = None,
    keep_resident: bool = False,
    pinned_results: bool = False,
) -> dict:
    """Fused pass over host buffers through ``wfb_process_host``.  Returns a dict with
    ``features`` (BASIC_FEATURES_DTYPE), ``hits`` (THRESHOLD_HIT_DTYPE), ``counts`` (int32).

    Records are expected in ``wave_offset`` order (what the records plugins produce); any other order works too, the
    call then runs a second time with the pool range of every chunk taken over all of its records.

    ``keep_resident``: the chunks are uploaded into one device buffer that holds the whole pool (``wfb_process_host_resident``)
    and the result carries ``run``, the DeviceRun of the records + pool now resident in HBM.  ``pinned_results``: the row
    arrays come from torch's caching pinned allocator (see ``to_host``)."""
    lib = _lib.load()
    _torch()
    rec = packed_records(records, explicit_dt)
    pool, is_f32 = check_pool(pool)
    n = len(rec)
    flags = (_lib.DO_FEATURES if features else 0) | (_lib.DO_HITS if hits else 0)
    rules = make_rules(thresholds, fixed_baselines)
    if lmax is None:  # a shard of a run passes the run-wide maximum (hit_finder.py:364); 0 = the library scans the rows
        lmax = 0
    p = make_params(flags=flags, pool_is_f32=is_f32, height_range=height_range, area_range=area_range,
                    threshold=threshold, left_extension=left_extension, right_extension=right_extension,
                    lmax=max(lmax, 0), n_rules=len(rules), signed_samples=signed_samples, row_base=row_base)
    torch = _torch()

    def _rows(count, dtype):
        nbytes = int(count) * dtype.itemsize
        if pinned_results and (1 << 20) <= nbytes <= PINNED_RESULT_MAX:
            try:
                quantum = 8 << 20  # (see to_host)
                return torch.empty(-(-nbytes // quantum) * quantum, dtype=torch.uint8, pin_memory=True)[:nbytes].numpy().view(dtype)
            except RuntimeError:
                pass
        return np.empty(int(count), dtype=dtype)

    feat = None
    if features:
        feat = out_features if out_features is not None else _rows(n, BASIC_FEATURES_DTYPE)
    counts = np.empty(n, dtype=np.int32) if (hits and want_counts) else None
    d_pool = d_meta = None
    if keep_resident and n:
        d_pool = torch.empty(len(pool) + 16, dtype=torch.float32 if is_f32 else torch.int16, device="cuda")[: len(pool)]
        d_meta = torch.empty(n * 48, dtype=torch.uint8, device="cuda")
    cap = int(hit_cap) if hit_cap is not None else max(1024, 8 * n)
    if out_hits is not None:
        cap = len(out_hits)
    hit_rows = None
    n_hits = C.c_int64(0)
    while True:
        if out_hits is not None and len(out_hits) >= cap:
            hit_rows = out_hits  # caller-provided (e.g. pinned) output rows
        else:
            hit_rows = _rows(cap if hits else 0, THRESHOLD_HIT_DTYPE)
        args = (_hptr(rec), n, _hptr(pool), len(pool), C.byref(p), _hptr(rules if len(rules) else None), _hptr(feat),
                _hptr(hit_rows if hits and cap else None), cap if hits else 0, _hptr(counts), C.byref(n_hits), int(chunk_records))
        if d_pool is not None:
            rc = lib.wfb_process_host_resident(*args, _ptr(d_pool), _ptr(d_meta))
        else:
            rc = lib.wfb_process_host(*args)
        _lib.check(rc, "wfb_process_host")
        if not hits or n_hits.value <= cap:
            break
        cap = int(n_hits.value)  # rare: more hits than the initial estimate, run again with room
    res = dict(features=feat, hits=hit_rows[: n_hits.value] if hits else None, counts=counts, n_hits=int(n_hits.value))
    if d_pool is not None:
        stats = np.zeros(3, dtype=np.int32)
        scratch = torch.empty(4, dtype=torch.int32, device="cuda")
        _lib.check(lib.wfb_meta_stats(_ptr(d_meta), n, _ptr(scratch), _hptr(stats), _stream()), "wfb_meta_stats")
        run = DeviceRun(d_meta, d_pool, n, is_f32, max(int(stats[0]), 0))
        run.dt_range = (int(stats[1]), int(stats[2]))
        res["run"] = run
    return res


# --------------------------------------------------------------------------------------------
# device-resident run
# --------------------------------------------------------------------------------------------


class DeviceRun:
    """records (as wfb_rec_meta) + wave_pool resident in HBM."""

    def __init__(self, meta, pool, n: int, pool_is_f32: int, lmax: int, records_rows=None, pool_base: int = 0, row_base: int = 0):
        self.meta = meta  # torch.uint8 [n*48]
        self.pool = pool  # torch tensor (uint16 stored as int16, or float32)
        self.n = int(n)
        self.pool_is_f32 = int(pool_is_f32)
        self.lmax = int(lmax)
        self.records_rows = records_rows
        self.pool_base = int(pool_base)
        self.row_base = int(row_base)
        self._ws = None
        self.dt_range = None  # (min, max) of the records' dt, when it was reduced on the device
        self.lmin = None  # shortest event_length, when it is known without a pass over the records (fixed-length runs)

    @property
    def pool_len(self) -> int:
        return int(self.pool.numel())

    @classmethod
    def from_host(cls, records: np.ndarray, pool: np.ndarray, explicit_dt: int | None = None, *, pool_base: int = 0, row_base: int = 0,
                  clamp_lengths: np.ndarray | None = None) -> "DeviceRun":
        torch = _torch()
        lib = _lib.load()
        rec = packed_records(records, explicit_dt)
        pool, is_f32 = check_pool(pool)
        n = len(rec)
        rows = upload(rec)
        d_pool = upload(pool, tail=16)
        meta = torch.empty(max(n, 1) * 48, dtype=torch.uint8, device="cuda")
        _lib.check(lib.wfb_records_unpack(_ptr(rows), n, _ptr(meta), _stream()), "wfb_records_unpack")
        if clamp_lengths is not None and n:
            d_clamp = upload(np.ascontiguousarray(clamp_lengths, dtype=np.int32))
            _lib.check(lib.wfb_meta_set_clamp(_ptr(meta), n, _ptr(d_clamp), _stream()), "wfb_meta_set_clamp")
            torch.cuda.current_stream().synchronize()
        # longest record and dt range from the device copy: no pass over the strided host rows
        stats = np.zeros(3, dtype=np.int32)
        scratch = torch.empty(4, dtype=torch.int32, device="cuda")
        _lib.check(lib.wfb_meta_stats(_ptr(meta), n, _ptr(scratch), _hptr(stats), _stream()), "wfb_meta_stats")
        run = cls(meta, d_pool, n, is_f32, max(int(stats[0]), 0), records_rows=rows, pool_base=pool_base, row_base=row_base)
        run.dt_range = (int(stats[1]), int(stats[2])) if n else None
        return run

    @classmethod
    def from_device_pool(cls, records: np.ndarray, d_pool, pool_is_f32: int = 0) -> "DeviceRun":
        """records rows from the host (small) + a sample pool that already lives on the device (it was produced there)."""
        torch = _torch()
        lib = _lib.load()
        rec = packed_records(records, None)
        n = len(rec)
        rows = upload(rec)
        meta = torch.empty(max(n, 1) * 48, dtype=torch.uint8, device="cuda")
        _lib.check(lib.wfb_records_unpack(_ptr(rows), n, _ptr(meta), _stream()), "wfb_records_unpack")
        lmax = int(rec["event_length"].max()) if n else 0
        return cls(meta, d_pool, n, int(pool_is_f32), max(lmax, 0), records_rows=rows)

    @classmethod
    def synth(cls, n: int, n_samples: int, n_channels: int, *, dt_ns: int = 2, seed: int = 1234, with_rows: bool = False,
              record_base: int = 0) -> "DeviceRun":
        """Synthetic run generated on the device.  ``record_base``: this is the time shard [record_base, record_base + n)
        of ONE run with that seed (timestamps, record ids and wave offsets are those of the whole run)."""
        torch = _torch()
        lib = _lib.load()
        pool = torch.empty(n * n_samples + 16, dtype=torch.int16, device="cuda")[: n * n_samples]
        meta = torch.empty(max(n, 1) * 48, dtype=torch.uint8, device="cuda")
        rows = torch.empty(n * 102, dtype=torch.uint8, device="cuda") if with_rows else None
        _lib.check(lib.wfb_synth_fill(_ptr(pool), _ptr(meta), _ptr(rows), n, n_samples, n_channels, dt_ns, seed, int(record_base), _stream()),
                   "wfb_synth_fill")
        run = cls(meta, pool, n, 0, n_samples, records_rows=rows, pool_base=int(record_base) * n_samples, row_base=int(record_base))
        run.lmin = n_samples
        return run

    def workspace(self):
        torch = _torch()
        need = _lib.load().wfb_features_hits_workspace_bytes(self.n)
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(need, dtype=torch.uint8, device="cuda")
        return self._ws

    def features_hits(
        self,
        *,
        features: bool = True,
        hits: bool = True,
        height_range=(40, 90),
        area_range=(0, None),
        threshold: float = 10.0,
        left_extension: int = 2,
        right_extension: int = 2,
        rules: np.ndarray | None = None,
        hit_cap: int | None = None,
        out=None,
        want_counts: bool = False,
        lmax: int | None = None,
        signed_samples: bool = False,
    ) -> dict:
        """One fused pass; returns device tensors (uint8 row buffers) + the int64 total tensor.
        Asynchronous: nothing is copied to the host."""
        torch = _torch()
        lib = _lib.load()
        flags = (_lib.DO_FEATURES if features else 0) | (_lib.DO_HITS if hits else 0)
        d_rules = None
        if rules is not None and len(rules):
            d_rules = upload(rules)
        p = make_params(flags=flags, pool_is_f32=self.pool_is_f32, height_range=height_range, area_range=area_range,
                        threshold=threshold, left_extension=left_extension, right_extension=right_extension,
                        lmax=self.lmax if lmax is None else lmax, n_rules=0 if d_rules is None else len(rules),
                        rules_dev=0 if d_rules is None else d_rules.data_ptr(), pool_base=self.pool_base, row_base=self.row_base,
                        signed_samples=signed_samples)
        out = out or {}
        n = self.n
        feat = out.get("features")
        if features and feat is None:
            feat = torch.empty(max(n, 1) * 36, dtype=torch.uint8, device="cuda")
        cap = int(hit_cap) if hit_cap is not None else max(1024, 8 * n)
        hit_rows = out.get("hits")
        if hits and hit_rows is None:
            hit_rows = torch.empty(max(cap, 1) * 60, dtype=torch.uint8, device="cuda")
        if hits and hit_rows is not None:
            cap = min(cap, hit_rows.numel() // 60) if hit_cap is not None else hit_rows.numel() // 60
        total = out.get("total")
        if total is None:
            total = torch.zeros(1, dtype=torch.int64, device="cuda")
        counts = out.get("counts")
        if hits and want_counts and counts is None:
            counts = torch.empty(max(n, 1), dtype=torch.int32, device="cuda")
        ws = self.workspace()
        rc = lib.wfb_features_hits(_ptr(self.pool), self.pool_len, _ptr(self.meta), n, C.byref(p), _ptr(feat if features else None),
                                   _ptr(hit_rows if hits else None), cap if hits else 0, _ptr(counts if hits else None),
                                   C.c_void_p(0), _ptr(total), _ptr(ws), ws.numel(), _stream())
        _lib.check(rc, "wfb_features_hits")
        return dict(features=feat, hits=hit_rows, total=total, counts=counts, cap=cap, rules=d_rules)

    def check(self):
        _lib.check(_lib.load().wfb_features_hits_check(_ptr(self.workspace()), _stream()), "wfb_features_hits")

    def run_to_host(self, **kw) -> dict:
        """features_hits + copy the rows to host numpy arrays (re-runs if the hit buffer was small)."""
        torch = _torch()
        res = self.features_hits(**kw)
        self.check()
        out = {}
        if res["features"] is not None and kw.get("features", True):
            out["features"] = to_host(res["features"][: self.n * 36]).view(BASIC_FEATURES_DTYPE)
        if kw.get("hits", True):
            total = int(res["total"].item())
            if total > res["cap"]:
                kw2 = dict(kw)
                kw2["hit_cap"] = total
                kw2.pop("out", None)
                res = self.features_hits(**kw2)
                torch.cuda.synchronize()
                total = int(res["total"].item())
            out["hits"] = to_host(res["hits"][: total * 60]).view(THRESHOLD_HIT_DTYPE)
            if res["counts"] is not None:
                out["counts"] = res["counts"][: self.n].cpu().numpy()
        return out

    def records_to_host(self) -> np.ndarray:
        if self.records_rows is None:
            raise ValueError("this DeviceRun holds no packed records rows")
        return self.records_rows.cpu().numpy().view(RECORDS_DTYPE)

    def pool_to_host(self) -> np.ndarray:
        a = self.pool.cpu().numpy()
        return a if self.pool_is_f32 else a.view(np.uint16)


# --------------------------------------------------------------------------------------------
# streaming: two device slots, chunk k + 1 uploads while chunk k computes
# --------------------------------------------------------------------------------------------


def records_host_scan(records_packed: np.ndarray, *, times: bool = False) -> dict:
    """One threaded pass over packed RECORDS rows on the host (``wfb_records_host_scan``; no device involved): the sample
    range the rows refer to, the longest record, the smallest dt and - with ``times`` - the timestamp / end time (ps)
    columns the chunk iteration needs."""
    rec = np.ascontiguousarray(records_packed)
    if rec.dtype != RECORDS_DTYPE:
        raise ValueError("records_host_scan expects packed RECORDS rows")
    n = len(rec)
    ts = np.empty(n, dtype=np.int64) if times else None
    end = np.empty(n, dtype=np.int64) if times else None
    stats = np.zeros(4, dtype=np.int64)
    _lib.check(_lib.load().wfb_records_host_scan(_hptr(rec) if n else C.c_void_p(0), n, _hptr(ts), _hptr(end), _hptr(stats)), "wfb_records_host_scan")
    return dict(lo=int(stats[0]), hi=int(stats[1]), lmax=int(stats[2]), dt_min=int(stats[3]), ts=ts, end=end)


class StagedChunk:
    """One chunk on its way through the device: slot buffers + the events that order the copy and the compute stream."""

    def __init__(self):
        self.slot = 0
        self.n = 0
        self.pool_len = 0
        self.pool_is_f32 = 0
        self.rows = self.pool = self.meta = None
        self.copied = self.done = None
        self.run = None
        self.out = {}


class StreamSlots:
    """Double-buffered host -> device staging for the streaming plugins (core/plugins/core/streaming.py:447-548 processes
    one chunk after the other on the host; here the chunks overlap on the device).

    ``stage`` enqueues the host-to-device copies of a chunk's packed record rows and of its sample range on the COPY
    stream (into the slot's device buffers); ``device_run`` makes the compute stream wait for them and unpacks the
    rows.  A slot is reused ``depth`` chunks later, after its owner has been finished (``finish`` waits for the slot's
    ``done`` event), so the upload of the next chunk(s) runs while the kernels of chunk k do."""

    def __init__(self, depth: int = 2):
        torch = _torch()
        self.depth = max(2, int(depth))
        self.copy_stream = torch.cuda.Stream()
        self.compute_stream = torch.cuda.Stream()
        self._dev = [dict() for _ in range(self.depth)]
        self._busy = [None] * self.depth
        self._k = 0
        self.bytes_uploaded = 0
        self.chunks = 0

    def _buffer(self, store: dict, name: str, nbytes: int, *, pinned: bool):
        torch = _torch()
        t = store.get(name)
        if t is None or t.numel() < nbytes:
            cap = max(int(nbytes * 1.25), 1 << 16)
            t = torch.empty(cap, dtype=torch.uint8, pin_memory=True) if pinned else torch.empty(cap, dtype=torch.uint8, device="cuda")
            store[name] = t
        return t

    def stage(self, records_packed: np.ndarray, pool: np.ndarray) -> StagedChunk:
        torch = _torch()
        slot = self._k % self.depth
        self._k += 1
        prev = self._busy[slot]
        if prev is not None and prev.done is not None:
            prev.done.synchronize()  # (already finished by the pipeline; a direct user of the class may not have)
        st = StagedChunk()
        st.slot = slot
        rec = np.ascontiguousarray(records_packed)
        pool, st.pool_is_f32 = check_pool(pool)
        st.n, st.pool_len = len(rec), len(pool)
        nb_rows, nb_pool = rec.nbytes, pool.nbytes
        d_rows = self._buffer(self._dev[slot], "rows", nb_rows + 64, pinned=False)
        d_pool = self._buffer(self._dev[slot], "pool", nb_pool + 64, pinned=False)
        # straight from the caller's arrays: DMA at link speed when they are pinned, the driver's staged copy when they are
        # pageable or memmap views (then the call returns once the source has been read, which is all the slot logic needs)
        lib = _lib.load()
        cs = C.c_void_p(self.copy_stream.cuda_stream)
        if nb_rows:
            _lib.check(lib.wfb_memcpy_h2d_async(_ptr(d_rows), C.c_void_p(rec.ctypes.data), nb_rows, cs), "wfb_memcpy_h2d_async")
        if nb_pool:
            _lib.check(lib.wfb_memcpy_h2d_async(_ptr(d_pool), C.c_void_p(pool.ctypes.data), nb_pool, cs), "wfb_memcpy_h2d_async")
        st.copied = torch.cuda.Event()
        st.copied.record(self.copy_stream)
        st.host_refs = (rec, pool)  # keep the sources alive until the copy has run
        st.rows = d_rows
        st.pool = d_pool[:nb_pool].view(torch.float32 if st.pool_is_f32 else torch.int16)
        self._busy[slot] = st
        self.bytes_uploaded += nb_rows + nb_pool
        self.chunks += 1
        return st

    def device_run(self, st: StagedChunk, *, lmax: int, pool_base: int = 0, row_base: int = 0) -> "DeviceRun":
        """Call inside ``with torch.cuda.stream(slots.compute_stream)``: the DeviceRun of the staged chunk."""
        torch = _torch()
        lib = _lib.load()
        torch.cuda.current_stream().wait_event(st.copied)
        meta = self._buffer(self._dev[st.slot], "meta", max(st.n, 1) * 48, pinned=False)
        _lib.check(lib.wfb_records_unpack(_ptr(st.rows), st.n, _ptr(meta), _stream()), "wfb_records_unpack")
        st.meta = meta
        st.run = DeviceRun(meta, st.pool, st.n, st.pool_is_f32, int(lmax), records_rows=st.rows, pool_base=int(pool_base), row_base=int(row_base))
        return st.run

    def mark_done(self, st: StagedChunk) -> None:
        torch = _torch()
        st.done = torch.cuda.Event()
        st.done.record(torch.cuda.current_stream())

    @staticmethod
    def finish(st: StagedChunk) -> None:
        if st.done is not None:
            st.done.synchronize()

    def close(self) -> None:
        """Wait for everything the slots still have in flight (a consumer that abandons the stream, an exception in a
        chunk): the slot buffers go back to the allocator when this object dies and must not be in use then."""
        self.copy_stream.synchronize()
        self.compute_stream.synchronize()
