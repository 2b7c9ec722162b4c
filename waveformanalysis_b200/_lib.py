"""ctypes binding of libwfb200.so (the C-ABI declared in include/wfb200.h).

There is no CPU fallback: if the shared library is missing, or no CUDA device is visible when
a compute entry point is called, the call raises.  Status codes map onto the exceptions the
reference plugins raise (ValueError for bad inputs, RuntimeError otherwise) so that
Context's error wrapping (core/context_execution.py:150-176) keeps working.
"""

from __future__ import annotations

import ctypes as C
import os
import threading

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("WFB200_LIB") or os.path.join(HERE, "libwfb200.so")  # WFB200_LIB: development override

WFB_OK = 0
WFB_ERR_INVALID = -1
WFB_ERR_CUDA = -2
WFB_ERR_LAYOUT = -3
WFB_ERR_NOMEM = -4

DO_FEATURES = 1
DO_HITS = 2
SLICE_END_NONE = 2**63 - 1
MAX_SOS_SECTIONS = 16
MAX_CHANNEL_KEYS = 8192


class RecMeta(C.Structure):
    _fields_ = [
        ("timestamp", C.c_int64),
        ("baseline", C.c_double),
        ("wave_offset", C.c_int64),
        ("event_length", C.c_int32),
        ("dt", C.c_int32),
        ("board", C.c_int16),
        ("channel", C.c_int16),
        ("polarity", C.c_uint8),
        ("pad_", C.c_uint8 * 3),
        ("record_id", C.c_int64),
    ]


assert C.sizeof(RecMeta) == 48


class ChanRule(C.Structure):
    _fields_ = [
        ("board", C.c_int32),
        ("channel", C.c_int32),
        ("threshold", C.c_double),
        ("fixed_baseline", C.c_double),
        ("has_threshold", C.c_int32),
        ("has_fixed_baseline", C.c_int32),
    ]


assert C.sizeof(ChanRule) == 32


class FHParams(C.Structure):
    _fields_ = [
        ("flags", C.c_int32),
        ("pool_is_f32", C.c_int32),
        ("height_start", C.c_int64),
        ("height_end", C.c_int64),
        ("area_start", C.c_int64),
        ("area_end", C.c_int64),
        ("threshold", C.c_double),
        ("left_extension", C.c_int32),
        ("right_extension", C.c_int32),
        ("lmax", C.c_int32),
        ("n_rules", C.c_int32),
        ("rules_dev", C.c_void_p),
        ("pool_base", C.c_int64),
        ("row_base", C.c_int64),
        ("signed_samples", C.c_int32),
        ("reserved_", C.c_int32),
    ]


class FilterCfg(C.Structure):
    _fields_ = [
        ("type", C.c_int32),
        ("sg_window", C.c_int32),
        ("sg_poly", C.c_int32),
        ("n_sections", C.c_int32),
        ("sos", (C.c_double * 6) * MAX_SOS_SECTIONS),
        ("zi", (C.c_double * 2) * MAX_SOS_SECTIONS),
    ]


class WidthParams(C.Structure):
    _fields_ = [
        ("rise_low", C.c_double),
        ("rise_high", C.c_double),
        ("fall_high", C.c_double),
        ("fall_low", C.c_double),
        ("sampling_rate", C.c_double),
        ("interpolation", C.c_int32),
        ("wave_is_f32", C.c_int32),
    ]


_vp, _i64, _i32, _sz, _dbl = C.c_void_p, C.c_int64, C.c_int32, C.c_size_t, C.c_double

# name -> (restype, argtypes): exactly the prototypes of include/wfb200.h
class PeakParams(C.Structure):  # wfb_peak_params
    _fields_ = [("wave_kind", C.c_int32), ("use_derivative", C.c_int32), ("height", C.c_double), ("prominence", C.c_double),
                ("width", C.c_double), ("threshold", C.c_double), ("has_threshold", C.c_int32), ("distance", C.c_int32),
                ("height_method", C.c_int32), ("height_window_extension", C.c_int32), ("lmax", C.c_int32), ("level_f32", C.c_int32),
                ("pool_base", C.c_int64)]


class GainRule(C.Structure):  # wfb_gain_rule
    _fields_ = [("board", C.c_int32), ("channel", C.c_int32), ("gain", C.c_double)]


class Range(C.Structure):  # wfb_range
    _fields_ = [("lo", C.c_double), ("hi", C.c_double), ("has_lo", C.c_int32), ("has_hi", C.c_int32), ("present", C.c_int32),
                ("reserved_", C.c_int32)]


class S1S2Params(C.Structure):  # wfb_s1s2_params
    _fields_ = [("s1_width", Range), ("s1_area", Range), ("s1_height", Range), ("s2_width", Range), ("s2_area", Range),
                ("s2_height", Range), ("width_in_samples", C.c_int32), ("conflict_policy", C.c_int32), ("feat_row_base", C.c_int64)]


WAVE_AOS_I16, WAVE_AOS_F32, WAVE_REC_U16, WAVE_REC_F32, WAVE_AOS_F32_AS_F64, WAVE_AOS_U16 = 0, 1, 2, 3, 4, 5

PROTOTYPES = {
    "wfb_last_error": (C.c_char_p, []),
    "wfb_version": (C.c_int, []),
    "wfb_device_info": (C.c_int, [C.POINTER(C.c_int)] * 3 + [C.c_char_p, C.c_int]),
    "wfb_memcpy_h2d": (C.c_int, [_vp, _vp, C.c_size_t, _vp]),
    "wfb_memcpy_h2d_async": (C.c_int, [_vp, _vp, C.c_size_t, _vp]),
    "wfb_records_host_scan": (C.c_int, [_vp, C.c_int64, _vp, _vp, _vp]),
    "wfb_records_unpack": (C.c_int, [_vp, _i64, _vp, _vp]),
    "wfb_structure_waveforms": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _i64, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _i64, _vp, _vp]),
    "wfb_meta_set_clamp": (C.c_int, [_vp, _i64, _vp, _vp]),
    "wfb_meta_stats": (C.c_int, [_vp, _i64, _vp, _vp, _vp]),
    "wfb_hit_columns": (C.c_int, [_vp, _i64, C.c_int32, _vp, _vp, _vp, _vp, _vp, _vp]),
    "wfb_merged_abs_windows": (C.c_int, [_vp, _vp, _vp, _i64, _vp, _vp, _vp]),
    "wfb_build_records": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i64, _i32, _i32, _i32, _i32, _i64, _vp, _vp, _vp, _vp, _sz, _vp]),
    "wfb_build_records_workspace_bytes": (_sz, [_i64]),
    "wfb_features_hits_workspace_bytes": (_sz, [_i64]),
    "wfb_features_hits": (C.c_int, [_vp, _i64, _vp, _i64, C.POINTER(FHParams), _vp, _vp, _i64, _vp, _vp, _vp, _vp, _sz, _vp]),
    "wfb_features_hits_check": (C.c_int, [_vp, _vp]),
    "wfb_process_host": (C.c_int, [_vp, _i64, _vp, _i64, C.POINTER(FHParams), _vp, _vp, _vp, _i64, _vp, C.POINTER(_i64), _i64]),
    "wfb_process_host_resident": (C.c_int, [_vp, _i64, _vp, _i64, C.POINTER(FHParams), _vp, _vp, _vp, _i64, _vp, C.POINTER(_i64), _i64, _vp, _vp]),
    "wfb_release_cache": (C.c_int, []),
    "wfb_group_abs_windows": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i64, _dbl, _vp, _vp, _vp, _vp, _sz, _vp]),
    "wfb_build_records_ragged": (C.c_int, [_vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i32, _i32, _i32, _i64, _vp, _vp, _i64, _vp, _vp, _sz, _vp]),
    "wfb_build_records_ragged_seq": (C.c_int, [_vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i32, _i32, _i32, _i64, _vp, _vp, _i64, _vp, _vp,
                                               _sz, _vp]),
    "wfb_find_peaks_workspace_bytes": (_sz, [_i64]),
    "wfb_find_peaks": (C.c_int, [_vp, _i64, _vp, _i64, C.POINTER(PeakParams), _vp, _i64, _vp, _vp, _vp, _sz, _vp]),
    "wfb_v1725_scan_host": (C.c_int, [_vp, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, C.POINTER(_i64), C.POINTER(_i64)]),
    "wfb_build_records_v1725_workspace_bytes": (_sz, [_i64]),
    "wfb_build_records_v1725": (C.c_int, [_vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i32, _vp, _vp, _i64, _vp, _vp, _sz, _vp]),
    "wfb_build_records_v1725_seq": (C.c_int, [_vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i32, _vp, _vp, _i64, _vp, _vp, _sz, _vp]),
    "wfb_record_split_points": (C.c_int, [_vp, _i64, _vp, _i64, _vp, _vp]),
    "wfb_merge_record_runs_workspace_bytes": (_sz, [_i64, _i64]),
    "wfb_merge_record_runs": (C.c_int, [_vp, _vp, _i64, _vp, _i64, _i64, _i64, _vp, _vp, _i64, _vp, _vp, _sz, _vp]),
    "wfb_hit_merge_workspace_bytes": (_sz, [_i64]),
    "wfb_hit_merge": (C.c_int, [_vp, _i64, _dbl, _dbl, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "wfb_filter_pool": (C.c_int, [_vp, _i32, _i64, _vp, _i64, _vp, _i32, _vp, _vp, _vp, _vp, _i64, _vp, _sz, _i32, _vp]),
    "wfb_filter_workspace_bytes": (_sz, [_i64, _i32]),
    "wfb_filter_plan": (C.c_int, [_vp, _i64, _vp, _vp, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp]),
    "wfb_apply_polarity": (C.c_int, [_vp, _vp, _i64, _vp, _i32, _vp]),
    "wfb_waveform_width": (C.c_int, [_vp, _i64, _i32, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _i64, C.POINTER(WidthParams), _vp, _vp, _vp]),
    "wfb_waveform_width_run_workspace_bytes": (_sz, [_i64]),
    "wfb_waveform_width_run": (C.c_int, [_vp, _i32, _i64, _vp, _i64, _i64, _i64, _vp, _i64, C.POINTER(WidthParams), _vp, _vp, _vp, _sz, _vp]),
    "wfb_width_integral": (C.c_int, [_vp, _i32, _i64, _vp, _i64, _dbl, _dbl, _dbl, _i64, _i64, _vp, _vp]),
    "wfb_group_workspace_bytes": (_sz, [_i64]),
    "wfb_group_hit_windows": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _dbl, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "wfb_group_time_window": (C.c_int, [_vp, _i64, _dbl, _vp, _vp, _vp, _sz, _vp]),
    "wfb_event_table_workspace_bytes": (_sz, [_i64]),
    "wfb_event_table": (C.c_int, [_vp, _vp, _i64, _i64] + [_vp] * 14 + [_vp, _sz, _vp]),
    "wfb_hit_event_table_workspace_bytes": (_sz, [_i64]),
    "wfb_hit_event_table": (C.c_int, [_vp, _vp, _i64, _i64] + [_vp] * 6 + [_i32] + [_vp] * 7 + [_vp, _sz, _vp]),
    "wfb_df_columns_workspace_bytes": (_sz, [_i64]),
    "wfb_df_columns": (C.c_int, [_vp, _vp, _i64, _vp, _i32, _i32] + [_vp] * 11 + [_vp, _sz, _vp]),
    "wfb_s1s2_classify": (C.c_int, [_vp, _i64, _vp, _i64, C.POINTER(S1S2Params), _vp, _vp]),
    "wfb_pair_events": (C.c_int, [_vp, _i64, _vp, _vp, _vp, _vp, _dbl, _i32, _vp, _vp, _vp, _vp, _vp]),
    "wfb_sort_pairs_i64": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _vp, _sz, _vp]),
    "wfb_sort_workspace_bytes": (_sz, [_i64]),
    "wfb_synth_fill": (C.c_int, [_vp, _vp, _vp, _i64, _i32, _i32, _i32, C.c_uint64, _i64, _vp]),
}

_lib = None
_lock = threading.Lock()


def load() -> C.CDLL:
    """Load libwfb200.so (once).  Raises RuntimeError if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise RuntimeError(
                    f"{LIB_PATH} is missing: build it with `python -m waveformanalysis_b200.build` "
                    "(there is no CPU fallback for the B200 plugins)"
                )
            lib = C.CDLL(LIB_PATH)
            for name, (res, args) in PROTOTYPES.items():
                fn = getattr(lib, name, None)
                if fn is None:  # an outdated build: calling it raises AttributeError (tests/test_cabi_symbols.py
                    continue    # checks that a current build exports everything the header declares)
                fn.restype = res
                fn.argtypes = args
            _lib = lib
    return _lib


def last_error() -> str:
    msg = load().wfb_last_error()
    return msg.decode("utf-8", "replace") if msg else ""


def check(rc: int, what: str = "") -> None:
    if rc == WFB_OK:
        return
    msg = last_error() or f"libwfb200 error {rc}"
    if what:
        msg = f"{what}: {msg}"
    if rc in (WFB_ERR_INVALID, WFB_ERR_LAYOUT):
        raise ValueError(msg)
    if rc == WFB_ERR_NOMEM:
        raise MemoryError(msg)
    raise RuntimeError(msg)
