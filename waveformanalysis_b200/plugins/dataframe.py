"""df / df_paired / s1_s2 on the B200: the step after the hot path.

Reference: core/plugins/builtin/cpu/dataframe.py:31-311 (DataFramePlugin),
core/plugins/builtin/cpu/event_analysis.py:109-144 + core/processing/analyzer.py:66-110 (PairedEventsPlugin),
core/plugins/builtin/cpu/s1_s2_classifier.py:72-228 (S1S2ClassifierPlugin).  Same ``provides``, options and
outputs; the sort / gather / calibration, the range cuts and the per-event columns run on the device.
"""

from __future__ import annotations

import logging
import warnings
from collections.abc import Mapping
from typing import Any

import numpy as np

from .. import ops
from ..channel_config import parse_channel_ref
from ..dtypes import BASIC_FEATURES_DTYPE, S1_S2_CLASSIFIER_DTYPE, WAVEFORM_WIDTH_DTYPE
from ..plugin_api import Option, Plugin
from ..wave_source import WAVE_SOURCE_AUTO, load_wave_input, resolve_wave_input_spec

logger = logging.getLogger(__name__)


def resolve_gain_values(channel_config: Any, run_id: str, have_channels: bool, plugin_name: str) -> dict:
    """{(board, channel): gain > 0} from a gain_adc_per_pe mapping (core/hardware/channel.py:571-619)."""
    if not have_channels or channel_config is None:
        return {}
    if not isinstance(channel_config, Mapping):
        warnings.warn(f"Plugin '{plugin_name}' run '{run_id}': channel config must be dict-like, cannot resolve 'gain_adc_per_pe'.",
                      UserWarning, stacklevel=3)
        return {}
    selected = channel_config
    run_block = selected.get(run_id)
    if isinstance(run_block, Mapping):
        selected = run_block
    if isinstance(selected.get("channels"), Mapping):
        selected = selected["channels"]
    values: dict = {}
    invalid: list = []
    for key, raw in selected.items():
        hw = parse_channel_ref(key)
        if hw is None:
            raise ValueError(f'Invalid channel key {key!r}; expected HardwareChannel, (board, channel), or "board:channel".')
        if isinstance(raw, Mapping):
            raw = raw.get("gain_adc_per_pe")
        try:
            value = float(raw)
        except (TypeError, ValueError):
            if raw is not None:
                invalid.append(f"board{hw[0]}:ch{hw[1]}")
            continue
        if value <= 0:
            invalid.append(f"board{hw[0]}:ch{hw[1]}")
            continue
        values[hw] = value
    if invalid:
        warnings.warn(f"Plugin '{plugin_name}' run '{run_id}': invalid 'gain_adc_per_pe' entries -> " + ", ".join(sorted(invalid)),
                      UserWarning, stacklevel=3)
    return values


class B200DataFramePlugin(Plugin):
    """The single-channel events DataFrame: device sort by timestamp + column gather + PE calibration."""

    provides = "df"
    depends_on = []
    description = "Build the initial single-channel events DataFrame."
    version = "1.7.0"
    save_when = "always"
    uses_run_config = True
    options = {
        "use_filtered": Option(default=False, type=bool, help="use filtered_waveforms"),
        "wave_source": Option(default=WAVE_SOURCE_AUTO, type=str, help="auto|records|st_waveforms|filtered_waveforms"),
        "gain_adc_per_pe": Option(default=None, type=dict, help='ADC/PE gain per "board:channel"; adds area_pe / height_pe'),
    }

    def resolve_depends_on(self, context: Any, run_id: str | None = None) -> list:
        spec = resolve_wave_input_spec(context, self, needs_wave_samples=False)
        return list(spec.depends_on) + ["basic_features"]

    @staticmethod
    def _run_config_gain(run_config: Any) -> Any:  # dataframe.py:100-113
        if not isinstance(run_config, dict):
            return None
        calibration = run_config.get("calibration")
        if isinstance(calibration, dict) and isinstance(calibration.get("gain_adc_per_pe"), dict):
            return calibration.get("gain_adc_per_pe")
        if isinstance(run_config.get("gain_adc_per_pe"), dict):
            return run_config.get("gain_adc_per_pe")
        return None

    def _resolve_gain_map(self, context: Any, run_id: str, have_channels: bool) -> tuple:
        """explicit config > run_config.json > none (dataframe.py:115-190); (gains, enabled)."""
        gain = context.get_config(self, "gain_adc_per_pe")
        explicit = False
        has_explicit = getattr(context, "has_explicit_config", None)
        if callable(has_explicit):
            try:
                explicit = bool(has_explicit(self, "gain_adc_per_pe"))
            except Exception:
                explicit = False
        if explicit:
            if isinstance(gain, dict):
                return resolve_gain_values(gain, run_id, have_channels, self.provides), bool(gain)
            return {}, False
        if isinstance(gain, dict) and gain:
            return resolve_gain_values(gain, run_id, have_channels, self.provides), True
        getter = getattr(context, "get_run_config", None)
        if callable(getter):
            try:
                run_gain = self._run_config_gain(getter(run_id))
                if isinstance(run_gain, dict):
                    return resolve_gain_values(run_gain, run_id, have_channels, self.provides), bool(run_gain)
            except Exception as exc:
                logger.warning("Failed to resolve gain from run config for run '%s': %s", run_id, exc)
        return {}, False

    def compute(self, context: Any, run_id: str, **kwargs) -> Any:
        import pandas as pd

        features = context.get_data(run_id, "basic_features")
        wave_input = load_wave_input(context, self, run_id, needs_wave_samples=False)
        if not isinstance(features, np.ndarray):
            raise ValueError("df expects basic_features as a single structured array")
        if wave_input.spec.is_records:
            from .features import B200BasicFeaturesPlugin

            basic_spec = resolve_wave_input_spec(context, B200BasicFeaturesPlugin(), needs_wave_samples=True)
            if not basic_spec.is_records:
                raise ValueError("df.wave_source=records requires basic_features.wave_source=records "
                                 f"(resolved as {basic_spec.source!r}).")
            source = wave_input.records
            if source is None:
                raise ValueError("df failed to load records input")
            name = "records"
        else:
            source = wave_input.waveform_data
            name = wave_input.spec.data_name
            if source is None:
                raise ValueError(f"df failed to load {name}")
        if len(source) != len(features):
            raise ValueError(f"basic_features length ({len(features)}) != {name} length ({len(source)})")
        names = source.dtype.names or ()
        # timestamp / board / channel of the source rows are what basic_features carries (basic_features.py:
        # 233-278 copies them); a source without board / channel columns reads zeros (dataframe.py:232-241)
        feats = np.ascontiguousarray(features, dtype=BASIC_FEATURES_DTYPE).copy()
        feats["timestamp"] = np.asarray(source["timestamp"], dtype=np.int64)
        feats["board"] = np.asarray(source["board"], dtype=np.int16) if "board" in names else 0
        feats["channel"] = np.asarray(source["channel"], dtype=np.int16) if "channel" in names else 0
        rid = np.asarray(source["record_id"], dtype=np.int64) if "record_id" in names else None
        have_channels = len(feats) > 0
        gains, enabled = self._resolve_gain_map(context, run_id, have_channels)
        cols = ops.df_columns(feats, rid, gains if enabled else None)
        return df_frame(cols, cols["order"], enabled)


DF_COLUMNS = ("timestamp", "record_id", "area", "height", "amp", "max_abs_diff", "board", "channel")


def df_frame(cols: dict, index, with_pe: bool):
    """The `df` DataFrame of ``df_columns`` output (host arrays); ``index`` = the rows' labels."""
    import pandas as pd

    data = {k: cols[k] for k in DF_COLUMNS}
    if with_pe:
        data["area_pe"] = cols["area_pe"]
        data["height_pe"] = cols["height_pe"]
    # sort_values keeps the original row labels: the index is the sort permutation
    return pd.DataFrame(data, index=pd.Index(index, dtype=np.int64))


class B200PairedEventsPlugin(Plugin):
    """Events whose time span fits the window, with delta_t and the per-channel area / height columns."""

    provides = "df_paired"
    depends_on = ["df_events"]
    description = "Pair grouped events across channels for coincidence analysis."
    save_when = "always"

    def compute(self, context: Any, run_id: str, **kwargs) -> Any:
        df_events = context.get_data(run_id, "df_events")
        n_channels = int(context.config.get("n_channels", 2))
        start = int(context.config.get("start_channel_slice", 6))
        tw = context.config.get("time_window_ns", 100.0)
        return pair_events_frame(df_events, n_channels, start, tw)


def _csr_of(df_events, key: str, dtype) -> tuple:
    col = df_events[key].to_numpy()
    lens = np.fromiter((len(x) for x in col), dtype=np.int64, count=len(col))
    offsets = np.zeros(len(col) + 1, dtype=np.int64)
    np.cumsum(lens, out=offsets[1:])
    flat = np.concatenate([np.asarray(x, dtype=dtype) for x in col]) if len(col) and offsets[-1] else np.zeros(0, dtype=dtype)
    return offsets, flat


def pair_events_frame(df_events, n_channels: int, start_channel_slice: int, time_window_ns):
    """EventAnalyzer.pair_events (analyzer.py:66-110) with the row work on the device."""
    tw = 100 if time_window_ns is None else time_window_ns
    n = len(df_events)
    if n == 0:
        return df_events[df_events["dt/ns"] <= tw].copy()
    areas_key = "areas" if "areas" in df_events.columns else "charges"
    heights_key = "heights" if "heights" in df_events.columns else "peaks"
    from .grouping import member_arrays_of

    csr = member_arrays_of(df_events)
    if isinstance(csr, dict) and len(csr.get("offsets", ())) == n + 1:
        offsets, ts, area, height = csr["offsets"], csr["timestamps"], csr["areas"], csr["heights"]
    else:
        offsets, ts = _csr_of(df_events, "timestamps", np.int64)
        _, area = _csr_of(df_events, areas_key, np.float32)
        _, height = _csr_of(df_events, heights_key, np.float32)
    out = ops.pair_events(offsets, ts, area, height, df_events["dt/ns"].to_numpy(dtype=np.float64), float(tw), n_channels)
    return paired_frame(df_events, offsets, out, n_channels, start_channel_slice)


def paired_frame(df_events, offsets: np.ndarray, out: dict, n_channels: int, start_channel_slice: int):
    """df_paired from the events frame, its CSR ``offsets`` and the pair_events columns of ALL its events (``keep``,
    ``delta_t``, ``area_ch``, ``height_ch``).  The float64 widening of a per-channel column depends on every kept
    event, so this runs once on the whole run's events."""
    keep = out["keep"]
    df_paired = df_events[keep].copy()
    if "delta_t" not in df_paired.columns and not df_paired.empty:
        df_paired["delta_t"] = out["delta_t"][keep]
    if not df_paired.empty:
        short = (offsets[1:] - offsets[:-1])[keep]
        for i in range(n_channels):
            # a column with a missing member holds python NaN next to float32 scalars: pandas widens it to float64
            widen = bool((short <= i).any())
            a = out["area_ch"][keep, i]
            h = out["height_ch"][keep, i]
            df_paired[f"area_ch{start_channel_slice + i}"] = a.astype(np.float64) if widen else a
            df_paired[f"height_ch{start_channel_slice + i}"] = h.astype(np.float64) if widen else h
    return df_paired


def _normalize_range(value):  # s1_s2_classifier.py:45-53
    if value is None:
        return None
    if not isinstance(value, tuple) or len(value) != 2:
        raise ValueError("range must be a tuple of (min, max)")
    lo, hi = value
    if lo is None and hi is None:
        return None
    return (None if lo is None else float(lo), None if hi is None else float(hi))


class B200S1S2ClassifierPlugin(Plugin):
    """S1 / S2 / unknown label per detected peak from width / area / height range cuts."""

    provides = "s1_s2"
    depends_on = ["waveform_width", "basic_features"]
    description = "Classify peaks into S1/S2 using width/area/height ranges."
    version = "0.4.0"
    save_when = "always"
    output_dtype = S1_S2_CLASSIFIER_DTYPE
    options = {
        "width_unit": Option(default="ns", type=str, choices=["ns", "samples"], help="unit of the width ranges"),
        "s1_width_range": Option(default=None, type=tuple, help="S1 width range (min, max) in width_unit"),
        "s2_width_range": Option(default=None, type=tuple, help="S2 width range (min, max) in width_unit"),
        "s1_area_range": Option(default=None, type=tuple, help="S1 area range (min, max)"),
        "s2_area_range": Option(default=None, type=tuple, help="S2 area range (min, max)"),
        "s1_height_range": Option(default=None, type=tuple, help="S1 height range (min, max)"),
        "s2_height_range": Option(default=None, type=tuple, help="S2 height range (min, max)"),
        "conflict_policy": Option(default="unknown", type=str, choices=["unknown", "prefer_s1", "prefer_s2"],
                                  help="what to do when both S1 and S2 match"),
        "strict": Option(default=False, type=bool, help="raise when no criteria are configured"),
    }

    def compute(self, context: Any, run_id: str, **_kwargs) -> np.ndarray:
        widths = context.get_data(run_id, "waveform_width")
        features = context.get_data(run_id, "basic_features")
        ranges = {k: _normalize_range(context.get_config(self, k)) for k in
                  ("s1_width_range", "s2_width_range", "s1_area_range", "s2_area_range", "s1_height_range", "s2_height_range")}
        if context.get_config(self, "strict") and all(v is None for v in ranges.values()):
            raise ValueError("No S1/S2 criteria configured; set ranges or disable strict.")
        if not isinstance(widths, np.ndarray):
            raise ValueError("s1_s2 expects waveform_width as a single array")
        if not isinstance(features, np.ndarray):
            raise ValueError("s1_s2 expects basic_features as a single array")
        if len(widths) == 0:
            return np.zeros(0, dtype=S1_S2_CLASSIFIER_DTYPE)
        if widths.dtype != WAVEFORM_WIDTH_DTYPE or features.dtype != BASIC_FEATURES_DTYPE:
            raise ValueError("s1_s2 (B200) expects the packed waveform_width / basic_features dtypes")
        return ops.s1s2_classify(widths, features, width_unit=context.get_config(self, "width_unit"),
                                 conflict_policy=context.get_config(self, "conflict_policy"), **ranges)
