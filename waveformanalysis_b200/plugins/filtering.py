"""wave_pool_filtered on the B200 (reference: core/plugins/builtin/cpu/records.py:334-438,
filtering.py:47-130 for the config validation)."""

from __future__ import annotations

import logging
from typing import Any

import numpy as np

from .. import ops
from ..channel_config import resolve_channel_values, unique_channels
from ..plugin_api import Option, Plugin

logger = logging.getLogger(__name__)
FILTER_ENGINE_VERSION = "3.0.0"
FILTER_OPTION_NAMES = ("filter_type", "lowcut", "highcut", "fs", "filter_order", "sg_window_size", "sg_poly_order")


def resolve_filter_config(values: dict) -> dict:
    """Validate one channel's filter options and design the filter (filtering.py:76-130)."""
    filter_type = str(values["filter_type"])
    if filter_type not in ("BW", "SG"):
        raise ValueError(f"unsupported filter type: {filter_type}. Use 'BW' or 'SG'.")
    if filter_type == "BW":
        lowcut, highcut, fs = float(values["lowcut"]), float(values["highcut"]), float(values["fs"])
        order = int(values["filter_order"])
        if fs <= 0:
            raise ValueError(f"fs ({fs}) must be > 0")
        if order <= 0:
            raise ValueError(f"filter order ({order}) must be > 0")
        if lowcut <= 0 or highcut <= 0:
            raise ValueError("cut-off frequencies must be > 0")
        if lowcut >= highcut:
            raise ValueError(f"lowcut ({lowcut}) must be smaller than highcut ({highcut})")
        if highcut >= fs / 2:
            raise ValueError(f"highcut ({highcut}) must be below the Nyquist frequency ({fs / 2})")
        return {"filter_type": "BW", "sos": ops.butter_bandpass_sos(order, lowcut, highcut, fs)}
    w, p = int(values["sg_window_size"]), int(values["sg_poly_order"])
    if w <= 0:
        raise ValueError(f"SG window size ({w}) must be > 0")
    if p < 0:
        raise ValueError(f"SG polynomial order ({p}) must be >= 0")
    if w % 2 == 0:
        w += 1
        logger.warning("SG window size adjusted to an odd value: %s", w)
    if p >= w:
        raise ValueError(f"SG polynomial order ({p}) must be smaller than the window size ({w})")
    return {"filter_type": "SG", "sg_window_size": w, "sg_poly_order": p}


def channel_filter_configs(channels, filter_options: dict, channel_config: Any, run_id: str | None) -> tuple[dict, dict]:
    """({(board, channel): designed filter} for ``channels``, the designed filter of the options themselves).

    ``filter_options``: values of the options in FILTER_OPTION_NAMES (missing ones take the plugin's defaults),
    overridden per channel by ``channel_config`` for ``run_id``.  Resolution is a function of (run_id, board, channel)
    alone, so processes that hold different channels of one run agree on every channel they share."""
    unknown = sorted(set(filter_options) - set(FILTER_OPTION_NAMES))
    if unknown:
        raise ValueError(f"unknown filter options {unknown}; expected a subset of {FILTER_OPTION_NAMES}")
    base_values = {k: B200WavePoolFilteredPlugin.options[k].default for k in FILTER_OPTION_NAMES}
    base_values.update(filter_options)
    default = resolve_filter_config(base_values)
    return {(b, c): resolve_filter_config(resolve_channel_values(channel_config, run_id, b, c, base_values)) for b, c in channels}, default


class B200WavePoolFilteredPlugin(Plugin):
    """Build a filtered wave_pool aligned to the existing records layout."""

    provides = "wave_pool_filtered"
    depends_on = ["records", "wave_pool"]
    description = "Build filtered wave_pool from records-backed raw waveforms."
    version = FILTER_ENGINE_VERSION
    save_when = "always"
    output_dtype = np.dtype(np.float32)
    options = {
        "filter_type": Option(default="SG", type=str, help="'BW' or 'SG'"),
        "lowcut": Option(default=0.1, type=float, help="BW low cut-off"),
        "highcut": Option(default=0.5, type=float, help="BW high cut-off"),
        "fs": Option(default=0.5, type=float, help="BW sampling rate (GHz)"),
        "filter_order": Option(default=4, type=int, help="BW order"),
        "sg_window_size": Option(default=11, type=int, help="SG window (odd)"),
        "sg_poly_order": Option(default=2, type=int, help="SG polynomial order"),
        "max_workers": Option(default=None, type=int, help="unused on the GPU (kept for config compatibility)"),
        "batch_size": Option(default=0, type=int, help="unused on the GPU (kept for config compatibility)"),
        "channel_config": Option(default=None, type=dict, help="per (board, channel) overrides of the filter options"),
    }

    def compute(self, context: Any, run_id: str, **kwargs) -> np.ndarray:
        records = context.get_data(run_id, "records")
        wave_pool = context.get_data(run_id, "wave_pool")
        if not isinstance(records, np.ndarray):
            raise ValueError("wave_pool_filtered expects records as a structured array")
        if not isinstance(wave_pool, np.ndarray):
            raise ValueError("wave_pool_filtered expects wave_pool as a numpy array")
        if records.dtype.names is None:
            raise ValueError("wave_pool_filtered expects structured records input")
        missing = [f for f in ("wave_offset", "event_length") if f not in records.dtype.names]
        if missing:
            raise ValueError(f"wave_pool_filtered records missing required fields: {missing}")
        if len(records) == 0 or len(wave_pool) == 0:
            return np.zeros(len(wave_pool), dtype=np.float32)
        batch_size = int(context.get_config(self, "batch_size"))
        if batch_size < 0:
            raise ValueError(f"batch_size ({batch_size}) must be >= 0")
        names = records.dtype.names
        boards = records["board"] if "board" in names else np.zeros(len(records), np.int16)
        channels = records["channel"] if "channel" in names else np.zeros(len(records), np.int16)
        base_values = {k: context.get_config(self, k) for k in FILTER_OPTION_NAMES}
        configs, default = channel_filter_configs(unique_channels(boards, channels), base_values, context.get_config(self, "channel_config"),
                                                  run_id)
        off = records["wave_offset"].astype(np.int64)
        ln = records["event_length"].astype(np.int64)
        if np.any((ln > 0) & ((off < 0) | (off + ln > len(wave_pool)))):
            raise ValueError("wave_pool_filtered found out-of-bounds wave slice")
        from .. import residency
        from ..dtypes import RECORDS_DTYPE

        if records.dtype != RECORDS_DTYPE or not residency.fits_device(int(wave_pool.nbytes) * 3):
            return ops.filter_pool(records, wave_pool, configs=configs, default=default)
        # the raw pool is (or becomes) resident; the filtered pool stays in HBM under the host array handed back, so a
        # hit / feature plugin with use_filtered finds it there (the reference shares its bundle: records.py:441-464)
        run = residency.device_run(run_id, records, wave_pool, "wave_pool")
        host, frun = ops.filter_pool(records, wave_pool, configs=configs, default=default, run=run, return_device=True)
        if frun is not None:
            residency.adopt_run(run_id, records, host, "wave_pool_filtered", frun)
        return host
