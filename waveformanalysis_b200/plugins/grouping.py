"""hit_grouped / df_events on the B200 (reference: core/plugins/builtin/cpu/event_analysis.py:23-106,
core/processing/event_grouping.py:99-471).  Sorting, window chaining / anchoring and event ids run
on the device; the pandas packaging of the ragged per-event columns stays on the host."""

from __future__ import annotations

from typing import Any

import numpy as np

from .. import ops
from ..plugin_api import Option, Plugin, check_dt_array, resolve_dt_config

HIT_GROUPED_COLUMNS = ["event_id", "t_min", "t_max", "dt/ns", "n_hits", "dt", "boards", "channels", "heights", "integrals",
                       "timestamps", "record_ids", "sample_starts", "sample_ends"]
DF_EVENTS_COLUMNS = ["event_id", "t_min", "t_max", "dt/ns", "n_hits", "channels", "areas", "heights", "timestamps"]


_MEMBER_ARRAYS: dict = {}


def stash_member_arrays(frame, arrays: dict) -> None:
    """Remember the flat member arrays of a df_events frame for as long as that frame object lives."""
    import weakref

    key = id(frame)
    _MEMBER_ARRAYS[key] = arrays
    weakref.finalize(frame, _MEMBER_ARRAYS.pop, key, None)


def member_arrays_of(frame):
    return _MEMBER_ARRAYS.get(id(frame))


class B200HitGroupedPlugin(Plugin):
    provides = "hit_grouped"
    depends_on = ["hit_merged", "hit_merged_components", "hit_threshold"]
    description = "Group merged hits across channels into event-level coincidence windows."
    version = "0.5.0"
    save_when = "always"
    options = {
        "time_window_ns": Option(default=100.0, type=float),
        "dt": Option(default=None, type=int, help="sample interval (ns), only used when hit_merged has no dt field"),
    }

    def compute(self, context: Any, run_id: str, **kwargs) -> Any:
        import pandas as pd

        hits = context.get_data(run_id, "hit_merged")
        time_window_ns = float(context.get_config(self, "time_window_ns"))
        explicit_dt = resolve_dt_config(context, self, deprecated_keys=("sampling_interval_ns", "dt_ns"))
        if not isinstance(hits, np.ndarray):
            raise ValueError("hits must be a single structured array")
        if len(hits) == 0:
            return pd.DataFrame(columns=HIT_GROUPED_COLUMNS)
        if time_window_ns < 0:
            raise ValueError("time_window_ns must be >= 0")
        names = hits.dtype.names or ()
        required = {"timestamp", "position", "board", "channel", "height", "integral", "record_id"}
        missing = sorted(required - set(names))
        if missing:
            raise KeyError(f"hits missing required fields: {missing}")
        sn, en = ("sample_start", "sample_end") if "sample_start" in names else ("edge_start", "edge_end")
        if sn not in names or en not in names:
            raise KeyError(f"hits missing required fields: {[sn, en]}")
        dt_scalar = check_dt_array(hits, explicit_dt, self.provides, "hit_merged")
        if dt_scalar is not None:
            h = np.zeros(len(hits), dtype=hits.dtype.descr + [("dt", "i4")])
            for n in names:
                h[n] = hits[n]
            h["dt"] = dt_scalar
            hits = h
        comp_rows = comp_hits = None
        if np.any((hits[sn] < 0) | (hits[en] < 0)):  # clusters merged across records: windows from the component hits
            comp_rows = context.get_data(run_id, "hit_merged_components")
            comp_hits = context.get_data(run_id, "hit_threshold")
        ev = ops.group_hit_windows(hits, time_window_ns, comp_rows, comp_hits)
        return hit_grouped_frame(ev, hit_member_columns(hits[ev["members"]]))


class B200GroupedEventsPlugin(Plugin):
    provides = "df_events"
    depends_on = ["df"]
    description = "Group events across channels within a configurable time window."
    save_when = "always"
    options = {"time_window_ns": Option(default=100.0, type=float)}

    def compute(self, context: Any, run_id: str, **kwargs) -> Any:
        import pandas as pd

        df = context.get_data(run_id, "df")
        tw = context.get_config(self, "time_window_ns")
        area_col = "area" if "area" in df.columns else "charge"
        height_col = "height" if "height" in df.columns else "peak"
        if area_col not in df.columns or height_col not in df.columns:
            raise KeyError("df must contain area/height (or charge/peak) columns")
        if len(df) == 0:
            return pd.DataFrame(columns=DF_EVENTS_COLUMNS)
        ts = df["timestamp"].to_numpy()
        ch = df["channel"].to_numpy()
        ev = ops.group_time_window(ts, ch, float(tw))
        m = ev["members"]
        areas, heights = df[area_col].to_numpy(), df[height_col].to_numpy()
        return events_frame(ev, ch[m], areas[m], heights[m], ts[m])


def events_frame(ev: dict, channels, areas, heights, timestamps):
    """The df_events DataFrame of an event table (``event_id``, ``t_min``, ``t_max``, ``dt_ns``, ``n_hits``, CSR
    ``offsets``) and its member columns, already in member order."""
    import pandas as pd

    off = np.asarray(ev["offsets"], dtype=np.int64)
    split = (lambda v: np.split(v, off[1:-1])) if len(off) > 1 else (lambda v: [])
    out = pd.DataFrame({
        "event_id": ev["event_id"], "t_min": ev["t_min"], "t_max": ev["t_max"], "dt/ns": ev["dt_ns"],
        "n_hits": np.asarray(ev["n_hits"]).astype(np.int32),
        "channels": split(channels), "areas": split(areas), "heights": split(heights), "timestamps": split(timestamps),
    })
    # the flat member arrays, for B200PairedEventsPlugin (saves re-flattening the object columns).  Kept beside the
    # frame, not in df.attrs: the Context saves DataFrames with to_parquet, which json-dumps the attrs
    # (core/storage/memmap.py:886)
    stash_member_arrays(out, {"offsets": off, "timestamps": timestamps, "areas": np.asarray(areas).astype(np.float32),
                              "heights": np.asarray(heights).astype(np.float32)})
    return out


def hit_member_columns(rows: np.ndarray) -> dict:
    """The hit_grouped list columns of hit rows (hit_merged with sample_start / sample_end, or edge_start / edge_end)
    already in member order, flat, in the plugin's dtypes."""
    names = rows.dtype.names
    sn, en = ("sample_start", "sample_end") if "sample_start" in names else ("edge_start", "edge_end")
    return {"dt": rows["dt"].astype(np.int32), "boards": rows["board"].astype(np.int16), "channels": rows["channel"].astype(np.int16),
            "heights": rows["height"].astype(np.float32), "integrals": rows["integral"].astype(np.float32),
            "timestamps": rows["timestamp"].astype(np.int64), "record_ids": rows["record_id"].astype(np.int64),
            "sample_starts": rows[sn].astype(np.int32), "sample_ends": rows[en].astype(np.int32)}


def hit_grouped_frame(ev: dict, members: dict):
    """The hit_grouped DataFrame of an event table (``event_id``, ``t_min``, ``t_max``, ``dt_ns``, ``n_hits``, CSR
    ``offsets``) and its flat member columns (``hit_member_columns``), already in member order."""
    import pandas as pd

    off = np.asarray(ev["offsets"], dtype=np.int64)
    split = (lambda v: np.split(v, off[1:-1])) if len(off) > 1 else (lambda v: [])
    cols = {"event_id": ev["event_id"], "t_min": ev["t_min"], "t_max": ev["t_max"], "dt/ns": ev["dt_ns"], "n_hits": ev["n_hits"]}
    cols.update({k: split(v) for k, v in members.items()})
    return pd.DataFrame(cols, columns=HIT_GROUPED_COLUMNS)
