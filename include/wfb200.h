/*
 * wfb200.h - C ABI of libwfb200.so: the B200 (sm_100a) hot path of WaveformAnalysis.
 *
 * Plain C: device/host pointers + sizes + POD parameter blocks, int status codes.
 * No torch / numpy types.  Every entry point cites the reference code it replaces
 * (paths relative to waveform_analysis/ in SnowingWolf/WaveformAnalysis).
 *
 * Conventions
 *   - "_dev" pointers are CUDA device pointers owned by the caller; the library never frees
 *     them.  Scratch comes from a caller-provided workspace (size from *_workspace_bytes).
 *   - `stream` is a cudaStream_t passed as void*; NULL = legacy default stream.  Calls are
 *     asynchronous with respect to the host unless stated otherwise and are re-entrant
 *     (the last error string is thread-local; the only state kept between calls are the
 *     per-device staging buffers of wfb_process_host / wfb_find_peaks, serialised by a mutex
 *     and freed by wfb_release_cache).
 *   - Every entry point that SORTS (wfb_sort_pairs_i64, wfb_build_records*, wfb_group_*,
 *     wfb_hit_merge, wfb_df_columns) synchronises the stream one to four times: the radix
 *     sort reads back which key digits differ (16 bytes) and skips the passes over constant
 *     digits.  They cannot be captured into a CUDA graph.
 *   - Packed row layouts are the reference numpy dtypes byte for byte:
 *       RECORDS_DTYPE         102 B  core/processing/dtypes.py:80-100
 *       BASIC_FEATURES_DTYPE   36 B  core/plugins/builtin/cpu/basic_features.py:29-40
 *       THRESHOLD_HIT_DTYPE    60 B  core/plugins/builtin/cpu/hit_finder.py:33-49
 *       WAVEFORM_WIDTH_DTYPE   56 B  core/plugins/builtin/cpu/waveform_width.py:22-37
 *       WAVEFORM_WIDTH_INTEGRAL_DTYPE 52 B  .../waveform_width_integral.py:25-39
 *   - Return value: 0 = WFB_OK, negative = error (wfb_last_error() has the text).
 */
#ifndef WFB200_H
#define WFB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define WFB_OK 0
#define WFB_ERR_INVALID (-1)  /* bad argument (maps to ValueError in the Python plugins) */
#define WFB_ERR_CUDA (-2)     /* CUDA runtime failure (RuntimeError) */
#define WFB_ERR_LAYOUT (-3)   /* records reference samples outside wave_pool (ValueError) */
#define WFB_ERR_NOMEM (-4)

#define WFB_POL_UNKNOWN 0
#define WFB_POL_POSITIVE 1
#define WFB_POL_NEGATIVE 2
#define WFB_POL_RAW_POSITIVE 3 /* positive pulses, raw float64 arithmetic (st_waveforms branch of
                                   basic_features.py:241-262; records polarity tag "rawpos") */

#define WFB_DO_FEATURES 1
#define WFB_DO_HITS 2

#define WFB_SLICE_END_NONE INT64_MAX /* python slice end=None */

/* Device-side record metadata, 48 bytes, 16-byte aligned: the fields of RECORDS_DTYPE the
 * kernels read (core/processing/dtypes.py:80-100), unpacked once by wfb_records_unpack. */
typedef struct wfb_rec_meta {
    int64_t timestamp;    /* ps */
    double baseline;      /* records["baseline"] */
    int64_t wave_offset;  /* first sample in wave_pool */
    int32_t event_length; /* samples */
    int32_t dt;           /* ns */
    int16_t board;
    int16_t channel;
    uint8_t polarity; /* WFB_POL_* ('positive' / 'negative' / anything else) */
    uint8_t pad_[3];  /* 0, or (edge clamp length + 1) little-endian: see wfb_meta_set_clamp */
    int64_t record_id;
} wfb_rec_meta;

/* Per-(board, channel) overrides resolved on the host from the reference's channel_config
 * (core/hardware/channel.py:412-431): hit_threshold.threshold (hit_finder.py:288-327) and
 * basic_features.fixed_baseline (basic_features.py:134-146). */
typedef struct wfb_chan_rule {
    int32_t board;
    int32_t channel;
    double threshold;
    double fixed_baseline;
    int32_t has_threshold;
    int32_t has_fixed_baseline;
} wfb_chan_rule;

/* Parameters of the fused baseline -> threshold hits -> basic_features pass. */
typedef struct wfb_fh_params {
    int32_t flags;        /* WFB_DO_FEATURES | WFB_DO_HITS */
    int32_t pool_is_f32;  /* 0: uint16 wave_pool, 1: float32 wave_pool_filtered */
    int64_t height_start; /* basic_features.height_range, python slice semantics */
    int64_t height_end;   /* WFB_SLICE_END_NONE for None */
    int64_t area_start;   /* basic_features.area_range */
    int64_t area_end;
    double threshold;        /* hit_threshold.threshold (default 10.0) */
    int32_t left_extension;  /* >= 0 */
    int32_t right_extension; /* >= 0 */
    int32_t lmax; /* padded matrix width = max event_length over ALL records of the run
                     (hit_finder.py:364); 0 = use the maximum over the records passed */
    int32_t n_rules;
    const wfb_chan_rule* rules_dev; /* n_rules entries on the device, may be NULL */
    int64_t pool_base;  /* sample index of pool_dev[0] inside the run's wave_pool */
    int64_t row_base;   /* event_index of the first record passed (basic_features.py:194) */
    int32_t signed_samples; /* 1: the 16-bit samples are int16 (st_waveforms rows), not uint16 */
    int32_t reserved_;
} wfb_fh_params;

const char* wfb_last_error(void);
int wfb_version(void);
/* Number of SMs / device name of the current device (diagnostics). */
int wfb_device_info(int* sm_count, int* cc_major, int* cc_minor, char* name, int name_len);

/* ---- K1: records ---------------------------------------------------------------------- */

/* Host -> device copy of any host array (pageable, read-only or memory-mapped: what the reference's Context hands to
 * plugins, core/context_execution.py:241-251) followed by a stream synchronise, so the source may be released at once.
 * Sources that are not pinned are copied through a ring of pinned 32 MB pieces by a few threads (the driver's own staged
 * copy runs on one); wfb_process_host(_resident) does the same for its chunks.  WFB_STAGED_H2D=0 switches that off. */
int wfb_memcpy_h2d(void* dst_dev, const void* src_host, size_t bytes, void* stream);
/* The same copy without the synchronise, for the streaming backend (core/plugins/core/streaming.py:447-548: chunk k + 1
 * is uploaded while chunk k computes).  The source must stay valid until the stream has passed the copy; a pageable
 * source is read before the call returns, a pinned one by DMA later. */
int wfb_memcpy_h2d_async(void* dst_dev, const void* src_host, size_t bytes, void* stream);
/* HOST helper of the chunk iteration (core/plugins/core/streaming.py:592-664, core/processing/chunk.py:345-385): one
 * threaded pass over n packed RECORDS rows.  ts_out[i] = timestamp, end_ps_out[i] = timestamp + max(event_length, 0) * dt *
 * 1000 (either may be NULL); stats[0..3] = first sample, one past the last sample the rows with event_length > 0 refer to
 * (0, 0 if there is none), the longest event_length, the smallest dt. */
int wfb_records_host_scan(const void* records_host, int64_t n, int64_t* ts_out, int64_t* end_ps_out, int64_t* stats);

/* RECORDS_DTYPE rows (102 B packed, device) -> wfb_rec_meta[n].  Replaces the per-record
 * field access of RecordsView (core/data/records_view.py:16-33). */
int wfb_records_unpack(const void* records_aos_dev, int64_t n, wfb_rec_meta* meta_dev, void* stream);

/* Longest record and the range of dt over the unpacked records, reduced on the device: out_host[0] = max event_length
 * (0 when n == 0), out_host[1] = min dt, out_host[2] = max dt.  Replaces three passes over the 102-byte strided host rows
 * (the dt validation of require_dt_array, _dt_compat.py:51-81, and the padded matrix width of hit_finder.py:364).
 * scratch_dev: 12 bytes.  Synchronises the stream. */
int wfb_meta_stats(const wfb_rec_meta* meta_dev, int64_t n, int32_t* scratch_dev, int32_t* out_host, void* stream);

/* Hit rows of record i have their edges clamped to clamp_len_dev[i] instead of event_length (a negative entry or a NULL
 * array restores event_length).  This is hit_threshold on structured st_waveforms / filtered_waveforms rows whose
 * `event_length` field differs from the row width: every sample of the row is scanned, the edges are clamped to the
 * source's event_length (hit_finder.py:183-230, 388-391).  Lengths up to 2^24 - 2. */
int wfb_meta_set_clamp(wfb_rec_meta* meta_dev, int64_t n, const int32_t* clamp_len_dev, void* stream);

/* ---- per-channel tables -------------------------------------------------------------------------------------------
 * A channel's key is board * 65536 + (channel & 0xFFFF) (the order of channel_config.unique_channels).  Key tables are
 * sorted, without duplicates, and hold at most WFB_MAX_CHANNEL_KEYS entries (they are staged in shared memory). */
#define WFB_MAX_CHANNEL_KEYS 8192

typedef struct wfb_polarity_entry {
    int32_t key;
    uint32_t image[8]; /* the 32 bytes of the RECORDS_DTYPE polarity field (U8, UTF-32) */
} wfb_polarity_entry;

/* records["polarity"] from channel metadata (records.py:40-63 of the reference): every record whose key is in the table
 * gets the entry's image in its packed row (records_aos_dev, may be NULL) and the matching WFB_POL_* code in its
 * wfb_rec_meta, decoded the way wfb_records_unpack decodes rows.  Other records, and the edge clamp in pad_, are left
 * as they are.  One thread per record. */
int wfb_apply_polarity(wfb_rec_meta* meta_dev, void* records_aos_dev, int64_t n, const wfb_polarity_entry* table_dev,
                       int32_t n_table, void* stream);

/* Raw int16 rows -> time-sorted records + wave_pool.  Replaces
 * _build_records_part_from_raw_array + _records_sort_order + _merge_records_part_refs
 * (core/processing/records_builder.py:212-302, 115-120, 341-426).
 *   samples_dev   int16[n * n_samples]  rows in input (per-channel file) order
 *   ts_dev        int64[n] timestamps already in ps; board_dev/channel_dev int16[n]
 *   baseline window [bl_start, bl_end) in samples (VX2730 default 0..40); if
 *   baselines_in_dev != NULL it is used instead (V1725 header baseline, v1725.py:99)
 * Outputs: records_aos_dev (n * 102 B, RECORDS_DTYPE), pool_dev uint16[n * n_samples],
 *          meta_dev (optional, may be NULL), in ascending (timestamp, pid=0, board, channel,
 *          input order); record_id = arange, wave_offset = record_id * n_samples,
 *          time = timestamp / 1000 + epoch_ns. */
int wfb_build_records(const int16_t* samples_dev, const int64_t* ts_dev, const int16_t* board_dev,
                      const int16_t* channel_dev, const double* baselines_in_dev, int64_t n,
                      int32_t n_samples, int32_t bl_start, int32_t bl_end, int32_t dt_ns,
                      int64_t epoch_ns, void* records_aos_dev, uint16_t* pool_dev,
                      wfb_rec_meta* meta_dev, void* workspace_dev, size_t workspace_bytes,
                      void* stream);
size_t wfb_build_records_workspace_bytes(int64_t n);

/* Raw int16 rows -> structured st_waveforms rows (ST_WAVEFORM_DTYPE: 76 header bytes + wave_length int16 samples,
 * core/processing/dtypes.py:36-64) in INPUT order.  Replaces WaveformStruct._structure_waveform
 * (core/plugins/builtin/cpu/waveforms.py:644-799): baseline = mean over the sample window [bl_start, bl_end) clamped to
 * the row (NaN when empty; baselines_in_dev overrides it), baseline_upstream from baseline_upstream_dev (NaN when NULL,
 * :762-771), polarity 'unknown', record_id = record_base + row (:909-911), dt, event_length = min(n_samples,
 * wave_length), samples copied / truncated, the rest of `wave` zero.  ts_dev already in ps. */
int wfb_structure_waveforms(const int16_t* samples_dev, const int64_t* ts_dev, const int16_t* board_dev,
                            const int16_t* channel_dev, const double* baselines_in_dev,
                            const double* baseline_upstream_dev, int64_t n, int32_t n_samples, int32_t wave_length,
                            int32_t bl_start, int32_t bl_end, int32_t dt_ns, int64_t record_base, void* rows_out_dev,
                            void* stream);

/* ---- K2 + K3: fused baseline / threshold hits / basic_features ----------------------------- */

size_t wfb_features_hits_workspace_bytes(int64_t n);

/* One pass over the samples of n records.  Replaces BasicFeaturesPlugin.compute (records
 * branch, basic_features.py:108-195) and ThresholdHitPlugin.compute +
 * _build_hits_from_signal_matrix (hit_finder.py:122-255, 329-413).
 *   pool_dev      uint16 or float32 samples; 16-byte aligned; pool_len samples
 *   feat_out_dev  n * 36 B BASIC_FEATURES rows (if WFB_DO_FEATURES)
 *   hit_out_dev   hit_cap * 60 B THRESHOLD_HIT rows in reference order: record-major, then
 *                 start sample (if WFB_DO_HITS).  Rows beyond hit_cap are counted, not stored.
 *   hit_counts_dev optional int32[n] per-record hit counts (may be NULL)
 *   hit_base_dev  optional const int64*: running hit total of previous calls (row offset of
 *                 this call's first hit); NULL = 0
 *   total_hits_dev int64*: receives hit_base + hits found by this call
 * The caller compares *total_hits_dev with hit_cap after synchronising and re-runs with a
 * larger buffer if it overflowed. */
int wfb_features_hits(const void* pool_dev, int64_t pool_len, const wfb_rec_meta* meta_dev,
                      int64_t n, const wfb_fh_params* params, void* feat_out_dev,
                      void* hit_out_dev, int64_t hit_cap, int32_t* hit_counts_dev,
                      const int64_t* hit_base_dev, int64_t* total_hits_dev, void* workspace_dev,
                      size_t workspace_bytes, void* stream);

/* Error flag of the last wfb_features_hits call that used this workspace: WFB_ERR_LAYOUT if a
 * record pointed outside the pool (RecordsView._validate_wave_bounds,
 * core/data/records_view.py:47-56).  Synchronises the stream. */
int wfb_features_hits_check(void* workspace_dev, void* stream);

/* Host-buffer front end of the same pass: the reference-facing call.  records_host is the
 * RECORDS_DTYPE array and pool_host the wave_pool exactly as Context hands them to a plugin;
 * outputs are host arrays.  Internally a chunked, triple-buffered H2D -> kernels -> D2H
 * pipeline on private streams (synchronous for the caller); hit rows are copied back two chunks
 * behind the compute stream.  wave_offsets must ascend with
 * the record index (always true for pools built by the reference, records_builder.py:300,408).
 * On return *n_hits is the number of hits found; if it exceeds hit_cap only the first hit_cap
 * rows were stored (call again with a larger buffer). */
int wfb_process_host(const void* records_host, int64_t n, const void* pool_host, int64_t pool_len,
                     const wfb_fh_params* params, const wfb_chan_rule* rules_host,
                     void* feat_out_host, void* hit_out_host, int64_t hit_cap,
                     int32_t* hit_counts_host, int64_t* n_hits, int64_t chunk_records);

/* The same pipeline, leaving the run RESIDENT: every chunk of the pool is uploaded into its place in pool_keep_dev (room
 * for pool_len elements, 16-byte aligned, readable up to the next 16-byte boundary) and every chunk's records are unpacked
 * into meta_keep_dev (n rows), so that later passes over the same run (wave_pool_filtered, widths, a second
 * configuration) find it in HBM - the device-side counterpart of the records bundle the reference's plugins share
 * (core/plugins/builtin/cpu/records.py:441-464).  The upload still overlaps the kernels and the copies back. */
int wfb_process_host_resident(const void* records_host, int64_t n, const void* pool_host, int64_t pool_len,
                              const wfb_fh_params* params, const wfb_chan_rule* rules_host, void* feat_out_host,
                              void* hit_out_host, int64_t hit_cap, int32_t* hit_counts_host, int64_t* n_hits,
                              int64_t chunk_records, void* pool_keep_dev, wfb_rec_meta* meta_keep_dev);

/* wfb_process_host keeps its streams, events and device staging buffers between calls (one set per
 * device, calls on one device are serialised).  This frees the device buffers; the reference has
 * no counterpart (its plugins hold no device state), call it when a Context is done with the GPU. */
int wfb_release_cache(void);

/* ---- wave_pool_filtered -------------------------------------------------------------------- */

#define WFB_FILTER_SG 0
#define WFB_FILTER_BW 1
#define WFB_MAX_SG_WINDOW 129
#define WFB_MAX_SOS_SECTIONS 16

/* One filter configuration (host side builds one per distinct resolved configuration;
 * filtering.py:47-130).  SG: taps = savgol coefficients (window), edge = (halflen x window)
 * projection rows for the first half-window (the last half-window uses the mirrored rows).
 * BW: sos[n_sections][6] and zi[n_sections][2] (sosfilt_zi). */
typedef struct wfb_filter_cfg {
    int32_t type;       /* WFB_FILTER_SG / WFB_FILTER_BW */
    int32_t sg_window;  /* requested window (odd); the kernel applies min(window, L) forced odd */
    int32_t sg_poly;
    int32_t n_sections;
    double sos[WFB_MAX_SOS_SECTIONS][6];
    double zi[WFB_MAX_SOS_SECTIONS][2];
} wfb_filter_cfg;

/* uint16 (or float32) pool -> float32 filtered pool aligned with the same wave_offsets.
 * Replaces WavePoolFilteredPlugin.compute -> filter_wave_pool_batch -> _apply_filter_core
 * (records.py:368-438, filtering.py:206-241, 377-407).
 *   cfg_index_dev  int32[n]: index into cfgs for each record; cfgs_dev: wfb_filter_cfg[n_cfg]
 *   sg_tables_dev  double tables built by the host for every distinct effective SG window,
 *                  see waveformanalysis_b200/filters.py (layout: per table [window taps |
 *                  halflen*window edge rows]); sg_table_offset_dev int32[n]: offset of the
 *                  record's table (or -1 = identity) */
int wfb_filter_pool(const void* pool_dev, int32_t pool_is_f32, int64_t pool_len,
                    const wfb_rec_meta* meta_dev, int64_t n, const wfb_filter_cfg* cfgs_dev,
                    int32_t n_cfg, const int32_t* cfg_index_dev, const double* sg_tables_dev,
                    const int32_t* sg_table_offset_dev, float* out_dev, int64_t pool_base,
                    void* workspace_dev, size_t workspace_bytes, int32_t lmax, void* stream);
/* Scratch for the Butterworth forward pass (float64, one row of lmax + 2*padlen per resident
 * thread); SG-only runs may pass a NULL workspace. */
size_t wfb_filter_workspace_bytes(int64_t n, int32_t lmax);

/* The per-record arguments of wfb_filter_pool, one thread per record: cfg_index_out[i] = cfg_of_key_dev[j] for the
 * entry j of keys_dev that holds record i's channel key, default_cfg when there is none.  For an SG configuration c
 * (sg_lut_off_of_cfg_dev[c] >= 0), sg_table_offset_out[i] = sg_lut_dev[sg_lut_off_of_cfg_dev[c] + min(max(L, 0),
 * sg_wcap_of_cfg_dev[c])] with L the record's event_length: the host lists the table offset of each effective window
 * min(window, L) (forced odd, -1 = identity when <= poly) for L = 0 .. wcap.  Otherwise -1. */
int wfb_filter_plan(const wfb_rec_meta* meta_dev, int64_t n, const int32_t* keys_dev, const int32_t* cfg_of_key_dev, int32_t n_keys,
                    int32_t default_cfg, const int32_t* sg_lut_dev, const int32_t* sg_lut_off_of_cfg_dev, const int32_t* sg_wcap_of_cfg_dev,
                    int32_t* cfg_index_out, int32_t* sg_table_offset_out, void* stream);

/* ---- waveform_width / waveform_width_integral --------------------------------------------- */

typedef struct wfb_width_params {
    double rise_low, rise_high, fall_high, fall_low;
    double sampling_rate; /* GHz */
    int32_t interpolation;
    int32_t wave_is_f32; /* 0: int16 samples (st_waveforms), 1: float32 (filtered_waveforms) */
} wfb_width_params;

/* Per hit: 10/90 (configurable) rise / fall / total widths with linear interpolation.
 * Replaces WaveformWidthPlugin._calculate_width_from_peak + _find_threshold_crossing
 * (waveform_width.py:205-374).  hit_row_dev[i] = row index of the waveform of hit i (or -1:
 * no matching record -> row dropped); waves are rows of `stride` samples (first `length`
 * valid).  valid_dev[i] = 1 if a row was produced (pv > 0 and position < length).
 * out_dev: n_hits * 56 B WAVEFORM_WIDTH rows (only rows with valid=1 are written). */
int wfb_waveform_width(const void* waves_dev, int64_t n_waves, int32_t length, int64_t stride,
                       const int64_t* hit_row_dev, const int64_t* hit_position_dev,
                       const int64_t* hit_timestamp_dev, const int16_t* hit_board_dev,
                       const int16_t* hit_channel_dev, const int64_t* hit_record_id_dev,
                       int64_t n_hits, const wfb_width_params* params, void* out_dev,
                       uint8_t* valid_dev, void* stream);

/* The same widths for hit rows that live on the device, against a device-resident run (records + pool, e.g. a time
 * shard).  hits_dev: n_hits packed HIT_DTYPE rows (48 B).  A hit's waveform is run row record_id - row_base, used only
 * when it lies in [0, n) and meta_dev[row].record_id == record_id (otherwise the hit gives no row, like a hit without a
 * matching waveform row in wfb_waveform_width); its samples are the record's own event_length samples at
 * pool_dev[wave_offset - pool_base].  A record whose samples lie outside [0, pool_len) gives no row either.
 * pool_is_f32: 0 = 16-bit samples read as int16 (what st_waveforms rows of the same samples hold), 1 = float32;
 * params->wave_is_f32 is not read.  out_dev receives the WAVEFORM_WIDTH rows (56 B, room for n_hits) compacted in hit
 * order, *n_out_dev (device int64) their number.  Asynchronous: nothing is read back. */
size_t wfb_waveform_width_run_workspace_bytes(int64_t n_hits);
int wfb_waveform_width_run(const void* pool_dev, int32_t pool_is_f32, int64_t pool_len, const wfb_rec_meta* meta_dev,
                           int64_t n, int64_t pool_base, int64_t row_base, const void* hits_dev, int64_t n_hits,
                           const wfb_width_params* params, void* out_dev, int64_t* n_out_dev, void* workspace_dev,
                           size_t workspace_bytes, void* stream);

/* Per record cumulative-charge quantile indices.  Replaces
 * WaveformWidthIntegralPlugin.compute records branch (waveform_width_integral.py:166-231).
 * pool_is_f32: 0 uint16 pool, 1 float32 pool, 2 int16 samples (structured st_waveforms rows used in place).
 * out_dev: n * 52 B WAVEFORM_WIDTH_INTEGRAL rows. */
int wfb_width_integral(const void* pool_dev, int32_t pool_is_f32, int64_t pool_len,
                       const wfb_rec_meta* meta_dev, int64_t n, double q_low, double q_high,
                       double dt_ns, int64_t pool_base, int64_t row_base, void* out_dev,
                       void* stream);

/* ---- K4: event grouping ------------------------------------------------------------------- */

size_t wfb_group_workspace_bytes(int64_t n_hits);

/* Chain clustering of absolute hit windows.  Replaces the sort + sequential chain of
 * group_hit_windows (core/processing/event_grouping.py:365-367, 418, 453-470).
 * Inputs are SoA columns of hit_merged (device).  Outputs (device, n_hits each):
 *   order_dev     int64: permutation lexsort((record_id, timestamp, dt, abs_start))
 *   event_id_dev  int64: event id of hit i (in input order)
 *   abs_start_dev / abs_end_dev  double: absolute windows in ps
 * *n_events_dev receives the number of events. */
int wfb_group_hit_windows(const int64_t* timestamp_dev, const int64_t* position_dev,
                          const int32_t* start_dev, const int32_t* end_dev, const int32_t* dt_dev,
                          const int64_t* record_id_dev, int64_t n_hits, double time_window_ns,
                          int64_t* order_dev, int64_t* event_id_dev, double* abs_start_dev,
                          double* abs_end_dev, int64_t* n_events_dev, void* workspace_dev,
                          size_t workspace_bytes, void* stream);

/* The same grouping for caller-provided absolute windows: hit_merged rows merged across records have no sample
 * window (sample_start / sample_end = -1) and take min / max of their component hits' windows
 * (event_grouping.py:369-414) - computed by the caller, then grouped here. */
int wfb_group_abs_windows(const int64_t* timestamp_dev, const double* abs_start_dev, const double* abs_end_dev,
                          const int32_t* dt_dev, const int64_t* record_id_dev, int64_t n, double time_window_ns,
                          int64_t* order_dev, int64_t* event_id_dev, int64_t* n_events_dev, void* workspace_dev,
                          size_t workspace_bytes, void* stream);

/* Grouping columns straight from packed hit rows on the device (row_bytes 60: THRESHOLD_HIT, 72: HIT_MERGED; the first
 * 60 bytes are laid out alike): timestamp, dt, record_id and - unless abs_start_dev is NULL - the absolute windows
 * timestamp + (edge - position) * dt * 1e3 (event_grouping.py:365-367).  Keeps the time-sharded multi-GPU grouping on the
 * device (no host round trip of the hit rows). */
int wfb_hit_columns(const void* rows_dev, int64_t n, int32_t row_bytes, int64_t* timestamp_dev, int32_t* dt_dev,
                    int64_t* record_id_dev, double* abs_start_dev, double* abs_end_dev, void* stream);

/* Absolute window of every HIT_MERGED row as min / max over the windows of its component hits (event_grouping.py:369-414;
 * rows merged across records carry no sample window of their own).  hits_dev / order_dev / merged_dev as passed to and
 * filled by wfb_hit_merge. */
int wfb_merged_abs_windows(const void* hits_dev, const int64_t* order_dev, const void* merged_dev, int64_t n_clusters,
                           double* abs_start_dev, double* abs_end_dev, void* stream);

/* Anchored fixed-window clustering of time-sorted timestamps.  Replaces
 * _find_cluster_boundaries_numba (event_grouping.py:477-510): cluster k starts at the first
 * timestamp > ts[anchor_k-1] + window.  ts_sorted_dev int64[n] ascending.
 * event_id_dev int64[n]; *n_events_dev. */
int wfb_group_time_window(const int64_t* ts_sorted_dev, int64_t n, double time_window_ns,
                          int64_t* event_id_dev, int64_t* n_events_dev, void* workspace_dev,
                          size_t workspace_bytes, void* stream);

/* The event table of wfb_group_time_window's events (event_grouping.py:99-283, the df_events columns).
 * ts_sorted_dev int64[n] ascending and event_id_dev int64[n] as wfb_group_time_window wrote them (events are
 * contiguous runs numbered 0 .. n_events - 1); channel_dev int16, area_dev / height_dev float32 (both optional) are
 * indexed by INPUT row; order_dev int64[n] maps sorted position -> input row (NULL: the rows are already sorted).
 * Writes offsets_dev[n_events + 1] (CSR), members_dev[n] (input rows, stably ordered by channel inside every event:
 * np.lexsort((arange, channel, event))), t_min / t_max (timestamps of the first / last member in that order),
 * dt_ns = (double)(t_max - t_min) / 1e3, n_hits, and the member-ordered timestamp / channel / area / height columns
 * (member_area_dev / member_height_dev NULL exactly when their inputs are).  Events of up to 32 members are ranked by
 * one warp each; larger ones by one stable radix sort of their rows.  Synchronises the stream once. */
size_t wfb_event_table_workspace_bytes(int64_t n);
int wfb_event_table(const int64_t* ts_sorted_dev, const int64_t* event_id_dev, int64_t n, int64_t n_events,
                    const int16_t* channel_dev, const int64_t* order_dev, const float* area_dev, const float* height_dev,
                    int64_t* offsets_dev, int64_t* members_dev, int64_t* t_min_dev, int64_t* t_max_dev, double* dt_ns_dev,
                    int64_t* n_hits_dev, int64_t* member_ts_dev, int16_t* member_channel_dev, float* member_area_dev,
                    float* member_height_dev, void* workspace_dev, size_t workspace_bytes, void* stream);

/* The event table of chain-clustered hit windows (event_grouping.py:418-471, the hit_grouped columns).
 * order_dev / event_id_dev int64[n] as wfb_group_hit_windows / wfb_group_abs_windows wrote them (order sorted by
 * (abs_start, dt, timestamp, record_id, input row); every event a contiguous run of it, numbered 0 .. n_events - 1);
 * board_dev / channel_dev int16, dt_dev int32 and abs_start_dev / abs_end_dev float64 are indexed by INPUT row
 * (timestamp and record_id enter through order).  Writes offsets_dev[n_events + 1] (CSR), members_dev[n] (input rows
 * in the order np.lexsort((record_id, timestamp, abs_start, dt, channel, board, event)), ties in input row order),
 * t_min = (int64) min abs_start and t_max = (int64) max abs_end of every event (truncated toward zero),
 * dt_ns = (double)(t_max - t_min) / 1e3 and n_hits.  rows_dev (optional, packed THRESHOLD_HIT or HIT_MERGED rows of
 * row_bytes = 60 or 72, 4-byte aligned) is gathered into member_rows_dev in member order.  Events of up to 32 members
 * are ranked by one warp each; larger ones by two stable radix sorts of their positions, by (board, channel, dt) and
 * then by event.  Synchronises the stream once. */
size_t wfb_hit_event_table_workspace_bytes(int64_t n);
int wfb_hit_event_table(const int64_t* order_dev, const int64_t* event_id_dev, int64_t n, int64_t n_events,
                        const int16_t* board_dev, const int16_t* channel_dev, const int32_t* dt_dev,
                        const double* abs_start_dev, const double* abs_end_dev, const void* rows_dev, int32_t row_bytes,
                        int64_t* offsets_dev, int64_t* members_dev, int64_t* t_min_dev, int64_t* t_max_dev,
                        double* dt_ns_dev, int64_t* n_hits_dev, void* member_rows_dev, void* workspace_dev,
                        size_t workspace_bytes, void* stream);

/* K1 for records of different lengths (channels / parts with different waveform widths,
 * records_builder.py:212-302 per part + :870-945 merge): like wfb_build_records, but every record names its
 * own int16 samples (byte offset into samples_dev + count) and the wave_pool is ragged (wave_offset = running
 * sum of the lengths in output order).  baselines_in_dev == NULL: mean of samples [bl_start, min(bl_end, len)). */
int wfb_build_records_ragged(const void* samples_dev, int64_t samples_bytes, const int64_t* sample_offset_dev,
                             const int32_t* n_samples_dev, const int64_t* timestamp_ps_dev, const int16_t* board_dev,
                             const int16_t* channel_dev, const double* baselines_in_dev, int64_t n, int32_t dt_ns,
                             int32_t bl_start, int32_t bl_end, int64_t epoch_ns, void* records_aos_dev, uint16_t* pool_dev,
                             int64_t pool_len, wfb_rec_meta* meta_dev, void* workspace_dev, size_t workspace_bytes, void* stream);
/* The same for a part of a run read from a subset of its row groups (distributed.build_records_sharded): seq_dev[i]
 * is the global index of row i (its index in the concatenation of ALL groups of the run, in group order) and
 * becomes the row's record_id; the local rows must follow the groups in group order.  Rows come out ordered by
 * (timestamp, board, channel, seq).  The workspace is wfb_build_records_v1725_workspace_bytes(n). */
int wfb_build_records_ragged_seq(const void* samples_dev, int64_t samples_bytes, const int64_t* sample_offset_dev,
                                 const int32_t* n_samples_dev, const int64_t* timestamp_ps_dev, const int16_t* board_dev,
                                 const int16_t* channel_dev, const double* baselines_in_dev, const int64_t* seq_dev, int64_t n,
                                 int32_t dt_ns, int32_t bl_start, int32_t bl_end, int64_t epoch_ns, void* records_aos_dev,
                                 uint16_t* pool_dev, int64_t pool_len, wfb_rec_meta* meta_dev, void* workspace_dev,
                                 size_t workspace_bytes, void* stream);

/* `hit` = scipy.signal.find_peaks per record (core/plugins/builtin/cpu/peak_finding.py:213-565
 * HitFinderPlugin._compute_peaks / _find_peaks_in_waveform / _calculate_peak_height).
 * wave_kind selects what the plugin calls `waveform` and the detection signal:
 *   WFB_WAVE_AOS_I16 / WFB_WAVE_AOS_F32: rows of st_waveforms / filtered_waveforms (meta.wave_offset in
 *     elements of that type); detection = -diff(wave) in the wave's own dtype, or baseline - wave;
 *   WFB_WAVE_REC_U16 / WFB_WAVE_REC_F32: records + wave_pool(_filtered); waveform = -RecordsView.signals()
 *     (float32 baseline subtraction, polarity-normalised) in float64; detection = +diff or the signal.
 * Conditions are lower bounds as the plugin passes them; distance <= 2 is a no-op (local maxima are at
 * least two samples apart).  Rows are packed HIT_DTYPE (48 B) in record order; peaks beyond row_cap are
 * counted in *total_out_dev but not stored.  Synchronises the stream (error flag read-back). */
#define WFB_WAVE_AOS_I16 0
#define WFB_WAVE_AOS_F32 1
#define WFB_WAVE_REC_U16 2
#define WFB_WAVE_REC_F32 3
#define WFB_WAVE_AOS_F32_AS_F64 4 /* float32 rows promoted to float64 first (signal_peaks_stream, signal_peaks.py:256-262) */
#define WFB_WAVE_AOS_U16 5        /* uint16 rows: np.diff and the negation wrap modulo 65536 (peak_finding.py:488-495) */
typedef struct wfb_peak_params {
    int32_t wave_kind;      /* WFB_WAVE_* */
    int32_t use_derivative; /* detect on the first difference (default) or on the level */
    double height;          /* find_peaks(height=) */
    double prominence;      /* find_peaks(prominence=) */
    double width;           /* find_peaks(width=), rel_height 0.5 */
    double threshold;       /* find_peaks(threshold=) when has_threshold */
    int32_t has_threshold;
    int32_t distance;       /* find_peaks(distance=) */
    int32_t height_method;  /* 0 "minmax", 1 "diff" (hit), 2 "diff" by float64 cumsum (signal_peaks_stream) */
    int32_t height_window_extension;
    int32_t lmax;           /* longest record (samples) */
    int32_t level_f32;      /* WFB_WAVE_AOS_F32 without derivative: baseline - wave in float32 (the baseline is np.mean of the float32 row) */
    int64_t pool_base;      /* records sources: record samples start at waves_dev[wave_offset - pool_base] (a time shard holds only its
                               own pool slice); the AoS sources require 0 */
} wfb_peak_params;
size_t wfb_find_peaks_workspace_bytes(int64_t n);
int wfb_find_peaks(const void* waves_dev, int64_t waves_len, const wfb_rec_meta* meta_dev, int64_t n,
                   const wfb_peak_params* params, void* rows_out_dev, int64_t row_cap, int32_t* counts_out_dev,
                   int64_t* total_out_dev, void* workspace_dev, size_t workspace_bytes, void* stream);

/* CAEN V1725 DAW_DEMO binary ingest (utils/formats/v1725.py:69-114, the per-waveform Python loop of
 * V1725Reader.iter_waves; core/processing/records_builder.py:164-209, 798-830).
 * wfb_v1725_scan_host walks the header chain of one .bin stream in HOST memory and fills one index entry
 * per waveform (payload byte offset, samples, channel, 48-bit sample-index timestamp, 16-bit baseline,
 * trunc flag); parsing stops at the first short read like the reference's reader.  capacity == 0 only
 * counts.  wfb_build_records_v1725 takes the stream bytes of all files (concatenated, offsets rebased, on
 * the device) plus the index columns and writes RECORDS_DTYPE rows, wave_pool and wfb_rec_meta in the
 * reference's order: timestamp_ps = timestamp * dt_ns * 1000, lexsort((seq, channel, board, pid,
 * timestamp)), ragged wave_offsets, baseline = header field, flags = trunc, time = timestamp_ps // 1000. */
int wfb_v1725_scan_host(const uint8_t* blob_host, int64_t n_bytes, int64_t capacity, int64_t* payload_offset,
                        int32_t* n_samples, int16_t* channel, int64_t* timestamp, uint16_t* baseline, uint8_t* trunc,
                        int64_t* n_records, int64_t* n_samples_total);
size_t wfb_build_records_v1725_workspace_bytes(int64_t n);
int wfb_build_records_v1725(const uint8_t* blob_dev, int64_t blob_bytes, const int64_t* payload_offset_dev,
                            const int32_t* n_samples_dev, const int64_t* timestamp_dev, const int16_t* board_dev,
                            const int16_t* channel_dev, const uint16_t* baseline_dev, const uint8_t* trunc_dev, int64_t n,
                            int32_t dt_ns, void* records_aos_dev, uint16_t* pool_dev, int64_t pool_len,
                            wfb_rec_meta* meta_dev, void* workspace_dev, size_t workspace_bytes, void* stream);
/* The same for a part of a run read from a subset of its files: seq_dev[i] is the global index of waveform i
 * (its index in the concatenation of ALL files of the run, in list order) and becomes the row's record_id;
 * the local index columns must follow the files in list order.  The workspace is
 * wfb_build_records_v1725_workspace_bytes(n). */
int wfb_build_records_v1725_seq(const uint8_t* blob_dev, int64_t blob_bytes, const int64_t* payload_offset_dev,
                                const int32_t* n_samples_dev, const int64_t* timestamp_dev, const int16_t* board_dev,
                                const int16_t* channel_dev, const uint16_t* baseline_dev, const uint8_t* trunc_dev,
                                const int64_t* seq_dev, int64_t n, int32_t dt_ns, void* records_aos_dev, uint16_t* pool_dev,
                                int64_t pool_len, wfb_rec_meta* meta_dev, void* workspace_dev, size_t workspace_bytes, void* stream);

/* Time shards of a run built on several GPUs (distributed.build_records_sharded_v1725).  Rows are ordered by
 * the key (timestamp, board, channel, record_id), record_id holding the global seq.
 * wfb_record_split_points: for each of n_keys keys (int64 timestamp, board, channel, record_id, 4 per key)
 * the number of the n sorted RECORDS rows whose key is smaller (lower bound).
 * wfb_merge_record_runs: rows_in holds n_runs strictly increasing runs, run r at rows
 * [run_offsets_host[r], run_offsets_host[r + 1]), and pool_in their samples in the same order (no gaps).
 * Writes the merged rows with record_id = record_base + i and wave_offset = pool_base + the running sum of
 * event_length, all other fields unchanged, the samples in output order (pool_len = the total) and
 * wfb_rec_meta rows.  A run that is not strictly increasing: WFB_ERR_INVALID, nothing written.
 * Synchronizes the stream once (after that check). */
int wfb_record_split_points(const void* rows_dev, int64_t n, const int64_t* keys_dev, int64_t n_keys, int64_t* out_dev,
                            void* stream);
size_t wfb_merge_record_runs_workspace_bytes(int64_t n, int64_t n_runs);
int wfb_merge_record_runs(const void* rows_in_dev, const uint16_t* pool_in_dev, int64_t n_in, const int64_t* run_offsets_host,
                          int64_t n_runs, int64_t record_base, int64_t pool_base, void* rows_out_dev, uint16_t* pool_out_dev,
                          int64_t pool_len, wfb_rec_meta* meta_out_dev, void* workspace_dev, size_t workspace_bytes, void* stream);

/* hit_merge (core/plugins/builtin/cpu/hit_merge.py:115-181 cluster chain, :256-322 merged rows) on
 * packed THRESHOLD_HIT rows: per hardware channel, hits ordered by absolute window start are chained
 * while merge_gap_ns > 0, dt matches, gap <= merge_gap_ns and total width <= max_total_width_ns.
 * Outputs, all in cluster order: order_dev[k] = index of the k-th hit (hit_merge_clusters.hit_index),
 * cluster_index_dev[k] (hit_merge_clusters.cluster_index), merged_dev = *n_clusters_dev packed
 * HIT_MERGED rows (72 B; room for n rows). */
size_t wfb_hit_merge_workspace_bytes(int64_t n);
int wfb_hit_merge(const void* hits_dev, int64_t n, double merge_gap_ns, double max_total_width_ns, int64_t* order_dev,
                  int64_t* cluster_index_dev, void* merged_dev, int64_t* n_clusters_dev, void* workspace_dev,
                  size_t workspace_bytes, void* stream);

/* Stable LSD radix sort of int64 keys carrying int64 values (device, n each); used by the
 * plugins for the time sort (records_builder.py:115-120, event_grouping.py:142). */
int wfb_sort_pairs_i64(const int64_t* keys_in_dev, const int64_t* vals_in_dev, int64_t* keys_out_dev,
                       int64_t* vals_out_dev, int64_t n, void* workspace_dev,
                       size_t workspace_bytes, void* stream);
size_t wfb_sort_workspace_bytes(int64_t n);

/* ---- the step after the path: df, s1_s2, df_paired ------------------------------------------ */

/* `df` (core/plugins/builtin/cpu/dataframe.py:192-311): the columns of the events DataFrame in
 * timestamp order.  feat_rows_dev = n packed BASIC_FEATURES rows (36 B); record_id_dev = int64[n]
 * or NULL (then record_id = row index, dataframe.py:222-226).  order_dev[k] = input row of the k-th
 * output row (a STABLE sort by timestamp; it is the index of df.sort_values("timestamp")).
 * gains_host: n_gains (board, channel, gain_adc_per_pe) entries with gain > 0; with_pe != 0 also fills
 * area_pe / height_pe = float64(value) / gain, NaN for channels without an entry (dataframe.py:296-309);
 * with_pe == 0: both may be NULL. */
typedef struct wfb_gain_rule {
    int32_t board, channel;
    double gain;
} wfb_gain_rule;
size_t wfb_df_columns_workspace_bytes(int64_t n);
int wfb_df_columns(const void* feat_rows_dev, const int64_t* record_id_dev, int64_t n, const wfb_gain_rule* gains_host,
                   int32_t n_gains, int32_t with_pe, int64_t* order_dev, int64_t* timestamp_dev, int64_t* record_id_out_dev,
                   float* area_dev, float* height_dev, float* amp_dev, float* max_abs_diff_dev, int16_t* board_dev,
                   int16_t* channel_dev, double* area_pe_dev, double* height_pe_dev, void* workspace_dev,
                   size_t workspace_bytes, void* stream);

/* `s1_s2` (core/plugins/builtin/cpu/s1_s2_classifier.py:133-228): one packed S1_S2_CLASSIFIER row (45 B)
 * per waveform_width row (56 B).  height / area come from feat_rows_dev[record_id - feat_row_base] (36-B rows) when
 * 0 <= record_id - feat_row_base < n_feat, else NaN (:170-180).  A range with present == 0 always passes; a NaN value fails
 * a present range (:54-68).  width_in_samples selects total_width_samples instead of total_width (:182).
 * conflict_policy: 0 unknown, 1 prefer_s1, 2 prefer_s2 (:194-204). */
typedef struct wfb_range {
    double lo, hi;
    int32_t has_lo, has_hi;
    int32_t present;
    int32_t reserved_;
} wfb_range;
typedef struct wfb_s1s2_params {
    wfb_range s1_width, s1_area, s1_height;
    wfb_range s2_width, s2_area, s2_height;
    int32_t width_in_samples;
    int32_t conflict_policy;
    int64_t feat_row_base;  /* record_id of feat_rows_dev[0]: a time shard's feature rows start at its first record */
} wfb_s1s2_params;
int wfb_s1s2_classify(const void* width_rows_dev, int64_t n_peaks, const void* feat_rows_dev, int64_t n_feat,
                      const wfb_s1s2_params* params, void* out_rows_dev, void* stream);

/* `df_paired` (core/processing/analyzer.py:66-110) on the grouped events in CSR form (event e owns members
 * [offsets[e], offsets[e+1]) of the member arrays, in df_events order): keep_dev[e] = dt_ns[e] <= time_window_ns,
 * delta_t_dev[e] = (last - first member timestamp) / 1000.0, area_ch_dev / height_ch_dev [e * n_channels + i] =
 * the i-th member's value or NaN when the event has fewer members (:98-108). */
int wfb_pair_events(const int64_t* offsets_dev, int64_t n_events, const int64_t* member_ts_dev,
                    const float* member_area_dev, const float* member_height_dev, const double* dt_ns_dev,
                    double time_window_ns, int32_t n_channels, uint8_t* keep_dev, double* delta_t_dev,
                    float* area_ch_dev, float* height_ch_dev, void* stream);

/* ---- synthetic input (bench / tests) ------------------------------------------------------- */

/* Fill pool_dev / meta_dev with a seeded synthetic run of n fixed-length records
 * (SURVEY.md 8(d): baseline 8000+10*channel, N(0,3) noise, 1-3 negative pulses), time-sorted. */
int wfb_synth_fill(uint16_t* pool_dev, wfb_rec_meta* meta_dev, void* records_aos_dev, int64_t n,
                   int32_t n_samples, int32_t n_channels, int32_t dt_ns, uint64_t seed,
                   int64_t record_base, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* WFB200_H */
