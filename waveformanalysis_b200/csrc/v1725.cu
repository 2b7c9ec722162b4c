// CAEN V1725 DAW_DEMO binary ingest: header-chain index on the host, records + wave_pool on the device.
//
// Reference: utils/formats/v1725.py:69-114 (V1725Reader.iter_waves: one Python object per waveform),
// core/processing/records_builder.py:164-209 (_build_records_from_wave_list), :798-830
// (build_records_from_v1725_files), :115-120 (_records_sort_order), formats/base.py:184-186
// (sample-index timestamps -> ps).
//
// The stream is a chain (every header gives the position of the next), so the index - 34 bytes per
// waveform - is built by one sequential pass over the headers on the host while the payload never
// leaves its buffer; everything proportional to the samples runs on the device: time sort of all
// files' waveforms, ragged wave_offsets by a scan, one warp per output record copying its samples
// straight out of the stream bytes.
#include <algorithm>

#include "common.cuh"
#include "sort_scan.cuh"

namespace wfb {

static size_t v_al256(size_t x) { return (x + 255) & ~(size_t)255; }

__global__ void v1725_keys_kernel(const short* __restrict__ board, const short* __restrict__ channel, long long n,
                                  unsigned long long* __restrict__ key, long long* __restrict__ val) {
    long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= n) return;
    key[i] = ((unsigned long long)(unsigned)((int)board[i] + 32768) << 16) | (unsigned long long)(unsigned)((int)channel[i] + 32768);
    val[i] = i;
}
__global__ void v1725_gather_ts_kernel(const long long* __restrict__ raw_ts, const long long* __restrict__ idx, long long n,
                                       long long dt_ps, unsigned long long* __restrict__ out) {
    long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i < n) out[i] = (unsigned long long)(raw_ts[idx[i]] * dt_ps);
}
__global__ void v1725_lengths_kernel(const int* __restrict__ n_samples, const long long* __restrict__ order, long long n,
                                     long long* __restrict__ len_sorted) {
    long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i < n) len_sorted[i] = n_samples[order[i]];
}

// halfword k (0..50) of the packed RECORDS_DTYPE row (core/processing/dtypes.py:80-100)
__device__ __forceinline__ uint16_t v1725_row_halfword(int k, long long ts, int board, int channel, double baseline, long long rid,
                                                       int dt, unsigned flags, long long wave_offset, int len, long long time_ns) {
    auto h64 = [](unsigned long long v, int q) { return (uint16_t)(v >> (16 * q)); };
    if (k < 4) return h64((unsigned long long)ts, k);
    if (k < 6) return 0;  // pid
    if (k == 6) return (uint16_t)board;
    if (k == 7) return (uint16_t)channel;
    if (k < 12) return h64((unsigned long long)__double_as_longlong(baseline), k - 8);
    if (k < 16) return h64(0x7ff8000000000000ull, k - 12);  // baseline_upstream = NaN
    if (k < 32) {
        const char* s = "unknown";
        int ci = (k - 16) >> 1;
        return ((k & 1) == 0 && ci < 7) ? (uint16_t)s[ci] : (uint16_t)0;
    }
    if (k < 36) return h64((unsigned long long)rid, k - 32);
    if (k < 38) return (uint16_t)((unsigned)dt >> (16 * (k - 36)));
    if (k == 38) return 0;  // trigger_type
    if (k < 41) return (uint16_t)(flags >> (16 * (k - 39)));
    if (k < 45) return h64((unsigned long long)wave_offset, k - 41);
    if (k < 47) return (uint16_t)((unsigned)len >> (16 * (k - 45)));
    return h64((unsigned long long)time_ns, k - 47);
}

// one warp per OUTPUT record: copy the payload (int16 reinterpreted as uint16), pack the row
__global__ void __launch_bounds__(256) v1725_gather_kernel(const uint8_t* __restrict__ blob, const long long* __restrict__ payload_off,
                                                          const int* __restrict__ n_samples, const long long* __restrict__ raw_ts,
                                                          const short* __restrict__ board, const short* __restrict__ channel,
                                                          const unsigned short* __restrict__ baseline,
                                                          const double* __restrict__ baseline_f64,
                                                          const unsigned char* __restrict__ trunc,
                                                          const long long* __restrict__ order, const long long* __restrict__ len_incl,
                                                          const long long* __restrict__ seq, long long n, int dt_ns, long long ts_scale, int bl_start, int bl_end,
                                                          long long epoch_ns, long long blob_bytes, long long pool_len,
                                                          uint16_t* __restrict__ rows, uint16_t* __restrict__ pool,
                                                          wfb_rec_meta* __restrict__ meta) {
    const int lane = lane_id();
    const long long r = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
    if (r >= n) return;
    const long long src = order[r];
    const int len = n_samples[src];
    const long long wave_offset = len_incl[r] - len;
    const long long rid = seq != nullptr ? seq[src] : r;
    // payloads start on 4-byte boundaries of the stream; the destination only on 2-byte ones
    const uint16_t* in = reinterpret_cast<const uint16_t*>(blob + payload_off[src]);
    uint16_t* out = pool + wave_offset;
    const bool ok = len >= 0 && payload_off[src] >= 0 && payload_off[src] + 2ll * len <= blob_bytes && wave_offset + len <= pool_len;
    long long bsum = 0;
    const int be = min(bl_end, len);
    if (ok)
        for (int j = lane; j < len; j += 32) {
            const uint16_t v = in[j];
            out[j] = v;
            if (j >= bl_start && j < be) bsum += (short)v;
        }
    const long long ts = raw_ts[src] * ts_scale;
    double bl;
    if (baseline_f64 != nullptr) bl = baseline_f64[src];
    else if (baseline != nullptr) bl = (double)baseline[src];
    else {  // mean of the baseline window over the available samples (records_builder.py:243-257): exact integer sum
        bsum = warp_sum_i64(bsum);
        bl = (be > bl_start) ? (double)bsum / (double)(be - bl_start) : __longlong_as_double(0x7ff8000000000000ll);
    }
    if (meta != nullptr && lane == 0) {
        wfb_rec_meta m;
        m.timestamp = ts;
        m.baseline = bl;
        m.wave_offset = wave_offset;
        m.event_length = len;
        m.dt = dt_ns;
        m.board = board[src];
        m.channel = channel[src];
        m.polarity = WFB_POL_UNKNOWN;
        m.pad_[0] = m.pad_[1] = m.pad_[2] = 0;
        m.record_id = rid;
        meta[r] = m;
    }
    if (rows != nullptr) {
        long long t = ts / 1000;  // floor division like numpy's //
        if ((ts % 1000) != 0 && ts < 0) --t;
        t += epoch_ns;
        const unsigned fl = trunc != nullptr ? (unsigned)trunc[src] : 0u;
        uint16_t* row = rows + r * (kRecordsRowBytes / 2);
        row[lane] = v1725_row_halfword(lane, ts, board[src], channel[src], bl, rid, dt_ns, fl, wave_offset, len, t);
        if (lane + 32 < 51) row[lane + 32] = v1725_row_halfword(lane + 32, ts, board[src], channel[src], bl, rid, dt_ns, fl, wave_offset, len, t);
    }
}

}  // namespace wfb

using namespace wfb;

static unsigned v_nb(long long n, int t = 256) { return (unsigned)((n + t - 1) / t); }

extern "C" int wfb_v1725_scan_host(const uint8_t* blob_host, int64_t n_bytes, int64_t capacity, int64_t* payload_offset,
                                   int32_t* n_samples, int16_t* channel, int64_t* timestamp, uint16_t* baseline, uint8_t* trunc,
                                   int64_t* n_records, int64_t* n_samples_total) {
    WFB_REQUIRE(n_bytes >= 0 && capacity >= 0 && n_records != nullptr, "wfb_v1725_scan_host: bad arguments");
    WFB_REQUIRE(n_bytes == 0 || blob_host != nullptr, "wfb_v1725_scan_host: NULL stream");
    const bool store = capacity > 0;
    WFB_REQUIRE(!store || (payload_offset && n_samples && channel && timestamp && baseline && trunc),
                "wfb_v1725_scan_host: NULL output column");
    int64_t pos = 0, count = 0, total = 0;
    bool stop = false;
    while (!stop && n_bytes - pos >= 16) {  // a short event header ends the stream (v1725.py:80-85)
        const uint8_t* ev = blob_host + pos;
        pos += 16;
        const unsigned mask = (unsigned)ev[4] + ((unsigned)ev[11] << 8);
        for (int c = 0; c < 16 && !stop; ++c) {
            if (!((mask >> c) & 1u)) continue;
            if (n_bytes - pos < 12) { stop = true; break; }  // short channel header
            const uint8_t* h = blob_host + pos;
            pos += 12;
            const int64_t size = ((int64_t)h[0] | ((int64_t)h[1] << 8) | ((int64_t)h[2] << 16)) & ((1 << 22) - 1);
            const int64_t sig = (size - 3) * 4;
            WFB_REQUIRE(sig >= 0, "V1725 channel header with size < 3 words at byte %lld", (long long)(pos - 12));
            if (n_bytes - pos < sig) { stop = true; break; }  // short waveform
            if (store) {
                WFB_REQUIRE(count < capacity, "wfb_v1725_scan_host: more than %lld waveforms", (long long)capacity);
                payload_offset[count] = pos;
                n_samples[count] = (int32_t)(sig / 2);
                channel[count] = (int16_t)c;
                int64_t ts = 0;
                for (int k = 5; k >= 0; --k) ts = (ts << 8) | h[4 + k];
                timestamp[count] = ts;
                baseline[count] = (uint16_t)(h[10] | (h[11] << 8));
                trunc[count] = (uint8_t)((h[3] >> 6) & 1);
            }
            ++count;
            total += sig / 2;
            pos += sig;
        }
    }
    *n_records = count;
    if (n_samples_total) *n_samples_total = total;
    return WFB_OK;
}

extern "C" size_t wfb_build_records_v1725_workspace_bytes(int64_t n) {
    const size_t m = v_al256((size_t)std::max<int64_t>(n, 1) * 8);
    return 6 * m + radix_sort_workspace_bytes(n) + scan_workspace_bytes(n) + 512;
}

// common device part: sort, ragged offsets, gather.  seq_dev != NULL: record_id = seq[source index] instead of the
// output position (a rank's part of a run numbered over all files, shard_records.cu)
static int build_records_ragged(const uint8_t* blob_dev, int64_t blob_bytes, const int64_t* payload_offset_dev, const int32_t* n_samples_dev,
                                const int64_t* timestamp_dev, long long ts_scale, const int16_t* board_dev, const int16_t* channel_dev,
                                const uint16_t* baseline_u16_dev, const double* baseline_f64_dev, const uint8_t* flags_dev,
                                const int64_t* seq_dev, int64_t n,
                                int32_t dt_ns, int32_t bl_start, int32_t bl_end, int64_t epoch_ns, void* records_aos_dev, uint16_t* pool_dev,
                                int64_t pool_len, wfb_rec_meta* meta_dev, void* workspace_dev, size_t workspace_bytes, cudaStream_t st,
                                const char* who) {
    WFB_REQUIRE(n >= 0 && blob_bytes >= 0 && pool_len >= 0, "%s: negative size", who);
    if (n == 0) return WFB_OK;
    WFB_REQUIRE(blob_dev && payload_offset_dev && n_samples_dev && timestamp_dev && board_dev && channel_dev && workspace_dev, "%s: NULL pointer", who);
    WFB_REQUIRE(pool_len == 0 || pool_dev != nullptr, "%s: NULL wave_pool", who);
    WFB_REQUIRE(((uintptr_t)blob_dev & 1) == 0, "%s: the sample bytes must be 2-byte aligned", who);
    WFB_REQUIRE(dt_ns > 0, "%s: dt_ns must be positive", who);
    WFB_REQUIRE(workspace_bytes >= wfb_build_records_v1725_workspace_bytes(n), "%s: workspace too small", who);
    uint8_t* ws = static_cast<uint8_t*>(workspace_dev);
    const size_t m = v_al256((size_t)n * 8);
    unsigned long long* kA = reinterpret_cast<unsigned long long*>(ws);
    long long* vA = reinterpret_cast<long long*>(ws + m);
    unsigned long long* kB = reinterpret_cast<unsigned long long*>(ws + 2 * m);
    long long* vB = reinterpret_cast<long long*>(ws + 3 * m);
    long long* len_sorted = reinterpret_cast<long long*>(ws + 4 * m);
    long long* len_incl = reinterpret_cast<long long*>(ws + 5 * m);
    uint8_t* sws = ws + 6 * m;
    const size_t sort_bytes = radix_sort_workspace_bytes(n);
    void* scan_ws = sws + sort_bytes;
    // lexsort((seq, channel, board, pid, timestamp)): stable sort by (board, channel), then by timestamp
    v1725_keys_kernel<<<v_nb(n), 256, 0, st>>>(board_dev, channel_dev, n, kA, vA);
    int rc = radix_sort_pairs(kA, vA, kB, vB, n, kKeyUnsigned, sws, sort_bytes, st);
    if (rc != WFB_OK) return rc;
    v1725_gather_ts_kernel<<<v_nb(n), 256, 0, st>>>(reinterpret_cast<const long long*>(timestamp_dev), vB, n, ts_scale, kA);
    rc = radix_sort_pairs(kA, vB, kB, vA, n, kKeySigned, sws, sort_bytes, st);
    if (rc != WFB_OK) return rc;
    // ragged wave offsets
    v1725_lengths_kernel<<<v_nb(n), 256, 0, st>>>(n_samples_dev, vA, n, len_sorted);
    rc = inclusive_scan_sum_i64(len_sorted, len_incl, n, scan_ws, st);
    if (rc != WFB_OK) return rc;
    v1725_gather_kernel<<<v_nb(n * 32), 256, 0, st>>>(blob_dev, reinterpret_cast<const long long*>(payload_offset_dev), n_samples_dev,
                                                      reinterpret_cast<const long long*>(timestamp_dev), board_dev, channel_dev,
                                                      baseline_u16_dev, baseline_f64_dev, flags_dev, vA, len_incl,
                                                      reinterpret_cast<const long long*>(seq_dev), n, dt_ns, ts_scale,
                                                      bl_start, bl_end, epoch_ns, blob_bytes, pool_len,
                                                      static_cast<uint16_t*>(records_aos_dev), pool_dev, meta_dev);
    WFB_CUDA(cudaGetLastError());
    return WFB_OK;
}

extern "C" int wfb_build_records_ragged(const void* samples_dev, int64_t samples_bytes, const int64_t* sample_offset_dev,
                                        const int32_t* n_samples_dev, const int64_t* timestamp_ps_dev, const int16_t* board_dev,
                                        const int16_t* channel_dev, const double* baselines_in_dev, int64_t n, int32_t dt_ns,
                                        int32_t bl_start, int32_t bl_end, int64_t epoch_ns, void* records_aos_dev, uint16_t* pool_dev,
                                        int64_t pool_len, wfb_rec_meta* meta_dev, void* workspace_dev, size_t workspace_bytes, void* stream) {
    return build_records_ragged(static_cast<const uint8_t*>(samples_dev), samples_bytes, sample_offset_dev, n_samples_dev, timestamp_ps_dev, 1,
                                board_dev, channel_dev, nullptr, baselines_in_dev, nullptr, nullptr, n, dt_ns, bl_start, bl_end, epoch_ns,
                                records_aos_dev, pool_dev, pool_len, meta_dev, workspace_dev, workspace_bytes,
                                static_cast<cudaStream_t>(stream), "wfb_build_records_ragged");
}

extern "C" int wfb_build_records_ragged_seq(const void* samples_dev, int64_t samples_bytes, const int64_t* sample_offset_dev,
                                            const int32_t* n_samples_dev, const int64_t* timestamp_ps_dev, const int16_t* board_dev,
                                            const int16_t* channel_dev, const double* baselines_in_dev, const int64_t* seq_dev, int64_t n,
                                            int32_t dt_ns, int32_t bl_start, int32_t bl_end, int64_t epoch_ns, void* records_aos_dev,
                                            uint16_t* pool_dev, int64_t pool_len, wfb_rec_meta* meta_dev, void* workspace_dev,
                                            size_t workspace_bytes, void* stream) {
    WFB_REQUIRE(n == 0 || seq_dev != nullptr, "wfb_build_records_ragged_seq: NULL seq");
    return build_records_ragged(static_cast<const uint8_t*>(samples_dev), samples_bytes, sample_offset_dev, n_samples_dev, timestamp_ps_dev, 1,
                                board_dev, channel_dev, nullptr, baselines_in_dev, nullptr, seq_dev, n, dt_ns, bl_start, bl_end, epoch_ns,
                                records_aos_dev, pool_dev, pool_len, meta_dev, workspace_dev, workspace_bytes,
                                static_cast<cudaStream_t>(stream), "wfb_build_records_ragged_seq");
}

static int build_v1725(const uint8_t* blob_dev, int64_t blob_bytes, const int64_t* payload_offset_dev, const int32_t* n_samples_dev,
                       const int64_t* timestamp_dev, const int16_t* board_dev, const int16_t* channel_dev, const uint16_t* baseline_dev,
                       const uint8_t* trunc_dev, const int64_t* seq_dev, int64_t n, int32_t dt_ns, void* records_aos_dev, uint16_t* pool_dev,
                       int64_t pool_len, wfb_rec_meta* meta_dev, void* workspace_dev, size_t workspace_bytes, void* stream, const char* who) {
    WFB_REQUIRE(n == 0 || (baseline_dev && trunc_dev), "%s: NULL pointer", who);
    WFB_REQUIRE(n == 0 || ((uintptr_t)blob_dev & 3) == 0, "%s: the stream must be 4-byte aligned", who);
    return build_records_ragged(blob_dev, blob_bytes, payload_offset_dev, n_samples_dev, timestamp_dev, (long long)dt_ns * 1000ll, board_dev,
                                channel_dev, baseline_dev, nullptr, trunc_dev, seq_dev, n, dt_ns, 0, 0, 0, records_aos_dev, pool_dev, pool_len,
                                meta_dev, workspace_dev, workspace_bytes, static_cast<cudaStream_t>(stream), who);
}

extern "C" int wfb_build_records_v1725(const uint8_t* blob_dev, int64_t blob_bytes, const int64_t* payload_offset_dev,
                                       const int32_t* n_samples_dev, const int64_t* timestamp_dev, const int16_t* board_dev,
                                       const int16_t* channel_dev, const uint16_t* baseline_dev, const uint8_t* trunc_dev, int64_t n,
                                       int32_t dt_ns, void* records_aos_dev, uint16_t* pool_dev, int64_t pool_len,
                                       wfb_rec_meta* meta_dev, void* workspace_dev, size_t workspace_bytes, void* stream) {
    return build_v1725(blob_dev, blob_bytes, payload_offset_dev, n_samples_dev, timestamp_dev, board_dev, channel_dev, baseline_dev, trunc_dev,
                       nullptr, n, dt_ns, records_aos_dev, pool_dev, pool_len, meta_dev, workspace_dev, workspace_bytes, stream,
                       "wfb_build_records_v1725");
}

extern "C" int wfb_build_records_v1725_seq(const uint8_t* blob_dev, int64_t blob_bytes, const int64_t* payload_offset_dev,
                                           const int32_t* n_samples_dev, const int64_t* timestamp_dev, const int16_t* board_dev,
                                           const int16_t* channel_dev, const uint16_t* baseline_dev, const uint8_t* trunc_dev,
                                           const int64_t* seq_dev, int64_t n, int32_t dt_ns, void* records_aos_dev, uint16_t* pool_dev,
                                           int64_t pool_len, wfb_rec_meta* meta_dev, void* workspace_dev, size_t workspace_bytes,
                                           void* stream) {
    WFB_REQUIRE(n == 0 || seq_dev != nullptr, "wfb_build_records_v1725_seq: NULL seq");
    return build_v1725(blob_dev, blob_bytes, payload_offset_dev, n_samples_dev, timestamp_dev, board_dev, channel_dev, baseline_dev, trunc_dev,
                       seq_dev, n, dt_ns, records_aos_dev, pool_dev, pool_len, meta_dev, workspace_dev, workspace_bytes, stream,
                       "wfb_build_records_v1725_seq");
}
