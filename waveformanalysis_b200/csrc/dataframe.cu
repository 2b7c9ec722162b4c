// The step after the hot path: columns of `df`, `s1_s2` labels, `df_paired` columns.
// Elementwise / gather kernels around the device radix sort; every row format is the reference's
// packed numpy dtype (dataframe.py:222-246, s1_s2_classifier.py:29-42, analyzer.py:66-110).
#include <cmath>
#include <vector>

#include "common.cuh"
#include "sort_scan.cuh"

namespace wfb {

constexpr int kFeatRow = 36;   // BASIC_FEATURES_DTYPE
constexpr int kWidthRow = 56;  // WAVEFORM_WIDTH_DTYPE
constexpr int kS1S2Row = 45;   // S1_S2_CLASSIFIER_DTYPE

__device__ __forceinline__ long long ld_i64_u4(const uint8_t* p) {  // int64 at a 4-byte aligned address
    const unsigned* q = reinterpret_cast<const unsigned*>(p);
    return (long long)(((unsigned long long)q[1] << 32) | q[0]);
}

__global__ void df_keys_kernel(const uint8_t* feat, long long n, unsigned long long* keys, long long* vals) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= n) return;
    keys[i] = (unsigned long long)ld_i64_u4(feat + i * kFeatRow + 16);
    vals[i] = i;
}

struct DfOut {
    long long* ts;
    long long* rid;
    float *area, *height, *amp, *mad;
    short *board, *channel;
    double *area_pe, *height_pe;
};

__global__ void df_gather_kernel(const uint8_t* feat, const long long* record_id, const long long* order, long long n,
                                 const wfb_gain_rule* gains, int n_gains, int with_pe, DfOut o) {
    const long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (k >= n) return;
    const long long src = order[k];
    const uint8_t* row = feat + src * kFeatRow;
    const float* f = reinterpret_cast<const float*>(row);
    const float height = f[0], amp = f[1], area = f[2], mad = f[3];
    const unsigned bc = *reinterpret_cast<const unsigned*>(row + 24);
    const short board = (short)(bc & 0xffffu), channel = (short)(bc >> 16);
    o.ts[k] = ld_i64_u4(row + 16);
    o.rid[k] = record_id ? record_id[src] : src;
    o.area[k] = area;
    o.height[k] = height;
    o.amp[k] = amp;
    o.mad[k] = mad;
    o.board[k] = board;
    o.channel[k] = channel;
    if (with_pe) {
        double g = nan("");
        for (int i = 0; i < n_gains; ++i)
            if (gains[i].board == (int)board && gains[i].channel == (int)channel) g = gains[i].gain;
        o.area_pe[k] = __ddiv_rn((double)area, g);
        o.height_pe[k] = __ddiv_rn((double)height, g);
    }
}

__device__ __forceinline__ bool in_range(double v, const wfb_range& r) {  // s1_s2_classifier.py:54-68
    if (!r.present) return true;
    if (isnan(v)) return false;
    if (r.has_lo && v < r.lo) return false;
    if (r.has_hi && v > r.hi) return false;
    return true;
}

__device__ __forceinline__ void put_bytes(uint8_t* dst, const void* src, int nbytes) {
    const uint8_t* s = static_cast<const uint8_t*>(src);
    for (int i = 0; i < nbytes; ++i) dst[i] = s[i];
}

constexpr int kS1S2Block = 128;

__global__ void __launch_bounds__(kS1S2Block) s1s2_kernel(const uint8_t* widths, long long n_peaks, const uint8_t* feat, long long n_feat,
                                                          const wfb_s1s2_params p, uint8_t* out) {
    __shared__ __align__(16) uint8_t stage[kS1S2Block * kS1S2Row];
    const long long base = blockIdx.x * (long long)kS1S2Block;
    const long long i = base + threadIdx.x;
    if (i < n_peaks) {
        const uint8_t* w = widths + i * kWidthRow;
        const float width_ns = *reinterpret_cast<const float*>(w + 8);
        const float width_samples = *reinterpret_cast<const float*>(w + 20);
        const long long peak_position = ld_i64_u4(w + 24);
        const long long ts = ld_i64_u4(w + 36);
        const unsigned bc = *reinterpret_cast<const unsigned*>(w + 44);
        const long long rid = ld_i64_u4(w + 48);
        const long long frow = rid - p.feat_row_base;
        float height = nanf(""), area = nanf("");
        if (frow >= 0 && frow < n_feat) {
            const float* f = reinterpret_cast<const float*>(feat + frow * kFeatRow);
            height = f[0];
            area = f[2];
        }
        const double wv = p.width_in_samples ? (double)width_samples : (double)width_ns;
        const bool s1_en = p.s1_width.present || p.s1_area.present || p.s1_height.present;
        const bool s2_en = p.s2_width.present || p.s2_area.present || p.s2_height.present;
        const bool s1 = s1_en && in_range(wv, p.s1_width) && in_range((double)area, p.s1_area) && in_range((double)height, p.s1_height);
        const bool s2 = s2_en && in_range(wv, p.s2_width) && in_range((double)area, p.s2_area) && in_range((double)height, p.s2_height);
        signed char label = 0;
        if (s1 && !s2) label = 1;
        else if (s2 && !s1) label = 2;
        else if (s1 && s2) label = (p.conflict_policy == 1) ? 1 : (p.conflict_policy == 2) ? 2 : 0;
        uint8_t* d = stage + threadIdx.x * kS1S2Row;
        d[0] = (uint8_t)label;
        put_bytes(d + 1, &width_ns, 4);
        put_bytes(d + 5, &width_samples, 4);
        put_bytes(d + 9, &height, 4);
        put_bytes(d + 13, &area, 4);
        put_bytes(d + 17, &ts, 8);
        put_bytes(d + 25, &bc, 4);
        put_bytes(d + 29, &rid, 8);
        put_bytes(d + 37, &peak_position, 8);
    }
    __syncthreads();
    const long long rows = min((long long)kS1S2Block, n_peaks - base);
    const int nbytes = (int)rows * kS1S2Row;
    uint8_t* dst = out + base * kS1S2Row;  // base * 45 is a multiple of 4 * 45 * 32: word aligned when out is
    if ((((uintptr_t)dst) & 3) == 0) {
        const int nw = nbytes >> 2;
        for (int k = threadIdx.x; k < nw; k += kS1S2Block) reinterpret_cast<unsigned*>(dst)[k] = reinterpret_cast<const unsigned*>(stage)[k];
        for (int k = (nw << 2) + threadIdx.x; k < nbytes; k += kS1S2Block) dst[k] = stage[k];
    } else {
        for (int k = threadIdx.x; k < nbytes; k += kS1S2Block) dst[k] = stage[k];
    }
}

__global__ void pair_events_kernel(const long long* offsets, long long n_events, const long long* ts, const float* area,
                                   const float* height, const double* dt_ns, double tw, int n_channels, uint8_t* keep,
                                   double* delta_t, float* area_ch, float* height_ch) {
    const long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (e >= n_events) return;
    const long long b = offsets[e], m = offsets[e + 1] - b;
    keep[e] = dt_ns[e] <= tw ? 1 : 0;
    delta_t[e] = (m > 0) ? __ddiv_rn((double)(ts[b + m - 1] - ts[b]), 1000.0) : nan("");
    for (int i = 0; i < n_channels; ++i) {
        const bool have = i < m;
        area_ch[e * n_channels + i] = have ? area[b + i] : nanf("");
        height_ch[e * n_channels + i] = have ? height[b + i] : nanf("");
    }
}

static size_t df_al(size_t x) { return (x + 255) & ~(size_t)255; }

}  // namespace wfb

using namespace wfb;

extern "C" size_t wfb_df_columns_workspace_bytes(int64_t n) {
    if (n < 1) n = 1;
    return 3 * df_al((size_t)n * 8) + radix_sort_workspace_bytes(n) + 64 * 1024 + 512;
}

extern "C" int wfb_df_columns(const void* feat_rows_dev, const int64_t* record_id_dev, int64_t n, const wfb_gain_rule* gains_host,
                              int32_t n_gains, int32_t with_pe, int64_t* order_dev, int64_t* timestamp_dev,
                              int64_t* record_id_out_dev, float* area_dev, float* height_dev, float* amp_dev,
                              float* max_abs_diff_dev, int16_t* board_dev, int16_t* channel_dev, double* area_pe_dev,
                              double* height_pe_dev, void* workspace_dev, size_t workspace_bytes, void* stream) {
    WFB_REQUIRE(n >= 0, "wfb_df_columns: negative size");
    if (n == 0) return WFB_OK;
    WFB_REQUIRE(feat_rows_dev && order_dev && timestamp_dev && record_id_out_dev && area_dev && height_dev && amp_dev &&
                    max_abs_diff_dev && board_dev && channel_dev,
                "wfb_df_columns: NULL pointer");
    WFB_REQUIRE(!with_pe || (area_pe_dev && height_pe_dev), "wfb_df_columns: calibrated columns requested without buffers");
    WFB_REQUIRE(n_gains >= 0 && (n_gains == 0 || gains_host), "wfb_df_columns: gains_host is NULL");
    WFB_REQUIRE((size_t)n_gains * sizeof(wfb_gain_rule) <= 64 * 1024, "wfb_df_columns: too many gain entries");
    WFB_REQUIRE(((uintptr_t)feat_rows_dev & 3) == 0, "wfb_df_columns: feat_rows_dev must be 4-byte aligned");
    WFB_REQUIRE(workspace_bytes >= wfb_df_columns_workspace_bytes(n), "wfb_df_columns: workspace too small");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    uint8_t* ws = static_cast<uint8_t*>(workspace_dev);
    const size_t m = df_al((size_t)n * 8);
    unsigned long long* kA = reinterpret_cast<unsigned long long*>(ws);
    unsigned long long* kB = reinterpret_cast<unsigned long long*>(ws + m);
    long long* vA = reinterpret_cast<long long*>(ws + 2 * m);
    wfb_gain_rule* d_gains = reinterpret_cast<wfb_gain_rule*>(ws + 3 * m);
    uint8_t* sws = ws + 3 * m + 64 * 1024;
    const uint8_t* feat = static_cast<const uint8_t*>(feat_rows_dev);
    const unsigned blocks = (unsigned)((n + 255) / 256);
    df_keys_kernel<<<blocks, 256, 0, st>>>(feat, n, kA, vA);
    WFB_CUDA(cudaGetLastError());
    int rc = radix_sort_pairs(kA, vA, kB, reinterpret_cast<long long*>(order_dev), n, kKeySigned, sws, radix_sort_workspace_bytes(n), st);
    if (rc != WFB_OK) return rc;
    if (with_pe && n_gains > 0) {
        // pageable source: the copy is staged before the call returns, the caller's array may go away
        WFB_CUDA(cudaMemcpyAsync(d_gains, gains_host, (size_t)n_gains * sizeof(wfb_gain_rule), cudaMemcpyHostToDevice, st));
    }
    DfOut o;
    o.ts = reinterpret_cast<long long*>(timestamp_dev);
    o.rid = reinterpret_cast<long long*>(record_id_out_dev);
    o.area = area_dev; o.height = height_dev; o.amp = amp_dev; o.mad = max_abs_diff_dev;
    o.board = board_dev; o.channel = channel_dev;
    o.area_pe = area_pe_dev; o.height_pe = height_pe_dev;
    df_gather_kernel<<<blocks, 256, 0, st>>>(feat, reinterpret_cast<const long long*>(record_id_dev), reinterpret_cast<const long long*>(order_dev), n,
                                              d_gains, with_pe ? n_gains : 0, with_pe, o);
    WFB_CUDA(cudaGetLastError());
    return WFB_OK;
}

extern "C" int wfb_s1s2_classify(const void* width_rows_dev, int64_t n_peaks, const void* feat_rows_dev, int64_t n_feat,
                                 const wfb_s1s2_params* params, void* out_rows_dev, void* stream) {
    WFB_REQUIRE(params != nullptr, "wfb_s1s2_classify: params is NULL");
    WFB_REQUIRE(n_peaks >= 0 && n_feat >= 0, "wfb_s1s2_classify: negative size");
    WFB_REQUIRE(params->conflict_policy >= 0 && params->conflict_policy <= 2, "wfb_s1s2_classify: unknown conflict_policy");
    if (n_peaks == 0) return WFB_OK;
    WFB_REQUIRE(width_rows_dev && out_rows_dev && (feat_rows_dev || n_feat == 0), "wfb_s1s2_classify: NULL pointer");
    WFB_REQUIRE(((uintptr_t)width_rows_dev & 3) == 0 && ((uintptr_t)feat_rows_dev & 3) == 0, "wfb_s1s2_classify: rows must be 4-byte aligned");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const unsigned blocks = (unsigned)((n_peaks + kS1S2Block - 1) / kS1S2Block);
    s1s2_kernel<<<blocks, kS1S2Block, 0, st>>>(static_cast<const uint8_t*>(width_rows_dev), n_peaks, static_cast<const uint8_t*>(feat_rows_dev),
                                               n_feat, *params, static_cast<uint8_t*>(out_rows_dev));
    WFB_CUDA(cudaGetLastError());
    return WFB_OK;
}

extern "C" int wfb_pair_events(const int64_t* offsets_dev, int64_t n_events, const int64_t* member_ts_dev,
                               const float* member_area_dev, const float* member_height_dev, const double* dt_ns_dev,
                               double time_window_ns, int32_t n_channels, uint8_t* keep_dev, double* delta_t_dev,
                               float* area_ch_dev, float* height_ch_dev, void* stream) {
    WFB_REQUIRE(n_events >= 0 && n_channels >= 0, "wfb_pair_events: negative size");
    if (n_events == 0) return WFB_OK;
    WFB_REQUIRE(offsets_dev && member_ts_dev && member_area_dev && member_height_dev && dt_ns_dev && keep_dev && delta_t_dev,
                "wfb_pair_events: NULL pointer");
    WFB_REQUIRE(n_channels == 0 || (area_ch_dev && height_ch_dev), "wfb_pair_events: per-channel buffers are NULL");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    pair_events_kernel<<<(unsigned)((n_events + 255) / 256), 256, 0, st>>>(
        reinterpret_cast<const long long*>(offsets_dev), n_events, reinterpret_cast<const long long*>(member_ts_dev), member_area_dev,
        member_height_dev, dt_ns_dev, time_window_ns, n_channels, keep_dev, delta_t_dev, area_ch_dev, height_ch_dev);
    WFB_CUDA(cudaGetLastError());
    return WFB_OK;
}
