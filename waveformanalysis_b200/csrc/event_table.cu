// The device event table of anchored fixed-window clustering (df_events, event_grouping.py:99-283): CSR offsets,
// members ordered by channel inside every event, t_min / t_max / dt/ns / n_hits and the member-ordered columns that
// df_events' list columns and wfb_pair_events read.
//
// Events are contiguous runs of the time-sorted rows (wfb_group_time_window numbers them 0, 1, ... in row order).
// The member order is np.lexsort((arange, channel, event)): by channel, equal channels in row order.
//   * events of up to 32 members: one warp per event ranks its members in registers - lane j's rank is the number of
//     members with a smaller channel, or the same channel and a smaller position - and scatters them;
//   * larger events: their rows are compacted (in row order) and ordered by ONE stable radix sort on the composite key
//     (event << 16 | channel + 32768), so a run that is one giant event stays O(n).
// t_min / t_max are the timestamps of the first / last member in that order (not the min / max), dt/ns is numpy's
// int64 difference over 1e3.
#include <algorithm>

#include "common.cuh"
#include "sort_scan.cuh"

namespace wfb {

static size_t et_al(size_t x) { return (x + 255) & ~(size_t)255; }

struct EtIn {
    const long long* ts;       // sorted positions
    const long long* ev;       // sorted positions
    const short* ch;           // input rows
    const long long* order;    // sorted position -> input row, or NULL (identity)
    const float* area;         // input rows, optional
    const float* height;       // input rows, optional
};
struct EtOut {
    long long* members;
    long long* ts;
    short* ch;
    float* area;
    float* height;
};

__device__ __forceinline__ void et_put(const EtIn& in, const EtOut& o, long long k, long long dst) {
    const long long src = in.order ? in.order[k] : k;
    o.members[dst] = src;
    o.ts[dst] = in.ts[k];
    o.ch[dst] = in.ch[src];
    if (o.area) o.area[dst] = in.area[src];
    if (o.height) o.height[dst] = in.height[src];
}

// offsets[e] = first row of event e, offsets[n_events] = n
__global__ void et_offsets_kernel(const long long* __restrict__ ev, long long n, long long n_events, long long* __restrict__ offsets) {
    const long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (k >= n) return;
    if (k == 0 || ev[k] != ev[k - 1]) offsets[ev[k]] = k;
    if (k == n - 1) offsets[n_events] = n;
}

// one warp per event: events of <= 32 members are ranked in registers; larger ones only add their rows to *n_big
__global__ void __launch_bounds__(256) et_small_kernel(EtIn in, const long long* __restrict__ offsets, long long n_events, EtOut o,
                                                       unsigned long long* __restrict__ n_big) {
    const long long e = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
    if (e >= n_events) return;
    const int lane = lane_id();
    const long long b = offsets[e];
    const long long m = offsets[e + 1] - b;
    if (m > 32) {
        if (lane == 0) atomicAdd(n_big, (unsigned long long)m);
        return;
    }
    const bool live = lane < m;
    const int c = live ? (int)in.ch[in.order ? in.order[b + lane] : b + lane] : 0x7fffffff;
    int rank = 0;
    for (int i = 0; i < (int)m; ++i) {
        const int ci = __shfl_sync(kFull, c, i);
        rank += (ci < c) || (ci == c && i < lane);
    }
    if (live) et_put(in, o, b + lane, b + rank);
}

// rows of events with more than 32 members (flag, for the compaction scan)
__global__ void et_big_flags_kernel(const long long* __restrict__ ev, const long long* __restrict__ offsets, long long n,
                                    long long* __restrict__ flag) {
    const long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (k >= n) return;
    const long long e = ev[k];
    flag[k] = (offsets[e + 1] - offsets[e]) > 32 ? 1 : 0;
}

__global__ void et_big_keys_kernel(const EtIn in, const long long* __restrict__ flag, const long long* __restrict__ incl, long long n,
                                   unsigned long long* __restrict__ keys, long long* __restrict__ vals) {
    const long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (k >= n || !flag[k]) return;
    const long long j = incl[k] - 1;
    const int c = (int)in.ch[in.order ? in.order[k] : k];
    keys[j] = ((unsigned long long)in.ev[k] << 16) | (unsigned long long)(unsigned)(c + 32768);
    vals[j] = k;
}

// the j-th sorted big row goes to offsets[e] + (j - first compacted index of event e)
__global__ void et_big_scatter_kernel(const EtIn in, const unsigned long long* __restrict__ keys, const long long* __restrict__ vals,
                                      long long n_big, const long long* __restrict__ offsets, const long long* __restrict__ incl, EtOut o) {
    const long long j = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (j >= n_big) return;
    const long long e = (long long)(keys[j] >> 16);
    const long long b = offsets[e];
    const long long first = incl[b] - 1;  // the event's first row is flagged
    et_put(in, o, vals[j], b + (j - first));
}

__global__ void et_stats_kernel(const long long* __restrict__ offsets, const long long* __restrict__ member_ts, long long n_events,
                                long long* __restrict__ t_min, long long* __restrict__ t_max, double* __restrict__ dt_ns,
                                long long* __restrict__ n_hits) {
    const long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (e >= n_events) return;
    const long long b = offsets[e], z = offsets[e + 1];
    const long long t0 = member_ts[b], t1 = member_ts[z - 1];
    t_min[e] = t0;
    t_max[e] = t1;
    dt_ns[e] = __ddiv_rn((double)(t1 - t0), 1e3);
    n_hits[e] = z - b;
}

}  // namespace wfb

using namespace wfb;

static unsigned et_nb(long long n, int t = 256) { return (unsigned)((n + t - 1) / t); }

extern "C" size_t wfb_event_table_workspace_bytes(int64_t n) {
    const size_t m = et_al((size_t)std::max<int64_t>(n, 1) * 8);
    return 6 * m + et_al(radix_sort_workspace_bytes(n)) + et_al(scan_workspace_bytes(n)) + 512;
}

extern "C" int wfb_event_table(const int64_t* ts_sorted_dev, const int64_t* event_id_dev, int64_t n, int64_t n_events,
                               const int16_t* channel_dev, const int64_t* order_dev, const float* area_dev, const float* height_dev,
                               int64_t* offsets_dev, int64_t* members_dev, int64_t* t_min_dev, int64_t* t_max_dev, double* dt_ns_dev,
                               int64_t* n_hits_dev, int64_t* member_ts_dev, int16_t* member_channel_dev, float* member_area_dev,
                               float* member_height_dev, void* workspace_dev, size_t workspace_bytes, void* stream) {
    WFB_REQUIRE(n >= 0 && n_events >= 0 && n_events <= n, "wfb_event_table: bad sizes");
    WFB_REQUIRE(n_events > 0 || n == 0, "wfb_event_table: rows without events");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (offsets_dev) WFB_CUDA(cudaMemsetAsync(offsets_dev, 0, 8, st));
    if (n == 0) return WFB_OK;
    WFB_REQUIRE(n_events < (1ll << 47), "wfb_event_table: too many events");
    WFB_REQUIRE(ts_sorted_dev && event_id_dev && channel_dev && offsets_dev && members_dev && t_min_dev && t_max_dev && dt_ns_dev &&
                    n_hits_dev && member_ts_dev && member_channel_dev && workspace_dev,
                "wfb_event_table: NULL pointer");
    WFB_REQUIRE((area_dev == nullptr) == (member_area_dev == nullptr) && (height_dev == nullptr) == (member_height_dev == nullptr),
                "wfb_event_table: area / height need both the input and the output column");
    WFB_REQUIRE(workspace_bytes >= wfb_event_table_workspace_bytes(n), "wfb_event_table: workspace too small");
    uint8_t* ws = static_cast<uint8_t*>(workspace_dev);
    const size_t m = et_al((size_t)n * 8);
    long long* flag = reinterpret_cast<long long*>(ws);
    long long* incl = reinterpret_cast<long long*>(ws + m);
    unsigned long long* kA = reinterpret_cast<unsigned long long*>(ws + 2 * m);
    long long* vA = reinterpret_cast<long long*>(ws + 3 * m);
    unsigned long long* kB = reinterpret_cast<unsigned long long*>(ws + 4 * m);
    long long* vB = reinterpret_cast<long long*>(ws + 5 * m);
    uint8_t* sws = ws + 6 * m;
    const size_t sort_bytes = radix_sort_workspace_bytes(n);
    void* scan_ws = sws + et_al(sort_bytes);
    unsigned long long* d_big = reinterpret_cast<unsigned long long*>(static_cast<uint8_t*>(scan_ws) + et_al(scan_workspace_bytes(n)));

    const EtIn in{reinterpret_cast<const long long*>(ts_sorted_dev), reinterpret_cast<const long long*>(event_id_dev), channel_dev,
                  reinterpret_cast<const long long*>(order_dev), area_dev, height_dev};
    const EtOut o{reinterpret_cast<long long*>(members_dev), reinterpret_cast<long long*>(member_ts_dev), member_channel_dev,
                  member_area_dev, member_height_dev};
    long long* offsets = reinterpret_cast<long long*>(offsets_dev);

    et_offsets_kernel<<<et_nb(n), 256, 0, st>>>(in.ev, n, n_events, offsets);
    WFB_CUDA(cudaMemsetAsync(d_big, 0, 8, st));
    et_small_kernel<<<et_nb(n_events * 32), 256, 0, st>>>(in, offsets, n_events, o, d_big);
    WFB_CUDA(cudaGetLastError());
    unsigned long long n_big = 0;
    WFB_CUDA(cudaMemcpyAsync(&n_big, d_big, 8, cudaMemcpyDeviceToHost, st));
    WFB_CUDA(cudaStreamSynchronize(st));
    if (n_big > 0) {
        et_big_flags_kernel<<<et_nb(n), 256, 0, st>>>(in.ev, offsets, n, flag);
        int rc = inclusive_scan_sum_i64(flag, incl, n, scan_ws, st);
        if (rc != WFB_OK) return rc;
        et_big_keys_kernel<<<et_nb(n), 256, 0, st>>>(in, flag, incl, n, kA, vA);
        rc = radix_sort_pairs(kA, vA, kB, vB, (long long)n_big, kKeyUnsigned, sws, sort_bytes, st);
        if (rc != WFB_OK) return rc;
        et_big_scatter_kernel<<<et_nb((long long)n_big), 256, 0, st>>>(in, kB, vB, (long long)n_big, offsets, incl, o);
        WFB_CUDA(cudaGetLastError());
    }
    et_stats_kernel<<<et_nb(n_events), 256, 0, st>>>(offsets, o.ts, n_events, reinterpret_cast<long long*>(t_min_dev),
                                                     reinterpret_cast<long long*>(t_max_dev), dt_ns_dev,
                                                     reinterpret_cast<long long*>(n_hits_dev));
    WFB_CUDA(cudaGetLastError());
    return WFB_OK;
}
