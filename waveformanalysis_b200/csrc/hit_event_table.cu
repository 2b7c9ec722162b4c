// The device event table of chain-clustered hit windows (hit_grouped, event_grouping.py:287-471): CSR offsets,
// members ordered by (board, channel, dt, abs_start, timestamp, record_id, input row) inside every event, t_min / t_max /
// dt/ns / n_hits and, optionally, the packed hit rows in member order.
//
// wfb_group_hit_windows / wfb_group_abs_windows leave `order` = lexsort((record_id, timestamp, dt, abs_start)) (stable,
// so ties keep the input row order) and number the events 0, 1, ... along it: every event is a contiguous run of
// `order`.  A stable sort of that run by (board, channel, dt) therefore gives the reference's member order
// np.lexsort((record_id, timestamp, abs_start, dt, channel, board, event)), and the three fields fit one 64-bit key:
//   * events of up to 32 members: one warp per event ranks its members in registers - lane j's rank is the number of
//     members with a smaller key, or the same key and a smaller position - and scatters them;
//   * larger events: their positions are compacted (in order) and sorted by two stable radix sorts, first by the
//     (board, channel, dt) key, then by the event, so a run that is one giant event stays O(n).
// t_min = (int64) min abs_start is the abs_start of the event's first position (abs_start is the primary sort key);
// t_max = (int64) max abs_end comes from one segmented running maximum over the positions.  The casts truncate toward
// zero like numpy's astype; dt/ns is numpy's int64 difference over 1e3.
#include <algorithm>

#include "common.cuh"
#include "sort_scan.cuh"

namespace wfb {

static size_t ht_al(size_t x) { return (x + 255) & ~(size_t)255; }

struct HtIn {
    const long long* order;  // sorted position -> input row
    const long long* ev;     // input rows
    const short* board;      // input rows
    const short* channel;
    const int* dt;
    const double* a0;
    const double* a1;
    const uint8_t* rows;     // input rows, optional (row_bytes each)
    int row_words;
};
struct HtOut {
    long long* members;
    uint8_t* rows;  // member order, optional
};

// (board, channel, dt) as one unsigned key in signed ascending order of each field
__device__ __forceinline__ unsigned long long ht_key(const HtIn& in, long long r) {
    const unsigned long long b = (unsigned)((int)in.board[r] + 32768), c = (unsigned)((int)in.channel[r] + 32768);
    return (b << 48) | (c << 32) | (unsigned long long)((unsigned)in.dt[r] ^ 0x80000000u);
}

__device__ __forceinline__ void ht_put(const HtIn& in, const HtOut& o, long long r, long long dst) {
    o.members[dst] = r;
    if (o.rows) {
        const unsigned* s = reinterpret_cast<const unsigned*>(in.rows) + r * in.row_words;
        unsigned* d = reinterpret_cast<unsigned*>(o.rows) + dst * in.row_words;
        for (int w = 0; w < in.row_words; ++w) d[w] = s[w];
    }
}

// offsets[e] = first position of event e, offsets[n_events] = n; the (abs_end, event) pairs of the running maximum
__global__ void ht_offsets_kernel(const HtIn in, long long n, long long n_events, long long* __restrict__ offsets,
                                  SegMax* __restrict__ sm) {
    const long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (k >= n) return;
    const long long r = in.order[k];
    const long long e = in.ev[r];
    if (k == 0 || in.ev[in.order[k - 1]] != e) offsets[e] = k;
    if (k == n - 1) offsets[n_events] = n;
    sm[k] = SegMax{in.a1[r], e};
}

__global__ void ht_stats_kernel(const HtIn in, const long long* __restrict__ offsets, const SegMax* __restrict__ pm, long long n_events,
                                long long* __restrict__ t_min, long long* __restrict__ t_max, double* __restrict__ dt_ns,
                                long long* __restrict__ n_hits) {
    const long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (e >= n_events) return;
    const long long b = offsets[e], z = offsets[e + 1];
    const long long t0 = (long long)in.a0[in.order[b]], t1 = (long long)pm[z - 1].v;
    t_min[e] = t0;
    t_max[e] = t1;
    dt_ns[e] = __ddiv_rn((double)(t1 - t0), 1e3);
    n_hits[e] = z - b;
}

// one warp per event: events of <= 32 members are ranked in registers; larger ones only add their rows to *n_big
__global__ void __launch_bounds__(256) ht_small_kernel(const HtIn in, const long long* __restrict__ offsets, long long n_events, HtOut o,
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
    const long long r = live ? in.order[b + lane] : 0;
    const unsigned long long key = live ? ht_key(in, r) : ~0ull;
    int rank = 0;
    for (int i = 0; i < (int)m; ++i) {
        const unsigned long long ki = __shfl_sync(kFull, key, i);
        rank += (ki < key) || (ki == key && i < lane);
    }
    if (live) ht_put(in, o, r, b + rank);
}

// positions of events with more than 32 members (flag, for the compaction scan)
__global__ void ht_big_flags_kernel(const HtIn in, const long long* __restrict__ offsets, long long n, long long* __restrict__ flag) {
    const long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (k >= n) return;
    const long long e = in.ev[in.order[k]];
    flag[k] = (offsets[e + 1] - offsets[e]) > 32 ? 1 : 0;
}

__global__ void ht_big_keys_kernel(const HtIn in, const long long* __restrict__ flag, const long long* __restrict__ incl, long long n,
                                   unsigned long long* __restrict__ keys, long long* __restrict__ vals) {
    const long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (k >= n || !flag[k]) return;
    const long long j = incl[k] - 1;
    keys[j] = ht_key(in, in.order[k]);
    vals[j] = k;
}

// second pass: the event of every (board, channel, dt)-sorted position
__global__ void ht_big_event_keys_kernel(const HtIn in, const long long* __restrict__ vals, long long n_big,
                                         unsigned long long* __restrict__ keys) {
    const long long j = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (j >= n_big) return;
    keys[j] = (unsigned long long)in.ev[in.order[vals[j]]];
}

// the j-th sorted big position goes to offsets[e] + (j - first compacted index of event e)
__global__ void ht_big_scatter_kernel(const HtIn in, const unsigned long long* __restrict__ keys, const long long* __restrict__ vals,
                                      long long n_big, const long long* __restrict__ offsets, const long long* __restrict__ incl, HtOut o) {
    const long long j = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (j >= n_big) return;
    const long long e = (long long)keys[j];
    const long long b = offsets[e];
    const long long first = incl[b] - 1;  // the event's first position is flagged
    ht_put(in, o, in.order[vals[j]], b + (j - first));
}

}  // namespace wfb

using namespace wfb;

static unsigned ht_nb(long long n, int t = 256) { return (unsigned)((n + t - 1) / t); }

extern "C" size_t wfb_hit_event_table_workspace_bytes(int64_t n) {
    const size_t m = ht_al((size_t)std::max<int64_t>(n, 1) * 8);
    return 6 * m + ht_al(radix_sort_workspace_bytes(n)) + 2 * ht_al(scan_workspace_bytes(n)) + 512;
}

extern "C" int wfb_hit_event_table(const int64_t* order_dev, const int64_t* event_id_dev, int64_t n, int64_t n_events,
                                   const int16_t* board_dev, const int16_t* channel_dev, const int32_t* dt_dev,
                                   const double* abs_start_dev, const double* abs_end_dev, const void* rows_dev, int32_t row_bytes,
                                   int64_t* offsets_dev, int64_t* members_dev, int64_t* t_min_dev, int64_t* t_max_dev,
                                   double* dt_ns_dev, int64_t* n_hits_dev, void* member_rows_dev, void* workspace_dev,
                                   size_t workspace_bytes, void* stream) {
    WFB_REQUIRE(n >= 0 && n_events >= 0 && n_events <= n, "wfb_hit_event_table: bad sizes");
    WFB_REQUIRE(n_events > 0 || n == 0, "wfb_hit_event_table: rows without events");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (offsets_dev) WFB_CUDA(cudaMemsetAsync(offsets_dev, 0, 8, st));
    if (n == 0) return WFB_OK;
    WFB_REQUIRE(order_dev && event_id_dev && board_dev && channel_dev && dt_dev && abs_start_dev && abs_end_dev && offsets_dev &&
                    members_dev && t_min_dev && t_max_dev && dt_ns_dev && n_hits_dev && workspace_dev,
                "wfb_hit_event_table: NULL pointer");
    WFB_REQUIRE((rows_dev == nullptr) == (member_rows_dev == nullptr), "wfb_hit_event_table: rows need both the input and the output");
    WFB_REQUIRE(rows_dev == nullptr || row_bytes == kHitRowBytes || row_bytes == 72, "wfb_hit_event_table: row_bytes must be 60 or 72");
    WFB_REQUIRE(((uintptr_t)rows_dev & 3) == 0 && ((uintptr_t)member_rows_dev & 3) == 0, "wfb_hit_event_table: rows must be 4-byte aligned");
    WFB_REQUIRE(workspace_bytes >= wfb_hit_event_table_workspace_bytes(n), "wfb_hit_event_table: workspace too small");
    uint8_t* ws = static_cast<uint8_t*>(workspace_dev);
    const size_t m = ht_al((size_t)n * 8);
    long long* flag = reinterpret_cast<long long*>(ws);
    long long* incl = reinterpret_cast<long long*>(ws + m);
    unsigned long long* kA = reinterpret_cast<unsigned long long*>(ws + 2 * m);
    long long* vA = reinterpret_cast<long long*>(ws + 3 * m);
    unsigned long long* kB = reinterpret_cast<unsigned long long*>(ws + 4 * m);
    long long* vB = reinterpret_cast<long long*>(ws + 5 * m);
    // the running maximum's pairs (16 B each) live in kA..vA and kB..vB: they are read before the big path sorts there
    SegMax* sm_in = reinterpret_cast<SegMax*>(kA);
    SegMax* sm_out = reinterpret_cast<SegMax*>(kB);
    uint8_t* sws = ws + 6 * m;
    const size_t sort_bytes = radix_sort_workspace_bytes(n);
    void* scan_ws = sws + ht_al(sort_bytes);
    unsigned long long* d_big =
        reinterpret_cast<unsigned long long*>(static_cast<uint8_t*>(scan_ws) + 2 * ht_al(scan_workspace_bytes(n)));

    const HtIn in{reinterpret_cast<const long long*>(order_dev), reinterpret_cast<const long long*>(event_id_dev), board_dev, channel_dev,
                  dt_dev, abs_start_dev, abs_end_dev, static_cast<const uint8_t*>(rows_dev), row_bytes / 4};
    const HtOut o{reinterpret_cast<long long*>(members_dev), static_cast<uint8_t*>(member_rows_dev)};
    long long* offsets = reinterpret_cast<long long*>(offsets_dev);

    ht_offsets_kernel<<<ht_nb(n), 256, 0, st>>>(in, n, n_events, offsets, sm_in);
    int rc = inclusive_scan_segmax(sm_in, sm_out, n, scan_ws, st);
    if (rc != WFB_OK) return rc;
    ht_stats_kernel<<<ht_nb(n_events), 256, 0, st>>>(in, offsets, sm_out, n_events, reinterpret_cast<long long*>(t_min_dev),
                                                     reinterpret_cast<long long*>(t_max_dev), dt_ns_dev,
                                                     reinterpret_cast<long long*>(n_hits_dev));
    WFB_CUDA(cudaMemsetAsync(d_big, 0, 8, st));
    ht_small_kernel<<<ht_nb(n_events * 32), 256, 0, st>>>(in, offsets, n_events, o, d_big);
    WFB_CUDA(cudaGetLastError());
    unsigned long long n_big = 0;
    WFB_CUDA(cudaMemcpyAsync(&n_big, d_big, 8, cudaMemcpyDeviceToHost, st));
    WFB_CUDA(cudaStreamSynchronize(st));
    if (n_big > 0) {
        ht_big_flags_kernel<<<ht_nb(n), 256, 0, st>>>(in, offsets, n, flag);
        rc = inclusive_scan_sum_i64(flag, incl, n, scan_ws, st);
        if (rc != WFB_OK) return rc;
        ht_big_keys_kernel<<<ht_nb(n), 256, 0, st>>>(in, flag, incl, n, kA, vA);
        rc = radix_sort_pairs(kA, vA, kB, vB, (long long)n_big, kKeyUnsigned, sws, sort_bytes, st);
        if (rc != WFB_OK) return rc;
        ht_big_event_keys_kernel<<<ht_nb((long long)n_big), 256, 0, st>>>(in, vB, (long long)n_big, kA);
        rc = radix_sort_pairs(kA, vB, kB, vA, (long long)n_big, kKeyUnsigned, sws, sort_bytes, st);
        if (rc != WFB_OK) return rc;
        ht_big_scatter_kernel<<<ht_nb((long long)n_big), 256, 0, st>>>(in, kB, vA, (long long)n_big, offsets, incl, o);
        WFB_CUDA(cudaGetLastError());
    }
    return WFB_OK;
}
