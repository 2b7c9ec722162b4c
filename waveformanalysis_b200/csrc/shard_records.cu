// Time shards of a V1725 run built on several GPUs: split points of locally sorted RECORDS rows and the merge of the
// sorted runs a rank receives from every rank (distributed.build_records_sharded_v1725).
//
// A run's global order is lexsort((seq, channel, board, pid = 0, timestamp)) over all files, seq = the waveform's index
// in the concatenation of all files (v1725.cu).  Every rank builds the rows of its own files with record_id = seq, so
// the key (timestamp, board, channel, record_id) is unique and read straight from the packed rows; key_less below is
// the one device definition of that order.
//
// The merge places record k of run r at k + (records of the other runs with a smaller key), each count one binary
// search in that run's keys; a stable radix sort of the received order would order equal (timestamp, board, channel)
// by source rank instead of by seq.  One warp per output record then copies the row (record_id and wave_offset
// renumbered for the shard's place in the run) and the samples, as v1725_gather_kernel does.
#include <algorithm>

#include "common.cuh"
#include "sort_scan.cuh"

namespace wfb {

struct RecKey {
    long long ts;
    long long id;
    unsigned bc;  // (board, channel) as one unsigned: board in the high half, both offset by 32768
};

__device__ __forceinline__ unsigned board_channel(int board, int channel) {
    return ((unsigned)(board + 32768) << 16) | (unsigned)(channel + 32768);
}

__device__ __forceinline__ RecKey row_key(const uint16_t* h) {  // timestamp@0, board@12, channel@14, record_id@64
    return RecKey{(long long)rd64(h), (long long)rd64(h + 32), board_channel((short)h[6], (short)h[7])};
}

__device__ __forceinline__ bool key_less(const RecKey& a, const RecKey& b) {
    if (a.ts != b.ts) return a.ts < b.ts;
    if (a.bc != b.bc) return a.bc < b.bc;
    return a.id < b.id;
}

// the run holding index i (runs may be empty): the last r with run_off[r] <= i
__device__ __forceinline__ int run_of(const long long* run_off, int n_runs, long long i) {
    int lo = 0, hi = n_runs;  // run_off[0] = 0 <= i < run_off[n_runs]
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (run_off[mid] <= i) lo = mid;
        else hi = mid;
    }
    return lo;
}

__global__ void split_points_kernel(const uint16_t* __restrict__ rows, long long n, const long long* __restrict__ keys, long long n_keys,
                                    long long* __restrict__ out) {
    const long long j = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (j >= n_keys) return;
    const long long* k = keys + 4 * j;
    const RecKey key{k[0], k[3], board_channel((int)k[1], (int)k[2])};
    long long lo = 0, hi = n;
    while (lo < hi) {
        const long long mid = (lo + hi) >> 1;
        if (key_less(row_key(rows + mid * (kRecordsRowBytes / 2)), key)) lo = mid + 1;
        else hi = mid;
    }
    out[j] = lo;
}

// compact keys + lengths; flag bit 0: a run is not strictly increasing, bit 1: a negative event_length
__global__ void merge_keys_kernel(const uint16_t* __restrict__ rows, long long n, const long long* __restrict__ run_off, int n_runs,
                                  RecKey* __restrict__ keys, long long* __restrict__ len, int* __restrict__ flag) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint16_t* h = rows + i * (kRecordsRowBytes / 2);
    const RecKey k = row_key(h);
    keys[i] = k;
    const int l = (int)rd32(h + 45);
    len[i] = l;
    int bad = l < 0 ? 2 : 0;
    if (run_off[run_of(run_off, n_runs, i)] != i && !key_less(row_key(h - kRecordsRowBytes / 2), k)) bad |= 1;
    if (bad) atomicOr(flag, bad);
}

// merge-by-rank: output position of every input record
__global__ void merge_rank_kernel(const RecKey* __restrict__ keys, long long n, const long long* __restrict__ run_off, int n_runs,
                                  const long long* __restrict__ len_in, long long* __restrict__ src_of, long long* __restrict__ len_out) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int r = run_of(run_off, n_runs, i);
    const RecKey k = keys[i];
    long long pos = i - run_off[r];
    for (int q = 0; q < n_runs; ++q) {
        if (q == r) continue;
        // equal keys (not produced by a valid build) still get distinct places: earlier runs first
        const bool upper = q < r;
        long long lo = run_off[q], hi = run_off[q + 1];
        const long long base = lo;
        while (lo < hi) {
            const long long mid = (lo + hi) >> 1;
            const bool before = upper ? !key_less(k, keys[mid]) : key_less(keys[mid], k);
            if (before) lo = mid + 1;
            else hi = mid;
        }
        pos += lo - base;
    }
    src_of[pos] = i;
    len_out[pos] = len_in[i];
}

// one warp per OUTPUT record: row with record_id / wave_offset renumbered, samples, wfb_rec_meta
__global__ void __launch_bounds__(256) merge_gather_kernel(const uint16_t* __restrict__ rows_in, const uint16_t* __restrict__ pool_in,
                                                           const long long* __restrict__ in_incl, const long long* __restrict__ src_of,
                                                           const long long* __restrict__ len_out, const long long* __restrict__ out_incl,
                                                           long long n, long long record_base, long long pool_base,
                                                           uint16_t* __restrict__ rows_out, uint16_t* __restrict__ pool_out,
                                                           wfb_rec_meta* __restrict__ meta_out) {
    const int lane = lane_id();
    const long long j = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
    if (j >= n) return;
    const long long src = src_of[j];
    const long long len = len_out[j];
    const long long out_off = out_incl[j] - len;
    const uint16_t* in = pool_in + (in_incl[src] - len);
    uint16_t* out = pool_out + out_off;
    for (long long t = lane; t < len; t += 32) out[t] = in[t];
    const long long rid = record_base + j, wo = pool_base + out_off;
    const uint16_t* h = rows_in + src * (kRecordsRowBytes / 2);
    uint16_t* o = rows_out + j * (kRecordsRowBytes / 2);
    for (int k = lane; k < kRecordsRowBytes / 2; k += 32) {
        uint16_t v = h[k];
        if (k >= 32 && k < 36) v = (uint16_t)((unsigned long long)rid >> (16 * (k - 32)));
        else if (k >= 41 && k < 45) v = (uint16_t)((unsigned long long)wo >> (16 * (k - 41)));
        o[k] = v;
    }
    if (lane == 0) {
        wfb_rec_meta m = rec_meta_from_row(h);
        m.record_id = rid;
        m.wave_offset = wo;
        meta_out[j] = m;
    }
}

}  // namespace wfb

using namespace wfb;

static unsigned s_nb(long long n, int t = 256) { return (unsigned)((n + t - 1) / t); }
static size_t s_al256(size_t x) { return (x + 255) & ~(size_t)255; }

extern "C" int wfb_record_split_points(const void* rows_dev, int64_t n, const int64_t* keys_dev, int64_t n_keys, int64_t* out_dev,
                                       void* stream) {
    WFB_REQUIRE(n >= 0 && n_keys >= 0, "wfb_record_split_points: negative size");
    if (n_keys == 0) return WFB_OK;
    WFB_REQUIRE(keys_dev && out_dev && (n == 0 || rows_dev), "wfb_record_split_points: NULL pointer");
    WFB_REQUIRE(((uintptr_t)rows_dev & 1) == 0, "wfb_record_split_points: rows must be 2-byte aligned");
    split_points_kernel<<<s_nb(n_keys), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        static_cast<const uint16_t*>(rows_dev), n, reinterpret_cast<const long long*>(keys_dev), n_keys, reinterpret_cast<long long*>(out_dev));
    WFB_CUDA(cudaGetLastError());
    return WFB_OK;
}

extern "C" size_t wfb_merge_record_runs_workspace_bytes(int64_t n, int64_t n_runs) {
    const size_t m = s_al256((size_t)std::max<int64_t>(n, 1) * 8);
    return s_al256((size_t)std::max<int64_t>(n, 1) * sizeof(RecKey)) + 5 * m + s_al256((size_t)(std::max<int64_t>(n_runs, 0) + 1) * 8) + 256 +
           scan_workspace_bytes(n);
}

extern "C" int wfb_merge_record_runs(const void* rows_in_dev, const uint16_t* pool_in_dev, int64_t n_in, const int64_t* run_offsets_host,
                                     int64_t n_runs, int64_t record_base, int64_t pool_base, void* rows_out_dev, uint16_t* pool_out_dev,
                                     int64_t pool_len, wfb_rec_meta* meta_out_dev, void* workspace_dev, size_t workspace_bytes, void* stream) {
    const char* who = "wfb_merge_record_runs";
    WFB_REQUIRE(n_in >= 0 && pool_len >= 0 && n_runs >= 1 && n_runs < (1 << 20), "%s: bad sizes", who);
    WFB_REQUIRE(run_offsets_host != nullptr && run_offsets_host[0] == 0 && run_offsets_host[n_runs] == n_in, "%s: bad run offsets", who);
    for (int64_t r = 0; r < n_runs; ++r) WFB_REQUIRE(run_offsets_host[r] <= run_offsets_host[r + 1], "%s: run offsets decrease", who);
    if (n_in == 0) {
        WFB_REQUIRE(pool_len == 0, "%s: samples without records", who);
        return WFB_OK;
    }
    WFB_REQUIRE(rows_in_dev && rows_out_dev && meta_out_dev && workspace_dev && (pool_len == 0 || (pool_in_dev && pool_out_dev)),
                "%s: NULL pointer", who);
    WFB_REQUIRE((((uintptr_t)rows_in_dev | (uintptr_t)rows_out_dev | (uintptr_t)pool_in_dev | (uintptr_t)pool_out_dev) & 1) == 0,
                "%s: rows and samples must be 2-byte aligned", who);
    WFB_REQUIRE(((uintptr_t)meta_out_dev & 15) == 0, "%s: meta must be 16-byte aligned", who);
    WFB_REQUIRE(workspace_bytes >= wfb_merge_record_runs_workspace_bytes(n_in, n_runs), "%s: workspace too small", who);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const long long n = n_in;
    uint8_t* ws = static_cast<uint8_t*>(workspace_dev);
    const size_t m = s_al256((size_t)n * 8);
    RecKey* keys = reinterpret_cast<RecKey*>(ws);
    ws += s_al256((size_t)n * sizeof(RecKey));
    long long* len_in = reinterpret_cast<long long*>(ws);
    long long* in_incl = reinterpret_cast<long long*>(ws + m);
    long long* src_of = reinterpret_cast<long long*>(ws + 2 * m);
    long long* len_out = reinterpret_cast<long long*>(ws + 3 * m);
    long long* out_incl = reinterpret_cast<long long*>(ws + 4 * m);
    ws += 5 * m;
    long long* run_off = reinterpret_cast<long long*>(ws);
    ws += s_al256((size_t)(n_runs + 1) * 8);
    int* flag = reinterpret_cast<int*>(ws);
    void* scan_ws = ws + 256;
    const int runs = (int)n_runs;

    WFB_CUDA(cudaMemcpyAsync(run_off, run_offsets_host, (size_t)(n_runs + 1) * 8, cudaMemcpyHostToDevice, st));
    WFB_CUDA(cudaMemsetAsync(flag, 0, sizeof(int), st));
    merge_keys_kernel<<<s_nb(n), 256, 0, st>>>(static_cast<const uint16_t*>(rows_in_dev), n, run_off, runs, keys, len_in, flag);
    WFB_CUDA(cudaGetLastError());
    int rc = inclusive_scan_sum_i64(len_in, in_incl, n, scan_ws, st);
    if (rc != WFB_OK) return rc;
    // the positions are a permutation only for strictly increasing runs: check before anything is scattered
    int h_flag = 0;
    long long h_total = 0;
    WFB_CUDA(cudaMemcpyAsync(&h_flag, flag, sizeof(int), cudaMemcpyDeviceToHost, st));
    WFB_CUDA(cudaMemcpyAsync(&h_total, in_incl + (n - 1), sizeof(long long), cudaMemcpyDeviceToHost, st));
    WFB_CUDA(cudaStreamSynchronize(st));
    WFB_REQUIRE(!(h_flag & 1), "%s: a run is not strictly increasing in (timestamp, board, channel, record_id)", who);
    WFB_REQUIRE(!(h_flag & 2), "%s: negative event_length", who);
    WFB_REQUIRE(h_total == pool_len, "%s: the records hold %lld samples, pool_len is %lld", who, h_total, (long long)pool_len);

    merge_rank_kernel<<<s_nb(n), 256, 0, st>>>(keys, n, run_off, runs, len_in, src_of, len_out);
    WFB_CUDA(cudaGetLastError());
    rc = inclusive_scan_sum_i64(len_out, out_incl, n, scan_ws, st);
    if (rc != WFB_OK) return rc;
    merge_gather_kernel<<<s_nb(n * 32), 256, 0, st>>>(static_cast<const uint16_t*>(rows_in_dev), pool_in_dev, in_incl, src_of, len_out,
                                                       out_incl, n, record_base, pool_base, static_cast<uint16_t*>(rows_out_dev),
                                                       pool_out_dev, meta_out_dev);
    WFB_CUDA(cudaGetLastError());
    return WFB_OK;
}
