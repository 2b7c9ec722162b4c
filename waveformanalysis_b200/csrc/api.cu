// C-ABI plumbing: errors, device info, RECORDS_DTYPE unpack, the host-buffer pipeline.
#include <limits.h>
#include <stdarg.h>

#include <algorithm>
#include <mutex>
#include <thread>
#include <vector>

#include "common.cuh"

namespace wfb {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int cuda_fail(cudaError_t e, const char* what) {
    set_error("CUDA error %d (%s) in %s", (int)e, cudaGetErrorString(e), what);
    return WFB_ERR_CUDA;
}

int sm_count() {
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 148;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) return 148;
    return n;
}

__global__ void records_unpack_kernel(const uint16_t* __restrict__ rows, long long n, wfb_rec_meta* __restrict__ meta) {
    long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= n) return;
    meta[i] = rec_meta_from_row(rows + i * (kRecordsRowBytes / 2));
}

// keeps the first non-zero error flag of the chunks of one wfb_process_host call (the per-call flag in the workspace
// is cleared by the next chunk that uses the slot)
__global__ void err_accumulate_kernel(const int* __restrict__ chunk_flag, int* __restrict__ run_flag) {
    if (*chunk_flag != 0 && *run_flag == 0) *run_flag = *chunk_flag;
}

__global__ void meta_stats_kernel(const wfb_rec_meta* __restrict__ meta, long long n, int* __restrict__ out) {
    int mx_len = 0, mn_dt = INT_MAX, mx_dt = INT_MIN;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        mx_len = max(mx_len, meta[i].event_length);
        mn_dt = min(mn_dt, meta[i].dt);
        mx_dt = max(mx_dt, meta[i].dt);
    }
    mx_len = __reduce_max_sync(kFull, mx_len);
    mn_dt = __reduce_min_sync(kFull, mn_dt);
    mx_dt = __reduce_max_sync(kFull, mx_dt);
    if (lane_id() == 0) {
        atomicMax(out + 0, mx_len);
        atomicMin(out + 1, mn_dt);
        atomicMax(out + 2, mx_dt);
    }
}

__global__ void meta_set_clamp_kernel(wfb_rec_meta* __restrict__ meta, long long n, const int* __restrict__ clamp) {
    long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int c = clamp ? clamp[i] : -1;
    const unsigned enc = (c >= 0) ? (unsigned)min(c, (1 << 24) - 2) + 1u : 0u;
    meta[i].pad_[0] = (uint8_t)(enc & 0xff);
    meta[i].pad_[1] = (uint8_t)((enc >> 8) & 0xff);
    meta[i].pad_[2] = (uint8_t)((enc >> 16) & 0xff);
}

}  // namespace wfb

using namespace wfb;

extern "C" int wfb_meta_stats(const wfb_rec_meta* meta_dev, int64_t n, int32_t* scratch_dev, int32_t* out_host, void* stream) {
    WFB_REQUIRE(n >= 0 && out_host != nullptr, "wfb_meta_stats: bad arguments");
    out_host[0] = 0;
    out_host[1] = INT_MAX;
    out_host[2] = INT_MIN;
    if (n == 0) return WFB_OK;
    WFB_REQUIRE(meta_dev && scratch_dev, "wfb_meta_stats: NULL pointer");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    WFB_CUDA(cudaMemcpyAsync(scratch_dev, out_host, 12, cudaMemcpyHostToDevice, st));
    meta_stats_kernel<<<(unsigned)std::min<long long>(2048, (n + 255) / 256), 256, 0, st>>>(meta_dev, n, scratch_dev);
    WFB_CUDA(cudaGetLastError());
    WFB_CUDA(cudaMemcpyAsync(out_host, scratch_dev, 12, cudaMemcpyDeviceToHost, st));
    WFB_CUDA(cudaStreamSynchronize(st));
    return WFB_OK;
}

extern "C" int wfb_meta_set_clamp(wfb_rec_meta* meta_dev, int64_t n, const int32_t* clamp_len_dev, void* stream) {
    WFB_REQUIRE(n >= 0, "wfb_meta_set_clamp: negative n");
    if (n == 0) return WFB_OK;
    WFB_REQUIRE(meta_dev != nullptr, "wfb_meta_set_clamp: NULL meta");
    meta_set_clamp_kernel<<<(unsigned)((n + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(meta_dev, n, clamp_len_dev);
    WFB_CUDA(cudaGetLastError());
    return WFB_OK;
}

static int staged_upload(void* dst_dev, const void* src_host, size_t bytes, cudaStream_t st);  // (below: needs the device's stager)

extern "C" int wfb_memcpy_h2d(void* dst_dev, const void* src_host, size_t bytes, void* stream) {
    if (bytes == 0) return WFB_OK;
    WFB_REQUIRE(dst_dev && src_host, "wfb_memcpy_h2d: NULL pointer");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    int rc = staged_upload(dst_dev, src_host, bytes, st);
    if (rc != WFB_OK) return rc;
    WFB_CUDA(cudaStreamSynchronize(st));  // pageable / memory-mapped sources: the caller may drop the array right away
    return WFB_OK;
}

extern "C" int wfb_memcpy_h2d_async(void* dst_dev, const void* src_host, size_t bytes, void* stream) {
    if (bytes == 0) return WFB_OK;
    WFB_REQUIRE(dst_dev && src_host, "wfb_memcpy_h2d_async: NULL pointer");
    WFB_CUDA(cudaMemcpyAsync(dst_dev, src_host, bytes, cudaMemcpyHostToDevice, static_cast<cudaStream_t>(stream)));
    return WFB_OK;
}

extern "C" const char* wfb_last_error(void) { return g_err; }
extern "C" int wfb_version(void) { return 100; }

extern "C" int wfb_device_info(int* sm, int* cc_major, int* cc_minor, char* name, int name_len) {
    int dev = 0;
    WFB_CUDA(cudaGetDevice(&dev));
    cudaDeviceProp prop;
    WFB_CUDA(cudaGetDeviceProperties(&prop, dev));
    if (sm) *sm = prop.multiProcessorCount;
    if (cc_major) *cc_major = prop.major;
    if (cc_minor) *cc_minor = prop.minor;
    if (name && name_len > 0) {
        strncpy(name, prop.name, name_len - 1);
        name[name_len - 1] = 0;
    }
    return WFB_OK;
}

extern "C" int wfb_records_unpack(const void* records_aos_dev, int64_t n, wfb_rec_meta* meta_dev, void* stream) {
    WFB_REQUIRE(n >= 0, "wfb_records_unpack: negative n");
    if (n == 0) return WFB_OK;
    WFB_REQUIRE(records_aos_dev && meta_dev, "wfb_records_unpack: NULL pointer");
    WFB_REQUIRE(((uintptr_t)records_aos_dev & 1) == 0, "wfb_records_unpack: records must be 2-byte aligned");
    WFB_REQUIRE(((uintptr_t)meta_dev & 15) == 0, "wfb_records_unpack: meta_dev must be 16-byte aligned");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    records_unpack_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(static_cast<const uint16_t*>(records_aos_dev), n, meta_dev);
    WFB_CUDA(cudaGetLastError());
    return WFB_OK;
}

// ---- host-buffer pipeline -----------------------------------------------------------------------
// Chunked over records: H2D (copy stream) -> unpack + fused kernel (compute stream) -> D2H of
// the feature rows; hit rows accumulate in one device buffer and are copied back at the end.
namespace {

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    int ensure(size_t bytes) {
        if (bytes <= cap) return WFB_OK;
        release();
        // grow with some slack so that runs of slightly different size reuse the buffer
        const size_t want = bytes + bytes / 8;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) {
            (void)cudaGetLastError();
            e = cudaMalloc(&p, bytes);
            if (e != cudaSuccess) {
                p = nullptr;
                set_error("cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e));
                return WFB_ERR_NOMEM;
            }
            cap = bytes;
            return WFB_OK;
        }
        cap = want;
        return WFB_OK;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
};

struct Slot {
    DevBuf pool, rows, meta, feat, counts, ws;
    cudaEvent_t copied = nullptr, computed = nullptr, drained = nullptr;
};

constexpr int kSlots = 3;
constexpr int kMaxDevices = 64;

// Streams, events and device buffers of wfb_process_host, kept between calls (one set per device,
// calls on the same device are serialised by the mutex).  wfb_release_cache() frees them; they
// are deliberately not freed at process exit (the CUDA context may already be gone).
// Pageable (or memory-mapped) host sources - what a Context hands to a plugin - would be staged by the driver on one
// thread at ~10 GB/s.  The stager copies them into a small ring of pinned pieces with a few threads and sends every piece
// by DMA as soon as it is full, so the upload runs at the speed the host can read its own memory.
constexpr int kStagePieces = 4;
constexpr size_t kStagePieceBytes = 32u << 20;
struct Stager {
    uint8_t* buf[kStagePieces] = {nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t sent[kStagePieces] = {nullptr, nullptr, nullptr, nullptr};
    int next = 0;
    bool ready = false;
    int init() {
        if (ready) return WFB_OK;
        for (int k = 0; k < kStagePieces; ++k) {
            WFB_CUDA(cudaHostAlloc(reinterpret_cast<void**>(&buf[k]), kStagePieceBytes, cudaHostAllocDefault));
            WFB_CUDA(cudaEventCreateWithFlags(&sent[k], cudaEventDisableTiming));
        }
        ready = true;
        return WFB_OK;
    }
    void release() {
        for (int k = 0; k < kStagePieces; ++k) {
            if (buf[k]) cudaFreeHost(buf[k]);
            if (sent[k]) cudaEventDestroy(sent[k]);
            buf[k] = nullptr;
            sent[k] = nullptr;
        }
        ready = false;
    }
};

bool host_pointer_is_pinned(const void* p) {
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return attr.type == cudaMemoryTypeHost || attr.type == cudaMemoryTypeManaged;
}

void parallel_memcpy(uint8_t* dst, const uint8_t* src, size_t bytes) {
    const int nt = (int)std::max<size_t>(1, std::min<size_t>(4, bytes >> 22));  // one thread per 4 MB, at most four
    if (nt == 1) {
        memcpy(dst, src, bytes);
        return;
    }
    std::vector<std::thread> th;
    const size_t per = ((bytes / nt) + 63) & ~(size_t)63;
    for (int t = 1; t < nt; ++t) {
        const size_t lo = std::min(bytes, per * t), hi = (t == nt - 1) ? bytes : std::min(bytes, per * (t + 1));
        th.emplace_back([=]() { memcpy(dst + lo, src + lo, hi - lo); });
    }
    memcpy(dst, src, std::min(bytes, per));
    for (auto& x : th) x.join();
}

// host -> device on `st`; the source may be released when the call returns unless it is pinned (then: after the stream
// has passed the copy, as with cudaMemcpyAsync)
int staged_h2d(Stager& sg, void* dst_dev, const void* src_host, size_t bytes, cudaStream_t st, bool src_pinned) {
    if (bytes == 0) return WFB_OK;
    static const bool off = [] { const char* e = getenv("WFB_STAGED_H2D"); return e && e[0] == '0'; }();
    if (src_pinned || off || bytes < (1u << 20)) {
        WFB_CUDA(cudaMemcpyAsync(dst_dev, src_host, bytes, cudaMemcpyHostToDevice, st));
        return WFB_OK;
    }
    int rc = sg.init();
    if (rc != WFB_OK) return rc;
    const uint8_t* src = static_cast<const uint8_t*>(src_host);
    uint8_t* dst = static_cast<uint8_t*>(dst_dev);
    for (size_t o = 0; o < bytes; o += kStagePieceBytes) {
        const size_t len = std::min(kStagePieceBytes, bytes - o);
        const int k = sg.next;
        sg.next = (sg.next + 1) % kStagePieces;
        WFB_CUDA(cudaEventSynchronize(sg.sent[k]));  // the piece's previous content has left
        parallel_memcpy(sg.buf[k], src + o, len);
        WFB_CUDA(cudaMemcpyAsync(dst + o, sg.buf[k], len, cudaMemcpyHostToDevice, st));
        WFB_CUDA(cudaEventRecord(sg.sent[k], st));
    }
    return WFB_OK;
}

struct HostPipe {
    std::mutex mu;
    bool ready = false;
    Stager stager;
    cudaStream_t s_copy = nullptr, s_comp = nullptr, s_out = nullptr;
    Slot slots[kSlots];
    DevBuf d_hits, d_rules, d_tot;
    long long* mailbox = nullptr;  // pinned: the running hit total after each chunk
    void release_buffers() {
        for (auto& s : slots) {
            s.pool.release(); s.rows.release(); s.meta.release(); s.feat.release(); s.counts.release(); s.ws.release();
        }
        d_hits.release(); d_rules.release(); d_tot.release();
        stager.release();
    }
};
HostPipe* g_pipes[kMaxDevices];
std::mutex g_pipes_mu;

HostPipe* host_pipe(int device) {
    std::lock_guard<std::mutex> lock(g_pipes_mu);
    if (device < 0 || device >= kMaxDevices) return nullptr;
    if (!g_pipes[device]) g_pipes[device] = new HostPipe();
    return g_pipes[device];
}

inline long long rec_i64(const uint8_t* row, int off) {
    long long v;
    memcpy(&v, row + off, 8);
    return v;
}
inline int rec_i32(const uint8_t* row, int off) {
    int v;
    memcpy(&v, row + off, 4);
    return v;
}

}  // namespace

static int staged_upload(void* dst_dev, const void* src_host, size_t bytes, cudaStream_t st) {
    const bool pinned = host_pointer_is_pinned(src_host);
    if (pinned || bytes < (4u << 20)) {
        WFB_CUDA(cudaMemcpyAsync(dst_dev, src_host, bytes, cudaMemcpyHostToDevice, st));
        return WFB_OK;
    }
    int device = 0;
    WFB_CUDA(cudaGetDevice(&device));
    HostPipe* hp = host_pipe(device);
    if (hp == nullptr) {
        WFB_CUDA(cudaMemcpyAsync(dst_dev, src_host, bytes, cudaMemcpyHostToDevice, st));
        return WFB_OK;
    }
    std::lock_guard<std::mutex> pipe_lock(hp->mu);
    return staged_h2d(hp->stager, dst_dev, src_host, bytes, st, false);
}

// pool_keep / meta_keep: device buffers for the WHOLE pool (pool_len elements, 16-byte aligned, readable to the next
// 16-byte boundary) and the records' metadata (n rows): every chunk is uploaded / unpacked straight into its place there
// instead of into the pipeline's slot buffers, so the run is resident in HBM when the call returns.
static int process_host_impl(const void* records_host, int64_t n, const void* pool_host, int64_t pool_len,
                             const wfb_fh_params* params, const wfb_chan_rule* rules_host, void* feat_out_host,
                             void* hit_out_host, int64_t hit_cap, int32_t* hit_counts_host, int64_t* n_hits,
                             int64_t chunk_records, void* pool_keep, wfb_rec_meta* meta_keep) {
    WFB_REQUIRE(params != nullptr && n_hits != nullptr, "wfb_process_host: NULL params / n_hits");
    WFB_REQUIRE(n >= 0 && pool_len >= 0 && hit_cap >= 0, "wfb_process_host: negative size");
    *n_hits = 0;
    if (n == 0) return WFB_OK;
    WFB_REQUIRE(records_host && pool_host, "wfb_process_host: NULL input");
    const int flags = params->flags;
    const bool do_feat = flags & WFB_DO_FEATURES, do_hits = flags & WFB_DO_HITS;
    WFB_REQUIRE(do_feat || do_hits, "wfb_process_host: flags select nothing");
    WFB_REQUIRE(!do_feat || feat_out_host, "wfb_process_host: feat_out_host is NULL");
    WFB_REQUIRE(!do_hits || hit_cap == 0 || hit_out_host, "wfb_process_host: hit_out_host is NULL");
    const size_t esz = params->pool_is_f32 ? 4 : 2;
    const uint8_t* rows = static_cast<const uint8_t*>(records_host);
    const uint8_t* pool = static_cast<const uint8_t*>(pool_host);
    if (chunk_records <= 0) chunk_records = 1 << 18;
    chunk_records = std::min<int64_t>(chunk_records, n);

    // padded matrix width = max event_length over the whole run (hit_finder.py:364)
    // (also without hits: a per-chunk maximum would cost a device round trip per chunk and make the kernel variant
    // depend on the chunk)
    int lmax = params->lmax;
    if (lmax <= 0) {  // strided read of 4 of every 102 bytes: a few threads hide the cache misses
        const int nt = (int)std::max<int64_t>(1, std::min<int64_t>(8, n >> 16));
        std::vector<int> part(nt, 0);
        auto scan = [&](int t) {
            int mx = 0;
            for (int64_t i = n * t / nt, e = n * (t + 1) / nt; i < e; ++i) mx = std::max(mx, rec_i32(rows + i * kRecordsRowBytes, 90));
            part[t] = mx;
        };
        std::vector<std::thread> th;
        for (int t = 1; t < nt; ++t) th.emplace_back(scan, t);
        scan(0);
        for (auto& x : th) x.join();
        for (int v : part) lmax = std::max(lmax, v);
    }
    bool scan_all = false;

    int device = 0;
    WFB_CUDA(cudaGetDevice(&device));
    HostPipe* hp = host_pipe(device);
    WFB_REQUIRE(hp != nullptr, "wfb_process_host: device index %d out of range", device);
    std::lock_guard<std::mutex> pipe_lock(hp->mu);
    int rc = WFB_OK;
    if (!hp->ready) {
        WFB_CUDA(cudaStreamCreateWithFlags(&hp->s_copy, cudaStreamNonBlocking));
        WFB_CUDA(cudaStreamCreateWithFlags(&hp->s_comp, cudaStreamNonBlocking));
        WFB_CUDA(cudaStreamCreateWithFlags(&hp->s_out, cudaStreamNonBlocking));
        for (auto& s : hp->slots) {
            WFB_CUDA(cudaEventCreateWithFlags(&s.copied, cudaEventDisableTiming));
            WFB_CUDA(cudaEventCreateWithFlags(&s.computed, cudaEventDisableTiming));
            WFB_CUDA(cudaEventCreateWithFlags(&s.drained, cudaEventDisableTiming));
        }
        WFB_CUDA(cudaHostAlloc(reinterpret_cast<void**>(&hp->mailbox), sizeof(long long) * kSlots, cudaHostAllocDefault));
        hp->ready = true;
    }
    cudaStream_t s_copy = hp->s_copy, s_comp = hp->s_comp, s_out = hp->s_out;
    Slot* slots = hp->slots;
    const bool pool_pinned = pool_len == 0 || host_pointer_is_pinned(pool_host);
    const bool rows_pinned = n == 0 || host_pointer_is_pinned(records_host);
    DevBuf &d_hits = hp->d_hits, &d_rules = hp->d_rules, &d_tot = hp->d_tot;
    auto cleanup = [&]() {  // leave the pipeline idle: nothing of this call is still in flight
        cudaStreamSynchronize(s_copy);
        cudaStreamSynchronize(s_comp);
        cudaStreamSynchronize(s_out);
    };
#define PH_CHECK(expr)                \
    do {                              \
        rc = (expr);                  \
        if (rc != WFB_OK) {           \
            cleanup();                \
            return rc;                \
        }                             \
    } while (0)
#define PH_CUDA(call)                                   \
    do {                                                \
        cudaError_t e__ = (call);                       \
        if (e__ != cudaSuccess) {                       \
            rc = cuda_fail(e__, #call);                 \
            cleanup();                                  \
            return rc;                                  \
        }                                               \
    } while (0)

again:
    if (do_hits) PH_CHECK(d_hits.ensure(std::max<size_t>((size_t)hit_cap * kHitRowBytes, 64)));
    PH_CHECK(d_tot.ensure(64));  // ping-pong running totals (bytes 0..15) and the run-wide error flag (byte 32)
    PH_CUDA(cudaMemsetAsync(d_tot.p, 0, 64, s_comp));
    int* const run_err = reinterpret_cast<int*>(static_cast<uint8_t*>(d_tot.p) + 32);
    wfb_fh_params p = *params;
    p.lmax = lmax;
    p.rules_dev = nullptr;
    if (p.n_rules > 0) {
        WFB_REQUIRE(rules_host != nullptr, "wfb_process_host: n_rules > 0 but rules_host is NULL");
        PH_CHECK(d_rules.ensure(sizeof(wfb_chan_rule) * p.n_rules));
        PH_CUDA(cudaMemcpyAsync(d_rules.p, rules_host, sizeof(wfb_chan_rule) * p.n_rules, cudaMemcpyHostToDevice, s_comp));
        p.rules_dev = static_cast<const wfb_chan_rule*>(d_rules.p);
    }

    // hit rows leave the device two chunks behind the compute stream: the running total of chunk j is
    // read from the pinned mailbox once its event has fired, then the new rows are copied on s_out
    long long hits_copied = 0;
    auto drain_hits = [&](int64_t j) -> int {
        Slot& sj = slots[j % kSlots];
        cudaError_t e = cudaEventSynchronize(sj.computed);
        if (e != cudaSuccess) return cuda_fail(e, "cudaEventSynchronize");
        const long long upto = std::min<long long>(hp->mailbox[j % kSlots], hit_cap);
        if (upto > hits_copied) {
            e = cudaStreamWaitEvent(s_out, sj.computed, 0);
            if (e == cudaSuccess)
                e = cudaMemcpyAsync(static_cast<uint8_t*>(hit_out_host) + (size_t)hits_copied * kHitRowBytes,
                                    static_cast<uint8_t*>(d_hits.p) + (size_t)hits_copied * kHitRowBytes,
                                    (size_t)(upto - hits_copied) * kHitRowBytes, cudaMemcpyDeviceToHost, s_out);
            if (e != cudaSuccess) return cuda_fail(e, "hit rows D2H");
            hits_copied = upto;
        }
        return WFB_OK;
    };

    // resident mode uploads EVERY sample of the pool (also those no record refers to): chunk ranges are stretched to tile
    // [0, pool_len); records out of wave_offset order get the whole pool in one copy before the first chunk
    long long keep_hi = 0;
    if (pool_keep && scan_all && pool_len > 0) PH_CHECK(staged_h2d(hp->stager, pool_keep, pool, (size_t)pool_len * esz, s_copy, pool_pinned));
    int64_t chunk_idx = 0;
    for (int64_t r0 = 0; r0 < n; r0 += chunk_records, ++chunk_idx) {
        const int64_t r1 = std::min<int64_t>(n, r0 + chunk_records), m = r1 - r0;
        Slot& s = slots[chunk_idx % kSlots];
        // pool range of the chunk.  Records built by the records plugins have wave_offsets that ascend with the record
        // index: the first and the last non-empty record bound the range.  If the device finds a record outside it
        // (filtered / reordered records), the call runs again with the range taken over every record.
        long long lo = -1, hi = -1;
        if (scan_all) {
            for (int64_t i = r0; i < r1; ++i) {
                const int len = rec_i32(rows + i * kRecordsRowBytes, 90);
                if (len <= 0) continue;
                const long long o = rec_i64(rows + i * kRecordsRowBytes, 82);
                lo = (lo < 0) ? o : std::min(lo, o);
                hi = std::max(hi, o + len);
            }
        } else {
            for (int64_t i = r0; i < r1; ++i) {
                if (rec_i32(rows + i * kRecordsRowBytes, 90) > 0) { lo = rec_i64(rows + i * kRecordsRowBytes, 82); break; }
            }
            for (int64_t i = r1 - 1; i >= r0; --i) {
                int len = rec_i32(rows + i * kRecordsRowBytes, 90);
                if (len > 0) { hi = rec_i64(rows + i * kRecordsRowBytes, 82) + len; break; }
            }
        }
        if (lo < 0) lo = hi = 0;
        if (lo > hi || hi > pool_len || lo < 0) {
            cleanup();
            if (!scan_all) {  // first / last record do not bound the chunk: records are not in wave_offset order
                scan_all = true;
                goto again;
            }
            set_error("records reference samples outside wave_pool bounds");
            return WFB_ERR_LAYOUT;
        }
        if (do_hits && hit_out_host && chunk_idx >= 2) PH_CHECK(drain_hits(chunk_idx - 2));
        if (pool_keep && !scan_all) {
            lo = std::min(lo, keep_hi);
            if (r1 == n) hi = pool_len;
            hi = std::max(hi, lo);
            keep_hi = std::max(keep_hi, hi);
        }
        const long long lo_al = lo & ~7ll;  // keep 16-byte alignment of record starts relative to the pool
        const size_t pool_bytes = (pool_keep && scan_all) ? 0 : (size_t)(hi - lo_al) * esz;
        // (re)allocation waits for the slot's previous work: only ever happens while the buffers grow
        const bool grow = (!pool_keep && pool_bytes + 64 > s.pool.cap) || (size_t)m * kRecordsRowBytes + 64 > s.rows.cap ||
                          wfb_features_hits_workspace_bytes(m) > s.ws.cap;
        if (grow) cleanup();
        if (!pool_keep) PH_CHECK(s.pool.ensure(pool_bytes + 64));
        PH_CHECK(s.rows.ensure((size_t)m * kRecordsRowBytes + 64));
        if (!meta_keep) PH_CHECK(s.meta.ensure((size_t)m * sizeof(wfb_rec_meta) + 64));
        void* const pool_dst = pool_keep ? static_cast<void*>(static_cast<uint8_t*>(pool_keep) + (size_t)lo_al * esz) : s.pool.p;
        wfb_rec_meta* const meta_dst = meta_keep ? meta_keep + r0 : static_cast<wfb_rec_meta*>(s.meta.p);
        if (do_feat) PH_CHECK(s.feat.ensure((size_t)m * kFeatRowBytes + 64));
        if (do_hits && hit_counts_host) PH_CHECK(s.counts.ensure((size_t)m * 4 + 64));
        PH_CHECK(s.ws.ensure(wfb_features_hits_workspace_bytes(m)));
        // the slot's previous results must have left the device before we overwrite them
        PH_CUDA(cudaStreamWaitEvent(s_copy, s.drained, 0));
        PH_CUDA(cudaStreamWaitEvent(s_copy, s.computed, 0));
        if (pool_bytes) PH_CHECK(staged_h2d(hp->stager, pool_dst, pool + (size_t)lo_al * esz, pool_bytes, s_copy, pool_pinned));
        PH_CHECK(staged_h2d(hp->stager, s.rows.p, rows + (size_t)r0 * kRecordsRowBytes, (size_t)m * kRecordsRowBytes, s_copy, rows_pinned));
        PH_CUDA(cudaEventRecord(s.copied, s_copy));
        PH_CUDA(cudaStreamWaitEvent(s_comp, s.copied, 0));
        PH_CUDA(cudaStreamWaitEvent(s_comp, s.drained, 0));
        PH_CHECK(wfb_records_unpack(s.rows.p, m, meta_dst, s_comp));
        p.pool_base = params->pool_base + lo_al;
        p.row_base = params->row_base + r0;
        int64_t* tot = static_cast<int64_t*>(d_tot.p);
        PH_CHECK(wfb_features_hits(pool_dst, hi - lo_al, meta_dst, m, &p, s.feat.p,
                                   d_hits.p, hit_cap, (do_hits && hit_counts_host) ? static_cast<int32_t*>(s.counts.p) : nullptr,
                                   tot + (chunk_idx & 1), tot + ((chunk_idx + 1) & 1), s.ws.p, s.ws.cap, s_comp));
        err_accumulate_kernel<<<1, 1, 0, s_comp>>>(reinterpret_cast<const int*>(static_cast<uint8_t*>(s.ws.p) + 4), run_err);
        PH_CUDA(cudaGetLastError());
        PH_CUDA(cudaMemcpyAsync(&hp->mailbox[chunk_idx % kSlots], tot + ((chunk_idx + 1) & 1), 8, cudaMemcpyDeviceToHost, s_comp));
        PH_CUDA(cudaEventRecord(s.computed, s_comp));
        PH_CUDA(cudaStreamWaitEvent(s_out, s.computed, 0));
        if (do_feat)
            PH_CUDA(cudaMemcpyAsync(static_cast<uint8_t*>(feat_out_host) + (size_t)r0 * kFeatRowBytes, s.feat.p,
                                    (size_t)m * kFeatRowBytes, cudaMemcpyDeviceToHost, s_out));
        if (do_hits && hit_counts_host)
            PH_CUDA(cudaMemcpyAsync(hit_counts_host + r0, s.counts.p, (size_t)m * 4, cudaMemcpyDeviceToHost, s_out));
        PH_CUDA(cudaEventRecord(s.drained, s_out));
    }
    {  // error flag of ANY chunk of the call (the workspaces are reused every kSlots chunks)
        int h_err = 0;
        PH_CUDA(cudaMemcpyAsync(&h_err, run_err, 4, cudaMemcpyDeviceToHost, s_comp));
        PH_CUDA(cudaStreamSynchronize(s_comp));
        if (h_err == 1) {
            cleanup();
            if (!scan_all) {  // records not in wave_offset order: take every record's range into account and run again
                scan_all = true;
                goto again;
            }
            set_error("records reference samples outside wave_pool bounds");
            return WFB_ERR_LAYOUT;
        }
        if (h_err == 2) {
            cleanup();
            set_error("lmax is smaller than the longest record passed");
            return WFB_ERR_INVALID;
        }
    }
    if (do_hits) {
        *n_hits = hp->mailbox[(chunk_idx - 1) % kSlots];
        if (hit_out_host) {
            if (chunk_idx >= 2) PH_CHECK(drain_hits(chunk_idx - 2));
            PH_CHECK(drain_hits(chunk_idx - 1));
        }
    }
    PH_CUDA(cudaStreamSynchronize(s_out));
    cleanup();
    return WFB_OK;
#undef PH_CHECK
#undef PH_CUDA
}

namespace wfb {
void release_peak_scratch();
}

extern "C" int wfb_process_host(const void* records_host, int64_t n, const void* pool_host, int64_t pool_len,
                                const wfb_fh_params* params, const wfb_chan_rule* rules_host, void* feat_out_host,
                                void* hit_out_host, int64_t hit_cap, int32_t* hit_counts_host, int64_t* n_hits,
                                int64_t chunk_records) {
    return process_host_impl(records_host, n, pool_host, pool_len, params, rules_host, feat_out_host, hit_out_host, hit_cap,
                             hit_counts_host, n_hits, chunk_records, nullptr, nullptr);
}

extern "C" int wfb_process_host_resident(const void* records_host, int64_t n, const void* pool_host, int64_t pool_len,
                                         const wfb_fh_params* params, const wfb_chan_rule* rules_host, void* feat_out_host,
                                         void* hit_out_host, int64_t hit_cap, int32_t* hit_counts_host, int64_t* n_hits,
                                         int64_t chunk_records, void* pool_keep_dev, wfb_rec_meta* meta_keep_dev) {
    WFB_REQUIRE(n == 0 || (pool_keep_dev && meta_keep_dev), "wfb_process_host_resident: NULL resident buffers");
    WFB_REQUIRE(((uintptr_t)pool_keep_dev & 15) == 0 && ((uintptr_t)meta_keep_dev & 15) == 0, "wfb_process_host_resident: resident buffers must be 16-byte aligned");
    return process_host_impl(records_host, n, pool_host, pool_len, params, rules_host, feat_out_host, hit_out_host, hit_cap,
                             hit_counts_host, n_hits, chunk_records, pool_keep_dev, meta_keep_dev);
}

// Host: one threaded pass over packed RECORDS rows (the strided numpy field reads it replaces cost one pass per field)
extern "C" int wfb_records_host_scan(const void* records_host, int64_t n, int64_t* ts_out, int64_t* end_ps_out, int64_t* stats) {
    WFB_REQUIRE(n >= 0 && stats != nullptr && (n == 0 || records_host != nullptr), "wfb_records_host_scan: bad arguments");
    const uint8_t* rows = static_cast<const uint8_t*>(records_host);
    const int nt = (int)std::max<int64_t>(1, std::min<int64_t>(8, n >> 15));
    struct Part { long long lo, hi, lmax, dt_min; };
    std::vector<Part> part(nt, Part{LLONG_MAX, LLONG_MIN, 0, LLONG_MAX});
    auto scan = [&](int t) {
        Part p{LLONG_MAX, LLONG_MIN, 0, LLONG_MAX};
        for (int64_t i = n * t / nt, e = n * (t + 1) / nt; i < e; ++i) {
            const uint8_t* r = rows + i * kRecordsRowBytes;
            const long long ts = rec_i64(r, 0), off = rec_i64(r, 82);
            const long long len = rec_i32(r, 90), dt = rec_i32(r, 72);
            if (ts_out) ts_out[i] = ts;
            if (end_ps_out) end_ps_out[i] = ts + std::max<long long>(len, 0) * dt * 1000;
            if (len > 0) {
                p.lo = std::min(p.lo, off);
                p.hi = std::max(p.hi, off + len);
                p.lmax = std::max(p.lmax, len);
            }
            p.dt_min = std::min(p.dt_min, dt);
        }
        part[t] = p;
    };
    std::vector<std::thread> th;
    for (int t = 1; t < nt; ++t) th.emplace_back(scan, t);
    scan(0);
    for (auto& x : th) x.join();
    Part a{LLONG_MAX, LLONG_MIN, 0, LLONG_MAX};
    for (const Part& p : part) {
        a.lo = std::min(a.lo, p.lo);
        a.hi = std::max(a.hi, p.hi);
        a.lmax = std::max(a.lmax, p.lmax);
        a.dt_min = std::min(a.dt_min, p.dt_min);
    }
    if (a.hi == LLONG_MIN) a.lo = a.hi = 0;  // no row with samples
    stats[0] = a.lo;
    stats[1] = a.hi;
    stats[2] = a.lmax;
    stats[3] = (n > 0) ? a.dt_min : 0;
    return WFB_OK;
}

extern "C" int wfb_release_cache(void) {
    wfb::release_peak_scratch();
    std::lock_guard<std::mutex> lock(g_pipes_mu);
    for (HostPipe* hp : g_pipes) {
        if (!hp) continue;
        std::lock_guard<std::mutex> pipe_lock(hp->mu);
        if (hp->ready) {
            cudaStreamSynchronize(hp->s_copy);
            cudaStreamSynchronize(hp->s_comp);
            cudaStreamSynchronize(hp->s_out);
        }
        hp->release_buffers();
    }
    return WFB_OK;
}
