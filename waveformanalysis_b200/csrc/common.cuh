// Shared device/host helpers for libwfb200 (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/wfb200.h"

namespace wfb {

// ---- error plumbing (thread-local last error, C-ABI status codes) ---------------------------
void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what);

#define WFB_CUDA(call)                                         \
    do {                                                       \
        cudaError_t e__ = (call);                              \
        if (e__ != cudaSuccess) return wfb::cuda_fail(e__, #call); \
    } while (0)

#define WFB_REQUIRE(cond, ...)            \
    do {                                  \
        if (!(cond)) {                    \
            wfb::set_error(__VA_ARGS__);  \
            return WFB_ERR_INVALID;       \
        }                                 \
    } while (0)

int sm_count();

constexpr int kRecordsRowBytes = 102;  // RECORDS_DTYPE
constexpr int kFeatRowBytes = 36;      // BASIC_FEATURES_DTYPE
constexpr int kHitRowBytes = 60;       // THRESHOLD_HIT_DTYPE
constexpr int kWidthRowBytes = 56;     // WAVEFORM_WIDTH_DTYPE
constexpr int kPeakRowBytes = 48;      // HIT_DTYPE
constexpr int kWidthIntRowBytes = 52;  // WAVEFORM_WIDTH_INTEGRAL_DTYPE

constexpr unsigned kFull = 0xffffffffu;

// ---- warp helpers ---------------------------------------------------------------------------
__device__ __forceinline__ int lane_id() { return threadIdx.x & 31; }

__device__ __forceinline__ double shfl_xor_f64(double v, int m) {
    int lo = __double2loint(v), hi = __double2hiint(v);
    lo = __shfl_xor_sync(kFull, lo, m);
    hi = __shfl_xor_sync(kFull, hi, m);
    return __hiloint2double(hi, lo);
}
__device__ __forceinline__ double shfl_f64(double v, int src) {
    int lo = __double2loint(v), hi = __double2hiint(v);
    lo = __shfl_sync(kFull, lo, src);
    hi = __shfl_sync(kFull, hi, src);
    return __hiloint2double(hi, lo);
}
__device__ __forceinline__ double shfl_up_f64(double v, int d) {
    int lo = __double2loint(v), hi = __double2hiint(v);
    lo = __shfl_up_sync(kFull, lo, d);
    hi = __shfl_up_sync(kFull, hi, d);
    return __hiloint2double(hi, lo);
}
__device__ __forceinline__ double warp_sum_f64(double v) {
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) v += shfl_xor_f64(v, m);
    return v;
}
__device__ __forceinline__ double warp_max_f64(double v) {
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) v = fmax(v, shfl_xor_f64(v, m));
    return v;
}
__device__ __forceinline__ double warp_min_f64(double v) {
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) v = fmin(v, shfl_xor_f64(v, m));
    return v;
}
__device__ __forceinline__ float warp_max_f32(float v) {
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) v = fmaxf(v, __shfl_xor_sync(kFull, v, m));
    return v;
}
__device__ __forceinline__ float warp_min_f32(float v) {
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) v = fminf(v, __shfl_xor_sync(kFull, v, m));
    return v;
}
__device__ __forceinline__ long long warp_sum_i64(long long v) {
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) {
        int lo = __shfl_xor_sync(kFull, (int)(v & 0xffffffffll), m);
        int hi = __shfl_xor_sync(kFull, (int)(v >> 32), m);
        v += ((long long)hi << 32) | (unsigned)lo;
    }
    return v;
}

// python seq[start:end] bounds for a sequence of length len (step 1)
__device__ __forceinline__ void resolve_slice(long long start, long long end, int len, int& lo, int& hi) {
    long long s = start < 0 ? (start + len < 0 ? 0 : start + len) : (start > len ? len : start);
    long long e = end < 0 ? (end + len < 0 ? 0 : end + len) : (end > len ? len : end);
    lo = (int)s;
    hi = (int)(e > s ? e : s);
}

// streaming (read-once) 16-byte load: keep it out of L1
__device__ __forceinline__ uint4 ldg_stream16(const void* p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}

// ---- RECORDS_DTYPE (102 B packed, 2-byte aligned rows) -> wfb_rec_meta -----------------------
// field offsets: core/processing/dtypes.py:80-100
//   timestamp i8@0  pid i4@8  board i2@12  channel i2@14  baseline f8@16  baseline_upstream f8@24
//   polarity U8@32 (UTF-32, 32 B)  record_id i8@64  dt i4@72  trigger_type i2@76  flags u4@78
//   wave_offset i8@82  event_length i4@90  time i8@94
__device__ __forceinline__ unsigned long long rd64(const uint16_t* h) {
    return (unsigned long long)h[0] | ((unsigned long long)h[1] << 16) | ((unsigned long long)h[2] << 32) |
           ((unsigned long long)h[3] << 48);
}
__device__ __forceinline__ unsigned rd32(const uint16_t* h) { return (unsigned)h[0] | ((unsigned)h[1] << 16); }

// The WFB_POL_* code of a polarity field (U8: 8 UTF-32 code units as 16 half-words): 'positive' / 'negative' / other,
// compared on the first code units and the last one so that e.g. 'pos' is not mistaken for 'positive'.  The one place
// that maps polarity strings to codes (wfb_records_unpack, wfb_apply_polarity).
__device__ __forceinline__ int polarity_code(const uint16_t* p) {
    unsigned c0 = rd32(p), c1 = rd32(p + 2), c7 = rd32(p + 14);
    int pol = WFB_POL_UNKNOWN;
    if (c7 == 'e') {
        // full 8-character compare
        const char* pos = "positive";
        const char* neg = "negative";
        bool isp = true, isn = true;
        for (int k = 0; k < 8; ++k) {
            unsigned ck = rd32(p + 2 * k);
            isp = isp && ck == (unsigned)pos[k];
            isn = isn && ck == (unsigned)neg[k];
        }
        pol = isp ? WFB_POL_POSITIVE : (isn ? WFB_POL_NEGATIVE : WFB_POL_UNKNOWN);
    }
    if (c0 == 'r' && c1 == 'a') {  // internal tag "rawpos" (waveformanalysis_b200/aos.py)
        const char* rp = "rawpos";
        bool isr = true;
        for (int k = 0; k < 8; ++k) isr = isr && rd32(p + 2 * k) == (k < 6 ? (unsigned)rp[k] : 0u);
        if (isr) pol = WFB_POL_RAW_POSITIVE;
    }
    return pol;
}

__device__ __forceinline__ wfb_rec_meta rec_meta_from_row(const uint16_t* h) {
    wfb_rec_meta m;
    m.timestamp = (long long)rd64(h + 0);
    m.board = (short)h[6];
    m.channel = (short)h[7];
    m.baseline = __longlong_as_double((long long)rd64(h + 8));
    m.polarity = (uint8_t)polarity_code(h + 16);
    m.pad_[0] = m.pad_[1] = m.pad_[2] = 0;
    m.record_id = (long long)rd64(h + 32);
    m.dt = (int)rd32(h + 36);
    m.wave_offset = (long long)rd64(h + 41);
    m.event_length = (int)rd32(h + 45);
    return m;
}

}  // namespace wfb
