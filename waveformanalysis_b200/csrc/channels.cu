// Per-channel tables applied on the device: polarity from channel metadata (wfb_apply_polarity) and the per-record
// filter configuration / Savitzky-Golay table of wfb_filter_pool (wfb_filter_plan).  Both look a record's channel key up
// in a small sorted table staged in shared memory; the grid is capped so that each block stages it once for many
// records.
#include <algorithm>

#include "common.cuh"

namespace wfb {

__device__ __forceinline__ int channel_key(const wfb_rec_meta& m) { return (int)m.board * 65536 + ((int)m.channel & 0xFFFF); }

// index of key in the sorted s_keys[0, n), -1 when absent
__device__ __forceinline__ int find_key(const int* s_keys, int n, int key) {
    int lo = 0, hi = n;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (s_keys[mid] < key) lo = mid + 1;
        else hi = mid;
    }
    return (lo < n && s_keys[lo] == key) ? lo : -1;
}

__global__ void __launch_bounds__(256) apply_polarity_kernel(wfb_rec_meta* __restrict__ meta, uint16_t* __restrict__ rows, long long n,
                                                             const wfb_polarity_entry* __restrict__ table, int n_table) {
    extern __shared__ int s_keys[];
    for (int j = threadIdx.x; j < n_table; j += blockDim.x) s_keys[j] = table[j].key;
    __syncthreads();
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const int e = find_key(s_keys, n_table, channel_key(meta[i]));
        if (e < 0) continue;
        uint16_t img[16];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const uint32_t w = table[e].image[k];
            img[2 * k] = (uint16_t)(w & 0xffffu);
            img[2 * k + 1] = (uint16_t)(w >> 16);
        }
        if (rows) {  // polarity U8 at byte 32 of the 2-byte aligned row
            uint16_t* p = rows + i * (kRecordsRowBytes / 2) + 16;
#pragma unroll
            for (int k = 0; k < 16; ++k) p[k] = img[k];
        }
        meta[i].polarity = (uint8_t)polarity_code(img);
    }
}

__global__ void __launch_bounds__(256) filter_plan_kernel(const wfb_rec_meta* __restrict__ meta, long long n, const int* __restrict__ keys,
                                                          const int* __restrict__ cfg_of_key, int n_keys, int default_cfg,
                                                          const int* __restrict__ sg_lut, const int* __restrict__ lut_off,
                                                          const int* __restrict__ wcap, int* __restrict__ cfg_index,
                                                          int* __restrict__ table_offset) {
    extern __shared__ int s_keys[];
    for (int j = threadIdx.x; j < n_keys; j += blockDim.x) s_keys[j] = keys[j];
    __syncthreads();
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const int e = find_key(s_keys, n_keys, channel_key(meta[i]));
        const int c = e < 0 ? default_cfg : cfg_of_key[e];
        const int lo = lut_off[c];
        int toff = -1;
        if (lo >= 0) toff = sg_lut[lo + min(max(meta[i].event_length, 0), wcap[c])];
        cfg_index[i] = c;
        table_offset[i] = toff;
    }
}

unsigned table_grid(long long n) { return (unsigned)std::max<long long>(1, std::min<long long>((n + 255) / 256, (long long)sm_count() * 8)); }

}  // namespace wfb

using namespace wfb;

extern "C" int wfb_apply_polarity(wfb_rec_meta* meta_dev, void* records_aos_dev, int64_t n, const wfb_polarity_entry* table_dev,
                                  int32_t n_table, void* stream) {
    WFB_REQUIRE(n >= 0 && n_table >= 0 && n_table <= WFB_MAX_CHANNEL_KEYS, "wfb_apply_polarity: bad size (n_table %d, at most %d)", (int)n_table,
                WFB_MAX_CHANNEL_KEYS);
    if (n == 0 || n_table == 0) return WFB_OK;
    WFB_REQUIRE(meta_dev && table_dev, "wfb_apply_polarity: NULL pointer");
    WFB_REQUIRE(((uintptr_t)records_aos_dev & 1) == 0, "wfb_apply_polarity: records must be 2-byte aligned");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    apply_polarity_kernel<<<table_grid(n), 256, (size_t)n_table * sizeof(int), st>>>(meta_dev, static_cast<uint16_t*>(records_aos_dev), n,
                                                                                     table_dev, n_table);
    WFB_CUDA(cudaGetLastError());
    return WFB_OK;
}

extern "C" int wfb_filter_plan(const wfb_rec_meta* meta_dev, int64_t n, const int32_t* keys_dev, const int32_t* cfg_of_key_dev, int32_t n_keys,
                               int32_t default_cfg, const int32_t* sg_lut_dev, const int32_t* sg_lut_off_of_cfg_dev,
                               const int32_t* sg_wcap_of_cfg_dev, int32_t* cfg_index_out, int32_t* sg_table_offset_out, void* stream) {
    WFB_REQUIRE(n >= 0 && n_keys >= 0 && n_keys <= WFB_MAX_CHANNEL_KEYS, "wfb_filter_plan: bad size (n_keys %d, at most %d)", (int)n_keys,
                WFB_MAX_CHANNEL_KEYS);
    WFB_REQUIRE(default_cfg >= 0, "wfb_filter_plan: negative default configuration");
    if (n == 0) return WFB_OK;
    WFB_REQUIRE(meta_dev && sg_lut_off_of_cfg_dev && sg_wcap_of_cfg_dev && cfg_index_out && sg_table_offset_out, "wfb_filter_plan: NULL pointer");
    WFB_REQUIRE(n_keys == 0 || (keys_dev && cfg_of_key_dev), "wfb_filter_plan: NULL key table");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    filter_plan_kernel<<<table_grid(n), 256, (size_t)n_keys * sizeof(int), st>>>(meta_dev, n, keys_dev, cfg_of_key_dev, n_keys, default_cfg,
                                                                                sg_lut_dev, sg_lut_off_of_cfg_dev, sg_wcap_of_cfg_dev,
                                                                                cfg_index_out, sg_table_offset_out);
    WFB_CUDA(cudaGetLastError());
    return WFB_OK;
}
