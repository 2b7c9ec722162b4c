// `hit`: scipy.signal.find_peaks per record on the device (HitFinderPlugin).
//
// Reference: core/plugins/builtin/cpu/peak_finding.py:213-565 (_compute_peaks, _find_peaks_in_waveform,
// _calculate_peak_height).  The arithmetic lives in scipy (un-vendored dependency, scipy>=1.7.0; restated
// from scipy/signal/_peak_finding.py and _peak_finding_utils.pyx, see oracle/np_oracle.py:find_peaks_1d):
//   local maxima (strict rise, plateau midpoint, strict fall) -> height >= hmin -> optional neighbour
//   threshold -> minimal distance (highest peaks first) -> prominence (bases = lowest samples up to the next
//   higher sample on each side) -> width at rel_height 0.5 with linearly interpolated crossings.
//
// One warp per record.  The record's waveform (float64, exact for int16 / float32 sources) and the
// detection signal are staged in shared memory; lanes test 32 positions per step for a local maximum and
// compact the survivors in order with ballots; prominence / width scans run one peak per lane.  Rows are
// variable in number: a counting pass, a device scan and an emitting pass (same code, rows switched on).
#include <algorithm>
#include <mutex>

#include "common.cuh"
#include "np_sum.cuh"
#include "sort_scan.cuh"

namespace wfb {

constexpr int kPeakWarps = 4;
constexpr int kPeakCache = 6;      // peaks per record the counting pass remembers (position, left / right edge)

struct PeakCacheEnt {  // 24 bytes
    double lip, rip;
    int pk, pad_;
};

// the record's waveform as the plugin sees it (float64, exact for int16 / float32 sources), read from global
// memory on demand: only the detection signal is staged in shared memory
struct Wave {
    const void* base;
    long long off;
    int load_kind;  // params->wave_kind
    float b32;
    bool pos;
    __device__ __forceinline__ double operator[](int i) const {
        if (load_kind == WFB_WAVE_AOS_I16) return (double)static_cast<const short*>(base)[off + i];
        if (load_kind == WFB_WAVE_AOS_U16) return (double)static_cast<const unsigned short*>(base)[off + i];
        if (load_kind == WFB_WAVE_AOS_F32 || load_kind == WFB_WAVE_AOS_F32_AS_F64) return (double)static_cast<const float*>(base)[off + i];
        const float s = (load_kind == WFB_WAVE_REC_U16) ? (float)static_cast<const unsigned short*>(base)[off + i]
                                                        : static_cast<const float*>(base)[off + i];
        // -RecordsView.signals(): signals = f32(w) - f32(b), negated once more for positive pulses (records_view.py:152-169)
        return pos ? (double)__fsub_rn(s, b32) : (double)__fsub_rn(b32, s);
    }
};

struct PeakRec {
    int kind, len, m;  // wave kind, samples, detection samples
    bool deriv;
    double baseline;
    Wave w;            // waveform values
    const double* x;   // shared: detection signal
};

__device__ __forceinline__ double detection_value(const PeakRec& r, int i) {
    if (r.deriv) {
        if (r.kind == WFB_WAVE_AOS_I16) {  // np.diff on int16 stays int16, so does the negation
            const short d = (short)((int)r.w[i + 1] - (int)r.w[i]);
            return (double)(short)(-(int)d);
        }
        if (r.kind == WFB_WAVE_AOS_U16) return (double)(((int)r.w[i] - (int)r.w[i + 1]) & 0xffff);  // uint16 diff and negation wrap
        if (r.kind == WFB_WAVE_AOS_F32) return (double)(-__fsub_rn((float)r.w[i + 1], (float)r.w[i]));
        if (r.kind == WFB_WAVE_AOS_F32_AS_F64) return -__dsub_rn(r.w[i + 1], r.w[i]);  // streaming: float64 copy of the row
        return __dsub_rn(r.w[i + 1], r.w[i]);  // records: +diff of the float64 signal
    }
    if (r.kind == WFB_WAVE_AOS_I16 || r.kind == WFB_WAVE_AOS_U16 || r.kind == WFB_WAVE_AOS_F32 || r.kind == WFB_WAVE_AOS_F32_AS_F64)
        return __dsub_rn(r.baseline, r.w[i]);
    return r.w[i];
}

struct DiffSrcF32 {  // np.diff(-waveform) for a float32 waveform
    Wave w;
    __device__ float operator()(int i) const { return __fsub_rn(-(float)w[i + 1], -(float)w[i]); }
};
struct DiffSrcF64 {
    Wave w;
    __device__ double operator()(int i) const { return __dsub_rn(-w[i + 1], -w[i]); }
};
template <typename S>
struct OffsetSrc {
    S s;
    int off;
    __device__ auto operator()(int i) const { return s(off + i); }
};

// peak_finding.py:567-614
__device__ float peak_height(const PeakRec& r, double edge_start, double edge_end, int method, int ext) {
    int s = max(0, (int)rint(edge_start));  // np.round: half to even
    int e = min(r.len - 1, (int)rint(edge_end));
    if (method == 2) {  // streaming "diff": cumsum(-diff(w)) in float64, clipped rounded edges (signal_peaks.py:370-381)
        const int max_idx = max(r.len - 1, 0);
        const int s2 = min(max((int)rint(edge_start), 0), max_idx), e2 = min(max((int)rint(edge_end), 0), max_idx);
        if (e2 <= s2) return 0.f;
        double cs = 0.0, at_s = 0.0;
        for (int j = 0; j < e2; ++j) {
            if (j == s2) at_s = cs;
            cs = __dadd_rn(cs, -__dsub_rn(r.w[j + 1], r.w[j]));
        }
        return (float)__dsub_rn(cs, at_s);
    }
    if (method == 1) {  // "diff": sum(diff(-w)[s:e]) in the waveform's own arithmetic
        if (e <= s) return 0.f;
        if (r.kind == WFB_WAVE_AOS_I16) {
            long long acc = 0;  // int16 diffs summed in int64
            for (int i = s; i < e; ++i) acc += (short)((int)(short)(-(int)r.w[i + 1]) - (int)(short)(-(int)r.w[i]));
            return (float)(double)acc;
        }
        if (r.kind == WFB_WAVE_AOS_U16) {
            unsigned long long acc = 0;  // uint16 diffs of the wrapped negation, summed in uint64
            for (int i = s; i < e; ++i) acc += (unsigned)(((int)r.w[i] - (int)r.w[i + 1]) & 0xffff);
            return (float)(double)acc;
        }
        if (r.kind == WFB_WAVE_AOS_F32) return numpy_pairwise_sum_t<float>(OffsetSrc<DiffSrcF32>{DiffSrcF32{r.w}, s}, e - s);
        return (float)numpy_pairwise_sum(OffsetSrc<DiffSrcF64>{DiffSrcF64{r.w}, s}, e - s);
    }
    ext = max(0, ext);
    const int a = max(0, s - ext), b = min(r.len, e + ext);
    if (b <= a) return __int_as_float(0x7fc00000);  // numpy raises on an empty window; cannot happen for found peaks
    double mx = r.w[a], mn = r.w[a];
    for (int i = a + 1; i < b; ++i) { mx = fmax(mx, r.w[i]); mn = fmin(mn, r.w[i]); }
    if (r.kind == WFB_WAVE_AOS_I16) return (float)(double)(short)((int)mx - (int)mn);
    if (r.kind == WFB_WAVE_AOS_U16) return (float)(double)(((int)mx - (int)mn) & 0xffff);
    if (r.kind == WFB_WAVE_AOS_F32) return __fsub_rn((float)mx, (float)mn);
    return (float)__dsub_rn(mx, mn);
}

// one packed HIT row (48 bytes) of a found peak
__device__ __forceinline__ void write_peak_row(uint8_t* rows, long long row, const PeakRec& r, const wfb_rec_meta& mrec,
                                               const wfb_peak_params& p, int pk, double lip, double rip) {
    const float hgt = peak_height(r, lip, rip, p.height_method, p.height_window_extension);
    const double step = __dmul_rn((double)mrec.dt, 1e3);
    const long long ti = (long long)__dadd_rn((double)mrec.timestamp, __dmul_rn((double)pk, step));
    unsigned* dst = reinterpret_cast<unsigned*>(rows + row * kPeakRowBytes);
    dst[0] = (unsigned)pk;
    dst[1] = 0u;
    dst[2] = __float_as_uint(hgt);
    dst[3] = 0u;  // integral (always 0.0 in the reference)
    dst[4] = __float_as_uint((float)lip);
    dst[5] = __float_as_uint((float)rip);
    dst[6] = (unsigned)mrec.dt;
    dst[7] = (unsigned)(ti & 0xffffffffll);
    dst[8] = (unsigned)((unsigned long long)ti >> 32);
    dst[9] = ((unsigned)(unsigned short)mrec.board) | ((unsigned)(unsigned short)mrec.channel << 16);
    dst[10] = (unsigned)(mrec.record_id & 0xffffffffll);
    dst[11] = (unsigned)((unsigned long long)mrec.record_id >> 32);
}

// emit pass for the records whose peaks all sit in the cache of the counting pass (the usual case): one THREAD per
// cache slot finishes a row - a warp per record would keep 2 of its 32 lanes busy
__global__ void __launch_bounds__(256) peaks_emit_cached_kernel(const void* __restrict__ waves, long long waves_len,
                                                               const wfb_rec_meta* __restrict__ meta, long long n, const wfb_peak_params p,
                                                               const int* __restrict__ counts, const long long* __restrict__ row_incl,
                                                               uint8_t* __restrict__ rows, long long row_cap,
                                                               const PeakCacheEnt* __restrict__ cache) {
    const long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    const long long rec = t / kPeakCache;
    const int k = (int)(t % kPeakCache);
    if (rec >= n) return;
    const int c = counts[rec];
    if (c > kPeakCache || k >= c) return;
    const wfb_rec_meta mrec = meta[rec];
    const bool records_src = p.wave_kind == WFB_WAVE_REC_U16 || p.wave_kind == WFB_WAVE_REC_F32;
    PeakRec r;
    r.kind = records_src ? WFB_WAVE_REC_U16 : p.wave_kind;
    r.len = mrec.event_length;  // validated by the counting pass (a rejected record has no peaks)
    r.deriv = p.use_derivative != 0;
    r.m = r.deriv ? max(r.len - 1, 0) : r.len;
    r.baseline = mrec.baseline;
    r.w = Wave{waves, mrec.wave_offset - p.pool_base, p.wave_kind, (float)mrec.baseline, mrec.polarity == WFB_POL_POSITIVE};
    r.x = nullptr;
    const PeakCacheEnt e = cache[rec * kPeakCache + k];
    const long long row = row_incl[rec] - c + k;
    if (row < row_cap) write_peak_row(rows, row, r, mrec, p, e.pk, e.lip, e.rip);
}

template <bool EMIT>
__global__ void __launch_bounds__(kPeakWarps * 32) find_peaks_kernel(const void* __restrict__ waves, long long waves_len,
                                                                     const wfb_rec_meta* __restrict__ meta, long long n,
                                                                     const wfb_peak_params p, int lcap, int* __restrict__ counts,
                                                                     const long long* __restrict__ row_incl,
                                                                     uint8_t* __restrict__ rows, long long row_cap, int* __restrict__ err,
                                                                     PeakCacheEnt* __restrict__ cache, uint8_t* __restrict__ gscratch) {
    extern __shared__ __align__(16) uint8_t smem[];
    const int warp = threadIdx.x >> 5, lane = lane_id();
    const int nwarps = blockDim.x >> 5;  // 4, 2 or 1: as many as fit the shared memory with records of lcap samples
    // per warp: x[lcap] doubles, peak positions int[lcap/2 + 2], keep flags; in shared memory, or (records too long
    // even for one warp per block) in a global scratch area that stays in L2
    const size_t per_warp = (((size_t)lcap * 8 + (size_t)(lcap / 2 + 2) * 4 + (size_t)(lcap / 2 + 2)) + 15) & ~(size_t)15;
    uint8_t* base = gscratch ? gscratch + ((size_t)blockIdx.x * nwarps + warp) * per_warp : smem + (size_t)warp * per_warp;
    double* x = reinterpret_cast<double*>(base);
    int* peaks = reinterpret_cast<int*>(x + lcap);
    uint8_t* keep = reinterpret_cast<uint8_t*>(peaks + (lcap / 2 + 2));

    auto do_record = [&](const long long rec) {
    const wfb_rec_meta mrec = meta[rec];
    int len = mrec.event_length;
    const long long off = mrec.wave_offset - p.pool_base;  // 0 for the AoS sources
    if (len < 0) len = 0;
    if (len > 0 && (off < 0 || off + len > waves_len)) {
        if (lane == 0) atomicExch(err, 1);
        len = 0;
    }
    if (len > lcap) {
        if (lane == 0) atomicExch(err, 2);
        len = 0;
    }
    const bool records_src = p.wave_kind == WFB_WAVE_REC_U16 || p.wave_kind == WFB_WAVE_REC_F32;
    PeakRec r;
    r.kind = records_src ? WFB_WAVE_REC_U16 : p.wave_kind;  // both records kinds share the float64 arithmetic
    r.len = len;
    r.deriv = p.use_derivative != 0;
    r.m = r.deriv ? max(len - 1, 0) : len;
    r.baseline = mrec.baseline;
    r.w = Wave{waves, off, p.wave_kind, (float)mrec.baseline, mrec.polarity == WFB_POL_POSITIVE};
    r.x = x;
    auto write_row = [&](long long row, int pk, double lip, double rip) { write_peak_row(rows, row, r, mrec, p, pk, lip, rip); };
    if (EMIT) {
        // records whose peaks all fit the cache are finished by peaks_emit_cached_kernel
        if (counts[rec] <= kPeakCache) return;
    }
    // ---- stage the detection signal.  The sample format is resolved once, outside the loop, and with the
    // derivative every sample is read from global memory once: lane i hands w[i] to its left neighbour's diff
    {
        const long long o = off;
        const float b32 = (float)mrec.baseline;
        const bool pos = mrec.polarity == WFB_POL_POSITIVE;
        auto stage = [&](auto loadf, auto difff, auto levelf) {
            const int m = r.m;
            if (r.deriv) {
                constexpr int U = 8;  // 32-sample groups in flight per pass: the loads are issued before any is used
                for (int b0 = 0; b0 < m; b0 += 32 * U) {
                    double wv[U];
#pragma unroll
                    for (int u = 0; u < U; ++u) {
                        const int i = b0 + 32 * u + lane;
                        wv[u] = (i <= m) ? loadf(i) : 0.0;  // m = len - 1: w[m] exists
                    }
                    const double wlast = (lane == 31 && b0 + 32 * U <= m) ? loadf(b0 + 32 * U) : 0.0;
#pragma unroll
                    for (int u = 0; u < U; ++u) {
                        const int i = b0 + 32 * u + lane;
                        double wn = shfl_f64(wv[u], (lane + 1) & 31);
                        const double nx = (u + 1 < U) ? shfl_f64(wv[(u + 1 < U) ? u + 1 : u], 0) : wlast;  // lane 31's successor
                        if (lane == 31) wn = nx;
                        if (i < m) x[i] = difff(wn, wv[u]);
                    }
                }
            } else {
                for (int i = lane; i < m; i += 32) x[i] = levelf(loadf(i));
            }
        };
        const double bl = r.baseline;
        auto lvl_sub = [&](double w) { return __dsub_rn(bl, w); };
        // float32 rows without a baseline field: the level is np.mean(row) (float32) minus the float32 row (peak_finding.py:508-511)
        auto lvl_sub32 = [&](double w) { return p.level_f32 ? (double)__fsub_rn((float)bl, (float)w) : __dsub_rn(bl, w); };
        auto lvl_id = [](double w) { return w; };
        switch (p.wave_kind) {
            case WFB_WAVE_AOS_U16:  // np.diff on uint16 and its negation wrap modulo 65536
                stage([&](int i) { return (double)static_cast<const unsigned short*>(waves)[o + i]; },
                      [](double wn, double wi) { return (double)(((int)wi - (int)wn) & 0xffff); }, lvl_sub);
                break;
            case WFB_WAVE_AOS_I16:  // np.diff on int16 stays int16, so does the negation
                stage([&](int i) { return (double)static_cast<const short*>(waves)[o + i]; },
                      [](double wn, double wi) { return (double)(short)(-(int)(short)((int)wn - (int)wi)); }, lvl_sub);
                break;
            case WFB_WAVE_AOS_F32:
                stage([&](int i) { return (double)static_cast<const float*>(waves)[o + i]; },
                      [](double wn, double wi) { return (double)(-__fsub_rn((float)wn, (float)wi)); }, lvl_sub32);
                break;
            case WFB_WAVE_AOS_F32_AS_F64:  // streaming: float64 copy of the row
                stage([&](int i) { return (double)static_cast<const float*>(waves)[o + i]; },
                      [](double wn, double wi) { return -__dsub_rn(wn, wi); }, lvl_sub);
                break;
            case WFB_WAVE_REC_U16:  // records: +diff of the float64 copy of -RecordsView.signals() (records_view.py:152-169)
                stage([&](int i) {
                          const float sv = (float)static_cast<const unsigned short*>(waves)[o + i];
                          return pos ? (double)__fsub_rn(sv, b32) : (double)__fsub_rn(b32, sv);
                      },
                      [](double wn, double wi) { return __dsub_rn(wn, wi); }, lvl_id);
                break;
            default:
                stage([&](int i) {
                          const float sv = static_cast<const float*>(waves)[o + i];
                          return pos ? (double)__fsub_rn(sv, b32) : (double)__fsub_rn(b32, sv);
                      },
                      [](double wn, double wi) { return __dsub_rn(wn, wi); }, lvl_id);
                break;
        }
    }
    __syncwarp();

    // ---- local maxima + height / threshold conditions, compacted in order
    const int m = r.m;
    int np = 0;
    for (int b0 = 0; b0 < m; b0 += 32) {
        const int i = b0 + lane;
        int pos = -1;
        // the height condition first: a plateau has one value, so x[pos] == x[i], and most samples (noise) fail it -
        // 32 samples without a candidate cost one load, one compare and one vote
        const double xi = (i >= 1 && i < m - 1) ? x[i] : 0.0;
        const bool cand = i >= 1 && i < m - 1 && xi >= p.height;
        if (!__any_sync(kFull, cand)) continue;
        if (cand && x[i - 1] < xi) {
            int ahead = i + 1;
            while (ahead < m - 1 && x[ahead] == xi) ++ahead;
            if (x[ahead] < xi) pos = (i + ahead - 1) >> 1;
        }
        if (pos >= 0 && p.has_threshold) {
            if (!(fmin(__dsub_rn(x[pos], x[pos - 1]), __dsub_rn(x[pos], x[pos + 1])) >= p.threshold)) pos = -1;
        }
        const unsigned bal = __ballot_sync(kFull, pos >= 0);
        if (pos >= 0) {
            const int k = np + __popc(bal & ((1u << lane) - 1u));
            peaks[k] = pos;
            keep[k] = 1;
        }
        np += __popc(bal);
    }
    __syncwarp();
    // ---- minimal distance: highest peaks first (stable order among equal heights: the later peak wins)
    if (p.distance > 2 && np > 1 && lane == 0) {
        for (int round = 0; round < np; ++round) {
            // the highest peak not yet visited: visited peaks are marked with bit 1 of keep
            int best = -1;
            for (int k = 0; k < np; ++k) {
                if (keep[k] & 2) continue;
                if (best < 0 || x[peaks[k]] >= x[peaks[best]]) best = k;
            }
            if (best < 0) break;
            keep[best] |= 2;
            if (!(keep[best] & 1)) continue;
            for (int k = best - 1; k >= 0 && peaks[best] - peaks[k] < p.distance; --k) keep[k] &= ~1;
            for (int k = best + 1; k < np && peaks[k] - peaks[best] < p.distance; ++k) keep[k] &= ~1;
        }
    }
    __syncwarp();
    // ---- prominence, width, rows: peaks one after the other, every scan done by the whole warp 32 samples at a
    // time (the tallest peaks scan the whole record: one lane would walk hundreds of samples alone)
    long long row0 = 0;
    if (EMIT) row0 = row_incl[rec] - counts[rec];
    int nout = 0;
    const double kInf = __longlong_as_double(0x7ff0000000000000ll);
    for (int q = 0; q < np; ++q) {
        if (!(keep[q] & 1)) continue;
        const int pk = peaks[q];
        const double xp = x[pk];
        // left side: samples pk, pk-1, ... while x <= xp; lowest value, among equals the one nearest to the peak
        double lmin = kInf;
        int lidx = -1;
        for (int hi = pk; hi >= 0; hi -= 32) {
            const int i = hi - lane;
            const bool in = i >= 0;
            const double xi = in ? x[i] : 0.0;
            const unsigned stop = __ballot_sync(kFull, in && xi > xp);
            const int nstop = stop ? __ffs(stop) - 1 : 32;  // lanes below nstop are still inside the scan
            if (in && lane < nstop && xi < lmin) { lmin = xi; lidx = i; }
            if (stop) break;
        }
        double rmin = kInf;
        int ridx = 0x7fffffff;
        for (int lo = pk; lo <= m - 1; lo += 32) {
            const int i = lo + lane;
            const bool in = i <= m - 1;
            const double xi = in ? x[i] : 0.0;
            const unsigned stop = __ballot_sync(kFull, in && xi > xp);
            const int nstop = stop ? __ffs(stop) - 1 : 32;
            if (in && lane < nstop && xi < rmin) { rmin = xi; ridx = i; }
            if (stop) break;
        }
        // each lane holds the nearest index of its own minimum (it scans away from the peak with a strict <)
        const double lm = warp_min_f64(lmin), rm = warp_min_f64(rmin);
        const int lb = __reduce_max_sync(kFull, (lmin == lm) ? lidx : -1);
        const int rb = __reduce_min_sync(kFull, (rmin == rm) ? ridx : 0x7fffffff);
        const double prom = __dsub_rn(xp, fmax(lm, rm));
        if (!(prom >= p.prominence)) continue;
        // width at half prominence: first sample at or below the level on each side, not beyond the bases
        const double h = __dsub_rn(xp, __dmul_rn(prom, 0.5));
        int il = lb;
        for (int hi = pk; hi > lb; hi -= 32) {
            const int i = hi - lane;
            const unsigned stop = __ballot_sync(kFull, i > lb && !(h < x[i]));
            if (stop) { il = hi - (__ffs(stop) - 1); break; }
        }
        int ir = rb;
        for (int lo = pk; lo < rb; lo += 32) {
            const int i = lo + lane;
            const unsigned stop = __ballot_sync(kFull, i < rb && !(h < x[i]));
            if (stop) { ir = lo + (__ffs(stop) - 1); break; }
        }
        double lip = (double)il, rip = (double)ir;
        if (x[il] < h) lip = __dadd_rn(lip, __ddiv_rn(__dsub_rn(h, x[il]), __dsub_rn(x[il + 1], x[il])));
        if (x[ir] < h) rip = __dsub_rn(rip, __ddiv_rn(__dsub_rn(h, x[ir]), __dsub_rn(x[ir - 1], x[ir])));
        if (!(__dsub_rn(rip, lip) >= p.width)) continue;
        if (EMIT && lane == 0) {
            const long long row = row0 + nout;
            if (row < row_cap) write_row(row, pk, lip, rip);
        }
        if (!EMIT && lane == 0 && nout < kPeakCache) cache[rec * kPeakCache + nout] = PeakCacheEnt{lip, rip, pk, 0};
        ++nout;
    }
    if (!EMIT && lane == 0) counts[rec] = nout;
    };
    for (long long rec = (long long)blockIdx.x * nwarps + warp; rec < n; rec += (long long)gridDim.x * nwarps) {
        do_record(rec);
        __syncwarp();  // the staging area is reused by the warp's next record
    }
}

__global__ void peaks_counts_to_i64_kernel(const int* __restrict__ counts, long long n, long long* __restrict__ out) {
    long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i < n) out[i] = counts[i];
}
__global__ void peaks_total_kernel(const long long* __restrict__ incl, long long n, long long* __restrict__ total) {
    if (blockIdx.x == 0 && threadIdx.x == 0) *total = n > 0 ? incl[n - 1] : 0;
}

}  // namespace wfb

using namespace wfb;

static size_t pk_al256(size_t x) { return (x + 255) & ~(size_t)255; }

// Staging area of wfb_find_peaks for records too long for shared memory: kept per device between calls (the stream
// order of the calls serialises its use), freed by wfb_release_cache().
namespace {
std::mutex g_scratch_mu;
void* g_scratch[64];
size_t g_scratch_cap[64];
int peak_scratch(size_t bytes, uint8_t** out) {
    std::lock_guard<std::mutex> lock(g_scratch_mu);
    int dev = 0;
    WFB_CUDA(cudaGetDevice(&dev));
    WFB_REQUIRE(dev >= 0 && dev < 64, "wfb_find_peaks: device index %d out of range", dev);
    if (g_scratch_cap[dev] < bytes) {
        if (g_scratch[dev]) {
            WFB_CUDA(cudaDeviceSynchronize());
            cudaFree(g_scratch[dev]);
            g_scratch[dev] = nullptr;
            g_scratch_cap[dev] = 0;
        }
        cudaError_t e = cudaMalloc(&g_scratch[dev], bytes);
        if (e != cudaSuccess) {
            (void)cudaGetLastError();
            g_scratch[dev] = nullptr;
            set_error("wfb_find_peaks: cudaMalloc(%zu) for the long-record staging area failed", bytes);
            return WFB_ERR_NOMEM;
        }
        g_scratch_cap[dev] = bytes;
    }
    *out = static_cast<uint8_t*>(g_scratch[dev]);
    return WFB_OK;
}
}  // namespace

namespace wfb {
void release_peak_scratch() {
    std::lock_guard<std::mutex> lock(g_scratch_mu);
    for (int d = 0; d < 64; ++d) {
        if (!g_scratch[d]) continue;
        int cur = 0;
        cudaGetDevice(&cur);
        cudaSetDevice(d);
        cudaFree(g_scratch[d]);
        cudaSetDevice(cur);
        g_scratch[d] = nullptr;
        g_scratch_cap[d] = 0;
    }
}
}  // namespace wfb

extern "C" size_t wfb_find_peaks_workspace_bytes(int64_t n) {
    const size_t m = pk_al256((size_t)std::max<int64_t>(n, 1) * 8);
    return 2 * m + pk_al256((size_t)std::max<int64_t>(n, 1) * 4) + scan_workspace_bytes(n) + 1024 +
           pk_al256((size_t)std::max<int64_t>(n, 1) * kPeakCache * sizeof(PeakCacheEnt));
}

extern "C" int wfb_find_peaks(const void* waves_dev, int64_t waves_len, const wfb_rec_meta* meta_dev, int64_t n,
                              const wfb_peak_params* params, void* rows_out_dev, int64_t row_cap, int32_t* counts_out_dev,
                              int64_t* total_out_dev, void* workspace_dev, size_t workspace_bytes, void* stream) {
    WFB_REQUIRE(params != nullptr && total_out_dev != nullptr, "wfb_find_peaks: NULL params / total");
    WFB_REQUIRE(n >= 0 && waves_len >= 0 && row_cap >= 0, "wfb_find_peaks: negative size");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (n == 0) {
        WFB_CUDA(cudaMemsetAsync(total_out_dev, 0, 8, st));
        return WFB_OK;
    }
    WFB_REQUIRE(meta_dev && workspace_dev && (waves_dev || waves_len == 0), "wfb_find_peaks: NULL pointer");
    WFB_REQUIRE(row_cap == 0 || rows_out_dev != nullptr, "wfb_find_peaks: NULL row buffer");
    WFB_REQUIRE(params->wave_kind >= WFB_WAVE_AOS_I16 && params->wave_kind <= WFB_WAVE_AOS_U16, "wfb_find_peaks: unknown wave_kind");
    WFB_REQUIRE(params->pool_base == 0 || params->wave_kind == WFB_WAVE_REC_U16 || params->wave_kind == WFB_WAVE_REC_F32,
                "wfb_find_peaks: pool_base %lld needs a records wave_kind (the AoS sources take pool_base 0)", (long long)params->pool_base);
    WFB_REQUIRE(params->height_method >= 0 && params->height_method <= 2, "unsupported height_method");
    WFB_REQUIRE(params->lmax > 0, "wfb_find_peaks: lmax must be the longest record");
    WFB_REQUIRE(workspace_bytes >= wfb_find_peaks_workspace_bytes(n), "wfb_find_peaks: workspace too small");
    const int lcap = (params->lmax + 1) & ~1;
    const size_t per_warp = (((size_t)lcap * 8 + (size_t)(lcap / 2 + 2) * 4 + (size_t)(lcap / 2 + 2)) + 15) & ~(size_t)15;
    // warps per block: as many (4, 2, 1) as fit the shared memory; longer records stage in a global scratch area
    // (a bounded persistent grid, so the area stays small enough for L2)
    int nwarps = kPeakWarps;
    while (nwarps > 1 && per_warp * nwarps > 200 * 1024) nwarps >>= 1;
    const bool in_global = per_warp * nwarps > 200 * 1024;
    if (in_global) nwarps = kPeakWarps;
    const size_t dyn = in_global ? 0 : per_warp * nwarps;
    unsigned grid = (unsigned)std::min<long long>((n + nwarps - 1) / nwarps, 0x7fffffff);
    uint8_t* gscratch = nullptr;
    if (in_global) {
        grid = (unsigned)std::min<long long>(grid, (long long)sm_count() * 2);
        const int rc_s = peak_scratch((size_t)grid * nwarps * per_warp, &gscratch);
        if (rc_s != WFB_OK) return rc_s;
    }
    uint8_t* ws = static_cast<uint8_t*>(workspace_dev);
    const size_t m = pk_al256((size_t)n * 8);
    long long* cnt64 = reinterpret_cast<long long*>(ws);
    long long* incl = reinterpret_cast<long long*>(ws + m);
    int* counts = reinterpret_cast<int*>(ws + 2 * m);
    int* err = reinterpret_cast<int*>(ws + 2 * m + pk_al256((size_t)n * 4));
    void* scan_ws = ws + 2 * m + pk_al256((size_t)n * 4) + 256;
    PeakCacheEnt* cache = reinterpret_cast<PeakCacheEnt*>(ws + 2 * m + pk_al256((size_t)n * 4) + 512 + pk_al256(scan_workspace_bytes(n)));
    WFB_CUDA(cudaMemsetAsync(err, 0, 4, st));
    wfb_peak_params p = *params;
    p.distance = (int)std::min<long long>(std::max<long long>(p.distance, 0), 1 << 30);
    WFB_CUDA(cudaFuncSetAttribute(find_peaks_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
    WFB_CUDA(cudaFuncSetAttribute(find_peaks_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
    find_peaks_kernel<false><<<grid, nwarps * 32, dyn, st>>>(waves_dev, waves_len, meta_dev, n, p, lcap, counts, nullptr, nullptr, 0, err, cache, gscratch);
    peaks_counts_to_i64_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(counts, n, cnt64);
    int rc = inclusive_scan_sum_i64(cnt64, incl, n, scan_ws, st);
    if (rc != WFB_OK) return rc;
    peaks_total_kernel<<<1, 32, 0, st>>>(incl, n, reinterpret_cast<long long*>(total_out_dev));
    if (row_cap > 0) {
        const long long slots = n * kPeakCache;
        peaks_emit_cached_kernel<<<(unsigned)((slots + 255) / 256), 256, 0, st>>>(waves_dev, waves_len, meta_dev, n, p, counts, incl,
                                                                               static_cast<uint8_t*>(rows_out_dev), row_cap, cache);
        find_peaks_kernel<true><<<grid, nwarps * 32, dyn, st>>>(waves_dev, waves_len, meta_dev, n, p, lcap, counts, incl,
                                                              static_cast<uint8_t*>(rows_out_dev), row_cap, err, cache, gscratch);
    }
    if (counts_out_dev) WFB_CUDA(cudaMemcpyAsync(counts_out_dev, counts, (size_t)n * 4, cudaMemcpyDeviceToDevice, st));
    WFB_CUDA(cudaGetLastError());
    int herr = 0;
    WFB_CUDA(cudaMemcpyAsync(&herr, err, 4, cudaMemcpyDeviceToHost, st));
    WFB_CUDA(cudaStreamSynchronize(st));
    if (herr == 1) {
        set_error("records reference samples outside the waveform buffer");
        return WFB_ERR_LAYOUT;
    }
    if (herr == 2) {
        set_error("a record is longer than params->lmax");
        return WFB_ERR_INVALID;
    }
    return WFB_OK;
}
