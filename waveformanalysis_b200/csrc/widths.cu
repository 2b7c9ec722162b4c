// waveform_width (per hit, threshold crossings with linear interpolation) and
// waveform_width_integral (per record, cumulative-charge quantiles).
//
// Reference: core/plugins/builtin/cpu/waveform_width.py:205-374,
//            core/plugins/builtin/cpu/waveform_width_integral.py:166-231.
#include <algorithm>

#include "common.cuh"
#include "np_sum.cuh"
#include "sort_scan.cuh"

namespace wfb {

// ---------------------------------------------------------------------------------------------
// waveform_width: one warp per hit.  numpy promotion rules are followed as the reference gets
// them: int16 rows -> everything float64; float32 rows -> baseline, corrected wave, thresholds
// and the interpolated crossing in float32, sums with the int64 peak position in float64.
// ---------------------------------------------------------------------------------------------

// np.mean of the first n (<= 50) float32 samples: numpy's pairwise sum for n < 128 keeps eight partial sums (r[k] takes
// samples k, k + 8, ...), folds them as ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)) and adds the tail n % 8 one by one.
// Computed by the warp: lanes 0..7 own the eight partial sums (each adds its samples in numpy's order), the
// fold is the same tree through shuffles, lane 0 adds the tail - the result is bit-identical, the dependent chain is six
// loads deep instead of fifty.  Returns the mean in every lane.
__device__ __forceinline__ float numpy_mean_f32_warp(const float* w, int n) {
    const int lane = lane_id();
    float res = 0.f;
    if (n < 8) {
        if (lane == 0)
            for (int i = 0; i < n; ++i) res = __fadd_rn(res, w[i]);
    } else {
        const int body = n - (n % 8);
        float r = 0.f;
        if (lane < 8) {
            r = w[lane];
            for (int i = 8 + lane; i < body; i += 8) r = __fadd_rn(r, w[i]);
        }
        const float p1 = __fadd_rn(r, __shfl_down_sync(kFull, r, 1));    // lanes 0, 2, 4, 6: r0+r1, r2+r3, r4+r5, r6+r7
        const float p2 = __fadd_rn(p1, __shfl_down_sync(kFull, p1, 2));  // lanes 0, 4
        res = __fadd_rn(p2, __shfl_down_sync(kFull, p2, 4));             // lane 0
        if (lane == 0)
            for (int i = body; i < n; ++i) res = __fadd_rn(res, w[i]);
    }
    res = __fdiv_rn(res, (float)n);
    return __shfl_sync(kFull, res, 0);
}

// first index in [lo, hi) where pred(i) holds, -1 if none; warp-cooperative
template <typename F>
__device__ __forceinline__ int warp_find_first(int lo, int hi, F pred) {
    const int lane = lane_id();
    // four 32-sample groups per pass: their loads are issued together, so a long scan (the rising edge is searched
    // from the start of the record) pays the memory latency once per 128 samples
    for (int base = lo; base < hi; base += 128) {
        const int i0 = base + lane, i1 = i0 + 32, i2 = i0 + 64, i3 = i0 + 96;
        const bool p0 = i0 < hi && pred(i0);
        const bool p1 = i1 < hi && pred(i1);
        const bool p2 = i2 < hi && pred(i2);
        const bool p3 = i3 < hi && pred(i3);
        const unsigned m0 = __ballot_sync(kFull, p0), m1 = __ballot_sync(kFull, p1);
        const unsigned m2 = __ballot_sync(kFull, p2), m3 = __ballot_sync(kFull, p3);
        if (m0) return base + __ffs(m0) - 1;
        if (m1) return base + 32 + __ffs(m1) - 1;
        if (m2) return base + 64 + __ffs(m2) - 1;
        if (m3) return base + 96 + __ffs(m3) - 1;
    }
    return -1;
}

// the same for two predicates over one scan (both thresholds of an edge are searched in the same slice): every
// sample is loaded once; the scan ends when both have been found
template <typename V, typename PA, typename PB>
__device__ __forceinline__ void warp_find_first2(int lo, int hi, V val, PA pa, PB pb, int& ia, int& ib) {
    const int lane = lane_id();
    ia = -1;
    ib = -1;
    for (int base = lo; base < hi && (ia < 0 || ib < 0); base += 128) {
        unsigned ma[4], mb[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int i = base + 32 * u + lane;
            const bool in = i < hi;
            const auto v = val(in ? i : lo);
            ma[u] = __ballot_sync(kFull, in && pa(v));
            mb[u] = __ballot_sync(kFull, in && pb(v));
        }
        if (ia < 0) {
            if (ma[0]) ia = base + __ffs(ma[0]) - 1;
            else if (ma[1]) ia = base + 32 + __ffs(ma[1]) - 1;
            else if (ma[2]) ia = base + 64 + __ffs(ma[2]) - 1;
            else if (ma[3]) ia = base + 96 + __ffs(ma[3]) - 1;
        }
        if (ib < 0) {
            if (mb[0]) ib = base + __ffs(mb[0]) - 1;
            else if (mb[1]) ib = base + 32 + __ffs(mb[1]) - 1;
            else if (mb[2]) ib = base + 64 + __ffs(mb[2]) - 1;
            else if (mb[3]) ib = base + 96 + __ffs(mb[3]) - 1;
        }
    }
}

// Where a hit's samples and its row fields come from.  `locate` gives the hit's waveform and its length (false: no
// waveform, the hit gives no row); the other members give the hit's own fields.
template <typename T>
struct WidthRowsSrc {  // structured rows of one width, hits as device columns (wfb_waveform_width)
    const T* waves;
    long long n_waves;
    int length;
    long long stride;
    const long long *row, *pos, *ts;
    const short *board, *channel;
    const long long* rid;
    __device__ __forceinline__ bool locate(long long hit, const T*& w, int& len) const {
        const long long r = row[hit];
        if (r < 0 || r >= n_waves) return false;
        w = waves + r * stride;
        len = length;
        return true;
    }
    __device__ __forceinline__ long long position(long long hit) const { return pos[hit]; }
    __device__ __forceinline__ long long timestamp(long long hit) const { return ts[hit]; }
    __device__ __forceinline__ unsigned board_channel(long long hit) const {
        return ((unsigned)(unsigned short)(board ? board[hit] : 0)) | ((unsigned)(unsigned short)channel[hit] << 16);
    }
    __device__ __forceinline__ long long record_id(long long hit) const { return rid[hit]; }
};

template <typename T>
struct WidthRunSrc {  // a device-resident run (records meta + pool slice), hits as packed HIT rows (wfb_waveform_width_run)
    const T* pool;
    long long pool_len;
    const wfb_rec_meta* meta;
    long long n, pool_base, row_base;
    const unsigned* hits;  // HIT_DTYPE rows as words
    __device__ __forceinline__ long long word64(long long hit, int k) const {
        const unsigned* h = hits + hit * (kPeakRowBytes / 4);
        return (long long)(((unsigned long long)h[k + 1] << 32) | h[k]);
    }
    __device__ __forceinline__ bool locate(long long hit, const T*& w, int& len) const {
        const long long rid = record_id(hit);
        const long long r = rid - row_base;
        if (r < 0 || r >= n || meta[r].record_id != rid) return false;
        const long long off = meta[r].wave_offset - pool_base;
        len = meta[r].event_length;
        if (off < 0 || len < 0 || off + len > pool_len) return false;
        w = pool + off;
        return true;
    }
    __device__ __forceinline__ long long position(long long hit) const { return word64(hit, 0); }
    __device__ __forceinline__ long long timestamp(long long hit) const { return word64(hit, 7); }
    __device__ __forceinline__ unsigned board_channel(long long hit) const { return hits[hit * (kPeakRowBytes / 4) + 9]; }
    __device__ __forceinline__ long long record_id(long long hit) const { return word64(hit, 10); }
};

// One hit, by its whole warp.  Returns whether the hit gives a row (the same value in every lane); with ROWS the row's
// 14 words are written to `out`, without it the work ends once that is known (the counting pass of the run variant).
template <typename T, bool ROWS, typename Src>
__device__ __forceinline__ bool width_of_hit(const Src& src, long long hit, const wfb_width_params& p, unsigned* __restrict__ out) {
    constexpr bool F32 = sizeof(T) == 4;
    const int lane = lane_id();
    const T* w = nullptr;
    int length = 0;
    if (!src.locate(hit, w, length)) return false;
    const long long pos64 = src.position(hit);
    if (!(pos64 < length && length > 0)) return false;
    // numpy negative indices wrap: position in [-length, 0) addresses from the end
    const long long posw = pos64 < 0 ? pos64 + length : pos64;
    if (!(posw >= 0 && posw < length)) return false;
    const int pos = (int)posw;
    const int nb = min(50, length);
    double bl64 = 0.0;
    float bl32 = 0.f;
    if (F32) {
        bl32 = numpy_mean_f32_warp(reinterpret_cast<const float*>(w), nb);
    } else {
        long long s = 0;
        for (int i = lane; i < nb; i += 32) s += (long long)w[i];
        s = warp_sum_i64(s);
        bl64 = (double)s / (double)nb;  // integer sum is exact, one division as np.mean
    }
    auto wc64 = [&](int i) -> double { return __dsub_rn((double)w[i], bl64); };
    auto wc32 = [&](int i) -> float { return __fsub_rn((float)w[i], bl32); };
    const double pv = F32 ? (double)wc32(pos) : wc64(pos);
    if (pv <= 0.0) return false;  // peak_value <= 0 (NaN compares false in the reference too: NaN <= 0 is False!)
    if (!ROWS) return true;
    // the slices wave[:pos] / wave[pos:] use the raw (possibly negative) position
    const int left_hi = pos;
    // thresholds
    double t64[4];
    float t32[4];
    const double fr[4] = {p.rise_low, p.rise_high, p.fall_high, p.fall_low};
    for (int k = 0; k < 4; ++k) {
        t64[k] = __dmul_rn(pv, fr[k]);
        t32[k] = __fmul_rn((float)pv, (float)fr[k]);
    }
    // crossing positions: value + kind (interpolated positions are float32 for float32 rows)
    double cross[4];
    bool found[4];
    // both thresholds of an edge in one scan: rising edge in wave[:pos], falling edge in wave[pos:]
    int idx4[4];
    if (F32) {
        const float ta = t32[0], tb = t32[1], tc = t32[2], td = t32[3];
        warp_find_first2(0, left_hi, [&](int i) { return wc32(i); }, [&](float v) { return v >= ta; }, [&](float v) { return v >= tb; }, idx4[0], idx4[1]);
        warp_find_first2(pos, length, [&](int i) { return wc32(i); }, [&](float v) { return v <= tc; }, [&](float v) { return v <= td; }, idx4[2], idx4[3]);
    } else {
        const double ta = t64[0], tb = t64[1], tc = t64[2], td = t64[3];
        warp_find_first2(0, left_hi, [&](int i) { return wc64(i); }, [&](double v) { return v >= ta; }, [&](double v) { return v >= tb; }, idx4[0], idx4[1]);
        warp_find_first2(pos, length, [&](int i) { return wc64(i); }, [&](double v) { return v <= tc; }, [&](double v) { return v <= td; }, idx4[2], idx4[3]);
    }
    for (int k = 0; k < 4; ++k) {
        const bool rising = k < 2;
        const int lo = rising ? 0 : pos;
        const int idx = idx4[k];
        found[k] = idx >= 0;
        cross[k] = 0.0;
        if (idx >= 0) {
            const int rel = idx - lo;  // index inside the slice
            if (!p.interpolation || rel == 0) {
                cross[k] = (double)rel;
            } else if (F32) {
                float y0 = wc32(idx - 1), y1 = wc32(idx);
                float dy = __fsub_rn(y1, y0);
                if (fabsf(dy) < 1e-10f) cross[k] = (double)rel;
                else cross[k] = (double)__fadd_rn((float)(rel - 1), __fdiv_rn(__fsub_rn(t32[k], y0), dy));
            } else {
                double y0 = wc64(idx - 1), y1 = wc64(idx);
                double dy = __dsub_rn(y1, y0);
                if (fabs(dy) < 1e-10) cross[k] = (double)rel;
                else cross[k] = __dadd_rn((double)(rel - 1), __ddiv_rn(__dsub_rn(t64[k], y0), dy));
            }
        }
    }
    double rts = 0.0, rt = 0.0, fts = 0.0, ft = 0.0, tws = 0.0, tw = 0.0;
    if (found[0] && found[1]) {
        rts = F32 ? (double)__fsub_rn((float)cross[1], (float)cross[0]) : __dsub_rn(cross[1], cross[0]);
        rt = F32 ? (double)__fdiv_rn((float)rts, (float)p.sampling_rate) : __ddiv_rn(rts, p.sampling_rate);
    }
    double fh = 0.0, fl = 0.0;
    if (found[2] && found[3]) {
        fh = __dadd_rn(cross[2], (double)pos64);  // + np.int64 position -> float64
        fl = __dadd_rn(cross[3], (double)pos64);
        fts = __dsub_rn(fl, fh);
        ft = __ddiv_rn(fts, p.sampling_rate);
    }
    if (found[0] && found[3]) {
        if (found[2]) {
            tws = __dsub_rn(fl, cross[0]);
            tw = __ddiv_rn(tws, p.sampling_rate);
        } else {  // fall_low_pos was not shifted by the peak position (waveform_width.py:294-306)
            tws = F32 ? (double)__fsub_rn((float)cross[3], (float)cross[0]) : __dsub_rn(cross[3], cross[0]);
            tw = F32 ? (double)__fdiv_rn((float)tws, (float)p.sampling_rate) : __ddiv_rn(tws, p.sampling_rate);
        }
    }
    if (lane < 14) {
        unsigned word;
        switch (lane) {
            case 0: word = __float_as_uint((float)rt); break;
            case 1: word = __float_as_uint((float)ft); break;
            case 2: word = __float_as_uint((float)tw); break;
            case 3: word = __float_as_uint((float)rts); break;
            case 4: word = __float_as_uint((float)fts); break;
            case 5: word = __float_as_uint((float)tws); break;
            case 6: word = (unsigned)(pos64 & 0xffffffffll); break;
            case 7: word = (unsigned)((unsigned long long)pos64 >> 32); break;
            case 8: word = __float_as_uint((float)pv); break;
            case 9: word = (unsigned)(src.timestamp(hit) & 0xffffffffll); break;
            case 10: word = (unsigned)((unsigned long long)src.timestamp(hit) >> 32); break;
            case 11: word = src.board_channel(hit); break;
            case 12: word = (unsigned)(src.record_id(hit) & 0xffffffffll); break;
            default: word = (unsigned)((unsigned long long)src.record_id(hit) >> 32); break;
        }
        out[lane] = word;
    }
    return true;
}

// six blocks of the float32 instance fit an SM at 40 registers (the row source's fields would otherwise take it to 46)
template <typename T>
__global__ void __launch_bounds__(256, sizeof(T) == 4 ? 6 : 5) waveform_width_kernel(const WidthRowsSrc<T> src, long long n_hits, const wfb_width_params p,
                                                            uint8_t* __restrict__ out, uint8_t* __restrict__ valid) {
    const long long hit = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
    if (hit >= n_hits) return;
    const bool ok = width_of_hit<T, true>(src, hit, p, reinterpret_cast<unsigned*>(out + hit * kWidthRowBytes));
    if (lane_id() == 0) valid[hit] = ok ? 1 : 0;
}

// wfb_waveform_width_run: a counting pass (which hits give a row), an inclusive scan of the counts, and the pass that
// writes every row at its place in hit order
template <typename T>
__global__ void __launch_bounds__(256) waveform_width_run_count_kernel(const WidthRunSrc<T> src, long long n_hits, const wfb_width_params p,
                                                                      long long* __restrict__ has_row) {
    const long long hit = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
    if (hit >= n_hits) return;
    const bool ok = width_of_hit<T, false>(src, hit, p, nullptr);
    if (lane_id() == 0) has_row[hit] = ok ? 1 : 0;
}

template <typename T>
__global__ void __launch_bounds__(256) waveform_width_run_kernel(const WidthRunSrc<T> src, long long n_hits, const wfb_width_params p,
                                                                const long long* __restrict__ has_row, const long long* __restrict__ row_incl,
                                                                uint8_t* __restrict__ out) {
    const long long hit = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
    if (hit >= n_hits || !has_row[hit]) return;
    width_of_hit<T, true>(src, hit, p, reinterpret_cast<unsigned*>(out + (row_incl[hit] - 1) * kWidthRowBytes));
}

// ---------------------------------------------------------------------------------------------
// waveform_width_integral: one THREAD per record, strictly sequential float64 arithmetic so the
// cumulative sums round exactly as np.cumsum and the total exactly as numpy's pairwise np.sum.
// ---------------------------------------------------------------------------------------------
template <typename T>
struct ChargeSrc {
    const T* w;
    double b;
    float b32;
    int mode;  // 0: unknown polarity (b - w in f64), 1: negative known (b32 - w in f32), 2: positive known,
               // 3: raw positive (w - b in f64; st_waveforms branch, waveform_width_integral.py:187-191)
    // one 16-byte chunk of the pool is kept in registers: a thread walks its record sequentially, so it issues
    // one load per 8 (uint16) / 4 (float32) samples instead of one per sample (32 sectors per warp load)
    const uint4* chunks;   // pool aligned down to 16 bytes
    long long first;       // element index of w[0] relative to `chunks`
    long long last;        // last chunk that may be read (the record's own last chunk)
    mutable long long cached;
    mutable uint4 q, qn;   // the current chunk and the one behind it, fetched one chunk ahead of its use
    __device__ __forceinline__ T sample(int i) const {
        constexpr int PER = 16 / (int)sizeof(T);
        const int e = (int)first + i;  // first < PER, i < 2^31 - PER
        const long long c = e / PER;
        if (c != cached) {
            q = (c == cached + 1) ? qn : __ldg(chunks + c);
            if (c + 1 <= last) qn = __ldg(chunks + c + 1);  // in flight while this chunk's samples are consumed
            cached = c;
        }
        const int k = e % PER;
        if (sizeof(T) == 2) {
            const unsigned word = (k < 4) ? ((k < 2) ? q.x : q.y) : ((k < 6) ? q.z : q.w);
            const unsigned short h = (unsigned short)(word >> ((k & 1) * 16));
            return *reinterpret_cast<const T*>(&h);
        }
        const unsigned word = (k < 2) ? ((k < 1) ? q.x : q.y) : ((k < 3) ? q.z : q.w);
        return *reinterpret_cast<const T*>(&word);
    }
    __device__ __forceinline__ double operator()(int i) const {
        const T wi = sample(i);
        double sig;
        if (mode == 0) sig = __dsub_rn(b, (double)wi);
        else if (mode == 1) sig = (double)__fsub_rn(b32, (float)wi);
        else if (mode == 2) sig = (double)__fsub_rn((float)wi, b32);
        else sig = __dsub_rn((double)wi, b);
        return (sig > 0.0 || isnan(sig)) ? sig : 0.0;  // np.maximum(sig, 0.0) keeps a NaN (fmax would drop it)
    }
};

// Fast path of waveform_width_integral for 16-bit samples whose record starts on a 16-byte boundary (every record of a
// fixed-length pool with L % 8 == 0): the SAME float64 operations in the SAME order as the generic path - numpy's pairwise
// np.sum (blocks of <= 128 with eight accumulators; every block starts at a multiple of eight) and the sequential
// np.cumsum - but eight samples come from one 16-byte load, the sample format and the polarity mode are resolved at
// compile time and nothing is indexed dynamically: ~9 instead of ~47 instructions per sample and pass.
template <typename T, int MODE>
struct ChargeTerm {
    double b;
    float b32;
    __device__ __forceinline__ double operator()(unsigned h) const {
        const T wi = (T)(unsigned short)h;  // uint16_t or short
        double sig;
        if (MODE == 0) sig = __dsub_rn(b, (double)wi);
        else if (MODE == 1) sig = (double)__fsub_rn(b32, (float)wi);
        else if (MODE == 2) sig = (double)__fsub_rn((float)wi, b32);
        else sig = __dsub_rn((double)wi, b);
        return fmax(sig, 0.0);
    }
    __device__ __forceinline__ void load8(const uint4* chunks, int i, double v[8]) const {  // samples i .. i + 7, i % 8 == 0
        const uint4 q = __ldg(chunks + (i >> 3));
        v[0] = (*this)(q.x & 0xffffu); v[1] = (*this)(q.x >> 16);
        v[2] = (*this)(q.y & 0xffffu); v[3] = (*this)(q.y >> 16);
        v[4] = (*this)(q.z & 0xffffu); v[5] = (*this)(q.z >> 16);
        v[6] = (*this)(q.w & 0xffffu); v[7] = (*this)(q.w >> 16);
    }
    __device__ __forceinline__ double at(const uint4* chunks, int i) const {
        const unsigned short* hw = reinterpret_cast<const unsigned short*>(chunks);
        return (*this)((unsigned)__ldg(hw + i));
    }
};

template <typename T, int MODE>
__device__ void width_integral_fast(const uint4* chunks, int L, const ChargeTerm<T, MODE> term, double q_low, double q_high, double& q_out,
                                    int& lo_out, int& hi_out) {
    // ---- q = np.sum: numpy's pairwise recursion, iterative (np_sum.cuh), blocks summed eight samples per load
    auto block = [&](int off, int len) -> double {
        if (len < 8) {
            double res = 0.0;
            for (int i = 0; i < len; ++i) res = __dadd_rn(res, term.at(chunks, off + i));
            return res;
        }
        double r[8], v[8];
        term.load8(chunks, off, r);
        int i;
        for (i = 8; i < len - (len % 8); i += 8) {
            term.load8(chunks, off + i, v);
#pragma unroll
            for (int k = 0; k < 8; ++k) r[k] = __dadd_rn(r[k], v[k]);
        }
        double res = __dadd_rn(__dadd_rn(__dadd_rn(r[0], r[1]), __dadd_rn(r[2], r[3])), __dadd_rn(__dadd_rn(r[4], r[5]), __dadd_rn(r[6], r[7])));
        for (; i < len; ++i) res = __dadd_rn(res, term.at(chunks, off + i));
        return res;
    };
    int st_off[24], st_len[24], st_state[24];
    double st_val[24];
    int sp = 0;
    st_off[0] = 0; st_len[0] = L; st_state[0] = 0;
    double ret = 0.0;
    while (sp >= 0) {
        const int off = st_off[sp], len = st_len[sp];
        if (st_state[sp] == 0) {
            if (len <= 128) {
                ret = block(off, len);
                --sp;
            } else {
                int n2 = len / 2;
                n2 -= n2 % 8;
                st_state[sp] = 1;
                ++sp;
                st_off[sp] = off; st_len[sp] = n2; st_state[sp] = 0;
            }
        } else if (st_state[sp] == 1) {
            int n2 = len / 2;
            n2 -= n2 % 8;
            st_val[sp] = ret;
            st_state[sp] = 2;
            ++sp;
            st_off[sp] = off + n2; st_len[sp] = len - n2; st_state[sp] = 0;
        } else {
            ret = __dadd_rn(st_val[sp], ret);
            --sp;
        }
    }
    const double q = ret;
    q_out = q;
    lo_out = hi_out = 0;
    if (!(q > 0.0 && isfinite(q))) return;
    // ---- np.cumsum + searchsorted(..., 'left'): the first index whose cumulative sum reaches the target
    const double tl = __dmul_rn(q_low, q), th = __dmul_rn(q_high, q);
    int lo = L, hi = L;
    bool fl = false, fh = false;
    double cs = 0.0;
    int i = 0;
    for (; i + 8 <= L && !fh; i += 8) {
        double v[8];
        term.load8(chunks, i, v);
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            cs = (i + k == 0) ? v[0] : __dadd_rn(cs, v[k]);
            if (!fl && cs >= tl) { lo = i + k; fl = true; }
            if (!fh && cs >= th) { hi = i + k; fh = true; }
        }
    }
    for (; i < L && !fh; ++i) {
        cs = (i == 0) ? term.at(chunks, 0) : __dadd_rn(cs, term.at(chunks, i));
        if (!fl && cs >= tl) { lo = i; fl = true; }
        if (!fh && cs >= th) { hi = i; fh = true; }
    }
    lo_out = lo;
    hi_out = hi;
}

template <typename T>
__global__ void __launch_bounds__(128) width_integral_kernel(const T* __restrict__ pool, long long pool_len,
                                                            const wfb_rec_meta* __restrict__ meta, long long n,
                                                            double q_low, double q_high, double dt, long long pool_base,
                                                            long long row_base, uint8_t* __restrict__ out) {
    const long long rec = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (rec >= n) return;
    const wfb_rec_meta m = meta[rec];
    long long off = m.wave_offset - pool_base;
    int L = m.event_length;
    if (L < 0 || off < 0 || off + L > pool_len) L = 0;
    ChargeSrc<T> x;
    x.w = pool + off;
    {
        constexpr int PER = 16 / (int)sizeof(T);
        const uintptr_t addr = reinterpret_cast<uintptr_t>(pool + off);
        x.chunks = reinterpret_cast<const uint4*>(addr & ~(uintptr_t)15);
        x.first = (long long)((addr & 15) / sizeof(T));
        x.cached = -2;  // neither this chunk nor its predecessor is in registers
        x.q = make_uint4(0u, 0u, 0u, 0u);
        x.qn = x.q;
        x.last = (L > 0) ? (x.first + L - 1) / PER : -1;
    }
    x.b = m.baseline;
    x.b32 = (float)m.baseline;
    x.mode = m.polarity == WFB_POL_NEGATIVE ? 1 : (m.polarity == WFB_POL_POSITIVE ? 2 : (m.polarity == WFB_POL_RAW_POSITIVE ? 3 : 0));
    double q = 0.0;
    int lo = 0, hi = 0;
    bool done = false;
    if (L > 0 && isnan(m.baseline)) {  // every signal sample is NaN: np.sum is NaN, the quantile indices stay 0
        q = __longlong_as_double(0x7ff8000000000000ll);
        done = true;
    }
    if constexpr (sizeof(T) == 2) {
        if (!done && L >= 8 && (reinterpret_cast<uintptr_t>(pool + off) & 15) == 0) {
            const uint4* ch = reinterpret_cast<const uint4*>(pool + off);
            switch (x.mode) {
                case 0: width_integral_fast<T, 0>(ch, L, ChargeTerm<T, 0>{x.b, x.b32}, q_low, q_high, q, lo, hi); break;
                case 1: width_integral_fast<T, 1>(ch, L, ChargeTerm<T, 1>{x.b, x.b32}, q_low, q_high, q, lo, hi); break;
                case 2: width_integral_fast<T, 2>(ch, L, ChargeTerm<T, 2>{x.b, x.b32}, q_low, q_high, q, lo, hi); break;
                default: width_integral_fast<T, 3>(ch, L, ChargeTerm<T, 3>{x.b, x.b32}, q_low, q_high, q, lo, hi); break;
            }
            done = true;
        }
    }
    if (!done) q = numpy_pairwise_sum(x, L);
    if (!done && q > 0.0 && isfinite(q)) {
        const double tl = __dmul_rn(q_low, q), th = __dmul_rn(q_high, q);
        lo = hi = L;  // searchsorted returns len when no element reaches the target
        bool fl = false, fh = false;
        double cs = 0.0;
        for (int i = 0; i < L; ++i) {
            cs = (i == 0) ? x(0) : __dadd_rn(cs, x(i));
            if (!fl && cs >= tl) { lo = i; fl = true; }
            if (!fh && cs >= th) { hi = i; fh = true; break; }
        }
    }
    const double ws = (double)max(hi - lo, 0);
    unsigned* dst = reinterpret_cast<unsigned*>(out + rec * kWidthIntRowBytes);
    dst[0] = __float_as_uint((float)__dmul_rn((double)lo, dt));
    dst[1] = __float_as_uint((float)__dmul_rn((double)hi, dt));
    dst[2] = __float_as_uint((float)__dmul_rn(ws, dt));
    dst[3] = __float_as_uint((float)lo);
    dst[4] = __float_as_uint((float)hi);
    dst[5] = __float_as_uint((float)ws);
    const long long qb = __double_as_longlong(q);
    dst[6] = (unsigned)(qb & 0xffffffffll);
    dst[7] = (unsigned)((unsigned long long)qb >> 32);
    dst[8] = (unsigned)(m.timestamp & 0xffffffffll);
    dst[9] = (unsigned)((unsigned long long)m.timestamp >> 32);
    dst[10] = ((unsigned)(unsigned short)m.board) | ((unsigned)(unsigned short)m.channel << 16);
    const long long ev = row_base + rec;
    dst[11] = (unsigned)(ev & 0xffffffffll);
    dst[12] = (unsigned)((unsigned long long)ev >> 32);
}

}  // namespace wfb

using namespace wfb;

extern "C" int wfb_waveform_width(const void* waves_dev, int64_t n_waves, int32_t length, int64_t stride,
                                  const int64_t* hit_row_dev, const int64_t* hit_position_dev,
                                  const int64_t* hit_timestamp_dev, const int16_t* hit_board_dev,
                                  const int16_t* hit_channel_dev, const int64_t* hit_record_id_dev, int64_t n_hits,
                                  const wfb_width_params* params, void* out_dev, uint8_t* valid_dev, void* stream) {
    WFB_REQUIRE(params != nullptr, "wfb_waveform_width: params is NULL");
    WFB_REQUIRE(n_hits >= 0 && n_waves >= 0 && length >= 0, "wfb_waveform_width: negative size");
    if (n_hits == 0) return WFB_OK;
    WFB_REQUIRE(hit_row_dev && hit_position_dev && hit_timestamp_dev && hit_channel_dev && hit_record_id_dev && out_dev && valid_dev,
                "wfb_waveform_width: NULL pointer");
    WFB_REQUIRE(params->sampling_rate != 0.0, "wfb_waveform_width: sampling_rate is 0");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const unsigned blocks = (unsigned)((n_hits * 32 + 255) / 256);
    const long long* row = reinterpret_cast<const long long*>(hit_row_dev);
    const long long* pos = reinterpret_cast<const long long*>(hit_position_dev);
    const long long* ts = reinterpret_cast<const long long*>(hit_timestamp_dev);
    const long long* rid = reinterpret_cast<const long long*>(hit_record_id_dev);
    if (params->wave_is_f32)
        waveform_width_kernel<float><<<blocks, 256, 0, st>>>(
            WidthRowsSrc<float>{static_cast<const float*>(waves_dev), n_waves, length, stride, row, pos, ts, hit_board_dev, hit_channel_dev, rid},
            n_hits, *params, static_cast<uint8_t*>(out_dev), valid_dev);
    else
        waveform_width_kernel<short><<<blocks, 256, 0, st>>>(
            WidthRowsSrc<short>{static_cast<const short*>(waves_dev), n_waves, length, stride, row, pos, ts, hit_board_dev, hit_channel_dev, rid},
            n_hits, *params, static_cast<uint8_t*>(out_dev), valid_dev);
    WFB_CUDA(cudaGetLastError());
    return WFB_OK;
}

static size_t wr_al256(size_t x) { return (x + 255) & ~(size_t)255; }

extern "C" size_t wfb_waveform_width_run_workspace_bytes(int64_t n_hits) {
    const size_t m = wr_al256((size_t)std::max<int64_t>(n_hits, 1) * 8);
    return 2 * m + scan_workspace_bytes(n_hits);
}

template <typename T>
static void launch_width_run(const WidthRunSrc<T>& src, long long n_hits, const wfb_width_params& p, long long* has_row, long long* incl,
                             void* scan_ws, uint8_t* out, int* rc, cudaStream_t st) {
    const unsigned blocks = (unsigned)((n_hits * 32 + 255) / 256);
    waveform_width_run_count_kernel<T><<<blocks, 256, 0, st>>>(src, n_hits, p, has_row);
    *rc = inclusive_scan_sum_i64(has_row, incl, n_hits, scan_ws, st);
    if (*rc != WFB_OK) return;
    waveform_width_run_kernel<T><<<blocks, 256, 0, st>>>(src, n_hits, p, has_row, incl, out);
}

extern "C" int wfb_waveform_width_run(const void* pool_dev, int32_t pool_is_f32, int64_t pool_len, const wfb_rec_meta* meta_dev,
                                      int64_t n, int64_t pool_base, int64_t row_base, const void* hits_dev, int64_t n_hits,
                                      const wfb_width_params* params, void* out_dev, int64_t* n_out_dev, void* workspace_dev,
                                      size_t workspace_bytes, void* stream) {
    WFB_REQUIRE(params != nullptr && n_out_dev != nullptr, "wfb_waveform_width_run: NULL params / count");
    WFB_REQUIRE(n_hits >= 0 && n >= 0 && pool_len >= 0, "wfb_waveform_width_run: negative size");
    WFB_REQUIRE(pool_is_f32 == 0 || pool_is_f32 == 1, "wfb_waveform_width_run: pool_is_f32 must be 0 or 1, got %d", pool_is_f32);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (n_hits == 0) {
        WFB_CUDA(cudaMemsetAsync(n_out_dev, 0, 8, st));
        return WFB_OK;
    }
    WFB_REQUIRE(hits_dev && out_dev && workspace_dev && (meta_dev || n == 0) && (pool_dev || pool_len == 0),
                "wfb_waveform_width_run: NULL pointer");
    WFB_REQUIRE(((uintptr_t)hits_dev & 3) == 0, "wfb_waveform_width_run: hit rows must be 4-byte aligned");
    WFB_REQUIRE(params->sampling_rate != 0.0, "wfb_waveform_width_run: sampling_rate is 0");
    WFB_REQUIRE(workspace_bytes >= wfb_waveform_width_run_workspace_bytes(n_hits), "wfb_waveform_width_run: workspace too small");
    uint8_t* ws = static_cast<uint8_t*>(workspace_dev);
    const size_t m = wr_al256((size_t)n_hits * 8);
    long long* has_row = reinterpret_cast<long long*>(ws);
    long long* incl = reinterpret_cast<long long*>(ws + m);
    void* scan_ws = ws + 2 * m;
    const unsigned* hits = static_cast<const unsigned*>(hits_dev);
    uint8_t* out = static_cast<uint8_t*>(out_dev);
    int rc = WFB_OK;
    if (pool_is_f32)
        launch_width_run(WidthRunSrc<float>{static_cast<const float*>(pool_dev), pool_len, meta_dev, n, pool_base, row_base, hits}, n_hits, *params,
                         has_row, incl, scan_ws, out, &rc, st);
    else
        launch_width_run(WidthRunSrc<short>{static_cast<const short*>(pool_dev), pool_len, meta_dev, n, pool_base, row_base, hits}, n_hits, *params,
                         has_row, incl, scan_ws, out, &rc, st);
    if (rc != WFB_OK) return rc;
    WFB_CUDA(cudaMemcpyAsync(n_out_dev, incl + n_hits - 1, 8, cudaMemcpyDeviceToDevice, st));
    WFB_CUDA(cudaGetLastError());
    return WFB_OK;
}

extern "C" int wfb_width_integral(const void* pool_dev, int32_t pool_is_f32, int64_t pool_len, const wfb_rec_meta* meta_dev,
                                  int64_t n, double q_low, double q_high, double dt_ns, int64_t pool_base, int64_t row_base,
                                  void* out_dev, void* stream) {
    WFB_REQUIRE(n >= 0 && pool_len >= 0, "wfb_width_integral: negative size");
    WFB_REQUIRE(q_low > 0 && q_high < 1 && q_low < q_high, "q_low/q_high invalid: q_low=%g, q_high=%g", q_low, q_high);
    if (n == 0) return WFB_OK;
    WFB_REQUIRE(meta_dev && out_dev, "wfb_width_integral: NULL pointer");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const unsigned blocks = (unsigned)((n + 127) / 128);
    if (pool_is_f32 == 1)
        width_integral_kernel<float><<<blocks, 128, 0, st>>>(static_cast<const float*>(pool_dev), pool_len, meta_dev, n, q_low, q_high,
                                                           dt_ns, pool_base, row_base, static_cast<uint8_t*>(out_dev));
    else if (pool_is_f32 == 2)  // int16 samples (structured st_waveforms rows used in place)
        width_integral_kernel<short><<<blocks, 128, 0, st>>>(static_cast<const short*>(pool_dev), pool_len, meta_dev, n, q_low, q_high,
                                                           dt_ns, pool_base, row_base, static_cast<uint8_t*>(out_dev));
    else
        width_integral_kernel<uint16_t><<<blocks, 128, 0, st>>>(static_cast<const uint16_t*>(pool_dev), pool_len, meta_dev, n, q_low,
                                                              q_high, dt_ns, pool_base, row_base, static_cast<uint8_t*>(out_dev));
    WFB_CUDA(cudaGetLastError());
    return WFB_OK;
}
