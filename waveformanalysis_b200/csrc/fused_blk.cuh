// Block-granular hit machinery of the lane-per-record kernel (included by fused_lpr.cu after the
// shared structs; uses WarpHits, LaneRec, FeatState, Ring and the sinks defined there).
//
// The streaming lane looks at its record 32 samples (one BLOCK = four 16-byte chunks) at a time.
// One packed min / max tree over the sixteen words classifies the block: QUIET (nothing above
// threshold), FULL (everything above) or MIXED.  Only blocks in which a run starts or ends are
// ITEMS: a MIXED block, a FULL block that follows a sample below threshold (a run starts with
// its first sample) and a QUIET block that follows a sample above threshold (the run ends with
// the block's first sample).  FULL blocks inside a run only update a per-lane aggregate (first
// minimum key and its block, sum) that travels with the owner's next item.
//
// An item is COPIED into a 64-slot per-warp ring in shared memory: the block's 64 bytes, the last
// word of the block in front (left extension), the first word of the block behind (right extension;
// written one step later, an item is complete once its owner has seen the next block) and the
// aggregate of the FULL blocks in front.  When 32 complete items wait, the warp runs a DENSE ROUND:
// lane t takes item t whoever owns it, builds the 32-bit above-threshold mask of the block with
// packed compares, and walks the runs of the block with bit operations; a run that is still open at
// the block end is staged and handed to the owner's next item (same round: through the stage rows;
// later rounds: through the per-owner carry).  Nothing is re-read from global memory except the one
// FULL block that holds a run's minimum when its position is needed.
//
// Semantics are those of lpr_round / hit_finder.py:329-413: runs of samples with key <= kmax, window
// [max(0, s - left), min(lmax, e + right)), first arg-min of the key inside the window, count and key
// sum of the samples on the signal side of the baseline; samples past the record end inside the window
// take the padding value (a true 0).  Extensions of at most two samples (the default is two).
#pragma once

namespace wfb {

constexpr int kBQRing = 64;    // item slots per warp: < 32 complete items + <= 32 pushed in the current step
#ifndef WFB_BQ_WORDS
#define WFB_BQ_WORDS 27
#endif
constexpr int kBQWords = WFB_BQ_WORDS;  // 32-bit words per slot; odd, so that the lanes' scalar accesses fall into distinct banks
constexpr int kBQPark = (kBQWords - 19) / 2;  // {key, sum} pairs of ended runs a slot can park (words 19 ..)
static_assert(kBQWords % 2 == 1 && kBQPark >= 1, "slot size");
// slot words: 0 last word of the previous block, 1..16 the block (offset-domain samples), 17 first word of the next
// block, 18 owner | block << 5, 19 first-minimum key of the FULL blocks in front (key << 16 | block) or ~0, 20 their
// raw sample sum; 19 .. 26 are reused by the round for the {key, sum} pairs of up to four runs that end in the block.
// As half-words: sample j of the block (j = -2 .. 33) sits at j + 2.
constexpr int kBQMaxExt = 2;

// bit j <=> (half-word j of d0..d3, xor cx) < k1; k1k1 = k1 | k1 << 16 with 1 <= k1 <= 65535
__device__ __forceinline__ unsigned lt_mask32(const uint4& d0, const uint4& d1, const uint4& d2, const uint4& d3, unsigned cx32, unsigned k1k1) {
    auto w2 = [&](unsigned w) {  // 1 per half-word that is below k1
        const unsigned t = __vminu2(w ^ cx32, k1k1);
        return __vminu2(k1k1 - t, 0x00010001u);
    };
    auto c8 = [&](const uint4& d) {
        unsigned m = __dp2a_lo(w2(d.w), 0x8040u, 0u);
        m = __dp2a_lo(w2(d.z), 0x2010u, m);
        m = __dp2a_lo(w2(d.y), 0x0804u, m);
        return __dp2a_lo(w2(d.x), 0x0201u, m);
    };
    return c8(d0) | (c8(d1) << 8) | (c8(d2) << 16) | (c8(d3) << 24);
}

// ---- dense round: lane t walks the runs of queued block item t -----------------------------------
// Fast path (thresholds >= 0): ONE unrolled, branch-free pass over the 32 positions keeps the running first-minimum
// key and sample sum of the current run in two registers; where a run ends the pair is parked in the item's own slot
// (its header words are in registers by then), so the per-run work that remains is a short loop over ENDED runs:
// extension samples, the carried-in fragment of the first one, the row entry.  A negative threshold (FULL blocks are
// items then, a run can cross a whole block) takes the general walker with per-sample loops.
template <typename Sink>
__device__ __forceinline__ void blk_round(WarpHits& ws, unsigned* bq, int qh, int qn, const LaneRec& r, const FHArgs& a, Sink& sink) {
    __syncwarp();  // pushes and completions are visible
    const int lane = lane_id();
    const bool act = lane < qn;
    unsigned* sl = bq + ((qh + (act ? lane : 0)) & (kBQRing - 1)) * kBQWords;
    const unsigned hdr = sl[18], fa_key = sl[19], fa_sum = sl[20];  // owner | block << 5, FULL key, FULL sum
    const unsigned prev_w = sl[0];
    const unsigned short* hw = reinterpret_cast<const unsigned short*>(sl) + 2;  // hw[j]: sample j of the block, j = -2 .. 33
    const int src = act ? (int)(hdr & 31u) : lane;  // owner lane
    const int B = (int)(hdr >> 5);
    // the owner's record constants
    const int o_kmax = __shfl_sync(kFull, r.kmax, src);
    const int o_mis = __shfl_sync(kFull, r.mis, src);
    const int o_len = __shfl_sync(kFull, r.len, src);
    const int o_wlim = __shfl_sync(kFull, r.wlim, src);
    const unsigned o_flags = __shfl_sync(kFull, (r.positive ? 1u : 0u) | (r.degen ? 2u : 0u), src);
    const bool o_pos = (o_flags & 1u) != 0u;
    const long long o_off = bcast_i64(r.off, src);
    sink.prepare(src, r);
    const int bias = r.bias;                       // uniform
    const unsigned cx = o_pos ? 0xffffu : 0u;      // offset-domain sample -> key
    const unsigned cx32 = cx | (cx << 16);
    const int padkv = o_pos ? 65535 - bias : bias;                    // key of a padding sample (true 0)
    const int kin = o_pos ? 65535 - (o_wlim + bias) : o_wlim + bias;  // signal side <=> key <= kin
    const int left = a.p.left_extension, right = a.p.right_extension;
    const int i0 = 32 * B - o_mis;  // record index of the block's first sample
    // positions of the block that belong to the record
    const int vlo = max(0, -i0), vhi = min(32, o_len - i0);
    unsigned vmask = 0u;
    if (act && vhi > vlo) vmask = (vhi >= 32 ? 0xffffffffu : ((1u << vhi) - 1u)) & ~((1u << vlo) - 1u);
    // does a run come in (the sample in front of the block is above threshold)?
    const bool in_open = act && i0 >= 1 && i0 - 1 < o_len && (int)((prev_w >> 16) ^ cx) <= o_kmax;
    const bool slow = __any_sync(kFull, act && ((o_flags & 2u) != 0u || o_kmax >= 65535));

    // one sample of the window by its position relative to the block (-2 .. 33)
    auto add_sample = [&](int rel, unsigned& key, unsigned& cnt, unsigned& skv) {
        const int i = i0 + rel;
        const int kv = (i < o_len) ? (int)((unsigned)hw[rel] ^ cx) : padkv;
        key = min(key, ((unsigned)kv << 16) + (unsigned)i);
        if (kv <= kin) { cnt += 1u; skv += (unsigned)kv; }
    };
    // an extension sample with key kv at block position rel
    auto ext_sample = [&](int rel, int kv, unsigned& key, unsigned& cnt, unsigned& skv) {
        key = min(key, ((unsigned)kv << 16) + (unsigned)(i0 + rel));
        if (kv <= kin) { cnt += 1u; skv += (unsigned)kv; }
    };
    // samples [ja, jb) of the block, all inside the record
    auto add_core = [&](int ja, int jb, unsigned& key, unsigned& cnt, unsigned& skv) {
        unsigned ki = (unsigned)(i0 + ja);
        for (int j = ja; j < jb; ++j, ++ki) {
            const unsigned kv = (unsigned)hw[j] ^ cx;
            key = min(key, (kv << 16) + ki);
            if ((int)kv <= kin) { cnt += 1u; skv += kv; }
        }
    };
    // the fragment carried in by the owner's previous item, with the FULL blocks between the two items
    auto carried_in = [&](unsigned ltp) {
        uint4 prev = ltp ? ws.stage[31 - __clz(ltp)] : ws.carry[src];
        if (fa_key != 0xffffffffu) {
            const unsigned fkv = fa_key >> 16;
            const int fb = (int)(fa_key & 0xffffu);
            const int bs = ((int)prev.x + o_mis) >> 5;  // block in which the run started
            const unsigned nfull = 32u * (unsigned)(B - bs - 1);
            if (fkv < (prev.y >> 16)) {  // the minimum lies in a FULL block: find its first position (L2)
                const uint4* g = reinterpret_cast<const uint4*>(static_cast<const uint16_t*>(a.pool) + (o_off - o_mis) + 32ll * fb);
                const uint4 g0 = __ldg(g), g1 = __ldg(g + 1), g2 = __ldg(g + 2), g3 = __ldg(g + 3);
                const unsigned cxr = (bias ? 0x8000u : 0u) ^ cx;
                unsigned eq = 0xffffffffu;
                if (fkv < 65535u) eq = lt_mask32(g0, g1, g2, g3, cxr | (cxr << 16), (fkv + 1u) | ((fkv + 1u) << 16));
                prev.y = (fkv << 16) + (unsigned)(32 * fb - o_mis + __ffs(eq) - 1);
            }
            prev.z += nfull;
            prev.w += o_pos ? nfull * 65535u - fa_sum : fa_sum;
        }
        return prev;
    };

    if (!slow) {
        // ---------------- fast path ----------------
        unsigned kvp[16];
#pragma unroll
        for (int w = 0; w < 16; ++w) kvp[w] = sl[1 + w] ^ cx32;
        if (__any_sync(kFull, vmask != 0xffffffffu)) {  // record start / end (or an idle lane): positions outside never count
#pragma unroll
            for (int w = 0; w < 16; ++w) {
                const unsigned b2 = (vmask >> (2 * w)) & 3u;
                kvp[w] |= ~((b2 & 1u) * 0xffffu + (b2 >> 1) * 0xffff0000u);
            }
        }
        unsigned* fst = sl + 19;  // kBQPark parked {key, sum} pairs: words 19 .. (the last one is overwritten by later runs)
        unsigned key = 0xffffffffu, sum = 0u, m32 = 0u;
        int nf = 0;  // runs that ended so far
        bool pprev = in_open;
#pragma unroll
        for (int j = 0; j < 32; ++j) {
            const unsigned kv = (j & 1) ? (kvp[j >> 1] >> 16) : (kvp[j >> 1] & 0xffffu);
            const bool p = (int)kv <= o_kmax;
            if (pprev && !p) {  // a run ended in front of j: park it (the fourth slot is overwritten by later ones)
                unsigned* f = fst + 2 * min(nf, kBQPark - 1);
                f[0] = key;
                f[1] = sum;
                ++nf;
                key = 0xffffffffu;
                sum = 0u;
            }
            if (p) {
                key = min(key, (kv << 16) + (unsigned)j);
                sum += kv;
                m32 |= 1u << j;
            }
            pprev = p;
        }
        const unsigned starts = m32 & ~((m32 << 1) | (in_open ? 1u : 0u));
        const int nstarts = __popc(starts);
        const bool has_trail = (m32 >> 31) != 0u;  // a run is still open at the block end
        ws.stage_n[lane] = nstarts;
        const unsigned peers = __match_any_sync(kFull, act ? src : 32 + lane);
        const unsigned ltp = peers & ((1u << lane) - 1u);
        __syncwarp();  // stage_n, and the parked pairs of this lane
        int ord_base = act ? ws.carry_n[src] : 0;  // runs of the record started in front of this item
        for (unsigned m = ltp; m; m &= m - 1) ord_base += ws.stage_n[__ffs(m) - 1];
        if (has_trail) {  // staged for the owner's next item (key and sum are those of the trailing run)
            const int js_tr = 32 - __clz(~m32);
            const int s_tr = i0 + js_tr;
            unsigned tkey = key + (unsigned)i0, cnt = (unsigned)(32 - js_tr), skv = sum;
            if (left >= 1 && s_tr >= 1) ext_sample(js_tr - 1, (int)((unsigned)hw[js_tr - 1] ^ cx), tkey, cnt, skv);
            if (left >= 2 && s_tr >= 2) ext_sample(js_tr - 2, (int)((unsigned)hw[js_tr - 2] ^ cx), tkey, cnt, skv);
            ws.stage[lane] = make_uint4((unsigned)s_tr, tkey, cnt, skv);
        }
        __syncwarp();
        unsigned em = ~m32 & ((m32 << 1) | (in_open ? 1u : 0u));  // bit j: a run ended in front of position j
        unsigned sm = starts;
        for (int k = 0; em; ++k) {
            const int je = __ffs(em) - 1;
            em &= em - 1u;
            const bool lead = in_open && k == 0;
            int js = 0;
            if (!lead) {
                js = __ffs(sm) - 1;
                sm &= sm - 1u;
            }
            unsigned hkey = 0xffffffffu, cnt = 0u, skv = 0u;
            if (k < kBQPark - 1 || (k == kBQPark - 1 && nf <= kBQPark)) {
                if (je > js) {  // (an incoming run that ends with the block's first sample has no sample here)
                    hkey = fst[2 * k] + (unsigned)i0;
                    skv = fst[2 * k + 1];
                    cnt = (unsigned)(je - js);
                }
            } else {
                add_core(js, je, hkey, cnt, skv);
            }
            int s = i0 + js, ord = ord_base + k - (in_open ? 1 : 0);
            if (lead) {
                const uint4 prev = carried_in(ltp);
                s = (int)prev.x;
                hkey = min(hkey, prev.y);
                cnt += prev.z;
                skv += prev.w;
            } else {  // left extension: the samples in front of the run belong to the record
                if (left >= 1 && s >= 1) ext_sample(js - 1, (int)((unsigned)hw[js - 1] ^ cx), hkey, cnt, skv);
                if (left >= 2 && s >= 2) ext_sample(js - 2, (int)((unsigned)hw[js - 2] ^ cx), hkey, cnt, skv);
            }
            const int e = i0 + je;
            if (right >= 1 && e < a.lmax) ext_sample(je, e < o_len ? (int)((unsigned)hw[je] ^ cx) : padkv, hkey, cnt, skv);
            if (right >= 2 && e + 1 < a.lmax) ext_sample(je + 1, e + 1 < o_len ? (int)((unsigned)hw[je + 1] ^ cx) : padkv, hkey, cnt, skv);
            sink.store((int)(hkey & 0xffffu), s, e, (int)(hkey >> 16), cnt, o_pos ? cnt * 65535u - skv : skv, ord, src, a);
        }
        __syncwarp();  // every read of stage / carry is done
        if (act && !(peers >> lane >> 1)) {  // the last item of this owner in the round
            if (has_trail) ws.carry[src] = ws.stage[lane];
            ws.carry_n[src] = ord_base + nstarts;
        }
        __syncwarp();
        return;
    }

    // ---------------- general walker ----------------
    const uint4 d0 = make_uint4(sl[1], sl[2], sl[3], sl[4]), d1 = make_uint4(sl[5], sl[6], sl[7], sl[8]);
    const uint4 d2 = make_uint4(sl[9], sl[10], sl[11], sl[12]), d3 = make_uint4(sl[13], sl[14], sl[15], sl[16]);
    const unsigned k1 = (unsigned)min(max(o_kmax + 1, 1), 65535);
    const unsigned lt = lt_mask32(d0, d1, d2, d3, cx32, k1 | (k1 << 16));
    const unsigned m32 = (o_kmax >= 65535) ? vmask : ((o_kmax >= 0) ? (lt & vmask) : 0u);
    const unsigned starts = m32 & ~((m32 << 1) | (in_open ? 1u : 0u));
    const int nstarts = __popc(starts);
    const bool has_trail = (m32 >> 31) != 0u;  // a run is still open at the block end
    ws.stage_n[lane] = nstarts;
    const unsigned peers = __match_any_sync(kFull, act ? src : 32 + lane);
    const unsigned ltp = peers & ((1u << lane) - 1u);
    __syncwarp();
    int ord_base = act ? ws.carry_n[src] : 0;  // runs of the record started in front of this item
    for (unsigned m = ltp; m; m &= m - 1) ord_base += ws.stage_n[__ffs(m) - 1];
    // the run still open at the block end: staged for the owner's next item.  A block that a run crosses
    // from end to end has to wait for the fragment in front of it.
    int js_tr = 32;
    bool passthru = false;
    if (has_trail) {
        js_tr = 32 - __clz(~m32);  // first sample of the trailing run (0: the whole block)
        passthru = in_open && js_tr == 0;
        unsigned key = 0xffffffffu, cnt = 0u, skv = 0u;
        const int s_tr = i0 + js_tr;
        if (!passthru)
            for (int x = min(left, s_tr); x >= 1; --x) add_sample(js_tr - x, key, cnt, skv);
        add_core(js_tr, 32, key, cnt, skv);
        ws.stage[lane] = make_uint4(passthru ? 0xffffffffu : (unsigned)s_tr, key, cnt, skv);
    }
    __syncwarp();
    {
        bool pending = passthru;
        while (__any_sync(kFull, pending)) {
            uint4 pv = make_uint4(0u, 0u, 0u, 0u);
            bool ready = false;
            if (pending) {
                pv = ltp ? ws.stage[31 - __clz(ltp)] : ws.carry[src];
                ready = pv.x != 0xffffffffu;
            }
            __syncwarp();
            if (pending && ready) {
                const uint4 own = ws.stage[lane];
                ws.stage[lane] = make_uint4(pv.x, min(pv.y, own.y), pv.z + own.z, pv.w + own.w);
                pending = false;
            }
            __syncwarp();
        }
    }
    // the run that comes in and ends in this block
    unsigned mm = m32;
    if (in_open && !passthru) {
        const uint4 prev = carried_in(ltp);
        const int t0 = __ffs(~m32) - 1;  // the run ends at the first position that is not above threshold
        unsigned key = prev.y, cnt = prev.z, skv = prev.w;
        add_core(0, t0, key, cnt, skv);
        const int e = i0 + t0;
        for (int x = 0; x < right; ++x)
            if (e + x < a.lmax) add_sample(t0 + x, key, cnt, skv);
        sink.store((int)(key & 0xffffu), (int)prev.x, e, (int)(key >> 16), cnt, o_pos ? cnt * 65535u - skv : skv, ord_base - 1, src, a);
        mm &= ~((1u << t0) - 1u);
    }
    if (has_trail) mm &= (js_tr > 0) ? ((1u << js_tr) - 1u) : 0u;  // the trailing run is staged, not finished here
    // runs that start and end in this block
    for (int k = 0; mm; ++k) {
        const int js = __ffs(mm) - 1;
        const int je = js + __ffs(~(mm >> js)) - 1;  // <= 31: the trailing run is gone
        const int s = i0 + js, e = i0 + je;
        unsigned key = 0xffffffffu, cnt = 0u, skv = 0u;
        for (int x = min(left, s); x >= 1; --x) add_sample(js - x, key, cnt, skv);
        add_core(js, je, key, cnt, skv);
        for (int x = 0; x < right; ++x)
            if (e + x < a.lmax) add_sample(je + x, key, cnt, skv);
        sink.store((int)(key & 0xffffu), s, e, (int)(key >> 16), cnt, o_pos ? cnt * 65535u - skv : skv, ord_base + k, src, a);
        mm &= ~((1u << je) - 1u);
    }
    __syncwarp();  // every read of stage / carry is done
    if (act && !(peers >> lane >> 1)) {  // the last item of this owner in the round
        if (has_trail) ws.carry[src] = ws.stage[lane];
        ws.carry_n[src] = ord_base + nstarts;
    }
    __syncwarp();
}

// ---- stream one record per lane through the slot ring, block items ---------------------------------
template <bool FEAT, bool SGN, typename Sink>
__device__ __forceinline__ void blk_stream(const FHArgs& a, const uint16_t* pool, const LaneRec& r, int sc, const Ring& ring,
                                           int p0, int p1, int c0, int c1, FeatState& fs, WarpHits& ws, unsigned* bq, Sink& sink) {
    const int lane = lane_id();
    const int mis = r.mis, vtotal = r.mis + r.len;
    const int nch = (r.len > 0) ? ((vtotal + 7) >> 3) : 0;
    const int nch_max = __reduce_max_sync(kFull, nch);
    // one block past the longest record of the warp: it completes the last items and closes runs that reach the record end
    const int nblk = (nch_max > 0) ? ((nch_max + 3) >> 2) + 1 : 0;
    const int bps = sc >> 2;  // blocks per segment
    const int nseg = (nblk + bps - 1) / bps;
    const bool known = r.pol == WFB_POL_POSITIVE || r.pol == WFB_POL_NEGATIVE;
    const float b32 = (float)r.b_feat;
    // Block ranges of the record, computed once.  Block B holds 32 samples of the record iff 0 <= 32 B - mis <= len - 32;
    // the blocks of [f0, f0 + fn0) and [f1, f1 + fn1) also take the straight feature path (whole chunks inside the area
    // slice, none in the height slice, unknown polarity).  A test is one unsigned compare: in front of a range the
    // difference wraps above its length.
    const unsigned whn = (unsigned)max(0, r.len - 31);
    int f0 = 0, f1 = 0;
    unsigned fn0 = 0u, fn1 = 0u;
    if (FEAT && r.len > 0 && !known) {
        const int wh0 = (((mis + 7) >> 3) + 3) >> 2, wh1 = (vtotal >> 3) >> 2;  // the blocks of 32 record samples
        const int lo = max(wh0, (((mis + max(c0, 1) + 7) >> 3) + 3) >> 2);
        const int hi = min(wh1, ((mis + min(c1, r.len)) >> 3) >> 2);
        const int ha = (p1 > p0) ? ((mis + p0) >> 3) >> 2 : 0;                // blocks in front of the height slice
        const int hb = (p1 > p0) ? (((mis + p1 + 7) >> 3) + 3) >> 2 : 0;      // blocks behind it
        f0 = lo;
        fn0 = (unsigned)max(0, min(hi, ha) - lo);
        f1 = max(lo, hb);
        fn1 = (unsigned)max(0, hi - f1);
    }
    const unsigned xm16 = r.positive ? 0xffffu : 0u;
    const int kfull = r.degen ? -1 : r.kmax;    // a block is FULL <=> its largest key <= kfull (never with a negative threshold)
    // hit state of the lane
    bool open = false;                          // the last sample of the previous block is above threshold
    unsigned fa_key = 0xffffffffu, fa_sum = 0u; // FULL blocks since the lane's last item
    unsigned hprev = 0u;                        // last word of the previous block
    int myslot = -1;                            // word 17 of the item pushed in the previous step (waits for its next word)
    int qn_c = 0, qn_i = 0, qh = 0;             // complete / incomplete items, ring head (warp-uniform)

    auto issue = [&](int s) {
        const int b = s % kNBuf;
        const int cb = s * sc;
        const int clo = cb, chi = min(nch, (s + 1) * sc);
        const unsigned bytes = chi > clo ? (unsigned)(chi - clo) * 16u : 0u;
        fence_proxy_async();
        if (ring.use2d) {
            __syncwarp();
            if (lane == 0) {
                mbar_arrive_expect_tx(&ring.bars[b], (unsigned)ring.buf_stride);
                tma_tensor2d_g2s(ring.slot + b * ring.buf_stride, ring.tmap, cb * 8, ring.row0, &ring.bars[b]);
            }
            return;
        }
        const unsigned total = __reduce_add_sync(kFull, bytes);
        if (lane == 0) {
            if (total) mbar_arrive_expect_tx(&ring.bars[b], total);
            else mbar_arrive(&ring.bars[b]);
        }
        __syncwarp();
        if (bytes) tma_bulk_g2s(ring.slot + b * ring.buf_stride, pool + (r.off - mis) + (long long)clo * 8, bytes, &ring.bars[b]);
    };
    // |x[i] - x[i-1]| of the four words of chunk q, packed, given the word in front of it
    auto absdiff4 = [](const uint4& q, unsigned pw, unsigned& e0, unsigned& e1, unsigned& e2, unsigned& e3) {
        const unsigned g0 = __funnelshift_r(pw, q.x, 16), g1 = __funnelshift_r(q.x, q.y, 16);
        const unsigned g2 = __funnelshift_r(q.y, q.z, 16), g3 = __funnelshift_r(q.z, q.w, 16);
        e0 = __vmaxu2(q.x, g0) - __vminu2(q.x, g0);
        e1 = __vmaxu2(q.y, g1) - __vminu2(q.y, g1);
        e2 = __vmaxu2(q.z, g2) - __vminu2(q.z, g2);
        e3 = __vmaxu2(q.w, g3) - __vminu2(q.w, g3);
    };
    auto feat_plain = [&](const uint4& q, unsigned csum) {
        unsigned e0, e1, e2, e3;
        absdiff4(q, fs.prev_w, e0, e1, e2, e3);
        fs.pdiff = __vimax3_u16x2(fs.pdiff, __vmaxu2(e0, e1), __vmaxu2(e2, e3));
        fs.isum32 += csum;
        fs.prev_w = q.w;
    };
    auto csum4 = [](const uint4& q, unsigned cs = 0u) {  // cs + the eight samples of q
        cs = __dp2a_lo(q.x, 0x0101u, cs);
        cs = __dp2a_lo(q.y, 0x0101u, cs);
        cs = __dp2a_lo(q.z, 0x0101u, cs);
        return __dp2a_lo(q.w, 0x0101u, cs);
    };
    // features of any chunk (record start / end, height range, known polarity)
    auto feat_generic = [&](uint4 q, int vc) {
        if (vc >= nch) return;
        const int v0 = vc * 8;
        const int lo = max(mis - v0, 0), hi = min(vtotal - v0, 8);
        const int i0 = v0 - mis;
        const bool whole = lo == 0 && hi == 8;
        // inside the area slice and the record (not its first sample), outside the height slice, unknown polarity
        const bool plain = !known && i0 >= max(c0, 1) && i0 + 8 <= min(c1, r.len) && (p1 <= p0 || i0 + 8 <= p0 || i0 >= p1);
        if (plain) {
            feat_plain(q, csum4(q));
        } else if (whole) {
            unsigned e0, e1, e2, e3;
            absdiff4(q, (i0 > 0) ? fs.prev_w : (q.x << 16), e0, e1, e2, e3);
            fs.pdiff = __vmaxu2(fs.pdiff, __vmaxu2(__vmaxu2(e0, e1), __vmaxu2(e2, e3)));
            const int jlo = max(0, p0 - i0), jhi = min(8, p1 - i0);
            if (jhi > jlo) {
                if (jlo == 0 && jhi == 8) {
                    fs.pmin = __vminu2(fs.pmin, __vminu2(__vminu2(q.x, q.y), __vminu2(q.z, q.w)));
                    fs.pmax = __vmaxu2(fs.pmax, __vmaxu2(__vmaxu2(q.x, q.y), __vmaxu2(q.z, q.w)));
                } else {
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        int w = u16_at(q, j);
                        if (j >= jlo && j < jhi) { fs.imin = min(fs.imin, w); fs.imax = max(fs.imax, w); }
                    }
                }
            }
            const int klo = max(0, c0 - i0), khi = min(8, c1 - i0);
            if (khi > klo) {
                if (klo == 0 && khi == 8 && !known) {
                    fs.isum32 += csum4(q);
                } else {
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        unsigned w = (unsigned)u16_at(q, j);
                        if (j >= klo && j < khi) {
                            if (!known) fs.isum32 += w;
                            else fs.dsum += (double)(r.positive ? __fsub_rn((float)w, b32) : __fsub_rn(b32, (float)w));
                        }
                    }
                }
            }
            fs.prev_w = q.w;
        } else {
            const int prev_s = (int)(fs.prev_w >> 16);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int w = u16_at(q, j);
                if (j >= lo && j < hi) {
                    const int i = i0 + j;
                    if (i > 0) fs.idiff = max(fs.idiff, abs(w - ((j == 0) ? prev_s : u16_at(q, j - 1))));
                    if (i >= p0 && i < p1) { fs.imin = min(fs.imin, w); fs.imax = max(fs.imax, w); }
                    if (i >= c0 && i < c1) {
                        if (!known) fs.isum32 += (unsigned)w;
                        else fs.dsum += (double)(r.positive ? __fsub_rn((float)w, b32) : __fsub_rn(b32, (float)w));
                    }
                }
            }
            fs.prev_w = q.w;
        }
    };

    if (nseg > 0) issue(0);
    for (int s = 0; s <= nseg; ++s) {  // s == nseg: nothing is streamed any more, the queue is drained
        const bool drain = s == nseg;
        const int b = s % kNBuf;
        if (!drain) {
            if (s + 1 < nseg) issue(s + 1);
            mbar_wait(&ring.bars[b], (*ring.phase_bits >> b) & 1u);
            *ring.phase_bits ^= 1u << b;
        }
        const uint8_t* buf = ring.slot + b * ring.buf_stride;
        const int tend = drain ? 1 : min(bps, nblk - s * bps);
        const int qmin = drain ? 1 : 32;  // a round runs when 32 complete items wait; the drain takes what is left
        if (drain) myslot = -1;           // the items of the last block lie behind their records: no next word
        for (int t = 0; t < tend; ++t) {
            const int B = s * bps + t;
            const uint4* blk = reinterpret_cast<const uint4*>(buf + t * 64);
            // the items pushed one step ago get the first word of their next block
            if (myslot >= 0) bq[myslot] = reinterpret_cast<const unsigned*>(blk)[0] ^ (SGN ? 0x80008000u : 0u);
            myslot = -1;
            qn_c += qn_i;
            while (qn_c >= qmin) {
                const int take = min(qn_c, 32);
                blk_round(ws, bq, qh, take, r, a, sink);
                qh = (qh + take) & (kBQRing - 1);
                qn_c -= take;
            }
            if (drain) break;
            uint4 q0 = blk[0], q1 = blk[1], q2 = blk[2], q3 = blk[3];
            if (SGN) {  // int16 -> offset binary
                q0.x ^= 0x80008000u; q0.y ^= 0x80008000u; q0.z ^= 0x80008000u; q0.w ^= 0x80008000u;
                q1.x ^= 0x80008000u; q1.y ^= 0x80008000u; q1.z ^= 0x80008000u; q1.w ^= 0x80008000u;
                q2.x ^= 0x80008000u; q2.y ^= 0x80008000u; q2.z ^= 0x80008000u; q2.w ^= 0x80008000u;
                q3.x ^= 0x80008000u; q3.y ^= 0x80008000u; q3.z ^= 0x80008000u; q3.w ^= 0x80008000u;
            }
            // class of the block; with features the sample sum of a block of 32 record samples serves the area and the FULL
            // aggregate, without them only the aggregate needs it
            bool any = false, full = false, last = false;
            unsigned kvmin = 0xffffu, ssum = 0u;
            if ((unsigned)(32 * B - mis) < whn) {
                if (FEAT) ssum = csum4(q1, csum4(q0)) + csum4(q3, csum4(q2));
                const unsigned mn2 = __vimin3_u16x2(
                    __vimin3_u16x2(__vimin3_u16x2(q0.x, q0.y, q0.z), __vimin3_u16x2(q0.w, q1.x, q1.y), __vimin3_u16x2(q1.z, q1.w, q2.x)),
                    __vimin3_u16x2(__vimin3_u16x2(q2.y, q2.z, q2.w), __vimin3_u16x2(q3.x, q3.y, q3.z), q3.w), 0xffffffffu);
                const unsigned mx2 = __vimax3_u16x2(
                    __vimax3_u16x2(__vimax3_u16x2(q0.x, q0.y, q0.z), __vimax3_u16x2(q0.w, q1.x, q1.y), __vimax3_u16x2(q1.z, q1.w, q2.x)),
                    __vimax3_u16x2(__vimax3_u16x2(q2.y, q2.z, q2.w), __vimax3_u16x2(q3.x, q3.y, q3.z), q3.w), 0u);
                const unsigned wmin = min(mn2 & 0xffffu, mn2 >> 16), wmax = max(mx2 & 0xffffu, mx2 >> 16);
                kvmin = (r.positive ? wmax : wmin) ^ xm16;
                const unsigned kvmax = (r.positive ? wmin : wmax) ^ xm16;
                any = (int)kvmin <= r.kmax;
                full = (int)kvmax <= kfull;
                last = (int)((q3.w >> 16) ^ xm16) <= r.kmax;
            } else if (4 * B < nch) {  // record start / end: by position
                const int i0 = 32 * B - mis;
                const unsigned short* hwb = reinterpret_cast<const unsigned short*>(blk);
                for (int j = 0; j < 32; ++j) {
                    const int i = i0 + j;
                    const unsigned w = (unsigned)hwb[j] ^ (SGN ? 0x8000u : 0u);
                    const bool ab = i >= 0 && i < r.len && (int)(w ^ xm16) <= r.kmax;
                    any = any || ab;
                    last = ab;
                }
            }
            if (FEAT) {
                if ((unsigned)(B - f0) < fn0 || (unsigned)(B - f1) < fn1) {  // inside the blocks of 32 record samples
                    unsigned e[16];
                    absdiff4(q0, fs.prev_w, e[0], e[1], e[2], e[3]);
                    absdiff4(q1, q0.w, e[4], e[5], e[6], e[7]);
                    absdiff4(q2, q1.w, e[8], e[9], e[10], e[11]);
                    absdiff4(q3, q2.w, e[12], e[13], e[14], e[15]);
                    fs.pdiff = __vimax3_u16x2(
                        __vimax3_u16x2(__vimax3_u16x2(e[0], e[1], e[2]), __vimax3_u16x2(e[3], e[4], e[5]), __vimax3_u16x2(e[6], e[7], e[8])),
                        __vimax3_u16x2(__vimax3_u16x2(e[9], e[10], e[11]), __vimax3_u16x2(e[12], e[13], e[14]), e[15]), fs.pdiff);
                    fs.isum32 += ssum;
                    fs.prev_w = q3.w;
                } else {
#pragma unroll 1
                    for (int c = 0; c < 4; ++c) {  // record start / end, height range, known polarity: chunk by chunk
                        uint4 q = blk[c];
                        if (SGN) { q.x ^= 0x80008000u; q.y ^= 0x80008000u; q.z ^= 0x80008000u; q.w ^= 0x80008000u; }
                        feat_generic(q, 4 * B + c);
                    }
                }
            }
            if (full && open) {
                fa_key = min(fa_key, (kvmin << 16) | (unsigned)B);
                fa_sum += FEAT ? ssum : csum4(q1, csum4(q0)) + csum4(q3, csum4(q2));
            }
            const bool item = full ? !open : (any || open);
            const unsigned bal = __ballot_sync(kFull, item);
            if (item) {
                const int slot = (qh + qn_c + __popc(bal & ((1u << lane) - 1u))) & (kBQRing - 1);
                unsigned* sl = bq + slot * kBQWords;
                sl[0] = hprev;
                sl[1] = q0.x; sl[2] = q0.y; sl[3] = q0.z; sl[4] = q0.w;
                sl[5] = q1.x; sl[6] = q1.y; sl[7] = q1.z; sl[8] = q1.w;
                sl[9] = q2.x; sl[10] = q2.y; sl[11] = q2.z; sl[12] = q2.w;
                sl[13] = q3.x; sl[14] = q3.y; sl[15] = q3.z; sl[16] = q3.w;
                sl[18] = (unsigned)lane | ((unsigned)B << 5);
                sl[19] = fa_key;
                sl[20] = fa_sum;
                myslot = slot * kBQWords + 17;
                fa_key = 0xffffffffu;
                fa_sum = 0u;
            }
            qn_i = __popc(bal);
            open = last;
            hprev = q3.w;
        }
        __syncwarp();  // every lane is done with buffer b before it is refilled
    }
}

}  // namespace wfb
