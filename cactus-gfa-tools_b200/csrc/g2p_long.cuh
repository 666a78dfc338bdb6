// g2p_long.cuh — the streaming conversion kernel for records k_short does not take: anything
// longer than kSLimit bytes or with more steps / ops than fit one 8-lane group, up to
// chromosome-scale assembly records (10^4 path steps, 10^5 CIGAR ops, hundreds of kB of text).
//
// One warp owns one record and never materialises it.  Two token streams run over the record
// text in global memory, forwards for '+' records and backwards for '-' records (flip_gaf,
// gaf2paf_main.cpp:92-131, becomes a change of direction):
//   step stream   '>' / '<' markers of the path column  (gafkluge.hpp:118-158)
//   op stream     op letters of the cg:Z: value          (for_each_cg, gafkluge.hpp:226-239)
// Each refill classifies 512 bytes (16 per lane, SWAR compares), ranks the hits with a shuffle
// prefix sum and scatters their positions into a shared ring.  Steps are consumed 31 at a time
// (one lane per step: token parse, table probe, quota), ops 32 at a time (one lane per op, four
// 64-bit shuffle prefix sums carried from window to window).  The split of the CIGAR at step
// boundaries (cigar_next_by_target, gaf2paf_main.cpp:71-90; SURVEY.md Appendix B.3-B.5) is a
// merge of two sorted sequences: a boundary B is resolved by a shuffle binary search in the
// first op window whose cumulative target length reaches it; the window only advances when an
// unresolved boundary lies beyond it.  State carried between windows / batches is O(1).
// PAF lines of a batch are formatted one per lane into a shared staging buffer and flushed with
// 128-bit stores.
//
// Like k_short, the kernel converts only canonical records and delegates everything else
// (including every error path of the reference) to the general kernel k_convert_list.
#pragma once
#include "g2p_short.cuh"

namespace g2p {

enum : u32 { ST_F_LONG = 0x20000u };   // status flag: record was converted by k_long

constexpr int kLWarps = 4;
constexpr int kLThreads = kLWarps * 32;
#ifndef G2P_LONG_RING
#define G2P_LONG_RING 256
#endif
constexpr u32 kLRing = G2P_LONG_RING;   // ring entries (power of two); a refill that would not fit flags the stream (record delegated)
constexpr u32 kLChunk = 512;     // bytes classified per refill
constexpr u32 kLBatch = 31;      // steps per batch; the next lane holds the batch's end boundary
constexpr u32 kLOutCap = 5120;   // staged PAF bytes per batch
constexpr u32 kLText = 2048;     // bytes of text each stream keeps in shared memory (power of two, multiple of kLChunk)
constexpr u32 kLHead = 64;       // cached query name / tp / rc text

template <bool WITH_OUT>
struct __align__(16) LWarpMemT {
    u32 sring[kLRing];
    u32 oring[kLRing];
    u8 stext[kLText];            // last chunks of the path column, addressed by (offset & (kLText-1))
    u8 otext[kLText];            // last chunks of the cg value
    u8 qname[kLHead], tp[kLHead], rc[kLHead];
    u32 tabs[32];
    u32 hdr[H_N];
    u32 tkeys[kSMaxTags];
    u8 out[WITH_OUT ? kLOutCap + 16 : 16];   // line staging of the streaming emit (fallback path only)
};
static_assert(sizeof(LWarpMemT<true>) % 16 == 0 && sizeof(LWarpMemT<false>) % 16 == 0, "warp slices must keep 16-byte alignment");
template <bool EMIT> constexpr size_t long_smem() { return sizeof(LWarpMemT<EMIT>) * kLWarps; }
#ifndef G2P_LONG_CTAS
#define G2P_LONG_CTAS 4   /* resident CTAs per SM the size pass of k_long is compiled for */
#endif

__device__ __forceinline__ u32 range16u(u32 lo, u32 hi) {   // bits [lo, hi), both clamped to 16
    lo = lo > 16u ? 16u : lo;
    hi = hi > 16u ? 16u : hi;
    return hi > lo ? (((1u << hi) - 1u) & ~((1u << lo) - 1u)) : 0u;
}
__device__ __forceinline__ u32 wscan32(u32 v, u32 lane) {
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const u32 t = __shfl_up_sync(0xffffffffu, v, d); if (lane >= (u32)d) v += t; }
    return v;
}
__device__ __forceinline__ u64 wscan64(u64 v, u32 lane) {
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const u64 t = __shfl_up_sync(0xffffffffu, v, d); if (lane >= (u32)d) v += t; }
    return v;
}

// L2 prefetch of the line holding p (no register is tied up by the request).
__device__ __forceinline__ void prefetch_l2(const void* p) {
#if !defined(G2P_HOSTSIM)
    asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
#else
    (void)p;
#endif
}

// 16 bytes from base[off..], base 4-byte aligned for off == 0 (global text or a shared text window).
__device__ __forceinline__ void ld16_unaligned(const u8* base4, u32 sh_bytes, u32& w0, u32& w1, u32& w2, u32& w3) {
    const u32* q = reinterpret_cast<const u32*>(base4);
    const u32 sh = sh_bytes * 8u;
    const u32 x0 = q[0], x1 = q[1], x2 = q[2], x3 = q[3], x4 = q[4];
    w0 = __funnelshift_r(x0, x1, sh); w1 = __funnelshift_r(x1, x2, sh);
    w2 = __funnelshift_r(x2, x3, sh); w3 = __funnelshift_r(x3, x4, sh);
}

// Positions (absolute offsets into the GAF buffer) of the marker / non-digit bytes of a text span,
// produced chunk by chunk in stream order into a shared ring.  All members are warp-uniform.
template <bool MARKERS>
struct TokStream {
    u32* ring;
    u8* text;          // shared copy of the most recent chunks
    const u8* gaf;
    u32 lo, hi;        // span [lo, hi)
    u32 cur;           // base of the next chunk (multiple of kLChunk)
    u32 head, count;
    u32 tlo, thi;      // offsets currently held in `text`: [tlo, thi)
    bool bwd, done, overflow;

    __device__ __forceinline__ void init(u32* ring_, u8* text_, const u8* gaf_, u32 lo_, u32 hi_, bool bwd_) {
        ring = ring_; text = text_; gaf = gaf_; lo = lo_; hi = hi_; bwd = bwd_;
        overflow = false;
        head = count = 0;
        tlo = thi = 0;
        done = hi_ <= lo_;
        cur = done ? 0u : (bwd_ ? ((hi_ - 1u) & ~(kLChunk - 1u)) : (lo_ & ~(kLChunk - 1u)));
    }
    // Pointer to the n bytes at offset x: the shared copy when it holds all of them without
    // wrapping, else global memory.
    __device__ __forceinline__ const u8* src(u32 x, u32 n) const {
        const u32 k = x & (kLText - 1u);
        return (x >= tlo && x + n <= thi && k + n <= kLText) ? text + k : gaf + x;
    }
    __device__ __forceinline__ void refill(const u8* /*gaf*/, u64 n, u32 lane) {
        const u32 off = cur + 16u * lane;
        u32 m = 0;
        {   // the chunk replaces the oldest one in the shared text window
            const uint4 v0 = ldg_vec_guarded(gaf, off, n);
            *reinterpret_cast<uint4*>(text + (off & (kLText - 1u))) = v0;
            if (thi == tlo) { tlo = cur; thi = cur + kLChunk; }
            else if (!bwd) { thi = cur + kLChunk; if (thi - tlo > kLText) tlo = thi - kLText; }
            else { tlo = cur; if (thi - tlo > kLText) thi = tlo + kLText; }
        }
        if (off < hi && off + 16u > lo) {
            const uint4 v = *reinterpret_cast<const uint4*>(text + (off & (kLText - 1u)));
            const u32 w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int k = 0; k < 4; ++k)
                m |= movemask4(MARKERS ? zero_bytes((w[k] & 0xFDFDFDFDu) ^ 0x3C3C3C3Cu) : nondigit_bytes(w[k])) << (4 * k);
            m &= range16u(lo > off ? lo - off : 0u, hi - off);
        }
        const u32 cnt = (u32)__popc(m);
        const u32 incl = wscan32(cnt, lane);
        const u32 total = __shfl_sync(0xffffffffu, incl, 31);
        if (count + total > kLRing) { overflow = true; done = true; __syncwarp(); return; }   // pathologically dense tokens
        if (!bwd) {
            u32 k = head + count + incl - cnt;
            while (m) { const u32 b = (u32)__ffs((int)m) - 1u; m &= m - 1u; ring[k & (kLRing - 1u)] = off + b; ++k; }
        } else {
            u32 k = head + count + (total - incl);
            while (m) { const u32 b = 31u - (u32)__clz((int)m); m &= ~(1u << b); ring[k & (kLRing - 1u)] = off + b; ++k; }
        }
        count += total;
        if (!bwd) { if (hi - cur <= kLChunk) done = true; else cur += kLChunk; }
        else { if (cur <= lo) done = true; else cur -= kLChunk; }
        if (!done && (lane & 7u) == 0) prefetch_l2(gaf + cur + 16u * lane);   // the chunk the next refill reads
        __syncwarp();
    }
    __device__ __forceinline__ void ensure(u32 need, const u8* gaf, u64 n, u32 lane) {
        while (count < need && !done) refill(gaf, n, lane);
    }
    __device__ __forceinline__ u32 at(u32 k) const { return ring[(head + k) & (kLRing - 1u)]; }
    __device__ __forceinline__ void pop(u32 k) { head = (head + k) & (kLRing - 1u); count -= k; }
};

struct StepTok2 {
    u32 name_a, nl;   // absolute offset / length of the name
    i32 tlen, sa, se;
};

// One path step token [p, q) (p = its marker, or pa-1 for an unprefixed path): name, optional
// ":start-end", table probe.  Text comes from the step stream's shared window when it holds the
// token.  Returns the lane's "not canonical" flag.
__device__ __forceinline__ u32 parse_step_global(const TokStream<true>& ss, u64 n, const LenTableView& T, u32 p, u32 q, bool prefixed, StepTok2& t) {
    t.name_a = p + 1;
    const u32 tl = q - t.name_a;
    t.nl = tl; t.tlen = 0; t.sa = 0; t.se = 0;
    if ((u64)t.name_a + 24 > n) return 1;
    u32 w0, w1, w2, w3;
    ld16_unaligned(ss.src(t.name_a & ~3u, 24), t.name_a & 3u, w0, w1, w2, w3);
    bool interval = false;
    if (prefixed) {
        u32 cm = movemask4(zero_bytes(w0 ^ 0x3A3A3A3Au)) | (movemask4(zero_bytes(w1 ^ 0x3A3A3A3Au)) << 4) |
                 (movemask4(zero_bytes(w2 ^ 0x3A3A3A3Au)) << 8) | (movemask4(zero_bytes(w3 ^ 0x3A3A3A3Au)) << 12);
        cm &= tl >= 16 ? 0xffffu : ((1u << tl) - 1u);
        if (cm) { t.nl = (u32)__ffs((int)cm) - 1u; interval = true; }
    }
    if (t.nl == 0 || t.nl > 16) return 1;
    const int nl = (int)t.nl;
    w0 = keep_bytes(w0, nl); w1 = keep_bytes(w1, nl - 4); w2 = keep_bytes(w2, nl - 8); w3 = keep_bytes(w3, nl - 12);
    i64 tl64 = 0;
    if (!table_lookup_key16(T, (u64)w0 | ((u64)w1 << 32), (u64)w2 | ((u64)w3 << 32), t.nl, tl64)) return 1;
    if (tl64 < 0 || tl64 > 0x7fffffffLL) return 1;
    t.tlen = (i32)tl64;
    t.se = t.tlen;
    if (interval) {
        const u32 i0 = t.name_a + t.nl + 1, il = q - i0;   // "start-end"
        const u8* tx = ss.src(i0, il);
        u32 k = 0, x = 0, nd = 0;
        while (k < il && nd < 10) { const u32 d = (u32)tx[k] - '0'; if (d > 9) break; x = x * 10u + d; ++nd; ++k; }
        if (nd == 0 || nd > 9 || k >= il || tx[k] != '-') return 1;
        t.sa = (i32)x;
        ++k; x = 0; nd = 0;
        while (k < il && nd < 10) { const u32 d = (u32)tx[k] - '0'; if (d > 9) break; x = x * 10u + d; ++nd; ++k; }
        if (nd == 0 || nd > 9 || k != il) return 1;
        t.se = (i32)x;
    }
    return t.se < t.sa ? 1u : 0u;
}

// Requests the table slot the step token [p, q) will probe, one batch ahead of its use: the probe
// is a dependent random access (DRAM or far L2) and was the largest single stall of the kernel.
__device__ __forceinline__ void prefetch_step_slot(const TokStream<true>& ss, u64 n, const LenTableView& T, u32 p, u32 q) {
    const u32 name_a = p + 1, tl = q - name_a;
    if ((u64)name_a + 24 > n || T.nslots == 0) return;
    u32 w0, w1, w2, w3;
    ld16_unaligned(ss.src(name_a & ~3u, 24), name_a & 3u, w0, w1, w2, w3);
    u32 cm = movemask4(zero_bytes(w0 ^ 0x3A3A3A3Au)) | (movemask4(zero_bytes(w1 ^ 0x3A3A3A3Au)) << 4) |
             (movemask4(zero_bytes(w2 ^ 0x3A3A3A3Au)) << 8) | (movemask4(zero_bytes(w3 ^ 0x3A3A3A3Au)) << 12);
    cm &= tl >= 16 ? 0xffffu : ((1u << tl) - 1u);
    const u32 nl = cm ? (u32)__ffs((int)cm) - 1u : tl;
    if (nl == 0 || nl > 16) return;
    const int k = (int)nl;
    w0 = keep_bytes(w0, k); w1 = keep_bytes(w1, k - 4); w2 = keep_bytes(w2, k - 8); w3 = keep_bytes(w3, k - 12);
    prefetch_l2(T.slots + slot_index((u64)w0 | ((u64)w1 << 32), (u64)w2 | ((u64)w3 << 32), nl, T.nslots));
}

struct LongArgs {
    const u8* gaf;
    u64 n;
    const u32* rec_start;
    LenTableView T;
    u64* out_off;
    u32* status;
    u8* out;
    const u32* list;       // records to convert (delegated by k_short)
    const u32* n_list;
    u32* deleg_list;       // size pass: records left to the general kernel
    u32* n_deleg;
    LineDesc* desc;        // size pass: line descriptors for k_emit_lines (one padded 32-slot block per batch)
    RecDesc* rdesc;
    u32* n_desc;
    u32* n_desc2;          // small batches (<= 8 lines) take blocks from the upper half of the array: desc_cap / 2 + ...
    u32 desc_cap;
    u32 small_max;         // batches of at most this many lines take a small block (0: every batch takes 32 slots)
    u32* need_legacy;      // set when a record could not be described (array full): k_long<true> emits it
    u32* cursor;           // size pass: shared cursor into `list` (warps take the next record when they are free)
};

template <bool EMIT>
__device__ __forceinline__ void long_record(const LongArgs& a, LWarpMemT<EMIT>* wm, const u32 r, const u32 lane, const u32* p10) {
    const u32 FULL = 0xffffffffu;
    const Grp<32> g;
    const u8* gaf = a.gaf;
    const u32 s = a.rec_start[r], len = a.rec_start[r + 1] - s - 1;
    const u8* rt = gaf + s;
    u64 o = 0, osize = 0;
    if (EMIT) {   // legacy emit: only records whose lines are not in the descriptor array
        const u32 st0 = a.status[r];
        if (!(st0 & ST_F_LONG) || (st0 & ST_F_DESC)) return;
        o = a.out_off[r];
        osize = a.out_off[r + 1] - o;
        if (osize == 0) return;
    }
    bool deleg = false;
    bool desc_fail = false;   // (size pass) some line of the record is not in the descriptor array
    u64 size = 0;
    u32 status = ST_OK | ST_F_LONG;
    do {
        if (len == 0) { deleg = true; break; }
        if (rt[0] == '*') { status = ST_SKIP | ST_F_LONG; break; }
        // ---------------- tabs
        u32 nt = 0;
        {
            const u64 end = (u64)s + len;
            for (u64 base = s & ~(kLChunk - 1u); base < end; base += kLChunk) {
                const u64 off = base + 16u * lane;
                u32 m = 0;
                if (off < end && off + 16 > s) {
                    const uint4 v = ldg_vec_guarded(gaf, off, a.n);
                    const u32 w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                    for (int k = 0; k < 4; ++k) m |= movemask4(zero_bytes(w[k] ^ 0x09090909u)) << (4 * k);
                    m &= range16u(s > off ? (u32)(s - off) : 0u, (u32)(end - off > 16 ? 16 : end - off));
                }
                if (!__any_sync(FULL, m != 0)) continue;
                const u32 cnt = (u32)__popc(m);
                const u32 incl = wscan32(cnt, lane);
                u32 k = nt + incl - cnt;
                while (m) { const u32 b = (u32)__ffs((int)m) - 1u; m &= m - 1u; if (k < 32) wm->tabs[k] = (u32)(off - s) + b; ++k; }
                nt += __shfl_sync(FULL, incl, 31);
                if (nt > kSMaxTabs) break;
            }
        }
        if (lane < 6) wm->hdr[H_CG_A + lane] = 0;
        __syncwarp();
        if (nt < 11 || nt > kSMaxTabs) { deleg = true; break; }
        u32 lbad = parse_fields<32>(g, rt, wm->tabs, nt, len, wm->hdr, wm->tkeys);
        if (__any_sync(FULL, lbad != 0)) { deleg = true; break; }
        const bool minus = wm->hdr[H_MINUS] != 0;
        const i32 qs = (i32)wm->hdr[H_QS], ps = (i32)wm->hdr[H_PS], pe = (i32)wm->hdr[H_PE];
        if (wm->hdr[H_CG_B] == 0 || wm->hdr[H_CG_A] >= wm->hdr[H_CG_B] || qs < 0 || ps < 0 || pe < 0) { deleg = true; break; }
        const u32 cA = s + wm->hdr[H_CG_A], cB = s + wm->hdr[H_CG_B];
        const u32 pA = s + wm->hdr[H_PATH_A], pB = s + wm->hdr[H_PATH_B];
        const u8 c0 = gaf[pA];
        const bool prefixed = c0 == '>' || c0 == '<';
        const bool empty_path = !prefixed && pB - pA == 1 && c0 == '*';

        LineRec R;
        R.qn_b = wm->hdr[H_QN_B];
        R.qlen = (i32)wm->hdr[H_QLEN]; R.m = (i32)wm->hdr[H_M]; R.b = (i32)wm->hdr[H_B]; R.mapq = (i32)wm->hdr[H_MAPQ];
        R.tp_a = wm->hdr[H_TP_A]; R.tp_b = wm->hdr[H_TP_B]; R.rc_a = wm->hdr[H_RC_A]; R.rc_b = wm->hdr[H_RC_B];
        R.gi_n = gi_fast(R.m, R.b, R.gi);
        if (R.gi_n == 0) { deleg = true; break; }
        const u32 const_len = line_const_len(R, p10);
        if (!EMIT) {
            desc_fail = !rec_desc_fits(R);
            if (!desc_fail && lane == 0) store_rec_desc(a.rdesc + r, R);
        }
        // query name and tp / rc text are the same for every line of the record: cache them
        const bool head_cached = R.qn_b <= kLHead && R.tp_b - R.tp_a <= kLHead && R.rc_b - R.rc_a <= kLHead;
        if (head_cached) {
            for (u32 k = lane; k < R.qn_b; k += 32) wm->qname[k] = rt[k];
            for (u32 k = lane; k < R.tp_b - R.tp_a; k += 32) wm->tp[k] = rt[R.tp_a + k];
            for (u32 k = lane; k < R.rc_b - R.rc_a; k += 32) wm->rc[k] = rt[R.rc_a + k];
            __syncwarp();
        }

        TokStream<true> ss;
        TokStream<false> os;
        // ---------------- '-' records: path length from the steps (flip_gaf, gaf2paf_main.cpp:111-131)
        i32 ps2 = ps, pe2 = pe;
        if (minus) {
            u64 L = 0;
            if (prefixed) {
                ss.init(wm->sring, wm->stext, gaf, pA, pB, false);
                for (;;) {
                    ss.ensure(33, gaf, a.n, lane);
                    const u32 nb_ = ss.count < 32u ? ss.count : 32u;
                    if (nb_ == 0) break;
                    u64 v = 0;
                    if (lane < nb_) {
                        const u32 p = ss.at(lane), q = lane + 1 < ss.count ? ss.at(lane + 1) : pB;
                        StepTok2 t;
                        lbad |= parse_step_global(ss, a.n, a.T, p, q, true, t);
                        v = (u64)(u32)(t.se - t.sa);
                    }
                    v = wscan64(v, lane);
                    L += __shfl_sync(FULL, v, 31);
                    __syncwarp();
                    ss.pop(nb_);
                }
            } else if (!empty_path) {
                StepTok2 t;
                ss.init(wm->sring, wm->stext, gaf, 0u, 0u, false);
                lbad |= parse_step_global(ss, a.n, a.T, pA - 1, pB, false, t);
                L = (u64)(u32)(t.se - t.sa);
            }
            if (__any_sync(FULL, lbad != 0) || L > 0x7fffffffULL) { deleg = true; break; }
            ps2 = (i32)L - pe; pe2 = (i32)L - ps;
        }
        const i32 W = pe2 - ps2;
        if (ps2 < 0 || W < 0) { deleg = true; break; }

        // ---------------- streams
        ss.init(wm->sring, wm->stext, gaf, prefixed ? pA : 0u, prefixed ? pB : 0u, minus);
        os.init(wm->oring, wm->otext, gaf, cA, cB, minus);
        // op window (one op per lane, inclusive prefixes carried across windows)
        u64 wEND = 0, wQ = 0, wM = 0, wNB = 0, cE = 0, cQ = 0, cM = 0, cNB = 0;
        u32 wlen = 0, wlp = 0, wds = 0, wk = 0, nwin = 0;
        u32 last_lp = cA - 1;          // fwd: letter position of the previous op
        u32 top_lp = 0;                // largest letter position seen (must be cB-1)
        bool win_valid = false, ops_done = false;
        u64 win_last = 0;              // cumulative target length at the end of the window
        auto load_window = [&]() {
            os.ensure(33, gaf, a.n, lane);
            nwin = os.count < 32u ? os.count : 32u;
            if (nwin == 0) { win_valid = false; ops_done = true; return; }
            u32 vE = 0, vQ = 0, vM = 0, vB = 0;   // op lengths < 10^8: a window's sums fit 32 bits
            wlen = 0; wlp = 0; wds = 0; wk = 0;
            const u32 mylp = lane < nwin ? os.at(lane) : 0u;
            u32 prev = __shfl_up_sync(FULL, mylp, 1);
            if (lane == 0) prev = last_lp;
            if (lane < nwin) {
                wlp = mylp;
                if (!minus) wds = prev + 1u;
                else wds = lane + 1 < os.count ? os.at(lane + 1) + 1u : cA;
                const u32 nd = wlp - wds;
                // digits + op letter: two call sites so that the common one works on a pointer the
                // compiler can prove to be shared memory (LDS instead of generic loads)
                auto parse_op = [&](const u8* tx) {
                    wk = (u32)tx[nd] - '=';
                    if (wk >= 28 || !((kOpMask >> wk) & 1u) || nd == 0 || nd > 8 || (nd > 1 && tx[0] == '0')) { lbad = 1; return; }
                    u32 x = 0;
                    for (u32 t = 0; t < nd; ++t) x = x * 10u + ((u32)tx[t] - '0');
                    if (x == 0) lbad = 1;
                    wlen = x;
                    vB = x;
                    vE = ((kTargetMask >> wk) & 1u) ? x : 0u;
                    vQ = ((kQueryMask >> wk) & 1u) ? x : 0u;
                    vM = ((kMatchMask >> wk) & 1u) ? x : 0u;
                };
                const u32 tk = wds & (kLText - 1u);
                if (wds >= os.tlo && wlp + 1u <= os.thi && tk + nd + 1u <= kLText) parse_op(wm->otext + tk);
                else parse_op(gaf + wds);
            }
            wEND = (u64)wscan32(vE, lane) + cE; wQ = (u64)wscan32(vQ, lane) + cQ; wM = (u64)wscan32(vM, lane) + cM; wNB = (u64)wscan32(vB, lane) + cNB;
            cE = __shfl_sync(FULL, wEND, nwin - 1); cQ = __shfl_sync(FULL, wQ, nwin - 1);
            cM = __shfl_sync(FULL, wM, nwin - 1); cNB = __shfl_sync(FULL, wNB, nwin - 1);
            win_last = cE;
            if (lane >= nwin) wEND = ~0ULL;
            const u32 hi_lp = __shfl_sync(FULL, wlp, minus ? 0 : (int)nwin - 1);
            if (hi_lp > top_lp) top_lp = hi_lp;
            last_lp = __shfl_sync(FULL, wlp, nwin - 1);
            __syncwarp();
            os.pop(nwin);
            win_valid = true;
        };

        // ---------------- merge of step boundaries and op windows
        u32 tbc = 0;                   // cumulative quota of the steps before the batch
        u32 prev_p = pB;               // bwd: marker position of the previous (text-later) step
        bool first_batch = true, steps_done = empty_path;
        u64 run = 0;                   // PAF bytes of the record so far
        bool fail = false;
        while (!steps_done) {
            // --- next batch of steps
            u32 nsb;
            bool has_last;
            if (prefixed) {
                ss.ensure(kLBatch + 1, gaf, a.n, lane);
                nsb = ss.count < kLBatch ? ss.count : kLBatch;
                has_last = ss.done && ss.count == nsb;
            } else { nsb = 1; has_last = true; }
            if (nsb == 0) { fail = true; break; }   // prefixed path without a marker cannot happen
            const bool is_step = lane < nsb;
            StepTok2 t;
            t.name_a = 0; t.nl = 0; t.tlen = 0; t.sa = 0; t.se = 0;
            bool rev = false;
            {
                u32 p = 0, q = 0;
                if (prefixed) {
                    const u32 myp = is_step ? ss.at(lane) : 0u;
                    if (!minus) q = lane + 1 < ss.count ? ss.at(lane + 1) : pB;
                    else { q = __shfl_up_sync(FULL, myp, 1); if (lane == 0) q = prev_p; }
                    p = myp;
                    prev_p = __shfl_sync(FULL, myp, (int)nsb - 1);
                } else { p = pA - 1; q = pB; }
                if (is_step) {
                    rev = (prefixed && *ss.src(p, 1) == '<') != minus;
                    lbad |= parse_step_global(ss, a.n, a.T, p, q, prefixed, t);
                }
            }
            __syncwarp();
            if (prefixed) ss.pop(nsb);
            if (prefixed && !has_last) {   // next batch: bring its markers in and request its table slots now
                ss.ensure(kLBatch + 1, gaf, a.n, lane);
                const u32 nn = ss.count < kLBatch ? ss.count : kLBatch;
                const u32 np = lane < nn ? ss.at(lane) : 0u;
                u32 nq;
                if (!minus) nq = lane + 1 < ss.count ? ss.at(lane + 1) : pB;
                else { nq = __shfl_up_sync(FULL, np, 1); if (lane == 0) nq = prev_p; }
                if (lane < nn) prefetch_step_slot(ss, a.n, a.T, np, nq);
            }
            const i32 slen = t.se - t.sa;
            const i32 so = (first_batch && lane == 0) ? ps2 : 0;
            const bool is_last = has_last && lane + 1 == nsb;
            const u32 qsum = wscan32(is_step && !is_last ? (u32)(slen - so) : 0u, lane);
            u32 B = tbc + qsum - (is_step && !is_last ? (u32)(slen - so) : 0u);
            i32 quota = slen - so, eo = 0;
            if (is_last) { quota = W - (i32)B; eo = slen - so - quota; }
            if (is_step && (quota < 0 || eo < 0)) lbad = 1;
            {   // end boundary of the batch on lane nsb
                const u32 endB = __shfl_sync(FULL, B + (u32)quota, (int)nsb - 1);
                if (lane == nsb) B = endB;
                tbc = endB;
            }
            if (!is_step) quota = 0;
            if (__any_sync(FULL, lbad != 0)) { fail = true; break; }
            if ((u32)W > 0x7fffffffu || tbc > (u32)W) { fail = true; break; }

            // --- resolve boundaries (lanes 0..nsb) against the op windows
            bool need = lane <= nsb && B != 0;
            u32 r_lp = 0, r_ds = 0, r_code = 0, r_rem = 0, r_t = 0;
            bool r_cut = false;
            u64 rCQ = 0, rCM = 0, rCB = 0;
            while (__any_sync(FULL, need)) {
                if (!win_valid && !ops_done) load_window();
                if (__any_sync(FULL, lbad != 0)) { fail = true; break; }
                if (!win_valid) { fail = true; break; }   // CIGAR shorter than the path (:80 assert)
                const bool mine = need && (u64)B <= win_last;
                u32 lo = 0, hi = nwin - 1;
#pragma unroll
                for (int it = 0; it < 5; ++it) {
                    const u32 mid = (lo + hi) >> 1;
                    const u64 v = __shfl_sync(FULL, wEND, (int)mid);
                    if (lo < hi) { if (v >= (u64)B) hi = mid; else lo = mid + 1; }
                }
                const u64 jE_ = __shfl_sync(FULL, wEND, (int)lo), jQ = __shfl_sync(FULL, wQ, (int)lo), jM = __shfl_sync(FULL, wM, (int)lo),
                          jB = __shfl_sync(FULL, wNB, (int)lo);
                const u32 jl = __shfl_sync(FULL, wlen, (int)lo), jlp = __shfl_sync(FULL, wlp, (int)lo), jds = __shfl_sync(FULL, wds, (int)lo),
                          jk = __shfl_sync(FULL, wk, (int)lo);
                if (mine) {
                    const u64 tj = jE_ - jl;   // e(B) always consumes target
                    const u64 off = (u64)B - tj;
                    rCQ = jQ - (((kQueryMask >> jk) & 1u) ? (u64)jl - off : 0ULL);
                    rCM = jM - (((kMatchMask >> jk) & 1u) ? (u64)jl - off : 0ULL);
                    rCB = jB - ((u64)jl - off);
                    r_cut = jE_ > (u64)B;
                    r_rem = (u32)(jE_ - (u64)B);
                    r_t = (u32)tj;
                    r_lp = jlp; r_ds = jds; r_code = jk;
                    need = false;
                }
                if (__any_sync(FULL, need)) { win_valid = false; if (ops_done) { fail = true; break; } }
            }
            if (fail) break;

            // --- per-step values
            const bool zeroS = B == 0;
            const u32 eB = __shfl_down_sync(FULL, B, 1);
            const u32 e_lp = __shfl_down_sync(FULL, r_lp, 1), e_ds = __shfl_down_sync(FULL, r_ds, 1), e_code = __shfl_down_sync(FULL, r_code, 1),
                      e_t = __shfl_down_sync(FULL, r_t, 1);
            const u64 eCQ = __shfl_down_sync(FULL, rCQ, 1), eCM = __shfl_down_sync(FULL, rCM, 1), eCB = __shfl_down_sync(FULL, rCB, 1);
            const bool live = is_step && quota > 0;
            const u64 q64 = live ? eCQ - rCQ : 0ULL, nm64 = live ? eCM - rCM : 0ULL, nb64 = live ? eCB - rCB : 0ULL;
            const u64 q0_64 = (u64)(u32)qs + rCQ;
            if (live && (q0_64 + q64 > 0x7fffffffULL || nm64 > 0x7fffffffULL || nb64 > 0x7fffffffULL)) lbad = 1;
            if (__any_sync(FULL, lbad != 0)) { fail = true; break; }
            const bool emit_line = live && nm64 > 0;
            LineStep Ls;
            Ls.rev = rev;
            Ls.q0 = (u32)q0_64; Ls.q1 = (u32)(q0_64 + q64);
            Ls.name_a = t.name_a - s; Ls.nl = t.nl; Ls.tlen = (u32)t.tlen;
            Ls.ts = (u32)(t.sa + (rev ? eo : so)); Ls.te = (u32)(t.se - (rev ? so : eo));
            Ls.nm = (u32)nm64; Ls.nb = (u32)nb64;
            Ls.lenS = 0; Ls.codeS = 0; Ls.codeE = (u8)('=' + e_code); Ls.mid_a = Ls.mid_b = 0;
            Ls.mid_fwd = rev == minus;
            Ls.lenE = eB - (e_t > B ? e_t : B);
            u32 line = 0;
            if (emit_line) {
                const bool cutS = !zeroS && r_cut;
                const bool single = cutS && r_lp == e_lp;
                if (!single) {
                    if (cutS) { Ls.lenS = r_rem; Ls.codeS = (u8)('=' + r_code); }
                    u32 ma, mb;
                    if (!minus) { ma = zeroS ? cA : r_lp + 1u; mb = e_ds; }
                    else { ma = e_lp + 1u; mb = zeroS ? cB : r_ds; }
                    if (mb > ma) { Ls.mid_a = ma - s; Ls.mid_b = mb - s; }
                }
                line = const_len + line_step_len(Ls, p10);
            }
            const u32 lincl = wscan32(line, lane);
            const u32 btot = __shfl_sync(FULL, lincl, 31);
            if (!EMIT && btot && !desc_fail) {
                // describe the batch's lines for k_emit_lines.  Full batches take one 32-slot block from the lower half of
                // the array (one block = one warp of k_emit_lines = one contiguous run of the output); batches of at most
                // 8 lines (the only batch of a 250-1000 byte record, the last batch of a long one) take as many slots as
                // they have lines, rounded up to four, from the upper half -- a fixed 32 per batch starved such records.
                const u32 em = __ballot_sync(FULL, emit_line);
                const u32 nem = (u32)__popc(em);
                const bool small = nem <= a.small_max;
                const u32 nalloc = small ? (nem + 3u) & ~3u : 32u;
                const u32 half = a.desc_cap / 2u;
                u32 base = 0;
                if (lane == 0) base = atomicAdd(small ? a.n_desc2 : a.n_desc, nalloc);
                base = __shfl_sync(FULL, base, 0);
                const u64 lo64 = run + (lincl - line);
                const u32 room = small ? a.desc_cap - half : half;
                LineDesc* blk = a.desc + (small ? half : 0u) + base;
                if (base > room || room - base < nalloc || run + btot > 0xffffffffULL) {
                    desc_fail = true;
                    if (base < room && lane < nalloc && base + lane < room) blk[lane].rec = kDescInvalid;
                } else {
                    const u32 rank = (u32)__popc(em & ((1u << lane) - 1u));
                    if (emit_line) store_line_desc(blk + rank, r, (u32)lo64, line, Ls);
                    if (lane >= nem && lane < nalloc) blk[lane].rec = kDescInvalid;
                }
            }
            if (EMIT && btot) {
                const u64 ob = o + run;
                const bool staged = btot <= kLOutCap;
                const u32 pad = (u32)(ob & 15u);
                if (emit_line) {
                    LineSrc S;
                    S.qname = head_cached ? wm->qname : rt;
                    S.tp = head_cached ? wm->tp : rt + R.tp_a;
                    S.rc = head_cached ? wm->rc : rt + R.rc_a;
                    S.name = ss.src(t.name_a, t.nl);
                    S.mid = os.src(s + Ls.mid_a, Ls.mid_b - Ls.mid_a);
                    write_line<false>((staged ? wm->out + pad + (lincl - line) : a.out + ob + (lincl - line)) + line, S, R, Ls);
                }
                if (staged) {
                    __syncwarp();
                    const u32 total = pad + btot;
                    u8* gb = a.out + (ob - pad);
                    const u32 full_b = total >> 4;
                    for (u32 u = (pad ? 1u : 0u) + lane; u < full_b; u += 32) reinterpret_cast<uint4*>(gb)[u] = reinterpret_cast<const uint4*>(wm->out)[u];
                    const u32 head_end = pad ? (total < 16u ? total : 16u) : 0u;
                    for (u32 b = pad + lane; b < head_end; b += 32) gb[b] = wm->out[b];
                    const u32 tail_a = full_b * 16u > head_end ? full_b * 16u : head_end;
                    for (u32 b = tail_a + lane; b < total; b += 32) gb[b] = wm->out[b];
                    __syncwarp();
                }
            }
            run += btot;
            first_batch = false;
            if (has_last) steps_done = true;
        }
        if (fail) { deleg = true; break; }
        // ---------------- the rest of the CIGAR is still validated (for_each_cg parses all of it)
        while (!ops_done) {
            load_window();
            if (__any_sync(FULL, lbad != 0)) break;
        }
        if (__any_sync(FULL, lbad != 0) || top_lp != cB - 1 || ss.overflow || os.overflow) { deleg = true; break; }
        size = run;
    } while (0);
    __syncwarp();
    if (!EMIT && lane == 0) {
        if (deleg) {
            a.status[r] = ST_OK;   // overwritten by the general kernel
            a.out_off[r] = 0;
            a.deleg_list[atomicAdd(a.n_deleg, 1u)] = r;
        } else {
            const bool described = !desc_fail && size != 0;
            a.status[r] = status | (described ? (u32)ST_F_DESC : 0u);
            a.out_off[r] = size;
            if (!described && size != 0) *a.need_legacy = 1u;
        }
    }
    (void)osize;
}

template <bool EMIT>
__global__ void __launch_bounds__(kLThreads, EMIT ? 4 : G2P_LONG_CTAS) k_long(const LongArgs a) {
    G2P_DYN_SMEM(smem);
    __shared__ u32 p10[10];
    if (threadIdx.x < 10) {
        u32 v = 1;
        for (u32 i = 0; i < threadIdx.x; ++i) v *= 10u;
        p10[threadIdx.x] = v;
    }
    __syncthreads();
    const u32 lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    LWarpMemT<EMIT>* wm = reinterpret_cast<LWarpMemT<EMIT>*>(smem) + warp;
    const u32 nl = *a.n_list;
    if (!EMIT && a.cursor) {
        // records differ in length by orders of magnitude and the grid may hold more warps than are resident:
        // every warp takes the next unconverted record when it is free
        for (;;) {
            u32 k = 0;
            if (lane == 0) k = atomicAdd(a.cursor, 1u);
            k = __shfl_sync(0xffffffffu, k, 0);
            if (k >= nl) break;
            long_record<EMIT>(a, wm, a.list[k], lane, p10);
            __syncwarp();
        }
        return;
    }
    for (u32 k = blockIdx.x * kLWarps + warp; k < nl; k += gridDim.x * kLWarps) {
        long_record<EMIT>(a, wm, a.list[k], lane, p10);
        __syncwarp();
    }
}

}  // namespace g2p
