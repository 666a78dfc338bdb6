// g2p_short.cuh — the short-record conversion kernel (SURVEY.md §8a rows a2-a10 for records
// of up to kSLimit bytes: short reads, 1..G-1 path steps, <= kSMaxOps CIGAR operations).
//
// G lanes (G = 8: four records per warp) own one GAF record.  The record is staged into
// shared memory with 128-bit coalesced loads and classified 16 bytes per lane with SWAR byte
// compares (tab / '>' '<' / non-digit bit masks); ranks come from shuffle prefix sums and the
// token positions are scattered to small shared arrays.  After that every phase is
// item-parallel inside the group:
//   columns + tags   one lane per field        (parse_gaf_record, gafkluge.hpp:84-204)
//   path steps       one lane per step         (gafkluge.hpp:118-158; table probe = gaf2paf_main.cpp:162-167)
//   cg operations    one lane per op + four shuffle prefix sums (for_each_cg, gafkluge.hpp:226-239)
//   split            one lane per step boundary: lower_bound of the cumulative step quota in the
//                    cumulative target length of the ops (cigar_next_by_target, gaf2paf_main.cpp:71-90,
//                    closed form in SURVEY.md Appendix B.3-B.5)
//   emit             one lane per PAF line into a shared staging buffer, flushed with 128-bit stores
//
// '-' strand records (flip_gaf, gaf2paf_main.cpp:92-131) are handled by index arithmetic: steps
// and ops are visited in reverse order, nothing is physically reversed.
//
// The kernel only converts records it can prove canonical (plain decimal columns of <= 9
// digits, names of <= 16 bytes present in the table, XX:T:value tags, strict CIGAR syntax...).
// Anything else -- including every record the reference would reject -- is *delegated*: its
// index is appended to a list that the general per-record kernel (k_convert_list, the
// streaming state machine of g2p_core.cuh) converts.  Results are identical either way; the
// delegate path is simply slower.
#pragma once
#include "g2p_core.cuh"

namespace g2p {

enum : u32 {
    ST_F_FAST = 0x10000u,  // status flag: record was converted by k_short (else by k_long / the general kernel)
    ST_F_DESC = 0x40000u   // its PAF lines are described in the line-descriptor array (emitted by k_emit_lines)
};

#ifndef G2P_SHORT_CTAS
#define G2P_SHORT_CTAS 6   /* resident CTAs per SM the size pass is compiled for (register budget) */
#endif
constexpr int kSG = 8;                 // lanes per record
constexpr int kSThreads = 256;         // 32 records per CTA
#ifndef G2P_S_LIMIT
#define G2P_S_LIMIT 240   /* tests build a variant with 0 to push every record through k_long */
#endif
constexpr u32 kSLimit = G2P_S_LIMIT;   // longest record (bytes, without '\n') taken by the fast path
constexpr u32 kSMaxTabs = 31;          // 12 columns + up to 20 tags
constexpr u32 kSMaxTags = 20;
constexpr u32 kSMaxOps = 24;

// header slots (u32 / i32) in shared memory
enum { H_QN_B = 0, H_QLEN = 1, H_QS = 2, H_QE = 3, H_MINUS = 4, H_PATH_A = 5, H_PLEN = 6, H_PS = 7, H_PE = 8, H_M = 9, H_B = 10,
       H_MAPQ = 11, H_CG_A = 12, H_CG_B = 13, H_TP_A = 14, H_TP_B = 15, H_RC_A = 16, H_RC_B = 17, H_PATH_B = 18, H_N = 20 };

struct __align__(16) SGroupMem {
    u8 text[288];                  // the record, staged at its global 16-byte phase
    u16 spos[16];                  // path-step marker positions (+ end); tag keys alias spos..opos
    u16 opos[kSMaxOps];            // positions of the CIGAR op letters
    u32 hdr[H_N];
    u16 tabs[32];
    u32 pEnd[kSMaxOps], pQ[kSMaxOps], pNM[kSMaxOps], pNB[kSMaxOps];   // inclusive prefix sums, normalised op order
};
constexpr u32 kShortRecsPerCta = kSThreads / kSG;
constexpr u32 kSMaxLines = 8;          // line-descriptor slots per record (a record has <= G-1 lines)
constexpr size_t kShortSmem = sizeof(SGroupMem) * kShortRecsPerCta;
static_assert(sizeof(SGroupMem) % 16 == 0, "group slices must keep 16-byte alignment");

template <int G>
struct Grp {
    u32 gl, gbase, gmask;
    __device__ __forceinline__ Grp() {
        const u32 lane = threadIdx.x & 31u;
        gl = lane & (u32)(G - 1);
        gbase = lane - gl;
        gmask = (G == 32) ? 0xffffffffu : (((1u << (G & 31)) - 1u) << gbase);
    }
    __device__ __forceinline__ bool any(bool p) const { return __any_sync(gmask, p) != 0; }
    __device__ __forceinline__ u32 ballot(bool p) const { return (__ballot_sync(gmask, p) >> gbase) & ((G == 32) ? 0xffffffffu : ((1u << (G & 31)) - 1u)); }
    template <class T> __device__ __forceinline__ T shfl(T v, int src) const { return __shfl_sync(gmask, v, src, G); }
    template <class T> __device__ __forceinline__ T up(T v, int d) const { return __shfl_up_sync(gmask, v, d, G); }
    template <class T> __device__ __forceinline__ T down(T v, int d) const { return __shfl_down_sync(gmask, v, d, G); }
    __device__ __forceinline__ void sync() const { __syncwarp(gmask); }
    __device__ __forceinline__ u32 incl_scan(u32 v) const {
#pragma unroll
        for (int d = 1; d < G; d <<= 1) { const u32 t = up(v, d); if (gl >= (u32)d) v += t; }
        return v;
    }
    __device__ __forceinline__ u32 excl_scan(u32 v, u32& total) const {
        const u32 incl = incl_scan(v);
        total = shfl(incl, G - 1);
        return incl - v;
    }
};

// ---- SWAR byte classification ------------------------------------------------------------
__device__ __forceinline__ u32 zero_bytes(u32 x) { return ~(((x & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | x) & 0x80808080u; }
__device__ __forceinline__ u32 movemask4(u32 m) { return ((m >> 7) * 0x01020408u) >> 24; }   // bit7 of byte k -> bit k
__device__ __forceinline__ u32 nondigit_bytes(u32 w) {
    const u32 hi3 = zero_bytes((w & 0xF0F0F0F0u) ^ 0x30303030u);            // high nibble == 3
    const u32 gt9 = (((w & 0x0F0F0F0Fu) + 0x06060606u) & 0x10101010u) << 3;   // low nibble >= 10
    return ~(hi3 & ~gt9) & 0x80808080u;
}
__device__ __forceinline__ u32 range16(int lo, int hi) {   // bits [lo, hi) of a 16-bit chunk mask
    lo = lo < 0 ? 0 : (lo > 16 ? 16 : lo);
    hi = hi < 0 ? 0 : (hi > 16 ? 16 : hi);
    return hi > lo ? (((1u << hi) - 1u) & ~((1u << lo) - 1u)) : 0u;
}

// 16 bytes from an arbitrarily aligned shared-memory address.
__device__ __forceinline__ void lds16_unaligned(const u8* p, u32& w0, u32& w1, u32& w2, u32& w3) {
    const uintptr_t a = reinterpret_cast<uintptr_t>(p);
    const u32* q = reinterpret_cast<const u32*>(a & ~(uintptr_t)3);
    const u32 sh = (u32)(a & 3) * 8;
    const u32 x0 = q[0], x1 = q[1], x2 = q[2], x3 = q[3], x4 = q[4];
    w0 = __funnelshift_r(x0, x1, sh); w1 = __funnelshift_r(x1, x2, sh);
    w2 = __funnelshift_r(x2, x3, sh); w3 = __funnelshift_r(x3, x4, sh);
}
__device__ __forceinline__ u32 keep_bytes(u32 w, int n) {   // keep the n lowest bytes of w (n may be <0 or >4)
    return n >= 4 ? w : (n <= 0 ? 0u : (w & ((1u << (8 * n)) - 1u)));
}

// ---- decimal helpers (32-bit) -------------------------------------------------------------
__device__ __forceinline__ u32 dlen_u32(u32 v, const u32* p10) {
    const u32 t = ((32u - (u32)__clz((int)(v | 1u))) * 1233u) >> 12;   // floor(log10) or one more
    return t + 1u - (u32)((v | 1u) < p10[t]);
}
__device__ __forceinline__ u32 dlen_i32(i32 v, const u32* p10) { return v < 0 ? 1u + dlen_u32(0u - (u32)v, p10) : dlen_u32((u32)v, p10); }
// gi:f: text for 0 <= floor(m/b*1000+0.5) <= 1000 (gaf2paf_main.cpp:248-253); returns 0 if outside.
// The text is returned packed (byte k of the text in bits [8k, 8k+8) of `pack`) so that it lives
// in registers and never forces a local-memory array.
__device__ __forceinline__ u32 gi_fast(i32 m, i32 b, u64& pack) {
    pack = '0';
    if (b <= 0) return 1;
    const double x = __ddiv_rn((double)m, (double)b);
    const double k = floor(__dadd_rn(__dmul_rn(x, 1000.0), 0.5));
    if (!(k >= 0.0 && k <= 1000.0)) return 0;
    const u32 ki = (u32)k;
    if (ki == 0) return 1;
    if (ki == 1000) { pack = '1'; return 1; }
    const u32 d0 = ki / 100, d1 = (ki / 10) % 10, d2 = ki % 10;
    pack = (u64)'0' | ((u64)'.' << 8) | ((u64)('0' + d0) << 16) | ((u64)('0' + d1) << 24) | ((u64)('0' + d2) << 32);
    return d2 ? 5 : (d1 ? 4 : 3);
}


// ---- record header: columns 1..12 and the optional tags, one lane per field ---------------
// (parse_gaf_record, gafkluge.hpp:84-204).  `rt` is the record text (shared or global memory),
// tabs[nt] its tab positions (11 <= nt <= kSMaxTabs), tkeys a scratch of kSMaxTags words.
// Results go to hdr[]; the return value is this lane's "not canonical" flag.  The caller must
// have zeroed hdr[H_CG_A..H_RC_B] and synchronised the group.  Ends with hdr/tkeys written but
// not yet synchronised for other lanes: the caller's next group vote orders them.
template <int G, class TabT>
__device__ __forceinline__ u32 parse_fields(const Grp<G>& g, const u8* rt, const TabT* tabs, u32 nt, u32 len, u32* hdr, u32* tkeys) {
    u32 lbad = 0;
    for (u32 f = g.gl; f < 12; f += G) {
        const u32 fa = f ? (u32)tabs[f - 1] + 1u : 0u;
        const u32 fb = f < nt ? (u32)tabs[f] : len;
        const u32 fl = fb - fa;
        if (fl == 0) { lbad = 1; continue; }
        if (f == 0) { hdr[H_QN_B] = fb; }
        else if (f == 4) {
            const u8 c = rt[fa];
            if (fl != 1 || (c != '+' && c != '-')) lbad = 1;
            hdr[H_MINUS] = c == '-';
        } else if (f == 5) { hdr[H_PATH_A] = fa; hdr[H_PATH_B] = fb; }
        else {
            i32 v = 0;
            if (fl == 1 && rt[fa] == '*') v = -1;
            else if (fl > 9) lbad = 1;
            else {
                u32 x = 0;
                for (u32 k = fa; k < fb; ++k) { const u32 d = (u32)rt[k] - '0'; if (d > 9) lbad = 1; x = x * 10u + d; }
                v = (i32)x;
                if (f == 11 && v >= 255) v = -1;   // gafkluge.hpp:176-183
            }
            hdr[f] = (u32)v;
        }
    }
    const u32 ntf = nt - 11;   // tag fields (possibly empty ones)
    for (u32 t0 = 0; t0 < ntf; t0 += G) {
        const u32 ti = t0 + g.gl;
        if (ti < ntf) {
            const u32 f = 12 + ti;
            const u32 fa = (u32)tabs[f - 1] + 1u, fb = f < nt ? (u32)tabs[f] : len, fl = fb - fa;
            u32 key = 0x10000u + ti;   // empty field: unique non-key
            if (fl) {
                if (fl < 5 || rt[fa + 2] != ':' || rt[fa + 4] != ':') lbad = 1;
                else {
                    key = (u32)rt[fa] | ((u32)rt[fa + 1] << 8);
                    if (key == ((u32)'c' | ((u32)'g' << 8))) { hdr[H_CG_A] = fa + 5; hdr[H_CG_B] = fb; }
                    else if (key == ((u32)'t' | ((u32)'p' << 8))) { hdr[H_TP_A] = fa + 3; hdr[H_TP_B] = fb; }
                    else if (key == ((u32)'r' | ((u32)'c' << 8))) { hdr[H_RC_A] = fa + 3; hdr[H_RC_B] = fb; }
                }
            }
            tkeys[ti] = key;
        }
    }
    g.sync();
    for (u32 t0 = 0; t0 < ntf; t0 += G) {   // duplicate tags (gafkluge.hpp:195-198)
        const u32 ti = t0 + g.gl;
        if (ti < ntf) {
            const u32 key = tkeys[ti];
            for (u32 j = 0; j < ti; ++j) if (tkeys[j] == key) lbad = 1;
        }
    }
    return lbad;
}

// ---- one PAF line (paf.hpp:83-95 + gaf2paf_main.cpp:228-256) -------------------------------
struct LineRec {    // constant over the lines of one record
    u32 qn_b;
    i32 qlen, mapq, m, b;
    u32 tp_a, tp_b, rc_a, rc_b;   // "type:value" spans of the tp / rc tags (b == 0: absent)
    u32 gi_n;
    u64 gi;               // gi:f: value text, byte k in bits [8k, 8k+8)
};
struct LineStep {
    u32 q0, q1, name_a, nl, tlen, ts, te, nm, nb;
    u32 lenS, lenE;        // explicit first / last piece lengths
    u32 mid_a, mid_b;      // text span of the pieces copied verbatim (empty if mid_b <= mid_a)
    u8 codeS, codeE;       // codeS == 0: no explicit first piece
    bool rev, mid_fwd;     // mid_fwd: the verbatim span is printed in text order
};
__device__ __forceinline__ u32 line_const_len(const LineRec& R, const u32* p10) {
    return R.qn_b + dlen_i32(R.qlen, p10) + 12u + dlen_i32(R.mapq, p10) + (R.tp_b ? 4u + (R.tp_b - R.tp_a) : 0u) +
           (R.rc_b ? 4u + (R.rc_b - R.rc_a) : 0u) + 6u + dlen_i32(R.m, p10) + 6u + dlen_i32(R.b, p10) + 6u + R.gi_n + 6u + 1u;
}
__device__ __forceinline__ u32 line_step_len(const LineStep& L, const u32* p10) {
    u32 n = L.nl + dlen_u32(L.q0, p10) + dlen_u32(L.q1, p10) + dlen_u32(L.tlen, p10) + dlen_u32(L.ts, p10) + dlen_u32(L.te, p10) +
            dlen_u32(L.nm, p10) + dlen_u32(L.nb, p10) + dlen_u32(L.lenE, p10) + 1u;
    if (L.codeS) n += dlen_u32(L.lenS, p10) + 1u;
    if (L.mid_b > L.mid_a) n += L.mid_b - L.mid_a;
    return n;
}
// Right-to-left writers: the line's length is known from the size pass, so the line is written
// from its last byte backwards -- decimal digits come out in the order they are produced and no
// digit-count pass is needed.
__device__ __forceinline__ u8* rput_u32(u8* p, u32 v) {
    do { const u32 q = v / 10u; *--p = (u8)('0' + (v - q * 10u)); v = q; } while (v);
    return p;
}
__device__ __forceinline__ u8* rput_i32(u8* p, i32 v) {
    if (v < 0) { p = rput_u32(p, 0u - (u32)v); *--p = '-'; return p; }
    return rput_u32(p, (u32)v);
}
__device__ __forceinline__ u8* rput_bytes(u8* p, const u8* s, u32 n) {
    for (u32 i = n; i-- > 0;) *--p = s[i];
    return p;
}
// The n bytes of a run of whole CIGAR tokens ("digits letter" with at most 8 digits, which every size pass checks) at
// src go to dst (either at any alignment), in text order or, with rev, in reverse token order with each token
// forwards: the byte at position i of the token [s, e] goes to dst[n-1-e + i-s].  The text is read as the aligned
// 32-bit words that hold it (never a word past it), four bytes per step; the token ends come from a rolling mask of
// the op letters among the next 12 bytes.  So every lane runs the same flat loop whatever the direction and the token
// structure of its text, where the nested scan-and-copy loops ran at 2-5 of 32 lanes on short-read lines.
__device__ __forceinline__ void put_tokens(u8* dst, const u8* src, u32 n, bool rev) {
    const uintptr_t sa = reinterpret_cast<uintptr_t>(src);
    const u32* sp = reinterpret_cast<const u32*>(sa & ~(uintptr_t)3);
    const u32 s8 = (u32)(sa & 3u) * 8u;
    const u32 na = n ? ((u32)(sa & 3u) + n + 3u) >> 2 : 0u;   // aligned words that hold the text
    auto ld = [&](u32 j) -> u32 { return j < na ? sp[j] : 0u; };
    auto letters = [](u32 w) -> u32 { return movemask4(nondigit_bytes(w)); };
    const u32 x0 = ld(0), x1 = ld(1), x2 = ld(2);
    u32 x3 = ld(3);
    u32 w0 = __funnelshift_r(x0, x1, s8), w1 = __funnelshift_r(x1, x2, s8), w2 = __funnelshift_r(x2, x3, s8);
    u32 roll = letters(w0) | (letters(w1) << 4) | (letters(w2) << 8);   // bit t: byte 4k + t is an op letter
    u32 s = 0;                                                          // start of the token that byte 4k is in
    for (u32 k = 0; 4u * k < n; ++k) {
#pragma unroll
        for (u32 b = 0; b < 4; ++b) {
            const u32 i = 4u * k + b;
            const u32 below = roll & ((1u << b) - 1u);
            const u32 ts = below ? 4u * k + 32u - (u32)__clz((int)below) : s;   // token start
            const u32 te = i + (u32)__ffs((int)(roll >> b)) - 1u;                // its op letter
            if (i < n) dst[rev ? n - 1u - te + i - ts : i] = (u8)(w0 >> (8u * b));
        }
        if (roll & 0xfu) s = 4u * k + 32u - (u32)__clz((int)(roll & 0xfu));
        const u32 x4 = ld(k + 4u);
        w0 = w1; w1 = w2; w2 = __funnelshift_r(x3, x4, s8); x3 = x4;
        roll = (roll >> 4) | (letters(w2) << 8);
    }
}
__device__ __forceinline__ u8* rput_tag(u8* p, u8 a, u8 b, u8 t) {   // "\tab:t:"
    p -= 6;
    p[0] = '\t'; p[1] = a; p[2] = b; p[3] = ':'; p[4] = t; p[5] = ':';
    return p;
}
// Where the variable-length pieces of a line are read from (any address space).
struct LineSrc {
    const u8* qname;   // R.qn_b bytes
    const u8* name;    // L.nl bytes
    const u8* tp;      // R.tp_b - R.tp_a bytes ("type:value")
    const u8* rc;
    const u8* mid;     // L.mid_b - L.mid_a bytes of CIGAR text copied verbatim
};
__device__ __forceinline__ LineSrc line_src(const u8* rt, const LineRec& R, const LineStep& L) {   // everything inside one record buffer
    LineSrc S;
    S.qname = rt; S.name = rt + L.name_a; S.tp = rt + R.tp_a; S.rc = rt + R.rc_a; S.mid = rt + L.mid_a;
    return S;
}
// Writes the line that ends at `pend` (exclusive); returns its first byte.  FLAT_MID: the verbatim CIGAR middle is
// printed by put_tokens once the other fields are written; else by byte loops, a token scan nested in a per-token copy
// for a reversed middle.  The flat loop pays on short-read lines (k_emit_lines<false>: emit 2.39 -> 2.21 ms per 10 M
// records on a B200) and costs on the long middles of 2 kB records (k_emit_lines<true>: 3.39 -> 3.62 ms).
template <bool FLAT_MID>
__device__ __forceinline__ u8* write_line(u8* pend, const LineSrc& S, const LineRec& R, const LineStep& L) {
    u8* p = pend;
    *--p = '\n';
    // pieces, reversed for '<' steps (gaf2paf_main.cpp:184-211); here in reverse output order
    if (!L.rev) { *--p = L.codeE; p = rput_u32(p, L.lenE); }
    else if (L.codeS) { *--p = L.codeS; p = rput_u32(p, L.lenS); }
    const u32 mlen = L.mid_b > L.mid_a ? L.mid_b - L.mid_a : 0u;
    u8* const pmid = p - mlen;   // FLAT_MID: written last, when the other fields are no longer live
    if (FLAT_MID || mlen == 0) p = pmid;
    else if (L.mid_fwd) p = rput_bytes(p, S.mid, mlen);
    else {
        u32 t = 0;   // output order is the reverse token order: first text token is written last
        while (t < mlen) {
            u32 e = t;
            while (S.mid[e] <= '9') ++e;   // the op letter ends the token
            for (u32 k = e + 1; k-- > t;) *--p = S.mid[k];
            t = e + 1;
        }
    }
    if (!L.rev) { if (L.codeS) { *--p = L.codeS; p = rput_u32(p, L.lenS); } }
    else { *--p = L.codeE; p = rput_u32(p, L.lenE); }
    p = rput_tag(p, 'c', 'g', 'Z');
    for (u32 i = R.gi_n; i-- > 0;) *--p = (u8)(R.gi >> (8 * i));
    p = rput_tag(p, 'g', 'i', 'f');
    p = rput_i32(p, R.b); p = rput_tag(p, 'g', 'l', 'i');
    p = rput_i32(p, R.m); p = rput_tag(p, 'g', 'm', 'i');
    if (R.rc_b) { p = rput_bytes(p, S.rc, R.rc_b - R.rc_a); p -= 4; p[0] = '\t'; p[1] = 'r'; p[2] = 'c'; p[3] = ':'; }
    if (R.tp_b) { p = rput_bytes(p, S.tp, R.tp_b - R.tp_a); p -= 4; p[0] = '\t'; p[1] = 't'; p[2] = 'p'; p[3] = ':'; }
    p = rput_i32(p, R.mapq); *--p = '\t';
    p = rput_u32(p, L.nb); *--p = '\t';
    p = rput_u32(p, L.nm); *--p = '\t';
    p = rput_u32(p, L.te); *--p = '\t';
    p = rput_u32(p, L.ts); *--p = '\t';
    p = rput_u32(p, L.tlen); *--p = '\t';
    p = rput_bytes(p, S.name, L.nl); *--p = '\t';
    *--p = L.rev ? '-' : '+'; *--p = '\t';
    p = rput_u32(p, L.q1); *--p = '\t';
    p = rput_u32(p, L.q0); *--p = '\t';
    p = rput_i32(p, R.qlen); *--p = '\t';
    p = rput_bytes(p, S.qname, R.qn_b);
    if (FLAT_MID) put_tokens(pmid, S.mid, mlen, !L.mid_fwd);
    return p;
}

// ---- left-to-right line writer: 32-bit words into (word-aligned) shared memory ------------------
struct WEmit {
    u32* wp;
    u32 lo, sh;   // pending bytes: the low `sh` bits of lo (sh in {0, 8, 16, 24})
    __device__ __forceinline__ void put(u32 v, u32 nbytes) {   // the nbytes low bytes of v (the rest zero), 1 <= nbytes <= 4
        lo |= v << sh;
        const u32 hi = __funnelshift_l(v, 0u, sh);   // what does not fit (0 when sh == 0)
        sh += 8u * nbytes;
        const u32 full = sh >> 5;                    // 0 or 1; straight-line code: one predicated store, selects
        if (full) *wp = lo;
        wp += full;
        lo = full ? hi : lo;
        sh &= 31u;
    }
    __device__ __forceinline__ void put4(u32 v) {
        *wp++ = lo | (v << sh);
        lo = __funnelshift_l(v, 0u, sh);
    }
    // n bytes from an arbitrarily aligned shared-memory address (reads up to 7 bytes past the span)
    __device__ __forceinline__ void copy(const u8* src, u32 n) {
        const uintptr_t sa = reinterpret_cast<uintptr_t>(src);
        const u32* sp = reinterpret_cast<const u32*>(sa & ~(uintptr_t)3);
        const u32 s8 = (u32)(sa & 3u) * 8u;
        u32 prev = *sp++;
        while (n >= 4u) {
            const u32 cur = *sp++;
            put4(__funnelshift_r(prev, cur, s8));
            prev = cur;
            n -= 4u;
        }
        if (n) {
            const u32 cur = *sp;
            put(__funnelshift_r(prev, cur, s8) & ((1u << (8u * n)) - 1u), n);
        }
    }
    // n <= 8 bytes (the short verbatim fields: tag values, column texts): no loop
    __device__ __forceinline__ void copy_small(const u8* src, u32 n) {
        const uintptr_t sa = reinterpret_cast<uintptr_t>(src);
        const u32* sp = reinterpret_cast<const u32*>(sa & ~(uintptr_t)3);
        const u32 s8 = (u32)(sa & 3u) * 8u;
        const u32 x0 = sp[0], x1 = sp[1];
        const u32 w0 = __funnelshift_r(x0, x1, s8);
        if (n <= 4u) { put(n == 4u ? w0 : w0 & ((1u << (8u * n)) - 1u), n); return; }
        const u32 w1 = __funnelshift_r(x1, sp[2], s8);
        put4(w0);
        put(n == 8u ? w1 : w1 & ((1u << (8u * (n - 4u))) - 1u), n - 4u);
    }
    // decimal digits of x < 10000, zero padded to four, most significant digit in the low byte
    static __device__ __forceinline__ u32 pack4(u32 x) {
        const u32 d3 = x / 1000u, r3 = x - d3 * 1000u, d2 = r3 / 100u, r2 = r3 - d2 * 100u, d1 = r2 / 10u, d0 = r2 - d1 * 10u;
        return (d3 | (d2 << 8) | (d1 << 16) | (d0 << 24)) + 0x30303030u;
    }
    __device__ __forceinline__ void num_unpadded4(u32 x) {   // x < 10000
        const u32 nd = 1u + (u32)(x >= 10u) + (u32)(x >= 100u) + (u32)(x >= 1000u);
        put(pack4(x) >> (8u * (4u - nd)), nd);
    }
    // decimal v followed by the byte sep
    __device__ __forceinline__ void num(u32 v, u32 sep) {
        if (v < 1000u) {   // digits and separator in one append
            const u32 d2 = v / 100u, r = v - d2 * 100u, d1 = r / 10u, d0 = r - d1 * 10u;
            const u32 nd = 1u + (u32)(v >= 10u) + (u32)(v >= 100u);
            const u32 w = ((d2 | (d1 << 8) | (d0 << 16)) + 0x303030u) | (sep << 24);
            put(w >> (8u * (3u - nd)), nd + 1u);
            return;
        }
        const u32 hi = v / 10000u, lo4 = v - hi * 10000u;
        if (hi == 0u) put4(pack4(lo4));
        else {
            const u32 hh = hi / 10000u, hl = hi - hh * 10000u;
            if (hh == 0u) num_unpadded4(hl);
            else { num_unpadded4(hh); put4(pack4(hl)); }
            put4(pack4(lo4));
        }
        put(sep, 1u);
    }
};

// ---- line descriptors: what the size pass hands to k_emit_lines ---------------------------
// One 64-byte descriptor per PAF line and one 32-byte header per record; k_emit_lines formats
// one line per thread from them without parsing the record again.
struct __align__(16) LineDesc {
    u32 rec;              // record index (0xFFFFFFFF: padding slot)
    u32 loff;             // byte offset of the line inside the record's output
    u32 q0, q1;
    u32 tlen, ts, te, nm;
    u32 nb, lenS, lenE;
    u32 name_a;           // record-relative offsets of the name and of the verbatim CIGAR span
    u32 mid_a, mid_len;
    u32 len;              // bytes of the whole line
    u8 nl, codeS, codeE, flags;   // flags: bit0 rev, bit1 mid_fwd
};
static_assert(sizeof(LineDesc) == 64, "LineDesc is four 16-byte vectors");
struct __align__(16) RecDesc {
    i32 qlen, m, b;
    i32 mapq;
    u32 tp_a, rc_a;       // record-relative offsets of the "type:value" text of tp / rc
    u16 qn_b, tp_len, rc_len;
    u8 gi_n, pad0;
    u8 gi[5];
    u8 pad1[11];
};
static_assert(sizeof(RecDesc) == 48, "RecDesc is three 16-byte vectors");
// Descriptors are packed to / unpacked from four (three) 16-byte vectors in registers: no struct
// whose address is taken, hence no local-memory traffic on either side.
__device__ __forceinline__ void store_line_desc(LineDesc* dst, u32 rec, u32 loff, u32 line, const LineStep& L) {
    uint4* out = reinterpret_cast<uint4*>(dst);
    out[0] = make_uint4(rec, loff, L.q0, L.q1);
    out[1] = make_uint4(L.tlen, L.ts, L.te, L.nm);
    out[2] = make_uint4(L.nb, L.lenS, L.lenE, L.name_a);
    out[3] = make_uint4(L.mid_a, L.mid_b > L.mid_a ? L.mid_b - L.mid_a : 0u, line,
                        (L.nl & 0xffu) | ((u32)L.codeS << 8) | ((u32)L.codeE << 16) | ((L.rev ? 1u : 0u) << 24) | ((L.mid_fwd ? 2u : 0u) << 24));
}
__device__ __forceinline__ void unpack_line_desc(const uint4& v0, const uint4& v1, const uint4& v2, const uint4& v3, u32& rec, u32& loff, u32& line,
                                                 LineStep& L) {
    rec = v0.x; loff = v0.y; L.q0 = v0.z; L.q1 = v0.w;
    L.tlen = v1.x; L.ts = v1.y; L.te = v1.z; L.nm = v1.w;
    L.nb = v2.x; L.lenS = v2.y; L.lenE = v2.z; L.name_a = v2.w;
    L.mid_a = v3.x; L.mid_b = v3.x + v3.y; line = v3.z;
    L.nl = v3.w & 0xffu; L.codeS = (u8)(v3.w >> 8); L.codeE = (u8)(v3.w >> 16);
    L.rev = ((v3.w >> 24) & 1u) != 0; L.mid_fwd = ((v3.w >> 24) & 2u) != 0;
}
// false when the record's constants do not fit the descriptor (very long name / tag text)
__device__ __forceinline__ bool rec_desc_fits(const LineRec& R) { return R.qn_b <= 0xffffu && R.tp_b - R.tp_a <= 0xffffu && R.rc_b - R.rc_a <= 0xffffu; }
__device__ __forceinline__ void store_rec_desc(RecDesc* dst, const LineRec& R) {
    uint4* out = reinterpret_cast<uint4*>(dst);
    out[0] = make_uint4((u32)R.qlen, (u32)R.m, (u32)R.b, (u32)R.mapq);
    out[1] = make_uint4(R.tp_a, R.rc_a, (R.qn_b & 0xffffu) | ((R.tp_b - R.tp_a) << 16), ((R.rc_b - R.rc_a) & 0xffffu) | (R.gi_n << 16));
    out[2] = make_uint4((u32)R.gi, (u32)(R.gi >> 32), 0u, 0u);
}
__device__ __forceinline__ void unpack_rec_desc(const uint4& v0, const uint4& v1, const uint4& v2, LineRec& R) {
    R.qlen = (i32)v0.x; R.m = (i32)v0.y; R.b = (i32)v0.z; R.mapq = (i32)v0.w;
    const u32 tp_len = v1.z >> 16, rc_len = v1.w & 0xffffu;
    R.qn_b = v1.z & 0xffffu;
    R.tp_a = v1.x; R.tp_b = tp_len ? v1.x + tp_len : 0u;
    R.rc_a = v1.y; R.rc_b = rc_len ? v1.y + rc_len : 0u;
    R.gi_n = (v1.w >> 16) & 0xffu;
    R.gi = (u64)v2.x | ((u64)v2.y << 32);
}
constexpr u32 kDescInvalid = 0xFFFFFFFFu;

__device__ __forceinline__ uint4 ldg_vec_guarded(const u8* base, u64 off, u64 n) {
    if (off + 16 <= n) return __ldg(reinterpret_cast<const uint4*>(base + off));
    u32 w[4] = {0, 0, 0, 0};
    for (u32 i = 0; i < 16; ++i)
        if (off + i < n) w[i >> 2] |= (u32)base[off + i] << (8 * (i & 3));
    return make_uint4(w[0], w[1], w[2], w[3]);
}

#if defined(G2P_HOSTSIM)
#define G2P_DYN_SMEM(name) u8* name = hs::g_dyn_smem
#else
#define G2P_DYN_SMEM(name) extern __shared__ __align__(16) u8 name[]
#endif

struct ShortArgs {
    const u8* gaf;
    u64 n;
    const u32* rec_start;
    u32 nrec;
    LenTableView T;
    u64* out_off;        // per-record PAF byte count (scanned into offsets afterwards)
    u64* line_off;       // per-record PAF line count (scanned into line offsets afterwards)
    u32* status;
    u32* deleg_list;     // indices of records left to k_long / the general kernel
    u32* n_deleg;
    LineDesc* sdesc;     // line descriptors: record r owns slots [r * kSMaxLines, (r + 1) * kSMaxLines)
    RecDesc* rdesc;      // per-record constants of the lines
};

// One record per G-lane group: PAF size, status and one line descriptor per PAF line -- or the
// record is delegated.
template <int G>
__global__ void __launch_bounds__(kSThreads, G2P_SHORT_CTAS) k_short(const ShortArgs a) {
    G2P_DYN_SMEM(smem);
    __shared__ u32 p10[10];
    if (threadIdx.x < 10) {
        u32 v = 1;
        for (u32 i = 0; i < threadIdx.x; ++i) v *= 10u;
        p10[threadIdx.x] = v;
    }
    __syncthreads();

    const Grp<G> g;
    const u32 gid = threadIdx.x / G;
    SGroupMem* gm = reinterpret_cast<SGroupMem*>(smem) + gid;
    const u32 r = blockIdx.x * (kSThreads / G) + gid;
    if (r >= a.nrec) return;
    const u32 s = a.rec_start[r], e = a.rec_start[r + 1];
    const u32 len = e - s - 1;

    bool deleg = false;      // group-uniform
    u32 size = 0;
    u32 status = ST_OK | ST_F_FAST;
    LineRec R;
    LineStep L;
    bool emit_line = false;
    u32 line = 0, loff = 0;
    do {
        if (len == 0 || len > kSLimit) { deleg = true; break; }
        // ---------------- phase 0: stage + classify
        const u32 A = s & ~15u, sh = s - A;
        const u32 nchunks = (sh + len + 15) >> 4;   // <= 16
        const u8* rt = gm->text + sh;
        constexpr int NIT = (16 + G - 1) / G;
        u32 tabm[NIT], mrkm[NIT], ndgm[NIT];
#pragma unroll
        for (int it = 0; it < NIT; ++it) {
            const u32 c = it * G + g.gl;
            tabm[it] = mrkm[it] = ndgm[it] = 0;
            if (c < nchunks) {
                const uint4 v = ldg_vec_guarded(a.gaf, (u64)A + 16u * c, a.n);
                reinterpret_cast<uint4*>(gm->text)[c] = v;
                const u32 w[4] = {v.x, v.y, v.z, v.w};
                u32 t = 0, m = 0, d = 0;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    t |= movemask4(zero_bytes(w[k] ^ 0x09090909u)) << (4 * k);
                    m |= movemask4(zero_bytes((w[k] & 0xFDFDFDFDu) ^ 0x3C3C3C3Cu)) << (4 * k);
                    d |= movemask4(nondigit_bytes(w[k])) << (4 * k);
                }
                const u32 vm = range16((int)sh - 16 * (int)c, (int)(sh + len) - 16 * (int)c);
                tabm[it] = t & vm; mrkm[it] = m & vm; ndgm[it] = d & vm;
            }
        }
        if (g.gl < 6) gm->hdr[H_CG_A + g.gl] = 0;
        u32 nt = 0;
#pragma unroll
        for (int it = 0; it < NIT; ++it) {
            u32 tot;
            u32 k = nt + g.excl_scan((u32)__popc(tabm[it]), tot);
            u32 m = tabm[it];
            const u32 base = 16u * (it * G + g.gl) - sh;
            while (m) {
                const u32 b = (u32)__ffs((int)m) - 1u;
                m &= m - 1u;
                if (k < 32) gm->tabs[k] = (u16)(base + b);
                ++k;
            }
            nt += tot;
        }
        g.sync();
        if (rt[0] == '*') { status = ST_SKIP | ST_F_FAST; break; }   // gaf2paf_main.cpp:360
        if (nt < 11 || nt > kSMaxTabs) { deleg = true; break; }
        // ---------------- phase 1: columns 1..12 and tags, one lane per field
        u32 lbad = parse_fields<G>(g, rt, gm->tabs, nt, len, gm->hdr, reinterpret_cast<u32*>(gm->spos));
        if (g.any(lbad != 0)) { deleg = true; break; }   // also orders the tkeys reads before the scatter below

        const bool minus = gm->hdr[H_MINUS] != 0;
        const i32 qs = (i32)gm->hdr[H_QS], ps = (i32)gm->hdr[H_PS], pe = (i32)gm->hdr[H_PE];
        const u32 ca = gm->hdr[H_CG_A], cb = gm->hdr[H_CG_B];
        const u32 pa = gm->hdr[H_PATH_A], pb = gm->hdr[H_PATH_B];
        if (cb == 0 || ca >= cb || qs < 0 || ps < 0 || pe < 0) { deleg = true; break; }
        const u8 c0 = rt[pa];
        const bool prefixed = c0 == '>' || c0 == '<';
        const bool empty_path = !prefixed && pb - pa == 1 && c0 == '*';

        // ---------------- phase 2: step markers and op letters -> positions
        u32 ns = 0, no = 0;
#pragma unroll
        for (int it = 0; it < NIT; ++it) {
            const int base = 16 * (it * G + (int)g.gl) - (int)sh;
            u32 mm = prefixed ? (mrkm[it] & range16((int)pa - base, (int)pb - base)) : 0u;
            u32 dm = ndgm[it] & range16((int)ca - base, (int)cb - base);
            u32 tot;
            const u32 ex = g.excl_scan((u32)__popc(mm) | ((u32)__popc(dm) << 16), tot);
            u32 k = ns + (ex & 0xffffu);
            while (mm) {
                const u32 b = (u32)__ffs((int)mm) - 1u;
                mm &= mm - 1u;
                if (k < 15) gm->spos[k] = (u16)(base + (int)b);
                ++k;
            }
            k = no + (ex >> 16);
            while (dm) {
                const u32 b = (u32)__ffs((int)dm) - 1u;
                dm &= dm - 1u;
                if (k < kSMaxOps) gm->opos[k] = (u16)(base + (int)b);
                ++k;
            }
            ns += tot & 0xffffu;
            no += tot >> 16;
        }
        if (!prefixed) ns = empty_path ? 0u : 1u;
        if (ns > (u32)(G - 1) || no == 0 || no > kSMaxOps) { deleg = true; break; }
        if (prefixed && g.gl == 0) gm->spos[ns] = (u16)pb;
        g.sync();
        if (gm->opos[no - 1] != cb - 1) { deleg = true; break; }   // digits after the last op letter

        // ---------------- phase 3: one lane per path step
        const u32 i = g.gl;             // normalised step index (and boundary index)
        const bool is_step = i < ns;
        u32 name_a = 0, nl = 0;
        i32 tlen = 0, sa = 0, se = 0;
        bool rev = false;
        if (is_step) {
            const u32 so_ = minus ? ns - 1 - i : i;
            u32 p, q;
            if (prefixed) { p = gm->spos[so_]; q = gm->spos[so_ + 1]; } else { p = pa - 1; q = pb; }
            rev = (prefixed && rt[p] == '<') != minus;
            name_a = p + 1;
            const u32 tl = q - name_a;
            u32 w0, w1, w2, w3;
            lds16_unaligned(rt + name_a, w0, w1, w2, w3);
            bool interval = false;
            nl = tl;
            if (prefixed) {
                u32 cm = movemask4(zero_bytes(w0 ^ 0x3A3A3A3Au)) | (movemask4(zero_bytes(w1 ^ 0x3A3A3A3Au)) << 4) |
                         (movemask4(zero_bytes(w2 ^ 0x3A3A3A3Au)) << 8) | (movemask4(zero_bytes(w3 ^ 0x3A3A3A3Au)) << 12);
                cm &= tl >= 16 ? 0xffffu : ((1u << tl) - 1u);
                if (cm) { nl = (u32)__ffs((int)cm) - 1u; interval = true; }
            }
            if (nl == 0 || nl > 16) lbad = 1;
            else {
                w0 = keep_bytes(w0, (int)nl); w1 = keep_bytes(w1, (int)nl - 4);
                w2 = keep_bytes(w2, (int)nl - 8); w3 = keep_bytes(w3, (int)nl - 12);
                i64 tl64 = 0;
                if (!table_lookup_key16(a.T, (u64)w0 | ((u64)w1 << 32), (u64)w2 | ((u64)w3 << 32), nl, tl64)) lbad = 1;
                else if (tl64 < 0 || tl64 > 0x7fffffffLL) lbad = 1;
                tlen = (i32)tl64;
                se = tlen;
                if (interval) {   // ":start-end" (gafkluge.hpp:131-146), plain digits only
                    u32 k = name_a + nl + 1, x = 0, nd = 0;
                    while (k < q && nd < 10) { const u32 d = (u32)rt[k] - '0'; if (d > 9) break; x = x * 10u + d; ++nd; ++k; }
                    if (nd == 0 || nd > 9 || k >= q || rt[k] != '-') lbad = 1;
                    sa = (i32)x;
                    ++k; x = 0; nd = 0;
                    while (k < q && nd < 10) { const u32 d = (u32)rt[k] - '0'; if (d > 9) break; x = x * 10u + d; ++nd; ++k; }
                    if (nd == 0 || nd > 9 || k != q) lbad = 1;
                    se = (i32)x;
                }
            }
        }
        const i32 slen = se - sa;
        if (is_step && slen < 0) lbad = 1;
        // flip_gaf: mirror the path interval about the summed step lengths (gaf2paf_main.cpp:111-131)
        i32 ps2 = ps, pe2 = pe;
        if (minus) {
            u32 lo = is_step && !lbad ? (u32)slen : 0u, hi = 0;   // 64-bit sum in two halves
#pragma unroll
            for (int d = 1; d < G; d <<= 1) {
                const u32 tlo = g.up(lo, d), thi = g.up(hi, d);
                if (g.gl >= (u32)d) { const u32 nlo = lo + tlo; hi += thi + (nlo < lo); lo = nlo; }
            }
            lo = g.shfl(lo, G - 1); hi = g.shfl(hi, G - 1);
            if (hi != 0 || lo > 0x7fffffffu) lbad = 1;
            ps2 = (i32)lo - pe; pe2 = (i32)lo - ps;
        }
        // quotas (gaf2paf_main.cpp:176-182) and cumulative boundaries B_i (Appendix B.3)
        const i32 W = pe2 - ps2;
        const i32 so = (i == 0) ? ps2 : 0;
        const bool is_last = is_step && i + 1 == ns;
        u32 tbc;
        u32 B = g.excl_scan(is_step && !is_last ? (u32)(slen - so) : 0u, tbc);
        i32 quota = slen - so, eo = 0;
        if (is_last) { quota = W - (i32)tbc; eo = slen - so - quota; }
        if (is_step && (so < 0 || quota < 0 || eo < 0)) lbad = 1;   // :178 assert / negative quota
        if (!is_step) { quota = 0; if (i == ns) B = (u32)W; }
        if (g.any(lbad != 0)) { deleg = true; break; }

        // ---------------- phase 4: one lane per CIGAR op, inclusive prefix sums
        {
            u32 cE = 0, cQ = 0, cM = 0, cB = 0;
            for (u32 j0 = 0; j0 < no; j0 += G) {
                const u32 j = j0 + g.gl;
                u32 vE = 0, vQ = 0, vM = 0, vB = 0;
                if (j < no) {
                    const u32 oo = minus ? no - 1 - j : j;
                    const u32 lp = gm->opos[oo];
                    const u32 ds = oo ? gm->opos[oo - 1] + 1u : ca;
                    const u32 nd = lp - ds;
                    const u32 k = (u32)rt[lp] - '=';
                    if (k >= 28 || !((kOpMask >> k) & 1u) || nd == 0 || nd > 7 || (nd > 1 && rt[ds] == '0')) lbad = 1;
                    else {
                        u32 x = 0;
                        for (u32 t = ds; t < lp; ++t) x = x * 10u + ((u32)rt[t] - '0');
                        if (x == 0) lbad = 1;
                        vB = x;
                        vE = ((kTargetMask >> k) & 1u) ? x : 0u;
                        vQ = ((kQueryMask >> k) & 1u) ? x : 0u;
                        vM = ((kMatchMask >> k) & 1u) ? x : 0u;
                    }
                }
                vE = g.incl_scan(vE) + cE; vQ = g.incl_scan(vQ) + cQ; vM = g.incl_scan(vM) + cM; vB = g.incl_scan(vB) + cB;
                if (j < no) { gm->pEnd[j] = vE; gm->pQ[j] = vQ; gm->pNM[j] = vM; gm->pNB[j] = vB; }
                cE = g.shfl(vE, G - 1); cQ = g.shfl(vQ, G - 1); cM = g.shfl(vM, G - 1); cB = g.shfl(vB, G - 1);
            }
        }
        if (g.any(lbad != 0)) { deleg = true; break; }   // (also a group barrier for the prefix arrays)

        // ---------------- phase 5: boundary i -> position in the op stream (lanes 0..ns)
        u32 bj = 0, bt = 0, bCQ = 0, bCM = 0, bCB = 0;
        bool bcut = false, bexh = false;
        if (i <= ns && B != 0) {
            u32 lo = 0, hi = no;
            while (lo < hi) { const u32 mid = (lo + hi) >> 1; if (gm->pEnd[mid] >= B) hi = mid; else lo = mid + 1; }
            bj = lo;
            if (bj == no) bexh = true;
            else {
                const u32 Ej = gm->pEnd[bj];
                bt = bj ? gm->pEnd[bj - 1] : 0u;
                const u32 off = B - bt;
                const u32 k = (u32)rt[gm->opos[minus ? no - 1 - bj : bj]] - '=';
                bCQ = (bj ? gm->pQ[bj - 1] : 0u) + (((kQueryMask >> k) & 1u) ? off : 0u);
                bCM = (bj ? gm->pNM[bj - 1] : 0u) + (((kMatchMask >> k) & 1u) ? off : 0u);
                bCB = (bj ? gm->pNB[bj - 1] : 0u) + off;
                bcut = Ej > B;
            }
        }
        // the end boundary of step i is the start boundary of step i+1
        const u32 ej = g.down(bj, 1), et = g.down(bt, 1), eCQ = g.down(bCQ, 1), eCM = g.down(bCM, 1), eCB = g.down(bCB, 1);
        const u32 eB = g.down(B, 1);
        const bool eexh = g.down((u32)bexh, 1) != 0;
        const bool live = is_step && quota > 0;
        if (live && eexh) lbad = 1;   // :80 assert(cur_len > target_len): CIGAR shorter than the path
        if (g.any(lbad != 0)) { deleg = true; break; }
        const u32 q = live ? eCQ - bCQ : 0u, nm = live ? eCM - bCM : 0u, nb = live ? eCB - bCB : 0u;
        emit_line = live && nm > 0;   // :225

        // PAF columns (gaf2paf_main.cpp:214-217).  Query consumed before step i == CQ at its start
        // boundary (the per-step sums telescope), so no scan over steps is needed.
        R.qn_b = gm->hdr[H_QN_B];
        R.qlen = (i32)gm->hdr[H_QLEN]; R.m = (i32)gm->hdr[H_M]; R.b = (i32)gm->hdr[H_B]; R.mapq = (i32)gm->hdr[H_MAPQ];
        R.tp_a = gm->hdr[H_TP_A]; R.tp_b = gm->hdr[H_TP_B]; R.rc_a = gm->hdr[H_RC_A]; R.rc_b = gm->hdr[H_RC_B];
        R.gi_n = gi_fast(R.m, R.b, R.gi);
        if (R.gi_n == 0 || !rec_desc_fits(R)) { deleg = true; break; }   // uniform: same m, b in the whole group
        L.rev = rev;
        L.q0 = (u32)qs + bCQ; L.q1 = L.q0 + q;
        L.name_a = name_a; L.nl = nl; L.tlen = (u32)tlen;
        L.ts = (u32)(sa + (rev ? eo : so)); L.te = (u32)(se - (rev ? so : eo));
        L.nm = nm; L.nb = nb;
        // pieces of the step: ops jS..jE (normalised order); first / last explicit, the rest verbatim
        L.lenS = 0; L.codeS = 0; L.codeE = 0; L.mid_a = L.mid_b = 0;
        L.mid_fwd = rev == minus;   // text order == output order
        L.lenE = eB - (et > B ? et : B);
        line = 0;
        if (emit_line) {
            const u32 jS = (B == 0) ? 0u : (bcut ? bj : bj + 1u);
            const bool cutS = B != 0 && bcut;
            const u32 jE = ej;
            u32 mS = jS;   // verbatim middle tokens: [mS, jE)
            if (jS < jE) {
                if (cutS) { L.lenS = gm->pEnd[jS] - B; L.codeS = rt[gm->opos[minus ? no - 1 - jS : jS]]; mS = jS + 1; }
                if (mS < jE) {
                    const u32 o1 = minus ? no - jE : mS, o2 = minus ? no - 1 - mS : jE - 1;   // original index range [o1, o2]
                    L.mid_a = o1 ? gm->opos[o1 - 1] + 1u : ca;
                    L.mid_b = gm->opos[o2] + 1u;
                }
            }
            L.codeE = rt[gm->opos[minus ? no - 1 - jE : jE]];
            line = line_const_len(R, p10) + line_step_len(L, p10);
        }
        loff = g.excl_scan(line, size);

    } while (0);

    // ---------------- results: sizes, status, descriptors (record r owns kSMaxLines slots)
    const bool fast = !deleg && size != 0;
    const u32 lmask = g.ballot(fast && emit_line);
    if (fast && emit_line)
        store_line_desc(a.sdesc + (size_t)r * kSMaxLines + (u32)__popc(lmask & ((1u << g.gl) - 1u)), r, loff, line, L);
    if (g.gl == 0) {
        if (deleg) {
            a.status[r] = ST_OK;   // overwritten by k_long / the general kernel
            a.out_off[r] = 0;
            a.line_off[r] = 0;
            a.deleg_list[atomicAdd(a.n_deleg, 1u)] = r;
        } else {
            a.status[r] = status | (fast ? (u32)ST_F_DESC : 0u);
            a.out_off[r] = size;
            a.line_off[r] = (u32)__popc(lmask);
            if (fast) store_rec_desc(a.rdesc + r, R);
        }
    }
}

// One PAF line per thread from its descriptor.  Line slots are dense and in output order (k_short's
// records through the line map, k_long's batches as 32-slot blocks), so the lines of a warp are
// contiguous in the output unless a record converted by another kernel lies between them.  Lines are formatted into a per-warp
// staging buffer and flushed with 128-bit stores.
// ---- TMA 1-D bulk copies (cp.async.bulk, SASS UBLKCP): shared <-> global without passing through
// registers, completion through an mbarrier (loads) or a bulk async-group (stores).  The emulator
// build (G2P_HOSTSIM) takes the plain load/store loops instead.
#if !defined(G2P_HOSTSIM)
__device__ __forceinline__ u32 smem_u32(const void* p) { return (u32)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(u64* bar, u32 count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(u64* bar, u32 bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, u32 bytes, u64* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)), "l"(src),
                 "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(u64* bar, u32 parity) {
    u32 ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void bulk_s2g(void* dst, const void* src, u32 bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(smem_u32(src)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
#endif

constexpr int kEThreads = 256;
#ifndef G2P_EMIT_TEXT_CAP
#define G2P_EMIT_TEXT_CAP 4096
#endif
// Staging buffers per warp: PAF bytes (out) and GAF bytes (text: the records its 32 lines come from; 0: read the
// text from global).  Dense runs (k_par / k_long lines of long records) take 5 kB + 4 kB, 3 CTAs per SM.  The
// line-map instantiation only stages one warp's run of k_rec lines -- 32 lines of ~130 bytes from ~14 records of
// at most kSLimit bytes: ~4.3 kB of PAF from ~2 kB of GAF in short-read input -- and takes direct stores or global
// reads for a run that does not fit, so its buffers are sized for 4 CTAs of 256 threads per SM (32 warps).
template <bool DENSE> struct EmitCap {
    static constexpr u32 out = DENSE ? 5120u : 4608u;
    static constexpr u32 text = DENSE || G2P_EMIT_TEXT_CAP == 0 ? (u32)G2P_EMIT_TEXT_CAP : 2496u;
    static constexpr size_t smem = (size_t)(kEThreads / 32) * (out + 16 + text + 32);
};
constexpr size_t kEmitSmem = EmitCap<true>::smem;        // dense runs (also enough for the line-map instantiation)
constexpr size_t kEmitSmemMap = EmitCap<false>::smem;
static_assert(4 * (kEmitSmemMap + 64 + 1024) <= 228 * 1024, "4 CTAs of the line-map instantiation per SM");

// What k_emit_lines needs to start all its loads at once for a line of a k_short record.
struct __align__(16) LineMapEnt {
    u32 desc_idx;     // r * kSMaxLines + j
    u32 rec_start;    // text offset of the record
    u64 out_off;      // output offset of the record
};

struct EmitArgs {
    const u8* gaf;
    u64 n;
    const u32* rec_start;
    const u64* out_off;
    const LineDesc* desc;
    const LineMapEnt* map;   // line slot -> descriptor + record offsets (k_short's records), or null: slot == descriptor index
    const RecDesc* rdesc;
    const u32* status;       // dense mode: a line is emitted only if its record kept ST_F_DESC (k_long may describe the first
                             // batches of a record and delegate it later)
    u32 n_slots;
    u8* out;
};

// DENSE = false: the lines of k_rec / k_short records through the line map (a.map, written by k_scan_apply2);
// DENSE = true: the dense descriptor array of k_par's runs and k_long's blocks (a.map == null).
template <bool DENSE>
__global__ void __launch_bounds__(kEThreads, DENSE ? 3 : 4) k_emit_lines(const EmitArgs a) {
    G2P_DYN_SMEM(smem);
    constexpr u32 kEOutCap = EmitCap<DENSE>::out, kETextCap = EmitCap<DENSE>::text;
    const u32 FULL = 0xffffffffu;
    const u32 lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    u8* sm = smem + (size_t)warp * (kEOutCap + 16 + kETextCap + 32);
    u8* sm_text = sm + kEOutCap + 16;
#if !defined(G2P_HOSTSIM)
    __shared__ __align__(8) u64 s_bar[kEThreads / 32];   // one mbarrier per warp (used once: parity 0)
    if (lane == 0) { mbar_init(&s_bar[warp], 1); fence_mbar_init(); }
    __syncwarp();
#endif
    const u32 slot = blockIdx.x * kEThreads + threadIdx.x;
    const bool in_range = slot < a.n_slots;
    uint4 v0 = make_uint4(kDescInvalid, 0u, 0u, 0u), v1 = make_uint4(0u, 0u, 0u, 0u), v2 = v1, v3 = v1;
    u32 rs = 0, re = 0;   // text span of this lane's record
    u64 obase = 0;
    const LineDesc* dp = a.desc + slot;
    if (!DENSE && in_range) {   // k_rec's / k_short's lines: one 16-byte entry tells where everything is
        const uint4 m = __ldg(reinterpret_cast<const uint4*>(a.map + slot));
        dp = a.desc + m.x;
        rs = m.y;
        re = rs + kSLimit + 1;   // upper bound of the record's end (its length is not needed exactly)
        obase = (u64)m.z | ((u64)m.w << 32);
    }
    if (in_range) {
        const uint4* src = reinterpret_cast<const uint4*>(dp);
        v0 = __ldg(src); v1 = __ldg(src + 1); v2 = __ldg(src + 2); v3 = __ldg(src + 3);
    }
    struct { u32 rec, loff, len; } d;
    LineRec R;
    LineStep L;
    unpack_line_desc(v0, v1, v2, v3, d.rec, d.loff, d.len, L);
    if (!in_range) d.len = 0;
    const bool valid = !DENSE ? in_range : (d.rec != kDescInvalid && (__ldg(a.status + d.rec) & ST_F_DESC) != 0);
    const u32 vmask = __ballot_sync(FULL, valid);
    if (vmask == 0) return;
    const int first = __ffs((int)vmask) - 1, last = 31 - __clz((int)vmask);
    u64 o = 0;
    // The text of the warp's records (one short span: ~14 short records, or the one or two few-kB
    // records a dense block comes from) is staged in shared memory with one TMA bulk copy.  With the
    // line map it starts before the descriptors arrive; dense blocks know their record only from them.
    bool text_staged = false, text_tma = false;
    u32 A = 0;
    auto stage_text = [&](u32 t0, u32 t1) {
        if ((u64)t1 > a.n) t1 = (u32)a.n;
        A = t0 & ~15u;
        text_staged = t1 > t0 && t1 - A <= kETextCap;
        if (text_staged) {
            const u32 nvec = (t1 - A + 15u) >> 4;
#if !defined(G2P_HOSTSIM)
            if ((u64)A + 16ull * nvec <= a.n) {   // whole vectors inside the buffer: one TMA bulk copy
                if (lane == 0) { mbar_expect_tx(&s_bar[warp], nvec * 16u); bulk_g2s(sm_text, a.gaf + A, nvec * 16u, &s_bar[warp]); }
                text_tma = true;
            } else
#endif
            {
                for (u32 v = lane; v < nvec; v += 32) reinterpret_cast<uint4*>(sm_text)[v] = ldg_vec_guarded(a.gaf, (u64)A + 16u * v, a.n);
            }
        }
    };
    if (!DENSE) stage_text(__shfl_sync(FULL, rs, first), __shfl_sync(FULL, re, last));
    if (valid) {
        const uint4* src = reinterpret_cast<const uint4*>(a.rdesc + d.rec);
        const uint4 r0 = __ldg(src), r1 = __ldg(src + 1), r2 = __ldg(src + 2);
        if (DENSE) { rs = a.rec_start[d.rec]; re = a.rec_start[d.rec + 1]; obase = a.out_off[d.rec]; }
        o = obase + d.loff;
        unpack_rec_desc(r0, r1, r2, R);
    }
    if (DENSE) {   // the warp's slots may belong to several records in any order (small batches): stage the span that covers them all
        u32 t0 = valid ? rs : 0xffffffffu, t1 = valid ? re : 0u;
        for (int o2 = 16; o2 > 0; o2 >>= 1) {
            const u32 x0 = __shfl_xor_sync(FULL, t0, o2), x1 = __shfl_xor_sync(FULL, t1, o2);
            t0 = x0 < t0 ? x0 : t0;
            t1 = x1 > t1 ? x1 : t1;
        }
        stage_text(t0, t1);
    }
    // A record too long to be staged whole (a warp of a k_par run: 32 consecutive path steps of ONE record): stage the
    // pieces its lines are made of -- query name, tp / rc values (the same for all lanes), the span of the lanes' node
    // names in the path column and the span of their verbatim CIGAR pieces in the cg tag.
    bool parts = false;
    LineSrc PS;
    PS.qname = PS.name = PS.tp = PS.rc = PS.mid = nullptr;
    if (DENSE && !text_staged && kETextCap != 0) {
        const u32 rec0 = __shfl_sync(FULL, d.rec, first);
        if (__all_sync(FULL, !valid || d.rec == rec0)) {
            const u32 rs0 = __shfl_sync(FULL, rs, first);
            const u32 qn = __shfl_sync(FULL, R.qn_b, first);
            const u32 tpa = __shfl_sync(FULL, R.tp_a, first), tpb = __shfl_sync(FULL, R.tp_b, first);
            const u32 rca = __shfl_sync(FULL, R.rc_a, first), rcb = __shfl_sync(FULL, R.rc_b, first);
            u32 n0 = valid ? L.name_a : 0xffffffffu, n1 = valid ? L.name_a + L.nl : 0u;
            const bool has_mid = valid && L.mid_b > L.mid_a;
            u32 m0 = has_mid ? L.mid_a : 0xffffffffu, m1 = has_mid ? L.mid_b : 0u;
            for (int o2 = 16; o2 > 0; o2 >>= 1) {
                const u32 x0 = __shfl_xor_sync(FULL, n0, o2), x1 = __shfl_xor_sync(FULL, n1, o2);
                const u32 y0 = __shfl_xor_sync(FULL, m0, o2), y1 = __shfl_xor_sync(FULL, m1, o2);
                n0 = x0 < n0 ? x0 : n0; n1 = x1 > n1 ? x1 : n1;
                m0 = y0 < m0 ? y0 : m0; m1 = y1 > m1 ? y1 : m1;
            }
            // regions (record-relative [from, to)): query name, tp, rc, names, CIGAR pieces
            const u32 from[5] = {0u, tpa, rca, n0, m0};
            const u32 to[5] = {qn, tpb, rcb, n1, m1};
            u32 base[5], al[5], off = 0;
#pragma unroll
            for (int r = 0; r < 5; ++r) {
                base[r] = off;
                al[r] = (rs0 + from[r]) & ~15u;   // absolute, 16-byte aligned start of the copy
                if (to[r] > from[r]) off += ((rs0 + to[r] - al[r]) + 15u) & ~15u;
            }
            if (off <= kETextCap) {
#pragma unroll
                for (int r = 0; r < 5; ++r) {
                    if (to[r] > from[r]) {
                        const u32 nvec = ((rs0 + to[r] - al[r]) + 15u) >> 4;
                        for (u32 v = lane; v < nvec; v += 32) reinterpret_cast<uint4*>(sm_text + base[r])[v] = ldg_vec_guarded(a.gaf, (u64)al[r] + 16u * v, a.n);
                    }
                }
                __syncwarp();
                parts = true;
                PS.qname = sm_text + base[0] + (rs0 - al[0]);
                PS.tp = sm_text + base[1] + (rs0 + tpa - al[1]);
                PS.rc = sm_text + base[2] + (rs0 + rca - al[2]);
                PS.name = sm_text + base[3] + (rs0 + L.name_a - al[3]);
                PS.mid = sm_text + base[4] + (rs0 + L.mid_a - al[4]);
            }
        }
    }
    if (text_staged) {
#if !defined(G2P_HOSTSIM)
        if (text_tma) {
            u32 spins = 0;
            while (!mbar_try_wait(&s_bar[warp], 0)) { if (++spins > (1u << 24)) __trap(); }
        } else
#endif
            __syncwarp();
    }
    (void)text_tma;
    const u8* rt = text_staged ? sm_text + (rs - A) : a.gaf + rs;
    // contiguity of the warp's lines in the output
    const u64 end = o + d.len;
    const u64 onext = __shfl_down_sync(FULL, o, 1);
    const bool vnext = __shfl_down_sync(FULL, (u32)valid, 1) != 0 && lane < 31;
    const bool gap = valid && vnext && onext != end;
    const bool holes = (vmask >> first) != (0xffffffffu >> (31 - (last - first)));
    const u64 o1 = __shfl_sync(FULL, end, last);
    // short records: one run that fits the buffer (32 lines of ~130 bytes); anything else goes straight to global
    if (__any_sync(FULL, gap) || holes || (!DENSE && (o1 - __shfl_sync(FULL, o, first)) + 15u > kEOutCap)) {
        if (valid) write_line<!DENSE>(a.out + o + d.len, parts ? PS : line_src(rt, R, L), R, L);
        return;
    }
    // The warp's lines are one contiguous run of the output.  It goes through the staging buffer in
    // sub-runs of at most kEOutCap bytes (one for short reads; the 31 lines of a full batch of a
    // 2 kB assembly record need two), each formatted in shared memory and flushed with one bulk store.
    u32 todo = vmask;
    do {   // (a single pass, known at compile time, for the short records' variant)
        const int f = DENSE ? __ffs((int)todo) - 1 : first;
        const u64 ob = __shfl_sync(FULL, o, f);
        const u32 pad = (u32)(ob & 15u);
        const bool fits = DENSE ? ((todo >> lane) & 1u) != 0 && (end - ob) + pad <= kEOutCap : valid;
        const u32 in = DENSE ? __ballot_sync(FULL, fits) : vmask;   // a prefix of `todo`: the lines are in output order
        if (DENSE && in == 0) {   // one line longer than the buffer
            if ((int)lane == f) write_line<!DENSE>(a.out + o + d.len, parts ? PS : line_src(rt, R, L), R, L);
            todo &= todo - 1u;
            continue;
        }
        const u64 oe = DENSE ? __shfl_sync(FULL, end, 31 - __clz((int)in)) : o1;
        if (fits) {
            // two instantiations so that the common one (staged lines, staged text) works on pointers the
            // compiler can prove to be shared memory: LDS / STS instead of generic 64-bit LD / ST
            if (text_staged) write_line<!DENSE>(sm + pad + (u32)(o - ob) + d.len, line_src(sm_text + (rs - A), R, L), R, L);
            else if (DENSE && parts) write_line<!DENSE>(sm + pad + (u32)(o - ob) + d.len, PS, R, L);
            else write_line<!DENSE>(sm + pad + (u32)(o - ob) + d.len, line_src(a.gaf + rs, R, L), R, L);   // long records: text from global
        }
        const u32 total = pad + (u32)(oe - ob);
        u8* gb = a.out + (ob - pad);
        const u32 full_b = total >> 4;
#if !defined(G2P_HOSTSIM)
        // the 16-byte aligned middle of the run leaves as one TMA bulk store
        fence_async_smem();
        __syncwarp();
        const u32 first_b = pad ? 1u : 0u;
        if (lane == 0 && full_b > first_b) { bulk_s2g(gb + 16u * first_b, sm + 16u * first_b, 16u * (full_b - first_b)); bulk_commit(); }
#else
        __syncwarp();
        for (u32 u = (pad ? 1u : 0u) + lane; u < full_b; u += 32) reinterpret_cast<uint4*>(gb)[u] = reinterpret_cast<const uint4*>(sm)[u];
#endif
        const u32 head_end = pad ? (total < 16u ? total : 16u) : 0u;
        for (u32 b = pad + lane; b < head_end; b += 32) gb[b] = sm[b];
        const u32 tail_a = full_b * 16u > head_end ? full_b * 16u : head_end;
        for (u32 b = tail_a + lane; b < total; b += 32) gb[b] = sm[b];
#if !defined(G2P_HOSTSIM)
        if (lane == 0) bulk_wait_read0();   // the staging buffer must outlive the copy's reads
#endif
        __syncwarp();
        todo &= ~in;
    } while (DENSE && todo);
}

}  // namespace g2p
