// g2p_filter.cuh — gaffilter on the device (SURVEY.md §8f N1; reference gaffilter_main.cpp:31-70, 205-343).
//
// The reference loads every GAF (or, with -p, PAF) record, builds one interval tree per query sequence over the
// closed query intervals [query_start, query_end - 1], and prints a record iff it "dominates" every qualifying
// record whose interval overlaps its own (primary over secondary, then MAPQ ratio, then block-length ratio; and / or
// mzgaf2paf's length rule).  The decision does not depend on the order in which overlaps are visited (the loop ANDs
// them), so the tree is replaced by a sort:
//
//   k_filter_parse      one thread per line: the columns and tags the filter reads (parse_gaf_record,
//                       gafkluge.hpp:84-204, or parse_paf_line, paf.hpp:48-80) -> one 80-byte row; 128-bit hash of the
//                       query name; sort key = hash32 << 32 | query_start
//   k_rs_hist / scatter LSD radix sort of (key, record) pairs, 4 bits per pass, stable
//   k_filter_ends, k_segmax<>, k_segmax_tiles
//                       per run of equal hash32: running maximum of the interval ends (segmented max-scan; bounds the
//                       backward scan)
//   k_filter_sweep      one thread per record: forwards while start_j <= stop_i, backwards while the running maximum
//                       of the ends reaches start_i; same qualifiers and the same double arithmetic as dominates()
//   k_filter_emit       size pass / scan / write pass of the kept records, re-serialised like the reference prints
//                       them (operator<<(GafRecord), gafkluge.hpp:288-323: tags in name order; operator<<(PafLine),
//                       paf.hpp:83-95, where cg is an ordinary tag because of the compare(0, 3, "cg:Z:") quirk)
//
// Records are kept in input order.  Anything the reference would die on (assert / uncaught exception) is reported as
// an abort status with the index of the first such line; nothing is printed then (the reference loads all records
// before it prints any).
//
// Inputs of any size and several GPUs go through the job (g2p_filter_job_*, see the bucket partition below and
// g2p_filter_job.hpp): the same kernels over newline-aligned chunks, the rows partitioned by query name.
#pragma once
#include "g2u_core.cuh"

namespace g2p {

struct FilterParams {
    double ratio, min_overlap_pct, min_identity;
    i64 min_overlap_len, min_block_len, min_mapq;
    u32 is_paf;
};

struct __attribute__((aligned(16))) FRow {
    u64 h0, h1;          // 128-bit key of the query name (exact bytes for names of <= 16 bytes)
    i64 qs, qe, qlen, block_length, matches;
    u64 rc;              // key of the rc value (0: no rc tag)
    i64 paf_bases;       // PAF mode: column 11 (num_bases), what "total block lengths filtered" adds up
    i32 mapq;
    u32 flags;           // kFRowPrimary, kFRowSkip, kFRowHasGi
    float gi;            // GAF mode: stof(gi) when present
    u32 name_len;
    u64 grec;            // record number: chunk << 32 | line of the chunk (the single call: the line)
};
static_assert(sizeof(FRow) == 96, "FRow is the 96-byte row the filter job keeps in host memory");
enum : u32 { kFRowPrimary = 1u, kFRowSkip = 2u, kFRowHasGi = 4u };

struct FilterMeta {
    u32 first_err;       // smallest failing line (0xFFFFFFFF: none)
    u32 err_status;
    u32 n_loaded;        // records loaded ('*' lines are not)
    u32 n_filtered;
    u64 filtered_len;    // "total block lengths filtered"
    u64 out_total;
    u32 unsupported;     // a query_start >= 2^32: not sortable here
    u32 assert_rec;      // smallest row on which an assertion of the reference's filter loop fires (0xFFFFFFFF: none)
    u64 assert_grec;     // ... its grec, input order across the chunks and partitions of the job (~0: none); the
                         // single call's rows are its lines, so there both are the line
};

// ---- stof of a tag value (gi:f:0.978): decimal digits, optional fraction and exponent; anything else -> false -----
// Correctly rounded (to nearest, ties to even) like std::stof, and false where stof throws std::out_of_range: a value that
// rounds (24 bits, unbounded exponent) to 2^128 or more, or to less than FLT_MIN.  Method: at most 19 significant digits
// go into an integer M (a non-zero digit beyond them sets `sticky`), value = M * 10^E.  A double estimate gives a 24-bit
// candidate m * 2^e within one unit of the result; exact comparisons of M * 10^E with the midpoints next to the candidate
// (288-bit integers) correct it.  When digits were dropped and a midpoint lies between M * 10^E and (M + 1) * 10^E the
// rounding is not decided by the digits kept: false (more than 19 significant digits within 10^-18 of a midpoint).
struct FBig { u32 w[9]; };   // 288 bits: M * 10^56 * 2^26 and M * 2^153 fit
G2P_HD void fbig_set(FBig& a, u64 v) {
    a.w[0] = (u32)v; a.w[1] = (u32)(v >> 32);
    for (int i = 2; i < 9; ++i) a.w[i] = 0;
}
G2P_HD void fbig_mul(FBig& a, u32 f) {
    u64 c = 0;
    for (int i = 0; i < 9; ++i) { const u64 t = (u64)a.w[i] * f + c; a.w[i] = (u32)t; c = t >> 32; }
}
G2P_HD void fbig_mul_pow10(FBig& a, u32 k) {
    for (; k >= 9; k -= 9) fbig_mul(a, 1000000000u);
    u32 p = 1;
    while (k--) p *= 10;
    fbig_mul(a, p);
}
G2P_HD void fbig_shl(FBig& a, u32 s) {
    const u32 ws = s >> 5, bs = s & 31u;
    for (int i = 8; i >= 0; --i) {
        const int j = i - (int)ws;
        const u32 hi = j >= 0 ? a.w[j] : 0u, lo = j >= 1 ? a.w[j - 1] : 0u;
        a.w[i] = bs ? (hi << bs) | (lo >> (32 - bs)) : hi;
    }
}
// sign of M * 10^E - n * 2^b
G2P_HD int fdec_cmp(u64 M, i32 E, u64 n, i32 b) {
    FBig x, y;
    fbig_set(x, M); fbig_set(y, n);
    if (E >= 0) fbig_mul_pow10(x, (u32)E); else fbig_mul_pow10(y, (u32)-E);
    if (b >= 0) fbig_shl(y, (u32)b); else fbig_shl(x, (u32)-b);
    for (int i = 8; i >= 0; --i) if (x.w[i] != y.w[i]) return x.w[i] < y.w[i] ? -1 : 1;
    return 0;
}
// sign of value - n * 2^b for a value in [M, M + 1) * 10^E (sticky: strictly inside); 2 = not decided
G2P_HD int fdec_cmp_value(u64 M, bool sticky, i32 E, u64 n, i32 b) {
    const int c = fdec_cmp(M, E, n, b);
    if (!sticky || c > 0) return c;
    if (c == 0) return 1;
    return fdec_cmp(M + 1, E, n, b) > 0 ? 2 : -1;
}
G2P_HD bool parse_float_text(const u8* s, u32 n, float& out) {
    u32 i = 0;
    bool neg = false;
    if (i < n && (s[i] == '+' || s[i] == '-')) { neg = s[i] == '-'; ++i; }
    u64 M = 0;
    u32 nd = 0, sig = 0;
    i32 E = 0;
    bool sticky = false;
    for (; i < n && s[i] >= '0' && s[i] <= '9'; ++i, ++nd) {
        const u32 d = s[i] - '0';
        if (sig < 19) { M = M * 10 + d; sig += M != 0; }
        else { ++E; sticky |= d != 0; }
    }
    if (i < n && s[i] == '.') {
        for (++i; i < n && s[i] >= '0' && s[i] <= '9'; ++i, ++nd) {
            const u32 d = s[i] - '0';
            if (sig < 19) { M = M * 10 + d; sig += M != 0; --E; }
            else sticky |= d != 0;
        }
    }
    if (nd == 0) return false;
    if (i < n && (s[i] == 'e' || s[i] == 'E')) {
        ++i;
        bool eneg = false;
        if (i < n && (s[i] == '+' || s[i] == '-')) { eneg = s[i] == '-'; ++i; }
        i32 x = 0;
        u32 ne = 0;
        for (; i < n && s[i] >= '0' && s[i] <= '9'; ++i, ++ne) if (x < 100000) x = x * 10 + (s[i] - '0');
        if (ne == 0) return false;
        E += eneg ? -x : x;
    }
    if (i != n) return false;   // (stof ignores trailing text; such values are not produced by gaf2paf: unsupported)
    if (M == 0) { out = neg ? -0.f : 0.f; return true; }
    if ((i32)sig - 1 + E >= 39) return false;   // >= 10^39: overflow
    if ((i32)sig + E <= -38) return false;      // < 10^-38: below FLT_MIN
    // estimate: |E| <= 56 roundings of a double, far below half a unit of the float
    double v = (double)M;
    for (i32 k = 0; k < E; ++k) v *= 10.0;
    for (i32 k = 0; k < -E; ++k) v /= 10.0;
    union { double d; u64 u; } db;
    db.d = v;
    const u64 mant = (db.u & ((1ULL << 52) - 1)) | (1ULL << 52);   // v = mant * 2^(exp - 1075), a normal double
    u64 m = (mant + (1ULL << 28)) >> 29;
    i32 e = (i32)((db.u >> 52) & 0x7ff) - 1075 + 29;
    if (m == (1ULL << 24)) { m >>= 1; ++e; }
    for (int it = 0; it < 3; ++it) {
        const int up = fdec_cmp_value(M, sticky, E, 2 * m + 1, e - 1);
        if (up == 2) return false;
        if (up > 0 || (up == 0 && (m & 1))) {
            if (++m == (1ULL << 24)) { m >>= 1; ++e; }
            continue;
        }
        const bool low = m == (1ULL << 23);   // the next float down is half a unit away
        const int dn = low ? fdec_cmp_value(M, sticky, E, 4 * m - 1, e - 2) : fdec_cmp_value(M, sticky, E, 2 * m - 1, e - 1);
        if (dn == 2) return false;
        if (dn < 0 || (dn == 0 && (m & 1))) {
            if (low) { m = (1ULL << 24) - 1; --e; } else --m;
            continue;
        }
        break;
    }
    if (e >= 105 || e < -149) return false;   // >= 2^128, < 2^-126 (stof: std::out_of_range)
    union { float f; u32 u; } fb;
    fb.u = (neg ? 0x80000000u : 0u) | ((u32)(e + 150) << 23) | ((u32)m & 0x7FFFFFu);
    out = fb.f;
    return true;
}

G2P_HD void filter_name_key(const u8* s, u32 n, u64& k0, u64& k1) {
    name_key(s, n, k0, k1);
    if (n > 16) k1 ^= (u64)n * 0x9E3779B97F4A7C15ULL;
}
G2P_HD u64 filter_value_key(const u8* s, u32 n) {
    u64 a, b;
    name_key(s, n, a, b);
    u64 h = mix64(a ^ mix64(b + n));
    return h ? h : 1;
}

// GAF mode: parse_gaf_record + the tags the filter reads.  Returns a status (ST_OK / ST_SKIP / abort codes).
G2P_HD u32 filter_parse_gaf(const u8* r, u32 len, FRow& row) {
    URecHdr h;
    const u32 st = u_parse_header(r, len, h);
    if (st != ST_OK) return st;
    filter_name_key(r, h.qn_b, row.h0, row.h1);
    row.name_len = h.qn_b;
    row.qs = h.qs; row.qe = h.qe; row.qlen = h.qlen;
    // an empty path leaves the six path columns unparsed in the reference (-1); u_parse_header reports them the same way
    row.block_length = h.b; row.matches = h.m;
    row.mapq = h.mapq;
    row.paf_bases = 0;
    row.flags = kFRowPrimary;
    row.rc = 0;
    row.gi = 0.f;
    u32 p = h.tags_from;
    while (p < len) {
        u32 e = p;
        while (e < len && r[e] != '\t') ++e;
        if (e - p >= 5 && r[p + 2] == ':') {
            // value = everything after the second colon (gafkluge.hpp:185-202 splits at the first two colons)
            u32 c2 = p + 3;
            while (c2 < e && r[c2] != ':') ++c2;
            const u32 va = c2 + 1 <= e ? c2 + 1 : e;
            if (r[p] == 't' && r[p + 1] == 'p') { if (!(e - va == 1 && r[va] == 'P')) row.flags &= ~kFRowPrimary; }
            else if (r[p] == 'r' && r[p + 1] == 'c') row.rc = e > va ? filter_value_key(r + va, e - va) : 0;
            else if (r[p] == 'g' && r[p + 1] == 'i') {
                float g;
                if (!parse_float_text(r + va, e - va, g)) return ST_ABORT_STOL;
                row.gi = g; row.flags |= kFRowHasGi;
            }
        }
        p = e + 1;
    }
    return ST_OK;
}

// PAF mode: parse_paf_line (paf.hpp:48-80).  Tokens are split at tabs, EMPTY TOKENS ARE DROPPED (split_delims), more
// than 12 are required, the numeric columns go through std::stol, every further token must split at ':' into exactly
// three non-empty parts.
G2P_HD u32 filter_parse_paf(const u8* r, u32 len, FRow& row) {
    if (len > 0 && r[0] == '*') return ST_SKIP;
    u32 p = 0, k = 0;
    i64 cols[12];
    u32 qn_a = 0, qn_b = 0;
    row.flags = kFRowPrimary;
    row.rc = 0; row.gi = 0.f;
    bool have_gl = false, have_gm = false;
    i64 gl = 0, gm = 0;
    while (p <= len) {
        u32 e = p;
        while (e < len && r[e] != '\t') ++e;
        if (e > p) {
            if (k == 0) { qn_a = p; qn_b = e; }
            else if (k == 4) { if (e - p != 1 || (r[p] != '+' && r[p] != '-')) return ST_ABORT_ASSERT; }
            else if (k == 5) { /* target name */ }
            else if (k < 12) {
                const u32 st = stol_span(r, p, e, cols[k]);
                if (st) return st;
            } else {
                // tag: exactly three non-empty ':'-separated parts
                u32 parts = 0, a = p, pa[3] = {0, 0, 0}, pb[3] = {0, 0, 0};
                while (a <= e) {
                    u32 b = a;
                    while (b < e && r[b] != ':') ++b;
                    if (b > a) { if (parts < 3) { pa[parts] = a; pb[parts] = b; } ++parts; }
                    a = b + 1;
                }
                if (parts != 3) return ST_ABORT_ASSERT;
                const u32 kn = pb[0] - pa[0];
                if (kn == 2) {
                    const u8 c0 = r[pa[0]], c1 = r[pa[0] + 1];
                    if (c0 == 't' && c1 == 'p') { if (!(pb[2] - pa[2] == 1 && r[pa[2]] == 'P')) row.flags &= ~kFRowPrimary; else row.flags |= kFRowPrimary; }
                    else if (c0 == 'r' && c1 == 'c') row.rc = filter_value_key(r + pa[2], pb[2] - pa[2]);
                    else if (c0 == 'g' && c1 == 'l') { const u32 st = stol_span(r, pa[2], pb[2], gl); if (st) return st; have_gl = true; }
                    else if (c0 == 'g' && c1 == 'm') { const u32 st = stol_span(r, pa[2], pb[2], gm); if (st) return st; have_gm = true; }
                }
            }
            ++k;
        }
        p = e + 1;
    }
    if (k <= 12) return ST_ABORT_ASSERT;   // assert(toks.size() > 12)
    filter_name_key(r + qn_a, qn_b - qn_a, row.h0, row.h1);
    row.name_len = qn_b - qn_a;
    row.qlen = cols[1]; row.qs = cols[2]; row.qe = cols[3];
    row.matches = have_gm ? gm : cols[9];
    row.block_length = have_gl ? gl : cols[10];
    row.paf_bases = cols[10];
    row.mapq = (i32)cols[11];   // (int64 stored into GafRecord's int32 mapq, no 255 rule in this mode)
    return ST_OK;
}

struct FilterArgs {
    const u8* text;
    const u32* rec_start;
    u32 nrec;
    FilterParams P;
    FRow* rows;
    u64* keys;      // [nrec]  hash32 << 32 | query_start   (skipped lines: all ones -> sorted to the end)
    u32* vals;      // [nrec]  record index
    FilterMeta* meta;
    u64 grec_base;  // chunk << 32 (0 for the single call)
};

// sort key of a loaded row: hash32 << 32 | query_start
G2P_HD u64 filter_sort_key(const FRow& row) {
    const u32 h32 = (u32)(row.h0 ^ (row.h0 >> 32) ^ row.h1 ^ (row.h1 >> 32));
    // (negative starts -- no real aligner writes them, std::stol reads them -- sort together with start 0: the
    // forward scan of k_filter_sweep never stops on a start <= 0)
    return ((u64)(h32 == 0xffffffffu ? 0xfffffffeu : h32) << 32) | (u64)(row.qs < 0 ? 0u : (u32)row.qs);
}

__global__ void __launch_bounds__(128) k_filter_parse(const FilterArgs a) {
    for (u32 r = blockIdx.x * blockDim.x + threadIdx.x; r < a.nrec; r += gridDim.x * blockDim.x) {
        const u32 s = a.rec_start[r], len = a.rec_start[r + 1] - s - 1;
        FRow row;
        row.h0 = row.h1 = 0; row.qs = row.qe = row.qlen = row.block_length = row.matches = 0; row.rc = 0; row.paf_bases = 0;
        row.mapq = 0; row.flags = 0; row.gi = 0.f; row.name_len = 0; row.grec = a.grec_base | r;
        u32 st = a.P.is_paf ? filter_parse_paf(a.text + s, len, row) : filter_parse_gaf(a.text + s, len, row);
        u64 key = ~0ULL;
        if ((st & 0xff) == ST_SKIP) row.flags |= kFRowSkip;
        else if (st != ST_OK) { row.flags |= kFRowSkip; atomicMin(&a.meta->first_err, r); }
        else {
            atomicAdd(&a.meta->n_loaded, 1u);
            if (row.qs > 0xFFFFFFF0LL) atomicExch(&a.meta->unsupported, 1u);
            key = filter_sort_key(row);
        }
        a.rows[r] = row;
        a.keys[r] = key;
        a.vals[r] = r;
    }
}
// status of one line, recomputed for the report (runs only on error)
__global__ void k_filter_diagnose(const FilterArgs a) {
    const u32 r = a.meta->first_err;
    if (r == 0xFFFFFFFFu) return;
    const u32 s = a.rec_start[r], len = a.rec_start[r + 1] - s - 1;
    FRow row;
    a.meta->err_status = a.P.is_paf ? filter_parse_paf(a.text + s, len, row) : filter_parse_gaf(a.text + s, len, row);
}

// ---- LSD radix sort, 4 bits per pass ---------------------------------------------------------------
constexpr u32 kRsThreads = 256, kRsItems = 8, kRsTile = kRsThreads * kRsItems;
__global__ void __launch_bounds__(kRsThreads) k_rs_hist(const u64* __restrict__ keys, u32 n, u32 shift, u64* __restrict__ hist, u32 nblk) {
    __shared__ u32 h[16];
    if (threadIdx.x < 16) h[threadIdx.x] = 0;
    __syncthreads();
    const u32 base = blockIdx.x * kRsTile + threadIdx.x * kRsItems;
    for (u32 i = 0; i < kRsItems; ++i)
        if (base + i < n) atomicAdd(&h[(u32)(keys[base + i] >> shift) & 15u], 1u);
    __syncthreads();
    if (threadIdx.x < 16) hist[(size_t)threadIdx.x * nblk + blockIdx.x] = h[threadIdx.x];   // digit-major: one exclusive scan gives every (digit, block) its base
}
__global__ void __launch_bounds__(kRsThreads) k_rs_scatter(const u64* __restrict__ keys, const u32* __restrict__ vals, u64* __restrict__ keys_out,
                                                          u32* __restrict__ vals_out, u32 n, u32 shift, const u64* __restrict__ hist, u32 nblk) {
    __shared__ u32 cnt[16 * kRsThreads];   // [digit][thread]
    __shared__ u32 wsum[kRsThreads / 32];
    __shared__ u64 gbase[16];
    const u32 t = threadIdx.x;
    for (u32 d = 0; d < 16; ++d) cnt[d * kRsThreads + t] = 0;
    if (t < 16) gbase[t] = hist[(size_t)t * nblk + blockIdx.x];
    const u32 base = blockIdx.x * kRsTile + t * kRsItems;
    u64 k[kRsItems];
    u32 v[kRsItems];
    for (u32 i = 0; i < kRsItems; ++i) {
        if (base + i < n) {
            k[i] = keys[base + i]; v[i] = vals[base + i];
            cnt[((u32)(k[i] >> shift) & 15u) * kRsThreads + t] += 1u;   // (own column: no race)
        }
    }
    __syncthreads();
    // exclusive scan of the 16 x 256 counters in digit-major order: thread t owns entries [16 t, 16 t + 16)
    u32 own[16], sum = 0;
    for (u32 i = 0; i < 16; ++i) { own[i] = cnt[16 * t + i]; sum += own[i]; }
    u32 incl = sum;
    for (int o = 1; o < 32; o <<= 1) { const u32 up = __shfl_up_sync(0xffffffffu, incl, o); if ((t & 31u) >= (u32)o) incl += up; }
    if ((t & 31u) == 31u) wsum[t >> 5] = incl;
    __syncthreads();
    u32 wpre = 0;
    for (u32 i = 0; i < (t >> 5); ++i) wpre += wsum[i];
    u32 run = wpre + incl - sum;
    for (u32 i = 0; i < 16; ++i) { cnt[16 * t + i] = run; run += own[i]; }
    __syncthreads();
    // cnt[d][t] is now the number of elements of the block that sort before thread t's first element with digit d
    __shared__ u32 dfirst[16];   // ... and cnt[d][0] the number of elements of the block with a smaller digit
    if (t < 16) dfirst[t] = cnt[t * kRsThreads];
    __syncthreads();
    for (u32 i = 0; i < kRsItems; ++i) {
        if (base + i < n) {
            const u32 d = (u32)(k[i] >> shift) & 15u;
            const u32 pos = cnt[d * kRsThreads + t]++;   // (own column: no race; the thread's elements stay in order)
            const u64 o = gbase[d] + (pos - dfirst[d]);
            keys_out[o] = k[i];
            vals_out[o] = v[i];
        }
    }
}

// ---- after the sort: position p holds record vals[p]; runs of equal hash32 are contiguous and ordered by query_start ----
// Closed interval of a record as the reference stores it: Interval(query_start, query_end - 1) = [min, max].
G2P_HD void filter_interval(const FRow& r, i64& lo, i64& hi) {
    const i64 a = r.qs, b = r.qe - 1;
    lo = a < b ? a : b;
    hi = a < b ? b : a;
}

// Running maximum of the interval ends inside each run of equal hash32: a segmented inclusive max-scan over the sorted
// order (a run is one query sequence -- with assembly contigs as queries a single run holds 10^5 alignments, so nothing
// here may walk a run serially).  k_filter_ends writes every entry's end, k_segmax<false> reduces 2048-entry tiles to
// (does a run start inside the tile?, maximum after the last start), k_segmax_tiles turns those into the value carried
// into every tile, k_segmax<true> rescans the tiles with their carry.
constexpr int kSegThreads = 256, kSegItems = 8;
constexpr u32 kSegTile = kSegThreads * kSegItems;
__device__ __forceinline__ bool filter_run_head(const u64* __restrict__ keys, u32 p) {
    const u64 k = keys[p];
    return p == 0 || k == ~0ULL || (u32)(keys[p - 1] >> 32) != (u32)(k >> 32);   // ('*' and failed lines: each one alone)
}
__global__ void __launch_bounds__(256) k_filter_ends(const u64* __restrict__ keys, const u32* __restrict__ vals, const FRow* __restrict__ rows,
                                                     u32 n, i64* __restrict__ prefmax) {
    for (u32 p = blockIdx.x * blockDim.x + threadIdx.x; p < n; p += gridDim.x * blockDim.x) {
        i64 hi = 0;
        if (keys[p] != ~0ULL) { i64 lo; filter_interval(rows[vals[p]], lo, hi); }
        prefmax[p] = hi;
    }
}
// (flag, value) of a sequence followed by another: the value after the last run start
__device__ __forceinline__ void segmax_join(bool& f, i64& v, bool f2, i64 v2) {
    v = f2 ? v2 : (v > v2 ? v : v2);
    f = f || f2;
}
template <bool APPLY>
__global__ void __launch_bounds__(kSegThreads) k_segmax(const u64* __restrict__ keys, u32 n, i64* __restrict__ x, i64* __restrict__ tile_val, u32* __restrict__ tile_flag,
                                                        const i64* __restrict__ carry_val) {
    __shared__ i64 wv[kSegThreads / 32];
    __shared__ u32 wf[kSegThreads / 32];
    const u32 base = blockIdx.x * kSegTile + threadIdx.x * kSegItems;
    const u32 lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    // the thread's items
    bool f = false;
    i64 v = INT64_MIN;
    bool hf[kSegItems];
    i64 hv[kSegItems];
#pragma unroll
    for (int i = 0; i < kSegItems; ++i) {
        const u32 p = base + i;
        hf[i] = p < n && filter_run_head(keys, p);
        hv[i] = p < n ? x[p] : INT64_MIN;
        if (p < n) segmax_join(f, v, hf[i], hv[i]);
    }
    // inclusive scan over the threads of the warp, then over the warps
    bool sf = f;
    i64 sv = v;
    for (int d = 1; d < 32; d <<= 1) {
        const u32 pf = __shfl_up_sync(0xffffffffu, (u32)sf, d);
        const i64 pv = __shfl_up_sync(0xffffffffu, sv, d);
        if (lane >= (u32)d) { bool nf = pf != 0; i64 nv = pv; segmax_join(nf, nv, sf, sv); sf = nf; sv = nv; }
    }
    if (lane == 31) { wv[warp] = sv; wf[warp] = sf; }
    __syncthreads();
    // what arrives at this thread from the left: the tile's carry, the warps before, the lanes before
    bool cf = false;
    i64 cv = APPLY ? carry_val[blockIdx.x] : INT64_MIN;
    for (u32 w = 0; w < warp; ++w) segmax_join(cf, cv, wf[w] != 0, wv[w]);
    {
        const u32 pf = __shfl_up_sync(0xffffffffu, (u32)sf, 1);
        const i64 pv = __shfl_up_sync(0xffffffffu, sv, 1);
        if (lane > 0) segmax_join(cf, cv, pf != 0, pv);
    }
    if (APPLY) {
#pragma unroll
        for (int i = 0; i < kSegItems; ++i) {
            const u32 p = base + i;
            if (p < n) { segmax_join(cf, cv, hf[i], hv[i]); x[p] = cv; }
        }
    } else if (threadIdx.x == kSegThreads - 1) {
        segmax_join(cf, cv, f, v);
        tile_val[blockIdx.x] = cv;
        tile_flag[blockIdx.x] = cf;
    }
}
__global__ void k_segmax_tiles(const i64* __restrict__ tile_val, const u32* __restrict__ tile_flag, u32 ntiles, i64* __restrict__ carry_val) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    bool f = false;
    i64 v = INT64_MIN;
    for (u32 t = 0; t < ntiles; ++t) { carry_val[t] = v; segmax_join(f, v, tile_flag[t] != 0, tile_val[t]); }
}

// dominates() of the reference (gaffilter_main.cpp:31-60), same operations in the same order (no contraction: the
// divisions are __ddiv_rn, the additions __dadd_rn)
G2P_HD double f_div(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __ddiv_rn(a, b);
#else
    volatile double r = a / b;
    return r;
#endif
}
G2P_HD double f_add(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __dadd_rn(a, b);
#else
    volatile double r = a + b;
    return r;
#endif
}
G2P_HD bool filter_dominates(const FRow& g1, const FRow& g2, double ratio) {
    const bool p1 = (g1.flags & kFRowPrimary) != 0, p2 = (g2.flags & kFRowPrimary) != 0;
    if (g1.qs >= g1.qe) return false;
    if (g2.qs >= g2.qe) return true;
    if (p1 && !p2) return true;
    if (p2 && !p1) return false;
    if (f_div((double)g1.mapq, f_add((double)g2.mapq, 0.000001)) >= ratio) return true;
    if (f_div((double)g2.mapq, f_add((double)g1.mapq, 0.000001)) >= ratio) return false;
    if (f_div((double)g1.block_length, f_add((double)g2.block_length, 0.000001)) >= ratio) return true;
    return false;
}
G2P_HD bool filter_dominates_mz(const FRow& g1, const FRow& g2, i64 thr) {   // dominates_mzgaf2paf (:63-66)
    return (g1.block_length >= thr && g2.block_length < thr) || (g1.block_length < thr && g2.block_length < thr);
}
// assert(identity >= 0) of the visit lambda (gaffilter_main.cpp:289): evaluated for EVERY interval the tree reports,
// the record's own included
G2P_HD bool filter_identity_negative(const FRow& rj) {
    return rj.matches != 0 && f_div((double)rj.block_length, (double)rj.matches) < 0.0;
}
// one overlapping record j against record i: false = i is filtered out (gaffilter_main.cpp:263-312); `boom`: one of the
// reference's assertions fires on this pair (identity >= 0, :289; oend >= ostart in overlap_size, :68) -- it aborts
G2P_HD bool filter_pair_ok(const FRow& ri, const FRow& rj, const FilterParams& P, bool& boom) {
    if (rj.h0 != ri.h0 || rj.h1 != ri.h1 || rj.name_len != ri.name_len) return true;   // another query sequence (hash32 collision)
    double identity = rj.matches ? f_div((double)rj.block_length, (double)rj.matches) : 0.0;
    if (identity < 0.0) boom = true;
    if (rj.flags & kFRowHasGi) { const double g = (double)rj.gi; identity = g < identity ? g : identity; }
    if (!(rj.mapq >= P.min_mapq && (rj.qlen <= P.min_block_len || rj.block_length >= P.min_block_len) && identity >= P.min_identity)) return true;
    if (!(ri.rc == rj.rc || ri.rc == 0 || rj.rc == 0)) return true;   // they map to different reference contigs
    const i64 ostart = ri.qs > rj.qs ? ri.qs : rj.qs, oend = ri.qe < rj.qe ? ri.qe : rj.qe;
    const i64 overlap = oend - ostart;
    if (overlap < 0) boom = true;
    if (!(ri.block_length == 0 || f_div((double)overlap, (double)ri.block_length) >= P.min_overlap_pct)) return true;
    bool dom = true;
    if (P.ratio != 0.0) dom = filter_dominates(ri, rj, P.ratio);
    if (dom && P.min_overlap_len) dom = filter_dominates_mz(ri, rj, P.min_overlap_len);
    return dom;
}

__global__ void __launch_bounds__(128) k_filter_sweep(const u64* __restrict__ keys, const u32* __restrict__ vals, const FRow* __restrict__ rows,
                                                      const i64* __restrict__ prefmax, u32 n, FilterParams P, u8* __restrict__ keep, FilterMeta* meta) {
    for (u32 p = blockIdx.x * blockDim.x + threadIdx.x; p < n; p += gridDim.x * blockDim.x) {
        if (keys[p] == ~0ULL) continue;   // '*' lines and failed lines: never loaded
        const u32 i = vals[p];
        const FRow ri = rows[i];
        const u32 h = (u32)(keys[p] >> 32);
        // query of visit_overlapping(query_start, end_point): end_point = query_end - 1 if query_end > query_start else query_end
        const i64 qstart = ri.qs, qstop = ri.qe > ri.qs ? ri.qe - 1 : ri.qe;
        bool ok = true, boom = false;
        // (The reference collects ALL overlapping intervals -- its assertions run on every one of them, the record's own
        // included -- and only then looks for one that is not dominated: the scans do not stop at the first such one.)
        {
            i64 lo, hi;
            filter_interval(ri, lo, hi);
            if (hi >= qstart && lo <= qstop && filter_identity_negative(ri)) boom = true;
        }
        // forwards: starts are ascending (the stored interval's lower end can be query_end - 1 < query_start only for
        // empty / inverted records, whose lower end is within one of their start)
        for (u32 q = p + 1; q < n && (u32)(keys[q] >> 32) == h; ++q) {
            const FRow rj = rows[vals[q]];
            i64 lo, hi;
            filter_interval(rj, lo, hi);
            if (rj.qs > qstop + 1 && rj.qs > 0) break;
            if (hi >= qstart && lo <= qstop) { const bool d = filter_pair_ok(ri, rj, P, boom); ok = ok && d; }
        }
        for (u32 q = p; q-- > 0 && (u32)(keys[q] >> 32) == h;) {
            if (prefmax[q] < qstart) break;   // nothing at or before q reaches the query
            const FRow rj = rows[vals[q]];
            i64 lo, hi;
            filter_interval(rj, lo, hi);
            if (hi >= qstart && lo <= qstop) { const bool d = filter_pair_ok(ri, rj, P, boom); ok = ok && d; }
        }
        if (boom) {   // (local row order is not input order across the job's buckets: grec is)
            atomicMin(&meta->assert_rec, i);
            atomicMin(reinterpret_cast<unsigned long long*>(&meta->assert_grec), (unsigned long long)rows[i].grec);
        }
        keep[i] = ok ? 1 : 0;
        if (!ok) {
            atomicAdd(&meta->n_filtered, 1u);
            atomicAdd(reinterpret_cast<unsigned long long*>(&meta->filtered_len), (unsigned long long)(P.is_paf ? ri.paf_bases : ri.block_length));
        }
    }
}

// ---- the job (inputs of any size, several GPUs): rows partitioned by query-name bucket -----------------------------
// Whether a record is kept depends only on the records with the same query name, so the rows of a chunk are
// partitioned by bucket = the top 8 bits of the name's hash32 and every range of buckets is decided on its own.
// Load pass: k_filter_bucket_key, 3 radix passes (stable: input order within a bucket, unloaded lines last),
// k_filter_bucket_offsets, k_filter_gather_rows -> the chunk layout.  Decide pass: k_filter_rekey over the rows of a
// range of buckets, then the sort, k_filter_ends / k_segmax and k_filter_sweep.  Emit pass: k_filter_scatter_keep.
constexpr u32 kFBuckets = 256;
__global__ void __launch_bounds__(128) k_filter_bucket_key(const u64* __restrict__ keys, u32 n, u64* __restrict__ pkeys) {
    for (u32 r = blockIdx.x * blockDim.x + threadIdx.x; r < n; r += gridDim.x * blockDim.x)
        pkeys[r] = keys[r] == ~0ULL ? (u64)kFBuckets : keys[r] >> 56;
}
// off[b] = first position whose bucket is >= b (b = 0 .. kFBuckets; off[kFBuckets] = loaded rows), over sorted pkeys
__global__ void __launch_bounds__(128) k_filter_bucket_offsets(const u64* __restrict__ pkeys, u32 n, u32* __restrict__ off) {
    for (u32 p = blockIdx.x * blockDim.x + threadIdx.x; p <= n; p += gridDim.x * blockDim.x) {
        const u32 lo = p == 0 ? 0u : (u32)pkeys[p - 1] + 1u;
        const u32 hi = p == n ? kFBuckets : (u32)pkeys[p];
        for (u32 b = lo; b <= hi && b <= kFBuckets; ++b) off[b] = p;
    }
}
__global__ void __launch_bounds__(128) k_filter_gather_rows(const FRow* __restrict__ rows, const u32* __restrict__ vals, u32 n, FRow* __restrict__ out) {
    for (u32 p = blockIdx.x * blockDim.x + threadIdx.x; p < n; p += gridDim.x * blockDim.x) out[p] = rows[vals[p]];
}
__global__ void __launch_bounds__(128) k_filter_rekey(const FRow* __restrict__ rows, u32 n, u64* __restrict__ keys, u32* __restrict__ vals) {
    for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        keys[i] = filter_sort_key(rows[i]);
        vals[i] = i;
    }
}
__global__ void __launch_bounds__(128) k_filter_scatter_keep(const u32* __restrict__ vals, const u8* __restrict__ keep_layout, u32 n, u8* __restrict__ keep) {
    for (u32 p = blockIdx.x * blockDim.x + threadIdx.x; p < n; p += gridDim.x * blockDim.x) keep[vals[p]] = keep_layout[p];
}

// ---- printing a kept record ---------------------------------------------------------------------------
// tags of [from, len) in name order (std::map iteration): repeated selection of the smallest key above the last one.
// The fields are collected in one scan (FTags); with more than kUMaxTags of them the text is rescanned for every field.
struct FTags {
    u32 n;                  // > kUMaxTags: more than fit
    u32 a[kUMaxTags];
    u16 len[kUMaxTags];     // bytes of the whole field
    u8 k[kUMaxTags];        // bytes of its name
    u32 last_a, last_n;
    bool have_last, left;
};
G2P_HD void filter_tags_collect(const u8* r, u32 from, u32 len, FTags& T) {
    T.n = 0; T.last_a = T.last_n = 0; T.have_last = false; T.left = true;
    u32 p0 = from;
    while (p0 < len && T.n <= kUMaxTags) {
        u32 e0 = p0;
        while (e0 < len && r[e0] != '\t') ++e0;
        if (e0 > p0) {
            u32 k0 = p0;
            while (k0 < e0 && r[k0] != ':') ++k0;
            if (T.n < kUMaxTags && k0 - p0 <= 255u && e0 - p0 <= 65535u) { T.a[T.n] = p0; T.len[T.n] = (u16)(e0 - p0); T.k[T.n] = (u8)(k0 - p0); ++T.n; }
            else T.n = kUMaxTags + 1;
        }
        p0 = e0 + 1;
    }
}
// prints the next tag in name order; T.left = false when there is none
template <class Sink>
G2P_HD void filter_tags_next(const u8* r, u32 from, u32 len, bool last_wins, FTags& T, Sink& S) {
    bool found = false;
    u32 best_a = 0, best_b = 0, best_k = 0;
    if (T.n <= kUMaxTags) {
        for (u32 j = 0; j < T.n; ++j) {
            const u32 p0 = T.a[j], kn = T.k[j];
            // (PAF mode: a repeated tag name overwrites the earlier one in the reference's std::map -- the last one is printed)
            const int cb = found ? u_key_cmp(r + p0, kn, r + best_a, best_k) : -1;
            if ((!T.have_last || u_key_cmp(r + p0, kn, r + T.last_a, T.last_n) > 0) && (cb < 0 || (cb == 0 && last_wins))) {
                found = true; best_a = p0; best_b = p0 + T.len[j]; best_k = kn;
            }
        }
    } else {
        u32 p0 = from;
        while (p0 < len) {
            u32 e0 = p0;
            while (e0 < len && r[e0] != '\t') ++e0;
            if (e0 > p0) {
                u32 k0 = p0;
                while (k0 < e0 && r[k0] != ':') ++k0;
                const u32 kn = k0 - p0;
                const int cb = found ? u_key_cmp(r + p0, kn, r + best_a, best_k) : -1;
                if ((!T.have_last || u_key_cmp(r + p0, kn, r + T.last_a, T.last_n) > 0) && (cb < 0 || (cb == 0 && last_wins))) {
                    found = true; best_a = p0; best_b = e0; best_k = kn;
                }
            }
            p0 = e0 + 1;
        }
    }
    if (!found) { T.left = false; return; }
    S.ch('\t');
    S.bytes(r + best_a, best_b - best_a);
    T.last_a = best_a; T.last_n = best_k; T.have_last = true;
}
template <class Sink>
G2P_HD void filter_put_tags_sorted(const u8* r, u32 from, u32 len, bool last_wins, Sink& S) {
    FTags T;
    filter_tags_collect(r, from, len, T);
    while (T.left) filter_tags_next(r, from, len, last_wins, T, S);
}

// operator<<(GafRecord) (gafkluge.hpp:288-323) of an unchanged record
template <class Sink>
G2P_HD u32 filter_print_gaf_head(const u8* r, u32 len, Sink& S) {   // the 12 columns; returns where the optional fields begin
    URecHdr h;
    u_parse_header(r, len, h);
    S.bytes(r, h.qn_b); S.ch('\t');
    u_put_int(S, h.qlen); S.ch('\t');
    u_put_int(S, h.qs); S.ch('\t');
    u_put_int(S, h.qe); S.ch('\t');
    S.ch(h.strand); S.ch('\t');
    if (h.empty_path) { for (int k = 0; k < 6; ++k) { S.ch('*'); S.ch('\t'); } }
    else {
        // steps are re-serialised token by token (operator<<(GafStep), gafkluge.hpp:274-283): ">name", or
        // ">name:start-end" with the two numbers as std::stol read them (">a:007-10:9" prints ">a:7-10"); a bare stable
        // name is printed as it is
        if (!h.prefixed) S.bytes(r + h.path_a, h.path_b - h.path_a);
        else {
            u32 p = h.path_a;
            while (p < h.path_b) {
                const u32 q = next_marker(r, p + 1, h.path_b);
                StepTok t;
                parse_step_token<false>(r, p, q, t);
                S.ch(r[p]);
                S.bytes(r + t.name_a, t.name_b - t.name_a);
                if (t.is_interval) { S.ch(':'); S.dec(t.start); S.ch('-'); S.dec(t.end); }
                p = q;
            }
        }
        S.ch('\t');
        u_put_int(S, h.plen); S.ch('\t');
        u_put_int(S, h.ps); S.ch('\t');
        u_put_int(S, h.pe); S.ch('\t');
        u_put_int(S, h.m); S.ch('\t');
        u_put_int(S, h.b); S.ch('\t');
    }
    S.dec(h.mapq == -1 ? 255 : (i64)h.mapq);
    return h.tags_from;
}
template <class Sink>
G2P_HD void filter_print_gaf(const u8* r, u32 len, Sink& S) {
    const u32 from = filter_print_gaf_head(r, len, S);
    filter_put_tags_sorted(r, from, len, false, S);
    S.ch('\n');
}

// operator<<(PafLine) (paf.hpp:83-95): 12 columns (numbers through stol), then every tag -- cg included, see the header -- in name order
template <class Sink>
G2P_HD u32 filter_print_paf_head(const u8* r, u32 len, Sink& S) {
    u32 p = 0, k = 0, tags_from = len;
    while (p <= len && k < 12) {
        u32 e = p;
        while (e < len && r[e] != '\t') ++e;
        if (e > p) {
            if (k) S.ch('\t');
            if (k == 0 || k == 4 || k == 5) S.bytes(r + p, e - p);
            else { i64 v = 0; stol_span(r, p, e, v); S.dec(v); }
            ++k;
            tags_from = e + 1 <= len ? e + 1 : len;
        }
        p = e + 1;
    }
    return tags_from;
}
template <class Sink>
G2P_HD void filter_print_paf(const u8* r, u32 len, Sink& S) {
    const u32 from = filter_print_paf_head(r, len, S);
    filter_put_tags_sorted(r, from, len, true, S);
    S.ch('\n');
}

// One record per thread, in phases with the warp meeting after each (as unstable_record_warp): the 12 columns, the
// collection of the optional fields, then one field per round of a warp-uniform loop.
template <class Sink>
__device__ __forceinline__ void filter_print_warp(bool act, const u8* r, u32 len, u32 is_paf, Sink& S) {
    const u32 FULL = 0xffffffffu;
    u32 from = 0;
    if (act) from = is_paf ? filter_print_paf_head(r, len, S) : filter_print_gaf_head(r, len, S);
    __syncwarp();
    FTags T;
    T.left = false;
    if (act) filter_tags_collect(r, from, len, T);
    __syncwarp();
    while (__any_sync(FULL, act && T.left)) {
        if (act && T.left) filter_tags_next(r, from, len, is_paf != 0, T, S);
    }
    if (act) S.ch('\n');
}

template <bool EMIT>
__global__ void __launch_bounds__(128) k_filter_emit(const u8* __restrict__ text, const u32* __restrict__ rec_start, u32 nrec, u32 is_paf,
                                                     const u8* __restrict__ keep, u64* __restrict__ out_off, u8* __restrict__ out) {
    for (u32 base = blockIdx.x * blockDim.x; base < nrec; base += gridDim.x * blockDim.x) {   // (uniform: every lane takes part)
        const u32 r = base + threadIdx.x;
        const bool act = r < nrec && keep[r] != 0;
        const u32 s = act ? rec_start[r] : 0u, len = act ? rec_start[r + 1] - s - 1 : 0u;
        if (!EMIT) {
            CountSink cs;
            filter_print_warp(act, text + s, len, is_paf, cs);
            if (r < nrec) out_off[r] = cs.n;
        } else {
            StoreSink ss(out + (act ? out_off[r] : 0));
            filter_print_warp(act, text + s, len, is_paf, ss);
        }
    }
}

}  // namespace g2p
