// g2p_filter_job_simt — the gaffilter job (g2p_filter_job_* in g2p_capi.cu: the kernels of csrc/g2p_filter.cuh over
// newline-aligned chunks, the rows partitioned by query name) executed on the CPU by the SIMT emulator.  TEST
// INFRASTRUCTURE ONLY; the launch sequences mirror the job's, its host bookkeeping is csrc/g2p_filter_job.hpp itself.
// g2p_filter_simt runs the single call the same way.
//
// usage: g2p_filter_job_simt [-p] [-r R] [-m M] [-o N] [-b N] [-q N] [-i X] [-c BYTES] [-P PARTS] <gaf|->
//          (stdout / stderr / exit code as g2p_filter_simt): the job's three passes -- load per newline-aligned chunk
//          of about BYTES (default: one chunk), decide per partition (at least PARTS of them), emit per chunk
//        g2p_filter_job_simt --plan CAP MIN_PARTS NGPU     (stdin: 256 bucket row counts)
//          the partition plan of g2p_fjob::plan_partitions: one "b0 b1 rows gpu" line per partition, or
//          "error: ..." and exit 3
#define HS_IMPLEMENTATION
#include "cuda_shim.hpp"

#include <iostream>
#include <string>

#include "../../cactus-gfa-tools_b200/csrc/g2p_kernels.cuh"
#include "../../cactus-gfa-tools_b200/csrc/g2p_filter_job.hpp"

using namespace g2p;

// one text block on the "device": aligned copy, line index, parse
struct Block {
    std::vector<uint4> tb;
    const u8* text = nullptr;
    u64 n = 0;
    u32 nrec = 0;
    std::vector<u32> rec;
    std::vector<FRow> rows;
    std::vector<u64> k1, k2, hist, blocks, off;
    std::vector<u32> v1, v2;
    u64 *keys = nullptr, *keys2 = nullptr;
    u32 *vals = nullptr, *vals2 = nullptr;
    std::vector<u8> keep;
    FilterMeta fm;
    FilterArgs fa;
    u32 nblk = 0, nh = 0, nscan_h = 0, nscan_r = 0;

    void alloc(u32 rows_n) {   // work arrays for rows_n rows (filter_work)
        nrec = rows_n;
        nblk = (nrec + kRsTile - 1) / kRsTile; nh = 16u * nblk;
        nscan_h = (nh + kScanTile - 1) / kScanTile; nscan_r = (nrec + kScanTile - 1) / kScanTile;
        rows.assign(nrec, FRow());
        k1.assign(nrec, 0); k2.assign(nrec, 0); hist.assign(nh + 2, 0); blocks.assign(std::max(nscan_h, nscan_r) * 2 + 2, 0); off.assign(nrec + 1, 0);
        v1.assign(nrec, 0); v2.assign(nrec, 0);
        keep.assign(nrec, 0);
        keys = k1.data(); keys2 = k2.data(); vals = v1.data(); vals2 = v2.data();
        std::memset(&fm, 0, sizeof fm);
        fm.first_err = 0xFFFFFFFFu;
        fm.assert_rec = 0xFFFFFFFFu;
        fm.assert_grec = ~0ULL;
    }
    void parse(const char* src, u64 bytes, u64 grec_base, const FilterParams& P) {
        n = bytes;
        tb.assign((n + 15) / 16 + 4, uint4{0, 0, 0, 0});
        u8* t = reinterpret_cast<u8*>(tb.data());
        if (n) std::memcpy(t, src, n);
        text = t;
        PipelineMeta meta;
        std::memset(&meta, 0, sizeof meta);
        const u32 ntiles = (u32)((n + kIdxTile - 1) / kIdxTile);
        std::vector<u32> tiles(ntiles + 1);
        if (ntiles) hs::launch(dim3(ntiles), dim3(kIdxThreads), 0, [&] { k_count_lines(text, n, tiles.data()); });
        hs::launch(dim3(1), dim3(1024), 0, [&] { k_scan_tiles(tiles.data(), ntiles, text, n, &meta); });
        rec.assign(meta.n_records + 2, 0);
        if (ntiles) hs::launch(dim3(ntiles), dim3(kIdxThreads), 0, [&] { k_fill_lines(text, n, tiles.data(), rec.data(), &meta); });
        alloc(meta.n_records);
        fa = FilterArgs{text, rec.data(), nrec, P, rows.data(), keys, vals, &fm, grec_base};
        if (nrec) hs::launch(dim3(4), dim3(128), 0, [&] { k_filter_parse(fa); });
    }
    void rsort(u32 passes) {
        for (u32 shift = 0; shift < 4 * passes; shift += 4) {
            hs::launch(dim3(nblk), dim3(kRsThreads), 0, [&] { k_rs_hist(keys, nrec, shift, hist.data(), nblk); });
            hs::launch(dim3(nscan_h), dim3(kScanThreads), 0, [&] { k_scan_reduce(hist.data(), nh, blocks.data()); });
            hs::launch(dim3(1), dim3(1024), 0, [&] { k_scan_blocks(blocks.data(), nscan_h, hist.data() + nh + 1); });
            hs::launch(dim3(nscan_h), dim3(kScanThreads), 0, [&] { k_scan_apply(hist.data(), nh, blocks.data(), hist.data() + nh + 1); });
            hs::launch(dim3(nblk), dim3(kRsThreads), 0, [&] { k_rs_scatter(keys, vals, keys2, vals2, nrec, shift, hist.data(), nblk); });
            std::swap(keys, keys2);
            std::swap(vals, vals2);
        }
    }
    bool decide(const FilterParams& P) {   // filter_decide
        rsort(16);
        for (u32 i = 1; i < nrec; ++i) if (keys[i - 1] > keys[i]) { std::fprintf(stderr, "g2p_filter_simt: sort order broken at %u\n", i); return false; }
        std::vector<i64> pmax(nrec);
        const u32 nseg = (nrec + kSegTile - 1) / kSegTile;
        std::vector<i64> tile_val(nseg), carry(nseg);
        std::vector<u32> tile_flag(nseg);
        hs::launch(dim3(4), dim3(256), 0, [&] { k_filter_ends(keys, vals, rows.data(), nrec, pmax.data()); });
        hs::launch(dim3(nseg), dim3(kSegThreads), 0, [&] { k_segmax<false>(keys, nrec, pmax.data(), tile_val.data(), tile_flag.data(), nullptr); });
        hs::launch(dim3(1), dim3(32), 0, [&] { k_segmax_tiles(tile_val.data(), tile_flag.data(), nseg, carry.data()); });
        hs::launch(dim3(nseg), dim3(kSegThreads), 0, [&] { k_segmax<true>(keys, nrec, pmax.data(), tile_val.data(), tile_flag.data(), carry.data()); });
        std::fill(keep.begin(), keep.end(), 0);
        hs::launch(dim3(4), dim3(128), 0, [&] { k_filter_sweep(keys, vals, rows.data(), pmax.data(), nrec, P, keep.data(), &fm); });
        return true;
    }
    void emit_sizes(u32 is_paf) {
        hs::launch(dim3(4), dim3(128), 0, [&] { k_filter_emit<false>(text, rec.data(), nrec, is_paf, keep.data(), off.data(), nullptr); });
        hs::launch(dim3(nscan_r), dim3(kScanThreads), 0, [&] { k_scan_reduce(off.data(), nrec, blocks.data()); });
        hs::launch(dim3(1), dim3(1024), 0, [&] { k_scan_blocks(blocks.data(), nscan_r, &fm.out_total); });
        hs::launch(dim3(nscan_r), dim3(kScanThreads), 0, [&] { k_scan_apply(off.data(), nrec, blocks.data(), &fm.out_total); });
    }
    void emit_text(u32 is_paf, std::vector<u8>& out) {
        out.assign(fm.out_total + 64, 0);
        hs::launch(dim3(4), dim3(128), 0, [&] { k_filter_emit<true>(text, rec.data(), nrec, is_paf, keep.data(), off.data(), out.data()); });
        out.resize(fm.out_total);
    }
    void diagnose() { if (fm.first_err != 0xFFFFFFFFu) hs::launch(dim3(1), dim3(1), 0, [&] { k_filter_diagnose(fa); }); }
    void partition(g2p_fjob::ChunkBook& bk) {   // filter_partition: afterwards vals[p] = line of layout position p
        bk.bytes = n;
        bk.lines = nrec;
        if (!nrec) return;
        hs::launch(dim3(4), dim3(128), 0, [&] { k_filter_bucket_key(keys, nrec, keys2); });
        std::swap(keys, keys2);
        rsort(3);
        hs::launch(dim3(3), dim3(128), 0, [&] { k_filter_bucket_offsets(keys, nrec, bk.off); });
        diagnose();
        bk.first_err = fm.first_err;
        bk.err_status = fm.err_status;
        bk.unsupported = fm.unsupported != 0;
    }
};


// newline-aligned pieces of about `bytes` (as gaffilter_main.cpp cuts an in-memory input)
static std::vector<std::pair<size_t, size_t>> cut(const std::string& t, size_t bytes) {
    std::vector<std::pair<size_t, size_t>> v;
    for (size_t pos = 0; pos < t.size();) {
        size_t end = std::min(t.size(), pos + bytes);
        if (end < t.size()) {
            const size_t nl = t.rfind('\n', end - 1);
            if (nl != std::string::npos && nl >= pos) end = nl + 1;
            else { const size_t q = t.find('\n', end); end = q == std::string::npos ? t.size() : q + 1; }
        }
        v.emplace_back(pos, end - pos);
        pos = end;
    }
    return v;
}

static int run_job(const std::string& text_s, const FilterParams& P, size_t chunk_bytes, int min_parts) {
    const auto pieces = cut(text_s, chunk_bytes);
    const size_t C = pieces.size();
    std::vector<g2p_fjob::ChunkBook> books(C);
    std::vector<std::vector<FRow>> lay(C);
    std::vector<std::vector<u8>> keep(C);
    // load pass
    for (size_t c = 0; c < C; ++c) {
        Block B;
        B.parse(text_s.data() + pieces[c].first, pieces[c].second, (u64)c << 32, P);
        B.partition(books[c]);
        books[c].loaded = true;
        const u32 nl = books[c].n_loaded();
        lay[c].resize(nl);
        if (nl) hs::launch(dim3(4), dim3(128), 0, [&] { k_filter_gather_rows(B.rows.data(), B.vals, nl, lay[c].data()); });
        keep[c].assign(nl, 0xEE);   // (every flag is written by exactly one partition)
    }
    // decide
    const std::vector<u64> bases = g2p_fjob::line_bases(books);
    u64 n_loaded = 0, line;
    u32 status;
    for (const auto& b : books) n_loaded += b.n_loaded();
    if (g2p_fjob::first_load_error(books, bases, line, status)) {
        std::fprintf(stderr, "abort: line %llu status %u\n", (unsigned long long)line, status & 0xff);
        return 134;
    }
    for (const auto& b : books) if (b.unsupported) { std::fprintf(stderr, "unsupported query_start\n"); return 98; }
    std::vector<g2p_fjob::Part> parts;
    const std::string perr = g2p_fjob::plan_partitions(g2p_fjob::bucket_rows(books), 0x7FFFFFFF, min_parts, 1, parts);
    if (!perr.empty()) { std::fprintf(stderr, "%s\n", perr.c_str()); return 97; }
    u64 n_filtered = 0, filtered_len = 0, assert_grec = ~0ULL;
    for (const auto& pt : parts) {
        if (!pt.rows) continue;
        Block B;
        B.alloc((u32)pt.rows);
        size_t pos = 0;
        for (size_t c = 0; c < C; ++c) {
            const size_t seg = books[c].seg_rows(pt.b0, pt.b1);
            std::copy(lay[c].begin() + books[c].seg_begin(pt.b0), lay[c].begin() + books[c].seg_begin(pt.b0) + seg, B.rows.begin() + pos);
            pos += seg;
        }
        if (pos != pt.rows) { std::fprintf(stderr, "g2p_filter_simt: partition rows %zu != planned %llu\n", pos, (unsigned long long)pt.rows); return 99; }
        hs::launch(dim3(4), dim3(128), 0, [&] { k_filter_rekey(B.rows.data(), B.nrec, B.keys, B.vals); });
        if (!B.decide(P)) return 99;
        pos = 0;
        for (size_t c = 0; c < C; ++c) {
            const size_t seg = books[c].seg_rows(pt.b0, pt.b1);
            std::copy(B.keep.begin() + pos, B.keep.begin() + pos + seg, keep[c].begin() + books[c].seg_begin(pt.b0));
            pos += seg;
        }
        n_filtered += B.fm.n_filtered;
        filtered_len += B.fm.filtered_len;
        assert_grec = std::min(assert_grec, B.fm.assert_grec);
    }
    for (const auto& k : keep) for (u8 f : k) if (f > 1) { std::fprintf(stderr, "g2p_filter_simt: a keep flag no partition wrote\n"); return 99; }
    if (assert_grec != ~0ULL) {
        std::fprintf(stderr, "abort: assertion of the filter loop on record %llu\n", (unsigned long long)g2p_fjob::global_line(bases, assert_grec));
        return 134;
    }
    std::fprintf(stderr, "[gaffilter]: Loaded %llu %s records\n[gaffilter]: Constructed interval trees\n", (unsigned long long)n_loaded, P.is_paf ? "PAF" : "GAF");
    // emit pass
    for (size_t c = 0; c < C; ++c) {
        Block B;
        B.parse(text_s.data() + pieces[c].first, pieces[c].second, (u64)c << 32, P);
        g2p_fjob::ChunkBook now;
        B.partition(now);
        const std::string diff = g2p_fjob::same_chunk(books[c], now);
        if (!diff.empty()) { std::fprintf(stderr, "g2p_filter_simt: chunk %zu differs (%s)\n", c, diff.c_str()); return 99; }
        if (!B.nrec) continue;
        const u32 nl = books[c].n_loaded();
        if (nl) hs::launch(dim3(4), dim3(128), 0, [&] { k_filter_scatter_keep(B.vals, keep[c].data(), nl, B.keep.data()); });
        B.emit_sizes(P.is_paf);
        std::vector<u8> out;
        B.emit_text(P.is_paf, out);
        std::fwrite(out.data(), 1, out.size(), stdout);
    }
    std::fprintf(stderr, "[gaffilter]: filtered %llu / %llu. total block lengths filtered: %lld\n", (unsigned long long)n_filtered, (unsigned long long)n_loaded,
                 (long long)filtered_len);
    return 0;
}

static int run_plan(char** argv) {
    const u64 cap = std::stoull(argv[0]);
    const int min_parts = std::atoi(argv[1]), ngpu = std::atoi(argv[2]);
    std::vector<u64> rows(g2p_fjob::kBuckets, 0);
    for (auto& r : rows) if (!(std::cin >> r)) return 2;
    std::vector<g2p_fjob::Part> parts;
    const std::string err = g2p_fjob::plan_partitions(rows, cap, min_parts, ngpu, parts);
    if (!err.empty()) { std::printf("error: %s\n", err.c_str()); return 3; }
    for (const auto& p : parts) std::printf("%d %d %llu %d\n", p.b0, p.b1, (unsigned long long)p.rows, p.gpu);
    return 0;
}

int main(int argc, char** argv) {
    if (argc == 5 && std::string(argv[1]) == "--plan") return run_plan(argv + 2);
    FilterParams P{0, 0, 0, 0, 0, 0, 0};
    const char* path = nullptr;
    size_t chunk_bytes = 0;
    int min_parts = 0;
    for (int i = 1; i < argc; ++i) {
        std::string a = argv[i];
        if (a == "-p") P.is_paf = 1;
        else if (a == "-r" && i + 1 < argc) P.ratio = std::stof(argv[++i]);
        else if (a == "-m" && i + 1 < argc) P.min_overlap_pct = std::stof(argv[++i]);
        else if (a == "-i" && i + 1 < argc) P.min_identity = std::stof(argv[++i]);
        else if (a == "-o" && i + 1 < argc) P.min_overlap_len = std::stol(argv[++i]);
        else if (a == "-b" && i + 1 < argc) P.min_block_len = std::stol(argv[++i]);
        else if (a == "-q" && i + 1 < argc) P.min_mapq = std::stol(argv[++i]);
        else if (a == "-c" && i + 1 < argc) chunk_bytes = std::stoull(argv[++i]);
        else if (a == "-P" && i + 1 < argc) min_parts = std::atoi(argv[++i]);
        else path = argv[i];
    }
    if (!path) return 1;
    std::string text_s;
    {
        FILE* f = std::strcmp(path, "-") == 0 ? stdin : std::fopen(path, "rb");
        if (!f) return 1;
        char buf[1 << 16];
        size_t k;
        while ((k = std::fread(buf, 1, sizeof buf, f)) > 0) text_s.append(buf, k);
    }
    return run_job(text_s, P, chunk_bytes ? chunk_bytes : (size_t)1 << 40, std::max(min_parts, 1));
}
