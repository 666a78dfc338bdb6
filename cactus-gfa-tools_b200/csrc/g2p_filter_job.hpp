// g2p_filter_job.hpp — host bookkeeping of the gaffilter job (g2p_filter_job_* in g2p_capi.cu, and its CPU emulation in
// the SIMT driver tests/hostsim/g2p_filter_job_simt.cpp): what the load pass records per chunk, the bucket -> partition
// planner, the (chunk, bucket) segments of the chunk layouts, and the global line numbering.  Pure host code.
//
// A chunk's layout holds its loaded rows in bucket order (input order within a bucket); bucket b is the rows
// [off[b], off[b + 1]).  A partition is a range of buckets [b0, b1); its rows are, for every chunk c, the segment
// [off(c, b0), off(c, b1)) of that chunk's layout, so a partition is one copy per (chunk, partition).
#pragma once
#include <algorithm>
#include <cstdint>
#include <string>
#include <vector>

namespace g2p_fjob {

constexpr int kBuckets = 256;
constexpr uint32_t kNone = 0xFFFFFFFFu;

struct ChunkBook {
    bool loaded = false;
    uint64_t bytes = 0;
    uint32_t lines = 0;                  // lines of the chunk (the line index's records)
    uint32_t off[kBuckets + 1] = {};     // off[kBuckets] = loaded rows of the chunk
    uint32_t first_err = kNone;          // smallest line of the chunk that fails to load
    uint32_t err_status = 0;             // its status
    bool unsupported = false;            // a loaded query_start >= 2^32 - 16
    uint32_t n_loaded() const { return off[kBuckets]; }
    uint64_t seg_begin(int b0) const { return off[b0]; }
    uint64_t seg_rows(int b0, int b1) const { return (uint64_t)off[b1] - off[b0]; }
};

// "" when the emit pass saw the chunk the load pass saw (bytes, lines, per-bucket rows), else what differs
inline std::string same_chunk(const ChunkBook& loaded, const ChunkBook& now) {
    if (loaded.bytes != now.bytes) return "byte count";
    if (loaded.lines != now.lines) return "line count";
    for (int b = 0; b <= kBuckets; ++b)
        if (loaded.off[b] != now.off[b]) return "bucket " + std::to_string(b) + " rows";
    return "";
}

struct Part {
    int b0, b1;        // buckets [b0, b1)
    uint64_t rows;
    int gpu;
};

// total rows of every bucket over the chunks
inline std::vector<uint64_t> bucket_rows(const std::vector<ChunkBook>& chunks) {
    std::vector<uint64_t> t(kBuckets, 0);
    for (const ChunkBook& c : chunks)
        for (int b = 0; b < kBuckets; ++b) t[b] += c.seg_rows(b, b + 1);
    return t;
}

// Contiguous bucket ranges of at most `cap` rows each, at least min(max(min_parts, ngpu, ceil(total / cap)), 256) of them,
// of about equal row counts; then assigned to the GPUs, largest first to the least loaded.  Returns "" or the reason
// no plan exists (one bucket alone exceeds `cap`).
inline std::string plan_partitions(const std::vector<uint64_t>& rows, uint64_t cap, int min_parts, int ngpu, std::vector<Part>& parts) {
    parts.clear();
    if (cap == 0) cap = 1;
    if (ngpu < 1) ngpu = 1;
    uint64_t total = 0;
    for (int b = 0; b < kBuckets; ++b) {
        if (rows[b] > cap)
            return "one query-name bucket holds " + std::to_string(rows[b]) + " records, more than the " + std::to_string(cap) +
                   " a GPU can decide at once (a single query sequence with about that many alignments)";
        total += rows[b];
    }
    const uint64_t want = std::min<uint64_t>(kBuckets, std::max<uint64_t>({(uint64_t)std::max(min_parts, 1), (uint64_t)ngpu, (total + cap - 1) / cap}));
    const uint64_t target = std::max<uint64_t>(1, (total + want - 1) / want);
    int b0 = 0;
    uint64_t cur = 0;
    for (int b = 0; b < kBuckets; ++b) {
        if (cur > 0 && cur + rows[b] > target) { parts.push_back(Part{b0, b, cur, 0}); b0 = b; cur = 0; }
        cur += rows[b];
    }
    parts.push_back(Part{b0, kBuckets, cur, 0});
    // (too few ranges -- few non-empty buckets, or the test hook -- : halve the widest range until there are enough)
    while (parts.size() < want) {
        size_t w = 0;
        for (size_t i = 1; i < parts.size(); ++i) if (parts[i].b1 - parts[i].b0 > parts[w].b1 - parts[w].b0) w = i;
        if (parts[w].b1 - parts[w].b0 < 2) break;
        const int mid = (parts[w].b0 + parts[w].b1) / 2;
        Part hi{mid, parts[w].b1, 0, 0};
        parts[w].b1 = mid;
        parts[w].rows = 0;
        for (int b = parts[w].b0; b < mid; ++b) parts[w].rows += rows[b];
        for (int b = mid; b < hi.b1; ++b) hi.rows += rows[b];
        parts.insert(parts.begin() + (long)w + 1, hi);
    }
    std::vector<size_t> order(parts.size());
    for (size_t i = 0; i < order.size(); ++i) order[i] = i;
    std::stable_sort(order.begin(), order.end(), [&](size_t a, size_t b) { return parts[a].rows > parts[b].rows; });
    std::vector<uint64_t> load(ngpu, 0);
    for (size_t i : order) {
        const int g = (int)(std::min_element(load.begin(), load.end()) - load.begin());
        parts[i].gpu = g;
        load[g] += parts[i].rows;
    }
    return "";
}

// global line number of the first line of every chunk (chunks in input order), plus the total at the end
inline std::vector<uint64_t> line_bases(const std::vector<ChunkBook>& chunks) {
    std::vector<uint64_t> base(chunks.size() + 1, 0);
    for (size_t c = 0; c < chunks.size(); ++c) base[c + 1] = base[c] + chunks[c].lines;
    return base;
}
inline uint64_t global_line(const std::vector<uint64_t>& bases, uint64_t grec) { return bases[grec >> 32] + (grec & 0xFFFFFFFFu); }

// the smallest global line that fails to load, over all chunks (false: none)
inline bool first_load_error(const std::vector<ChunkBook>& chunks, const std::vector<uint64_t>& bases, uint64_t& line, uint32_t& status) {
    for (size_t c = 0; c < chunks.size(); ++c)
        if (chunks[c].first_err != kNone) { line = bases[c] + chunks[c].first_err; status = chunks[c].err_status; return true; }
    return false;
}

}  // namespace g2p_fjob
