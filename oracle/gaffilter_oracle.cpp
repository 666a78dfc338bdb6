// gaffilter_oracle — CPU restatement of the reference's gaffilter (gaffilter_main.cpp:31-70, 205-343).
//
// TEST INFRASTRUCTURE ONLY.  Nothing under oracle/ is linked, imported or executed by the
// product (libg2p.so, gaf2paf, gaf2unstable, gaffilter); only tests/ may run it, as the checker.
//
// Parity status: PINNED.  Every gaffilter run stored in tests/golden/reference_runs.json (the
// 41 "gaffilter_inputs" and 9 "gaffilter" entries) must be reproduced -- exit code, stdout md5,
// summary line (tests/test_filter.py::test_gaffilter_oracle_reproduces_stored_runs) -- and,
// where the reference build oracle/_ref/gaffilter exists, seeded differential runs against it.
//
// It states the rules the way the reference does and shares no code with the device
// implementation (csrc/g2p_filter.cuh): every record is loaded into std containers, records are
// grouped by the exact query-name string (no hash), the overlapping records of each record are
// found by a plain search over its group, the qualifiers and dominates() are evaluated in double
// in the reference's order of operations (build with -ffp-contract=off), the two assertions of
// the filter loop abort, kept records are re-serialised with their tags in name order (std::map).
// Inputs the reference would die on (asserts, uncaught exceptions) give exit code 134 and no
// output, without reproducing the message.
//
// usage: gaffilter_oracle [-r N] [-m N] [-o N] [-b N] [-q N] [-i N] [-p] <gaf|->   (argv as gaffilter)
#include <getopt.h>

#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <sstream>
#include <stdexcept>
#include <string>
#include <unordered_map>
#include <vector>

namespace {

struct Abort : std::runtime_error {
    using std::runtime_error::runtime_error;
};
void require(bool ok, const char* what) { if (!ok) throw Abort(what); }

// ---- one loaded record: what the filter reads, and what it prints when the record is kept
struct Step { std::string name; bool rev = false, stable = false, interval = false; int64_t start = 0, end = 0; };
struct Rec {
    std::string qname;
    int64_t qlen = 0, qs = 0, qe = 0;
    int64_t matches = 0, block_length = 0;   // GAF columns 10 / 11; PAF: gm / gl tags, else columns 10 / 11
    int64_t summed_length = 0;               // what "total block lengths filtered" adds: GAF block_length, PAF column 11
    int32_t mapq = 0;
    bool primary = true;
    std::string rc;                          // empty: no rc
    bool has_gi = false;
    float gi = 0.f;
    // printing
    char strand = '+';
    std::string target;                      // PAF column 6
    int64_t plen = 0, ps = 0, pe = 0;
    int64_t paf_columns[2] = {0, 0};         // PAF columns 10 / 11 and 12 as std::stol read them
    int64_t paf_mapq = 0;
    std::vector<Step> path;
    std::map<std::string, std::string> tags; // name -> "name:type:value" as printed
};

int64_t gaf_int(const std::string& s) { return s == "*" ? -1 : std::stol(s); }   // gafkluge.hpp:30-34
std::string int_str(int64_t v) { return v == -1 ? "*" : std::to_string(v); }    // gafkluge.hpp:25-29

// parse_gaf_record (gafkluge.hpp:84-204) and the tags gaffilter reads from it
void parse_gaf(const std::string& line, Rec& r) {
    std::vector<std::string> col;
    {
        std::istringstream in(line);
        std::string tok;
        while (std::getline(in, tok, '\t')) col.push_back(tok);
    }
    require(col.size() >= 12, "fewer than 12 columns");
    for (int k = 0; k < 12; ++k) require(!col[k].empty(), "empty column");
    r.qname = col[0];
    r.qlen = gaf_int(col[1]); r.qs = gaf_int(col[2]); r.qe = gaf_int(col[3]);
    require(col[4].size() == 1 && (col[4][0] == '+' || col[4][0] == '-' || col[4][0] == '*'), "strand");
    r.strand = col[4][0];
    const std::string& p = col[5];
    if (p[0] == '<' || p[0] == '>') {   // gafkluge.hpp:118-147
        size_t i = 0;
        while (i < p.size()) {
            size_t j = i + 1;
            while (j < p.size() && p[j] != '<' && p[j] != '>') ++j;
            Step s;
            s.rev = p[i] == '<';
            const std::string tok = p.substr(i + 1, j - i - 1);
            const size_t c = tok.find(':');
            if (c == std::string::npos) s.name = tok;
            else {
                s.name = tok.substr(0, c);
                s.stable = s.interval = true;
                const size_t d = tok.find('-', c + 1);
                require(d != std::string::npos, "range without '-'");
                s.start = std::stol(tok.substr(c + 1, d - c));
                s.end = std::stol(tok.substr(d + 1));
            }
            r.path.push_back(s);
            i = j;
        }
    } else if (p != "*") {              // a bare stable contig: one step (gafkluge.hpp:148-157)
        Step s;
        s.name = p;
        s.stable = true;
        r.path.push_back(s);
    }
    r.plen = gaf_int(col[6]); r.ps = gaf_int(col[7]); r.pe = gaf_int(col[8]);
    r.matches = gaf_int(col[9]); r.block_length = gaf_int(col[10]);
    r.summed_length = r.block_length;
    if (col[11] == "*") r.mapq = -1;
    else { const int v = std::stoi(col[11]); r.mapq = v >= 255 ? -1 : v; }   // gafkluge.hpp:176-183
    std::map<std::string, std::pair<std::string, std::string>> opt;
    for (size_t k = 12; k < col.size(); ++k) {   // gafkluge.hpp:185-202
        const std::string& f = col[k];
        if (f.empty()) continue;
        const size_t c1 = f.find(':'), c2 = c1 == std::string::npos ? c1 : f.find(':', c1 + 1);
        require(f.size() >= 5 && c1 != std::string::npos && c2 != std::string::npos, "optional tag");
        const std::string key = f.substr(0, c1);
        require(!opt.count(key), "duplicate tag");
        opt[key] = {f.substr(c1 + 1, c2 - c1 - 1), f.substr(c2 + 1)};
        r.tags[key] = f;
    }
    // gaffilter_main.cpp: a record is primary unless its tp is not P; rc names the reference contig; gi through std::stof
    if (opt.count("tp")) r.primary = opt["tp"].second == "P";
    if (opt.count("rc")) r.rc = opt["rc"].second;
    if (opt.count("gi")) { r.gi = std::stof(opt["gi"].second); r.has_gi = true; }
}

// parse_paf_line (paf.hpp:48-80): split_delims drops empty tokens
std::vector<std::string> split_delims(const std::string& s, char d) {
    std::vector<std::string> v;
    size_t a = 0;
    while (a <= s.size()) {
        size_t b = s.find(d, a);
        if (b == std::string::npos) b = s.size();
        if (b > a) v.push_back(s.substr(a, b - a));
        a = b + 1;
    }
    return v;
}
void parse_paf(const std::string& line, Rec& r) {
    const std::vector<std::string> t = split_delims(line, '\t');
    require(t.size() > 12, "fewer than 13 PAF tokens");
    r.qname = t[0];
    r.qlen = std::stol(t[1]); r.qs = std::stol(t[2]); r.qe = std::stol(t[3]);
    require(t[4] == "+" || t[4] == "-", "strand");
    r.strand = t[4][0];
    r.target = t[5];
    r.plen = std::stol(t[6]); r.ps = std::stol(t[7]); r.pe = std::stol(t[8]);
    r.paf_columns[0] = r.matches = std::stol(t[9]);
    r.paf_columns[1] = r.block_length = r.summed_length = std::stol(t[10]);
    const int64_t mapq = std::stol(t[11]);
    r.mapq = (int32_t)mapq;   // (an int64 stored into the GafRecord's int32 mapq; no 255 rule in this mode)
    std::map<std::string, std::string> val;
    for (size_t k = 12; k < t.size(); ++k) {
        const std::vector<std::string> parts = split_delims(t[k], ':');
        require(parts.size() == 3, "PAF tag without three parts");
        val[parts[0]] = parts[2];   // (a repeated name: the last one wins)
        r.tags[parts[0]] = parts[0] + ":" + parts[1] + ":" + parts[2];
    }
    if (val.count("tp")) r.primary = val["tp"] == "P";
    if (val.count("rc")) r.rc = val["rc"];
    if (val.count("gl")) r.block_length = std::stol(val["gl"]);
    if (val.count("gm")) r.matches = std::stol(val["gm"]);
    r.paf_mapq = mapq;
}


// operator<<(GafRecord) (gafkluge.hpp:288-323) / operator<<(PafLine) (paf.hpp:83-95): tags in name order
void print_gaf(const Rec& r, std::string& out) {
    out += r.qname + "\t" + int_str(r.qlen) + "\t" + int_str(r.qs) + "\t" + int_str(r.qe) + "\t";
    out.push_back(r.strand);
    out += "\t";
    if (r.path.empty()) out += "*\t*\t*\t*\t*\t*\t";
    else {
        for (const Step& s : r.path) {   // operator<<(GafStep), gafkluge.hpp:274-283
            if (!s.stable || s.interval) out.push_back(s.rev ? '<' : '>');
            out += s.name;
            if (s.interval) out += ":" + std::to_string(s.start) + "-" + std::to_string(s.end);
        }
        out += "\t" + int_str(r.plen) + "\t" + int_str(r.ps) + "\t" + int_str(r.pe) + "\t" + int_str(r.matches) + "\t" + int_str(r.block_length) + "\t";
    }
    out += std::to_string(r.mapq == -1 ? 255 : r.mapq);
    for (const auto& t : r.tags) out += "\t" + t.second;
    out += "\n";
}
void print_paf(const Rec& r, std::string& out) {
    out += r.qname + "\t" + std::to_string(r.qlen) + "\t" + std::to_string(r.qs) + "\t" + std::to_string(r.qe) + "\t";
    out.push_back(r.strand);
    out += "\t" + r.target + "\t" + std::to_string(r.plen) + "\t" + std::to_string(r.ps) + "\t" + std::to_string(r.pe) + "\t" +
           std::to_string(r.paf_columns[0]) + "\t" + std::to_string(r.paf_columns[1]) + "\t" + std::to_string(r.paf_mapq);
    for (const auto& t : r.tags) out += "\t" + t.second;
    out += "\n";
}

struct Options {
    double ratio = 0, min_overlap_pct = 0, min_identity = 0;   // std::stof, widened
    int64_t min_overlap_len = 0, min_block_len = 0, min_mapq = 0;
    bool paf = false;
};

// dominates() (gaffilter_main.cpp:31-60)
bool dominates(const Rec& g1, const Rec& g2, double ratio) {
    if (g1.qs >= g1.qe) return false;
    if (g2.qs >= g2.qe) return true;
    if (g1.primary && !g2.primary) return true;
    if (g2.primary && !g1.primary) return false;
    if ((double)g1.mapq / ((double)g2.mapq + 0.000001) >= ratio) return true;
    if ((double)g2.mapq / ((double)g1.mapq + 0.000001) >= ratio) return false;
    if ((double)g1.block_length / ((double)g2.block_length + 0.000001) >= ratio) return true;
    return false;
}
// dominates_mzgaf2paf() (gaffilter_main.cpp:63-66)
bool dominates_mz(const Rec& g1, const Rec& g2, int64_t thr) {
    return (g1.block_length >= thr && g2.block_length < thr) || (g1.block_length < thr && g2.block_length < thr);
}

// The closed interval the reference stores for a record: Interval(query_start, query_end - 1), endpoints ordered
int64_t lo_of(const Rec& r) { return std::min(r.qs, r.qe - 1); }
int64_t hi_of(const Rec& r) { return std::max(r.qs, r.qe - 1); }

// The records of one query sequence sorted by the lower end of their interval, in blocks that know the highest upper end
// among them: the search for the intervals that meet [a, b] skips blocks that end before a and stops at the first block
// that starts after b.
struct Group {
    static constexpr size_t kBlock = 64;
    std::vector<size_t> idx;
    std::vector<int64_t> lo, hi, block_hi;
    void build(const std::vector<Rec>& recs) {
        std::sort(idx.begin(), idx.end(), [&](size_t a, size_t b) { return lo_of(recs[a]) < lo_of(recs[b]); });
        for (size_t k : idx) { lo.push_back(lo_of(recs[k])); hi.push_back(hi_of(recs[k])); }
        for (size_t b = 0; b < idx.size(); b += kBlock) {
            int64_t m = INT64_MIN;
            for (size_t k = b; k < std::min(idx.size(), b + kBlock); ++k) m = std::max(m, hi[k]);
            block_hi.push_back(m);
        }
    }
    template <class F>
    void visit(int64_t a, int64_t b, F&& f) const {
        for (size_t blk = 0; blk < block_hi.size() && lo[blk * kBlock] <= b; ++blk) {
            if (block_hi[blk] < a) continue;
            for (size_t k = blk * kBlock; k < std::min(idx.size(), (blk + 1) * kBlock); ++k)
                if (lo[k] <= b && hi[k] >= a) f(idx[k]);
        }
    }
};

// The filter loop (gaffilter_main.cpp:243-330) for record i: false = filtered out.  Every interval of the query's tree
// that overlaps [query_start, end_point] is visited (end_point = query_end - 1 if query_end > query_start, else
// query_end); the decision ANDs over all of them.
bool keep_record(const std::vector<Rec>& recs, const Group& g, size_t i, const Options& O) {
    const Rec& r = recs[i];
    const int64_t end_point = r.qe > r.qs ? r.qe - 1 : r.qe;
    bool keep = true;
    g.visit(r.qs, end_point, [&](size_t j) {
        const Rec& o = recs[j];
        double identity = o.matches ? (double)o.block_length / (double)o.matches : 0.0;
        if (identity < 0.0) std::abort();   // assert(identity >= 0) (:289), the record's own interval included
        if (o.has_gi) identity = std::min(identity, (double)o.gi);
        if (j == i) return;
        // qualifiers of the overlapping record (-q, -b, -i)
        if (!(o.mapq >= O.min_mapq && (o.qlen <= O.min_block_len || o.block_length >= O.min_block_len) && identity >= O.min_identity)) return;
        if (!r.rc.empty() && !o.rc.empty() && r.rc != o.rc) return;   // they map to different reference contigs
        // overlap_size (:68-70)
        const int64_t ostart = std::max(r.qs, o.qs), oend = std::min(r.qe, o.qe);
        if (oend < ostart) std::abort();   // assert(oend >= ostart)
        const int64_t overlap = oend - ostart;
        if (r.block_length != 0 && (double)overlap / (double)r.block_length < O.min_overlap_pct) return;   // -m
        bool dom = true;
        if (O.ratio != 0) dom = dominates(r, o, O.ratio);
        if (dom && O.min_overlap_len) dom = dominates_mz(r, o, O.min_overlap_len);
        keep = keep && dom;
    });
    return keep;
}

void help(char** argv) {
    std::fprintf(stderr, "usage: %s [options] <gaf> > output.gaf\n", argv[0]);
}

int run(int argc, char** argv) {
    Options O;
    optind = 1;
    static const struct option long_options[] = {
        {"help", no_argument, 0, 'h'},
        {"ratio", required_argument, 0, 'r'},
        {"min-overlap", required_argument, 0, 'm'},
        {"min-overlap-length", required_argument, 0, 'o'},
        {"min-block-length", required_argument, 0, 'b'},
        {"min-mapq", required_argument, 0, 'q'},
        {"min-identity", required_argument, 0, 'i'},
        {"paf", no_argument, 0, 'p'},
        {0, 0, 0, 0}};
    while (true) {
        int option_index = 0;
        const int c = getopt_long(argc, argv, "h:r:m:po:b:q:i:", long_options, &option_index);
        if (c == -1) break;
        switch (c) {
            case 'r': O.ratio = std::stof(optarg); break;
            case 'm': O.min_overlap_pct = std::stof(optarg); break;
            case 'o': O.min_overlap_len = std::stol(optarg); break;
            case 'p': O.paf = true; break;
            case 'b': O.min_block_len = std::stol(optarg); break;
            case 'i': O.min_identity = std::stof(optarg); break;
            case 'q': O.min_mapq = std::stol(optarg); break;
            default: help(argv); return 1;
        }
    }
    if (argc <= 1) { help(argv); return 1; }
    if (O.ratio == 0 && O.min_overlap_len == 0) {
        std::fprintf(stderr, "[gaffilter] error: at least one of -r or -o must be used to specify filter\n");
        return 1;
    }
    if (optind >= argc) { std::fprintf(stderr, "[gaffilter] error: too few arguments\n"); help(argv); return 1; }
    const std::string path = argv[optind];
    std::string text;
    {
        FILE* f = path == "-" ? stdin : std::fopen(path.c_str(), "rb");
        if (!f) { std::fprintf(stderr, "[gaffilter] error: unable to open input: %s\n", path.c_str()); return 1; }
        char buf[1 << 16];
        size_t k;
        while ((k = std::fread(buf, 1, sizeof buf, f)) > 0) text.append(buf, k);
        if (f != stdin) std::fclose(f);
    }
    // load every record (lines starting with '*' are skipped); the query's records form one group
    std::vector<Rec> recs;
    std::unordered_map<std::string, size_t> group_of;
    std::vector<Group> groups;
    std::vector<size_t> rec_group;
    {
        std::istringstream lines(text);
        std::string line;
        while (std::getline(lines, line)) {
            if (line[0] == '*') continue;
            Rec r;
            if (O.paf) parse_paf(line, r); else parse_gaf(line, r);
            auto it = group_of.emplace(r.qname, groups.size()).first;
            if (it->second == groups.size()) groups.emplace_back();
            groups[it->second].idx.push_back(recs.size());
            rec_group.push_back(it->second);
            recs.push_back(std::move(r));
        }
    }
    for (Group& g : groups) g.build(recs);
    std::string out;
    size_t n_filtered = 0;
    uint64_t filtered_len = 0;   // (an int64_t in the reference: wraps, printed signed)
    for (size_t i = 0; i < recs.size(); ++i) {
        if (keep_record(recs, groups[rec_group[i]], i, O)) {
            if (O.paf) print_paf(recs[i], out); else print_gaf(recs[i], out);
        } else {
            ++n_filtered;
            filtered_len += (uint64_t)recs[i].summed_length;
        }
    }
    std::fprintf(stderr, "[gaffilter]: Loaded %zu %s records\n[gaffilter]: Constructed interval trees\n", recs.size(), O.paf ? "PAF" : "GAF");
    std::fwrite(out.data(), 1, out.size(), stdout);
    std::fflush(stdout);
    std::fprintf(stderr, "[gaffilter]: filtered %zu / %zu. total block lengths filtered: %lld\n", n_filtered, recs.size(), (long long)filtered_len);
    return 0;
}

}  // namespace

int main(int argc, char** argv) {
    try {
        return run(argc, argv);
    } catch (const std::exception& e) {   // the reference's uncaught exceptions and assertions: SIGABRT, nothing printed
        std::fprintf(stderr, "abort: %s\n", e.what());
        return 134;
    }
}
