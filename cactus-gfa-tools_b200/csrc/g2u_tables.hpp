// g2u_tables.hpp — the flat arrays gaf2unstable's kernels read, and its warning text, on the host.
//
// g2p_load_rgfa builds one RgfaHost per rGFA and keeps it: every context that loads or shares the tables uploads
// the same arrays (g2p_capi.cu), and g2p_format_unstable_warning reads its node -> reference contig map.  The CPU
// stub of the C-ABI (tests/hostsim/g2u_stub_capi.cpp) runs the per-record code on the same arrays.
#pragma once
#include <set>
#include <string>
#include <vector>

#include "g2p_table.hpp"
#include "g2u_core.cuh"
#include "g2u_rgfa.hpp"

namespace g2p {

struct RgfaHost {
    RgfaTables T;
    HostLenTable contigs;        // stable contig name -> contig index (UnstableView::contigs)
    std::vector<u32> begin;      // [ncontig + 1] into nodes
    std::vector<UNode> nodes;    // per contig, sorted by SO
    std::vector<u8> names;
    std::vector<u32> refoff;     // [nref + 1] into refnames
    std::vector<u8> refnames;
    std::string node_lengths;    // the -o file, rows in the reference's order
    HostLenTable node_table;     // node name -> length: what `gaf2paf -l <the -o file>` would load

    // host pointers into the arrays above (the device copy has the same layout)
    UnstableView view() const {
        UnstableView v;
        v.contigs = contigs.view();
        v.contig_begin = begin.data(); v.nodes = nodes.data(); v.node_names = names.data();
        v.ref_off = refoff.data(); v.ref_names = refnames.data();
        return v;
    }
};

// Flattens H.T (built by build_rgfa_tables, without an exit code): contig hash -> index, nodes per contig sorted by
// SO, names, node -> reference contig, the -o text and its lengths table.  false: that table does not parse.
inline bool flatten_rgfa(RgfaHost& H) {
    const RgfaTables& T = H.T;
    H.contigs.reserve_for(T.mapping.size());
    u32 ci = 0;
    for (const auto& cs : T.mapping) {
        H.contigs.put(reinterpret_cast<const u8*>(cs.first.data()), (u32)cs.first.size(), (i64)ci++);
        H.begin.push_back((u32)H.nodes.size());
        i64 cum = 0;
        for (const RgfaNode& nd : cs.second) {
            UNode u;
            u.offset = nd.offset; u.cum = cum; u.length = (u32)nd.length;
            u.name_off = (u32)H.names.size(); u.name_len = (u32)nd.name.size();
            H.names.insert(H.names.end(), nd.name.begin(), nd.name.end());
            int64_t id;
            u.ref = -1;
            if (rgfa_detail::node_id_of(nd.name, id)) {
                auto it = T.node_to_contig.find(id);
                if (it != T.node_to_contig.end()) u.ref = (i32)it->second;
            }
            cum += nd.length;
            H.nodes.push_back(u);
            H.node_lengths += nd.name;
            H.node_lengths += '\t';
            H.node_lengths += std::to_string(nd.length);
            H.node_lengths += '\n';
        }
    }
    H.begin.push_back((u32)H.nodes.size());
    if (H.contigs.arena.empty()) H.contigs.arena.push_back(0);
    H.refoff.assign(1, 0);
    for (const std::string& c : T.ref_contigs) { H.refnames.insert(H.refnames.end(), c.begin(), c.end()); H.refoff.push_back((u32)H.refnames.size()); }
    // no array is empty: the device copies need a valid base address
    if (H.names.empty()) H.names.push_back(0);
    if (H.refnames.empty()) H.refnames.push_back(0);
    if (H.nodes.empty()) H.nodes.push_back(UNode{0, 0, 0, 0, 0, -1});
    return build_len_table(H.node_lengths.data(), H.node_lengths.size(), H.node_table) == ST_OK;
}

// "[gaf2unstable] warning: Target path spans multiple reference contigs a, b, \nthe (unstable) record is\n<line>\n"
// (gaf2unstable_main.cpp:165-171): contig names in ascending contig-id order; the record printed
// there does not carry an rc tag of its own making, which is what the output line holds as well.
// false: the line has fewer than six columns.
inline bool format_unstable_warning(const RgfaTables& T, const char* line, size_t len, std::string& m) {
    // column 6 = the path
    size_t a = 0;
    for (int c = 0; c < 5 && a < len; ++c) { const void* t = std::memchr(line + a, '\t', len - a); if (!t) return false; a = static_cast<const char*>(t) - line + 1; }
    const void* te = std::memchr(line + a, '\t', len - a);
    const size_t b = te ? static_cast<const char*>(te) - line : len;
    std::set<int64_t> ids;
    size_t p = a;
    while (p < b) {
        size_t q = p + 1;
        while (q < b && line[q] != '>' && line[q] != '<') ++q;
        int64_t id;
        if (rgfa_detail::node_id_of(std::string(line + p + 1, q - p - 1), id)) {
            auto it = T.node_to_contig.find(id);
            if (it != T.node_to_contig.end()) ids.insert(it->second);
        }
        p = q;
    }
    m = "[gaf2unstable] warning: Target path spans multiple reference contigs ";
    for (int64_t id : ids) { m += T.ref_contigs[(size_t)id]; m += ", "; }
    m += "\nthe (unstable) record is\n";
    size_t ll = len;
    while (ll > 0 && line[ll - 1] == '\n') --ll;
    m.append(line, ll);
    m += "\n";
    return true;
}

}  // namespace g2p
