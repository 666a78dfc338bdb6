// g2u_hostsim — CPU instantiation of the gaf2unstable per-record code (g2u_core.cuh) and of the
// host-side rGFA tables and warning text (g2u_rgfa.hpp, g2u_tables.hpp).
//
// TEST INFRASTRUCTURE ONLY: never linked into libg2p.so or the executables.  Mirrors
// g2p_load_rgfa + run_unstable (g2p_capi.cu) with plain host arrays so that CPU-only CI can check
// the rewrite against the reference binary and the golden vectors.
//
// usage: g2u_hostsim -g graph.gfa [-o node-lengths.tsv] <gaf|->      (stdout / exit code as gaf2unstable)
// stderr: the reference's multi-contig warnings, verbatim; on a record the reference aborts on, "abort: status N" last.
//
// Built with -DG2U_SIMT (build/g2u_simt): the kernels themselves, run by the SIMT emulator (cuda_shim.hpp) over the whole
// input -- size pass, scan, emit pass, then the warnings as run_unstable (g2p_capi.cu) builds them: the first n_deleg
// entries of warn_list, sorted, cut at first_err.
//   default            k_unstable<false/true>, 64-thread CTAs like run_unstable, the grid capped at G2U_SIMT_CTAS CTAs
//                      (default 3) so that the grid-stride loop takes several turns
//   G2U_SIMT_STAGED=1  k_unstable_staged<false/true> (build/g2u_simt_small, built with tiny staging buffers, always)
//   G2P_SIMT_STATS=1   prints the kernel, the grid, the stride turns and the listed warnings to stderr
#if defined(G2U_SIMT)
#define HS_IMPLEMENTATION
#include "cuda_shim.hpp"
#include "../../cactus-gfa-tools_b200/csrc/g2p_kernels.cuh"
#endif
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../cactus-gfa-tools_b200/csrc/g2u_tables.hpp"

#ifndef G2U_SIMT_STAGED_ONLY
#define G2U_SIMT_STAGED_ONLY 0
#endif

using namespace g2p;

static bool slurp(const char* path, std::string& out) {
    FILE* f = std::strcmp(path, "-") == 0 ? stdin : std::fopen(path, "rb");
    if (!f) return false;
    char buf[1 << 16];
    size_t k;
    while ((k = std::fread(buf, 1, sizeof buf, f)) > 0) out.append(buf, k);
    if (f != stdin) std::fclose(f);
    return true;
}

int main(int argc, char** argv) {
    const char *gfa = nullptr, *olen = nullptr, *in = nullptr;
    for (int i = 1; i < argc; ++i) {
        if (!std::strcmp(argv[i], "-g") && i + 1 < argc) gfa = argv[++i];
        else if (!std::strcmp(argv[i], "-o") && i + 1 < argc) olen = argv[++i];
        else in = argv[i];
    }
    if (!gfa || !in) { std::fprintf(stderr, "usage: g2u_hostsim -g graph.gfa [-o lengths.tsv] <gaf>\n"); return 1; }
    std::string rg, gaf;
    if (!slurp(gfa, rg)) { std::fprintf(stderr, "[gaf2unstable] error: Could not open %s\n", gfa); return 1; }
    if (!slurp(in, gaf)) { std::fprintf(stderr, "[gaf2unstable] error: unable to open input: %s\n", in); return 1; }
    RgfaHost H;
    build_rgfa_tables(rg.data(), rg.size(), H.T);
    if (H.T.exit_code) { std::fputs(H.T.error.c_str(), stderr); std::fputc('\n', stderr); return H.T.exit_code; }
    if (!flatten_rgfa(H)) { std::fprintf(stderr, "hostsim: node lengths table\n"); return 99; }
    if (olen) {
        FILE* o = std::fopen(olen, "wb");
        if (!o) { std::fprintf(stderr, "[gaf2unstable] error: unable to open output: %s\n", olen); return 1; }
        std::fwrite(H.node_lengths.data(), 1, H.node_lengths.size(), o);
        std::fclose(o);
    }
    const UnstableView V = H.view();
    auto warn = [&](const u8* line, size_t len) {
        std::string m;
        format_unstable_warning(H.T, reinterpret_cast<const char*>(line), len, m);
        std::fputs(m.c_str(), stderr);
    };

#if defined(G2U_SIMT)
    {
        const u64 n = gaf.size();
        std::vector<uint4> buf((n + 15) / 16 + 4);
        u8* text = reinterpret_cast<u8*>(buf.data());
        std::memcpy(text, gaf.data(), n);
        std::vector<u32> rec{0};
        for (u64 i = 0; i < n; ++i) if (text[i] == '\n') rec.push_back((u32)i + 1);
        if (n && text[n - 1] != '\n') rec.push_back((u32)n + 1);   // unterminated last line: virtual newline, as the line index does
        const u32 nrec = (u32)rec.size() - 1;
        if (nrec == 0) return 0;
        rec.push_back(0);
        std::vector<u64> off(nrec + 1, 0);
        std::vector<u32> status(nrec), wl(nrec, 0xFFFFFFFFu);
        PipelineMeta meta;
        std::memset(&meta, 0, sizeof meta);
        meta.first_err = 0xFFFFFFFFu;
        const bool staged = G2U_SIMT_STAGED_ONLY || (std::getenv("G2U_SIMT_STAGED") && std::atoi(std::getenv("G2U_SIMT_STAGED")) != 0);
        const u32 cap = std::getenv("G2U_SIMT_CTAS") ? (u32)std::atoi(std::getenv("G2U_SIMT_CTAS")) : 3u;
        const u32 ncta = std::min<u32>((nrec + kListThreads - 1) / kListThreads, cap ? cap : 1u);   // run_unstable: capped at n_sm * 32
        const u32 ncta_s = (nrec + kUThreads - 1) / kUThreads;
        auto pass = [&](auto emit, u8* out) {
            constexpr bool E = decltype(emit)::value;
            if (staged) hs::launch(dim3(ncta_s), dim3(kUThreads), unstable_smem<E>(), [&] { k_unstable_staged<E>(text, n, rec.data(), nrec, V, off.data(), status.data(), out, &meta, wl.data()); });
            else hs::launch(dim3(ncta), dim3(kListThreads), 0, [&] { k_unstable<E>(text, rec.data(), nrec, V, off.data(), status.data(), out, &meta, wl.data()); });
        };
        pass(std::false_type{}, nullptr);
        u64 run = 0;
        for (u32 r = 0; r <= nrec; ++r) { const u64 c = r < nrec ? off[r] : 0; off[r] = run; run += c; }
        std::vector<u8> outb(run + 64, 0xEE);
        pass(std::true_type{}, outb.data());
        if (std::getenv("G2P_SIMT_STATS")) {
            const u32 per = staged ? kUThreads : ncta * kListThreads;
            std::fprintf(stderr, "g2u_simt: %s, %u records, %u CTAs of %u threads, %u stride turns, %u warnings listed\n",
                         staged ? "k_unstable_staged" : "k_unstable", nrec, staged ? ncta_s : ncta, staged ? kUThreads : (u32)kListThreads,
                         staged ? 1u : (nrec + per - 1) / per, meta.n_deleg);
        }
        const u32 stop = meta.first_err == 0xFFFFFFFFu ? nrec : meta.first_err;
        std::fwrite(outb.data(), 1, off[stop], stdout);
        std::fflush(stdout);
        std::vector<u32> listed(wl.begin(), wl.begin() + meta.n_deleg);
        std::sort(listed.begin(), listed.end());
        for (u32 r : listed) {
            if (r >= stop) break;
            warn(outb.data() + off[r], off[r + 1] - off[r]);
        }
        if (stop != nrec) { std::fprintf(stderr, "abort: status %u\n", status[stop] & 0xff); return 134; }
        return 0;
    }
#endif
    if (!gaf.empty() && gaf.back() != '\n') gaf.push_back('\n');
    const u8* base = reinterpret_cast<const u8*>(gaf.data());
    std::string out;
    for (size_t i = 0; i < gaf.size();) {
        const char* nl = static_cast<const char*>(std::memchr(gaf.data() + i, '\n', gaf.size() - i));
        const u32 len = (u32)(nl - (gaf.data() + i));
        CountSink cs;
        u32 ea, eb;
        const u32 st = unstable_record(base + i, len, V, cs, ea, eb);
        if (st_is_abort(st)) {
            std::fwrite(out.data(), 1, out.size(), stdout);
            std::fflush(stdout);
            std::fprintf(stderr, "abort: status %u\n", st & 0xff);
            return 134;
        }
        if ((st & 0xff) != ST_SKIP) {
            const size_t o0 = out.size();
            out.resize(o0 + cs.n);
            StoreSink ss(reinterpret_cast<u8*>(&out[o0]));
            unstable_record(base + i, len, V, ss, ea, eb);
            if ((size_t)(ss.p - reinterpret_cast<u8*>(&out[o0])) != cs.n) { std::fprintf(stderr, "hostsim: pass mismatch\n"); return 99; }
            if ((st & 0xff) == ST_WARN_MULTIREF) warn(reinterpret_cast<const u8*>(&out[o0]), cs.n);
        }
        i = (size_t)(nl - gaf.data()) + 1;
    }
    std::fwrite(out.data(), 1, out.size(), stdout);
    return 0;
}
