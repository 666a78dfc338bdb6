// gaf2unstable — drop-in command line for the reference tool of the same name
// (reference gaf2unstable_main.cpp:177-301): same options (and option quirks), same stdout
// bytes, same stderr messages and exit codes; the per-record rewrite runs on B200 GPUs through
// the C-ABI of libg2p.so (include/g2p.h).
//
//   gaf2unstable [options] <gaf>
//     -g, --rgfa FILE   (uncompressed) minigraph rGFA
//     -o FILE           write "node<TAB>length" for every rGFA node (input of gaf2paf -l)
//
// Environment (argv stays identical to the reference):
//   G2P_GPUS=N        shard the input over the first N GPUs of the box by newline-aligned
//                     byte ranges; outputs and warnings are printed in input order (default 1)
//   G2P_DEVICE=K      first device ordinal (default 0)
//   G2P_CHUNK_MB=M    bytes of GAF per GPU call (default: 16 for short records, up to 512 for long ones)
//   G2P_IO_THREADS=T  threads of the parallel pread / pwrite of regular files
//   G2P_STATS=1       timing summary on stderr
//
// The rGFA tables are built once on the host (g2p_load_rgfa on the first GPU's context, while the
// other contexts are created) and copied to every other GPU (g2p_share_rgfa).  The host side is the
// reader -> per-GPU converter -> writer pipeline of cli_pipeline.hpp.
#include <fcntl.h>
#include <getopt.h>
#include <signal.h>
#include <unistd.h>

#include <cerrno>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "cli_pipeline.hpp"

namespace {

void help(char** argv) {
    fprintf(stderr,
            "usage: %s [options] <gaf> \n"
            "Replace stable sequences in path steps, ex >chr1:500-1000, with the unstable graph node names, ex >s1:1-100>s2:100-600\n"
            "\n"
            "options: \n"
            "    -g, --rGFA FILE           (uncompressed) minigraph rGFA, required to look up unstable mappings\n"
            "    -o, --out-lengths FILE    Output lengths of all minigraph sequences in given file (can be passed to gaf2paf)\n",
            argv[0]);
}

}  // namespace

int main(int argc, char** argv) {
    std::string rgfa_path, node_lengths_path;
    int c;
    optind = 1;
    while (true) {
        // the long form of -o maps to a value the switch does not handle (reference :196-226)
        static const struct option long_options[] = {
            {"help", no_argument, 0, 'h'}, {"rgfa", required_argument, 0, 'g'}, {"out-lengths", required_argument, 0, '0'}, {0, 0, 0, 0}};
        int option_index = 0;
        c = getopt_long(argc, argv, "hg:o:", long_options, &option_index);
        if (c == -1) break;
        switch (c) {
            case 'h':
                // falls through to `rgfa_path = optarg` with optarg == NULL in the reference: SIGSEGV
                raise(SIGSEGV);
                return 139;
            case 'g': rgfa_path = optarg; break;
            case 'o': node_lengths_path = optarg; break;
            case '?':
                help(argv);
                exit(1);
            default: abort();
        }
    }
    if (argc <= 1) { help(argv); return 1; }
    if (optind >= argc) {
        fprintf(stderr, "[gaf2unstable] error: too few arguments\n");
        help(argv);
        return 1;
    }
    const std::string in_gaf_path = argv[optind++];
    if (optind < argc - 1) {
        fprintf(stderr, "[gaf2unstable] error: too many arguments\n");
        help(argv);
        return 1;
    }
    if (rgfa_path.empty()) {
        fprintf(stderr, "[gaf2unstable] error: -g option required\n");
        return 1;
    }
    {   // the reference opens the GAF before it reads the rGFA (gaf2unstable_main.cpp:248-262)
        if (in_gaf_path != "-") {
            int fd = open(in_gaf_path.c_str(), O_RDONLY);
            if (fd == -1) {
                fprintf(stderr, "[gaf2unstable] error: unable to open input: %s\n", in_gaf_path.c_str());
                return 1;
            }
            close(fd);
        }
    }
    std::string rgfa;
    if (!cli::read_file(rgfa_path, rgfa)) {
        fprintf(stderr, "[gaf2unstable] error: Could not open %s\n", rgfa_path.c_str());
        return 1;
    }
    {   // the reference maps the file O_RDWR and asserts on failure (gfakluge.hpp:570-573)
        int fd = open(rgfa_path.c_str(), O_RDWR);
        if (fd == -1) abort();
        close(fd);
    }

    const int ngpu = (int)std::max(1L, cli::env_long("G2P_GPUS", 1));
    const int dev0 = (int)cli::env_long("G2P_DEVICE", 0);
    const bool stats = cli::env_long("G2P_STATS", 0) != 0;
    using clk = std::chrono::steady_clock;
    auto secs = [](clk::time_point t) { return std::chrono::duration<double>(clk::now() - t).count(); };

    // one context per GPU, created concurrently (CUDA context creation is the bulk of the start-up time); the first one
    // builds the rGFA tables meanwhile
    std::vector<g2p_ctx*> ctx(ngpu, nullptr);
    std::vector<int> crc(ngpu, G2P_OK);
    std::vector<std::thread> th;
    for (int g = 1; g < ngpu; ++g) th.emplace_back([&, g] { crc[g] = g2p_create(dev0 + g, &ctx[g]); });
    crc[0] = g2p_create(dev0, &ctx[0]);
    int ref_rc = 0, rc = G2P_OK;
    std::vector<char> msg(1 << 16);
    double load_s = 0;
    if (crc[0] == G2P_OK) {
        const auto t = clk::now();
        rc = g2p_load_rgfa(ctx[0], rgfa.data(), rgfa.size(), &ref_rc, msg.data(), msg.size());
        load_s = secs(t);
    }
    for (auto& t : th) t.join();
    th.clear();
    if (crc[0] != G2P_OK) {
        fprintf(stderr, "[gaf2unstable] error: no usable CUDA device (this build has no CPU path)\n");
        return 1;
    }
    if (rc == G2P_E_TABLE) {
        fputs(msg.data(), stderr);
        if (ref_rc == 1) return 1;
        abort();
    }
    if (rc != G2P_OK) { fprintf(stderr, "[gaf2unstable] error: %s\n", g2p_last_error(ctx[0])); return 1; }
    std::string().swap(rgfa);
    for (int g = 1; g < ngpu; ++g)
        if (crc[g] != G2P_OK) {
            fprintf(stderr, "[gaf2unstable] error: no usable CUDA device %d (this build has no CPU path)\n", dev0 + g);
            return 1;
        }

    if (!node_lengths_path.empty()) {
        FILE* o = fopen(node_lengths_path.c_str(), "wb");
        if (!o) {
            fprintf(stderr, "[gaf2unstable] error: unable to open output: %s\n", node_lengths_path.c_str());
            return 1;
        }
        const char* tsv = nullptr;
        size_t n = 0;
        g2p_rgfa_node_lengths(ctx[0], &tsv, &n);
        fwrite(tsv, 1, n, o);
        fclose(o);
    }

    // the tables of the first context go to the others: no second pass over the rGFA
    const auto t_share = clk::now();
    std::vector<int> src(ngpu, G2P_OK);
    for (int g = 1; g < ngpu; ++g) th.emplace_back([&, g] { src[g] = g2p_share_rgfa(ctx[g], ctx[0]); });
    for (auto& t : th) t.join();
    const double share_s = secs(t_share);
    for (int g = 1; g < ngpu; ++g)
        if (src[g] != G2P_OK) { fprintf(stderr, "[gaf2unstable] error: %s\n", g2p_last_error(ctx[g])); return 1; }

    size_t chunk = (size_t)std::max(1L, cli::env_long("G2P_CHUNK_MB", 16)) << 20;
    if (cli::env_long("G2P_CHUNK_BYTES", 0) > 0) chunk = (size_t)cli::env_long("G2P_CHUNK_BYTES", 0);   // tests: tiny chunks
    cli::Pipeline P;
    P.tool = "gaf2unstable";
    P.chunk_bytes = chunk;
    P.chunk_auto = !getenv("G2P_CHUNK_MB") && !getenv("G2P_CHUNK_BYTES");
    P.ctx = ctx;
    P.convert = [](g2p_ctx* cx, cli::Chunk& c) {
        int r = g2p_unstable_host(cx, c.buf, c.n, &c.out, &c.res);
        if (r != G2P_OK) return r;
        // the reference prints its multi-contig warning while it converts the record: keep the texts with the chunk
        const g2p_warn* warns = nullptr;
        size_t nw = 0;
        g2p_unstable_warnings(cx, &warns, &nw);
        std::vector<char> wmsg(1 << 16);
        for (size_t i = 0; i < nw; ++i) {
            if (wmsg.size() < warns[i].out_len + 4096) wmsg.resize(warns[i].out_len + 4096);
            g2p_format_unstable_warning(cx, c.out + warns[i].out_off, warns[i].out_len, wmsg.data(), wmsg.size());
            c.err_text += wmsg.data();
        }
        return r;
    };
    P.on_record_error = [](cli::Chunk& c) {
        fprintf(stderr, "terminate: gaf2unstable cannot convert record %llu of this block (status %u)\n", (unsigned long long)c.res.err_record,
                c.res.rec_status);
        fflush(stderr);
        abort();   // reference: assert / uncaught exception -> SIGABRT
    };
    const auto t0 = clk::now();
    if (stats) fprintf(stderr, "[gaf2unstable] stats: contexts ready\n");
    const int prc = P.run({in_gaf_path});
    if (stats)
        fprintf(stderr, "[gaf2unstable] stats: records=%llu in=%llu B out=%llu B device=%.3f ms wall=%.3f s gpus=%d rgfa=%.3f s share=%.3f s\n",
                (unsigned long long)P.tot_rec, (unsigned long long)P.tot_in, (unsigned long long)P.tot_out, P.device_ms, secs(t0), ngpu, load_s,
                share_s);
    for (g2p_ctx* c : P.ctx) g2p_destroy(c);
    return prc;
}
