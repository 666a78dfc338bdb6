// gaffilter — drop-in command line for the reference tool of the same name (reference gaffilter_main.cpp:68-352):
// same options, same stdout bytes, same stderr lines and exit codes; loading, overlap search and the dominance test
// run on a B200 through g2p_filter_host (include/g2p.h, csrc/g2p_filter.cuh).
//
//   gaffilter [options] <gaf> > output.gaf
//     -r N  -m N  -o N  -q N  -b N  -i N  -p        (see help)
//
// Environment: G2P_DEVICE=K (device ordinal).  The whole input is one call (< 4 GiB), like the reference, which holds
// every record in memory before it prints the first one.
#include <getopt.h>
#include <sys/stat.h>
#include <unistd.h>

#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <iostream>
#include <string>
#include <thread>
#include <vector>

#include "cli_pipeline.hpp"

using namespace std;

static void help(char** argv) {
    cerr << "usage: " << argv[0] << " [options] <gaf> > output.gaf" << endl
         << "Filter GAF record if its query interval overlaps another query interval and\n"
         << "  1) the record is secondary and the overlapping record is primary or\n"
         << "  2) the record's MAPQ is lower than {ratio, see -r} times the overlapping record's MAPQ or\n"
         << "  3) the record's block length is less than {ratio, see -r} times larger than the overlapping record's block length (and its MAPQ isn't higher)" << endl
         << "  Also: the -o option can be used to mimic mzgaf2paf's query overlap filter" << endl
         << endl
         << "options: " << endl
         << "    -r, --ratio N                   If two query blocks overlap, and one is Nx bigger than the other, the bigger one is kept (otherwise both deleted) [0]" << endl
         << "    -m, --min-overlap N             Ignore overlaps that consitute <N% of the length [0]" << endl
         << "    -o, --min-overlap-length N      If >= 2 query regions with size >= N overlap, ignore the query region.  If 1 query region with size >= N overlaps any regions of size <= N, ignore the smaller ones only. Works separate to -r/-m but can be used in conjunction with them to combine the two filters (0 = disable) [0]" << endl
         << "    -q, --min-mapq N                Don't let an interval with MAPQ < N cause something to be filtered out" << endl
         << "    -b, --min-block-length N        Don't let an interval with block length < N cause something to be filtered out" << endl
         << "    -i, --min-identity N            Don't let an interval with identity < N cause something to be filtered out" << endl
         << "    -p, --paf                       Input is PAF, not GAF" << endl;
}

int main(int argc, char** argv) {
    g2p_filter_params P;
    memset(&P, 0, sizeof P);
    int c;
    optind = 1;
    while (true) {
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
        int option_index = 0;
        c = getopt_long(argc, argv, "h:r:m:po:b:q:i:", long_options, &option_index);
        if (c == -1) break;
        switch (c) {
            case 'r': P.ratio = stof(optarg); break;             // (std::stof like the reference: a float widened to double)
            case 'm': P.min_overlap_pct = stof(optarg); break;
            case 'o': P.min_overlap_len = std::stol(optarg); break;
            case 'p': P.is_paf = 1; break;
            case 'b': P.min_block_len = std::stol(optarg); break;
            case 'i': P.min_identity = std::stof(optarg); break;
            case 'q': P.min_mapq = std::stol(optarg); break;
            case 'h':
            case '?':
                help(argv);
                exit(1);
            default: abort();
        }
    }
    if (argc <= 1) { help(argv); return 1; }
    if (P.ratio == 0 && P.min_overlap_len == 0) {
        cerr << "[gaffilter] error: at least one of -r or -o must be used to specify filter" << endl;
        return 1;
    }
    if (optind >= argc) {
        cerr << "[gaffilter] error: too few arguments" << endl;
        help(argv);
        return 1;
    }
    const string gaf_path = argv[optind++];
    const uint64_t kSingleLimit = 0xFFFFFFF0ULL;   // g2p_filter_host: < 4 GiB (32-bit line index and record numbers)
    const int ngpu = (int)std::max(1L, cli::env_long("G2P_GPUS", 1));
    const int dev0 = (int)cli::env_long("G2P_DEVICE", 0);
    const bool tiny_chunks = cli::env_long("G2P_CHUNK_BYTES", 0) > 0;   // (tests)
    size_t chunk = (size_t)std::min(std::max(1L, cli::env_long("G2P_CHUNK_MB", 512)), 3072L) << 20;
    if (tiny_chunks) chunk = (size_t)cli::env_long("G2P_CHUNK_BYTES", 0);
    bool use_job = ngpu > 1 || tiny_chunks;
    bool stream_file = false;   // the job reads the file itself, twice
    string text;
    if (gaf_path == "-") {
        char buf[1 << 16];
        size_t k;
        while ((k = fread(buf, 1, sizeof buf, stdin)) > 0) text.append(buf, k);
    } else {
        struct stat st;
        FILE* f = fopen(gaf_path.c_str(), "rb");
        const bool regular = f && fstat(fileno(f), &st) == 0 && S_ISREG(st.st_mode);
        if (f) fclose(f);
        if (regular && (use_job || (uint64_t)st.st_size >= kSingleLimit)) use_job = stream_file = true;
        else if (!cli::read_file(gaf_path, text)) {
            cerr << "[gaffilter] error: unable to open input: " << gaf_path << endl;
            return 1;
        }
    }
    if (!stream_file && text.size() >= kSingleLimit) use_job = true;
    if (!use_job) {
        g2p_ctx* ctx = nullptr;
        if (g2p_create(dev0, &ctx) != G2P_OK) {
            cerr << "[gaffilter] error: no usable CUDA device (this build has no CPU path)" << endl;
            return 1;
        }
        const char* out = nullptr;
        g2p_filter_result res;
        const int rc = g2p_filter_host(ctx, text.data(), text.size(), &P, &out, &res);
        if (rc != G2P_OK) { cerr << "[gaffilter] error: " << g2p_last_error(ctx) << endl; return 1; }
        if (res.rec_status != G2P_REC_OK) {
            // the reference dies while it loads the records (assert / uncaught exception): nothing was printed yet
            cerr << "terminate: gaffilter cannot parse line " << res.err_record << " (status " << res.rec_status << ")" << endl;
            abort();
        }
        cerr << "[gaffilter]: Loaded " << res.n_loaded << (P.is_paf ? " PAF" : " GAF") << " records" << endl;
        cerr << "[gaffilter]: Constructed interval trees" << endl;
        cli::write_seq(1, out, res.out_bytes);
        cerr << "[gaffilter]: filtered " << res.n_filtered << " / " << res.n_loaded << ". total block lengths filtered: " << (long long)res.filtered_len << endl;   // (an int64_t in the reference: a sum beyond 2^63 prints negative)
        g2p_destroy(ctx);
        return 0;
    }

    // ---- the job: load pass, decide, emit pass over the same chunks (chunk s on GPU s % N) ----
    auto t0 = std::chrono::steady_clock::now();
    std::vector<g2p_ctx*> ctxs(ngpu, nullptr);
    std::vector<int> crc(ngpu, G2P_OK);
    {
        std::vector<std::thread> th;
        for (int g = 0; g < ngpu; ++g) th.emplace_back([&, g] { crc[g] = g2p_create(dev0 + g, &ctxs[g]); });
        for (auto& t : th) t.join();
    }
    for (int g = 0; g < ngpu; ++g)
        if (crc[g] != G2P_OK) {
            cerr << "[gaffilter] error: no usable CUDA device (this build has no CPU path)" << endl;
            return 1;
        }
    g2p_filter_job* job = nullptr;
    if (g2p_filter_job_create(ctxs.data(), ngpu, &P, &job) != G2P_OK) { cerr << "[gaffilter] error: cannot create the filter job" << endl; return 1; }
    auto fail = [&](g2p_ctx* ctx) {
        cerr << "[gaffilter] error: " << g2p_last_error(ctx) << endl;
        fflush(stderr);
        _exit(1);   // (other threads may be inside CUDA calls)
    };
    // in-memory input: newline-aligned pieces of about `chunk` bytes
    std::vector<std::pair<size_t, size_t>> pieces;
    if (!stream_file) {
        for (size_t pos = 0; pos < text.size();) {
            size_t end = std::min(text.size(), pos + chunk);
            if (end < text.size()) {
                const void* nl = memrchr(text.data() + pos, '\n', end - pos);
                if (nl) end = (size_t)(static_cast<const char*>(nl) - text.data()) + 1;
                else { const size_t q = text.find('\n', end); end = q == string::npos ? text.size() : q + 1; }
            }
            pieces.emplace_back(pos, end - pos);
            pos = end;
        }
    }
    auto run_pass = [&](bool emit) {
        if (stream_file) {
            cli::Pipeline L;
            L.tool = "gaffilter";
            L.chunk_bytes = chunk;
            L.chunk_auto = false;   // (both passes must cut the file at the same places)
            L.ctx = ctxs;
            L.convert = [&, emit](g2p_ctx*, cli::Chunk& c) {
                std::memset(&c.res, 0, sizeof c.res);
                if (!emit) return g2p_filter_job_load(job, c.seq, c.buf, c.n);
                g2p_filter_result r;
                const int rc = g2p_filter_job_emit(job, c.seq, c.buf, c.n, &c.out, &r);
                c.res.out_bytes = r.out_bytes;
                return rc;
            };
            L.on_record_error = [](cli::Chunk&) { abort(); };   // (the job reports no per-chunk record status)
            L.run({gaf_path});
            return;
        }
        if (!emit) {
            std::vector<std::thread> th;
            for (int g = 0; g < ngpu; ++g)
                th.emplace_back([&, g] {
                    for (size_t s = (size_t)g; s < pieces.size(); s += (size_t)ngpu)
                        if (g2p_filter_job_load(job, s, text.data() + pieces[s].first, pieces[s].second) != G2P_OK) fail(ctxs[g]);
                });
            for (auto& t : th) t.join();
            return;
        }
        for (size_t s = 0; s < pieces.size(); ++s) {
            const char* out = nullptr;
            g2p_filter_result r;
            if (g2p_filter_job_emit(job, s, text.data() + pieces[s].first, pieces[s].second, &out, &r) != G2P_OK) fail(ctxs[s % ngpu]);
            cli::write_seq(1, out, r.out_bytes);
        }
    };
    run_pass(false);
    g2p_filter_result res;
    if (g2p_filter_job_decide(job, &res) != G2P_OK) { cerr << "[gaffilter] error: " << g2p_last_error(ctxs[0]) << endl; return 1; }
    if (res.rec_status != G2P_REC_OK) {
        cerr << "terminate: gaffilter cannot parse line " << res.err_record << " (status " << res.rec_status << ")" << endl;
        abort();
    }
    cerr << "[gaffilter]: Loaded " << res.n_loaded << (P.is_paf ? " PAF" : " GAF") << " records" << endl;
    cerr << "[gaffilter]: Constructed interval trees" << endl;
    run_pass(true);
    cerr << "[gaffilter]: filtered " << res.n_filtered << " / " << res.n_loaded << ". total block lengths filtered: " << (long long)res.filtered_len << endl;
    if (cli::env_long("G2P_STATS", 0)) {
        g2p_filter_job_stats js;
        g2p_filter_job_get_stats(job, &js);
        const double wall = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
        fprintf(stderr, "[gaffilter] stats: gpus=%d load=%.3f ms decide=%.3f ms emit=%.3f ms h2d=%llu B d2h=%llu B wall=%.3f s\n", ngpu, js.load_ms, js.decide_ms,
                js.emit_ms, (unsigned long long)js.h2d_bytes, (unsigned long long)js.d2h_bytes, wall);
    }
    g2p_filter_job_destroy(job);
    for (g2p_ctx* c : ctxs) g2p_destroy(c);
    return 0;
}
