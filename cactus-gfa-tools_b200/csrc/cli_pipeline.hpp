// cli_pipeline.hpp — the host side of the two drop-in executables (gaf2paf, gaf2unstable):
// a three-stage pipeline around the C-ABI's host-buffer calls.
//
//   reader      cuts the inputs (argv order, "-" = stdin) into newline-aligned chunks and fills pinned
//               buffers; regular files are read with parallel pread()s straight into pinned memory
//   converters  one host thread per GPU: chunk s goes to GPU s % N (sharding by newline-aligned byte
//               ranges, SURVEY.md §8e), one C-ABI call per chunk
//   writer      the calling thread: writes the chunks' outputs to stdout in input order (parallel
//               pwrite()s when stdout is a regular file), prints the per-chunk stderr text in order and
//               stops at the first failing record like the reference's exit()/abort()
//
// Two input slots per GPU, and the library keeps two pinned output buffers per context (a result stays
// valid until the next-but-one call, include/g2p.h), so that reading chunk s+N, converting chunk s and
// writing chunk s-N overlap.  The reference's process boundary (gaf2paf_main.cpp:342-374,
// gaf2unstable_main.cpp:288-297) is unchanged: stdout carries the records of all inputs in order.
#pragma once
#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <cerrno>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/g2p.h"

namespace cli {

inline long env_long(const char* k, long dflt) {
    const char* v = getenv(k);
    return v && *v ? strtol(v, nullptr, 10) : dflt;
}

inline bool read_file(const std::string& path, std::string& out) {
    FILE* f = fopen(path.c_str(), "rb");
    if (!f) return false;
    char buf[1 << 16];
    size_t k;
    while ((k = fread(buf, 1, sizeof buf, f)) > 0) out.append(buf, k);
    fclose(f);
    return true;
}

inline void write_seq(int fd, const char* p, size_t n) {
    while (n) {
        ssize_t k = ::write(fd, p, n);
        if (k < 0) {
            if (errno == EINTR) continue;
            _exit(1);   // downstream closed: nothing sensible left to do
        }
        p += k;
        n -= (size_t)k;
    }
}

// smallest span one I/O thread gets (tests lower it to exercise the parallel paths on small files)
inline size_t io_min_bytes() {
    static const size_t v = (size_t)std::max(1L, env_long("G2P_IO_MIN_BYTES", 1L << 20));
    return v;
}

inline int io_threads() {
    static const int t = (int)std::max(1L, std::min(16L, env_long("G2P_IO_THREADS", std::max(1u, std::thread::hardware_concurrency() / 2))));
    return t;
}

// n bytes at file offset off -> buf, with several pread()s in flight (page cache / tmpfs copies run at
// memcpy speed per thread, so one thread caps a 1.4 GB input at ~0.5 s)
inline bool pread_parallel(int fd, char* buf, size_t n, off_t off) {
    const size_t kMin = io_min_bytes();
    const int T = (int)std::min<size_t>((size_t)io_threads(), std::max<size_t>(1, n / kMin));
    bool ok = true;
    auto part = [&](size_t a, size_t b) {
        while (a < b) {
            ssize_t k = ::pread(fd, buf + a, b - a, off + (off_t)a);
            if (k < 0) { if (errno == EINTR) continue; ok = false; return; }
            if (k == 0) { ok = false; return; }
            a += (size_t)k;
        }
    };
    if (T <= 1) { part(0, n); return ok; }
    std::vector<std::thread> th;
    for (int t = 1; t < T; ++t) th.emplace_back(part, n * t / T, n * (t + 1) / T);
    part(0, n / T);
    for (auto& x : th) x.join();
    return ok;
}

// stdout writer: sequential write(), or parallel pwrite() when fd 1 is a regular file not opened O_APPEND
struct OutWriter {
    bool par = false;
    off_t pos = 0;
    OutWriter() {
        struct stat st;
        const int fl = fcntl(1, F_GETFL);
        if (fstat(1, &st) == 0 && S_ISREG(st.st_mode) && fl != -1 && !(fl & O_APPEND) && io_threads() > 1) {
            pos = lseek(1, 0, SEEK_CUR);
            par = pos != (off_t)-1;
        }
    }
    void write(const char* p, size_t n) {
        const size_t kMin = io_min_bytes();
        if (!par || n < 2 * kMin) {
            write_seq(1, p, n);
            if (par) pos += (off_t)n;
            return;
        }
        const int T = (int)std::min<size_t>((size_t)io_threads(), n / kMin);
        auto part = [&](size_t a, size_t b) {
            while (a < b) {
                ssize_t k = ::pwrite(1, p + a, b - a, pos + (off_t)a);
                if (k < 0) { if (errno == EINTR) continue; _exit(1); }
                a += (size_t)k;
            }
        };
        std::vector<std::thread> th;
        for (int t = 1; t < T; ++t) th.emplace_back(part, n * t / T, n * (t + 1) / T);
        part(0, n / T);
        for (auto& x : th) x.join();
        pos += (off_t)n;
        lseek(1, pos, SEEK_SET);
    }
};

struct Chunk {
    char* buf = nullptr;       // pinned input
    size_t cap = 0, n = 0;
    const char* out = nullptr; // library-owned pinned output of this chunk's call
    g2p_result res;
    int rc = G2P_OK;
    std::string err_text;      // stderr text that belongs before this chunk's output (gaf2unstable warnings)
    std::string open_error;    // non-empty: not a data chunk -- an input could not be opened (printed in order, then exit 1)
    int state = 0;             // 0 free, 1 filled, 2 converted
    size_t seq = 0;            // chunk number, in input order
};

struct Pipeline {
    std::vector<g2p_ctx*> ctx;          // one per GPU
    size_t chunk_bytes = 16u << 20;
    bool chunk_auto = true;             // size the chunks from the records: short reads 16 MB (small pinned buffers, early overlap of
                                        // read / convert / write), long records up to 512 MB (a GPU call must hold enough of them)
    const char* tool = "gaf2paf";
    // one C-ABI call: fills c.out, c.res (and c.err_text); returns G2P_*
    std::function<int(g2p_ctx*, Chunk&)> convert;
    // called by the writer after a chunk's output is on stdout and its record status is not OK: prints the
    // reference's message and terminates the process
    std::function<void(Chunk&)> on_record_error;

    uint64_t tot_rec = 0, tot_in = 0, tot_out = 0;
    double device_ms = 0;

    int run(const std::vector<std::string>& inputs) {
        const int ngpu = (int)ctx.size(), nslots = 2 * ngpu;
        std::vector<Chunk> slots(nslots);
        std::mutex mu;
        std::condition_variable cv;
        size_t total = (size_t)-1;   // number of chunks, known when the reader is done
        bool stop = false;

        auto ensure_cap = [&](Chunk& c, size_t want, size_t keep) -> bool {
            if (want <= c.cap) return true;
            const size_t cap = want + (want >> 3) + (1u << 20);
            char* nb = static_cast<char*>(g2p_host_alloc(cap));
            if (!nb) return false;
            if (keep) memcpy(nb, c.buf, keep);
            if (c.buf) g2p_host_free(c.buf);
            c.buf = nb; c.cap = cap;
            return true;
        };

        std::thread reader([&] {
            size_t s = 0;
            auto acquire = [&]() -> Chunk* {   // the next slot, once the writer has released it
                Chunk& c = slots[s % nslots];
                std::unique_lock<std::mutex> lk(mu);
                cv.wait(lk, [&] { return c.state == 0 || stop; });
                return stop ? nullptr : &c;
            };
            auto publish = [&](Chunk& c) {
                std::lock_guard<std::mutex> g(mu);
                c.seq = s;
                c.state = c.open_error.empty() ? 1 : 2;
                ++s;
                cv.notify_all();
            };
            auto fail = [&](const std::string& msg) {   // reported by the writer, in order
                Chunk* c = acquire();
                if (!c) return;
                c->n = 0; c->open_error = msg;
                publish(*c);
            };
            bool aborted = false;
            for (const std::string& path : inputs) {
                if (aborted) break;
                const bool is_stdin = path == "-";
                const int fd = is_stdin ? 0 : ::open(path.c_str(), O_RDONLY);
                if (fd < 0) {
                    fail("[" + std::string(tool) + "] error: unable to open input: " + path + "\n");
                    break;
                }
                struct stat st;
                const bool regular = fstat(fd, &st) == 0 && S_ISREG(st.st_mode) && st.st_size > 0 && lseek(fd, 0, SEEK_CUR) == 0;
                if (regular) {
                    const size_t size = (size_t)st.st_size;
                    size_t pos = 0;
                    if (chunk_auto) {   // mean record length of the first MiB
                        std::vector<char> probe(std::min<size_t>(size, 1u << 20));
                        const ssize_t got = ::pread(fd, probe.data(), probe.size(), 0);
                        size_t nl = 1;
                        for (ssize_t i = 0; i < got; ++i) nl += probe[i] == '\n';
                        const size_t mean = got > 0 ? (size_t)got / nl : 128;
                        chunk_bytes = std::min<size_t>(std::max<size_t>(mean * 65536u, 16u << 20), 512u << 20);
                    }
                    while (pos < size) {
                        Chunk* c = acquire();
                        if (!c) { aborted = true; break; }
                        size_t want = std::min(chunk_bytes, size - pos), n = 0;
                        for (;;) {
                            if (!ensure_cap(*c, want + 1, 0) || !pread_parallel(fd, c->buf, want, (off_t)pos)) {
                                fail("[" + std::string(tool) + "] error: cannot read " + path + "\n");
                                aborted = true;
                                break;
                            }
                            if (pos + want >= size) { n = want; break; }
                            const void* nl = memrchr(c->buf, '\n', want);
                            if (nl) { n = (size_t)(static_cast<const char*>(nl) - c->buf) + 1; break; }
                            if (want >= 0xE0000000ULL) {
                                fail("[" + std::string(tool) + "] error: line longer than 4 GiB\n");
                                aborted = true;
                                break;
                            }
                            want = std::min(want * 2, size - pos);   // a single line longer than the chunk
                        }
                        if (aborted) break;
                        c->n = n;
                        c->open_error.clear();
                        publish(*c);
                        pos += n;
                    }
                } else {
                    // pipe / stdin / empty or special file: sequential read(), the bytes after the last newline
                    // are carried into the next chunk
                    std::string carry;
                    bool eof = false;
                    while (!eof) {
                        Chunk* c = acquire();
                        if (!c) { aborted = true; break; }
                        size_t have = 0;
                        for (;;) {
                            if (!ensure_cap(*c, carry.size() + chunk_bytes + 1, 0)) { aborted = true; break; }
                            memcpy(c->buf, carry.data(), carry.size());
                            have = carry.size();
                            carry.clear();
                            while (have < chunk_bytes) {
                                ssize_t k = ::read(fd, c->buf + have, chunk_bytes - have);
                                if (k < 0) { if (errno == EINTR) continue; k = 0; }
                                if (k == 0) { eof = true; break; }
                                have += (size_t)k;
                            }
                            if (eof) break;
                            const void* nl = memrchr(c->buf, '\n', have);
                            if (nl) {
                                const size_t cut = (size_t)(static_cast<const char*>(nl) - c->buf) + 1;
                                carry.assign(c->buf + cut, have - cut);
                                have = cut;
                                break;
                            }
                            carry.assign(c->buf, have);   // a single line longer than the chunk: keep reading it
                            if (carry.size() >= 0xE0000000ULL) { aborted = true; break; }
                            chunk_bytes = std::max(chunk_bytes, carry.size() * 2);
                        }
                        if (aborted) { fail("[" + std::string(tool) + "] error: line longer than 4 GiB\n"); break; }
                        if (have == 0 && eof) break;
                        c->n = have;
                        c->open_error.clear();
                        publish(*c);
                    }
                }
                if (!is_stdin) ::close(fd);
            }
            std::lock_guard<std::mutex> g(mu);
            total = s;
            cv.notify_all();
        });

        std::vector<std::thread> conv;
        for (int g = 0; g < ngpu; ++g) {
            conv.emplace_back([&, g] {
                for (size_t s = (size_t)g;; s += (size_t)ngpu) {
                    Chunk& c = slots[s % nslots];
                    {
                        std::unique_lock<std::mutex> lk(mu);
                        // chunk s is in its slot when s chunks before it ... simply: the slot is filled and it is this GPU's turn
                        cv.wait(lk, [&] { return stop || s >= total || c.state == 1 || (c.state == 2 && !c.open_error.empty()); });
                        if (stop || s >= total) return;
                        if (c.state == 2) continue;   // an open-error marker: the writer handles it
                    }
                    c.err_text.clear();
                    c.rc = convert(ctx[g], c);
                    std::lock_guard<std::mutex> lk(mu);
                    c.state = 2;
                    cv.notify_all();
                }
            });
        }

        OutWriter ow;
        int exit_code = 0;
        for (size_t s = 0;; ++s) {
            Chunk& c = slots[s % nslots];
            {
                std::unique_lock<std::mutex> lk(mu);
                cv.wait(lk, [&] { return s >= total || c.state == 2; });
                if (s >= total && c.state != 2) break;
                if (s >= total) break;
            }
            auto halt = [&] {
                std::lock_guard<std::mutex> lk(mu);
                stop = true;
                cv.notify_all();
            };
            if (!c.open_error.empty()) {
                fputs(c.open_error.c_str(), stderr);
                exit_code = 1;
                halt();
                break;
            }
            if (c.rc != G2P_OK) {
                fprintf(stderr, "[%s] error: GPU conversion failed: %s\n", tool, g2p_last_error(ctx[s % ngpu]));
                exit_code = 1;
                halt();
                break;
            }
            if (!c.err_text.empty()) fputs(c.err_text.c_str(), stderr);
            ow.write(c.out, c.res.out_bytes);
            device_ms += c.res.device_ms;
            tot_rec += c.res.n_records; tot_in += c.n; tot_out += c.res.out_bytes;
            if (c.res.rec_status != G2P_REC_OK) {
                fflush(stderr);
                on_record_error(c);   // does not return
                _exit(1);
            }
            std::lock_guard<std::mutex> lk(mu);
            c.state = 0;
            cv.notify_all();
        }
        if (exit_code) {
            // threads may be inside CUDA calls: leave without tearing the process down under them
            fflush(stderr);
            _exit(exit_code);
        }
        reader.join();
        for (auto& t : conv) t.join();
        for (auto& c : slots) if (c.buf) g2p_host_free(c.buf);
        return 0;
    }
};

}  // namespace cli
