// g2u_stub_capi — a CPU stand-in for the entry points of the C-ABI (include/g2p.h) that the gaf2unstable executable calls.
//
// TEST INFRASTRUCTURE ONLY: never part of libg2p.so or of the shipped executables.  CPU-only CI links
// csrc/gaf2unstable_main.cpp against this file (build/gaf2unstable_stub) so that the HOST logic of the drop-in
// executable -- the reader / converter / writer pipeline of cli_pipeline.hpp, G2P_GPUS round-robin, ordered output
// and warnings, the rGFA tables loaded once and shared, error and exit-code paths -- runs without a GPU.
// The tables are built by the library's own host code (g2u_rgfa.hpp build_rgfa_tables, g2u_tables.hpp flatten_rgfa,
// format_unstable_warning) and the per-record code is the product's scalar device code (g2u_core.cuh unstable_record)
// instantiated for the host, exactly like build/g2u_hostsim; results are double-buffered per context as the real
// library's are.  (tests/hostsim/g2p_stub_capi.cpp is the same for gaf2paf.)
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <string>
#include <vector>

#include "../../include/g2p.h"
#include "../../cactus-gfa-tools_b200/csrc/g2u_tables.hpp"

using namespace g2p;

struct g2p_ctx {
    std::vector<u8> out[2];
    int cur = 0;
    std::string err;
    std::shared_ptr<const RgfaHost> rgfa;
    bool have_rgfa = false;
    std::vector<g2p_warn> warns;
};

extern "C" {

int g2p_create(int device, g2p_ctx** out) {
    if (!out || device < 0 || device >= 64) return G2P_E_NO_DEVICE;
    *out = new g2p_ctx();
    return G2P_OK;
}
void g2p_destroy(g2p_ctx* ctx) { delete ctx; }
const char* g2p_last_error(const g2p_ctx* ctx) { return ctx ? ctx->err.c_str() : "no context"; }
void* g2p_host_alloc(size_t bytes) { return std::malloc(bytes ? bytes : 1); }
void g2p_host_free(void* p) { std::free(p); }

int g2p_load_rgfa(g2p_ctx* ctx, const char* rgfa, size_t n, int* ref_exit_code, char* msg, size_t msg_cap) {
    if (!ctx || (!rgfa && n)) return G2P_E_ARG;
    if (ref_exit_code) *ref_exit_code = 0;
    if (msg && msg_cap) msg[0] = 0;
    auto H = std::make_shared<RgfaHost>();
    ctx->rgfa = H;
    ctx->have_rgfa = false;
    build_rgfa_tables(rgfa, n, H->T);
    if (H->T.exit_code) {
        if (ref_exit_code) *ref_exit_code = H->T.exit_code;
        if (msg && msg_cap) std::snprintf(msg, msg_cap, "%s", H->T.exit_code == 1 ? H->T.error.c_str() : "");
        ctx->err = "rGFA: " + H->T.error;
        return G2P_E_TABLE;
    }
    if (!flatten_rgfa(*H)) { ctx->err = "node lengths table"; return G2P_E_TABLE; }
    ctx->have_rgfa = true;
    return G2P_OK;
}

int g2p_share_rgfa(g2p_ctx* dst, const g2p_ctx* src) {
    if (!dst || !src || dst == src) return G2P_E_ARG;
    if (!src->have_rgfa) return G2P_E_NOTABLE;
    dst->rgfa = src->rgfa;
    dst->have_rgfa = true;
    return G2P_OK;
}

int g2p_rgfa_node_lengths(g2p_ctx* ctx, const char** tsv, size_t* n) {
    if (!ctx || !tsv || !n) return G2P_E_ARG;
    if (!ctx->have_rgfa) return G2P_E_NOTABLE;
    *tsv = ctx->rgfa->node_lengths.data();
    *n = ctx->rgfa->node_lengths.size();
    return G2P_OK;
}

// run_unstable's results: every line is a record ('*' lines print nothing), the output stops before the first record
// the reference aborts on, and the records before it whose path spans several reference contigs are listed
int g2p_unstable_host(g2p_ctx* ctx, const char* gaf, size_t n, const char** out, g2p_result* res) {
    if (!ctx || !res || !out || (!gaf && n)) return G2P_E_ARG;
    if (!ctx->have_rgfa) return G2P_E_NOTABLE;
    std::memset(res, 0, sizeof *res);
    ctx->warns.clear();
    std::vector<u8>& o = ctx->out[ctx->cur ^= 1];
    o.clear();
    const UnstableView V = ctx->rgfa->view();
    const u8* base = reinterpret_cast<const u8*>(gaf);
    size_t i = 0;
    u64 r = 0;
    while (i < n) {
        const void* nl = std::memchr(gaf + i, '\n', n - i);
        const size_t e = nl ? (size_t)(static_cast<const char*>(nl) - gaf) : n;
        CountSink cs;
        u32 ea = 0, eb = 0;
        const u32 st = unstable_record(base + i, (u32)(e - i), V, cs, ea, eb);
        if (st_is_error(st)) {
            res->rec_status = st & 0xff;
            res->rec_aux = (st >> 8) & 0xff;
            res->err_record = r;
            ++r;
            break;
        }
        if ((st & 0xff) != ST_SKIP) {
            const size_t at = o.size();
            o.resize(at + cs.n + 64);
            StoreSink ss(o.data() + at);
            unstable_record(base + i, (u32)(e - i), V, ss, ea, eb);
            o.resize(at + cs.n);
            if ((st & 0xff) == ST_WARN_MULTIREF) ctx->warns.push_back(g2p_warn{r, at, cs.n});
        }
        ++r;
        i = e + 1;
    }
    res->n_records = r;
    res->out_bytes = o.size();
    o.push_back(0);
    *out = reinterpret_cast<const char*>(o.data());
    return G2P_OK;
}

int g2p_unstable_warnings(g2p_ctx* ctx, const g2p_warn** warns, size_t* n) {
    if (!ctx || !warns || !n) return G2P_E_ARG;
    *warns = ctx->warns.data();
    *n = ctx->warns.size();
    return G2P_OK;
}

int g2p_format_unstable_warning(g2p_ctx* ctx, const char* line, size_t len, char* buf, size_t cap) {
    if (!ctx || !line || !buf || cap == 0 || !ctx->rgfa) return G2P_E_ARG;
    buf[0] = 0;
    std::string m;
    if (!format_unstable_warning(ctx->rgfa->T, line, len, m)) return G2P_E_ARG;
    std::snprintf(buf, cap, "%s", m.c_str());
    return G2P_OK;
}

}  // extern "C"
