// g2p_capi.cu — C-ABI (include/g2p.h) over the sm_100a kernels.
//
// Owns all CUDA state: the device copy of the name->length table, grow-only work
// buffers (record index, status, output offsets, PAF output) and the pinned host
// staging used by the host-buffer entry point.  No CPU conversion path exists here:
// every byte of PAF is produced by k_convert<true>.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <mutex>
#include <set>
#include <thread>
#include <vector>
#include <cctype>
#include <chrono>
#include <sched.h>
#include <cstring>
#include <new>
#include <string>

#include "../../include/g2p.h"
#include "g2p_kernels.cuh"
#include "g2p_table.hpp"
#include "g2u_rgfa.hpp"
#include "g2p_errfmt.hpp"
#include "g2p_filter_job.hpp"
#include <memory>

using namespace g2p;

namespace {

// Pipeline counters go to the host through a kernel that stores into mapped pinned memory, not
// through cudaMemcpyAsync: a small D2H copy queues on the copy engine BEHIND the 200 MB output copy
// of another chunk (measured: every pipeline of g2p_convert_host stalled 4-9 ms on its two counter
// read-backs), a store from a kernel does not.
__global__ void k_meta_to_host(const g2p::PipelineMeta* __restrict__ src, g2p::PipelineMeta* __restrict__ dst) {
    const uint32_t* s = reinterpret_cast<const uint32_t*>(src);
    volatile uint32_t* d = reinterpret_cast<volatile uint32_t*>(dst);
    for (uint32_t i = threadIdx.x; i < sizeof(g2p::PipelineMeta) / 4; i += blockDim.x) d[i] = s[i];
    __threadfence_system();
}
static_assert(sizeof(g2p::PipelineMeta) % 4 == 0, "PipelineMeta is copied as 32-bit words");
__global__ void k_words_to_host(const uint32_t* __restrict__ src, uint32_t* __restrict__ dst, uint32_t nwords) {
    volatile uint32_t* d = dst;
    for (uint32_t i = threadIdx.x; i < nwords; i += blockDim.x) d[i] = src[i];
    __threadfence_system();
}
inline cudaError_t meta_to_host(void* h_meta, const void* d_meta, cudaStream_t st) {
    k_meta_to_host<<<1, 32, 0, st>>>(static_cast<const g2p::PipelineMeta*>(d_meta), static_cast<g2p::PipelineMeta*>(h_meta));
    return cudaGetLastError();
}

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

struct PinBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFreeHost(p);
        p = nullptr; cap = 0;
        size_t want = bytes + bytes / 8 + 4096;
        cudaError_t e = cudaHostAlloc(&p, want, cudaHostAllocMapped | cudaHostAllocPortable);   // also device-addressable (unified addressing)
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
};

}  // namespace

// One pipeline instance: a stream plus the grow-only work buffers of one in-flight chunk.
struct Worker {
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[10] = {};  // 0..4: general pipeline (index, size, scan, emit), 5..6: k_fuse, 8..9: k_par
    DevBuf f_rows, f_keys, f_keys2, f_vals, f_vals2, f_pmax, f_keep, f_hist, f_meta, f_seg, f_lay, f_boff;   // gaffilter
    DevBuf d_mid, d_in, d_tiles, d_rec, d_status, d_off, d_blocks, d_out, d_meta, d_list, d_list2, d_desc, d_rdesc, d_sdesc, d_loff, d_map, d_lsort, d_perm, d_fuse;
    DevBuf p_recs, p_tb, p_toff, p_bs, p_step, p_op, d_list3;   // k_par (g2p_par.cuh)
    PinBuf h_meta, h_fmeta, h_par;
    bool init() {
        if (cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking) != cudaSuccess) return false;
        for (auto& e : ev) if (cudaEventCreate(&e) != cudaSuccess) return false;
        return d_meta.ensure(sizeof(PipelineMeta)) == cudaSuccess && h_meta.ensure(sizeof(PipelineMeta)) == cudaSuccess &&
               h_fmeta.ensure(sizeof(FuseMeta)) == cudaSuccess && h_par.ensure(64) == cudaSuccess;
    }
    void release() {
        for (DevBuf* b : {&f_rows, &f_keys, &f_keys2, &f_vals, &f_vals2, &f_pmax, &f_keep, &f_hist, &f_meta, &f_seg, &f_lay, &f_boff, &d_mid, &d_in, &d_tiles, &d_rec, &d_status, &d_off, &d_blocks, &d_out, &d_meta, &d_list, &d_list2, &d_desc, &d_rdesc, &d_sdesc, &d_loff, &d_map, &d_lsort, &d_perm, &d_fuse, &p_recs, &p_tb, &p_toff, &p_bs, &p_step, &p_op, &d_list3}) b->release();
        h_meta.release();
        h_fmeta.release();
        h_par.release();
        for (auto& e : ev) if (e) cudaEventDestroy(e);
        if (stream) cudaStreamDestroy(stream);
    }
};

constexpr int kWorkers = 3;            // chunks in flight in g2p_convert_host: H2D / kernels / D2H overlap
constexpr size_t kHostChunk = 48u << 20;   // bytes of GAF per chunk (cut at a newline)

struct g2p_ctx {
    int device = 0;
    int n_sm = 148;
    std::string err;
    std::mutex err_mu;
    // table
    DevBuf d_slots, d_arena;
    LenTableView table{nullptr, nullptr, 0};
    uint64_t table_entries = 0;
    bool have_table = false;
    Worker w[kWorkers];
    PinBuf h_outs[2];                // pinned result buffers of the host-buffer calls, used alternately: a result stays valid until the next-but-one call
    int h_cur = 0;
    PinBuf& next_out() { h_cur ^= 1; return h_outs[h_cur]; }
    // gaf2unstable tables
    DevBuf u_slots, u_arena, u_begin, u_nodes, u_names, u_refoff, u_refnames;
    DevBuf n_slots, n_arena;              // node name -> length table of the rGFA (what gaf2unstable -o writes, loaded like gaf2paf -l)
    LenTableView node_table{nullptr, nullptr, 0};
    std::string warn_text;                // stderr text of the gaf2unstable stage of the last g2p_unstable_convert_* call
    const u8* warn_mid = nullptr;         // (built on demand from the intermediate GAF, which stays in the worker's d_mid buffer)
    bool warn_pending = false;
    UnstableView uview{};
    bool have_rgfa = false;
    RgfaTables* rgfa = nullptr;
    std::string node_lengths;
    std::vector<g2p_warn> warns;
    size_t host_chunk = kHostChunk;
    bool host_chunk_fixed = false;   // G2P_HOST_CHUNK_MB given: no adaptation to the record length
    bool two_pass_index = true;      // default: counting index (count, scan, fill); G2P_ONE_PASS_INDEX=1 selects k_index1 (measured slower, see profiles/r01_summary.md)
    bool have_cpus = false;          // CPUs of the GPU's NUMA node (G2P_NUMA_BIND=0: none)
    cpu_set_t cpus;
    bool len_sort = false;           // G2P_LEN_SORT=1: global counting sort of the records by length class before k_rec (default off: in-CTA sort only)
    bool size_kernel_short = false;  // G2P_SIZE_KERNEL=short: k_short (8 lanes per record) instead of k_rec (thread per record)
    uint32_t rec_chunks_override = 0; // G2P_REC_CHUNKS: k_rec slot capacity in 16-byte chunks
    bool unstable_staged = false;    // G2P_UNSTABLE_STAGED=1: gaf2unstable's records and output go through shared memory (k_unstable_staged).  Measured slower
                                     // (1.10 vs 0.97 ms per 294 k records): the per-record code is bound by SIMT divergence (profiles/r02_k_unstable.txt),
                                     // not by the latency of its byte loads, and the staging buffers cost occupancy
    bool par = true;                 // G2P_PAR=0: records k_rec does not take go straight to k_long (one warp per record) instead of the token-parallel kernels
    u32 long_small_max = 8;          // G2P_LONG_SMALL: k_long batches of at most this many lines take a small descriptor block (0: always 32 slots)
    uint64_t desc_cap_override = 0;  // G2P_DESC_CAP (tests): line-descriptor slots, to exercise the overflow fallback
    int fuse_mode = 1;               // G2P_FUSE: 0 never run the one-pass kernel k_fuse; 2 always try it first; 1 (default) when it pays:
                                     // k_fuse takes records of up to 1000 bytes at one speed, the two-pass pipeline is faster on records its
                                     // thread-per-record size pass k_rec takes (<= 240 bytes: 7.2 vs 9.3 ms per 10 M records) and slower on longer
                                     // ones (k_par; ~9x slower with k_long) -- so: mean record length > 200 bytes, or k_rec left > 1/32 of the
                                     // previous call's records to the long-record kernels
    std::atomic<int> prefer_fuse{0};
    int fuse_cfg = 6;                // k_fuse configuration (tile bytes, table sizes; g2p_fuse.cuh); moves to a denser one, and stays there, when a tile
                                     // holds more records / path steps than its tables (G2P_FUSE_CFG picks the first one)
    uint64_t fuse_out_cap_override = 0;   // G2P_FUSE_OUT_CAP (tests): initial output capacity of k_fuse, to exercise the grow-and-rerun path
    void set_err(const std::string& m) { std::lock_guard<std::mutex> g(err_mu); err = m; }
};

#define G2P_CUDA(call)                                                                        \
    do {                                                                                      \
        cudaError_t e__ = (call);                                                             \
        if (e__ != cudaSuccess) {                                                             \
            ctx->set_err(std::string(#call) + ": " + cudaGetErrorString(e__));                \
            return G2P_E_CUDA;                                                                \
        }                                                                                     \
    } while (0)

extern "C" {

// Host-side locality (opt-in, G2P_NUMA_BIND=1; the default leaves the caller's affinity mask alone):
// the calling thread (and the worker threads it will start, which inherit its mask)
// is restricted to the CPUs of the GPU's NUMA node, so that the pinned buffers it allocates are placed in
// that node's memory and the PCIe copies of several GPUs of one box do not all cross the socket link
// (on the single-NUMA-node VM this round was measured on it is a no-op: 8 ranks move 35 GB of host memory
// per step at ~115 GB/s with or without it).
// Nothing happens when sysfs has no node for the device or the node's CPUs are not in the current mask.
// The mask is computed once per context against the mask the process had when the first context was
// created, and applied to the thread that creates the context and to every thread that enters
// g2p_convert_host with it (several contexts, one host thread per GPU: each thread ends up on its own
// GPU's node).
static bool gpu_numa_cpus(int device, cpu_set_t* want) {
    const char* bind = std::getenv("G2P_NUMA_BIND");   // opt-in: a library must not change its host's CPU affinity by default
    if (!bind || std::atoi(bind) == 0) return false;
    static std::mutex mu;
    static bool have_orig = false;
    static cpu_set_t orig;
    {
        std::lock_guard<std::mutex> g(mu);
        if (!have_orig) {
            if (sched_getaffinity(0, sizeof orig, &orig) != 0) return false;
            have_orig = true;
        }
    }
    char bus[32] = {0};
    if (cudaDeviceGetPCIBusId(bus, (int)sizeof bus, device) != cudaSuccess) return false;
    for (char* q = bus; *q; ++q) *q = (char)std::tolower((unsigned char)*q);
    char path[160];
    std::snprintf(path, sizeof path, "/sys/bus/pci/devices/%s/numa_node", bus);
    FILE* f = std::fopen(path, "r");
    if (!f) return false;
    int node = -1;
    const int got = std::fscanf(f, "%d", &node);
    std::fclose(f);
    if (got != 1 || node < 0) return false;
    std::snprintf(path, sizeof path, "/sys/devices/system/node/node%d/cpulist", node);
    f = std::fopen(path, "r");
    if (!f) return false;
    char list[4096] = {0};
    const bool have = std::fgets(list, (int)sizeof list, f) != nullptr;
    std::fclose(f);
    if (!have) return false;
    CPU_ZERO(want);
    int n_want = 0;
    for (char* q = list; *q;) {   // "0-31,64-95"
        char* end = nullptr;
        const long a = std::strtol(q, &end, 10);
        if (end == q) break;
        long b = a;
        q = end;
        if (*q == '-') { b = std::strtol(q + 1, &end, 10); q = end; }
        for (long c = a; c <= b && c < CPU_SETSIZE; ++c)
            if (c >= 0 && CPU_ISSET((int)c, &orig)) { CPU_SET((int)c, want); ++n_want; }
        if (*q == ',') ++q; else break;
    }
    return n_want > 0;
}

int g2p_create(int device, g2p_ctx** out) {
    if (!out) return G2P_E_ARG;
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev <= 0 || device < 0 || device >= ndev) return G2P_E_NO_DEVICE;
    if (cudaSetDevice(device) != cudaSuccess) return G2P_E_NO_DEVICE;
    g2p_ctx* ctx = new (std::nothrow) g2p_ctx();
    if (!ctx) return G2P_E_ARG;
    ctx->device = device;
    ctx->have_cpus = gpu_numa_cpus(device, &ctx->cpus);
    if (ctx->have_cpus) sched_setaffinity(0, sizeof ctx->cpus, &ctx->cpus);   // before the pinned buffers are allocated
    for (auto& w : ctx->w)
        if (!w.init()) { g2p_destroy(ctx); return G2P_E_NO_DEVICE; }
    cudaFuncSetAttribute(k_short<kSG>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kShortSmem);
    cudaFuncSetAttribute(k_rec, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rec_smem(kRMaxChunks));
    if (const char* c = std::getenv("G2P_SIZE_KERNEL")) ctx->size_kernel_short = std::strcmp(c, "short") == 0;
    if (const char* c = std::getenv("G2P_LEN_SORT")) ctx->len_sort = std::atoi(c) != 0;
    if (const char* c = std::getenv("G2P_REC_CHUNKS")) ctx->rec_chunks_override = (u32)std::min(std::max(std::atoi(c), (int)kRMinChunks), (int)kRMaxChunks);
    cudaFuncSetAttribute(k_emit_lines<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kEmitSmem);
    cudaFuncSetAttribute(k_emit_lines<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kEmitSmem);
    cudaFuncSetAttribute(k_long<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)long_smem<true>());
    cudaFuncSetAttribute(k_long<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)long_smem<false>());
    cudaFuncSetAttribute(k_unstable_staged<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)unstable_smem<false>());
    cudaFuncSetAttribute(k_unstable_staged<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)unstable_smem<true>());
    cudaDeviceGetAttribute(&ctx->n_sm, cudaDevAttrMultiProcessorCount, device);
    if (const char* c = std::getenv("G2P_ONE_PASS_INDEX")) ctx->two_pass_index = std::atoi(c) == 0;
    if (const char* c = std::getenv("G2P_PAR")) ctx->par = std::atoi(c) != 0;
    if (const char* c = std::getenv("G2P_UNSTABLE_STAGED")) ctx->unstable_staged = std::atoi(c) != 0;
    if (const char* c = std::getenv("G2P_LONG_SMALL")) ctx->long_small_max = (u32)std::min(16, std::max(0, std::atoi(c)));
    if (const char* c = std::getenv("G2P_DESC_CAP")) ctx->desc_cap_override = std::strtoull(c, nullptr, 10);
    if (const char* c = std::getenv("G2P_FUSE")) ctx->fuse_mode = std::min(2, std::max(0, std::atoi(c)));
    if (const char* c = std::getenv("G2P_FUSE_OUT_CAP")) ctx->fuse_out_cap_override = std::strtoull(c, nullptr, 10);
    cudaFuncSetAttribute(k_fuse<FuseCfg0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FuseCfg0::kSmem);
    cudaFuncSetAttribute(k_fuse<FuseCfg1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FuseCfg1::kSmem);
    cudaFuncSetAttribute(k_fuse<FuseCfg2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FuseCfg2::kSmem);
    cudaFuncSetAttribute(k_fuse<FuseCfg3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FuseCfg3::kSmem);
    cudaFuncSetAttribute(k_fuse<FuseCfg4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FuseCfg4::kSmem);
    cudaFuncSetAttribute(k_fuse<FuseCfg5>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FuseCfg5::kSmem);
    cudaFuncSetAttribute(k_fuse<FuseCfg6>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FuseCfg6::kSmem);
    cudaFuncSetAttribute(k_fuse<FuseCfg7>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FuseCfg7::kSmem);
    cudaFuncSetAttribute(k_fuse<FuseCfg8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FuseCfg8::kSmem);
    if (const char* c = std::getenv("G2P_FUSE_CFG")) { const int v = std::atoi(c); if (v >= 0 && v < kFuseCfgs) ctx->fuse_cfg = v; }
    if (const char* c = std::getenv("G2P_HOST_CHUNK_MB")) {
        long v = std::atol(c);
        if (v > 0) { ctx->host_chunk = (size_t)v << 20; ctx->host_chunk_fixed = true; }
    }
    *out = ctx;
    return G2P_OK;
}

void g2p_destroy(g2p_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    ctx->d_slots.release();
    ctx->d_arena.release();
    for (DevBuf* b : {&ctx->u_slots, &ctx->u_arena, &ctx->u_begin, &ctx->u_nodes, &ctx->u_names, &ctx->u_refoff, &ctx->u_refnames, &ctx->n_slots, &ctx->n_arena}) b->release();
    delete ctx->rgfa;
    for (auto& w : ctx->w) w.release();
    for (auto& b : ctx->h_outs) b.release();
    delete ctx;
}

const char* g2p_last_error(const g2p_ctx* ctx) { return ctx ? ctx->err.c_str() : "no context"; }

void* g2p_host_alloc(size_t bytes) {
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) return nullptr;
    return p;
}
void g2p_host_free(void* p) { if (p) cudaFreeHost(p); }

int g2p_copy_to_device(void* d_dst, const void* h_src, size_t bytes) {
    return cudaMemcpy(d_dst, h_src, bytes, cudaMemcpyHostToDevice) == cudaSuccess ? G2P_OK : G2P_E_CUDA;
}
int g2p_copy_to_host(void* h_dst, const void* d_src, size_t bytes) {
    return cudaMemcpy(h_dst, d_src, bytes, cudaMemcpyDeviceToHost) == cudaSuccess ? G2P_OK : G2P_E_CUDA;
}

int g2p_load_lengths(g2p_ctx* ctx, const char* tsv, size_t n) {
    if (!ctx || (!tsv && n)) return G2P_E_ARG;
    G2P_CUDA(cudaSetDevice(ctx->device));
    HostLenTable t;
    u32 st = build_len_table(tsv, n, t);
    if (st != ST_OK) { ctx->set_err("lengths table: std::stol would throw"); return G2P_E_TABLE; }
    G2P_CUDA(cudaDeviceSynchronize());
    G2P_CUDA(ctx->d_slots.ensure(t.slots.size() * sizeof(LenSlot)));
    G2P_CUDA(ctx->d_arena.ensure(t.arena.size()));
    G2P_CUDA(cudaMemcpy(ctx->d_slots.p, t.slots.data(), t.slots.size() * sizeof(LenSlot), cudaMemcpyHostToDevice));
    G2P_CUDA(cudaMemcpy(ctx->d_arena.p, t.arena.data(), t.arena.size(), cudaMemcpyHostToDevice));
    ctx->table.slots = static_cast<const LenSlot*>(ctx->d_slots.p);
    ctx->table.arena = static_cast<const u8*>(ctx->d_arena.p);
    ctx->table.nslots = (u32)t.slots.size();
    ctx->table_entries = t.n_entries;
    ctx->have_table = true;
    return G2P_OK;
}

uint64_t g2p_table_entries(const g2p_ctx* ctx) { return ctx ? ctx->table_entries : 0; }

// Line index into w.d_rec; leaves meta (n_lines, n_records) in w.h_meta.  Default: the counting
// kernels (count, scan, fill: two reads of the text, no inter-CTA dependency).  The one-pass
// variant (k_index1: TMA tiles + decoupled look-back, index capacity of one record per 32 bytes with
// the counting kernels as its overflow fallback) is selectable but measured slower on B200: its
// 16 KiB tiles are too small to amortise the ticket / TMA / look-back latency chain.
static int run_index(g2p_ctx* ctx, Worker& w, const u8* d_text, size_t n, cudaStream_t st, uint32_t* launches) {
    const u32 ntiles = (u32)((n + kIdxTile - 1) / kIdxTile);
    G2P_CUDA(w.d_tiles.ensure(((size_t)ntiles + 2) * sizeof(u64)));
    PipelineMeta* d_meta = static_cast<PipelineMeta*>(w.d_meta.p);
    const PipelineMeta* hm = static_cast<const PipelineMeta*>(w.h_meta.p);
    if (ntiles && !ctx->two_pass_index) {
        const u64 cap64 = std::min<u64>((u64)n / 32 + 1024, 0xFFFFFFF0ULL);
        G2P_CUDA(w.d_rec.ensure((size_t)cap64 * sizeof(u32)));
        u64* d_status = static_cast<u64*>(w.d_tiles.p);
        u32* d_ticket = reinterpret_cast<u32*>(d_status + ntiles);
        G2P_CUDA(cudaMemsetAsync(d_status, 0, ((size_t)ntiles + 1) * sizeof(u64), st));
        k_index1<<<ntiles, kIdxThreads, 0, st>>>(d_text, n, ntiles, d_status, d_ticket, static_cast<u32*>(w.d_rec.p), (u32)cap64, d_meta);
        ++*launches;
        G2P_CUDA(meta_to_host(w.h_meta.p, d_meta, st)); ++*launches;
        G2P_CUDA(cudaStreamSynchronize(st));
        G2P_CUDA(cudaGetLastError());
        if ((u64)hm->n_records + 2 <= cap64) return G2P_OK;
        // more lines than the capacity guess: count first
    }
    u32* d_tiles = static_cast<u32*>(w.d_tiles.p);
    if (ntiles) { k_count_lines<<<ntiles, kIdxThreads, 0, st>>>(d_text, n, d_tiles); ++*launches; }
    k_scan_tiles<<<1, 1024, 0, st>>>(d_tiles, ntiles, d_text, n, d_meta);
    ++*launches;
    G2P_CUDA(meta_to_host(w.h_meta.p, d_meta, st)); ++*launches;
    G2P_CUDA(cudaStreamSynchronize(st));
    G2P_CUDA(w.d_rec.ensure(((size_t)hm->n_records + 2) * sizeof(u32)));
    if (ntiles) {
        k_fill_lines<<<ntiles, kIdxThreads, 0, st>>>(d_text, n, d_tiles, static_cast<u32*>(w.d_rec.p), d_meta);
        ++*launches;
    }
    G2P_CUDA(cudaGetLastError());
    return G2P_OK;
}

int g2p_index_lines(g2p_ctx* ctx, const void* d_text, size_t n, const uint32_t** d_starts, uint64_t* n_lines, void* stream) {
    if (!ctx || !d_starts || !n_lines) return G2P_E_ARG;
    if (n >= 0xFFFFFFF0ULL) return G2P_E_TOOBIG;
    G2P_CUDA(cudaSetDevice(ctx->device));
    Worker& w = ctx->w[0];
    cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : w.stream;
    uint32_t launches = 0;
    int rc = run_index(ctx, w, static_cast<const u8*>(d_text), n, st, &launches);
    if (rc) return rc;
    G2P_CUDA(cudaStreamSynchronize(st));
    *d_starts = static_cast<const uint32_t*>(w.d_rec.p);
    *n_lines = static_cast<const PipelineMeta*>(w.h_meta.p)->n_records;
    return G2P_OK;
}

// The one-pass path: k_fuse converts the whole block if every record is a canonical short record.  *done is set
// when the result is complete; otherwise (some record needs k_long / the general kernel, or fails) nothing of
// it is used and the caller runs the general pipeline.  The output buffer is sized by a bound (3x the input, or
// what earlier calls needed) and grown + the kernel run again when the exact size, which k_fuse always reports,
// exceeds it.
static void launch_fuse(int cfg, u32 ntiles, cudaStream_t st, const FuseArgs& fa) {
    switch (cfg) {
        case 0: k_fuse<FuseCfg0><<<ntiles, kFThreads, FuseCfg0::kSmem, st>>>(fa); break;
        case 1: k_fuse<FuseCfg1><<<ntiles, kFThreads, FuseCfg1::kSmem, st>>>(fa); break;
        case 2: k_fuse<FuseCfg2><<<ntiles, kFThreads, FuseCfg2::kSmem, st>>>(fa); break;
        case 3: k_fuse<FuseCfg3><<<ntiles, kFThreads, FuseCfg3::kSmem, st>>>(fa); break;
        case 4: k_fuse<FuseCfg4><<<ntiles, kFThreads, FuseCfg4::kSmem, st>>>(fa); break;
        case 5: k_fuse<FuseCfg5><<<ntiles, kFThreads, FuseCfg5::kSmem, st>>>(fa); break;
        case 6: k_fuse<FuseCfg6><<<ntiles, kFThreads, FuseCfg6::kSmem, st>>>(fa); break;
        case 7: k_fuse<FuseCfg7><<<ntiles, kFThreads, FuseCfg7::kSmem, st>>>(fa); break;
        default: k_fuse<FuseCfg8><<<ntiles, kFThreads, FuseCfg8::kSmem, st>>>(fa); break;
    }
}

static int run_fused(g2p_ctx* ctx, Worker& w, const u8* d_gaf, size_t n, cudaStream_t st, g2p_result* res, u8** d_out, bool* done, bool* not_convertible) {
    *done = false;
    *not_convertible = false;
    if (n == 0) return G2P_OK;
    const FuseMeta* hm = static_cast<const FuseMeta*>(w.h_fmeta.p);
    if (w.d_out.cap == 0 || ctx->fuse_out_cap_override) G2P_CUDA(w.d_out.ensure(ctx->fuse_out_cap_override ? (size_t)ctx->fuse_out_cap_override : n * 3 + (1u << 20)));
    G2P_CUDA(cudaEventRecord(w.ev[5], st));
    bool grown = false;
    for (;;) {
        const int cfg = ctx->fuse_cfg;
        const u32 tile = fuse_cfg_tile(cfg);
        const u32 ntiles = (u32)((n + tile - 1) / tile);
        const size_t fbytes = sizeof(FuseMeta) + 16 + (size_t)ntiles * sizeof(u64);
        G2P_CUDA(w.d_fuse.ensure(fbytes));
        u8* fb = static_cast<u8*>(w.d_fuse.p);
        FuseMeta* d_fm = reinterpret_cast<FuseMeta*>(fb);
        G2P_CUDA(cudaMemsetAsync(fb, 0, fbytes, st));
        FuseArgs fa{d_gaf, (u64)n, ntiles, ctx->table, static_cast<u8*>(w.d_out.p), (u64)(ctx->fuse_out_cap_override && !grown ? ctx->fuse_out_cap_override : w.d_out.cap),
                    reinterpret_cast<u64*>(fb + sizeof(FuseMeta) + 16), reinterpret_cast<u32*>(fb + sizeof(FuseMeta)), d_fm};
        launch_fuse(cfg, ntiles, st, fa);
        k_words_to_host<<<1, 32, 0, st>>>(reinterpret_cast<const uint32_t*>(d_fm), static_cast<uint32_t*>(w.h_fmeta.p), sizeof(FuseMeta) / 4);
        res->gpu_launches += 2;
        G2P_CUDA(cudaEventRecord(w.ev[6], st));
        G2P_CUDA(cudaStreamSynchronize(st));
        G2P_CUDA(cudaGetLastError());
        if (hm->fallback) {
            // only capacity reasons (records or path steps per tile): a smaller tile converts the same input
            if (!(hm->fallback & kFuseNotConvertible) && fuse_cfg_denser(cfg) >= 0) { ctx->fuse_cfg = fuse_cfg_denser(cfg); continue; }
            *not_convertible = (hm->fallback & kFuseNotConvertible) != 0;
            if (hm->fallback & (kFuseTimeoutLoad | kFuseTimeoutLookback))
                std::fprintf(stderr, "libg2p: k_fuse gave up a spin wait (flags 0x%x); the general pipeline converts this block\n", hm->fallback);
            cudaEventElapsedTime(&res->fused_ms, w.ev[5], w.ev[6]);   // (time spent on the attempt; n_fused stays 0)
            return G2P_OK;
        }
        if (!hm->overflow) {
            res->n_records = hm->n_records;
            res->out_bytes = hm->out_total;
            res->n_fused = hm->n_records;
            cudaEventElapsedTime(&res->fused_ms, w.ev[5], w.ev[6]);
            res->device_ms += res->fused_ms;
            *d_out = static_cast<u8*>(w.d_out.p);
            *done = true;
            return G2P_OK;
        }
        if (grown) return G2P_OK;   // (not reached with a consistent out_total; the general pipeline takes over)
        G2P_CUDA(w.d_out.ensure(hm->out_total + 256));   // the exact size is known now
        grown = true;
    }
}

// The device pipeline on one worker: index, size pass, scan, emit pass.  Returns with the stream
// synchronised; *d_out is the worker's output buffer.
// three 64-bit device words -> pinned host memory (same reason as k_meta_to_host)
__global__ void k_par_counts_to_host(const u64* a, const u64* b, const u64* c, u64* dst) {
    volatile u64* d = dst;
    if (threadIdx.x == 0) { d[0] = a ? *a : 0; d[1] = b ? *b : 0; d[2] = c ? *c : 0; }
    __threadfence_system();
}

// The token-parallel kernels (g2p_par.cuh) on the `nlist` records k_rec left: sizes, status and line descriptors
// for the canonical ones, the rest listed in w.d_list3 / meta->n_reject for k_long.  *done = false: nothing was
// converted (no room for the descriptors, or nothing to do) and k_long takes the whole list.
static int run_par(g2p_ctx* ctx, Worker& w, const u8* d_gaf, size_t n, cudaStream_t st, u32 nlist, LongArgs& la, PipelineMeta* d_meta, u32* launches, bool* done) {
    *done = false;
    auto scan64 = [&](u64* x, u32 cnt) {
        const u32 nb = (cnt + kScanTile - 1) / kScanTile;
        k_scan_reduce<<<nb, kScanThreads, 0, st>>>(x, cnt, static_cast<u64*>(w.p_bs.p));
        k_scan_blocks<<<1, 1024, 0, st>>>(static_cast<u64*>(w.p_bs.p), nb, x + cnt);
        k_scan_apply<<<nb, kScanThreads, 0, st>>>(x, cnt, static_cast<u64*>(w.p_bs.p), x + cnt);
        *launches += 3;
    };
    auto scan4 = [&](uint4* x, u32 cnt) {
        const u32 nb = (cnt + kScanTile - 1) / kScanTile;
        k_scan4_reduce<<<nb, kScanThreads, 0, st>>>(x, cnt, static_cast<uint4*>(w.p_bs.p));
        k_scan4_blocks<<<1, 1024, 0, st>>>(static_cast<uint4*>(w.p_bs.p), nb, x + cnt);
        k_scan4_apply<<<nb, kScanThreads, 0, st>>>(x, cnt, static_cast<uint4*>(w.p_bs.p));
        *launches += 3;
    };
    G2P_CUDA(w.p_recs.ensure((size_t)nlist * sizeof(ParRec)));
    G2P_CUDA(w.p_tb.ensure(((size_t)nlist + 1) * 2 * sizeof(u64)));
    G2P_CUDA(w.p_bs.ensure(((size_t)nlist / kScanTile + 2) * sizeof(uint4)));
    G2P_CUDA(w.d_list3.ensure((size_t)nlist * sizeof(u32)));
    ParArgs pa;
    std::memset(&pa, 0, sizeof pa);
    pa.gaf = d_gaf; pa.n = (u64)n; pa.rec_start = la.rec_start; pa.T = la.T; pa.list = la.list; pa.nlist = nlist;
    pa.recs = static_cast<ParRec*>(w.p_recs.p);
    pa.tile_base = static_cast<u64*>(w.p_tb.p); pa.slot_scan = pa.tile_base + nlist + 1;
    pa.out_off = la.out_off; pa.status = la.status; pa.rdesc = la.rdesc; pa.desc = la.desc;
    pa.reject_list = static_cast<u32*>(w.d_list3.p); pa.n_reject = &d_meta->n_reject; pa.n_desc = la.n_desc; pa.n_desc2 = la.n_desc2;
    pa.small_max = ctx->long_small_max ? ctx->long_small_max : 0u;
    const u32 grec = (nlist + 255) / 256;
    volatile u64* hp = static_cast<volatile u64*>(w.h_par.p);
    k_par_plan<<<grec, 256, 0, st>>>(pa); ++*launches;
    scan64(pa.tile_base, nlist);
    k_par_counts_to_host<<<1, 32, 0, st>>>(pa.tile_base + nlist, nullptr, nullptr, static_cast<u64*>(w.h_par.p)); ++*launches;
    G2P_CUDA(cudaStreamSynchronize(st));
    const u64 ntiles = hp[0];
    if (ntiles == 0 || ntiles > 0x7FFFFF00ULL) return G2P_OK;
    pa.ntiles = (u32)ntiles;
    G2P_CUDA(w.p_toff.ensure(((size_t)ntiles + 1) * (sizeof(uint4) + sizeof(u64) + sizeof(uint2))));
    G2P_CUDA(w.p_bs.ensure(((size_t)ntiles / kScanTile + 2) * sizeof(uint4)));
    pa.tile_osum = static_cast<uint4*>(w.p_toff.p);
    pa.tile_off = reinterpret_cast<u64*>(pa.tile_osum + ntiles + 1);
    pa.tile_map = reinterpret_cast<uint2*>(pa.tile_off + ntiles + 1);
    k_par_tilemap<<<grec, 256, 0, st>>>(pa); ++*launches;
    k_par_tabs<<<pa.ntiles, kPThreads, 0, st>>>(pa);
    k_par_head<<<(nlist + 127) / 128, 128, 0, st>>>(pa);
    k_par_count<<<pa.ntiles, kPThreads, 0, st>>>(pa);
    *launches += 3;
    scan64(pa.tile_off, pa.ntiles);
    scan4(pa.tile_osum, pa.ntiles);
    k_par_ranges<<<grec, 256, 0, st>>>(pa); ++*launches;
    scan64(pa.slot_scan, nlist);
    k_par_counts_to_host<<<1, 32, 0, st>>>(pa.tile_off + pa.ntiles, pa.slot_scan + nlist, nullptr, static_cast<u64*>(w.h_par.p)); ++*launches;
    G2P_CUDA(cudaStreamSynchronize(st));
    pa.nsteps = (u32)hp[0]; pa.nops = (u32)(hp[0] >> 32);
    const u64 big = (u32)hp[1], small = hp[1] >> 32;
    if (pa.nsteps == 0 || pa.nops == 0) return G2P_OK;
    // room for the records' descriptor runs in both halves of the array (k_long's blocks follow them), at most 12 bytes of descriptors per input byte
    const u64 need = 2 * std::max<u64>(std::max<u64>(big, small) + 2048, la.desc_cap / 2u);
    if (need > la.desc_cap) {
        if (ctx->desc_cap_override || need > 3 * (u64)n / 16 + 8192 || need > 0xFFFFFF00ULL) return G2P_OK;
        G2P_CUDA(w.d_desc.ensure((size_t)need * sizeof(LineDesc)));
        la.desc = static_cast<LineDesc*>(w.d_desc.p);
        la.desc_cap = (u32)need;
        pa.desc = la.desc;
    }
    pa.half = la.desc_cap / 2u;
    // per step: sval (16), sx, lx (8 + 8), spos, srec (4 + 4); per op: ox (16), opos, ot (4 + 4)
    const size_t ns1 = (size_t)pa.nsteps + 1, no1 = (size_t)pa.nops + 1;
    G2P_CUDA(w.p_step.ensure(ns1 * 40 + 64));
    G2P_CUDA(w.p_op.ensure(no1 * 24 + 64));
    G2P_CUDA(w.p_bs.ensure((ns1 / kScanTile + 2) * sizeof(uint4)));
    {
        u8* b = static_cast<u8*>(w.p_step.p);
        pa.sval = reinterpret_cast<uint4*>(b); b += ns1 * 16;
        pa.sx = reinterpret_cast<u64*>(b); b += ns1 * 8;
        pa.lx = reinterpret_cast<u64*>(b); b += ns1 * 8;
        pa.spos = reinterpret_cast<u32*>(b); b += ns1 * 4;
        pa.srec = reinterpret_cast<u32*>(b);
        u8* c = static_cast<u8*>(w.p_op.p);
        pa.ox = reinterpret_cast<uint4*>(c); c += no1 * 16;
        pa.opos = reinterpret_cast<u32*>(c); c += no1 * 4;
        pa.ot = reinterpret_cast<u32*>(c);
    }
    const u32 gmax = (u32)ctx->n_sm * 16u;
    const u32 gstep = std::min<u32>((pa.nsteps + 127) / 128, gmax);
    k_par_slots<<<grec, 256, 0, st>>>(pa);
    k_par_fill<<<pa.ntiles, kPThreads, 0, st>>>(pa);
    k_par_steps<<<gstep, 128, 0, st>>>(pa);
    *launches += 3;
    scan64(pa.sx, pa.nsteps);
    k_par_totals<<<grec, 256, 0, st>>>(pa);
    k_par_lines<<<gstep, 128, 0, st>>>(pa);
    *launches += 2;
    scan64(pa.lx, pa.nsteps);
    k_par_finish<<<grec, 256, 0, st>>>(pa);
    k_par_place<<<gstep, 128, 0, st>>>(pa);
    *launches += 2;
    G2P_CUDA(cudaGetLastError());
    la.list = pa.reject_list;
    la.n_list = &d_meta->n_reject;
    *done = true;
    return G2P_OK;
}

static int run_pipeline(g2p_ctx* ctx, Worker& w, const u8* d_gaf, size_t n, cudaStream_t st, g2p_result* res, u8** d_out) {
    std::memset(res, 0, sizeof *res);
    *d_out = nullptr;
    bool fuse_tried = false, fuse_nc = false;
    if (ctx->fuse_mode == 2) {   // always: before anything else
        bool done = false;
        int frc = run_fused(ctx, w, d_gaf, n, st, res, d_out, &done, &fuse_nc);
        if (frc || done) return frc;
        fuse_tried = true;
    }
    uint32_t launches = res->gpu_launches;
    G2P_CUDA(cudaEventRecord(w.ev[0], st));
    int rc = run_index(ctx, w, d_gaf, n, st, &launches);
    if (rc) return rc;
    G2P_CUDA(cudaEventRecord(w.ev[1], st));
    PipelineMeta* hm = static_cast<PipelineMeta*>(w.h_meta.p);
    PipelineMeta* d_meta = static_cast<PipelineMeta*>(w.d_meta.p);
    const u32 nrec = hm->n_records;
    res->n_records = nrec;
    // when it pays (see g2p_ctx::fuse_mode); a mean above k_fuse's record limit says it cannot take the block at all
    if (ctx->fuse_mode == 1 && nrec && (u64)n / nrec <= kFLimit && ((u64)n / nrec > 200 || ctx->prefer_fuse.load())) {
        res->gpu_launches = launches;
        bool done = false;
        int frc = run_fused(ctx, w, d_gaf, n, st, res, d_out, &done, &fuse_nc);
        if (frc) return frc;
        if (done) {
            cudaEventElapsedTime(&res->index_ms, w.ev[0], w.ev[1]);
            res->device_ms += res->index_ms;
            return G2P_OK;
        }
        launches = res->gpu_launches;
        fuse_tried = true;
        if (fuse_nc) ctx->prefer_fuse.store(0);
    }
    if (nrec == 0) {
        G2P_CUDA(w.d_out.ensure(256));
        *d_out = static_cast<u8*>(w.d_out.p);
        G2P_CUDA(cudaStreamSynchronize(st));
        res->gpu_launches = launches;
        return G2P_OK;
    }
    G2P_CUDA(w.d_status.ensure((size_t)nrec * sizeof(u32)));
    G2P_CUDA(w.d_off.ensure(((size_t)nrec + 1) * sizeof(u64)));
    const u32 nscan = (nrec + kScanTile - 1) / kScanTile;
    G2P_CUDA(w.d_blocks.ensure((size_t)nscan * 2 * sizeof(u64)));
    G2P_CUDA(w.d_list.ensure((size_t)nrec * sizeof(u32)));
    G2P_CUDA(w.d_list2.ensure((size_t)nrec * sizeof(u32)));
    u32* d_rec = static_cast<u32*>(w.d_rec.p);
    u32* d_status = static_cast<u32*>(w.d_status.p);
    u64* d_off = static_cast<u64*>(w.d_off.p);
    u64* d_blocks = static_cast<u64*>(w.d_blocks.p);
    u32* d_list = static_cast<u32*>(w.d_list.p);
    u32* d_list2 = static_cast<u32*>(w.d_list2.p);
    const u32 ncta = (nrec + kShortRecsPerCta - 1) / kShortRecsPerCta;
    const u32 nlong = (u32)ctx->n_sm * 6u;
    const u32 nlist = std::min<u32>((nrec + kListThreads - 1) / kListThreads, (u32)ctx->n_sm * 16u);
    // line descriptors: k_short's records own kSMaxLines slots each (sparse, addressed through the
    // line map); k_long reserves one block per batch in a dense array, as many slots as the batch has lines
    // (~1 line per 40 bytes of text), and falls back to its streaming emit when that array is full
    const u64 desc_cap64 = std::min<u64>((u64)n / 8 + 2048, 0xFFFFFF00ULL);   // two halves: full batches / small batches
    const u32 desc_cap = ctx->desc_cap_override ? (u32)std::min<u64>(ctx->desc_cap_override, desc_cap64) : (u32)desc_cap64;
    G2P_CUDA(w.d_desc.ensure((size_t)desc_cap * sizeof(LineDesc)));
    G2P_CUDA(w.d_sdesc.ensure((size_t)nrec * kSMaxLines * sizeof(LineDesc)));
    G2P_CUDA(w.d_rdesc.ensure((size_t)nrec * sizeof(RecDesc)));
    G2P_CUDA(w.d_loff.ensure(((size_t)nrec + 1) * sizeof(u64)));
    LineDesc* d_desc = static_cast<LineDesc*>(w.d_desc.p);
    LineDesc* d_sdesc = static_cast<LineDesc*>(w.d_sdesc.p);
    RecDesc* d_rdesc = static_cast<RecDesc*>(w.d_rdesc.p);
    u64* d_loff = static_cast<u64*>(w.d_loff.p);
    ShortArgs sa{d_gaf, (u64)n, d_rec, nrec, ctx->table, d_off, d_loff, d_status, d_list, &d_meta->n_deleg, d_sdesc, d_rdesc};
    LongArgs la{d_gaf, (u64)n, d_rec, ctx->table, d_off, d_status, nullptr, d_list, &d_meta->n_deleg, d_list2, &d_meta->n_deleg2,
                d_desc, d_rdesc, &d_meta->n_desc, &d_meta->n_desc2, desc_cap, ctx->long_small_max, &d_meta->legacy_long, &d_meta->long_cursor};

    // pass 1: sizes, status, line descriptors.  k_short takes the short canonical records, k_long
    // what it left, the general kernel what neither converts (non-canonical or erroneous records).
    if (ctx->size_kernel_short) k_short<kSG><<<ncta, kSThreads, kShortSmem, st>>>(sa);
    else {
        const u32 chunks = ctx->rec_chunks_override ? ctx->rec_chunks_override : rec_chunks_for((u64)n, nrec);
        const u32* d_perm = nullptr;
        if (ctx->len_sort && nrec > kRThreads) {   // order the records by length class: counting sort with the u64 scan kernels
            const u32 nsort = (nrec + kLenSortRecs - 1) / kLenSortRecs, nm = kLenBins * nsort;
            const u32 nscan_m = (nm + kScanTile - 1) / kScanTile;
            G2P_CUDA(w.d_lsort.ensure(((size_t)nm + 1 + nscan_m) * sizeof(u64)));
            G2P_CUDA(w.d_perm.ensure((size_t)nrec * sizeof(u32)));
            u64* d_m = static_cast<u64*>(w.d_lsort.p);
            u64* d_mb = d_m + nm + 1;
            k_len_hist<<<nsort, 256, 0, st>>>(d_rec, nrec, nsort, d_m);
            k_scan_reduce<<<nscan_m, kScanThreads, 0, st>>>(d_m, nm, d_mb);
            k_scan_blocks<<<1, 1024, 0, st>>>(d_mb, nscan_m, d_m + nm);
            k_scan_apply<<<nscan_m, kScanThreads, 0, st>>>(d_m, nm, d_mb, d_m + nm);
            k_len_scatter<<<nsort, 256, 0, st>>>(d_rec, nrec, nsort, d_m, static_cast<u32*>(w.d_perm.p));
            launches += 5;
            d_perm = static_cast<const u32*>(w.d_perm.p);
        }
        RecArgs ra{sa, chunks, d_perm};
        k_rec<<<(nrec + kRThreads - 1) / kRThreads, kRThreads, rec_smem(chunks), st>>>(ra);
    }
    ++launches;
    u32 desc_cap_now = desc_cap;
    bool par_done = false;
    if (ctx->par && !ctx->size_kernel_short) {
        // how many records did k_rec leave?  (one small read-back; the stream is synchronised again before the emit pass anyway)
        k_words_to_host<<<1, 32, 0, st>>>(&d_meta->n_deleg, &hm->n_deleg, 1); ++launches;
        G2P_CUDA(cudaStreamSynchronize(st));
        const u32 n_left = hm->n_deleg;
        if (n_left) {
            G2P_CUDA(cudaEventRecord(w.ev[8], st));
            rc = run_par(ctx, w, d_gaf, n, st, n_left, la, d_meta, &launches, &par_done);
            if (rc) return rc;
            G2P_CUDA(cudaEventRecord(w.ev[9], st));
            d_desc = la.desc;
            desc_cap_now = la.desc_cap;
        }
        if (n_left) {
            k_long<false><<<nlong, kLThreads, long_smem<false>(), st>>>(la);
            k_convert_list<false><<<nlist, kListThreads, 0, st>>>(d_gaf, d_rec, ctx->table, d_off, d_status, nullptr, d_meta, d_list2, &d_meta->n_deleg2);
            launches += 2;
        }
    } else {
        k_long<false><<<nlong, kLThreads, long_smem<false>(), st>>>(la);
        k_convert_list<false><<<nlist, kListThreads, 0, st>>>(d_gaf, d_rec, ctx->table, d_off, d_status, nullptr, d_meta, d_list2, &d_meta->n_deleg2);
        launches += 2;
    }
    G2P_CUDA(cudaEventRecord(w.ev[2], st));
    // exclusive scans: byte counts -> output offsets, line counts -> line slots (+ the line map)
    G2P_CUDA(w.d_map.ensure((size_t)nrec * kSMaxLines * sizeof(LineMapEnt)));
    LineMapEnt* d_map = static_cast<LineMapEnt*>(w.d_map.p);
    k_scan_reduce2<<<nscan, kScanThreads, 0, st>>>(d_off, d_loff, nrec, d_blocks, d_blocks + nscan);
    k_scan_blocks2<<<1, 1024, 0, st>>>(d_blocks, d_blocks + nscan, nscan, &d_meta->out_total, &d_meta->lines_total);
    k_scan_apply2<<<nscan, kScanThreads, 0, st>>>(d_off, d_loff, nrec, d_blocks, d_blocks + nscan, &d_meta->out_total, &d_meta->lines_total, d_rec, d_map);
    launches += 3;
    G2P_CUDA(meta_to_host(w.h_meta.p, d_meta, st)); ++launches;
    G2P_CUDA(cudaStreamSynchronize(st));
    const u64 out_total = hm->out_total;
    res->n_long = hm->n_deleg;
    res->n_delegated = hm->n_deleg2;
    res->n_par = par_done ? hm->n_deleg - hm->n_reject : 0u;
    if (par_done) cudaEventElapsedTime(&res->par_ms, w.ev[8], w.ev[9]);
    G2P_CUDA(w.d_out.ensure(out_total + 256));
    u8* d_o = static_cast<u8*>(w.d_out.p);
    // pass 2: emit
    G2P_CUDA(cudaEventRecord(w.ev[3], st));
    la.out = d_o;
    if (hm->lines_total) {   // k_short's records: line slot -> descriptor through the map
        if (hm->lines_total > 0xFFFFFF00ULL) { ctx->set_err("too many PAF lines in one call: split the input"); return G2P_E_TOOBIG; }
        const u32 nl = (u32)hm->lines_total;
        EmitArgs ea{d_gaf, (u64)n, d_rec, d_off, d_sdesc, d_map, d_rdesc, d_status, nl, d_o};
        k_emit_lines<false><<<(nl + kEThreads - 1) / kEThreads, kEThreads, kEmitSmem, st>>>(ea);
        ++launches;
    }
    const u32 half = desc_cap_now / 2u;
    const u32 n_slots = std::min<u32>(hm->n_desc, half);
    if (n_slots) {           // k_par's / k_long's records, full batches: dense 32-slot blocks
        EmitArgs ea{d_gaf, (u64)n, d_rec, d_off, d_desc, nullptr, d_rdesc, d_status, n_slots, d_o};
        k_emit_lines<true><<<(n_slots + kEThreads - 1) / kEThreads, kEThreads, kEmitSmem, st>>>(ea);
        ++launches;
    }
    const u32 n_slots2 = std::min<u32>(hm->n_desc2, desc_cap_now - half);
    if (n_slots2) {          // ... and their small batches
        EmitArgs ea{d_gaf, (u64)n, d_rec, d_off, d_desc + half, nullptr, d_rdesc, d_status, n_slots2, d_o};
        k_emit_lines<true><<<(n_slots2 + kEThreads - 1) / kEThreads, kEThreads, kEmitSmem, st>>>(ea);
        ++launches;
    }
    if (hm->legacy_long) {   // records k_long could not describe (descriptor array full)
        k_long<true><<<nlong, kLThreads, long_smem<true>(), st>>>(la);
        ++launches;
    }
    if (hm->n_deleg2) {
        k_convert_list<true><<<nlist, kListThreads, 0, st>>>(d_gaf, d_rec, ctx->table, d_off, d_status, d_o, d_meta, d_list2, &d_meta->n_deleg2);
        ++launches;
    }
    G2P_CUDA(cudaEventRecord(w.ev[4], st));
    res->out_bytes = out_total;
    if (hm->first_err != 0xFFFFFFFFu) {
        k_diagnose<<<1, 1, 0, st>>>(d_gaf, d_rec, ctx->table, d_off, d_meta);
        ++launches;
        G2P_CUDA(meta_to_host(w.h_meta.p, d_meta, st)); ++launches;
    }
    G2P_CUDA(cudaStreamSynchronize(st));
    G2P_CUDA(cudaGetLastError());
    if (hm->first_err != 0xFFFFFFFFu) {
        res->rec_status = hm->err_status & 0xff;
        res->rec_aux = (hm->err_status >> 8) & 0xff;
        res->err_record = hm->first_err;
        res->err_name_off = (u64)hm->err_rec_start + hm->err_a;
        res->err_name_len = hm->err_b - hm->err_a;
        res->out_bytes = hm->err_out_end;   // what the reference has written before it stops
    }
    cudaEventElapsedTime(&res->index_ms, w.ev[0], w.ev[1]);
    cudaEventElapsedTime(&res->size_ms, w.ev[1], w.ev[2]);
    cudaEventElapsedTime(&res->emit_ms, w.ev[3], w.ev[4]);
    cudaEventElapsedTime(&res->device_ms, fuse_tried ? w.ev[5] : w.ev[0], w.ev[4]);
    if (fuse_tried && ctx->fuse_mode == 1) cudaEventElapsedTime(&res->device_ms, w.ev[0], w.ev[4]);   // (the attempt came after the index)
    res->gpu_launches = launches;
    // many records needed k_long and nothing says k_fuse cannot take them: try it first next time
    if (ctx->fuse_mode == 1 && !fuse_nc) ctx->prefer_fuse.store((u64)res->n_long * 32u > nrec ? 1 : 0);
    *d_out = d_o;
    return G2P_OK;
}

int g2p_convert_device(g2p_ctx* ctx, const void* d_gaf_v, size_t n, void** d_out, g2p_result* res, void* stream) {
    if (!ctx || !res || !d_out) return G2P_E_ARG;
    if (!ctx->have_table) return G2P_E_NOTABLE;
    if (n >= 0xFFFFFFF0ULL) return G2P_E_TOOBIG;
    if ((reinterpret_cast<uintptr_t>(d_gaf_v) & 15) != 0) { ctx->set_err("d_gaf must be 16-byte aligned"); return G2P_E_ARG; }
    G2P_CUDA(cudaSetDevice(ctx->device));
    Worker& w = ctx->w[0];
    cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : w.stream;
    u8* d_o = nullptr;
    int rc = run_pipeline(ctx, w, static_cast<const u8*>(d_gaf_v), n, st, res, &d_o);
    *d_out = d_o;
    return rc;
}

// Host-buffer entry point.  The input is cut into newline-aligned chunks; kWorkers host threads
// each drive one chunk at a time through its own stream (H2D, pipeline, D2H), so the copies of
// one chunk overlap the kernels of another.  Output bytes land in one pinned buffer in input
// order; everything after the first failing record is dropped, like the reference's exit.
int g2p_convert_host(g2p_ctx* ctx, const char* gaf, size_t n, const char** out, g2p_result* res) {
    if (!ctx || !res || !out || (!gaf && n)) return G2P_E_ARG;
    if (!ctx->have_table) return G2P_E_NOTABLE;
    if (n >= 0xFFFFFFF0ULL) return G2P_E_TOOBIG;
    *out = nullptr;
    std::memset(res, 0, sizeof *res);
    G2P_CUDA(cudaSetDevice(ctx->device));
    if (ctx->have_cpus) sched_setaffinity(0, sizeof ctx->cpus, &ctx->cpus);   // the worker threads inherit the mask
    PinBuf& h_out = ctx->next_out();

    // newline-aligned chunk boundaries.  Chunks must hold enough records to fill the GPU: short
    // reads do at 48 MB, chromosome-scale records (one warp each in k_long) need more.
    size_t chunk = ctx->host_chunk;
    if (!ctx->host_chunk_fixed && n > chunk) {
        const size_t probe = std::min<size_t>(n, 4u << 20);
        size_t nl = 1;
        for (const char* q = gaf; (q = static_cast<const char*>(std::memchr(q, '\n', gaf + probe - q))) != nullptr; ++q) ++nl;
        const size_t avg = probe / nl;
        chunk = std::min<size_t>(std::max<size_t>(chunk, avg * 4096), 768u << 20);
    }
    std::vector<size_t> cut{0};
    while (cut.back() < n) {
        // the first chunks are smaller (1/3, 2/3 of a chunk): the output copy, which bounds the call
        // (PCIe D2H), starts after the first chunk's H2D + kernels
        const size_t k = cut.size();
        size_t e = cut.back() + (ctx->host_chunk_fixed || k > 2 ? chunk : chunk * k / 3);
        if (e >= n) e = n;
        else {
            const void* nl = std::memchr(gaf + e - 1, '\n', n - (e - 1));
            e = nl ? (size_t)(static_cast<const char*>(nl) - gaf) + 1 : n;
        }
        cut.push_back(e);
    }
    const size_t nchunks = cut.size() - 1;
    if (nchunks == 0) {
        G2P_CUDA(h_out.ensure(1));
        *out = static_cast<const char*>(h_out.p);
        return G2P_OK;
    }

    struct Shared {
        std::mutex mu;
        std::condition_variable cv;
        size_t published = 0;        // chunks whose output offset is known (prefix valid up to here)
        size_t copied = 0;           // chunks (in order) whose D2H has completed
        std::vector<u64> off;        // output offset of chunk i
        std::vector<u64> recs;       // records before chunk i
        size_t stop_at;              // first chunk with an error (chunks after it are ignored)
        int rc = G2P_OK;
    } S;
    S.off.assign(nchunks + 1, 0);
    S.recs.assign(nchunks + 1, 0);
    S.stop_at = nchunks;
    std::vector<g2p_result> cres(nchunks);
    std::vector<char> done(nchunks, 0);
    // first guess of the output size: keep what earlier calls needed, else 3x the input
    if (h_out.cap == 0) G2P_CUDA(h_out.ensure(n * 3 + (1 << 20)));

    // G2P_TRACE=1: host-clock timeline of every chunk on stderr (ms since the call started)
    const bool trace = std::getenv("G2P_TRACE") != nullptr;
    const auto t_call = std::chrono::steady_clock::now();
    auto now_ms = [&] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_call).count(); };
    auto worker = [&](int wi) {
        cudaSetDevice(ctx->device);
        Worker& w = ctx->w[wi];
        for (size_t i = wi; i < nchunks; i += kWorkers) {
            {
                std::lock_guard<std::mutex> g(S.mu);
                if (i > S.stop_at || S.rc != G2P_OK) break;
            }
            const size_t a = cut[i], len = cut[i + 1] - cut[i];
            const double t_begin = trace ? now_ms() : 0.0;
            int rc = G2P_OK;
            u8* d_o = nullptr;
            g2p_result r;
            std::memset(&r, 0, sizeof r);
            if (w.d_in.ensure(len + 256) != cudaSuccess) rc = G2P_E_CUDA;
            if (rc == G2P_OK && cudaMemcpyAsync(w.d_in.p, gaf + a, len, cudaMemcpyHostToDevice, w.stream) != cudaSuccess) rc = G2P_E_CUDA;
            if (rc == G2P_OK) rc = run_pipeline(ctx, w, static_cast<const u8*>(w.d_in.p), len, w.stream, &r, &d_o);
            const double t_piped = trace ? now_ms() : 0.0;
            // publish this chunk's output offset (in chunk order)
            std::unique_lock<std::mutex> lk(S.mu);
            S.cv.wait(lk, [&] { return S.published == i || S.rc != G2P_OK || i > S.stop_at; });
            if (S.rc != G2P_OK || i > S.stop_at) break;   // an earlier chunk failed: this one is never reached
            if (rc != G2P_OK) { S.rc = rc; S.cv.notify_all(); break; }
            cres[i] = r;
            S.off[i + 1] = S.off[i] + r.out_bytes;
            S.recs[i + 1] = S.recs[i] + r.n_records;
            if (r.rec_status != G2P_REC_OK) S.stop_at = i;
            if (S.off[i + 1] + 1 > h_out.cap) {
                // grow the pinned output: wait for the copies of earlier chunks, then move what is there
                S.cv.wait(lk, [&] { return S.copied == i || S.rc != G2P_OK; });
                PinBuf nb;
                if (S.rc == G2P_OK && nb.ensure(S.off[i + 1] + (n - cut[i + 1]) * 4 + (1 << 20)) != cudaSuccess) { S.rc = G2P_E_CUDA; ctx->set_err("pinned output allocation failed"); }
                if (S.rc != G2P_OK) { S.cv.notify_all(); break; }
                std::memcpy(nb.p, h_out.p, S.off[i]);
                h_out.release();
                h_out = nb;
            }
            char* dst = static_cast<char*>(h_out.p) + S.off[i];
            S.published = i + 1;
            S.cv.notify_all();
            lk.unlock();
            const double t_pub = trace ? now_ms() : 0.0;
            cudaError_t ce = cudaSuccess;
            if (r.out_bytes) ce = cudaMemcpyAsync(dst, d_o, r.out_bytes, cudaMemcpyDeviceToHost, w.stream);
            if (ce == cudaSuccess) ce = cudaStreamSynchronize(w.stream);
            if (trace) std::fprintf(stderr, "g2p trace: chunk %zu worker %d in %zu out %llu: begin %.2f piped %.2f (device %.2f) published %.2f copied %.2f\n", i, wi, len,
                                    (unsigned long long)r.out_bytes, t_begin, t_piped, r.device_ms, t_pub, now_ms());
            lk.lock();
            if (ce != cudaSuccess) { S.rc = G2P_E_CUDA; ctx->set_err(std::string("D2H: ") + cudaGetErrorString(ce)); S.cv.notify_all(); break; }
            done[i] = 1;
            while (S.copied < nchunks && done[S.copied]) ++S.copied;
            S.cv.notify_all();
        }
    };
    if (nchunks == 1) worker(0);
    else {
        std::vector<std::thread> th;
        const int nw = (int)std::min<size_t>(kWorkers, nchunks);
        for (int wi = 1; wi < nw; ++wi) th.emplace_back(worker, wi);
        worker(0);
        for (auto& t : th) t.join();
    }
    if (S.rc != G2P_OK) return S.rc;
    // aggregate
    const size_t last = std::min(S.stop_at, nchunks - 1);
    for (size_t i = 0; i <= last; ++i) {
        const g2p_result& r = cres[i];
        res->n_records += r.n_records;
        res->gpu_launches += r.gpu_launches;
        res->device_ms += r.device_ms; res->emit_ms += r.emit_ms; res->size_ms += r.size_ms; res->index_ms += r.index_ms;
        res->fused_ms += r.fused_ms; res->n_fused += r.n_fused;
        res->n_delegated += r.n_delegated; res->n_long += r.n_long;
        res->par_ms += r.par_ms; res->n_par += r.n_par;
    }
    res->out_bytes = S.off[last + 1];
    if (S.stop_at < nchunks) {
        const g2p_result& r = cres[S.stop_at];
        res->rec_status = r.rec_status; res->rec_aux = r.rec_aux;
        res->err_record = S.recs[S.stop_at] + r.err_record;
        res->err_name_off = cut[S.stop_at] + r.err_name_off;
        res->err_name_len = r.err_name_len;
    }
    *out = static_cast<const char*>(h_out.p);
    return G2P_OK;
}

// ---------------------------------------------------------------------------------------
// gaf2unstable
// ---------------------------------------------------------------------------------------
int g2p_load_rgfa(g2p_ctx* ctx, const char* rgfa, size_t n, int* ref_exit_code, char* msg, size_t msg_cap) {
    if (!ctx || (!rgfa && n)) return G2P_E_ARG;
    if (ref_exit_code) *ref_exit_code = 0;
    if (msg && msg_cap) msg[0] = 0;
    G2P_CUDA(cudaSetDevice(ctx->device));
    delete ctx->rgfa;
    ctx->rgfa = new RgfaTables();
    RgfaTables& T = *ctx->rgfa;
    build_rgfa_tables(rgfa, n, T);
    if (T.exit_code) {
        if (ref_exit_code) *ref_exit_code = T.exit_code;
        if (msg && msg_cap) std::snprintf(msg, msg_cap, "%s", T.exit_code == 1 ? T.error.c_str() : "");
        ctx->set_err("rGFA: " + T.error);
        ctx->have_rgfa = false;
        return G2P_E_TABLE;
    }
    // flatten: contig hash -> index, nodes per contig sorted by SO, names, node -> reference contig
    HostLenTable ct;
    ct.reserve_for(T.mapping.size());
    std::vector<u32> begin;
    std::vector<UNode> nodes;
    std::vector<u8> names;
    ctx->node_lengths.clear();
    u32 ci = 0;
    for (const auto& cs : T.mapping) {
        ct.put(reinterpret_cast<const u8*>(cs.first.data()), (u32)cs.first.size(), (i64)ci++);
        begin.push_back((u32)nodes.size());
        i64 cum = 0;
        for (const RgfaNode& nd : cs.second) {
            UNode u;
            u.offset = nd.offset; u.cum = cum; u.length = (u32)nd.length;
            u.name_off = (u32)names.size(); u.name_len = (u32)nd.name.size();
            names.insert(names.end(), nd.name.begin(), nd.name.end());
            int64_t id;
            u.ref = -1;
            if (rgfa_detail::node_id_of(nd.name, id)) {
                auto it = T.node_to_contig.find(id);
                if (it != T.node_to_contig.end()) u.ref = (i32)it->second;
            }
            cum += nd.length;
            nodes.push_back(u);
            ctx->node_lengths += nd.name;
            ctx->node_lengths += '\t';
            ctx->node_lengths += std::to_string(nd.length);
            ctx->node_lengths += '\n';
        }
    }
    begin.push_back((u32)nodes.size());
    if (ct.arena.empty()) ct.arena.push_back(0);
    std::vector<u32> refoff{0};
    std::vector<u8> refnames;
    for (const std::string& c : T.ref_contigs) { refnames.insert(refnames.end(), c.begin(), c.end()); refoff.push_back((u32)refnames.size()); }
    if (names.empty()) names.push_back(0);
    if (refnames.empty()) refnames.push_back(0);
    if (nodes.empty()) nodes.push_back(UNode{0, 0, 0, 0, 0, -1});
    G2P_CUDA(cudaDeviceSynchronize());
    auto up = [&](DevBuf& b, const void* src, size_t bytes) -> cudaError_t {
        cudaError_t e = b.ensure(bytes ? bytes : 16);
        if (e != cudaSuccess) return e;
        return bytes ? cudaMemcpy(b.p, src, bytes, cudaMemcpyHostToDevice) : cudaSuccess;
    };
    G2P_CUDA(up(ctx->u_slots, ct.slots.data(), ct.slots.size() * sizeof(LenSlot)));
    G2P_CUDA(up(ctx->u_arena, ct.arena.data(), ct.arena.size()));
    G2P_CUDA(up(ctx->u_begin, begin.data(), begin.size() * sizeof(u32)));
    G2P_CUDA(up(ctx->u_nodes, nodes.data(), nodes.size() * sizeof(UNode)));
    G2P_CUDA(up(ctx->u_names, names.data(), names.size()));
    G2P_CUDA(up(ctx->u_refoff, refoff.data(), refoff.size() * sizeof(u32)));
    G2P_CUDA(up(ctx->u_refnames, refnames.data(), refnames.size()));
    ctx->uview.contigs.slots = static_cast<const LenSlot*>(ctx->u_slots.p);
    ctx->uview.contigs.arena = static_cast<const u8*>(ctx->u_arena.p);
    ctx->uview.contigs.nslots = (u32)ct.slots.size();
    ctx->uview.contig_begin = static_cast<const u32*>(ctx->u_begin.p);
    ctx->uview.nodes = static_cast<const UNode*>(ctx->u_nodes.p);
    ctx->uview.node_names = static_cast<const u8*>(ctx->u_names.p);
    ctx->uview.ref_off = static_cast<const u32*>(ctx->u_refoff.p);
    ctx->uview.ref_names = static_cast<const u8*>(ctx->u_refnames.p);
    {   // the node-lengths table of the fused gaf2unstable | gaf2paf path: exactly what `gaf2paf -l <the -o file>` would load
        HostLenTable nt;
        if (build_len_table(ctx->node_lengths.data(), ctx->node_lengths.size(), nt) != ST_OK) { ctx->set_err("node lengths table"); return G2P_E_TABLE; }
        G2P_CUDA(up(ctx->n_slots, nt.slots.data(), nt.slots.size() * sizeof(LenSlot)));
        G2P_CUDA(up(ctx->n_arena, nt.arena.data(), nt.arena.size()));
        ctx->node_table.slots = static_cast<const LenSlot*>(ctx->n_slots.p);
        ctx->node_table.arena = static_cast<const u8*>(ctx->n_arena.p);
        ctx->node_table.nslots = (u32)nt.slots.size();
    }
    ctx->have_rgfa = true;
    return G2P_OK;
}

int g2p_rgfa_node_lengths(g2p_ctx* ctx, const char** tsv, size_t* n) {
    if (!ctx || !tsv || !n) return G2P_E_ARG;
    if (!ctx->have_rgfa) return G2P_E_NOTABLE;
    *tsv = ctx->node_lengths.data();
    *n = ctx->node_lengths.size();
    return G2P_OK;
}

static int run_unstable(g2p_ctx* ctx, Worker& w, const u8* d_gaf, size_t n, cudaStream_t st, g2p_result* res, u8** d_out) {
    std::memset(res, 0, sizeof *res);
    *d_out = nullptr;
    ctx->warns.clear();
    uint32_t launches = 0;
    G2P_CUDA(cudaEventRecord(w.ev[0], st));
    int rc = run_index(ctx, w, d_gaf, n, st, &launches);
    if (rc) return rc;
    G2P_CUDA(cudaEventRecord(w.ev[1], st));
    PipelineMeta* hm = static_cast<PipelineMeta*>(w.h_meta.p);
    PipelineMeta* d_meta = static_cast<PipelineMeta*>(w.d_meta.p);
    const u32 nrec = hm->n_records;
    res->n_records = nrec;
    G2P_CUDA(w.d_out.ensure(256));
    *d_out = static_cast<u8*>(w.d_out.p);
    if (nrec == 0) { G2P_CUDA(cudaStreamSynchronize(st)); res->gpu_launches = launches; return G2P_OK; }
    G2P_CUDA(w.d_status.ensure((size_t)nrec * sizeof(u32)));
    G2P_CUDA(w.d_off.ensure(((size_t)nrec + 1) * sizeof(u64)));
    const u32 nscan = (nrec + kScanTile - 1) / kScanTile;
    G2P_CUDA(w.d_blocks.ensure((size_t)nscan * sizeof(u64)));
    G2P_CUDA(w.d_list.ensure((size_t)nrec * sizeof(u32)));
    u32* d_rec = static_cast<u32*>(w.d_rec.p);
    u32* d_status = static_cast<u32*>(w.d_status.p);
    u64* d_off = static_cast<u64*>(w.d_off.p);
    u64* d_blocks = static_cast<u64*>(w.d_blocks.p);
    u32* d_list = static_cast<u32*>(w.d_list.p);
    const u32 ncta = std::min<u32>((nrec + kListThreads - 1) / kListThreads, (u32)ctx->n_sm * 32u);
    const u32 ncta_s = (nrec + kUThreads - 1) / kUThreads;
    if (ctx->unstable_staged) k_unstable_staged<false><<<ncta_s, kUThreads, unstable_smem<false>(), st>>>(d_gaf, (u64)n, d_rec, nrec, ctx->uview, d_off, d_status, nullptr, d_meta, d_list);
    else k_unstable<false><<<ncta, kListThreads, 0, st>>>(d_gaf, d_rec, nrec, ctx->uview, d_off, d_status, nullptr, d_meta, d_list);
    ++launches;
    G2P_CUDA(cudaEventRecord(w.ev[2], st));
    k_scan_reduce<<<nscan, kScanThreads, 0, st>>>(d_off, nrec, d_blocks);
    k_scan_blocks<<<1, 1024, 0, st>>>(d_blocks, nscan, &d_meta->out_total);
    k_scan_apply<<<nscan, kScanThreads, 0, st>>>(d_off, nrec, d_blocks, &d_meta->out_total);
    launches += 3;
    G2P_CUDA(meta_to_host(w.h_meta.p, d_meta, st)); ++launches;
    G2P_CUDA(cudaStreamSynchronize(st));
    const u64 out_total = hm->out_total;
    G2P_CUDA(w.d_out.ensure(out_total + 256));
    u8* d_o = static_cast<u8*>(w.d_out.p);
    G2P_CUDA(cudaEventRecord(w.ev[3], st));
    if (ctx->unstable_staged) k_unstable_staged<true><<<ncta_s, kUThreads, unstable_smem<true>(), st>>>(d_gaf, (u64)n, d_rec, nrec, ctx->uview, d_off, d_status, d_o, d_meta, d_list);
    else k_unstable<true><<<ncta, kListThreads, 0, st>>>(d_gaf, d_rec, nrec, ctx->uview, d_off, d_status, d_o, d_meta, d_list);
    ++launches;
    G2P_CUDA(cudaEventRecord(w.ev[4], st));
    G2P_CUDA(cudaStreamSynchronize(st));
    G2P_CUDA(cudaGetLastError());
    res->out_bytes = out_total;
    const u32 first_err = hm->first_err;
    std::vector<u64> off;
    if (first_err != 0xFFFFFFFFu || hm->n_deleg) {
        off.resize((size_t)nrec + 1);
        G2P_CUDA(cudaMemcpy(off.data(), d_off, off.size() * sizeof(u64), cudaMemcpyDeviceToHost));
    }
    if (first_err != 0xFFFFFFFFu) {
        u32 stv = 0;
        G2P_CUDA(cudaMemcpy(&stv, d_status + first_err, sizeof(u32), cudaMemcpyDeviceToHost));
        res->rec_status = stv & 0xff;
        res->rec_aux = (stv >> 8) & 0xff;
        res->err_record = first_err;
        res->out_bytes = off[first_err];
    }
    if (hm->n_deleg) {
        std::vector<u32> wl(hm->n_deleg);
        G2P_CUDA(cudaMemcpy(wl.data(), d_list, wl.size() * sizeof(u32), cudaMemcpyDeviceToHost));
        std::sort(wl.begin(), wl.end());
        for (u32 r : wl) {
            if (first_err != 0xFFFFFFFFu && r >= first_err) break;
            ctx->warns.push_back(g2p_warn{r, off[r], off[r + 1] - off[r]});
        }
    }
    cudaEventElapsedTime(&res->index_ms, w.ev[0], w.ev[1]);
    cudaEventElapsedTime(&res->size_ms, w.ev[1], w.ev[2]);
    cudaEventElapsedTime(&res->emit_ms, w.ev[3], w.ev[4]);
    cudaEventElapsedTime(&res->device_ms, w.ev[0], w.ev[4]);
    res->gpu_launches = launches;
    *d_out = d_o;
    return G2P_OK;
}

int g2p_unstable_device(g2p_ctx* ctx, const void* d_gaf_v, size_t n, void** d_out, g2p_result* res, void* stream) {
    if (!ctx || !res || !d_out) return G2P_E_ARG;
    if (!ctx->have_rgfa) return G2P_E_NOTABLE;
    if (n >= 0xFFFFFFF0ULL) return G2P_E_TOOBIG;
    if ((reinterpret_cast<uintptr_t>(d_gaf_v) & 15) != 0) { ctx->set_err("d_gaf must be 16-byte aligned"); return G2P_E_ARG; }
    G2P_CUDA(cudaSetDevice(ctx->device));
    Worker& w = ctx->w[0];
    cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : w.stream;
    u8* d_o = nullptr;
    int rc = run_unstable(ctx, w, static_cast<const u8*>(d_gaf_v), n, st, res, &d_o);
    *d_out = d_o;
    return rc;
}

int g2p_unstable_host(g2p_ctx* ctx, const char* gaf, size_t n, const char** out, g2p_result* res) {
    if (!ctx || !res || !out || (!gaf && n)) return G2P_E_ARG;
    if (!ctx->have_rgfa) return G2P_E_NOTABLE;
    if (n >= 0xFFFFFFF0ULL) return G2P_E_TOOBIG;
    *out = nullptr;
    G2P_CUDA(cudaSetDevice(ctx->device));
    Worker& w = ctx->w[0];
    PinBuf& h_out = ctx->next_out();
    G2P_CUDA(w.d_in.ensure(n + 256));
    if (n) G2P_CUDA(cudaMemcpyAsync(w.d_in.p, gaf, n, cudaMemcpyHostToDevice, w.stream));
    u8* d_o = nullptr;
    int rc = run_unstable(ctx, w, static_cast<const u8*>(w.d_in.p), n, w.stream, res, &d_o);
    if (rc) return rc;
    G2P_CUDA(h_out.ensure(res->out_bytes + 1));
    if (res->out_bytes) G2P_CUDA(cudaMemcpyAsync(h_out.p, d_o, res->out_bytes, cudaMemcpyDeviceToHost, w.stream));
    G2P_CUDA(cudaStreamSynchronize(w.stream));
    *out = static_cast<const char*>(h_out.p);
    return G2P_OK;
}

// ---- N2: gaf2unstable | gaf2paf without the intermediate text leaving the device (README.md:55-58 pipeline) -------
// Stage 1 (k_unstable) writes the node-space GAF into a device buffer, stage 2 (the gaf2paf pipeline, with the node
// lengths of the same rGFA as its -l table) reads it from there: no D2H / host / H2D round trip of the intermediate.
static int run_unstable_convert(g2p_ctx* ctx, Worker& w, const u8* d_gaf, size_t n, cudaStream_t st, g2p_result* res, u8** d_out) {
    g2p_result r1;
    u8* d_mid = nullptr;
    ctx->warn_text.clear();
    int rc = run_unstable(ctx, w, d_gaf, n, st, &r1, &d_mid);
    if (rc) return rc;
    (void)d_mid;
    std::swap(w.d_out, w.d_mid);   // the intermediate GAF stays in d_mid (until the next call); the converter writes d_out
    ctx->warn_mid = static_cast<const u8*>(w.d_mid.p);
    ctx->warn_pending = !ctx->warns.empty();
    const LenTableView saved = ctx->table;
    const bool saved_have = ctx->have_table;
    ctx->table = ctx->node_table;
    ctx->have_table = true;
    rc = run_pipeline(ctx, w, static_cast<const u8*>(w.d_mid.p), (size_t)r1.out_bytes, st, res, d_out);
    ctx->table = saved;
    ctx->have_table = saved_have;
    if (rc) return rc;
    res->unstable_ms = r1.device_ms;
    res->device_ms += r1.device_ms;
    res->gpu_launches += r1.gpu_launches;
    res->mid_bytes = r1.out_bytes;
    if (res->rec_status != G2P_REC_OK) res->stage = 2;
    else if (r1.rec_status != G2P_REC_OK) {   // stage 1 stopped at a record: everything before it was converted
        res->rec_status = r1.rec_status; res->rec_aux = r1.rec_aux; res->err_record = r1.err_record;
        res->stage = 1;
    }
    // stage 2 counts the records of the intermediate GAF ('*' lines are dropped by stage 1)
    return G2P_OK;
}

int g2p_unstable_convert_device(g2p_ctx* ctx, const void* d_gaf_v, size_t n, void** d_out, g2p_result* res, void* stream) {
    if (!ctx || !res || !d_out) return G2P_E_ARG;
    if (!ctx->have_rgfa) return G2P_E_NOTABLE;
    if (n >= 0xFFFFFFF0ULL) return G2P_E_TOOBIG;
    if ((reinterpret_cast<uintptr_t>(d_gaf_v) & 15) != 0) { ctx->set_err("d_gaf must be 16-byte aligned"); return G2P_E_ARG; }
    G2P_CUDA(cudaSetDevice(ctx->device));
    Worker& w = ctx->w[0];
    cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : w.stream;
    u8* d_o = nullptr;
    int rc = run_unstable_convert(ctx, w, static_cast<const u8*>(d_gaf_v), n, st, res, &d_o);
    *d_out = d_o;
    return rc;
}

int g2p_unstable_convert_host(g2p_ctx* ctx, const char* gaf, size_t n, const char** out, g2p_result* res) {
    if (!ctx || !res || !out || (!gaf && n)) return G2P_E_ARG;
    if (!ctx->have_rgfa) return G2P_E_NOTABLE;
    if (n >= 0xFFFFFFF0ULL) return G2P_E_TOOBIG;
    *out = nullptr;
    G2P_CUDA(cudaSetDevice(ctx->device));
    Worker& w = ctx->w[0];
    PinBuf& h_out = ctx->next_out();
    G2P_CUDA(w.d_in.ensure(n + 256));
    if (n) G2P_CUDA(cudaMemcpyAsync(w.d_in.p, gaf, n, cudaMemcpyHostToDevice, w.stream));
    u8* d_o = nullptr;
    int rc = run_unstable_convert(ctx, w, static_cast<const u8*>(w.d_in.p), n, w.stream, res, &d_o);
    if (rc) return rc;
    G2P_CUDA(h_out.ensure(res->out_bytes + 1));
    if (res->out_bytes) G2P_CUDA(cudaMemcpyAsync(h_out.p, d_o, res->out_bytes, cudaMemcpyDeviceToHost, w.stream));
    G2P_CUDA(cudaStreamSynchronize(w.stream));
    *out = static_cast<const char*>(h_out.p);
    return G2P_OK;
}

int g2p_unstable_convert_warnings(g2p_ctx* ctx, const char** text, size_t* n) {
    if (!ctx || !text || !n) return G2P_E_ARG;
    if (ctx->warn_pending) {
        // the stage-1 warnings (gaf2unstable_main.cpp:165-171) quote the record it wrote: fetch those lines from the
        // intermediate GAF -- here, not inside the conversion call
        G2P_CUDA(cudaSetDevice(ctx->device));
        for (const g2p_warn& wn : ctx->warns) {
            std::vector<char> line(wn.out_len + 1), msg(wn.out_len + 4096);
            G2P_CUDA(cudaMemcpy(line.data(), ctx->warn_mid + wn.out_off, wn.out_len, cudaMemcpyDeviceToHost));
            g2p_format_unstable_warning(ctx, line.data(), wn.out_len, msg.data(), msg.size());
            ctx->warn_text += msg.data();
        }
        ctx->warn_pending = false;
    }
    *text = ctx->warn_text.data();
    *n = ctx->warn_text.size();
    return G2P_OK;
}

int g2p_unstable_warnings(g2p_ctx* ctx, const g2p_warn** warns, size_t* n) {
    if (!ctx || !warns || !n) return G2P_E_ARG;
    *warns = ctx->warns.data();
    *n = ctx->warns.size();
    return G2P_OK;
}

// "[gaf2unstable] warning: Target path spans multiple reference contigs a, b, \nthe (unstable) record is\n<line>\n"
// (gaf2unstable_main.cpp:165-171): contig names in ascending contig-id order; the record printed
// there does not carry an rc tag of its own making, which is what the output line holds as well.
int g2p_format_unstable_warning(g2p_ctx* ctx, const char* line, size_t len, char* buf, size_t cap) {
    if (!ctx || !line || !buf || cap == 0 || !ctx->rgfa) return G2P_E_ARG;
    buf[0] = 0;
    const RgfaTables& T = *ctx->rgfa;
    // column 6 = the path
    size_t a = 0;
    for (int c = 0; c < 5 && a < len; ++c) { const void* t = std::memchr(line + a, '\t', len - a); if (!t) return G2P_E_ARG; a = static_cast<const char*>(t) - line + 1; }
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
    std::string m = "[gaf2unstable] warning: Target path spans multiple reference contigs ";
    for (int64_t id : ids) { m += T.ref_contigs[(size_t)id]; m += ", "; }
    m += "\nthe (unstable) record is\n";
    size_t ll = len;
    while (ll > 0 && line[ll - 1] == '\n') --ll;
    m.append(line, ll);
    m += "\n";
    std::snprintf(buf, cap, "%s", m.c_str());
    return G2P_OK;
}

// ---- N1: gaffilter on the device ------------------------------------------------------------------------
// The launch sequences of the single call (run_filter) and of the job (g2p_filter_job_*): parse, sort, sweep, emit.
struct FilterWork {
    u32 n = 0, grid = 0, nblk = 0, nh = 0, nscan_h = 0, nscan_r = 0;
    FRow* rows = nullptr;
    u64 *keys = nullptr, *keys2 = nullptr, *hist = nullptr, *d_blocks = nullptr, *d_off = nullptr;
    u32 *vals = nullptr, *vals2 = nullptr;
    i64* pmax = nullptr;
    u8* keep = nullptr;
    FilterMeta* d_fm = nullptr;
};

// work buffers for n rows (and n lines of text: d_off) + a cleared FilterMeta
static int filter_work(g2p_ctx* ctx, Worker& w, u32 n, cudaStream_t st, FilterWork& f) {
    f.n = n;
    f.nblk = (n + kRsTile - 1) / kRsTile; f.nh = 16u * f.nblk;
    f.nscan_h = (f.nh + kScanTile - 1) / kScanTile; f.nscan_r = (n + kScanTile - 1) / kScanTile;
    f.grid = std::max<u32>(1u, std::min<u32>((n + 127) / 128, (u32)ctx->n_sm * 16u));
    G2P_CUDA(w.f_rows.ensure((size_t)n * sizeof(FRow)));
    G2P_CUDA(w.f_keys.ensure((size_t)n * 8)); G2P_CUDA(w.f_keys2.ensure((size_t)n * 8));
    G2P_CUDA(w.f_vals.ensure((size_t)n * 4)); G2P_CUDA(w.f_vals2.ensure((size_t)n * 4));
    G2P_CUDA(w.f_pmax.ensure((size_t)n * 8));
    G2P_CUDA(w.f_keep.ensure((size_t)n));
    G2P_CUDA(w.f_hist.ensure(((size_t)f.nh + 2 + f.nscan_h + f.nscan_r) * 8));
    G2P_CUDA(w.f_meta.ensure(sizeof(FilterMeta)));
    G2P_CUDA(w.d_off.ensure(((size_t)n + 1) * sizeof(u64)));
    G2P_CUDA(w.d_blocks.ensure((size_t)std::max(f.nscan_r, f.nscan_h) * 2 * sizeof(u64)));
    f.d_fm = static_cast<FilterMeta*>(w.f_meta.p);
    FilterMeta init;
    std::memset(&init, 0, sizeof init);
    init.first_err = 0xFFFFFFFFu;
    init.assert_rec = 0xFFFFFFFFu;
    init.assert_grec = ~0ULL;
    G2P_CUDA(cudaMemcpyAsync(f.d_fm, &init, sizeof init, cudaMemcpyHostToDevice, st));
    f.keys = static_cast<u64*>(w.f_keys.p); f.keys2 = static_cast<u64*>(w.f_keys2.p);
    f.vals = static_cast<u32*>(w.f_vals.p); f.vals2 = static_cast<u32*>(w.f_vals2.p);
    f.rows = static_cast<FRow*>(w.f_rows.p);
    f.hist = static_cast<u64*>(w.f_hist.p);
    f.d_blocks = static_cast<u64*>(w.d_blocks.p);
    f.d_off = static_cast<u64*>(w.d_off.p);
    f.pmax = static_cast<i64*>(w.f_pmax.p);
    f.keep = static_cast<u8*>(w.f_keep.p);
    return G2P_OK;
}

// line index + k_filter_parse of a text block; f.n = 0 (and no buffers) for an empty one
static int filter_parse(g2p_ctx* ctx, Worker& w, const u8* d_text, size_t n, const FilterParams& P, u64 grec_base, cudaStream_t st,
                        uint32_t* launches, FilterWork& f, FilterArgs& fa) {
    int rc = run_index(ctx, w, d_text, n, st, launches);
    if (rc) return rc;
    const u32 nrec = static_cast<const PipelineMeta*>(w.h_meta.p)->n_records;
    f = FilterWork();
    if (nrec == 0) return G2P_OK;
    rc = filter_work(ctx, w, nrec, st, f);
    if (rc) return rc;
    fa = FilterArgs{d_text, static_cast<const u32*>(w.d_rec.p), nrec, P, f.rows, f.keys, f.vals, f.d_fm, grec_base};
    k_filter_parse<<<f.grid, 128, 0, st>>>(fa);
    ++*launches;
    return G2P_OK;
}

// stable LSD radix sort of (f.keys, f.vals) on the low 4 * passes bits; the result is in (f.keys, f.vals)
static void filter_rsort(FilterWork& f, u32 passes, cudaStream_t st, uint32_t* launches) {
    for (u32 shift = 0; shift < 4 * passes; shift += 4) {
        k_rs_hist<<<f.nblk, kRsThreads, 0, st>>>(f.keys, f.n, shift, f.hist, f.nblk);
        k_scan_reduce<<<f.nscan_h, kScanThreads, 0, st>>>(f.hist, f.nh, f.d_blocks);
        k_scan_blocks<<<1, 1024, 0, st>>>(f.d_blocks, f.nscan_h, f.hist + f.nh + 1);
        k_scan_apply<<<f.nscan_h, kScanThreads, 0, st>>>(f.hist, f.nh, f.d_blocks, f.hist + f.nh + 1);
        k_rs_scatter<<<f.nblk, kRsThreads, 0, st>>>(f.keys, f.vals, f.keys2, f.vals2, f.n, shift, f.hist, f.nblk);
        std::swap(f.keys, f.keys2);
        std::swap(f.vals, f.vals2);
        *launches += 5;
    }
}

// sort by (hash32, query_start), running maximum of the interval ends, sweep: keep[] in the order of f.rows
static int filter_decide(g2p_ctx* ctx, Worker& w, FilterWork& f, const FilterParams& P, cudaStream_t st, uint32_t* launches) {
    filter_rsort(f, 16, st, launches);
    {   // segmented max-scan of the interval ends over the sorted order
        const u32 nseg = (f.n + kSegTile - 1) / kSegTile;
        G2P_CUDA(w.f_seg.ensure((size_t)nseg * 24 + 64));
        i64* tile_val = static_cast<i64*>(w.f_seg.p);
        i64* carry = tile_val + nseg;
        u32* tile_flag = reinterpret_cast<u32*>(carry + nseg);
        k_filter_ends<<<f.grid, 256, 0, st>>>(f.keys, f.vals, f.rows, f.n, f.pmax);
        k_segmax<false><<<nseg, kSegThreads, 0, st>>>(f.keys, f.n, f.pmax, tile_val, tile_flag, nullptr);
        k_segmax_tiles<<<1, 32, 0, st>>>(tile_val, tile_flag, nseg, carry);
        k_segmax<true><<<nseg, kSegThreads, 0, st>>>(f.keys, f.n, f.pmax, tile_val, tile_flag, carry);
        *launches += 3;
    }
    G2P_CUDA(cudaMemsetAsync(f.keep, 0, f.n, st));
    k_filter_sweep<<<f.grid, 128, 0, st>>>(f.keys, f.vals, f.rows, f.pmax, f.n, P, f.keep, f.d_fm);
    *launches += 2;
    return G2P_OK;
}

// size pass and scan of the kept lines of a text block (total -> f.d_fm->out_total)
static void filter_emit_sizes(FilterWork& f, const u8* d_text, const u32* d_rec, u32 is_paf, cudaStream_t st, uint32_t* launches) {
    k_filter_emit<false><<<f.grid, 128, 0, st>>>(d_text, d_rec, f.n, is_paf, f.keep, f.d_off, nullptr);
    k_scan_reduce<<<f.nscan_r, kScanThreads, 0, st>>>(f.d_off, f.n, f.d_blocks);
    k_scan_blocks<<<1, 1024, 0, st>>>(f.d_blocks, f.nscan_r, &f.d_fm->out_total);
    k_scan_apply<<<f.nscan_r, kScanThreads, 0, st>>>(f.d_off, f.n, f.d_blocks, &f.d_fm->out_total);
    *launches += 4;
}

static int filter_emit_text(g2p_ctx* ctx, Worker& w, FilterWork& f, const u8* d_text, const u32* d_rec, u32 is_paf, u64 out_total, cudaStream_t st,
                            uint32_t* launches, u8** d_out) {
    G2P_CUDA(w.d_out.ensure(out_total + 256));
    *d_out = static_cast<u8*>(w.d_out.p);
    k_filter_emit<true><<<f.grid, 128, 0, st>>>(d_text, d_rec, f.n, is_paf, f.keep, f.d_off, *d_out);
    ++*launches;
    return G2P_OK;
}

static FilterParams filter_params(const g2p_filter_params* gp) {
    return FilterParams{gp->ratio, gp->min_overlap_pct, gp->min_identity, gp->min_overlap_len, gp->min_block_len, gp->min_mapq, gp->is_paf ? 1u : 0u};
}

static int run_filter(g2p_ctx* ctx, Worker& w, const u8* d_text, size_t n, const g2p_filter_params* gp, cudaStream_t st, g2p_filter_result* res, u8** d_out) {
    std::memset(res, 0, sizeof *res);
    *d_out = nullptr;
    uint32_t launches = 0;
    G2P_CUDA(cudaEventRecord(w.ev[0], st));
    const FilterParams P = filter_params(gp);
    FilterWork f;
    FilterArgs fa;
    int rc = filter_parse(ctx, w, d_text, n, P, 0, st, &launches, f, fa);
    if (rc) return rc;
    G2P_CUDA(w.d_out.ensure(256));
    *d_out = static_cast<u8*>(w.d_out.p);
    if (f.n == 0) { G2P_CUDA(cudaStreamSynchronize(st)); res->gpu_launches = launches; return G2P_OK; }
    rc = filter_decide(ctx, w, f, P, st, &launches);
    if (rc) return rc;
    const u32* d_rec = static_cast<const u32*>(w.d_rec.p);
    filter_emit_sizes(f, d_text, d_rec, P.is_paf, st, &launches);
    k_filter_diagnose<<<1, 1, 0, st>>>(fa);
    ++launches;
    FilterMeta hm;
    G2P_CUDA(cudaMemcpyAsync(&hm, f.d_fm, sizeof hm, cudaMemcpyDeviceToHost, st));
    G2P_CUDA(cudaStreamSynchronize(st));
    G2P_CUDA(cudaGetLastError());
    res->n_loaded = hm.n_loaded;
    if (hm.first_err == 0xFFFFFFFFu && hm.unsupported) { ctx->set_err("gaffilter: a query_start >= 2^32 is not supported by the device sort"); return G2P_E_ARG; }
    if (hm.first_err != 0xFFFFFFFFu) {   // the reference dies while it loads the records: nothing is printed
        res->rec_status = hm.err_status & 0xff;
        if (res->rec_status < G2P_REC_ABORT) res->rec_status = G2P_REC_ABORT + 8;
        res->err_record = hm.first_err;
        res->gpu_launches = launches;
        return G2P_OK;
    }
    if (hm.assert_grec != ~0ULL) {   // an assertion of the reference's filter loop (gaffilter_main.cpp:68, :289): it aborts
        res->rec_status = G2P_REC_ABORT + 9;
        res->err_record = hm.assert_grec;
        res->gpu_launches = launches;
        return G2P_OK;
    }
    res->n_filtered = hm.n_filtered;
    res->filtered_len = hm.filtered_len;
    res->out_bytes = hm.out_total;
    u8* d_o = nullptr;
    rc = filter_emit_text(ctx, w, f, d_text, d_rec, P.is_paf, hm.out_total, st, &launches, &d_o);
    if (rc) return rc;
    G2P_CUDA(cudaEventRecord(w.ev[4], st));
    G2P_CUDA(cudaStreamSynchronize(st));
    G2P_CUDA(cudaGetLastError());
    cudaEventElapsedTime(&res->device_ms, w.ev[0], w.ev[4]);
    res->gpu_launches = launches;
    *d_out = d_o;
    return G2P_OK;
}

int g2p_filter_device(g2p_ctx* ctx, const void* d_text, size_t n, const g2p_filter_params* params, void** d_out, g2p_filter_result* res, void* stream) {
    if (!ctx || !res || !d_out || !params) return G2P_E_ARG;
    if (n >= 0xFFFFFFF0ULL) return G2P_E_TOOBIG;
    if ((reinterpret_cast<uintptr_t>(d_text) & 15) != 0) { ctx->set_err("d_text must be 16-byte aligned"); return G2P_E_ARG; }
    G2P_CUDA(cudaSetDevice(ctx->device));
    Worker& w = ctx->w[1];   // (not worker 0: the text may be worker 0's own output buffer, a PAF made by g2p_convert_device)
    cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : w.stream;
    u8* d_o = nullptr;
    int rc = run_filter(ctx, w, static_cast<const u8*>(d_text), n, params, st, res, &d_o);
    *d_out = d_o;
    return rc;
}

int g2p_filter_host(g2p_ctx* ctx, const char* text, size_t n, const g2p_filter_params* params, const char** out, g2p_filter_result* res) {
    if (!ctx || !res || !out || !params || (!text && n)) return G2P_E_ARG;
    if (n >= 0xFFFFFFF0ULL) return G2P_E_TOOBIG;
    *out = nullptr;
    G2P_CUDA(cudaSetDevice(ctx->device));
    Worker& w = ctx->w[1];
    PinBuf& h_out = ctx->next_out();
    G2P_CUDA(w.d_in.ensure(n + 256));
    if (n) G2P_CUDA(cudaMemcpyAsync(w.d_in.p, text, n, cudaMemcpyHostToDevice, w.stream));
    u8* d_o = nullptr;
    int rc = run_filter(ctx, w, static_cast<const u8*>(w.d_in.p), n, params, w.stream, res, &d_o);
    if (rc) return rc;
    G2P_CUDA(h_out.ensure(res->out_bytes + 1));
    if (res->out_bytes) G2P_CUDA(cudaMemcpyAsync(h_out.p, d_o, res->out_bytes, cudaMemcpyDeviceToHost, w.stream));
    G2P_CUDA(cudaStreamSynchronize(w.stream));
    *out = static_cast<const char*>(h_out.p);
    return G2P_OK;
}

// ---- the gaffilter job: inputs of any size over one or more contexts (g2p_filter_job.hpp, g2p_filter.cuh) ----------
// Load pass per chunk: parse, partition the loaded rows by query-name bucket, chunk layout -> host memory.  Decide:
// per range of buckets, the rows of every chunk's segment -> one GPU, sort + sweep, keep flags -> host memory (in
// layout order, per chunk).  Emit pass per chunk: parse and partition again, keep flags scattered to the lines, print.
namespace {
struct HostArr {   // pinned (portable: any context copies from / to it) when possible, else pageable
    void* p = nullptr;
    bool pinned = false;
    bool alloc(size_t bytes) {
        if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable) == cudaSuccess) { pinned = true; return true; }
        (void)cudaGetLastError();
        p = std::malloc(bytes ? bytes : 1);
        return p != nullptr;
    }
    void release() {
        if (p) { if (pinned) cudaFreeHost(p); else std::free(p); }
        p = nullptr;
    }
};
struct JobChunk {
    g2p_fjob::ChunkBook book;
    HostArr rows, keep;   // the chunk layout (FRow), its keep flags (u8)
};
}  // namespace

struct g2p_filter_job {
    std::vector<g2p_ctx*> ctxs;
    g2p_filter_params params;
    int min_parts = 1;                          // G2P_FILTER_PARTS (tests): at least this many partitions
    std::mutex mu;
    std::vector<std::unique_ptr<JobChunk>> chunks;
    bool decided = false, printable = false;    // printable: decide found no error
    g2p_filter_job_stats stats{};
    ~g2p_filter_job() {
        for (auto& c : chunks) if (c) { c->rows.release(); c->keep.release(); }
    }
    void add_stats(int pass, double ms, uint64_t h2d, uint64_t d2h) {
        std::lock_guard<std::mutex> g(mu);
        (pass == 0 ? stats.load_ms : pass == 1 ? stats.decide_ms : stats.emit_ms) += ms;
        stats.h2d_bytes += h2d;
        stats.d2h_bytes += d2h;
    }
};

// bucket partition of a parsed chunk (f.keys / f.vals: after it, vals[p] = line of layout position p); h_off <- offsets
static int filter_partition(g2p_ctx* ctx, Worker& w, FilterWork& f, cudaStream_t st, uint32_t* launches, uint32_t* h_off) {
    G2P_CUDA(w.f_boff.ensure((kFBuckets + 1) * sizeof(u32)));
    u32* d_boff = static_cast<u32*>(w.f_boff.p);
    k_filter_bucket_key<<<f.grid, 128, 0, st>>>(f.keys, f.n, f.keys2);
    std::swap(f.keys, f.keys2);
    filter_rsort(f, 3, st, launches);   // 9 bits: buckets 0..255, unloaded lines 256
    k_filter_bucket_offsets<<<std::min<u32>(f.n / 128 + 1, (u32)ctx->n_sm * 16u), 128, 0, st>>>(f.keys, f.n, d_boff);
    *launches += 2;
    G2P_CUDA(cudaMemcpyAsync(h_off, d_boff, (kFBuckets + 1) * sizeof(u32), cudaMemcpyDeviceToHost, st));
    G2P_CUDA(cudaStreamSynchronize(st));
    G2P_CUDA(cudaGetLastError());
    return G2P_OK;
}

int g2p_filter_job_create(g2p_ctx* const* ctxs, int nctx, const g2p_filter_params* params, g2p_filter_job** out) {
    if (!ctxs || nctx < 1 || !params || !out) return G2P_E_ARG;
    *out = nullptr;
    for (int i = 0; i < nctx; ++i) if (!ctxs[i]) return G2P_E_ARG;
    g2p_filter_job* J = new (std::nothrow) g2p_filter_job();
    if (!J) return G2P_E_ARG;
    J->ctxs.assign(ctxs, ctxs + nctx);
    J->params = *params;
    if (const char* v = std::getenv("G2P_FILTER_PARTS")) J->min_parts = std::max(1, std::min(std::atoi(v), (int)kFBuckets));
    *out = J;
    return G2P_OK;
}

void g2p_filter_job_destroy(g2p_filter_job* J) { delete J; }

int g2p_filter_job_load(g2p_filter_job* J, uint64_t chunk, const char* text, size_t n) {
    if (!J || (!text && n) || chunk > 0xFFFFFFFFull) return G2P_E_ARG;
    g2p_ctx* ctx = J->ctxs[chunk % J->ctxs.size()];
    if (J->decided) { ctx->set_err("gaffilter job: load after decide"); return G2P_E_ARG; }
    if (n >= 0xFFFFFFF0ULL) { ctx->set_err("gaffilter job: a chunk must be < 4 GiB"); return G2P_E_TOOBIG; }
    G2P_CUDA(cudaSetDevice(ctx->device));
    Worker& w = ctx->w[1];
    cudaStream_t st = w.stream;
    uint32_t launches = 0;
    G2P_CUDA(cudaEventRecord(w.ev[0], st));
    G2P_CUDA(w.d_in.ensure(n + 256));
    if (n) G2P_CUDA(cudaMemcpyAsync(w.d_in.p, text, n, cudaMemcpyHostToDevice, st));
    const u8* d_text = static_cast<const u8*>(w.d_in.p);
    std::unique_ptr<JobChunk> C(new JobChunk());
    C->book.loaded = true;
    C->book.bytes = n;
    FilterWork f;
    FilterArgs fa;
    int rc = filter_parse(ctx, w, d_text, n, filter_params(&J->params), chunk << 32, st, &launches, f, fa);
    if (rc) return rc;
    C->book.lines = f.n;
    uint64_t d2h = 0;
    if (f.n) {
        rc = filter_partition(ctx, w, f, st, &launches, C->book.off);
        if (rc) return rc;
        const u32 nl = C->book.n_loaded();
        G2P_CUDA(w.f_lay.ensure((size_t)nl * sizeof(FRow) + 16));
        FRow* lay = static_cast<FRow*>(w.f_lay.p);
        if (nl) { k_filter_gather_rows<<<f.grid, 128, 0, st>>>(f.rows, f.vals, nl, lay); ++launches; }
        k_filter_diagnose<<<1, 1, 0, st>>>(fa);
        ++launches;
        FilterMeta hm;
        G2P_CUDA(cudaMemcpyAsync(&hm, f.d_fm, sizeof hm, cudaMemcpyDeviceToHost, st));
        if (!C->rows.alloc((size_t)nl * sizeof(FRow)) || !C->keep.alloc(nl)) { ctx->set_err("gaffilter job: out of host memory for the rows"); return G2P_E_ARG; }
        if (nl) G2P_CUDA(cudaMemcpyAsync(C->rows.p, lay, (size_t)nl * sizeof(FRow), cudaMemcpyDeviceToHost, st));
        G2P_CUDA(cudaEventRecord(w.ev[4], st));
        G2P_CUDA(cudaStreamSynchronize(st));
        G2P_CUDA(cudaGetLastError());
        C->book.first_err = hm.first_err;
        C->book.err_status = hm.err_status;
        C->book.unsupported = hm.unsupported != 0;
        d2h = (size_t)nl * sizeof(FRow);
    } else {
        G2P_CUDA(cudaEventRecord(w.ev[4], st));
        G2P_CUDA(cudaStreamSynchronize(st));
        if (!C->rows.alloc(0) || !C->keep.alloc(0)) return G2P_E_ARG;
    }
    float ms = 0;
    cudaEventElapsedTime(&ms, w.ev[0], w.ev[4]);
    J->add_stats(0, ms, n, d2h);
    std::lock_guard<std::mutex> g(J->mu);
    if (J->chunks.size() <= chunk) J->chunks.resize(chunk + 1);
    if (J->chunks[chunk]) { ctx->set_err("gaffilter job: chunk " + std::to_string(chunk) + " loaded twice"); C->rows.release(); C->keep.release(); return G2P_E_ARG; }
    J->chunks[chunk] = std::move(C);
    return G2P_OK;
}

namespace {
struct PartOut { uint64_t n_filtered = 0, filtered_len = 0, assert_grec = ~0ULL; float ms = 0; uint32_t launches = 0; };
}

// one partition on one context: the chunks' segments up, decide, keep flags back into the chunks' keep arrays
static int job_decide_part(g2p_filter_job* J, g2p_ctx* ctx, const g2p_fjob::Part& pt, PartOut& o) {
    if (pt.rows == 0) return G2P_OK;
    G2P_CUDA(cudaSetDevice(ctx->device));
    Worker& w = ctx->w[1];
    cudaStream_t st = w.stream;
    FilterWork f;
    int rc = filter_work(ctx, w, (u32)pt.rows, st, f);
    if (rc) return rc;
    G2P_CUDA(cudaEventRecord(w.ev[0], st));
    size_t pos = 0;
    for (auto& C : J->chunks) {
        const size_t seg = C->book.seg_rows(pt.b0, pt.b1);
        if (seg) G2P_CUDA(cudaMemcpyAsync(f.rows + pos, static_cast<const FRow*>(C->rows.p) + C->book.seg_begin(pt.b0), seg * sizeof(FRow), cudaMemcpyHostToDevice, st));
        pos += seg;
    }
    k_filter_rekey<<<f.grid, 128, 0, st>>>(f.rows, f.n, f.keys, f.vals);
    ++o.launches;
    rc = filter_decide(ctx, w, f, filter_params(&J->params), st, &o.launches);
    if (rc) return rc;
    pos = 0;
    for (auto& C : J->chunks) {
        const size_t seg = C->book.seg_rows(pt.b0, pt.b1);
        if (seg) G2P_CUDA(cudaMemcpyAsync(static_cast<u8*>(C->keep.p) + C->book.seg_begin(pt.b0), f.keep + pos, seg, cudaMemcpyDeviceToHost, st));
        pos += seg;
    }
    FilterMeta hm;
    G2P_CUDA(cudaMemcpyAsync(&hm, f.d_fm, sizeof hm, cudaMemcpyDeviceToHost, st));
    G2P_CUDA(cudaEventRecord(w.ev[4], st));
    G2P_CUDA(cudaStreamSynchronize(st));
    G2P_CUDA(cudaGetLastError());
    cudaEventElapsedTime(&o.ms, w.ev[0], w.ev[4]);
    o.n_filtered = hm.n_filtered;
    o.filtered_len = hm.filtered_len;
    o.assert_grec = hm.assert_grec;
    J->add_stats(1, 0, pt.rows * sizeof(FRow), pt.rows);
    return G2P_OK;
}

int g2p_filter_job_decide(g2p_filter_job* J, g2p_filter_result* res) {
    if (!J || !res) return G2P_E_ARG;
    std::memset(res, 0, sizeof *res);
    g2p_ctx* ctx0 = J->ctxs[0];
    if (J->decided) { ctx0->set_err("gaffilter job: decided twice"); return G2P_E_ARG; }
    J->decided = true;
    std::vector<g2p_fjob::ChunkBook> books;
    for (size_t c = 0; c < J->chunks.size(); ++c) {
        if (!J->chunks[c]) { ctx0->set_err("gaffilter job: chunk " + std::to_string(c) + " was not loaded"); return G2P_E_ARG; }
        books.push_back(J->chunks[c]->book);
    }
    const std::vector<uint64_t> bases = g2p_fjob::line_bases(books);
    for (const auto& b : books) res->n_loaded += b.n_loaded();
    // a line that fails to load anywhere wins (the reference dies while it loads: nothing is printed)
    uint64_t line;
    uint32_t status;
    if (g2p_fjob::first_load_error(books, bases, line, status)) {
        res->rec_status = status & 0xff;
        if (res->rec_status < G2P_REC_ABORT) res->rec_status = G2P_REC_ABORT + 8;
        res->err_record = line;
        return G2P_OK;
    }
    for (const auto& b : books)
        if (b.unsupported) { ctx0->set_err("gaffilter: a query_start >= 2^32 is not supported by the device sort"); return G2P_E_ARG; }
    // capacity: the rows one GPU can decide at once (~130 B of device memory per row)
    uint64_t cap = 0x7FFFFFFFull;
    for (g2p_ctx* ctx : J->ctxs) {
        size_t fr = 0, tot = 0;
        G2P_CUDA(cudaSetDevice(ctx->device));
        G2P_CUDA(cudaMemGetInfo(&fr, &tot));
        cap = std::min<uint64_t>(cap, (uint64_t)(fr * 0.85) / 130);
    }
    std::vector<g2p_fjob::Part> parts;
    const std::string perr = g2p_fjob::plan_partitions(g2p_fjob::bucket_rows(books), cap, J->min_parts, (int)J->ctxs.size(), parts);
    if (!perr.empty()) { ctx0->set_err("gaffilter: " + perr); return G2P_E_TOOBIG; }
    std::vector<PartOut> outs(parts.size());
    std::vector<int> rcs(J->ctxs.size(), G2P_OK);
    {
        std::vector<std::thread> th;
        for (size_t g = 0; g < J->ctxs.size(); ++g)
            th.emplace_back([&, g] {
                for (size_t i = 0; i < parts.size() && rcs[g] == G2P_OK; ++i)
                    if (parts[i].gpu == (int)g) rcs[g] = job_decide_part(J, J->ctxs[g], parts[i], outs[i]);
            });
        for (auto& t : th) t.join();
    }
    for (size_t g = 0; g < J->ctxs.size(); ++g)
        if (rcs[g] != G2P_OK) {
            if (g) ctx0->set_err(g2p_last_error(J->ctxs[g]));
            return rcs[g];
        }
    uint64_t assert_grec = ~0ULL;
    for (const PartOut& o : outs) {
        res->n_filtered += o.n_filtered;
        res->filtered_len += o.filtered_len;   // (mod 2^64, like the single call's sum)
        assert_grec = std::min(assert_grec, o.assert_grec);
        res->device_ms += o.ms;
        res->gpu_launches += o.launches;
    }
    J->add_stats(1, res->device_ms, 0, 0);
    for (auto& C : J->chunks) C->rows.release();   // (the emit pass needs the keep flags only)
    if (assert_grec != ~0ULL) {   // an assertion of the reference's filter loop: it aborts
        res->n_filtered = res->filtered_len = 0;
        res->rec_status = G2P_REC_ABORT + 9;
        res->err_record = g2p_fjob::global_line(bases, assert_grec);
        return G2P_OK;
    }
    J->printable = true;
    return G2P_OK;
}

int g2p_filter_job_emit(g2p_filter_job* J, uint64_t chunk, const char* text, size_t n, const char** out, g2p_filter_result* res) {
    if (!J || !out || !res || (!text && n)) return G2P_E_ARG;
    std::memset(res, 0, sizeof *res);
    *out = nullptr;
    g2p_ctx* ctx = J->ctxs[chunk % J->ctxs.size()];
    if (!J->printable) { ctx->set_err("gaffilter job: emit before a decide without errors"); return G2P_E_ARG; }
    if (chunk >= J->chunks.size()) { ctx->set_err("gaffilter job: chunk " + std::to_string(chunk) + " was not loaded"); return G2P_E_ARG; }
    if (n >= 0xFFFFFFF0ULL) return G2P_E_TOOBIG;
    const JobChunk& C = *J->chunks[chunk];
    G2P_CUDA(cudaSetDevice(ctx->device));
    Worker& w = ctx->w[1];
    cudaStream_t st = w.stream;
    PinBuf& h_out = ctx->next_out();
    uint32_t launches = 0;
    G2P_CUDA(cudaEventRecord(w.ev[0], st));
    G2P_CUDA(w.d_in.ensure(n + 256));
    if (n) G2P_CUDA(cudaMemcpyAsync(w.d_in.p, text, n, cudaMemcpyHostToDevice, st));
    const u8* d_text = static_cast<const u8*>(w.d_in.p);
    const FilterParams P = filter_params(&J->params);
    FilterWork f;
    FilterArgs fa;
    int rc = filter_parse(ctx, w, d_text, n, P, chunk << 32, st, &launches, f, fa);
    if (rc) return rc;
    g2p_fjob::ChunkBook now;
    now.bytes = n;
    now.lines = f.n;
    if (f.n) {
        rc = filter_partition(ctx, w, f, st, &launches, now.off);
        if (rc) return rc;
    }
    const std::string diff = g2p_fjob::same_chunk(C.book, now);
    if (!diff.empty()) { ctx->set_err("gaffilter job: chunk " + std::to_string(chunk) + " differs from the one loaded (" + diff + ")"); return G2P_E_ARG; }
    uint64_t out_total = 0;
    if (f.n) {
        const u32 nl = C.book.n_loaded();
        G2P_CUDA(w.f_lay.ensure((size_t)nl + 16));
        u8* d_klay = static_cast<u8*>(w.f_lay.p);
        if (nl) G2P_CUDA(cudaMemcpyAsync(d_klay, C.keep.p, nl, cudaMemcpyHostToDevice, st));
        G2P_CUDA(cudaMemsetAsync(f.keep, 0, f.n, st));
        if (nl) { k_filter_scatter_keep<<<f.grid, 128, 0, st>>>(f.vals, d_klay, nl, f.keep); ++launches; }
        const u32* d_rec = static_cast<const u32*>(w.d_rec.p);
        filter_emit_sizes(f, d_text, d_rec, P.is_paf, st, &launches);
        G2P_CUDA(cudaMemcpyAsync(&out_total, &f.d_fm->out_total, sizeof out_total, cudaMemcpyDeviceToHost, st));
        G2P_CUDA(cudaStreamSynchronize(st));
        u8* d_o = nullptr;
        rc = filter_emit_text(ctx, w, f, d_text, d_rec, P.is_paf, out_total, st, &launches, &d_o);
        if (rc) return rc;
        G2P_CUDA(h_out.ensure(out_total + 1));
        if (out_total) G2P_CUDA(cudaMemcpyAsync(h_out.p, d_o, out_total, cudaMemcpyDeviceToHost, st));
        const u8* k = static_cast<const u8*>(C.keep.p);
        for (u32 i = 0; i < nl; ++i) res->n_filtered += k[i] == 0;
        res->n_loaded = nl;
    } else {
        G2P_CUDA(h_out.ensure(1));
    }
    G2P_CUDA(cudaEventRecord(w.ev[4], st));
    G2P_CUDA(cudaStreamSynchronize(st));
    G2P_CUDA(cudaGetLastError());
    cudaEventElapsedTime(&res->device_ms, w.ev[0], w.ev[4]);
    res->out_bytes = out_total;
    res->gpu_launches = launches;
    J->add_stats(2, res->device_ms, n + C.book.n_loaded(), out_total);
    *out = static_cast<const char*>(h_out.p);
    return G2P_OK;
}

int g2p_filter_job_get_stats(const g2p_filter_job* J, g2p_filter_job_stats* s) {
    if (!J || !s) return G2P_E_ARG;
    *s = J->stats;
    return G2P_OK;
}

int g2p_format_error(const g2p_result* res, const char* gaf, size_t n, char* buf, size_t cap) {
    return g2p_errfmt::format_error(res, gaf, n, buf, cap);
}

}  // extern "C"
