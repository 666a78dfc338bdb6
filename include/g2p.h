/* g2p.h — C-ABI of the B200 GAF->PAF conversion library (libg2p.so).
 *
 * The reference (cactus-gfa-tools) has no library / plugin / FFI surface: its only
 * stable interface is the process boundary of the `gaf2paf` and `gaf2unstable`
 * executables (SURVEY.md §1, §8b).  This header is therefore the boundary the new
 * build defines between the C++ host drivers (same argv, same stdout/stderr/exit
 * codes as the reference) and the CUDA side.  Each entry point names the reference
 * code it replaces.
 *
 * Conventions: plain pointers and sizes only; every function returns 0 on success or
 * a negative G2P_E_* code (no exceptions cross the boundary); the caller owns host
 * buffers it passes in; the library owns every device buffer and the pinned result
 * buffers it hands back.  Device results are valid until the next call on the same
 * context; the pinned host results of the *_host calls are double-buffered per context
 * and stay valid until the next-but-one *_host call (or g2p_destroy), so that a caller
 * can write result i to its sink while call i+1 runs.  One context per GPU; calls on one context must be serialised by the
 * caller; different contexts may be driven from different host threads.
 *
 * There is no CPU fallback: without a CUDA device g2p_create fails with
 * G2P_E_NO_DEVICE and nothing else can be called.
 */
#ifndef G2P_H
#define G2P_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct g2p_ctx g2p_ctx;

enum {
    G2P_OK = 0,
    G2P_E_NO_DEVICE = -1,   /* no usable CUDA device / driver */
    G2P_E_CUDA = -2,        /* a CUDA call failed; see g2p_last_error */
    G2P_E_ARG = -3,         /* bad argument */
    G2P_E_TABLE = -4,       /* lengths table could not be parsed (reference would abort in std::stol) */
    G2P_E_NOTABLE = -5,     /* convert called before g2p_load_lengths */
    G2P_E_TOOBIG = -6       /* a single call is limited to < 4 GiB of GAF text: split at a newline */
};

/* Status of the first failing record in input order, mirroring the reference's two
 * error classes (SURVEY.md §5): */
enum {
    G2P_REC_OK = 0,
    G2P_REC_ERR_NAME = 1,   /* "[gaf2paf] error: unable to find X in lengths map", exit 1 (gaf2paf_main.cpp:118,163) */
    G2P_REC_ERR_NOCG = 2,   /* "[gaf2paf] error: cg cigar not found…", exit 1 (gaf2paf_main.cpp:365-368) */
    G2P_REC_ABORT = 16      /* >= 16: the reference dies with SIGABRT (assert / uncaught exception), rc 134 */
};

typedef struct g2p_result {
    uint64_t n_records;     /* GAF lines seen (including skipped '*' lines) */
    uint64_t out_bytes;     /* bytes of PAF produced; on error: everything the reference would have flushed */
    uint32_t rec_status;    /* G2P_REC_* of the first failing record (0 = none) */
    uint32_t rec_aux;       /* GAF column number for column parse errors */
    uint64_t err_record;    /* index of the failing record */
    uint64_t err_name_off;  /* byte offset in the input of the missing name (G2P_REC_ERR_NAME) */
    uint32_t err_name_len;
    uint32_t gpu_launches;  /* kernels launched by this call */
    float device_ms;        /* CUDA-event time of the device pipeline (index .. emit) */
    float emit_ms;          /* CUDA-event time of the emit kernel alone */
    float size_ms;          /* CUDA-event time of the size kernel alone */
    float index_ms;         /* CUDA-event time of the line index kernels */
    uint32_t n_delegated;   /* records converted by the general per-record kernel (non-canonical or erroneous records) */
    uint32_t n_long;        /* records converted by the streaming kernel k_long (incl. those it passed on) */
    float fused_ms;         /* CUDA-event time of the one-pass kernel k_fuse (0 when it did not produce the result) */
    uint32_t n_fused;       /* records converted by k_fuse (all of them, or 0 when the general pipeline ran) */
    float unstable_ms;      /* g2p_unstable_convert_*: CUDA-event time of the gaf2unstable stage (included in device_ms) */
    uint32_t stage;         /* g2p_unstable_convert_*: 1 / 2 = rec_status comes from the gaf2unstable / gaf2paf stage */
    uint64_t mid_bytes;     /* g2p_unstable_convert_*: bytes of the intermediate node-space GAF (it never leaves the device) */
    float par_ms;           /* CUDA-event time of the token-parallel kernels k_par_* (part of size_ms) */
    uint32_t n_par;         /* records converted by them (n_long counts what k_rec left; n_long - n_par went on to k_long) */
} g2p_result;

/* Context bound to one CUDA device. */
int g2p_create(int device, g2p_ctx** out);
void g2p_destroy(g2p_ctx* ctx);
const char* g2p_last_error(const g2p_ctx* ctx);

/* Pinned host memory helpers (cudaHostAlloc) so that callers can read files straight
 * into DMA-able memory. */
void* g2p_host_alloc(size_t bytes);
void g2p_host_free(void* p);

/* Synchronous copies between host and device memory (cudaMemcpy) for callers that hold raw
 * device addresses but do not link the CUDA runtime themselves (tests, bench harness). */
int g2p_copy_to_device(void* d_dst, const void* h_src, size_t bytes);
int g2p_copy_to_host(void* h_dst, const void* d_src, size_t bytes);

/* Replaces get_len_map (gaf2paf_main.cpp:22-45): parse a "name<TAB>length…" table held
 * in host memory and upload the open-addressing name->length table. */
int g2p_load_lengths(g2p_ctx* ctx, const char* tsv, size_t n);
uint64_t g2p_table_entries(const g2p_ctx* ctx);

/* Replaces the record loop of gaf2paf main() (gaf2paf_main.cpp:357-373) with
 * parse_gaf_record / flip_gaf / gaf2paf (gafkluge.hpp:84-204, gaf2paf_main.cpp:92-264)
 * for a newline-delimited block of GAF text already resident in device memory.
 *   d_gaf   device pointer, 16-byte aligned; n < 4 GiB bytes; whole lines (a final
 *           line may lack its '\n').
 *   d_out   receives a library-owned device pointer to the PAF bytes.
 *   stream  a cudaStream_t (NULL = default stream).  The call returns after the
 *           stream has been synchronised. */
int g2p_convert_device(g2p_ctx* ctx, const void* d_gaf, size_t n, void** d_out, g2p_result* res, void* stream);

/* Same conversion for GAF text in host memory: host->device copy, device pipeline,
 * device->host copy into a library-owned pinned buffer returned in *out.  This is the
 * call the gaf2paf executable makes for every input chunk. */
int g2p_convert_host(g2p_ctx* ctx, const char* gaf, size_t n, const char** out, g2p_result* res);

/* The line index on its own (first kernel of the pipeline): offsets of line starts of a
 * device-resident text block.  *d_starts receives a library-owned device array of
 * n_lines+1 uint32 offsets (last = n, or n+1 when the final line lacks '\n'). */
int g2p_index_lines(g2p_ctx* ctx, const void* d_text, size_t n, const uint32_t** d_starts, uint64_t* n_lines, void* stream);

/* ---- gaf2unstable (config 2: stable -> unstable node coordinates) ---------------------- */

/* Replaces get_unstable_mapping (gaf2unstable_main.cpp:34-68) and rgfa2contig
 * (rgfa-split.cpp:35-161): scans the S and L lines of a minigraph rGFA held in host memory
 * (gfakluge.hpp:757-967 semantics), builds stable contig -> nodes sorted by SO and node ->
 * reference contig on the host, and uploads them as flat arrays.  When the reference would
 * die on this rGFA, returns G2P_E_TABLE with *ref_exit_code = 1 or 134 and its stderr text
 * (exit 1 cases) in msg. */
int g2p_load_rgfa(g2p_ctx* ctx, const char* rgfa, size_t n, int* ref_exit_code, char* msg, size_t msg_cap);

/* Contents of the -o node-lengths file (gaf2unstable_main.cpp:274-285), rows in the
 * reference's order.  Library-owned, valid until the next g2p_load_rgfa / g2p_destroy. */
int g2p_rgfa_node_lengths(g2p_ctx* ctx, const char** tsv, size_t* n);

/* Replaces the record loop of gaf2unstable main() (gaf2unstable_main.cpp:288-297) with
 * parse_gaf_record / gaf2unstable / operator<<(GafRecord) (gafkluge.hpp:84-204, :288-323,
 * gaf2unstable_main.cpp:70-175) for a newline-delimited block of GAF text.  On a record the
 * reference would abort on, res->rec_status >= G2P_REC_ABORT, res->err_record names it and
 * out_bytes covers the records before it. */
int g2p_unstable_device(g2p_ctx* ctx, const void* d_gaf, size_t n, void** d_out, g2p_result* res, void* stream);
int g2p_unstable_host(g2p_ctx* ctx, const char* gaf, size_t n, const char** out, g2p_result* res);

/* Records of the last g2p_unstable_* call whose path spans several reference contigs
 * (gaf2unstable_main.cpp:165-171), in record order: their output line is out + out_off. */
typedef struct g2p_warn {
    uint64_t record;
    uint64_t out_off;
    uint64_t out_len;   /* including the trailing newline */
} g2p_warn;
int g2p_unstable_warnings(g2p_ctx* ctx, const g2p_warn** warns, size_t* n);
/* The reference's stderr text for one such output line. */
int g2p_format_unstable_warning(g2p_ctx* ctx, const char* out_line, size_t len, char* buf, size_t cap);

/* The reference's two-stage pipeline `gaf2unstable in.gaf -g graph.gfa -o L | gaf2paf - -l L` (README.md:55-58,
 * test/gaf2paf.t:36-37) as ONE call: stage 1 (gaf2unstable_main.cpp:109-175) writes the node-space GAF into device
 * memory, stage 2 (gaf2paf_main.cpp:134-264) converts it from there with the node lengths of the same rGFA as its
 * lengths table -- the intermediate text makes no device->host->device round trip.  Needs g2p_load_rgfa; the -l table
 * of g2p_load_lengths is not touched.  Output: the PAF bytes of the pipeline; res->stage tells which stage stopped at
 * a record (stage 1: the reference's gaf2unstable aborts; the records before it are converted). */
int g2p_unstable_convert_device(g2p_ctx* ctx, const void* d_gaf, size_t n, void** d_out, g2p_result* res, void* stream);
int g2p_unstable_convert_host(g2p_ctx* ctx, const char* gaf, size_t n, const char** out, g2p_result* res);
/* stderr text of the gaf2unstable stage of the last g2p_unstable_convert_* call (its multi-contig warnings). */
int g2p_unstable_convert_warnings(g2p_ctx* ctx, const char** text, size_t* n);

/* ---- gaffilter (SURVEY.md §8f N1): the query-overlap filter on GAF or PAF text that is already on the device ----------
 * Replaces the whole of gaffilter's main() after option parsing (gaffilter_main.cpp:186-343): load all records, one
 * interval tree per query, keep a record iff it dominates every qualifying overlapping record (dominates :31-60,
 * dominates_mzgaf2paf :63-66), print the kept records in input order re-serialised like operator<<(GafRecord) /
 * operator<<(PafLine).  Parameters as the reference's options (-r/-m/-i go through std::stof there: pass the float
 * value widened to double).  A PAF made by g2p_convert_device can be filtered where it lies: no D2H of the unfiltered PAF. */
typedef struct g2p_filter_params {
    double ratio;              /* -r */
    double min_overlap_pct;    /* -m */
    double min_identity;       /* -i */
    int64_t min_overlap_len;   /* -o */
    int64_t min_block_len;     /* -b */
    int64_t min_mapq;          /* -q */
    int32_t is_paf;            /* -p */
    int32_t pad;
} g2p_filter_params;
typedef struct g2p_filter_result {
    uint64_t n_loaded;         /* "[gaffilter]: Loaded N ... records" */
    uint64_t n_filtered;       /* "[gaffilter]: filtered X / N. total block lengths filtered: Y" */
    uint64_t filtered_len;
    uint64_t out_bytes;
    uint32_t rec_status;       /* 0, or >= G2P_REC_ABORT: the reference dies on line err_record (nothing is printed) */
    uint32_t gpu_launches;
    uint64_t err_record;
    float device_ms;
    uint32_t pad;
} g2p_filter_result;
int g2p_filter_device(g2p_ctx* ctx, const void* d_text, size_t n, const g2p_filter_params* params, void** d_out, g2p_filter_result* res, void* stream);
int g2p_filter_host(g2p_ctx* ctx, const char* text, size_t n, const g2p_filter_params* params, const char** out, g2p_filter_result* res);

/* gaffilter on inputs of any size and on several GPUs.  Whether a record is kept depends only on the records with the
 * same query name, so the job partitions the rows by query name (256 buckets of the name hash) and decides each range of
 * buckets on its own, on any context.  Three passes over the same newline-aligned chunks (each < 4 GiB, numbered from 0
 * in input order; chunk c runs on ctxs[c % nctx]):
 *   load    (every chunk)  parse; the loaded rows, in bucket order, go to host memory (~97 B per record in all)
 *   decide  (once)         the totals and the status of the whole input, as g2p_filter_host reports them for it: a line
 *                          that fails to load wins (its global line number), then a query_start >= 2^32 (G2P_E_ARG, the
 *                          same message), then a filter-loop assertion (the smallest global line); nothing may be
 *                          printed unless rec_status is 0.  G2P_E_TOOBIG when one bucket alone has more records than a
 *                          GPU can sort (a single query with ~10^9 alignments).  Uses one host thread per context.
 *   emit    (every chunk)  the kept records of the chunk, printed like g2p_filter_host prints them; the chunk must be
 *                          the one loaded (bytes, lines and bucket counts are checked: G2P_E_ARG otherwise).  *out is
 *                          double-buffered per context like the *_host results; res->n_loaded / n_filtered count the chunk.
 * load and emit calls of chunks on different contexts may run concurrently from different host threads.
 * G2P_FILTER_PARTS=k (tests) forces at least k partitions. */
typedef struct g2p_filter_job g2p_filter_job;
typedef struct g2p_filter_job_stats {
    double load_ms, decide_ms, emit_ms;   /* CUDA-event time summed over the calls of each pass */
    uint64_t h2d_bytes, d2h_bytes;        /* bytes copied over PCIe by the job's calls */
} g2p_filter_job_stats;
int g2p_filter_job_create(g2p_ctx* const* ctxs, int nctx, const g2p_filter_params* params, g2p_filter_job** out);
int g2p_filter_job_load(g2p_filter_job* job, uint64_t chunk, const char* text, size_t n);
int g2p_filter_job_decide(g2p_filter_job* job, g2p_filter_result* res);
int g2p_filter_job_emit(g2p_filter_job* job, uint64_t chunk, const char* text, size_t n, const char** out, g2p_filter_result* res);
int g2p_filter_job_get_stats(const g2p_filter_job* job, g2p_filter_job_stats* stats);
void g2p_filter_job_destroy(g2p_filter_job* job);

/* Formats the stderr line the reference prints for a failed record (empty for aborts,
 * whose text comes from the C++ runtime).  `gaf` is the host copy of the input. */
int g2p_format_error(const g2p_result* res, const char* gaf, size_t n, char* buf, size_t cap);

#ifdef __cplusplus
}
#endif
#endif /* G2P_H */
