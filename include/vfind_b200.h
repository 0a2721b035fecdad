/*
 * vfind_b200.h — C ABI of the B200-native variant-recovery path.
 *
 * This is the drop-in boundary for vFind's `find_variants` hot path.  The reference
 * (nsbuitrago/vfind, /root/reference) has no FFI of its own for this path: the whole
 * path is Rust behind one PyO3 function (src/lib.rs:168-320).  The entry points below
 * are what a `vfind-b200-sys` FFI crate would bind from that function's body — one
 * entry point per stage of `find_variants` — and what vfind_b200/api.py binds with ctypes.
 * INTEGRATION.md shows both bindings.
 *
 * Conventions: plain pointers and sizes, no C++/torch types; every function returns a
 * vfb_status (0 = ok); on failure vfb_last_error() (thread-local) describes it.  Device
 * pointers are CUDA device addresses in the calling process's primary context.  There is
 * no CPU fallback anywhere behind this interface: without a CUDA device every compute
 * entry point fails with VFB_ERR_CUDA.
 */
#ifndef VFIND_B200_H
#define VFIND_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VFB_ABI_VERSION 1

typedef enum vfb_status {
    VFB_OK = 0,
    VFB_ERR_VALUE = 1,   /* -> Python ValueError   (src/lib.rs:107-109)                     */
    VFB_ERR_IO = 2,      /* -> Python OSError      (File::open `?`, src/lib.rs:233)          */
    VFB_ERR_FORMAT = 3,  /* malformed gzip/FASTQ: the reference panics (src/lib.rs:308)      */
    VFB_ERR_CUDA = 4,    /* CUDA runtime failure / no device                                 */
    VFB_ERR_ARG = 5,     /* bad argument to this ABI (null pointer, unsupported size)        */
    VFB_ERR_NOMEM = 6
} vfb_status;

#define VFB_NONE 0xFFFFFFFFu

/* Arguments of find_variants (src/lib.rs:219-231), in the reference's order, followed by
 * GPU-side knobs that the reference does not have (all optional, 0 = default). */
typedef struct vfb_params {
    uint32_t struct_size;             /* sizeof(vfb_params), for ABI evolution              */
    const uint8_t *prefix;            /* adapters.0                      src/lib.rs:221     */
    uint64_t prefix_len;
    const uint8_t *suffix;            /* adapters.1                                          */
    uint64_t suffix_len;
    int32_t match_score;              /* :222 */
    int32_t mismatch_score;           /* :223 */
    int32_t gap_open_penalty;         /* :224 (positive = penalty, README.md:137-138)       */
    int32_t gap_extend_penalty;       /* :225 */
    double accept_prefix_alignment;   /* :226 */
    double accept_suffix_alignment;   /* :227 */
    uint32_t n_threads;               /* :228 host ingest threads (inflate/parse)           */
    uint64_t queue_len;               /* :229 batches in flight                             */
    int32_t skip_translation;         /* :230 */
    int32_t show_progress;            /* :231 stored; the reference's spinner is never ticked — progress is
                                         reported through vfb_set_progress                                */
    /* ---- additions ---- */
    int32_t device;                   /* CUDA ordinal; -1 = current device                  */
    int32_t diagnostics;              /* keep per-read diagnostics of the last batch        */
    uint64_t batch_reads;             /* max reads per device batch (0 = 8 Mi)              */
    uint64_t batch_bytes;             /* max text bytes per device batch (0 = 2 GiB)        */
    uint64_t table_capacity_hint;     /* expected distinct variants (0 = grow on demand)    */
    int32_t debug_hash_bits;          /* tests only: keep this many hash bits (0 = all 64)  */
    int32_t force_generic_dp;         /* tests only: use the unpacked fallback DP kernel    */
    int32_t dp_compute_all;           /* 1 = run the suffix DP even when the prefix failed
                                         (what the reference does, src/lib.rs:278-286; the
                                         result table is identical either way)              */
    int32_t force_general_scan;       /* tests only: use the byte-wise scan kernel          */
    int32_t dp_mode;                  /* 0 = auto (windowed DP where its filter applies, full DP in
                                         diagnostics mode), 1 = always the full DP, 2 = windowed DP even
                                         in diagnostics mode (scores of rejected alignments are then
                                         lower bounds or absent)                              */
    int32_t debug_win_cap;            /* tests only: > 0 caps the window list of the windowed DP   */
    int32_t both_strands;             /* 1 = a read without a region (start, end located, start < end <= len) is
                                         searched once more as its reverse complement; a region found there is
                                         counted in the same table (at most one strand counts per read)       */
    double collapse_ratio;            /* 0 = off; else (finite, >= 1) vfb_finish folds every key into a more abundant key of
                                         the same length one byte substitution away, as vfb_collapse does, before the
                                         table leaves the device (the count table itself keeps every key)               */
} vfb_params;

/* One read inside a text buffer: text[off .. off+len). */
typedef struct vfb_span {
    uint32_t off;
    uint32_t len;
} vfb_span;

/* Per-read diagnostics, field-compatible with the oracle's vfo_read_diag. */
typedef struct vfb_read_diag {
    int32_t exact_prefix;   /* leftmost exact position or -1         src/lib.rs:148   */
    int32_t exact_suffix;
    int32_t score_prefix;   /* DP score; INT32_MIN when no DP ran    src/lib.rs:156   */
    int32_t len_prefix;     /* DP length statistic; -1 when no DP    src/lib.rs:159   */
    int32_t score_suffix;
    int32_t len_suffix;
    int32_t start;          /* region boundaries or -1               src/lib.rs:278-286 */
    int32_t end;
} vfb_read_diag;

/* The result: HashMap<String,u64> unzipped to columns (src/lib.rs:312-317), Arrow-style.
 * Row i is data[offsets[i] .. offsets[i+1]) with counts[i].  Row order is unspecified. */
typedef struct vfb_table {
    uint64_t rows;
    uint64_t key_bytes;
    uint64_t *offsets;      /* rows + 1 */
    uint8_t *data;          /* key_bytes */
    uint64_t *counts;       /* rows */
    void *owner;            /* non-null: the columns live in pinned memory owned by that context
                               and stay valid until its next vfb_finish / vfb_destroy */
} vfb_table;

/* Arrow C Data Interface structs (the stable ABI of the Apache Arrow specification), declared here so that
 * callers need no Arrow headers. */
typedef struct vfb_arrow_schema {
    const char *format, *name, *metadata;
    int64_t flags, n_children;
    struct vfb_arrow_schema **children, *dictionary;
    void (*release)(struct vfb_arrow_schema *);
    void *private_data;
} vfb_arrow_schema;
typedef struct vfb_arrow_array {
    int64_t length, null_count, offset, n_buffers, n_children;
    const void **buffers;
    struct vfb_arrow_array **children, *dictionary;
    void (*release)(struct vfb_arrow_array *);
    void *private_data;
} vfb_arrow_array;

typedef struct vfb_stats {
    uint64_t reads;             /* reads submitted since create/reset                  */
    uint64_t dp_prefix;         /* prefix alignments performed                         */
    uint64_t dp_suffix;
    uint64_t dp_cells;          /* sum of adapter_len * read_len over alignments       */
    uint64_t counted;           /* reads that contributed to the table                 */
    uint64_t unique;            /* distinct keys                                       */
    uint64_t text_bytes;        /* sum of read lengths                                 */
    uint64_t kernel_launches;   /* kernels launched by this library since create/reset */
    uint64_t h2d_bytes;
    uint64_t d2h_bytes;
    /* device time per stage in ms (CUDA events on the compute stream), summed over
     * batches; only filled when vfb_set_profiling(ctx, 1). */
    double ms_scan, ms_worklist, ms_dp, ms_translate, ms_count, ms_total;
    uint64_t dp_kernel_launches;
    int32_t dp_kernel_kind;     /* 1 = packed DPX kernel, 2 = generic fallback, 3 = windowed packed DPX */
    int32_t reserved;
    uint64_t dp_cells_computed; /* cells the DP kernels actually evaluated (== dp_cells for the full DP) */
    uint64_t dp_windows;        /* windows the filter produced (windowed DP)            */
    double ms_dp_filter, ms_dp_window;   /* parts of ms_dp: k2_filter and k2_dp_window (profiling only) */
    uint64_t fused_batches;     /* batches whose key kernel probed the count table itself (k34_keys_count)   */
    uint64_t fused_hits;        /* counted reads whose key never left the key kernel (row already in the table) */
    uint64_t reverse_reads;     /* both_strands: reads searched as their reverse complement                  */
    uint64_t reverse_counted;   /* both_strands: reads counted from the reverse strand                       */
} vfb_stats;

typedef struct vfb_ctx vfb_ctx;

const char *vfb_last_error(void);
int vfb_abi_version(void);

/* Fill *p with the reference's defaults (src/lib.rs:169-182). */
void vfb_default_params(vfb_params *p);

/* Setup half of find_variants (src/lib.rs:236-261): validates both thresholds
 * (VFB_ERR_VALUE with the reference's message), builds the adapter profiles, converts
 * `thr * match * len` (evaluated in f64 exactly as :260-261) to integer accept bounds. */
int vfb_create(const vfb_params *p, vfb_ctx **out);
int vfb_destroy(vfb_ctx *ctx);

/* Clear the count table and the statistics (keeps allocations). */
int vfb_reset(vfb_ctx *ctx);
int vfb_set_profiling(vfb_ctx *ctx, int enabled);

/* Progress of vfb_run_file (the reference creates an indicatif spinner when show_progress is set but never
 * ticks it, src/lib.rs:265-269, :310; here the flag can mean something).  The callback runs on the thread that
 * is inside vfb_run_file, at most about ten times per second and once at the end: records queued so far,
 * compressed bytes consumed so far, compressed size of the file. */
typedef void (*vfb_progress_fn)(uint64_t records, uint64_t bytes_done, uint64_t bytes_total, void *user);
int vfb_set_progress(vfb_ctx *ctx, vfb_progress_fn fn, void *user);

/* The per-read hot loop (worker + reducer closures, src/lib.rs:275-306) over a batch of
 * reads held in HOST memory: host->device copies happen inside.  `text`/`spans` may be
 * pageable or pinned.  Asynchronous: pageable input is staged before the call returns; PINNED input is
 * copied straight from the caller's buffer by the copy engine, so it must stay unmodified until vfb_sync /
 * vfb_finish (or until two further submits have returned: two batches are in flight at most).
 * A span is text[off .. off+len) and must lie inside the buffer (VFB_ERR_ARG otherwise); spans may overlap or
 * repeat. */
int vfb_submit_host(vfb_ctx *ctx, const uint8_t *text, uint64_t text_bytes,
                    const vfb_span *spans, uint64_t n_reads);

/* Same, reads already resident in device memory (any size: split internally).  The spans are validated on the
 * device (one small kernel and an 16-byte read-back per batch). */
int vfb_submit_device(vfb_ctx *ctx, const uint8_t *d_text, uint64_t text_bytes,
                      const vfb_span *d_spans, uint64_t n_reads);

/* Whole find_variants ingest (src/lib.rs:233-234, :271-308): gzip (multi-member) FASTQ
 * file -> inflate -> parse -> batches -> the hot loop.  VFB_ERR_IO if it cannot be
 * opened, VFB_ERR_FORMAT on malformed gzip/FASTQ. */
int vfb_run_file(vfb_ctx *ctx, const char *path, uint64_t *n_reads);

/* vfb_run_file with input options.  VFB_INPUT_ALLOW_TEXT: a file that does not start with the gzip magic is read
 * as uncompressed FASTQ text (the reference accepts gzip only and panics on anything else, src/lib.rs:233, :308 —
 * which is what vfb_run_file and flags = 0 do).  May be called for several files on one context: the table
 * accumulates across calls (SURVEY §8(f) next-4: plain-text and multi-file front-ends). */
#define VFB_INPUT_ALLOW_TEXT 1u
int vfb_run_file_ex(vfb_ctx *ctx, const char *path, uint32_t flags, uint64_t *n_reads_out);

/* Host-only front half of vfb_run_file (no GPU needed): inflate `path` chunk by chunk exactly as
 * the ingest does (serial gzip, or member-parallel on n_threads for block-gzip/BGZF input) and
 * return the submitted text, the complete lines in it and the number of chunks.  `out` may be
 * NULL to only count.  For tests of the inflate / cut / carry logic. */
int vfb_debug_inflate_file(const char *path, uint32_t n_threads, uint8_t *out, uint64_t out_cap,
                           uint64_t *n_bytes, uint64_t *n_lines, uint64_t *n_chunks);

int vfb_sync(vfb_ctx *ctx);

/* Use the caller's CUDA stream (a cudaStream_t) as the context's compute stream, so that the caller's events and
 * collectives order with the library's work.  The caller keeps ownership of the stream.
 *
 * Streams: the hot loop of consecutive batches runs on two internal LANE streams (the ALU-bound alignment kernels of
 * one batch share the SMs with the memory-bound scan / key / count kernels of its neighbours).  A lane forks from
 * the compute stream when its batch is submitted — whatever the caller queued there before (a kernel that
 * produces the reads, say) is seen — and is joined back by vfb_sync, vfb_finish, the merge calls, vfb_table_clear
 * and vfb_fence.  A caller that records its own events or queues its own consumers on the compute stream calls
 * vfb_fence first: it makes the compute stream wait (on the device, not the host) for everything submitted so
 * far.  vfb_set_lanes(ctx, 1) runs every batch on the compute stream itself (the round-1 behaviour; per-stage
 * profiling times are only meaningful then). */
int vfb_set_compute_stream(vfb_ctx *ctx, void *stream);
int vfb_fence(vfb_ctx *ctx);
int vfb_set_lanes(vfb_ctx *ctx, int n_lanes);

/* `variants.into_iter().unzip()` (src/lib.rs:312): waits for all batches, compacts the
 * table into Arrow-style columns on the device and copies them into pinned host buffers
 * owned by the context (see vfb_table.owner).  Call vfb_table_free when done with the
 * view.  The context stays usable. */
int vfb_finish(vfb_ctx *ctx, vfb_table *out);
void vfb_table_free(vfb_table *t);

/* vfb_finish, exported as one Arrow struct array {sequence: large_utf8, count: uint64} (= the DataFrame of
 * src/lib.rs:312-319) over the pinned host columns themselves: zero copies.  The pinned buffers leave the context
 * and are released (to the pinned pool) by the array's release callback, so the result outlives the context. */
int vfb_finish_arrow(vfb_ctx *ctx, vfb_arrow_array *out_array, vfb_arrow_schema *out_schema);

int vfb_get_stats(vfb_ctx *ctx, vfb_stats *out);

/* collapse_ratio (directional clustering of sequencing errors).  Rows are ordered by count descending, then key bytes
 * ascending (unsigned).  Key a may be the parent of key b when both have the same length and differ in exactly one byte,
 * a comes first in the order and (double)count(a) >= ratio * (double)count(b) (one IEEE multiply, no FMA).  parent(b)
 * is the first such a; every row's count goes to the end of its parent chain, and only those roots are returned.
 * Rows with count 0 take no part and are not returned.  Wrong for libraries whose true members are one substitution
 * apart (single-mutant scans): the most abundant member absorbs its neighbours.
 *
 * What the last collapsing finish did: rows with a non-zero count before, roots after, and ms = elapsed time on the
 * device stream from the first collapse kernel to the last (the host waits between some launches for a 4-byte flag, and
 * that wait is included).  All zero until a finish has collapsed.  A collapse takes at most 2^29 rows with a count
 * (VFB_ERR_ARG beyond). */
typedef struct vfb_collapse_info {
    uint64_t rows_in;
    uint64_t rows_out;
    double ms;
} vfb_collapse_info;
int vfb_get_collapse_info(vfb_ctx *ctx, vfb_collapse_info *out);

/* The same collapse over host columns (in->data holds in->key_bytes bytes, offsets[0] <= ... <= offsets[rows] <=
 * key_bytes; owner ignored): uploaded to `device` (-1 = current), collapsed and compacted there, downloaded into malloc'd
 * columns (out->owner = NULL; vfb_table_free frees them).  Counts must be below 2^56.  VFB_ERR_VALUE for a ratio that is
 * not a finite number >= 1 and for a key that appears twice.  debug_hash_bits: tests only, as in vfb_params.  `info`
 * may be NULL. */
int vfb_collapse(const vfb_table *in, double ratio, int device, int debug_hash_bits, vfb_table *out, vfb_collapse_info *info);

/* umi_length: count distinct molecules per variant from a UMI inside the read.  The UMI of a counted read is bytes
 * [umi_offset, umi_offset + umi_length) of the read in the orientation its region was found in (the read as submitted,
 * or its reverse complement for a read counted by the both_strands reverse pass), compared as raw bytes.  The key
 * kernels append it to the key, so the table counts (variant, UMI) pairs; vfb_finish groups them by variant on the
 * device and returns one row per variant with count = reads and molecules = distinct UMIs ("unique" method: no error
 * correction, a UMI with a sequencing error is one more molecule).  A read with a key that is shorter than
 * umi_offset + umi_length is not counted (vfb_umi_info.reads_short).
 *
 * vfb_set_umi: umi_length 0 = off (the default), at most 64; umi_offset + umi_length <= 65536; an offset needs a length.
 * Only while the table is empty (after vfb_create, vfb_reset or vfb_table_clear): VFB_ERR_ARG otherwise.  VFB_ERR_VALUE
 * for bad values and with collapse_ratio set (not supported together).  Validated before any device use.  Every context
 * of a merge must use the same setting: with UMIs on, a row's owner is owner(hash(variant bytes)), so all rows of one
 * variant land on one part. */
int vfb_set_umi(vfb_ctx *ctx, uint32_t umi_offset, uint32_t umi_length);
/* pairs: distinct (variant, UMI) rows grouped by the last finish; rows_out: variant rows it returned; reads_short:
 * reads dropped for a short UMI since create or reset; ms: device time of the group-by, measured as
 * vfb_collapse_info.ms is. */
typedef struct vfb_umi_info {
    uint64_t pairs;
    uint64_t rows_out;
    uint64_t reads_short;
    double ms;
} vfb_umi_info;
int vfb_get_umi_info(vfb_ctx *ctx, vfb_umi_info *out);
/* The molecules column of the last vfb_finish (pinned, rows entries aligned with its rows), owned and invalidated as the
 * table's columns are.  VFB_ERR_ARG when UMIs are off.  vfb_finish_arrow returns it as a third child
 * `molecules: uint64`. */
int vfb_get_molecules(vfb_ctx *ctx, const uint64_t **col);

/* Diagnostics of the most recent batch (requires params.diagnostics = 1 and that the
 * last submit was a single batch).  Parity tests compare these with the oracle. */
int vfb_get_diag(vfb_ctx *ctx, vfb_read_diag *out, uint64_t n_reads);
/* both_strands: the diagnostics of the reverse-complement pass over the same batch, in the batch's read order.  Reads
 * that were not retried (they have a forward region, or are empty) carry the "absent" markers: positions and
 * boundaries -1, scores INT32_MIN, lengths -1.  Positions refer to the reverse complement of the read. */
int vfb_get_diag_reverse(vfb_ctx *ctx, vfb_read_diag *out, uint64_t n_reads);

/* ---- multi-GPU (no reference equivalent; SURVEY §8(e)) ----
 * Reads shard across devices with no data-path collective; the only exchange is the final merge of the per-device
 * tables.  Keys are owned by part = owner(hash(key)) in [0, n_parts).
 *
 * (1) One process, several devices: a vfb_multi is one context per device behind one handle.  vfb_multi_run_file
 * deals the file's block-gzip segments (or inflated chunks) round robin to the devices; vfb_multi_finish merges
 * the tables over peer copies (NVLink) — every device keeps the keys it owns and receives the others' counts for
 * them — and returns ONE table, each device writing its partition into its piece of the host columns.  This is what
 * find_variants(path, ..., devices=[...]) calls.  devices = NULL / n_devices = 0 means all visible devices.
 * vfb_multi_ctx gives the per-device contexts for vfb_submit_host / vfb_submit_device. */
typedef struct vfb_multi vfb_multi;
int vfb_device_count(void);            /* visible CUDA devices (0 without a driver) */
int vfb_multi_create(const vfb_params *p, const int32_t *devices, uint32_t n_devices, vfb_multi **out);
int vfb_multi_destroy(vfb_multi *m);
uint32_t vfb_multi_devices(const vfb_multi *m);
vfb_ctx *vfb_multi_ctx(vfb_multi *m, uint32_t i);
int vfb_multi_run_file(vfb_multi *m, const char *path, uint32_t flags, uint64_t *n_reads);
int vfb_multi_set_progress(vfb_multi *m, vfb_progress_fn fn, void *user);
int vfb_multi_sync(vfb_multi *m);
int vfb_multi_reset(vfb_multi *m);
int vfb_multi_merge(vfb_multi *m);      /* afterwards context i holds exactly the keys it owns, with global counts */
int vfb_multi_finish(vfb_multi *m, vfb_table *out);          /* merge + export; columns owned by m            */
int vfb_multi_finish_arrow(vfb_multi *m, vfb_arrow_array *out_array, vfb_arrow_schema *out_schema);
int vfb_multi_get_stats(vfb_multi *m, vfb_stats *out);       /* summed over the devices                       */
/* With collapse_ratio set, vfb_multi_finish* collapse the merged table on the first device (the merge partitions keys by
 * hash, so neighbours sit on different devices); this reports that collapse. */
int vfb_multi_get_collapse_info(vfb_multi *m, vfb_collapse_info *out);
/* umi_length on every device (vfb_set_umi).  Each device groups the variants it owns after the merge and writes its
 * piece of the columns, molecules included; the info is summed over the devices (ms: the largest). */
int vfb_multi_set_umi(vfb_multi *m, uint32_t umi_offset, uint32_t umi_length);
int vfb_multi_get_umi_info(vfb_multi *m, vfb_umi_info *out);
int vfb_multi_get_molecules(vfb_multi *m, const uint64_t **col);

/* (2) One process per device (torchrun, MPI): the same keep-your-own-keys merge over NCCL send/recv, queued on the
 * context's compute stream, one host synchronisation.  libnccl.so.2 is loaded at run time (VFB_NCCL_LIB names
 * another path); the communicator comes from a 128-byte id made on one rank and carried to the others by the
 * caller's control plane.  `comm` is an ncclComm_t (vfb_nccl_comm_init, or the caller's own). */
int vfb_nccl_available(void);
int vfb_nccl_unique_id(uint8_t *id128);
int vfb_nccl_comm_init(const uint8_t *id128, uint32_t n_ranks, uint32_t rank, int device, void **comm_out);
int vfb_nccl_comm_destroy(void *comm);
int vfb_merge_nccl(vfb_ctx *ctx, void *comm, uint32_t rank, uint32_t n_ranks);
/* (NCCL ranks collapse nothing themselves: the gathered result goes through vfb_collapse.) */

/* (3) Any other transport: export the local table as n_parts self-describing chunks in device memory (every row,
 * the rank's own included), exchange them, clear, absorb the received chunks (the round-1 interface; the gloo
 * tests drive it). */
int vfb_table_partition_sizes(vfb_ctx *ctx, uint32_t n_parts, uint64_t *chunk_bytes /* n_parts */);
int vfb_table_partition_fill(vfb_ctx *ctx, uint32_t n_parts, uint8_t *d_buf,
                             const uint64_t *chunk_offsets /* n_parts */);
int vfb_table_clear(vfb_ctx *ctx);
int vfb_table_absorb(vfb_ctx *ctx, const uint8_t *d_chunk, uint64_t chunk_bytes);
/* The key hash the table and the partitioning use, and the owner rule (host functions). */
uint64_t vfb_hash_key(const uint8_t *key, uint32_t len);
uint32_t vfb_key_owner(uint64_t hash, uint32_t n_parts);
/* Host-side view of a chunk (for CPU tests of the exchange plumbing). */
int vfb_chunk_rows(const uint8_t *h_chunk, uint64_t chunk_bytes, uint64_t *rows);

/* ---- synthetic reads (bench + tests; BASELINE.json configs, SURVEY §8(d)) ---- */
typedef struct vfb_synth_cfg {
    uint64_t seed;
    uint32_t read_len;        /* L */
    uint32_t adapter_len;     /* A (both adapters) */
    uint32_t region_len;      /* V, multiple of 3 */
    uint32_t n_variants;      /* U library size */
    uint32_t zipf;            /* 1 = octave-Zipf(s~1) over the library, 0 = uniform */
    uint32_t p_err_ppm;       /* per-adapter probability of being mutated, in 1e-6 */
    uint32_t indel_ppm;       /* probability that one edit is an indel, in 1e-6 (rest substitutions) */
    uint32_t force_indel;     /* 1 = first edit of a mutated adapter is always an indel (config #3) */
    uint32_t frameshift_ppm;  /* fraction of library entries with V±1 */
    uint32_t noise_ppm;       /* per-base substitution noise inside the region */
    uint32_t n_ppm;           /* per-base probability of an 'N' inside the region */
    uint32_t reserved;
} vfb_synth_cfg;

/* The two adapters the generator embeds (deterministic in cfg->seed). */
int vfb_synth_adapters(const vfb_synth_cfg *cfg, uint8_t *prefix, uint8_t *suffix);
/* Reads [first, first+n) as fixed-stride records: text[i*read_len ..), spans[i] = {i*read_len, read_len}.
 * Host and device produce identical bytes. */
int vfb_synth_host(const vfb_synth_cfg *cfg, uint64_t first, uint64_t n, uint8_t *text, vfb_span *spans);
int vfb_synth_device(const vfb_synth_cfg *cfg, uint64_t first, uint64_t n, uint8_t *d_text,
                     vfb_span *d_spans, int device);

/* ---- measurement helpers ---- */
/* Dependent-free integer microbenchmark on `device`: peak lane-ops/s of the INT32 ALU
 * pipe (IADD3/VIADDMNMX mix) and of ALU+FMA-pipe dual issue (IADD3 + IMAD).  Giga-ops/s. */
int vfb_measure_int_peak(int device, double *alu_gops, double *dual_gops);

/* Test hook for the GPU inflater: `members` holds n_members x {z_off, z_len, out_off, isize}
 * (uint32 each) describing whole gzip members inside z; the text lands in out.  *first_bad is
 * the first member that failed (bad deflate data, CRC-32 or ISIZE mismatch) or 0xFFFFFFFF. */
int vfb_debug_gpu_inflate(const uint8_t *z, uint64_t z_bytes, const uint32_t *members, uint32_t n_members,
                          uint8_t *out, uint64_t out_bytes, int device, uint32_t *first_bad, double *kernel_ms);

/* Test hook for the arithmetic fast path of the key kernel's translate (src/lib.rs:16-44): runs the HOST build of
 * the code the kernel uses (csrc/translate_fast.h) on twelve bases; aa receives four amino acids, *canonical is 1
 * when all twelve bytes are A/C/G/T/U of either case (only then does the kernel take this path). No GPU needed. */
int vfb_debug_translate12(const uint8_t *bases12, uint8_t *aa4, int *canonical);

/* Test hook for both_strands: the reverse complement the device gather writes (csrc/kernels_strand.cu, host build of
 * the same base map): out[i] = complement(in[n-1-i]), A<->T, C<->G, a<->t, c<->g, U->A, u->a, other bytes unchanged. */
int vfb_debug_revcomp(const uint8_t *in, uint64_t n, uint8_t *out);

/* Test hook for the windowed alignment path (what vfb_create decides for one adapter; no GPU needed): *accept_bound
 * receives the integer T with score >= T <=> score as f64 > accept_alignment * match_score * adapter_len
 * (src/lib.rs:157, :260-261), *max_edits the K of csrc/kernels_dpw.cu — the most edits an alignment with score >= T can
 * hold — or -1 when the edit-distance filter does not apply (non-positive edit costs, adapter > 64, 3K > adapter_len). */
int vfb_debug_window_plan(int32_t match_score, int32_t mismatch_score, int32_t gap_open_penalty, int32_t gap_extend_penalty,
                          uint32_t adapter_len, double accept_alignment, int32_t *accept_bound, int32_t *max_edits);

/* The packed DP word vfb_create picks for one adapter (csrc/kernels_dp.cu, DpLayout), so that a model of the DP
 * kernels can run on the library's own constants. */
typedef struct vfb_dp_layout_info {
    int32_t packed;           /* 1 = a packed kernel runs (the fields below are set), 0 = the unpacked one */
    int32_t max_edits;        /* K of the windowed path, -1 = the full-matrix kernel runs */
    int32_t accept_bound;     /* T: accept iff score >= T */
    uint32_t lcap;            /* longest read the packed kernels take; longer ones go to the unpacked kernel */
    int32_t S0, LB, XB;       /* score << S0 | q << (LB+XB) | x << LB | len */
    int32_t c_eopen, c_eext, c_fopen, c_fext;
    int32_t hmask, lowmask, lenmask;
    int32_t neg_e, neg_f;
    int32_t w_match, w_mismatch, w_wild;
} vfb_dp_layout_info;

/* What vfb_create decides for one adapter of a context without diagnostics (or with dp_mode 2) when dp_mode != 1,
 * and the full-matrix choice when dp_mode == 1.  Host code only, no GPU needed. */
int vfb_debug_dp_layout(int32_t match_score, int32_t mismatch_score, int32_t gap_open_penalty, int32_t gap_extend_penalty,
                        uint32_t adapter_len, double accept_alignment, int32_t dp_mode, vfb_dp_layout_info *out);

/* Pinned host memory for callers without their own allocator. */
int vfb_host_alloc(void **p, uint64_t bytes);
int vfb_host_free(void *p);

/* Pinned staging buffers (ingest segments, result columns) are cached process-wide between calls,
 * because page-locking costs more than a small run; this frees the cache (VFB_PINNED_POOL_MB caps it,
 * default 4096). */
int vfb_pinned_pool_trim(void);
/* Device buffers are cached the same way (cudaMalloc / cudaFree cost milliseconds apiece; VFB_DEVICE_POOL_MB caps
 * the cache per device, default 24576). */
int vfb_device_pool_trim(void);

#ifdef __cplusplus
}
#endif
#endif
