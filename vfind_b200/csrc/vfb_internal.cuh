// Internal declarations shared by the kernels and the host API (not part of the C ABI).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>

#include "../../include/vfind_b200.h"

#define VFB_MAX_PACKED_ADAPTER 64   // longest adapter the register-resident DP kernel takes
#define VFB_MAX_ADAPTER 1024        // longest adapter the fallback DP kernel takes
#define VFB_MAX_SCAN_ADAPTER 256    // adapters are passed by value to the scan kernel

namespace vfb {

void set_error(const std::string &msg);
// VFB_TRACE=1: timestamped lines on stderr (allocations, table growth, ingest phases)
bool trace_on();
void trace(const char *fmt, ...);
int cuda_fail(cudaError_t e, const char *what, const char *file, int line);
// process-wide cache of pinned host buffers (api.cu)
void *pinned_acquire(size_t want, size_t *cap_out);
void pinned_release(void *p, size_t cap);
void pinned_pool_trim();

#define VFB_CUDA(call)                                                         \
    do {                                                                       \
        cudaError_t e__ = (call);                                              \
        if (e__ != cudaSuccess) return vfb::cuda_fail(e__, #call, __FILE__, __LINE__); \
    } while (0)

// ---------------------------------------------------------------- adapters
struct AdapterBytes {
    uint8_t b[VFB_MAX_SCAN_ADAPTER];
    uint32_t len;
};

// Read-base / adapter-base codes of the alignment alphabet: parasail Matrix::create(b"ATCG")
// (/root/reference/src/lib.rs:236) is case-insensitive; everything else is the wildcard.
__host__ __device__ __forceinline__ int dp_code(uint8_t c)
{
    switch (c) {
    case 'A': case 'a': return 0;
    case 'C': case 'c': return 1;
    case 'G': case 'g': return 2;
    case 'T': case 't': return 3;
    default: return 4;
    }
}

// ---------------------------------------------------------------- packed DP word layout
// One 32-bit word carries (score | q | x | len), low to high: len [0,LB), x [LB,LB+XB),
// q [LB+XB, LB+XB+2), score [S0,32).  Signed integer comparison of two words compares the
// scores first, then the transient priority fields, so one VIMNMX3 / VIADDMNMX selects the
// winner of a cell under parasail's tie rules and carries its alignment length along:
//   q: source priority inside H = max(D,F,E): diag 2 > F 1 > E 0
//   x: number of consecutive gap extensions; an extension (x>=1) beats an opening (x=0)
//      at equal score ("tie -> extend").
struct DpLayout {
    int S0, LB, XB;
    int c_eopen, c_eext;   // E: H_left + c_eopen  vs  E_left + c_eext
    int c_fopen, c_fext;   // F: H_up + c_fopen    vs  F_up + c_fext   (both carry q=1)
    int hmask;             // clears q and x after the H max
    int lowmask;           // (1<<S0)-1
    int lenmask;           // (1<<LB)-1
    int neg_e, neg_f;      // border values of E and F ("-inf")
    int w_match, w_mismatch, w_wild;   // diagonal increments incl. +1 length and q=2
    int one;               // the constant 1 (opaque to the compiler: keeps adds on the FMA pipe)
};

struct DpScoring {
    int match, mismatch, open, extend;
};

// Returns false if the parameters do not fit the packed layout (then the fallback runs).  `windowed`: sized for
// the windowed DP too, whose windows start from a -inf border and so reach lower scores than the full matrix.
bool make_dp_layout(const DpScoring &s, uint32_t adapter_len, bool windowed, DpLayout *out);

struct DpJob {
    const uint8_t *text;
    const vfb_span *spans;
    const uint32_t *worklist;     // read indices needing this alignment
    const uint32_t *n_items;      // device counter
    uint32_t *bound;              // start[] (prefix) or end[] (suffix): written on accept
    int32_t *diag_score;          // nullable, indexed by read
    int32_t *diag_len;
    unsigned long long *cells;    // device counter: sum A*L over alignments
    // prefix pass only: reads it accepts whose suffix is still missing go on the suffix worklist
    uint32_t *next_list, *n_next;
    const uint32_t *other_bound;
    int is_prefix;
    int min_accept;               // accept iff score >= min_accept
    uint32_t adapter_len;
    uint8_t adapter_code[VFB_MAX_PACKED_ADAPTER];
};

// Longest read the layout can take; longer items are appended to `fallback`.
uint32_t dp_lcap(const DpLayout &lay, uint32_t adapter_len, int extend);
int launch_dp_packed_ex(const DpJob &job, const DpLayout &lay, uint32_t lcap, uint32_t *fallback,
                        uint32_t *n_fallback, int sm_count, cudaStream_t st);

// Windowed DP (kernels_dpw.cu): bit-parallel filter -> DP on the flagged windows -> resolve.
// K = dpw_max_edits(...) >= 0 when the filter applies to this adapter / scoring / bound.
int dpw_max_edits(const DpScoring &s, uint32_t adapter_len, int min_accept);
uint32_t dpw_item_bytes();
int launch_dp_windowed(const DpJob &job, const DpLayout &lay, int K, uint32_t lcap, uint32_t max_items,
                       void *wins, uint32_t *n_wins, uint32_t win_cap, unsigned long long *best_key,
                       unsigned long long *cb_val, uint32_t *fallback, uint32_t *n_fallback,
                       unsigned long long *cells_computed, uint32_t *work_cursors /* [0] and [32], zeroed */, int sm_count, cudaStream_t st,
                       cudaEvent_t ev_filter_done = nullptr, cudaEvent_t ev_windows_done = nullptr);

struct DpGenericJob {
    DpJob base;
    const uint8_t *d_adapter_code;   // adapter codes in device memory (any length)
    DpScoring sc;
    int32_t *scratch;                // 4 * adapter_len * n_threads ints
    uint32_t n_threads;
};
int launch_dp_generic(const DpGenericJob &job, int sm_count, cudaStream_t st);
uint32_t dp_generic_threads(int sm_count);

// ---------------------------------------------------------------- scan + worklist
struct ScanJob {
    const uint8_t *text;
    const vfb_span *spans;
    uint32_t n_reads;
    uint64_t text_bytes;   // bytes of text the spans address (sizes the scan tiles; 0 = unknown)
    uint32_t *start;   // prefix boundary: pos + A, or VFB_NONE
    uint32_t *end;     // suffix boundary: pos, or VFB_NONE
    // DP worklists built by the scan (null = that alignment is disabled)
    uint32_t *list_pre, *n_pre;   // reads without an exact prefix
    uint32_t *list_suf, *n_suf;   // reads without an exact suffix whose prefix is already located
    int compute_all;              // 1: list every suffix miss (what the reference computes)
    int force_general;            // tests: use the byte-wise kernel
};
// Shared-memory tile for 32 reads that sit text_bytes / n_reads apart on average (scan and key kernels), at most
// VFB_TILE_BYTES_MAX.  The tile launchers static_assert that a block of one warp at that size fits
// VFB_SMEM_BLOCK_MAX, the shared memory an sm_100 block may have, so they always launch.
#define VFB_TILE_BYTES_MAX (96u * 1024u)
#define VFB_SMEM_BLOCK_MAX (227u * 1024u)
uint32_t vfb_tile_bytes_for(uint64_t text_bytes, uint32_t n_reads);
int launch_scan(const ScanJob &job, const AdapterBytes &prefix, const AdapterBytes &suffix,
                int sm_count, cudaStream_t st);

// ---------------------------------------------------------------- translate + count
struct KeyJob {
    const uint8_t *text;
    const vfb_span *spans;
    const uint32_t *start, *end;
    uint32_t n_reads;
    uint64_t text_bytes;      // bytes of text the spans address (sizes the tiles; 0 = unknown)
    int skip_translation;
    uint8_t *keys;            // key arena of the batch; keys are bump-allocated, 16-byte aligned
    uint64_t *koff;           // per read: offset of its key in `keys`
    unsigned long long *key_cursor;   // device bump pointer (zeroed per batch)
    uint32_t *klen;           // 0 = no key
    uint64_t *khash;
    int hash_bits;            // 0 = 64
    uint32_t flank_bytes;     // prefix + suffix adapter length: a region is at most a read minus this (sizes key blocks)
};
int launch_keys(const KeyJob &job, cudaStream_t st);
struct DevTable;
// Fused keys + count (k34_keys_count): reads whose key already has a row in `tab` are counted by the key kernel;
// the others are left in job.koff / klen / khash as a compact list of *n_miss entries for launch_insert
// (InsertJob::n_keys_dev).  -1: the tile kernel does not apply to this batch (run launch_keys + launch_insert).
int launch_keys_count(const KeyJob &job, const DevTable &tab, uint32_t *n_miss, cudaStream_t st);

// Open-addressing table in device memory.  A slot is ONE 32-byte sector of four words:
//   [0] (tag << 32 | ref)   tag = high 32 hash bits, ref = row id + 1 (bit31 clear) or, only inside the
//                           insert kernel of the batch that created it, 0x80000000 | batch read index; 0 = empty
//   [1] count               the atomicAdd lands in the sector the probe has just pulled into L2
//   [2] arena offset, [3] key length of the row (written by k4_publish): the key compare needs no
//                           row_off[] / row_len[] look-ups
// Equality is always decided on full key bytes.
#define VFB_SLOT_WORDS 4
struct DevTable {
    unsigned long long *slots;   // capacity * VFB_SLOT_WORDS words
    uint64_t capacity;           // power of two
    // rows (distinct keys), append-only
    uint64_t *row_hash;
    uint64_t *row_off;           // into arena
    uint32_t *row_len;
    uint32_t *row_slot;          // the slot that holds the row's count: export and merge walk rows, not the slot array
    uint64_t row_capacity;
    uint8_t *arena;              // keys, each padded to 16 bytes
    uint64_t arena_capacity;
    // device counters: [0] rows, [1] arena bytes, [2] counted reads
    unsigned long long *counters;
};

struct InsertJob {
    const uint8_t *keys;
    const uint32_t *klen;
    const uint64_t *khash;
    const unsigned long long *kcount;   // nullable: per-key count (absorb); else 1
    const uint64_t *koff;               // nullable: per-key byte offset into keys; else i * key_stride
    uint32_t key_stride;
    uint32_t n_keys;
    const uint32_t *n_keys_dev = nullptr;   // nullable: device word holding the list's true length (<= n_keys)
    uint32_t *owner_slot;               // scratch, n_keys: slot claimed by this key or VFB_NONE
};
int launch_insert(const DevTable &t, const InsertJob &job, cudaStream_t st);
int launch_rehash(const DevTable &old_t, const DevTable &new_t, cudaStream_t st);
int launch_export_counts(const DevTable &t, uint64_t rows, unsigned long long *row_count, cudaStream_t st);
// Export of the rows with a non-zero count, in two passes: sizes (block_bytes / block_rows hold ceil(rows/1024)
// words of scratch each; totals[0] = key bytes, totals[1] = exported rows), then offsets (+ byte_base), counts and
// the keys back to back.
int launch_export_sizes(const DevTable &t, uint64_t rows, const unsigned long long *row_count,
                        unsigned long long *block_bytes, unsigned long long *block_rows, unsigned long long *totals,
                        cudaStream_t st);
int launch_export_gather(const DevTable &t, uint64_t rows, const unsigned long long *row_count,
                         const unsigned long long *block_bytes, const unsigned long long *block_rows,
                         unsigned long long byte_base, unsigned long long *offsets, unsigned long long *counts,
                         uint8_t *data, cudaStream_t st);

// ---------------------------------------------------------------- merge chunks
// Chunk layout (all sections 16-byte aligned):
//   header {magic, rows, key_area_bytes, reserved} u64 x4
//   hash   u64 x rows | count u64 x rows | koff u64 x rows | klen u32 x rows | key area
struct ChunkHeader {
    uint64_t magic, rows, key_bytes, reserved;
};
#define VFB_CHUNK_MAGIC 0x5646423230304b31ull
__host__ __device__ __forceinline__ uint64_t vfb_align16(uint64_t x) { return (x + 15) & ~15ull; }
__host__ __device__ __forceinline__ uint64_t chunk_bytes_for(uint64_t rows, uint64_t key_bytes)
{
    return sizeof(ChunkHeader) + vfb_align16(rows * 8) * 3 + vfb_align16(rows * 4) + vfb_align16(key_bytes);
}
// `self` < n_parts: rows owned by that part stay where they are (keep-own merge); self >= n_parts: every row
// with a non-zero count is exported.  `release`: the rows written to a chunk give up their count (they keep their
// slot, so a later read with the same key finds the row again).
int launch_partition_count(const DevTable &t, uint64_t rows, uint32_t n_parts,
                           uint32_t self, unsigned long long *part_rows, unsigned long long *part_keybytes,
                           cudaStream_t st);
int launch_partition_fill(const DevTable &t, uint64_t rows, uint32_t n_parts, uint32_t self, bool release,
                          uint8_t *buf, const uint64_t *d_chunk_off, const uint64_t *d_part_rows,
                          const uint64_t *d_part_keybytes, unsigned long long *cursors,
                          cudaStream_t st);

// ---------------------------------------------------------------- FASTQ parse (ingest)
// d_text holds n_lines complete lines (n_records = n_lines / 4 records, text starts at a record
// boundary, every line ends with a newline).  tile_scratch: parse_tile_words(n_bytes) u64.
int launch_parse(const uint8_t *d_text, uint32_t n_bytes, uint32_t n_lines, uint32_t n_records,
                 unsigned long long *tile_scratch, uint32_t *line_end, vfb_span *spans, uint32_t *err,
                 cudaStream_t st);
uint64_t parse_tile_words(uint32_t n_bytes);
// Split form for text inflated on the device (the host learns the line count in between).  d_text is 16-byte
// aligned; its first `skip` (< 16) bytes are not part of the text (they are neither counted nor framed).
int launch_parse_count(const uint8_t *d_text, uint32_t n_bytes, uint32_t skip, unsigned long long *tile_scratch, cudaStream_t st);
int launch_parse_index(const uint8_t *d_text, uint32_t n_bytes, uint32_t skip, uint32_t n_lines, uint32_t n_records,
                       const unsigned long long *tile_scratch, uint32_t *line_end, vfb_span *spans, uint32_t *err,
                       uint8_t *tail, uint32_t tail_cap, uint32_t *info, cudaStream_t st);

// ---------------------------------------------------------------- GPU inflate (ingest)
// One block-gzip member: where it sits in the compressed buffer, where its text goes.
struct vfb_member {
    uint32_t z_off, z_len, out_off, isize;
};
// *d_first_bad must be 0xFFFFFFFF before the launch; it receives the smallest failing member.
int launch_inflate(const uint8_t *d_z, const vfb_member *d_members, uint32_t n_members, uint8_t *d_out,
                   uint32_t *d_first_bad, cudaStream_t st);

// ---------------------------------------------------------------- single-stream gzip on the device (kernels_inflate.cu)
// Bit positions are relative to the word-aligned compressed segment d_z32 (at most 2^32 bits = 512 MiB).
#define VFB_GZ_WIN 32768u
#define VFB_GZ_PIECE 65536u        // newline counts come per piece of this many text bytes
#define VFB_GZ_CRC_PIECE 16384u    // CRC-32 values come per piece of this many text bytes
struct vfb_gz_chain_out {          // = GzChainOut
    uint32_t n_live, end_kind, end_bit, reserved;
    unsigned long long total_text;
};
#define VFB_GZ_RES_BYTES 32        // sizeof(GzChunkRes)
int launch_gz_search(const uint32_t *d_z32, uint32_t n_words, uint32_t lo_bit, uint32_t hi_bit, uint32_t *d_cand, uint32_t *d_n_cand,
                     uint32_t cand_cap, uint32_t *d_list, uint32_t list_cap, cudaStream_t st);
int launch_gz_decode(const uint32_t *d_z32, uint32_t n_words, const uint32_t *d_starts, uint32_t n_chunks, uint32_t n_decode,
                     uint16_t *d_out16, uint32_t cap, uint32_t max_span_bits, void *d_res, cudaStream_t st);
int launch_gz_chain(const void *d_res, const uint32_t *d_starts, uint32_t n_chunks, const uint16_t *d_out16, uint32_t cap,
                    uint32_t limit_bit, const uint8_t *d_first_window, uint32_t *d_live, unsigned long long *d_text_off,
                    uint8_t *d_win_store, uint8_t *d_out_window, void *d_out, cudaStream_t st);
int launch_gz_resolve(const uint32_t *d_live, const unsigned long long *d_text_off, uint32_t n_live, unsigned long long total_text,
                      const uint16_t *d_out16, uint32_t cap, const uint8_t *d_win_store, uint8_t *d_text, uint32_t *d_piece_nl,
                      uint32_t *d_piece_crc, int first_window_known, uint32_t *d_flag_unknown, cudaStream_t st);

// ---------------------------------------------------------------- both_strands (kernels_strand.cu)
// Reverse complements of the reads that have no forward region, gathered back to back into `out` (16-byte aligned
// base; the caller keeps 16 readable bytes before it and after the gathered text, which is at most 2^32 - 1 bytes).
// out_spans / src are compact: entry i is the i-th gathered read and its index in the batch.  `cursor` (zeroed before
// the launch) ends as gathered reads << 32 | gathered bytes; *n_gathered is incremented by the gathered reads.
struct StrandJob {
    const vfb_span *spans;
    const uint32_t *start, *end;      // the forward pass's final boundaries
    uint32_t n;
    const uint8_t *text;
    uint8_t *out;
    vfb_span *out_spans;
    uint32_t *src;
    unsigned long long *cursor, *n_gathered;
};
int launch_strand_gather(const StrandJob &job, int sm_count, cudaStream_t st);
// *t64 -= counters[2] (after = false) or += counters[2] (after = true): brackets the reverse pass's counting.
int launch_strand_tally(unsigned long long *t64, const unsigned long long *counters, bool after, cudaStream_t st);

// ---------------------------------------------------------------- misc
int launch_synth(const vfb_synth_cfg &cfg, uint64_t first, uint64_t n, uint8_t *d_text,
                 vfb_span *d_spans, cudaStream_t st);
int measure_int_peak(int device, double *alu_gops, double *dual_gops);
// d_out[0] += sum of span lengths, d_out[1] += spans outside [0, text_bytes)
int launch_span_check(const vfb_span *d_spans, uint64_t n, uint64_t text_bytes, unsigned long long *d_out, cudaStream_t st);

extern thread_local uint64_t g_launches;   // kernels launched by this thread's calls
}  // namespace vfb

// Internal hooks between ingest.cu and api.cu (not part of the C ABI).
// Queue one chunk of inflated FASTQ text held in PINNED host memory: H2D copy, GPU parse, the
// hot loop.  `copied` is recorded on the copy stream once the host buffer may be reused.
int vfb_internal_submit_fastq(vfb_ctx *ctx, const uint8_t *pinned_text, uint64_t n_bytes, uint64_t n_lines,
                              uint64_t record_base, cudaEvent_t copied);
// The same for a chunk whose text is [host_text (pinned, host_len bytes) | dev_text (dev_len bytes in the memory of device
// dev_device)]: the device part is copied device to device (or peer to peer); synchronous for that copy, so the caller may
// let go of dev_text when the call returns.
int vfb_internal_submit_fastq_dev(vfb_ctx *ctx, const uint8_t *host_text, uint64_t host_len, const uint8_t *dev_text, uint64_t dev_len,
                                  int dev_device, uint64_t n_lines, uint64_t record_base, cudaEvent_t copied);
// One segment of block-gzip members, in two phases (api.cu).  begin: the compressed members (pieces of PINNED host
// memory, back to back on the device; members[].z_off counts from the first piece) are copied and inflated on the
// ingest stream — asynchronous; `release(arg)` runs on a driver thread once the pieces have been copied (it must
// not call CUDA).  finish: `carry` (the text after the previous segment's last complete record) goes in front,
// records are framed, the hot loop is queued; synchronous for the values it returns: records processed, the text
// after the last complete record (tail, at most VFB_TAIL_CAP bytes), the first member that failed to inflate
// (UINT32_MAX = none).  Segments of one context finish in the order they began.
#define VFB_TAIL_CAP (16u << 20)
struct vfb_zpiece {
    const uint8_t *p;
    uint64_t len;
};
int vfb_internal_bgzf_begin(vfb_ctx *ctx, const vfb_zpiece *pieces, uint32_t n_pieces, const vfb::vfb_member *members,
                            uint32_t n_members, uint64_t text_bytes, void (*release)(void *), void *release_arg, int *slot);
int vfb_internal_bgzf_finish(vfb_ctx *ctx, int slot, const uint8_t *carry, uint64_t carry_len, uint64_t record_base,
                             uint64_t *n_records, uint8_t *tail, uint64_t *tail_len, uint32_t *bad_member);
// Host threads the ingest may use to inflate block-gzip members in parallel (params.n_threads).
int vfb_internal_ingest_threads(vfb_ctx *ctx);
void vfb_internal_progress(vfb_ctx *ctx, uint64_t records, uint64_t bytes_done, uint64_t bytes_total, bool final);
// After vfb_sync: global index of the first malformed record, or UINT64_MAX.
int vfb_internal_parse_error(vfb_ctx *ctx, uint64_t *first_bad_record);
