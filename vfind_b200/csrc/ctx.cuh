// The context behind the C ABI (struct vfb_ctx) and its buffer types.  Shared by api.cu (one device) and
// multi.cu (several devices in one process); not part of the C ABI.
#pragma once
#include <chrono>
#include <string>
#include <vector>

#include "vfb_internal.cuh"

namespace vfb {

// Process-wide caches of device and pinned host buffers (api.cu): cudaMalloc / cudaFree cost 2-8 ms apiece in
// a process that holds a lot of device memory, page-locking about 1 ms per MB — more than a whole small run.
// Buffers released by a context are kept (VFB_DEVICE_POOL_MB per device, default 24576; VFB_PINNED_POOL_MB,
// default 4096) and handed to the next one; vfb_device_pool_trim() / vfb_pinned_pool_trim() free them.
void *device_acquire(int device, size_t want, size_t *cap_out);
void device_release(int device, void *p, size_t cap);
void device_pool_trim();

struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    int dev = -1;
    int ensure(size_t bytes, bool keep = false, cudaStream_t st = 0)
    {
        if (bytes <= cap) return VFB_OK;
        if (dev < 0) VFB_CUDA(cudaGetDevice(&dev));
        const size_t want = bytes + bytes / 4 + 256;
        size_t ncap = 0;
        void *np = device_acquire(dev, want, &ncap);
        if (!np) {
            set_error("out of device memory allocating " + std::to_string(want) + " bytes");
            return VFB_ERR_NOMEM;
        }
        if (p) {
            if (keep && cap) VFB_CUDA(cudaMemcpyAsync(np, p, cap, cudaMemcpyDeviceToDevice, st));
            // what cudaFree did implicitly: nothing queued anywhere on the device may still use the old buffer
            // when it goes back to the cache
            VFB_CUDA(cudaDeviceSynchronize());
            device_release(dev, p, cap);
        }
        p = np;
        cap = ncap;
        return VFB_OK;
    }
    // the caller has made sure that no queued work uses the buffer (vfb_destroy synchronises its streams first)
    void release()
    {
        if (p) device_release(dev, p, cap);
        p = nullptr;
        cap = 0;
    }
    template <class T> T *as() const { return reinterpret_cast<T *>(p); }
};

// The adapter sides, indexes of vfb_ctx::side and of the per-side arrays below.
enum { PRE = 0, SUF = 1 };

// What vfb_create decides for one adapter.  win_k >= 0 <=> this side runs the windowed DP (filter -> windows ->
// resolve), and then `packed` is set too; plan_packed_dp is the one place that decides it.
struct AdapterSide {
    std::string seq;
    AdapterBytes ad;
    bool align = false;                 // the threshold is below 1: reads without an exact match are aligned
    int min_accept = 0;
    bool packed = false;                // the packed kernels run on `lay` (else only the unpacked one)
    DpLayout lay;
    uint32_t lcap = 0;
    int win_k = -1;                     // Myers threshold of the windowed DP
    DevBuf d_code;                      // adapter codes for the unpacked kernel
};

// The per-read diagnostics columns of one pass, by adapter side.
struct DiagBufs {
    DevBuf exact[2], score[2], len[2];
    int ensure(size_t bytes)
    {
        for (int s = 0; s < 2; ++s)
            for (DevBuf *b : {&exact[s], &score[s], &len[s]})
                if (int rc = b->ensure(bytes)) return rc;
        return VFB_OK;
    }
    void release()
    {
        for (int s = 0; s < 2; ++s) { exact[s].release(); score[s].release(); len[s].release(); }
    }
};

struct PinBuf {
    void *p = nullptr;
    size_t cap = 0;
    int ensure(size_t bytes)
    {
        if (bytes <= cap) return VFB_OK;
        release();
        p = pinned_acquire(bytes + bytes / 8 + 4096, &cap);
        if (!p) {
            cap = 0;
            set_error("cannot allocate pinned host memory");
            return VFB_ERR_NOMEM;
        }
        return VFB_OK;
    }
    void release()
    {
        pinned_release(p, cap);
        p = nullptr;
        cap = 0;
    }
};

// The hot loop of consecutive batches runs on two LANES (streams with their own per-batch scratch), so that the
// ALU-bound DP kernels of one batch share the SMs with the memory-bound scan / key / count kernels of its
// neighbours; only the table insert (K4) is serialised between the lanes.
#define VFB_LANES 2
struct Lane {
    cudaStream_t st = nullptr;          // scan, keys, count (and everything else of the batch)
    cudaStream_t st_dp = nullptr;       // split mode: the alignment kernels, at a lower priority than `st`
    cudaEvent_t ev_scanned = nullptr, ev_aligned = nullptr;
    cudaEvent_t done = nullptr;         // the lane's last batch has finished
    bool pending = false;               // `done` has not been joined into the compute stream yet
    DevBuf d_start, d_end, d_c32, d_t64;
    DevBuf d_list[2], d_fb[2];          // per side: DP worklist, reads for the next kernel of the fallback chain
    DevBuf d_keys, d_koff, d_klen, d_khash, d_owner;
    DevBuf d_wins, d_bestkey, d_cbval, d_fb2;   // windowed DP: window items, per-item results, second fallback list
    // both_strands: the reverse pass's text (reverse complements, padded), compact spans, original read indices and
    // boundaries (the forward boundaries stay in d_start / d_end)
    DevBuf d_rtext, d_rspans, d_rsrc, d_rstart, d_rend;
    uint32_t win_cap = 0;
};

struct Slot {
    DevBuf d_text, d_spans;
    PinBuf h_text, h_spans;
    cudaEvent_t copied = nullptr, computed[VFB_LANES] = {nullptr, nullptr};
    unsigned busy = 0;                  // lanes whose `computed` event is pending
};

// One block-gzip segment in flight on the device (ingest): its text buffer, spans and the events that order the
// ingest stream (H2D, inflate, parse) with the compute stream (K1..K4).
#define VFB_SEG_SLOTS 3
struct SegSlot {
    DevBuf text, z, members, spans;
    cudaEvent_t copied = nullptr, inflated = nullptr, parsed = nullptr;       // recorded on st_copy / st_ingest / st_parse
    bool used = false;                                                        // `inflated` has been recorded at least once
    cudaEvent_t computed[VFB_LANES] = {nullptr, nullptr};                     // recorded on the lanes
    unsigned busy = 0;                                  // lanes whose `computed` event is pending
    uint64_t text_bytes = 0, z_bytes = 0;
    uint32_t n_members = 0;
};

// device counters of one batch
enum { C_NPRE = 0, C_NSUF, C_FBPRE, C_FBSUF, C_FB2PRE, C_FB2SUF, C_NWINPRE, C_NWINSUF,
       // work cursors of the filter / window kernels (dynamic distribution), each in a 128-byte line of its own: the
       // counters above take millions of atomics per launch, a cursor in their line would queue behind them
       C_WORKPRE = 32, C_WORKPRE2 = 64, C_WORKSUF = 96, C_WORKSUF2 = 128,
       C_NMISS = 160,        // fused key + count kernel: keys left for the insert kernels
       C_COUNT32 = 192 };
// 64-bit device counters
// (T_GATHER: the gather cursor of the batch; T_REVREADS / T_REVCOUNTED: both_strands statistics; T_UMISHORT: reads
// dropped for a short UMI)
enum { T_CELLS = 0, T_DPPRE, T_DPSUF, T_KEYBYTES, T_CELLSCOMP, T_WINDOWS, T_GATHER, T_REVREADS, T_REVCOUNTED, T_UMISHORT,
       T_COUNT64 };

}  // namespace vfb

struct vfb_ctx {
    vfb_params prm;                       // prm.prefix / prm.suffix point into side[].seq
    vfb::AdapterSide side[2];
    vfb::DpScoring sc;
    vfb::DevBuf d_generic_scratch;
    uint32_t generic_threads = 0;

    int device = 0, sm_count = 148;
    cudaStream_t st_compute = nullptr, st_copy = nullptr;
    cudaStream_t st_ingest = nullptr;     // H2D of compressed members + inflate, segment after segment
    cudaStream_t st_parse = nullptr;      // record framing of a segment (highest priority: it is the serial link
                                          // between segments and must not queue behind the next segment's inflate)
    vfb::Slot slots[2];
    uint64_t batch_seq = 0;
    uint64_t batch_reads = 0, batch_bytes = 0;

    // per-batch scratch, one set per lane
    vfb::Lane lanes[VFB_LANES];
    int n_lanes = VFB_LANES;                    // 1: every batch on the compute stream itself (diagnostics, vfb_set_lanes)
    bool fused_count = true;                    // the key kernel probes the table itself (VFB_FUSED_COUNT=0: K3 then K4 over every read)
    uint64_t lane_seq = 0;
    cudaEvent_t ev_fork = nullptr, ev_k4 = nullptr;   // compute stream -> lane; the previous batch's insert is done
    bool k4_pending = false;
    vfb::DevBuf d_aligned_text;     // aligned copy of an unaligned caller buffer (vfb_submit_device)
    vfb::DevBuf d_span_sum;         // vfb_submit_device: sum of the span lengths of a batch
    // diagnostics of the forward pass and (both_strands) of the reverse pass, the latter in compact (gathered) order
    vfb::DiagBufs diag_fwd, diag_rev;
    uint64_t diag_n = 0;
    bool diag_valid = false;

    // table
    vfb::DevTable tab{};
    vfb::DevBuf t_slots, t_row_hash, t_row_off, t_row_len, t_row_slot, t_arena, t_counters, t_row_count;
    vfb::DevBuf t_row_mol;                // umi_length: molecules of the group each exported row represents
    // Host-side upper bounds of rows / arena bytes = the last counter snapshot that has come back + what the batches
    // queued since may add.  A snapshot (rows, arena bytes) is copied to pinned memory behind every batch's insert
    // and picked up without blocking: the bounds stay within a few batches of the truth and no batch waits for them.
    uint64_t ub_rows = 0, ub_arena = 0;
    struct CtrSnap { cudaEvent_t ev = nullptr; uint64_t add_rows = 0, add_bytes = 0; bool pending = false; };
    static constexpr int N_SNAP = 16;
    CtrSnap snaps[N_SNAP];
    vfb::PinBuf snap_pin;                 // N_SNAP x 2 u64
    uint64_t snap_head = 0, snap_tail = 0;   // [tail, head) are pending, in batch order
    uint64_t base_rows = 0, base_arena = 0;  // the newest snapshot seen

    // ingest, GPU inflate path: segments in flight, tail / info landing zones
    vfb::SegSlot seg[VFB_SEG_SLOTS];
    vfb::DevBuf g_tail, g_info;
    vfb::PinBuf g_pin;               // carry staging + tail/info landing zone
    uint64_t g_seq = 0;

    // ingest: GPU FASTQ parse scratch and the first-malformed-record word
    vfb::DevBuf p_tiles, p_line_end, p_err;      // p_err: u32 chunk-relative + u64 global (at +8)
    bool p_err_init = false;

    // export: device-side Arrow compaction and pinned host columns
    vfb::DevBuf x_block_bytes, x_block_rows, x_offsets, x_counts, x_data, x_mol;
    vfb::PinBuf h_offsets, h_counts, h_data, h_mol;
    uint64_t x_rows = 0, x_bytes = 0, x_table_rows = 0;   // vfb_internal_export_sizes -> _write

    // merge scratch
    vfb::DevBuf m_part_rows, m_part_keys, m_cursors, m_chunk_off, m_send, m_recv;
    vfb::PinBuf m_pin;                    // part sizes landing zone
    std::vector<uint64_t> h_part_rows, h_part_keys;
    uint32_t m_self = 0xFFFFFFFFu;        // `self` of the last partition_sizes call
    cudaEvent_t m_filled = nullptr;       // the send buffer is complete (recorded on st_compute)

    bool profiling = false;
    vfb_progress_fn progress_fn = nullptr;
    void *progress_user = nullptr;
    std::chrono::steady_clock::time_point progress_last{};
    bool own_compute_stream = true;
    std::vector<cudaEvent_t> evpool;   // 12 events per profiled batch, resolved at sync time
    size_t ev_used = 0;
    vfb_stats stats{};
    vfb_collapse_info collapse_info{};   // the last finish that collapsed (collapse_ratio)
    uint32_t umi_offset = 0, umi_len = 0;   // vfb_set_umi (umi_len 0 = off)
    vfb_umi_info umi_info{};             // the last finish that grouped UMIs (reads_short comes from the lanes)
    bool table_used = false;             // a batch or an absorb may have added rows since create / clear
    bool mol_valid = false;              // h_mol holds the molecules of the last vfb_finish
};

// ---- internal hooks between api.cu, ingest.cu and multi.cu (not part of the C ABI)
// Export in two passes, so that several contexts can write consecutive pieces of ONE set of host columns:
// sizes (synchronous: rows with a non-zero count and their key bytes), then offsets (+ byte_base) / counts / keys
// copied to the given PINNED host pointers on the compute stream (asynchronous; vfb_sync waits).  `collapse`: the
// exported counts are collapsed first (prm.collapse_ratio; the count table keeps its rows and counts).
int vfb_internal_export_sizes(vfb_ctx *ctx, uint64_t *rows, uint64_t *key_bytes, bool collapse);
// With UMIs on, h_molecules receives x_rows molecule counts.
int vfb_internal_export_write(vfb_ctx *ctx, uint64_t byte_base, uint64_t *h_offsets, uint64_t *h_counts, uint8_t *h_data,
                              uint64_t *h_molecules = nullptr);
// Merge building blocks.  export: partition the rows (all of them, or with self < n_parts only the rows other
// parts own) into one chunk per part in the context's send buffer; sizes land in chunk_bytes / chunk_offsets
// (synchronous for them), `m_filled` is recorded when the buffer is complete; exported rows give up their count
// when `release` is set.  absorb_known: vfb_table_absorb without reading the chunk header back.
int vfb_internal_merge_export(vfb_ctx *ctx, uint32_t n_parts, uint32_t self, bool release, uint64_t *chunk_bytes,
                              uint64_t *chunk_offsets, uint64_t *part_rows, uint64_t *part_keys);
int vfb_internal_absorb_known(vfb_ctx *ctx, const uint8_t *d_chunk, uint64_t rows, uint64_t key_bytes);
int vfb_internal_partition_count(vfb_ctx *ctx, uint32_t n_parts, uint32_t self, uint64_t *table_rows);
int vfb_internal_partition_fill(vfb_ctx *ctx, uint32_t n_parts, uint32_t self, bool release, uint8_t *d_buf, const uint64_t *chunk_offsets);
// `molecules` (umi_length; an empty buffer = none) becomes a third child.
int vfb_internal_arrow_wrap(vfb::PinBuf offsets, vfb::PinBuf data, vfb::PinBuf counts, uint64_t rows,
                            vfb_arrow_array *out_array, vfb_arrow_schema *out_schema, vfb::PinBuf molecules = vfb::PinBuf());
// vfb_set_umi's checks that need no device
int vfb_internal_umi_check(const vfb_ctx *ctx, uint32_t umi_offset, uint32_t umi_length);
// One file over n_ctx contexts, one per device (ingest.cu).
int vfb_internal_run_file(vfb_ctx **ctxs, uint32_t n_ctx, const char *path, uint32_t flags, uint64_t *n_reads_out);
void bump_launches_for(vfb_ctx *ctx, uint64_t launches_before);
