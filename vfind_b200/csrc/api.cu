// Host side of the C ABI (include/vfind_b200.h): context, batching, streams, table growth.
//
// Mirrors the setup + hot loop of find_variants (/root/reference/src/lib.rs:233-320): the
// reference's `parallel_fastq(reader, n_threads, queue_len, WORK, REDUCE)` becomes batches of
// reads moving through  H2D copy -> K1 scan -> worklists -> K2 DP -> K3 keys -> K4 count  on a
// compute stream, with the next batch's copy overlapping on a second stream.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <sched.h>
#include <string>
#include <thread>
#include <vector>

#include "hash.h"
#include "synth.h"
#include "ctx.cuh"

namespace vfb {

thread_local std::string g_error;
thread_local uint64_t g_launches = 0;

void set_error(const std::string &msg) { g_error = msg; }

int cuda_fail(cudaError_t e, const char *what, const char *file, int line)
{
    char buf[512];
    snprintf(buf, sizeof buf, "CUDA error %d (%s) at %s:%d: %s", (int)e, cudaGetErrorString(e), file, line, what);
    g_error = buf;
    return VFB_ERR_CUDA;
}

}  // namespace vfb (reopened below)

#include <atomic>
#include <chrono>
#include <cstdarg>
#include <mutex>
#include <thread>
#include <utility>
#include <vector>
namespace vfb {
bool trace_on()
{
    static int on = -1;
    if (on < 0) on = getenv("VFB_TRACE") ? 1 : 0;
    return on == 1;
}
void trace(const char *fmt, ...)
{
    if (!trace_on()) return;
    static const auto t0 = std::chrono::steady_clock::now();
    const double ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    fprintf(stderr, "[vfb %9.1f ms] ", ms);
    va_list ap;
    va_start(ap, fmt);
    vfprintf(stderr, fmt, ap);
    va_end(ap);
    fputc('\n', stderr);
}

// Process-wide cache of pinned host buffers: page-locking costs about 1 ms per MB, more than a
// whole small run.  Buffers released by a context / an ingest are kept (up to VFB_PINNED_POOL_MB,
// default 4096: a call on a plain gzip file holds 0.9 GB of staging — three 128 MB text chunks, two 254 MB compressed
// segments — plus its result columns, and the previous call's result is usually still alive; with a 1 GB cap every call
// page-locked 0.1-0.5 GB anew, 0.08-0.5 s on a 0.3 s call) and handed to the next one; vfb_pinned_pool_trim() frees them.
struct PinnedPool {
    std::mutex mu;
    std::vector<std::pair<void *, size_t>> idle;
    size_t bytes = 0;
};
static PinnedPool &pinned_pool()
{
    static PinnedPool *p = new PinnedPool;      // never destroyed: the driver may be gone at exit
    return *p;
}
void *pinned_acquire(size_t want, size_t *cap_out)
{
    PinnedPool &pp = pinned_pool();
    {
        std::lock_guard<std::mutex> lk(pp.mu);
        int best = -1;
        for (size_t i = 0; i < pp.idle.size(); ++i)
            // (a close fit only: a result column of 60 MB must not walk off with an 81 MB staging buffer that the
            // next call will want back -- page-locking a fresh one costs more than the call's kernels)
            if (pp.idle[i].second >= want && pp.idle[i].second <= want + want / 8 + (64u << 10) &&
                (best < 0 || pp.idle[i].second < pp.idle[(size_t)best].second)) best = (int)i;
        if (best >= 0) {
            void *p = pp.idle[(size_t)best].first;
            *cap_out = pp.idle[(size_t)best].second;
            pp.bytes -= *cap_out;
            pp.idle.erase(pp.idle.begin() + best);
            return p;
        }
    }
    void *p = nullptr;
    if (want >= (8u << 20)) trace("cudaMallocHost %zu MB", want >> 20);
    if (cudaMallocHost(&p, want) != cudaSuccess) {
        cudaGetLastError();
        pinned_pool_trim();                      // give the cache back and try once more
        if (cudaMallocHost(&p, want) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    }
    *cap_out = want;
    return p;
}
void pinned_release(void *p, size_t cap)
{
    if (!p) return;
    static size_t limit = 0;
    if (!limit) {
        const char *e = getenv("VFB_PINNED_POOL_MB");
        limit = ((size_t)(e ? strtoull(e, nullptr, 10) : 4096ull) << 20) + 1;
    }
    PinnedPool &pp = pinned_pool();
    std::vector<void *> evict;
    bool keep = false;
    {
        std::lock_guard<std::mutex> lk(pp.mu);
        if (cap < limit) {
            // the buffer just used is the one the next call will ask for: make room for it by letting the
            // longest-idle buffers go (a finished 100 M-read context leaves ~1 GB of result columns behind,
            // which used to crowd out the ingest's staging buffers and made every later call page-lock anew)
            while (pp.bytes + cap >= limit && !pp.idle.empty()) {
                evict.push_back(pp.idle.front().first);
                pp.bytes -= pp.idle.front().second;
                pp.idle.erase(pp.idle.begin());
            }
            pp.idle.emplace_back(p, cap);
            pp.bytes += cap;
            keep = true;
        }
    }
    for (void *q : evict) cudaFreeHost(q);
    if (!keep) cudaFreeHost(p);
}
void pinned_pool_trim()
{
    PinnedPool &pp = pinned_pool();
    std::vector<std::pair<void *, size_t>> all;
    {
        std::lock_guard<std::mutex> lk(pp.mu);
        all.swap(pp.idle);
        pp.bytes = 0;
    }
    for (auto &b : all) cudaFreeHost(b.first);
}

// Device buffers: one idle list per device.  A buffer fits a request when it is at least as large and at most
// twice as large (+1 MB): device memory is plentiful, a fresh cudaMalloc is what costs.
struct DevicePool {
    std::mutex mu;
    std::vector<std::vector<std::pair<void *, size_t>>> idle;   // per device
    std::vector<size_t> bytes;
};
static DevicePool &device_pool()
{
    static DevicePool *p = new DevicePool;       // never destroyed: the driver may be gone at exit
    return *p;
}
static size_t device_pool_limit()
{
    static size_t limit = 0;
    if (!limit) {
        const char *e = getenv("VFB_DEVICE_POOL_MB");
        limit = ((size_t)(e ? strtoull(e, nullptr, 10) : 24576ull) << 20) + 1;
    }
    return limit;
}
void *device_acquire(int device, size_t want, size_t *cap_out)
{
    DevicePool &dp = device_pool();
    {
        std::lock_guard<std::mutex> lk(dp.mu);
        if ((size_t)device < dp.idle.size()) {
            auto &v = dp.idle[(size_t)device];
            int best = -1;
            for (size_t i = 0; i < v.size(); ++i)
                if (v[i].second >= want && v[i].second <= 2 * want + (1u << 20) &&
                    (best < 0 || v[i].second < v[(size_t)best].second)) best = (int)i;
            if (best >= 0) {
                void *p = v[(size_t)best].first;
                *cap_out = v[(size_t)best].second;
                dp.bytes[(size_t)device] -= *cap_out;
                v.erase(v.begin() + best);
                return p;
            }
        }
    }
    void *p = nullptr;
    if (want >= (8u << 20)) trace("cudaMalloc %zu MB on device %d", want >> 20, device);
    if (cudaMalloc(&p, want) != cudaSuccess) {
        cudaGetLastError();
        device_pool_trim();                     // give the cache back and try once more
        if (cudaMalloc(&p, want) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    }
    *cap_out = want;
    return p;
}
void device_release(int device, void *p, size_t cap)
{
    if (!p) return;
    DevicePool &dp = device_pool();
    const size_t limit = device_pool_limit();
    std::vector<void *> evict;
    bool keep = false;
    {
        std::lock_guard<std::mutex> lk(dp.mu);
        if (device >= 0 && cap < limit) {
            if ((size_t)device >= dp.idle.size()) { dp.idle.resize((size_t)device + 1); dp.bytes.resize((size_t)device + 1, 0); }
            auto &v = dp.idle[(size_t)device];
            while (dp.bytes[(size_t)device] + cap >= limit && !v.empty()) {     // longest idle first
                evict.push_back(v.front().first);
                dp.bytes[(size_t)device] -= v.front().second;
                v.erase(v.begin());
            }
            v.emplace_back(p, cap);
            dp.bytes[(size_t)device] += cap;
            keep = true;
        }
    }
    if (!evict.empty() || !keep) {
        int cur = -1;
        cudaGetDevice(&cur);
        if (cur != device && device >= 0) cudaSetDevice(device);
        for (void *q : evict) cudaFree(q);
        if (!keep) cudaFree(p);
        if (cur != device && cur >= 0) cudaSetDevice(cur);
    }
}
void device_pool_trim()
{
    DevicePool &dp = device_pool();
    std::vector<std::vector<std::pair<void *, size_t>>> all;
    {
        std::lock_guard<std::mutex> lk(dp.mu);
        all.swap(dp.idle);
        dp.bytes.clear();
    }
    int cur = -1;
    cudaGetDevice(&cur);
    for (size_t d = 0; d < all.size(); ++d) {
        if (all[d].empty()) continue;
        cudaSetDevice((int)d);
        for (auto &b : all[d]) cudaFree(b.first);
    }
    if (cur >= 0) cudaSetDevice(cur);
}

}  // namespace vfb

using namespace vfb;

// Profiling: events are recorded on the compute stream without blocking; the per-stage
// times are accumulated when the stream is next synchronised.
static int prof_events(vfb_ctx *c, cudaEvent_t **out)
{
    if (c->ev_used + 12 > c->evpool.size()) {
        size_t old = c->evpool.size();
        c->evpool.resize(old + 96, nullptr);
        for (size_t i = old; i < c->evpool.size(); ++i) VFB_CUDA(cudaEventCreate(&c->evpool[i]));
    }
    *out = &c->evpool[c->ev_used];
    c->ev_used += 12;
    return VFB_OK;
}

static int prof_resolve(vfb_ctx *c)
{
    for (size_t b = 0; b + 12 <= c->ev_used; b += 12) {
        cudaEvent_t *ev = &c->evpool[b];
        float ms;
        VFB_CUDA(cudaEventElapsedTime(&ms, ev[0], ev[1])); c->stats.ms_scan += ms;
        VFB_CUDA(cudaEventElapsedTime(&ms, ev[1], ev[2])); c->stats.ms_worklist += ms;
        VFB_CUDA(cudaEventElapsedTime(&ms, ev[2], ev[3])); c->stats.ms_dp += ms;
        VFB_CUDA(cudaEventElapsedTime(&ms, ev[3], ev[4])); c->stats.ms_worklist += ms;
        VFB_CUDA(cudaEventElapsedTime(&ms, ev[4], ev[5])); c->stats.ms_dp += ms;
        VFB_CUDA(cudaEventElapsedTime(&ms, ev[5], ev[6])); c->stats.ms_translate += ms;
        VFB_CUDA(cudaEventElapsedTime(&ms, ev[6], ev[7])); c->stats.ms_count += ms;
        VFB_CUDA(cudaEventElapsedTime(&ms, ev[0], ev[7])); c->stats.ms_total += ms;
        // windowed DP: [2] filter [8] windows [9] resolve + fallbacks [3] for the prefix, [4] [10] [11] [5] for the suffix
        for (int s = 0; s < 2; ++s)
            if (c->side[s].win_k >= 0) {
                VFB_CUDA(cudaEventElapsedTime(&ms, ev[2 + 2 * s], ev[8 + 2 * s])); c->stats.ms_dp_filter += ms;
                VFB_CUDA(cudaEventElapsedTime(&ms, ev[8 + 2 * s], ev[9 + 2 * s])); c->stats.ms_dp_window += ms;
            }
    }
    c->ev_used = 0;
    return VFB_OK;
}

static int bump_launches(vfb_ctx *c, uint64_t before)
{
    c->stats.kernel_launches += g_launches - before;
    return VFB_OK;
}
void bump_launches_for(vfb_ctx *c, uint64_t before) { bump_launches(c, before); }

// ------------------------------------------------------------------------------------ helpers
// Everything the lanes have been given so far is ordered before whatever is queued next on the compute stream.
static int lanes_join(vfb_ctx *c)
{
    for (auto &ln : c->lanes)
        if (ln.pending) {
            VFB_CUDA(cudaStreamWaitEvent(c->st_compute, ln.done, 0));
            ln.pending = false;
        }
    c->k4_pending = false;
    return VFB_OK;
}

static int table_alloc(vfb_ctx *c, uint64_t capacity, uint64_t rows_cap, uint64_t arena_cap)
{
    int rc;
    if ((rc = c->t_slots.ensure(capacity * 8 * VFB_SLOT_WORDS))) return rc;
    if ((rc = c->t_row_hash.ensure(rows_cap * 8, true, c->st_compute))) return rc;
    if ((rc = c->t_row_off.ensure(rows_cap * 8, true, c->st_compute))) return rc;
    if ((rc = c->t_row_len.ensure(rows_cap * 4, true, c->st_compute))) return rc;
    if ((rc = c->t_row_slot.ensure(rows_cap * 4, true, c->st_compute))) return rc;
    if ((rc = c->t_arena.ensure(arena_cap, true, c->st_compute))) return rc;
    c->tab.slots = c->t_slots.as<unsigned long long>();
    c->tab.capacity = capacity;
    c->tab.row_hash = c->t_row_hash.as<uint64_t>();
    c->tab.row_off = c->t_row_off.as<uint64_t>();
    c->tab.row_len = c->t_row_len.as<uint32_t>();
    c->tab.row_slot = c->t_row_slot.as<uint32_t>();
    c->tab.row_capacity = rows_cap;
    c->tab.arena = c->t_arena.as<uint8_t>();
    c->tab.arena_capacity = arena_cap;
    c->tab.counters = c->t_counters.as<unsigned long long>();
    return VFB_OK;
}

static uint64_t pow2_at_least(uint64_t v)
{
    uint64_t p = 1024;
    while (p < v) p <<= 1;
    return p;
}

static int table_init(vfb_ctx *c)
{
    int rc;
    if ((rc = c->t_counters.ensure(8 * 8))) return rc;
    uint64_t hint = c->prm.table_capacity_hint;
    // without a hint: room for 2 M distinct variants (about 250 MB in all) before the first rehash — a rehash stalls the
    // pipeline, and the buffers come from the device pool after the first call
    uint64_t cap = pow2_at_least(hint ? hint * 2 : (1u << 22));
    uint64_t rows = hint ? hint : (1u << 21);
    if ((rc = table_alloc(c, cap, rows, rows * 96))) return rc;
    VFB_CUDA(cudaMemsetAsync(c->tab.slots, 0, cap * 8 * VFB_SLOT_WORDS, c->st_compute));
    VFB_CUDA(cudaMemsetAsync(c->tab.counters, 0, 8 * 8, c->st_compute));
    c->ub_rows = 0;
    c->ub_arena = 0;
    return VFB_OK;
}

// Counter snapshots: see vfb_ctx::snaps.
static void snaps_poll(vfb_ctx *c, bool wait_oldest)
{
    while (c->snap_tail < c->snap_head) {
        vfb_ctx::CtrSnap &sn = c->snaps[c->snap_tail % vfb_ctx::N_SNAP];
        cudaError_t e = wait_oldest ? cudaEventSynchronize(sn.ev) : cudaEventQuery(sn.ev);
        wait_oldest = false;
        if (e != cudaSuccess) { cudaGetLastError(); break; }
        const uint64_t *v = reinterpret_cast<const uint64_t *>(c->snap_pin.p) + 2 * (c->snap_tail % vfb_ctx::N_SNAP);
        c->base_rows = v[0];
        c->base_arena = v[1];
        sn.pending = false;
        ++c->snap_tail;
    }
    uint64_t r = c->base_rows, a = c->base_arena;
    for (uint64_t k = c->snap_tail; k < c->snap_head; ++k) {
        r += c->snaps[k % vfb_ctx::N_SNAP].add_rows;
        a += c->snaps[k % vfb_ctx::N_SNAP].add_bytes;
    }
    c->ub_rows = r;
    c->ub_arena = a;
}

// Called once the inserts of a batch that may add (new_keys, new_bytes) have been queued on `st`.
static int snaps_push(vfb_ctx *c, uint64_t new_keys, uint64_t new_bytes, cudaStream_t st)
{
    if (!c->snap_pin.p) {
        int rc = c->snap_pin.ensure(vfb_ctx::N_SNAP * 16);
        if (rc) return rc;
        for (auto &sn : c->snaps) VFB_CUDA(cudaEventCreateWithFlags(&sn.ev, cudaEventDisableTiming));
    }
    if (c->snap_head - c->snap_tail >= (uint64_t)vfb_ctx::N_SNAP) snaps_poll(c, true);
    vfb_ctx::CtrSnap &sn = c->snaps[c->snap_head % vfb_ctx::N_SNAP];
    sn.add_rows = new_keys; sn.add_bytes = new_bytes; sn.pending = true;
    uint64_t *dst = reinterpret_cast<uint64_t *>(c->snap_pin.p) + 2 * (c->snap_head % vfb_ctx::N_SNAP);
    VFB_CUDA(cudaMemcpyAsync(dst, c->tab.counters, 16, cudaMemcpyDeviceToHost, st));
    VFB_CUDA(cudaEventRecord(sn.ev, st));
    ++c->snap_head;
    return VFB_OK;
}

static void snaps_reset(vfb_ctx *c)           // the table was cleared (after a join + on the compute stream)
{
    while (c->snap_tail < c->snap_head) {
        cudaEventSynchronize(c->snaps[c->snap_tail % vfb_ctx::N_SNAP].ev);
        c->snaps[c->snap_tail % vfb_ctx::N_SNAP].pending = false;
        ++c->snap_tail;
    }
    c->base_rows = c->base_arena = 0;
    c->ub_rows = c->ub_arena = 0;
}

// Make room for `new_keys` more keys of `new_bytes` padded key bytes (upper bounds).  The caller queues the inserts
// and then calls snaps_push with the same numbers.  `stream_of_batches`: the caller is one of a run of batches like this
// one (a submit), not a one-off (a merge's absorb).
static int table_reserve(vfb_ctx *c, uint64_t new_keys, uint64_t new_bytes, bool stream_of_batches)
{
    snaps_poll(c, false);
    uint64_t want_rows = c->ub_rows + new_keys, want_arena = c->ub_arena + new_bytes;
    auto fits = [&]() {
        return want_rows * 2 <= c->tab.capacity && want_rows <= c->tab.row_capacity &&
               want_arena <= c->tab.arena_capacity && want_rows < 0x7FFFFFF0ull;
    };
    if (fits()) return VFB_OK;
    // the bounds say no: wait for the true counters (everything queued so far), then grow if it is still needed —
    // geometrically, so that this happens O(log) times
    trace("table_reserve: bounds exceeded (rows %llu + %llu of %llu, arena %llu + %llu of %llu MB): sync",
          (unsigned long long)c->ub_rows, (unsigned long long)new_keys, (unsigned long long)c->tab.row_capacity,
          (unsigned long long)(c->ub_arena >> 20), (unsigned long long)(new_bytes >> 20), (unsigned long long)(c->tab.arena_capacity >> 20));
    { const int jrc = lanes_join(c); if (jrc) return jrc; }
    unsigned long long ctr[2];
    VFB_CUDA(cudaMemcpyAsync(ctr, c->tab.counters, sizeof ctr, cudaMemcpyDeviceToHost, c->st_compute));
    VFB_CUDA(cudaStreamSynchronize(c->st_compute));
    c->stats.d2h_bytes += sizeof ctr;
    while (c->snap_tail < c->snap_head) { c->snaps[c->snap_tail % vfb_ctx::N_SNAP].pending = false; ++c->snap_tail; }
    c->base_rows = c->ub_rows = ctr[0];
    c->base_arena = c->ub_arena = ctr[1];
    want_rows = c->ub_rows + new_keys;
    want_arena = c->ub_arena + new_bytes;
    if (!stream_of_batches) {
        if (fits()) return VFB_OK;
    } else {
        // The bounds of the batches still in flight (each counts ALL its reads as new rows) are what failed, so room for
        // this batch alone would only bring the next batch back here, with another wait for the counters (which halves
        // the pace of a plain-gzip file's chunks): unless there is room for a pipeline's worth of batches like this one,
        // grow now — once, geometrically.  Only where that is a modest step (at most four times what there is, or a few
        // GB in absolute terms: a file's chunks of 128 MB of text must always qualify, or the call's pace depends on
        // how many batches happened to be in flight): batches of millions of reads each are worth a wait for the
        // counters, not a table sized for seventeen of them; and never for a merge's absorb.
        const uint64_t ahead = (uint64_t)vfb_ctx::N_SNAP + 1;
        const uint64_t rows_ahead = c->ub_rows + ahead * new_keys, arena_ahead = c->ub_arena + ahead * new_bytes;
        const bool roomy = rows_ahead * 2 <= c->tab.capacity && rows_ahead <= c->tab.row_capacity && arena_ahead <= c->tab.arena_capacity;
        const uint64_t rows_step = std::max<uint64_t>(4 * c->tab.row_capacity, 32ull << 20);
        const uint64_t arena_step = std::max<uint64_t>(4 * c->tab.arena_capacity, 4ull << 30);
        const bool modest = rows_ahead <= rows_step && arena_ahead <= arena_step;
        if (fits() && (roomy || !modest || rows_ahead >= 0x7FFFFFF0ull)) return VFB_OK;
        if (fits()) {
            trace("table_reserve: growing ahead of need (rows %llu, %llu per batch)", (unsigned long long)c->ub_rows, (unsigned long long)new_keys);
            want_rows = rows_ahead;
            want_arena = arena_ahead;
        }
    }
    if (want_rows >= 0x7FFFFFF0ull) {
        set_error("more than 2^31 distinct variants are not supported");
        return VFB_ERR_ARG;
    }
    int rc;
    uint64_t rows_cap = c->tab.row_capacity, arena_cap = c->tab.arena_capacity;
    if (want_rows > rows_cap) rows_cap = 2 * want_rows;
    if (want_arena > arena_cap) arena_cap = 2 * want_arena;
    if (want_rows * 2 > c->tab.capacity) {
        // rehash into a larger slot array
        uint64_t ncap = pow2_at_least(want_rows * 4);
        trace("table rehash %llu -> %llu slots", (unsigned long long)c->tab.capacity, (unsigned long long)ncap);
        DevBuf nslots;
        if ((rc = nslots.ensure(ncap * 8 * VFB_SLOT_WORDS))) return rc;
        VFB_CUDA(cudaMemsetAsync(nslots.p, 0, ncap * 8 * VFB_SLOT_WORDS, c->st_compute));
        DevTable nt = c->tab;
        nt.slots = nslots.as<unsigned long long>();
        nt.capacity = ncap;
        if ((rc = launch_rehash(c->tab, nt, c->st_compute))) return rc;
        VFB_CUDA(cudaStreamSynchronize(c->st_compute));
        c->t_slots.release();
        c->t_slots = nslots;
        c->tab.capacity = ncap;
    }
    if ((rc = table_alloc(c, c->tab.capacity, rows_cap, arena_cap))) return rc;
    return VFB_OK;
}

static void fill_adapter(AdapterBytes *a, const std::string &s)
{
    memset(a, 0, sizeof *a);
    a->len = (uint32_t)s.size();
    memcpy(a->b, s.data(), s.size());
}

// score as f64 > min  <=>  score >= floor(min) + 1   (any finite min)   src/lib.rs:157,260-261
static int accept_bound(double thr, int32_t match, size_t len)
{
    volatile double a = thr * (double)match;
    volatile double m = a * (double)len;
    double f = std::floor((double)m);
    if (f > 2.0e9) return INT32_MAX;
    if (f < -2.0e9) return INT32_MIN + 1;
    return (int)f + 1;
}

// The packed DP of one adapter: the windowed path (K >= 0) when it is wanted, the filter applies and the window's
// wider score range fits the packed word; else the full-matrix kernel (K = -1) when its range fits; else false (the
// unpacked kernel runs).  The full kernel that takes the windowed path's fallback reads runs on the same layout.
static bool plan_packed_dp(const DpScoring &sc, uint32_t A, int min_accept, bool want_window, DpLayout *lay,
                           uint32_t *lcap, int *K)
{
    *K = want_window ? dpw_max_edits(sc, A, min_accept) : -1;
    if (*K >= 0 && !make_dp_layout(sc, A, true, lay)) *K = -1;
    if (*K < 0 && !make_dp_layout(sc, A, false, lay)) return false;
    *lcap = dp_lcap(*lay, A, sc.extend);
    return true;
}

// ------------------------------------------------------------------------------------ ABI
extern "C" {

const char *vfb_last_error(void) { return g_error.c_str(); }
int vfb_abi_version(void) { return VFB_ABI_VERSION; }

void vfb_default_params(vfb_params *p)
{
    memset(p, 0, sizeof *p);
    p->struct_size = sizeof *p;
    p->match_score = 3;            // src/lib.rs:172-181
    p->mismatch_score = -2;
    p->gap_open_penalty = 5;
    p->gap_extend_penalty = 2;
    p->accept_prefix_alignment = 0.75;
    p->accept_suffix_alignment = 0.75;
    p->n_threads = 3;
    p->queue_len = 2;
    p->skip_translation = 0;
    p->show_progress = 1;
    p->device = -1;
}

static int preflight(double thr, bool *skip)
{
    // src/lib.rs:100-110 (NaN fails both tests and reaches the error)
    if (thr > 0. && thr < 1.) { *skip = false; return VFB_OK; }
    if (thr == 1.) { *skip = true; return VFB_OK; }
    set_error("Accept alignment threshold must be between 0 and 1.");
    return VFB_ERR_VALUE;
}

int vfb_create(const vfb_params *p, vfb_ctx **out)
{
    trace("vfb_create");
    if (!p || !out) { set_error("null argument"); return VFB_ERR_ARG; }
    if (p->struct_size != sizeof(vfb_params)) { set_error("vfb_params size mismatch"); return VFB_ERR_ARG; }
    if ((p->prefix_len && !p->prefix) || (p->suffix_len && !p->suffix)) { set_error("null adapter"); return VFB_ERR_ARG; }
    const uint8_t *const seq[2] = {p->prefix, p->suffix};
    const uint64_t len[2] = {p->prefix_len, p->suffix_len};
    const double thr[2] = {p->accept_prefix_alignment, p->accept_suffix_alignment};
    bool skip[2];
    int rc;
    for (int s = 0; s < 2; ++s)
        if ((rc = preflight(thr[s], &skip[s]))) return rc;   // :239, :249
    if (len[PRE] > VFB_MAX_SCAN_ADAPTER || len[SUF] > VFB_MAX_SCAN_ADAPTER) {
        set_error("adapters longer than 256 bases are not supported");
        return VFB_ERR_ARG;
    }
    if ((!skip[PRE] && len[PRE] == 0) || (!skip[SUF] && len[SUF] == 0)) {
        // Profile::new on an empty adapter fails and the reference unwraps it (src/lib.rs:124-126)
        set_error("Error creating profile for adapter: empty adapter");
        return VFB_ERR_VALUE;
    }
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        set_error("no CUDA device available (this library has no CPU fallback)");
        return VFB_ERR_CUDA;
    }
    vfb_ctx *c = new vfb_ctx();
    c->prm = *p;
    for (int s = 0; s < 2; ++s) {
        AdapterSide &side = c->side[s];
        side.seq.assign((const char *)seq[s], len[s]);
        fill_adapter(&side.ad, side.seq);
        side.align = !skip[s];
        side.min_accept = accept_bound(thr[s], p->match_score, len[s]);
    }
    c->prm.prefix = (const uint8_t *)c->side[PRE].seq.data();
    c->prm.suffix = (const uint8_t *)c->side[SUF].seq.data();
    c->sc = DpScoring{p->match_score, p->mismatch_score, p->gap_open_penalty, p->gap_extend_penalty};
    c->batch_reads = p->batch_reads ? p->batch_reads : (8ull << 20);
    c->batch_bytes = p->batch_bytes ? p->batch_bytes : (2ull << 30);
    if (c->batch_reads > 0x7FFFFFFFull) c->batch_reads = 0x7FFFFFFFull;
    if (c->batch_bytes > 0xFFFFFFFFull) c->batch_bytes = 0xFFFFFFFFull;

    auto fail = [&](int code) { vfb_destroy(c); return code; };
    if (p->device >= 0) {
        if ((e = cudaSetDevice(p->device)) != cudaSuccess) return fail(cuda_fail(e, "cudaSetDevice", __FILE__, __LINE__));
        c->device = p->device;
    } else if ((e = cudaGetDevice(&c->device)) != cudaSuccess) {
        return fail(cuda_fail(e, "cudaGetDevice", __FILE__, __LINE__));
    }
    // (cudaGetDeviceProperties takes milliseconds; one attribute does not)
    if ((e = cudaDeviceGetAttribute(&c->sm_count, cudaDevAttrMultiProcessorCount, c->device)) != cudaSuccess)
        return fail(cuda_fail(e, "cudaDeviceGetAttribute", __FILE__, __LINE__));
    trace("vfb_create: device %d, %d SMs", c->device, c->sm_count);
    // the parse stream outranks everything: the short record-framing kernels of a segment sit on the critical path
    // of the segment chain and must queue neither behind K1..K4 nor behind the next segment's inflate
    int prio_lo = 0, prio_hi = 0;
    cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
    if ((e = cudaStreamCreateWithFlags(&c->st_compute, cudaStreamNonBlocking)) != cudaSuccess ||
        (e = cudaStreamCreateWithFlags(&c->st_copy, cudaStreamNonBlocking)) != cudaSuccess ||
        (e = cudaStreamCreateWithPriority(&c->st_ingest, cudaStreamNonBlocking, prio_lo)) != cudaSuccess ||
        (e = cudaStreamCreateWithPriority(&c->st_parse, cudaStreamNonBlocking, prio_hi)) != cudaSuccess)
        return fail(cuda_fail(e, "cudaStreamCreate", __FILE__, __LINE__));
    auto new_event = [&](cudaEvent_t *ev) { return (e = cudaEventCreateWithFlags(ev, cudaEventDisableTiming)) == cudaSuccess; };
    bool ev_ok = new_event(&c->m_filled) && new_event(&c->ev_fork) && new_event(&c->ev_k4);
    for (auto &s : c->slots) ev_ok = ev_ok && new_event(&s.copied) && new_event(&s.computed[0]) && new_event(&s.computed[1]);
    for (auto &g : c->seg) ev_ok = ev_ok && new_event(&g.copied) && new_event(&g.inflated) && new_event(&g.parsed) && new_event(&g.computed[0]) && new_event(&g.computed[1]);
    for (auto &ln : c->lanes)
        ev_ok = ev_ok && new_event(&ln.done) && new_event(&ln.ev_scanned) && new_event(&ln.ev_aligned) &&
                (e = cudaStreamCreateWithPriority(&ln.st, cudaStreamNonBlocking, prio_hi)) == cudaSuccess &&
                (e = cudaStreamCreateWithPriority(&ln.st_dp, cudaStreamNonBlocking, prio_lo)) == cudaSuccess;
    c->fused_count = true;
    if (const char *se = getenv("VFB_FUSED_COUNT")) c->fused_count = atoi(se) != 0;
    if (!ev_ok) return fail(cuda_fail(e, "cudaEventCreate / cudaStreamCreate", __FILE__, __LINE__));
    // two lanes unless the per-read diagnostics of "the last batch" are wanted
    c->n_lanes = VFB_LANES;
    if (p->diagnostics) c->n_lanes = 1;

    // DP setup: packed layout when the scores fit, else the fallback kernel
    const bool want_window = p->dp_mode != 1 && (!p->diagnostics || p->dp_mode == 2);
    for (AdapterSide &side : c->side) {
        if (!side.align) continue;
        const std::string &ad = side.seq;
        if (ad.size() > VFB_MAX_ADAPTER) { set_error("adapter too long for alignment"); return fail(VFB_ERR_ARG); }
        long long worst = (long long)(std::abs((long long)c->sc.match) + std::abs((long long)c->sc.mismatch) +
                                      std::abs((long long)c->sc.open) + std::abs((long long)c->sc.extend));
        if (worst > (1 << 20)) { set_error("alignment scores beyond +-2^20 are not supported"); return fail(VFB_ERR_ARG); }
        if (!p->force_generic_dp)
            side.packed = plan_packed_dp(c->sc, (uint32_t)ad.size(), side.min_accept, want_window, &side.lay, &side.lcap, &side.win_k);
        std::vector<uint8_t> code(ad.size());
        for (size_t i = 0; i < ad.size(); ++i) code[i] = (uint8_t)dp_code((uint8_t)ad[i]);
        if ((rc = side.d_code.ensure(code.size()))) return fail(rc);
        if ((e = cudaMemcpy(side.d_code.p, code.data(), code.size(), cudaMemcpyHostToDevice)) != cudaSuccess)
            return fail(cuda_fail(e, "cudaMemcpy", __FILE__, __LINE__));
    }
    const AdapterSide &pre = c->side[PRE], &suf = c->side[SUF];
    if (pre.align || suf.align) {
        c->generic_threads = dp_generic_threads(c->sm_count);
        size_t amax = pre.seq.size() > suf.seq.size() ? pre.seq.size() : suf.seq.size();
        if ((rc = c->d_generic_scratch.ensure(4 * amax * (size_t)c->generic_threads * sizeof(int32_t)))) return fail(rc);
    }
    for (auto &ln : c->lanes) {
        if ((rc = ln.d_c32.ensure(C_COUNT32 * 4))) return fail(rc);
        if ((rc = ln.d_t64.ensure(T_COUNT64 * 8))) return fail(rc);
        if ((e = cudaMemset(ln.d_t64.p, 0, T_COUNT64 * 8)) != cudaSuccess)
            return fail(cuda_fail(e, "cudaMemset", __FILE__, __LINE__));
    }
    trace("vfb_create: streams, events, DP setup done");
    if ((rc = table_init(c))) return fail(rc);
    trace("vfb_create: table ready");
    c->stats.dp_kernel_kind = (pre.win_k >= 0 || suf.win_k >= 0) ? 3 : (pre.packed || suf.packed) ? 1 : (pre.align || suf.align) ? 2 : 0;
    *out = c;
    return VFB_OK;
}

int vfb_destroy(vfb_ctx *c)
{
    if (!c) return VFB_OK;
    cudaSetDevice(c->device);
    if (c->st_compute) cudaStreamSynchronize(c->st_compute);
    if (c->st_copy) cudaStreamSynchronize(c->st_copy);
    if (c->st_ingest) cudaStreamSynchronize(c->st_ingest);
    if (c->st_parse) cudaStreamSynchronize(c->st_parse);
    for (auto &ln : c->lanes) { if (ln.st) cudaStreamSynchronize(ln.st); if (ln.st_dp) cudaStreamSynchronize(ln.st_dp); }
    for (auto &s : c->slots) {
        s.d_text.release(); s.d_spans.release(); s.h_text.release(); s.h_spans.release();
        if (s.copied) cudaEventDestroy(s.copied);
        for (auto &ev : s.computed) if (ev) cudaEventDestroy(ev);
    }
    for (auto &g : c->seg) {
        g.text.release(); g.z.release(); g.members.release(); g.spans.release();
        if (g.parsed) cudaEventDestroy(g.parsed);
        if (g.inflated) cudaEventDestroy(g.inflated);
        if (g.copied) cudaEventDestroy(g.copied);
        for (auto &ev : g.computed) if (ev) cudaEventDestroy(ev);
    }
    for (auto &ln : c->lanes) {
        DevBuf *lb[] = {&ln.d_start, &ln.d_end, &ln.d_list[PRE], &ln.d_list[SUF], &ln.d_fb[PRE], &ln.d_fb[SUF], &ln.d_c32, &ln.d_t64, &ln.d_keys,
                        &ln.d_koff, &ln.d_klen, &ln.d_khash, &ln.d_owner, &ln.d_wins, &ln.d_bestkey, &ln.d_cbval, &ln.d_fb2,
                        &ln.d_rtext, &ln.d_rspans, &ln.d_rsrc, &ln.d_rstart, &ln.d_rend};
        for (auto *b : lb) b->release();
        if (ln.done) cudaEventDestroy(ln.done);
        if (ln.ev_scanned) cudaEventDestroy(ln.ev_scanned);
        if (ln.ev_aligned) cudaEventDestroy(ln.ev_aligned);
        if (ln.st) cudaStreamDestroy(ln.st);
        if (ln.st_dp) cudaStreamDestroy(ln.st_dp);
    }
    if (c->ev_fork) cudaEventDestroy(c->ev_fork);
    if (c->ev_k4) cudaEventDestroy(c->ev_k4);
    for (auto &side : c->side) side.d_code.release();
    c->diag_fwd.release(); c->diag_rev.release();
    DevBuf *bufs[] = {&c->d_generic_scratch, &c->t_slots,
                      &c->t_row_hash, &c->t_row_off, &c->t_row_len, &c->t_row_slot, &c->t_arena, &c->t_counters, &c->t_row_count,
                      &c->m_part_rows, &c->m_part_keys, &c->m_cursors, &c->m_chunk_off, &c->m_send, &c->m_recv,
                      &c->d_aligned_text, &c->d_span_sum,
                      &c->x_block_bytes, &c->x_block_rows, &c->x_offsets, &c->x_counts, &c->x_data,
                      &c->p_tiles, &c->p_line_end, &c->p_err, &c->g_tail, &c->g_info};
    for (auto *b : bufs) b->release();
    c->g_pin.release(); c->m_pin.release(); c->snap_pin.release();
    for (auto &sn : c->snaps) if (sn.ev) cudaEventDestroy(sn.ev);
    c->h_offsets.release(); c->h_counts.release(); c->h_data.release();
    for (auto &ev : c->evpool) if (ev) cudaEventDestroy(ev);
    if (c->m_filled) cudaEventDestroy(c->m_filled);
    if (c->st_compute && c->own_compute_stream) cudaStreamDestroy(c->st_compute);
    if (c->st_copy) cudaStreamDestroy(c->st_copy);
    if (c->st_ingest) cudaStreamDestroy(c->st_ingest);
    if (c->st_parse) cudaStreamDestroy(c->st_parse);
    delete c;
    return VFB_OK;
}

int vfb_set_profiling(vfb_ctx *c, int enabled)
{
    if (!c) { set_error("null context"); return VFB_ERR_ARG; }
    c->profiling = enabled != 0;
    return VFB_OK;
}

int vfb_set_progress(vfb_ctx *c, vfb_progress_fn fn, void *user)
{
    if (!c) { set_error("null context"); return VFB_ERR_ARG; }
    c->progress_fn = fn;
    c->progress_user = user;
    c->progress_last = std::chrono::steady_clock::time_point{};
    return VFB_OK;
}

int vfb_table_clear(vfb_ctx *c)
{
    if (!c) { set_error("null context"); return VFB_ERR_ARG; }
    VFB_CUDA(cudaSetDevice(c->device));
    { const int jrc = lanes_join(c); if (jrc) return jrc; }
    snaps_reset(c);
    VFB_CUDA(cudaMemsetAsync(c->tab.slots, 0, c->tab.capacity * 8 * VFB_SLOT_WORDS, c->st_compute));
    VFB_CUDA(cudaMemsetAsync(c->tab.counters, 0, 8 * 8, c->st_compute));
    return VFB_OK;
}

int vfb_reset(vfb_ctx *c)
{
    int rc = vfb_table_clear(c);
    if (rc) return rc;
    for (auto &ln : c->lanes) VFB_CUDA(cudaMemsetAsync(ln.d_t64.p, 0, T_COUNT64 * 8, c->st_compute));
    int kind = c->stats.dp_kernel_kind;
    memset(&c->stats, 0, sizeof c->stats);
    c->stats.dp_kernel_kind = kind;
    c->diag_valid = false;
    return VFB_OK;
}

}  // extern "C"

// ------------------------------------------------------------------------------------ batch
__global__ void k_accumulate(unsigned long long *t64, const uint32_t *c32, uint32_t win_cap)
{
    t64[T_DPPRE] += c32[C_NPRE];
    t64[T_DPSUF] += c32[C_NSUF];
    t64[T_WINDOWS] += (c32[C_NWINPRE] < win_cap ? c32[C_NWINPRE] : win_cap) + (c32[C_NWINSUF] < win_cap ? c32[C_NWINSUF] : win_cap);
}

// What one pass over a batch reads and writes: the forward pass works on the batch's text and the lane's d_start /
// d_end, the reverse pass (both_strands) on the gathered reverse complements and d_rstart / d_rend.  `bound` holds
// them by side (start: prefix, end: suffix); `diag` is null without diagnostics.
struct Pass {
    const uint8_t *text;
    const vfb_span *spans;
    uint32_t *bound[2];
    const DiagBufs *diag;
};

// The alignments of adapter side `s`, as a fallback chain: the windowed DP (filter -> DP on the flagged windows ->
// resolve) passes the reads it cannot take to the packed full-matrix kernel, which passes the reads too long for the
// packed word (normally none) to the unpacked one.  Each stage runs only where vfb_create planned it.
static int run_dp(vfb_ctx *c, Lane &ln, cudaStream_t st, const Pass &ps, int s, uint32_t n_batch, cudaEvent_t *pev)
{
    int rc;
    const AdapterSide &side = c->side[s];
    uint32_t *c32 = ln.d_c32.as<uint32_t>();
    DpJob job;
    memset(&job, 0, sizeof job);
    job.text = ps.text;
    job.spans = ps.spans;
    job.worklist = ln.d_list[s].as<uint32_t>();
    job.n_items = c32 + C_NPRE + s;
    job.bound = ps.bound[s];
    if (ps.diag) {
        job.diag_score = ps.diag->score[s].as<int32_t>();
        job.diag_len = ps.diag->len[s].as<int32_t>();
    }
    job.cells = ln.d_t64.as<unsigned long long>() + T_CELLS;
    if (s == PRE && c->side[SUF].align && !(c->prm.dp_compute_all || c->prm.diagnostics)) {
        job.next_list = ln.d_list[SUF].as<uint32_t>();
        job.n_next = c32 + C_NSUF;
        job.other_bound = ps.bound[SUF];
    }
    job.is_prefix = s == PRE;
    job.min_accept = side.min_accept;
    job.adapter_len = (uint32_t)side.seq.size();
    if (side.packed)
        for (size_t i = 0; i < side.seq.size(); ++i) job.adapter_code[i] = (uint8_t)dp_code((uint8_t)side.seq[i]);
    DpJob rest = job;                   // the reads the next stage of the chain takes
    uint32_t *fb = ln.d_fb[s].as<uint32_t>(), *nfb = c32 + C_FBPRE + s;
    if (side.win_k >= 0) {
        if ((rc = launch_dp_windowed(job, side.lay, side.win_k, side.lcap, n_batch, ln.d_wins.p, c32 + C_NWINPRE + s,
                                     ln.win_cap, ln.d_bestkey.as<unsigned long long>(), ln.d_cbval.as<unsigned long long>(),
                                     fb, nfb, ln.d_t64.as<unsigned long long>() + T_CELLSCOMP,
                                     c32 + C_WORKPRE + 64 * s /* the window cursor sits 32 words on */, c->sm_count, st,
                                     pev ? pev[8 + 2 * s] : nullptr, pev ? pev[9 + 2 * s] : nullptr)))
            return rc;
        rest.worklist = fb;
        rest.n_items = nfb;
        fb = ln.d_fb2.as<uint32_t>();
        nfb = c32 + C_FB2PRE + s;
        c->stats.dp_kernel_launches += 3;
    }
    if (side.packed) {
        if ((rc = launch_dp_packed_ex(rest, side.lay, side.lcap, fb, nfb, c->sm_count, st))) return rc;
        rest.worklist = fb;
        rest.n_items = nfb;
        c->stats.dp_kernel_launches += 1;
    }
    DpGenericJob gj;
    gj.base = rest;
    gj.d_adapter_code = side.d_code.as<uint8_t>();
    gj.sc = c->sc;
    gj.scratch = c->d_generic_scratch.as<int32_t>();
    gj.n_threads = c->generic_threads;
    if ((rc = launch_dp_generic(gj, c->sm_count, st))) return rc;
    c->stats.dp_kernel_launches += 1;
    return VFB_OK;
}

// Scan and alignments of one pass (see Pass), queued on `st` with the alignment kernels on `sd`.
static int queue_scan_dp(vfb_ctx *c, Lane &ln, cudaStream_t st, cudaStream_t sd, const Pass &ps, uint32_t n,
                         uint64_t text_bytes_hint, cudaEvent_t *pev)
{
    int rc;
    const bool prof = pev != nullptr, diag = c->prm.diagnostics != 0, split = sd != st;
    if (prof) VFB_CUDA(cudaEventRecord(pev[0], st));
    VFB_CUDA(cudaMemsetAsync(ln.d_c32.p, 0, C_COUNT32 * 4, st));
    VFB_CUDA(cudaMemsetAsync(ln.d_t64.as<unsigned long long>() + T_KEYBYTES, 0, 8, st));
    ScanJob sj;
    memset(&sj, 0, sizeof sj);
    sj.text = ps.text; sj.spans = ps.spans; sj.n_reads = n; sj.text_bytes = text_bytes_hint;
    sj.start = ps.bound[PRE]; sj.end = ps.bound[SUF];
    if (c->side[PRE].align) { sj.list_pre = ln.d_list[PRE].as<uint32_t>(); sj.n_pre = ln.d_c32.as<uint32_t>() + C_NPRE; }
    if (c->side[SUF].align) { sj.list_suf = ln.d_list[SUF].as<uint32_t>(); sj.n_suf = ln.d_c32.as<uint32_t>() + C_NSUF; }
    sj.compute_all = (c->prm.dp_compute_all || diag) ? 1 : 0;
    sj.force_general = c->prm.force_general_scan;
    if ((rc = launch_scan(sj, c->side[PRE].ad, c->side[SUF].ad, c->sm_count, st))) return rc;
    if (prof) VFB_CUDA(cudaEventRecord(pev[1], st));
    if (diag) {
        for (int s = 0; s < 2; ++s)
            VFB_CUDA(cudaMemcpyAsync(ps.diag->exact[s].p, ps.bound[s], (size_t)n * 4, cudaMemcpyDeviceToDevice, st));
        // "no DP ran" markers: score = INT32_MIN (0x80000000), len = -1
        for (int s = 0; s < 2; ++s) VFB_CUDA(cudaMemsetAsync(ps.diag->len[s].p, 0xFF, (size_t)n * 4, st));
        for (int s = 0; s < 2; ++s) VFB_CUDA(cudaMemsetAsync(ps.diag->score[s].p, 0, (size_t)n * 4, st));
    }
    // DP.  The prefix pass runs first: reads it rejects need no suffix alignment (no region
    // either way, src/lib.rs:288), reads it accepts join the suffix worklist if they need one.
    // split mode: the (ALU-bound) alignment kernels of the batch run on the lane's lower-priority stream, so that the
    // other lane's memory-bound kernels get SM resources as soon as alignment blocks retire
    if (split) {
        VFB_CUDA(cudaEventRecord(ln.ev_scanned, st));
        VFB_CUDA(cudaStreamWaitEvent(sd, ln.ev_scanned, 0));
    }
    for (int s = 0; s < 2; ++s) {
        if (prof) VFB_CUDA(cudaEventRecord(pev[2 + 2 * s], st));
        if (c->side[s].align) if ((rc = run_dp(c, ln, sd, ps, s, n, pev))) return rc;
        if (prof) VFB_CUDA(cudaEventRecord(pev[3 + 2 * s], st));
    }
    k_accumulate<<<1, 1, 0, sd>>>(ln.d_t64.as<unsigned long long>(), ln.d_c32.as<uint32_t>(), ln.win_cap);
    ++g_launches;
    if (split) {
        VFB_CUDA(cudaEventRecord(ln.ev_aligned, sd));
        VFB_CUDA(cudaStreamWaitEvent(st, ln.ev_aligned, 0));
    }
    return VFB_OK;
}

// Keys and count of one pass.  `probe`: the fused key kernel may look the keys up in the table (it is not known to be
// empty).  The caller has ordered the previous batch's inserts before this pass (ev_k4) unless `k4_wait` is set, in
// which case this waits for them in front of the first kernel that touches the table.
static int queue_keys_count(vfb_ctx *c, Lane &ln, cudaStream_t st, const Pass &ps, uint32_t n, uint64_t text_bytes_hint,
                            bool probe, bool k4_wait, cudaEvent_t *pev)
{
    int rc;
    KeyJob kj;
    kj.text = ps.text; kj.spans = ps.spans;
    kj.start = ps.bound[PRE]; kj.end = ps.bound[SUF];
    kj.n_reads = n; kj.text_bytes = text_bytes_hint; kj.skip_translation = c->prm.skip_translation;
    kj.keys = ln.d_keys.as<uint8_t>(); kj.koff = ln.d_koff.as<uint64_t>();
    kj.key_cursor = ln.d_t64.as<unsigned long long>() + T_KEYBYTES;
    kj.klen = ln.d_klen.as<uint32_t>(); kj.khash = ln.d_khash.as<uint64_t>();
    kj.hash_bits = c->prm.debug_hash_bits;
    kj.flank_bytes = (uint32_t)(c->side[PRE].seq.size() + c->side[SUF].seq.size());
    // the table work of a batch claims slots by batch-relative index, and the fused key kernel reads slots without
    // fences: one batch at a time from here on
    bool k4_waited = false;
    InsertJob ij;
    ij.keys = kj.keys; ij.klen = kj.klen; ij.khash = kj.khash; ij.kcount = nullptr; ij.koff = kj.koff;
    ij.key_stride = 0; ij.n_keys = n; ij.owner_slot = ln.d_owner.as<uint32_t>();
    int frc = -1;
    if (c->fused_count && probe) {
        if (k4_wait) { VFB_CUDA(cudaStreamWaitEvent(st, c->ev_k4, 0)); k4_waited = true; }
        frc = launch_keys_count(kj, c->tab, ln.d_c32.as<uint32_t>() + C_NMISS, st);
        if (frc > 0) return frc;
        if (frc == VFB_OK) { ij.n_keys_dev = ln.d_c32.as<uint32_t>() + C_NMISS; ++c->stats.fused_batches; }
    }
    if (frc != VFB_OK && (rc = launch_keys(kj, st))) return rc;
    if (pev) VFB_CUDA(cudaEventRecord(pev[6], st));

    if (k4_wait && !k4_waited) VFB_CUDA(cudaStreamWaitEvent(st, c->ev_k4, 0));
    if ((rc = launch_insert(c->tab, ij, st))) return rc;
    return VFB_OK;
}

// both_strands needs every offset of the gathered text in 32 bits: a batch's span lengths may sum to at most this.
#define VFB_STRAND_TEXT_MAX 0xFFFFFFFFull

// The hot loop over one device-resident batch (all work queued on the compute stream).
// span_len_ub bounds the SUM of the batch's span lengths (it sizes the key space: spans may overlap or repeat, so
// the text range they address is not a bound); text_bytes_hint is the text this batch's reads are spread over (it
// sizes the shared-memory tiles of the scan and key kernels; 0 = span_len_ub).
//
// both_strands: forward scan -> forward DP -> gather of the reads without a forward region (their reverse
// complements, k_strand_gather) -> forward keys and count -> reverse scan -> reverse DP -> reverse keys and count, all
// on the lane, the reverse pass reusing the lane's scratch.  The reverse pass runs over n reads: the span list is
// zeroed first, so the entries past the gathered ones are empty reads, which no kernel does work for.  A read yields a
// key on at most one strand, so the batch's bounds on new rows and key bytes are those of one pass.
static int process_batch(vfb_ctx *c, const uint8_t *d_text, const vfb_span *d_spans, uint32_t n,
                         uint64_t span_len_ub, uint64_t text_bytes_hint = 0, unsigned *lanes_used = nullptr)
{
    const uint64_t span_bytes_upper = span_len_ub;
    if (!text_bytes_hint) text_bytes_hint = span_bytes_upper;
    int rc;
    if (n == 0) return VFB_OK;
    const bool both = c->prm.both_strands != 0;
    if (both && span_len_ub > VFB_STRAND_TEXT_MAX) { set_error("both_strands: the reads of a batch exceed 4 GiB"); return VFB_ERR_ARG; }
    // the lane: with two lanes consecutive batches alternate, each on its own stream, forked from the compute stream
    // (whatever produced the batch's inputs was ordered into that stream by the caller)
    const int li = c->n_lanes > 1 ? (int)(c->lane_seq++ & 1u) : 0;
    Lane &ln = c->lanes[li];
    cudaStream_t st = c->n_lanes > 1 ? ln.st : c->st_compute;
    if (lanes_used) *lanes_used |= 1u << li;
    const bool prof = c->profiling;
    // scratch
    if ((rc = ln.d_start.ensure((size_t)n * 4))) return rc;
    if ((rc = ln.d_end.ensure((size_t)n * 4))) return rc;
    for (int s = 0; s < 2; ++s)
        if (c->side[s].align) { if ((rc = ln.d_list[s].ensure((size_t)n * 4))) return rc; if ((rc = ln.d_fb[s].ensure((size_t)n * 4))) return rc; }
    // keys: sum of padded key lengths <= bytes/(3|1) + 16 per read
    const uint64_t key_bytes_ub = (c->prm.skip_translation ? span_bytes_upper : span_bytes_upper / 3) + 16ull * n;
    if ((rc = ln.d_keys.ensure(key_bytes_ub))) return rc;
    if ((rc = ln.d_koff.ensure((size_t)n * 8))) return rc;
    if ((rc = ln.d_klen.ensure((size_t)n * 4))) return rc;
    if ((rc = ln.d_khash.ensure((size_t)n * 8))) return rc;
    if ((rc = ln.d_owner.ensure((size_t)n * 4))) return rc;
    if (c->side[PRE].win_k >= 0 || c->side[SUF].win_k >= 0) {
        const uint32_t cap = n < 0x3FFFFFFFu ? n * 2u + 1024u : 0x7FFFFFFFu;
        if ((rc = ln.d_wins.ensure((size_t)cap * dpw_item_bytes()))) return rc;
        ln.win_cap = (uint32_t)(ln.d_wins.cap / dpw_item_bytes());
        if (c->prm.debug_win_cap > 0 && (uint32_t)c->prm.debug_win_cap < ln.win_cap) ln.win_cap = (uint32_t)c->prm.debug_win_cap;
        if ((rc = ln.d_bestkey.ensure((size_t)n * 8))) return rc;
        if ((rc = ln.d_cbval.ensure((size_t)n * 8))) return rc;
        if ((rc = ln.d_fb2.ensure((size_t)n * 4))) return rc;
    }
    const bool diag = c->prm.diagnostics != 0;
    if (diag && (rc = c->diag_fwd.ensure((size_t)n * 4))) return rc;
    Pass fwd{d_text, d_spans, {ln.d_start.as<uint32_t>(), ln.d_end.as<uint32_t>()}, diag ? &c->diag_fwd : nullptr};
    Pass rev{};
    if (both) {
        // the gathered text sits 16 bytes into its buffer and is followed by 16 more: the kernels load aligned 16-byte
        // chunks around each read
        if ((rc = ln.d_rtext.ensure(span_len_ub + 32))) return rc;
        if ((rc = ln.d_rspans.ensure((size_t)n * 8))) return rc;
        if ((rc = ln.d_rsrc.ensure((size_t)n * 4))) return rc;
        if ((rc = ln.d_rstart.ensure((size_t)n * 4))) return rc;
        if ((rc = ln.d_rend.ensure((size_t)n * 4))) return rc;
        if (diag && (rc = c->diag_rev.ensure((size_t)n * 4))) return rc;
        rev = Pass{ln.d_rtext.as<uint8_t>() + 16, ln.d_rspans.as<vfb_span>(), {ln.d_rstart.as<uint32_t>(), ln.d_rend.as<uint32_t>()},
                   diag ? &c->diag_rev : nullptr};
    }
    if ((rc = table_reserve(c, n, key_bytes_ub, true))) return rc;
    cudaEvent_t *pev = nullptr, *pev_rev = nullptr;
    if (prof) {
        // two consecutive groups of 12 events with both_strands (taken before either pointer is kept: the pool may grow)
        const size_t first = c->ev_used;
        if ((rc = prof_events(c, &pev))) return rc;
        if (both && (rc = prof_events(c, &pev_rev))) return rc;
        pev = &c->evpool[first];
        if (both) pev_rev = pev + 12;
    }
    if (c->n_lanes > 1) {
        VFB_CUDA(cudaEventRecord(c->ev_fork, c->st_compute));
        VFB_CUDA(cudaStreamWaitEvent(st, c->ev_fork, 0));
    }
    const bool split = c->n_lanes > 1 && !prof;
    cudaStream_t sd = split ? ln.st_dp : st;
    if ((rc = queue_scan_dp(c, ln, st, sd, fwd, n, text_bytes_hint, pev))) return rc;
    unsigned long long *t64 = ln.d_t64.as<unsigned long long>();
    if (both) {
        VFB_CUDA(cudaMemsetAsync(ln.d_rspans.p, 0, (size_t)n * 8, st));
        VFB_CUDA(cudaMemsetAsync(t64 + T_GATHER, 0, 8, st));
        StrandJob sj{d_spans, fwd.bound[PRE], fwd.bound[SUF], n, d_text, ln.d_rtext.as<uint8_t>() + 16, ln.d_rspans.as<vfb_span>(),
                     ln.d_rsrc.as<uint32_t>(), t64 + T_GATHER, t64 + T_REVREADS};
        if ((rc = launch_strand_gather(sj, c->sm_count, st))) return rc;
    }
    // (a table that is known to be empty — the first batch after a clear — has nothing to find: the probe would
    // only cost)
    const bool k4_wait = c->n_lanes > 1 && c->k4_pending;
    if ((rc = queue_keys_count(c, ln, st, fwd, n, text_bytes_hint, c->ub_rows > 0, k4_wait, pev))) return rc;
    if (both) {
        if (prof) VFB_CUDA(cudaEventRecord(pev[7], st));
        if ((rc = queue_scan_dp(c, ln, st, sd, rev, n, text_bytes_hint, pev_rev))) return rc;
        // the forward pass may have added rows: the reverse keys always probe
        if ((rc = launch_strand_tally(t64 + T_REVCOUNTED, c->tab.counters, false, st))) return rc;
        if ((rc = queue_keys_count(c, ln, st, rev, n, text_bytes_hint, true, false, pev_rev))) return rc;
        if ((rc = launch_strand_tally(t64 + T_REVCOUNTED, c->tab.counters, true, st))) return rc;
        pev = pev_rev;
    }
    if ((rc = snaps_push(c, n, key_bytes_ub, st))) return rc;
    if (c->n_lanes > 1) {
        VFB_CUDA(cudaEventRecord(c->ev_k4, st));
        c->k4_pending = true;
        VFB_CUDA(cudaEventRecord(ln.done, st));
        ln.pending = true;
    }
    if (prof) VFB_CUDA(cudaEventRecord(pev[7], st));
    c->stats.reads += n;
    c->diag_n = n;
    c->diag_valid = diag;
    return VFB_OK;
}

// A staging slot may be refilled once the batches that read it are done: on whichever lanes they ran.
static int slot_wait(Slot &s)
{
    for (int li = 0; li < VFB_LANES; ++li)
        if (s.busy & (1u << li)) VFB_CUDA(cudaEventSynchronize(s.computed[li]));
    s.busy = 0;
    return VFB_OK;
}

static int mark_computed(vfb_ctx *c, cudaEvent_t *ev, unsigned *busy, unsigned lanes_used)
{
    if (c->n_lanes <= 1) {
        VFB_CUDA(cudaEventRecord(ev[0], c->st_compute));
        *busy = 1u;
        return VFB_OK;
    }
    *busy = 0;
    for (int li = 0; li < VFB_LANES; ++li)
        if (lanes_used & (1u << li)) {
            VFB_CUDA(cudaEventRecord(ev[li], c->lanes[li].st));
            *busy |= 1u << li;
        }
    return VFB_OK;
}

extern "C" {

int vfb_submit_device(vfb_ctx *c, const uint8_t *d_text, uint64_t text_bytes, const vfb_span *d_spans,
                      uint64_t n_reads)
{
    if (!c || (n_reads && (!d_text || !d_spans))) { set_error("null argument"); return VFB_ERR_ARG; }
    if (text_bytes > 0x100000000ull) { set_error("a text buffer is addressed with 32-bit offsets: at most 4 GiB per call"); return VFB_ERR_ARG; }
    VFB_CUDA(cudaSetDevice(c->device));
    const uint64_t before = g_launches;
    uint64_t done = 0;
    int rc = VFB_OK;
    // The kernels pull 16-byte ALIGNED chunks around each read.  That stays inside the caller's
    // buffer iff both of its ends are 16-byte aligned; otherwise the text is first copied into
    // an aligned, padded buffer of ours (one extra pass over it) so that no load can leave
    // memory the caller handed over.
    const uintptr_t a_lo = reinterpret_cast<uintptr_t>(d_text), a_hi = a_lo + text_bytes;
    if ((a_lo | a_hi) & 15u) {
        const size_t shift = a_lo & 15u;
        if ((rc = c->d_aligned_text.ensure(text_bytes + 48))) return rc;
        uint8_t *dst = c->d_aligned_text.as<uint8_t>() + shift;      // same alignment phase as the source
        VFB_CUDA(cudaMemcpyAsync(dst, d_text, text_bytes, cudaMemcpyDeviceToDevice, c->st_compute));
        d_text = dst;
    }
    if ((rc = c->d_span_sum.ensure(16))) return rc;
    uint64_t n = 0;
    while (done < n_reads) {
        if (!n) n = n_reads - done < c->batch_reads ? n_reads - done : c->batch_reads;
        // the spans are the caller's: every one must lie inside the buffer, and the key space of the batch is
        // bounded by the sum of their lengths (overlapping and repeated spans are legal)
        unsigned long long chk[2] = {0, 0};
        VFB_CUDA(cudaMemsetAsync(c->d_span_sum.p, 0, 16, c->st_compute));
        if ((rc = launch_span_check(d_spans + done, n, text_bytes, c->d_span_sum.as<unsigned long long>(), c->st_compute))) break;
        VFB_CUDA(cudaMemcpyAsync(chk, c->d_span_sum.p, 16, cudaMemcpyDeviceToHost, c->st_compute));
        VFB_CUDA(cudaStreamSynchronize(c->st_compute));
        c->stats.d2h_bytes += 16;
        if (chk[1]) { set_error("span outside the text buffer"); rc = VFB_ERR_ARG; break; }
        if (c->prm.both_strands && chk[0] > VFB_STRAND_TEXT_MAX) {
            // the gathered reverse complements need 32-bit offsets: only overlapping spans get here; halve and measure again
            if (n == 1) { set_error("both_strands: a read longer than 4 GiB"); rc = VFB_ERR_ARG; break; }
            n /= 2;
            continue;
        }
        if ((rc = process_batch(c, d_text, d_spans + done, (uint32_t)n, chk[0],
                                (uint64_t)((double)text_bytes * (double)n / (double)n_reads) + 1))) break;
        done += n;
        n = 0;
    }
    bump_launches(c, before);
    return rc;
}

int vfb_submit_host(vfb_ctx *c, const uint8_t *text, uint64_t text_bytes, const vfb_span *spans, uint64_t n_reads)
{
    if (!c || (n_reads && (!text || !spans))) { set_error("null argument"); return VFB_ERR_ARG; }
    if (text_bytes > 0x100000000ull) { set_error("a text buffer is addressed with 32-bit offsets: at most 4 GiB per call"); return VFB_ERR_ARG; }
    VFB_CUDA(cudaSetDevice(c->device));
    const uint64_t before = g_launches;
    cudaPointerAttributes at;
    bool pinned_text = false, pinned_spans = false;
    if (cudaPointerGetAttributes(&at, text) == cudaSuccess) pinned_text = at.type == cudaMemoryTypeHost; else cudaGetLastError();
    if (cudaPointerGetAttributes(&at, spans) == cudaSuccess) pinned_spans = at.type == cudaMemoryTypeHost; else cudaGetLastError();
    int rc = VFB_OK;
    uint64_t done = 0;
    while (done < n_reads && rc == VFB_OK) {
        // cut a batch: up to batch_reads reads whose text range fits batch_bytes.  The common case — the next
        // batch_reads spans fit — is checked on several threads (min / max / sum / bounds over 12.5 M spans take
        // 37 ms on one core, and the copy cannot be queued before the range is known)
        uint64_t n = 0, lo = UINT64_MAX, hi = 0, len_sum = 0;
        bool cut = false;
        {
            const uint64_t cand = n_reads - done < c->batch_reads ? n_reads - done : c->batch_reads;
            int nt = (int)std::thread::hardware_concurrency();
            if (nt > 8) nt = 8;
            if (cand >= (1u << 20) && nt > 1) {
                struct Part { uint64_t lo = UINT64_MAX, hi = 0, sum = 0; bool bad = false; };
                std::vector<Part> parts((size_t)nt);
                auto scan = [&](int t) {
                    const uint64_t a = done + cand * (uint64_t)t / (uint64_t)nt, b = done + cand * (uint64_t)(t + 1) / (uint64_t)nt;
                    Part p;
                    for (uint64_t i = a; i < b; ++i) {
                        const vfb_span s = spans[i];
                        const uint64_t e = (uint64_t)s.off + s.len;
                        p.lo = s.off < p.lo ? s.off : p.lo;
                        p.hi = e > p.hi ? e : p.hi;
                        p.sum += s.len;
                        p.bad |= e > text_bytes;
                    }
                    parts[(size_t)t] = p;
                };
                std::vector<std::thread> pool;
                for (int t = 1; t < nt; ++t) pool.emplace_back(scan, t);
                scan(0);
                for (auto &t : pool) t.join();
                Part all;
                for (const Part &p : parts) {
                    all.lo = p.lo < all.lo ? p.lo : all.lo;
                    all.hi = p.hi > all.hi ? p.hi : all.hi;
                    all.sum += p.sum;
                    all.bad |= p.bad;
                }
                if (!all.bad && all.hi >= all.lo && all.hi - all.lo <= c->batch_bytes &&
                    !(c->prm.both_strands && all.sum > VFB_STRAND_TEXT_MAX)) {
                    n = cand; lo = all.lo; hi = all.hi; len_sum = all.sum;
                    cut = true;
                }
            }
        }
        while (!cut && done + n < n_reads && n < c->batch_reads) {
            const vfb_span s = spans[done + n];
            if ((uint64_t)s.off + s.len > text_bytes) { set_error("span outside the text buffer"); rc = VFB_ERR_ARG; break; }
            const uint64_t nlo = s.off < lo ? s.off : lo, nhi = (uint64_t)s.off + s.len > hi ? (uint64_t)s.off + s.len : hi;
            if (n > 0 && nhi - nlo > c->batch_bytes) break;
            // both_strands: the gathered reverse complements need 32-bit offsets (only overlapping spans get here)
            if (n > 0 && c->prm.both_strands && len_sum + s.len > VFB_STRAND_TEXT_MAX) break;
            lo = nlo; hi = nhi; len_sum += s.len; ++n;
        }
        if (rc) break;
        if (n == 0) { set_error("a read is larger than batch_bytes"); rc = VFB_ERR_ARG; break; }
        if (hi < lo) { lo = 0; hi = 0; }
        const uint64_t bytes = hi - lo;
        Slot &s = c->slots[c->batch_seq & 1];
        if ((rc = slot_wait(s))) break;
        if ((rc = s.d_text.ensure(bytes + 32))) break;     // aligned 16-byte loads may run past the last read
        if ((rc = s.d_spans.ensure(n * sizeof(vfb_span)))) break;
        const uint8_t *src_text = text + lo;
        const vfb_span *src_spans = spans + done;
        if (!pinned_text) {
            if ((rc = s.h_text.ensure(bytes))) break;
            memcpy(s.h_text.p, src_text, bytes);
            src_text = (const uint8_t *)s.h_text.p;
        }
        if (!pinned_spans) {
            if ((rc = s.h_spans.ensure(n * sizeof(vfb_span)))) break;
            memcpy(s.h_spans.p, src_spans, n * sizeof(vfb_span));
            src_spans = (const vfb_span *)s.h_spans.p;
        }
        VFB_CUDA(cudaMemcpyAsync(s.d_spans.p, src_spans, n * sizeof(vfb_span), cudaMemcpyHostToDevice, c->st_copy));
        if (bytes) VFB_CUDA(cudaMemcpyAsync(s.d_text.p, src_text, bytes, cudaMemcpyHostToDevice, c->st_copy));
        VFB_CUDA(cudaEventRecord(s.copied, c->st_copy));
        VFB_CUDA(cudaStreamWaitEvent(c->st_compute, s.copied, 0));
        c->stats.h2d_bytes += bytes + n * sizeof(vfb_span);
        // span offsets stay relative to the caller's buffer: bias the device base by -lo
        const uint8_t *d_base = s.d_text.as<uint8_t>() - lo;
        unsigned used = 0;
        rc = process_batch(c, d_base, s.d_spans.as<vfb_span>(), (uint32_t)n, len_sum, bytes, &used);
        if (rc) break;
        if ((rc = mark_computed(c, s.computed, &s.busy, used))) break;
        ++c->batch_seq;
        done += n;
    }
    bump_launches(c, before);
    return rc;
}

}  // extern "C"

__global__ void k_parse_err_fold(uint32_t *err32, unsigned long long base, unsigned long long *global)
{
    if (*err32 != 0xFFFFFFFFu) atomicMin(global, base + *err32);
    *err32 = 0xFFFFFFFFu;
}

static int submit_fastq_impl(vfb_ctx *c, const uint8_t *pinned_text, uint64_t host_len, const uint8_t *dev_text, uint64_t dev_len,
                            int dev_device, uint64_t n_lines, uint64_t record_base, cudaEvent_t copied)
{
    const uint64_t n_bytes = host_len + dev_len;
    if (n_bytes > 0xFFFFFFF0ull || n_lines > 0xFFFFFFF0ull) { set_error("ingest chunk too large"); return VFB_ERR_ARG; }
    VFB_CUDA(cudaSetDevice(c->device));
    const uint64_t before = g_launches;
    const uint32_t n_rec = (uint32_t)(n_lines / 4);
    int rc;
    if (!c->p_err_init) {
        if ((rc = c->p_err.ensure(16))) return rc;
        VFB_CUDA(cudaMemsetAsync(c->p_err.p, 0xFF, 16, c->st_compute));
        c->p_err_init = true;
    }
    Slot &s = c->slots[c->batch_seq & 1];
    const bool tr = trace_on() && dev_len;
    const auto tt0 = std::chrono::steady_clock::now();
    auto tms = [&]() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - tt0).count(); };
    if ((rc = slot_wait(s))) return rc;
    const double t_wait = tms();
    if ((rc = s.d_text.ensure(n_bytes + 32))) return rc;
    if ((rc = s.d_spans.ensure((size_t)(n_rec ? n_rec : 1) * sizeof(vfb_span)))) return rc;
    if ((rc = c->p_tiles.ensure(parse_tile_words((uint32_t)n_bytes) * 8 + 8))) return rc;
    if ((rc = c->p_line_end.ensure((n_lines ? n_lines : 1) * 4))) return rc;
    if (host_len) VFB_CUDA(cudaMemcpyAsync(s.d_text.p, pinned_text, host_len, cudaMemcpyHostToDevice, c->st_copy));
    if (copied) VFB_CUDA(cudaEventRecord(copied, c->st_copy));
    if (dev_len) {
        // text that is already in device memory (plain gzip decoded on the device): device to device, or peer to peer
        uint8_t *dst = s.d_text.as<uint8_t>() + host_len;
        if (dev_device == c->device) VFB_CUDA(cudaMemcpyAsync(dst, dev_text, dev_len, cudaMemcpyDeviceToDevice, c->st_copy));
        else VFB_CUDA(cudaMemcpyPeerAsync(dst, c->device, dev_text, dev_device, dev_len, c->st_copy));
    }
    VFB_CUDA(cudaEventRecord(s.copied, c->st_copy));
    VFB_CUDA(cudaStreamWaitEvent(c->st_compute, s.copied, 0));
    c->stats.h2d_bytes += host_len;
    if (dev_len) VFB_CUDA(cudaEventSynchronize(s.copied));      // the caller lets go of dev_text when this returns
    const double t_copy = tms();
    unsigned used = 0;
    if (n_rec) {
        if ((rc = launch_parse(s.d_text.as<uint8_t>(), (uint32_t)n_bytes, (uint32_t)n_lines, n_rec,
                               c->p_tiles.as<unsigned long long>(), c->p_line_end.as<uint32_t>(),
                               s.d_spans.as<vfb_span>(), c->p_err.as<uint32_t>(), c->st_compute))) return rc;
        k_parse_err_fold<<<1, 1, 0, c->st_compute>>>(c->p_err.as<uint32_t>(), record_base,
                                                     reinterpret_cast<unsigned long long *>(c->p_err.as<uint8_t>() + 8));
        ++g_launches;
        // batches inside the chunk
        uint32_t done = 0;
        while (done < n_rec) {
            const uint32_t n = n_rec - done < c->batch_reads ? n_rec - done : (uint32_t)c->batch_reads;
            if ((rc = process_batch(c, s.d_text.as<uint8_t>(), s.d_spans.as<vfb_span>() + done, n, n_bytes,
                                    (uint64_t)((double)n_bytes * (double)n / (double)n_rec) + 1, &used))) return rc;
            done += n;
        }
    }
    if ((rc = mark_computed(c, s.computed, &s.busy, used))) return rc;
    if (tr) trace("submit_fastq_dev: slot wait %.2f ms, allocations + copies %.2f, parse + batches queued %.2f", t_wait, t_copy - t_wait, tms() - t_copy);
    ++c->batch_seq;
    bump_launches(c, before);
    return VFB_OK;
}

int vfb_internal_submit_fastq(vfb_ctx *c, const uint8_t *pinned_text, uint64_t n_bytes, uint64_t n_lines,
                              uint64_t record_base, cudaEvent_t copied)
{
    return submit_fastq_impl(c, pinned_text, n_bytes, nullptr, 0, -1, n_lines, record_base, copied);
}

int vfb_internal_submit_fastq_dev(vfb_ctx *c, const uint8_t *host_text, uint64_t host_len, const uint8_t *dev_text, uint64_t dev_len,
                                  int dev_device, uint64_t n_lines, uint64_t record_base, cudaEvent_t copied)
{
    return submit_fastq_impl(c, host_text, host_len, dev_text, dev_len, dev_device, n_lines, record_base, copied);
}

// ---- block-gzip segments, in two phases so that several segments (on one device or on several) overlap:
// begin  = H2D of the compressed members + inflate, independent of every other segment;
// finish = what needs the text carried over from the previous segment (the bytes after its last complete record):
//          carry in front of the inflated text, newline count, record framing, tail out, then the hot loop.
// The inflated text sits VFB_TAIL_CAP bytes into its buffer, so that the carry fits in front of it whatever its
// length; the parse kernels want a 16-byte aligned base and skip the (< 16) bytes between it and the carry.
int vfb_internal_bgzf_begin(vfb_ctx *c, const vfb_zpiece *pieces, uint32_t n_pieces, const vfb_member *members,
                            uint32_t n_members, uint64_t text_bytes, void (*release)(void *), void *release_arg, int *slot_out)
{
    uint64_t z_bytes = 0;
    for (uint32_t i = 0; i < n_pieces; ++i) z_bytes += pieces[i].len;
    if (text_bytes + VFB_TAIL_CAP > 0xFFFFFF00ull || z_bytes > 0xFFFFFF00ull) { set_error("ingest segment too large"); return VFB_ERR_ARG; }
    VFB_CUDA(cudaSetDevice(c->device));
    const uint64_t before = g_launches;
    int rc;
    if (!c->p_err_init) {
        if ((rc = c->p_err.ensure(16))) return rc;
        VFB_CUDA(cudaMemsetAsync(c->p_err.p, 0xFF, 16, c->st_ingest));
        c->p_err_init = true;
    }
    const int slot = (int)(c->g_seq % VFB_SEG_SLOTS);
    ++c->g_seq;
    SegSlot &g = c->seg[slot];
    if ((rc = g.text.ensure(VFB_TAIL_CAP + text_bytes + 64))) return rc;
    if ((rc = g.z.ensure(z_bytes + 64))) return rc;
    if ((rc = g.members.ensure((size_t)(n_members ? n_members : 1) * sizeof(vfb_member) + 16))) return rc;
    if ((rc = c->g_info.ensure(64 * VFB_SEG_SLOTS))) return rc;
    // the compressed bytes travel on the copy stream, so that this segment's H2D overlaps the previous segment's
    // inflate (both used to queue on the ingest stream: 1 ms of copy in front of every 5.5 ms inflate); the slot's
    // compressed buffer is free once the inflate that last read it is done
    if (g.used) VFB_CUDA(cudaStreamWaitEvent(c->st_copy, g.inflated, 0));
    uint64_t zo = 0;
    for (uint32_t i = 0; i < n_pieces; ++i) {
        if (pieces[i].len) VFB_CUDA(cudaMemcpyAsync(g.z.as<uint8_t>() + zo, pieces[i].p, pieces[i].len, cudaMemcpyHostToDevice, c->st_copy));
        zo += pieces[i].len;
    }
    if (release) VFB_CUDA(cudaLaunchHostFunc(c->st_copy, release, release_arg));
    if (n_members) VFB_CUDA(cudaMemcpyAsync(g.members.p, members, (size_t)n_members * sizeof(vfb_member), cudaMemcpyHostToDevice, c->st_copy));
    VFB_CUDA(cudaEventRecord(g.copied, c->st_copy));
    VFB_CUDA(cudaStreamWaitEvent(c->st_ingest, g.copied, 0));
    c->stats.h2d_bytes += z_bytes + (uint64_t)n_members * sizeof(vfb_member);
    // the hot loop that last read this slot's text must be done before the inflate overwrites it
    for (int li = 0; li < VFB_LANES; ++li)
        if (g.busy & (1u << li)) VFB_CUDA(cudaStreamWaitEvent(c->st_ingest, g.computed[li], 0));
    g.used = true;
    uint32_t *d_bad = c->g_info.as<uint32_t>() + 16 * slot + 8;
    VFB_CUDA(cudaMemsetAsync(d_bad, 0xFF, 4, c->st_ingest));
    if ((rc = launch_inflate(g.z.as<uint8_t>(), g.members.as<vfb_member>(), n_members, g.text.as<uint8_t>() + VFB_TAIL_CAP, d_bad, c->st_ingest))) return rc;
    VFB_CUDA(cudaEventRecord(g.inflated, c->st_ingest));
    g.text_bytes = text_bytes; g.z_bytes = z_bytes; g.n_members = n_members;
    *slot_out = slot;
    bump_launches(c, before);
    return VFB_OK;
}

int vfb_internal_bgzf_finish(vfb_ctx *c, int slot, const uint8_t *carry, uint64_t carry_len, uint64_t record_base,
                             uint64_t *n_records, uint8_t *tail, uint64_t *tail_len, uint32_t *bad_member)
{
    *n_records = 0; *tail_len = 0; *bad_member = 0xFFFFFFFFu;
    if (carry_len > VFB_TAIL_CAP) { set_error("a FASTQ record is larger than 16 MiB"); return VFB_ERR_FORMAT; }
    VFB_CUDA(cudaSetDevice(c->device));
    const uint64_t before = g_launches;
    SegSlot &g = c->seg[slot];
    cudaStream_t si = c->st_parse;
    VFB_CUDA(cudaStreamWaitEvent(si, g.inflated, 0));
    int rc;
    const uint64_t front = VFB_TAIL_CAP - carry_len;           // where the carried bytes start in the buffer
    const uint32_t skip = (uint32_t)(front & 15u);
    const uint8_t *base = g.text.as<uint8_t>() + (front & ~(uint64_t)15);
    const uint64_t used = skip + carry_len + g.text_bytes;      // bytes from `base`
    if ((rc = c->g_tail.ensure(VFB_TAIL_CAP))) return rc;
    if ((rc = c->g_pin.ensure(VFB_TAIL_CAP + 64))) return rc;
    if ((rc = c->p_tiles.ensure(parse_tile_words((uint32_t)used) * 8 + 8))) return rc;
    uint8_t *pin = (uint8_t *)c->g_pin.p;
    if (carry_len) {
        memcpy(pin, carry, carry_len);
        VFB_CUDA(cudaMemcpyAsync(g.text.as<uint8_t>() + front, pin, carry_len, cudaMemcpyHostToDevice, si));
        c->stats.h2d_bytes += carry_len;
    }
    unsigned long long lines = 0;
    uint32_t bad = 0xFFFFFFFFu;
    uint32_t *d_info = c->g_info.as<uint32_t>() + 16 * slot;
    if (used > skip) {
        if ((rc = launch_parse_count(base, (uint32_t)used, skip, c->p_tiles.as<unsigned long long>(), si))) return rc;
        const uint64_t n_tiles = parse_tile_words((uint32_t)used) - 1;
        VFB_CUDA(cudaMemcpyAsync(&lines, c->p_tiles.as<unsigned long long>() + n_tiles, 8, cudaMemcpyDeviceToHost, si));
    }
    VFB_CUDA(cudaMemcpyAsync(&bad, d_info + 8, 4, cudaMemcpyDeviceToHost, si));
    VFB_CUDA(cudaStreamSynchronize(si));
    c->stats.d2h_bytes += 12;
    *bad_member = bad;
    if (bad != 0xFFFFFFFFu || used <= skip) { bump_launches(c, before); return VFB_OK; }
    const uint32_t n_rec = (uint32_t)(lines / 4);
    if ((rc = c->p_line_end.ensure((lines ? lines : 1) * 4))) return rc;
    if ((rc = g.spans.ensure((size_t)(n_rec ? n_rec : 1) * sizeof(vfb_span)))) return rc;
    if ((rc = launch_parse_index(base, (uint32_t)used, skip, (uint32_t)lines, n_rec, c->p_tiles.as<unsigned long long>(),
                                 c->p_line_end.as<uint32_t>(), g.spans.as<vfb_span>(), c->p_err.as<uint32_t>(),
                                 c->g_tail.as<uint8_t>(), VFB_TAIL_CAP, d_info, si))) return rc;
    if (n_rec) {
        k_parse_err_fold<<<1, 1, 0, si>>>(c->p_err.as<uint32_t>(), record_base,
                                          reinterpret_cast<unsigned long long *>(c->p_err.as<uint8_t>() + 8));
        ++g_launches;
    }
    uint32_t *h_info = reinterpret_cast<uint32_t *>(pin + VFB_TAIL_CAP);
    VFB_CUDA(cudaMemcpyAsync(h_info, d_info, 8, cudaMemcpyDeviceToHost, si));
    // the tail is normally a fraction of one record: fetch a first page with the info, the rest if needed
    VFB_CUDA(cudaMemcpyAsync(pin, c->g_tail.p, 65536, cudaMemcpyDeviceToHost, si));
    VFB_CUDA(cudaEventRecord(g.parsed, si));
    VFB_CUDA(cudaStreamSynchronize(si));
    const uint32_t tl = h_info[1];
    if (tl > VFB_TAIL_CAP) { set_error("a FASTQ record is larger than 16 MiB"); return VFB_ERR_FORMAT; }
    if (tl > 65536) {
        VFB_CUDA(cudaMemcpyAsync(pin, c->g_tail.p, tl, cudaMemcpyDeviceToHost, si));
        VFB_CUDA(cudaStreamSynchronize(si));
    }
    memcpy(tail, pin, tl);
    *tail_len = tl;
    c->stats.d2h_bytes += 8 + tl;
    if (n_rec) {
        VFB_CUDA(cudaStreamWaitEvent(c->st_compute, g.parsed, 0));
        uint32_t done = 0;
        unsigned lanes_used = 0;
        g.busy = 0;
        while (done < n_rec) {
            const uint32_t n = n_rec - done < c->batch_reads ? n_rec - done : (uint32_t)c->batch_reads;
            if ((rc = process_batch(c, base, g.spans.as<vfb_span>() + done, n, used,
                                    (uint64_t)((double)used * (double)n / (double)n_rec) + 1, &lanes_used))) return rc;
            done += n;
        }
        if ((rc = mark_computed(c, g.computed, &g.busy, lanes_used))) return rc;
    }
    *n_records = n_rec;
    bump_launches(c, before);
    return VFB_OK;
}

void vfb_internal_progress(vfb_ctx *c, uint64_t records, uint64_t bytes_done, uint64_t bytes_total, bool final)
{
    if (!c->progress_fn) return;
    const auto now = std::chrono::steady_clock::now();
    if (!final && std::chrono::duration<double>(now - c->progress_last).count() < 0.1) return;
    c->progress_last = now;
    c->progress_fn(records, bytes_done, bytes_total, c->progress_user);
}

int vfb_internal_ingest_threads(vfb_ctx *c)
{
    // The reference's n_threads (src/lib.rs:228, default 3) are its worker threads; here they inflate /
    // read.  A B200 host has cores to spare and the GPU side is never the bottleneck of a gzip file, so the
    // ingest takes at least min(hardware threads, 32) unless VFB_INGEST_THREADS says otherwise.
    int t = c->prm.n_threads < 1 ? 1 : (int)(c->prm.n_threads > 256 ? 256 : c->prm.n_threads);
    if (const char *e = getenv("VFB_INGEST_THREADS")) {
        const int v = atoi(e);
        if (v >= 1) return v > 256 ? 256 : v;
    }
    int hw = (int)std::thread::hardware_concurrency();
    if (hw > 32) hw = 32;
    return t > hw ? t : hw;
}

int vfb_internal_parse_error(vfb_ctx *c, uint64_t *first_bad)
{
    *first_bad = UINT64_MAX;
    if (!c->p_err_init) return VFB_OK;
    VFB_CUDA(cudaSetDevice(c->device));
    unsigned long long v = 0;
    VFB_CUDA(cudaMemcpy(&v, c->p_err.as<uint8_t>() + 8, 8, cudaMemcpyDeviceToHost));
    *first_bad = v;
    // re-arm
    VFB_CUDA(cudaMemset(c->p_err.p, 0xFF, 16));
    return VFB_OK;
}

extern "C" {

int vfb_sync(vfb_ctx *c)
{
    if (!c) { set_error("null context"); return VFB_ERR_ARG; }
    VFB_CUDA(cudaSetDevice(c->device));
    VFB_CUDA(cudaStreamSynchronize(c->st_copy));
    VFB_CUDA(cudaStreamSynchronize(c->st_ingest));
    VFB_CUDA(cudaStreamSynchronize(c->st_parse));
    { const int jrc = lanes_join(c); if (jrc) return jrc; }
    VFB_CUDA(cudaStreamSynchronize(c->st_compute));
    for (auto &s : c->slots) s.busy = 0;
    for (auto &g : c->seg) g.busy = 0;
    return prof_resolve(c);
}

int vfb_fence(vfb_ctx *c)
{
    if (!c) { set_error("null context"); return VFB_ERR_ARG; }
    VFB_CUDA(cudaSetDevice(c->device));
    return lanes_join(c);
}

int vfb_set_lanes(vfb_ctx *c, int n)
{
    if (!c || n < 1 || n > VFB_LANES) { set_error("lanes: 1 or 2"); return VFB_ERR_ARG; }
    int rc = vfb_sync(c);
    if (rc) return rc;
    if (c->prm.diagnostics) n = 1;
    c->n_lanes = n;
    return VFB_OK;
}

int vfb_set_compute_stream(vfb_ctx *c, void *stream)
{
    if (!c) { set_error("null context"); return VFB_ERR_ARG; }
    int rc = vfb_sync(c);
    if (rc) return rc;
    if (c->own_compute_stream && c->st_compute) cudaStreamDestroy(c->st_compute);
    c->st_compute = (cudaStream_t)stream;
    c->own_compute_stream = false;
    return VFB_OK;
}

int vfb_get_stats(vfb_ctx *c, vfb_stats *out)
{
    if (!c || !out) { set_error("null argument"); return VFB_ERR_ARG; }
    int rc = vfb_sync(c);
    if (rc) return rc;
    unsigned long long t64[T_COUNT64] = {0}, ctr[4];
    for (auto &ln : c->lanes) {
        unsigned long long one[T_COUNT64];
        VFB_CUDA(cudaMemcpy(one, ln.d_t64.p, sizeof one, cudaMemcpyDeviceToHost));
        for (int k = 0; k < T_COUNT64; ++k) t64[k] += one[k];
    }
    VFB_CUDA(cudaMemcpy(ctr, c->tab.counters, sizeof ctr, cudaMemcpyDeviceToHost));
    c->stats.dp_cells = t64[T_CELLS];
    c->stats.dp_prefix = t64[T_DPPRE];
    c->stats.dp_suffix = t64[T_DPSUF];
    c->stats.dp_cells_computed = t64[T_CELLSCOMP];
    c->stats.dp_windows = t64[T_WINDOWS];
    c->stats.unique = ctr[0];
    c->stats.counted = ctr[2];
    c->stats.fused_hits = ctr[3];
    c->stats.reverse_reads = t64[T_REVREADS];
    c->stats.reverse_counted = t64[T_REVCOUNTED];
    *out = c->stats;
    return VFB_OK;
}

}  // extern "C"

// The first n rows of a pass's diagnostics columns and boundaries (device) -> vfb_read_diag rows (host).
static int diag_fetch(vfb_ctx *c, const DiagBufs &d, const DevBuf &start, const DevBuf &end, size_t n, vfb_read_diag *out)
{
    if (!n) return VFB_OK;
    std::vector<uint32_t> ep(n), es(n), st(n), en(n);
    std::vector<int32_t> sp(n), lp(n), ss(n), ls(n);
    VFB_CUDA(cudaMemcpy(ep.data(), d.exact[PRE].p, n * 4, cudaMemcpyDeviceToHost));
    VFB_CUDA(cudaMemcpy(es.data(), d.exact[SUF].p, n * 4, cudaMemcpyDeviceToHost));
    VFB_CUDA(cudaMemcpy(st.data(), start.p, n * 4, cudaMemcpyDeviceToHost));
    VFB_CUDA(cudaMemcpy(en.data(), end.p, n * 4, cudaMemcpyDeviceToHost));
    VFB_CUDA(cudaMemcpy(sp.data(), d.score[PRE].p, n * 4, cudaMemcpyDeviceToHost));
    VFB_CUDA(cudaMemcpy(lp.data(), d.len[PRE].p, n * 4, cudaMemcpyDeviceToHost));
    VFB_CUDA(cudaMemcpy(ss.data(), d.score[SUF].p, n * 4, cudaMemcpyDeviceToHost));
    VFB_CUDA(cudaMemcpy(ls.data(), d.len[SUF].p, n * 4, cudaMemcpyDeviceToHost));
    const uint32_t A = (uint32_t)c->side[PRE].seq.size();
    for (size_t i = 0; i < n; ++i) {
        vfb_read_diag r;
        r.exact_prefix = ep[i] == VFB_NONE ? -1 : (int32_t)(ep[i] - A);
        r.exact_suffix = es[i] == VFB_NONE ? -1 : (int32_t)es[i];
        r.score_prefix = lp[i] < 0 ? INT32_MIN : sp[i];
        r.len_prefix = lp[i];
        r.score_suffix = ls[i] < 0 ? INT32_MIN : ss[i];
        r.len_suffix = ls[i];
        r.start = st[i] == VFB_NONE ? -1 : (int32_t)st[i];
        r.end = en[i] == VFB_NONE ? -1 : (int32_t)en[i];
        out[i] = r;
    }
    return VFB_OK;
}

extern "C" {

int vfb_get_diag(vfb_ctx *c, vfb_read_diag *out, uint64_t n_reads)
{
    if (!c || !out) { set_error("null argument"); return VFB_ERR_ARG; }
    if (!c->prm.diagnostics || !c->diag_valid) { set_error("diagnostics were not enabled for the last batch"); return VFB_ERR_ARG; }
    if (n_reads != c->diag_n) { set_error("diagnostics cover exactly the last batch"); return VFB_ERR_ARG; }
    int rc = vfb_sync(c);
    if (rc) return rc;
    const size_t n = (size_t)n_reads;
    if ((rc = diag_fetch(c, c->diag_fwd, c->lanes[0].d_start, c->lanes[0].d_end, n, out))) return rc;
    c->stats.d2h_bytes += n * 32;
    return VFB_OK;
}

int vfb_get_diag_reverse(vfb_ctx *c, vfb_read_diag *out, uint64_t n_reads)
{
    if (!c || !out) { set_error("null argument"); return VFB_ERR_ARG; }
    if (!c->prm.diagnostics || !c->diag_valid) { set_error("diagnostics were not enabled for the last batch"); return VFB_ERR_ARG; }
    if (!c->prm.both_strands) { set_error("the context was created without both_strands"); return VFB_ERR_ARG; }
    if (n_reads != c->diag_n) { set_error("diagnostics cover exactly the last batch"); return VFB_ERR_ARG; }
    int rc = vfb_sync(c);
    if (rc) return rc;
    const size_t n = (size_t)n_reads;
    unsigned long long cursor = 0;
    VFB_CUDA(cudaMemcpy(&cursor, c->lanes[0].d_t64.as<unsigned long long>() + T_GATHER, 8, cudaMemcpyDeviceToHost));
    const size_t m = (size_t)(cursor >> 32);            // gathered reads, in compact order
    std::vector<vfb_read_diag> rows(m);
    std::vector<uint32_t> src(m);
    if ((rc = diag_fetch(c, c->diag_rev, c->lanes[0].d_rstart, c->lanes[0].d_rend, m, rows.data()))) return rc;
    if (m) VFB_CUDA(cudaMemcpy(src.data(), c->lanes[0].d_rsrc.p, m * 4, cudaMemcpyDeviceToHost));
    c->stats.d2h_bytes += 8 + m * 36;
    const vfb_read_diag absent = {-1, -1, INT32_MIN, -1, INT32_MIN, -1, -1, -1};
    for (size_t i = 0; i < n; ++i) out[i] = absent;
    for (size_t i = 0; i < m; ++i) {
        if (src[i] >= n) { set_error("reverse diagnostics: read index out of range"); return VFB_ERR_CUDA; }
        out[src[i]] = rows[i];
    }
    return VFB_OK;
}

}  // extern "C"

// Export, pass 1: slot counts -> row counts, sizes of what will be exported (rows with a non-zero count).
int vfb_internal_export_sizes(vfb_ctx *c, uint64_t *rows_out, uint64_t *bytes_out)
{
    *rows_out = 0; *bytes_out = 0;
    int rc = vfb_sync(c);
    if (rc) return rc;
    const uint64_t before = g_launches;
    unsigned long long ctr[3];
    VFB_CUDA(cudaMemcpy(ctr, c->tab.counters, sizeof ctr, cudaMemcpyDeviceToHost));
    const uint64_t rows = ctr[0];
    c->x_table_rows = rows; c->x_rows = 0; c->x_bytes = 0;
    if (rows == 0) return VFB_OK;
    const uint64_t nb = (rows + 1023) / 1024;
    if ((rc = c->t_row_count.ensure(rows * 8))) return rc;
    if ((rc = c->x_block_bytes.ensure((nb + 2) * 8))) return rc;
    if ((rc = c->x_block_rows.ensure(nb * 8))) return rc;
    unsigned long long *d_totals = c->x_block_bytes.as<unsigned long long>() + nb;
    if ((rc = launch_export_counts(c->tab, rows, c->t_row_count.as<unsigned long long>(), c->st_compute))) return rc;
    if ((rc = launch_export_sizes(c->tab, rows, c->t_row_count.as<unsigned long long>(), c->x_block_bytes.as<unsigned long long>(),
                                  c->x_block_rows.as<unsigned long long>(), d_totals, c->st_compute))) return rc;
    unsigned long long totals[2] = {0, 0};
    VFB_CUDA(cudaMemcpyAsync(totals, d_totals, 16, cudaMemcpyDeviceToHost, c->st_compute));
    VFB_CUDA(cudaStreamSynchronize(c->st_compute));
    c->stats.d2h_bytes += 16 + sizeof ctr;
    c->x_bytes = totals[0]; c->x_rows = totals[1];
    *rows_out = c->x_rows; *bytes_out = c->x_bytes;
    bump_launches(c, before);
    return VFB_OK;
}

// Export, pass 2 (asynchronous on the compute stream): h_offsets receives x_rows offsets (byte_base + ...; the
// closing offset is the caller's), h_counts x_rows counts, h_data x_bytes key bytes.  Pinned destinations.
int vfb_internal_export_write(vfb_ctx *c, uint64_t byte_base, uint64_t *h_offsets, uint64_t *h_counts, uint8_t *h_data)
{
    VFB_CUDA(cudaSetDevice(c->device));
    if (c->x_rows == 0) return VFB_OK;
    const uint64_t before = g_launches;
    int rc;
    if ((rc = c->x_offsets.ensure(c->x_rows * 8))) return rc;
    if ((rc = c->x_counts.ensure(c->x_rows * 8))) return rc;
    if ((rc = c->x_data.ensure(c->x_bytes ? c->x_bytes : 16))) return rc;
    if ((rc = launch_export_gather(c->tab, c->x_table_rows, c->t_row_count.as<unsigned long long>(),
                                   c->x_block_bytes.as<unsigned long long>(), c->x_block_rows.as<unsigned long long>(), byte_base,
                                   c->x_offsets.as<unsigned long long>(), c->x_counts.as<unsigned long long>(),
                                   c->x_data.as<uint8_t>(), c->st_compute))) return rc;
    VFB_CUDA(cudaMemcpyAsync(h_offsets, c->x_offsets.p, c->x_rows * 8, cudaMemcpyDeviceToHost, c->st_compute));
    VFB_CUDA(cudaMemcpyAsync(h_counts, c->x_counts.p, c->x_rows * 8, cudaMemcpyDeviceToHost, c->st_compute));
    if (c->x_bytes) VFB_CUDA(cudaMemcpyAsync(h_data, c->x_data.p, c->x_bytes, cudaMemcpyDeviceToHost, c->st_compute));
    c->stats.d2h_bytes += c->x_rows * 16 + c->x_bytes;
    bump_launches(c, before);
    return VFB_OK;
}

extern "C" {

int vfb_finish(vfb_ctx *c, vfb_table *out)
{
    if (!c || !out) { set_error("null argument"); return VFB_ERR_ARG; }
    memset(out, 0, sizeof *out);
    uint64_t rows = 0, bytes = 0;
    int rc = vfb_internal_export_sizes(c, &rows, &bytes);
    if (rc) return rc;
    // The columns are compacted on the device and land in pinned host buffers owned by the
    // context (valid until the next vfb_finish / vfb_destroy on it).
    if ((rc = c->h_offsets.ensure((rows + 1) * 8))) return rc;
    if ((rc = c->h_counts.ensure((rows ? rows : 1) * 8))) return rc;
    if ((rc = c->h_data.ensure(bytes ? bytes : 16))) return rc;
    out->rows = rows;
    out->key_bytes = bytes;
    out->offsets = (uint64_t *)c->h_offsets.p;
    out->counts = (uint64_t *)c->h_counts.p;
    out->data = (uint8_t *)c->h_data.p;
    out->owner = c;
    if ((rc = vfb_internal_export_write(c, 0, out->offsets, out->counts, out->data))) return rc;
    VFB_CUDA(cudaStreamSynchronize(c->st_compute));
    out->offsets[rows] = bytes;
    return VFB_OK;
}

// ---- Arrow C Data Interface (https://arrow.apache.org/docs/format/CDataInterface.html): the result as a struct
// array {sequence: large_utf8, count: uint64} whose buffers ARE the pinned host columns — nothing is copied on the
// way to pyarrow / polars.  Ownership of the pinned buffers moves from the context into the exported array; its
// release callback hands them back to the pinned pool.
namespace {
struct ArrowHolder {
    std::atomic<int> refs{0};
    PinBuf offsets, data, counts;
    vfb_arrow_array children[2];
    vfb_arrow_array *child_ptrs[2];
    const void *seq_bufs[3], *cnt_bufs[2], *top_bufs[1];
};
void holder_unref(ArrowHolder *h)
{
    if (h->refs.fetch_sub(1) == 1) {
        h->offsets.release(); h->data.release(); h->counts.release();
        delete h;
    }
}
void arrow_child_release(vfb_arrow_array *a)
{
    if (!a || !a->release) return;
    ArrowHolder *h = static_cast<ArrowHolder *>(a->private_data);
    a->release = nullptr;
    holder_unref(h);
}
void arrow_top_release(vfb_arrow_array *a)
{
    if (!a || !a->release) return;
    ArrowHolder *h = static_cast<ArrowHolder *>(a->private_data);
    for (int i = 0; i < 2; ++i)                     // children the consumer has not moved out
        if (h->children[i].release) h->children[i].release(&h->children[i]);
    a->release = nullptr;
    holder_unref(h);
}
struct SchemaHolder {
    vfb_arrow_schema children[2];
    vfb_arrow_schema *child_ptrs[2];
};
void schema_child_release(vfb_arrow_schema *s) { if (s) s->release = nullptr; }
void schema_top_release(vfb_arrow_schema *s)
{
    if (!s || !s->release) return;
    SchemaHolder *h = static_cast<SchemaHolder *>(s->private_data);
    for (int i = 0; i < 2; ++i)
        if (h->children[i].release) h->children[i].release(&h->children[i]);
    s->release = nullptr;
    delete h;
}
}  // namespace

}  // extern "C"

// Wraps three pinned columns (ownership moves into the array) as the Arrow struct array of vfb_finish_arrow.
int vfb_internal_arrow_wrap(PinBuf offsets, PinBuf data, PinBuf counts, uint64_t rows, vfb_arrow_array *out_array,
                            vfb_arrow_schema *out_schema)
{
    ArrowHolder *h = new ArrowHolder;
    h->offsets = offsets; h->data = data; h->counts = counts;
    h->refs = 3;
    h->seq_bufs[0] = nullptr; h->seq_bufs[1] = offsets.p; h->seq_bufs[2] = data.p;
    h->cnt_bufs[0] = nullptr; h->cnt_bufs[1] = counts.p;
    h->top_bufs[0] = nullptr;
    vfb_arrow_array &seq = h->children[0], &cnt = h->children[1];
    memset(&seq, 0, sizeof seq); memset(&cnt, 0, sizeof cnt);
    seq.length = (int64_t)rows; seq.n_buffers = 3; seq.buffers = h->seq_bufs;
    seq.release = arrow_child_release; seq.private_data = h;
    cnt.length = (int64_t)rows; cnt.n_buffers = 2; cnt.buffers = h->cnt_bufs;
    cnt.release = arrow_child_release; cnt.private_data = h;
    h->child_ptrs[0] = &seq; h->child_ptrs[1] = &cnt;
    memset(out_array, 0, sizeof *out_array);
    out_array->length = (int64_t)rows; out_array->n_buffers = 1; out_array->buffers = h->top_bufs;
    out_array->n_children = 2; out_array->children = h->child_ptrs;
    out_array->release = arrow_top_release; out_array->private_data = h;

    SchemaHolder *sh = new SchemaHolder;
    memset(sh->children, 0, sizeof sh->children);
    sh->children[0].format = "U"; sh->children[0].name = "sequence"; sh->children[0].release = schema_child_release;
    sh->children[1].format = "L"; sh->children[1].name = "count"; sh->children[1].release = schema_child_release;
    sh->child_ptrs[0] = &sh->children[0]; sh->child_ptrs[1] = &sh->children[1];
    memset(out_schema, 0, sizeof *out_schema);
    out_schema->format = "+s"; out_schema->name = ""; out_schema->n_children = 2; out_schema->children = sh->child_ptrs;
    out_schema->release = schema_top_release; out_schema->private_data = sh;
    return VFB_OK;
}

extern "C" {

int vfb_finish_arrow(vfb_ctx *c, vfb_arrow_array *out_array, vfb_arrow_schema *out_schema)
{
    if (!c || !out_array || !out_schema) { set_error("null argument"); return VFB_ERR_ARG; }
    vfb_table t;
    int rc = vfb_finish(c, &t);
    if (rc) return rc;
    // the context gives its pinned columns away; its next vfb_finish takes fresh ones from the pool
    PinBuf o = c->h_offsets, d = c->h_data, n = c->h_counts;
    c->h_offsets = PinBuf(); c->h_data = PinBuf(); c->h_counts = PinBuf();
    return vfb_internal_arrow_wrap(o, d, n, t.rows, out_array, out_schema);
}

void vfb_table_free(vfb_table *t)
{
    if (!t) return;
    if (!t->owner) {
        free(t->offsets);
        free(t->data);
        free(t->counts);
    }
    memset(t, 0, sizeof *t);
}

// ------------------------------------------------------------------------------------ merge
}  // extern "C"

// Pass 1 of a partition (asynchronous): slot counts -> row counts, rows and padded key bytes per part; the
// results stay on the device, m_part_rows = [rows per part (n_parts) | key bytes per part (n_parts)].
int vfb_internal_partition_count(vfb_ctx *c, uint32_t n_parts, uint32_t self, uint64_t *table_rows)
{
    int rc = vfb_sync(c);
    if (rc) return rc;
    const uint64_t before = g_launches;
    unsigned long long ctr[3];
    VFB_CUDA(cudaMemcpy(ctr, c->tab.counters, sizeof ctr, cudaMemcpyDeviceToHost));
    const uint64_t rows = ctr[0];
    c->x_table_rows = rows;
    c->m_self = self;
    if ((rc = c->m_part_rows.ensure((size_t)n_parts * 16))) return rc;
    VFB_CUDA(cudaMemsetAsync(c->m_part_rows.p, 0, (size_t)n_parts * 16, c->st_compute));
    if (rows && (rc = launch_partition_count(c->tab, rows, n_parts, self, c->m_part_rows.as<unsigned long long>(),
                                             c->m_part_rows.as<unsigned long long>() + n_parts, c->st_compute))) return rc;
    if (table_rows) *table_rows = rows;
    bump_launches(c, before);
    return VFB_OK;
}

// Pass 2 (asynchronous): one chunk per part (not for `self`) at d_buf + chunk_offsets[p]; part sizes as counted.
int vfb_internal_partition_fill(vfb_ctx *c, uint32_t n_parts, uint32_t self, bool release, uint8_t *d_buf, const uint64_t *chunk_offsets)
{
    VFB_CUDA(cudaSetDevice(c->device));
    const uint64_t before = g_launches;
    int rc;
    if ((rc = c->m_cursors.ensure((size_t)n_parts * 16))) return rc;
    if ((rc = c->m_chunk_off.ensure((size_t)n_parts * 8))) return rc;
    VFB_CUDA(cudaMemsetAsync(c->m_cursors.p, 0, (size_t)n_parts * 16, c->st_compute));
    // (pageable source: staged by the driver before the call returns)
    VFB_CUDA(cudaMemcpyAsync(c->m_chunk_off.p, chunk_offsets, (size_t)n_parts * 8, cudaMemcpyHostToDevice, c->st_compute));
    if ((rc = launch_partition_fill(c->tab, c->x_table_rows, n_parts, self, release, d_buf,
                                    c->m_chunk_off.as<uint64_t>(), c->m_part_rows.as<uint64_t>(),
                                    c->m_part_rows.as<uint64_t>() + n_parts, c->m_cursors.as<unsigned long long>(), c->st_compute)))
        return rc;
    bump_launches(c, before);
    return VFB_OK;
}

static int partition_fetch(vfb_ctx *c, uint32_t n_parts)
{
    c->h_part_rows.assign(n_parts, 0);
    c->h_part_keys.assign(n_parts, 0);
    std::vector<uint64_t> tmp((size_t)n_parts * 2);
    VFB_CUDA(cudaMemcpyAsync(tmp.data(), c->m_part_rows.p, (size_t)n_parts * 16, cudaMemcpyDeviceToHost, c->st_compute));
    VFB_CUDA(cudaStreamSynchronize(c->st_compute));
    c->stats.d2h_bytes += (uint64_t)n_parts * 16;
    for (uint32_t p = 0; p < n_parts; ++p) { c->h_part_rows[p] = tmp[p]; c->h_part_keys[p] = tmp[n_parts + p]; }
    return VFB_OK;
}

int vfb_internal_merge_export(vfb_ctx *c, uint32_t n_parts, uint32_t self, bool release, uint64_t *chunk_bytes,
                              uint64_t *chunk_offsets, uint64_t *part_rows, uint64_t *part_keys)
{
    int rc;
    if ((rc = vfb_internal_partition_count(c, n_parts, self, nullptr))) return rc;
    if ((rc = partition_fetch(c, n_parts))) return rc;
    uint64_t total = 0;
    for (uint32_t p = 0; p < n_parts; ++p) {
        const uint64_t r = c->h_part_rows[p], k = c->h_part_keys[p];
        chunk_bytes[p] = (p == self || r == 0) ? 0 : chunk_bytes_for(r, k);
        chunk_offsets[p] = total;
        total += chunk_bytes[p];
        if (part_rows) part_rows[p] = p == self ? 0 : r;
        if (part_keys) part_keys[p] = p == self ? 0 : k;
    }
    if ((rc = c->m_send.ensure(total ? total : 16))) return rc;
    if (total) {
        if ((rc = vfb_internal_partition_fill(c, n_parts, self, release, c->m_send.as<uint8_t>(), chunk_offsets))) return rc;
    }
    VFB_CUDA(cudaEventRecord(c->m_filled, c->st_compute));
    return VFB_OK;
}

int vfb_internal_absorb_known(vfb_ctx *c, const uint8_t *d_chunk, uint64_t rows, uint64_t key_bytes)
{
    if (rows == 0) return VFB_OK;
    if (rows > 0x7FFFFFFFull) { set_error("chunk too large"); return VFB_ERR_ARG; }
    VFB_CUDA(cudaSetDevice(c->device));
    const uint64_t before = g_launches;
    int rc;
    if ((rc = lanes_join(c))) return rc;
    if ((rc = table_reserve(c, rows, key_bytes, false))) return rc;
    if ((rc = c->lanes[0].d_owner.ensure(rows * 4))) return rc;
    const uint64_t n = rows;
    const uint8_t *base = d_chunk + sizeof(ChunkHeader);
    InsertJob ij;
    ij.khash = reinterpret_cast<const uint64_t *>(base);
    ij.kcount = reinterpret_cast<const unsigned long long *>(base + vfb_align16(n * 8));
    ij.koff = reinterpret_cast<const uint64_t *>(base + vfb_align16(n * 8) * 2);
    ij.klen = reinterpret_cast<const uint32_t *>(base + vfb_align16(n * 8) * 3);
    ij.keys = base + vfb_align16(n * 8) * 3 + vfb_align16(n * 4);
    ij.key_stride = 0;
    ij.n_keys = (uint32_t)n;
    ij.owner_slot = c->lanes[0].d_owner.as<uint32_t>();
    if ((rc = launch_insert(c->tab, ij, c->st_compute))) return rc;
    if ((rc = snaps_push(c, rows, key_bytes, c->st_compute))) return rc;
    bump_launches(c, before);
    return VFB_OK;
}

extern "C" {

int vfb_table_partition_sizes(vfb_ctx *c, uint32_t n_parts, uint64_t *chunk_bytes)
{
    if (!c || !chunk_bytes || n_parts == 0 || n_parts > 1024) { set_error("bad argument"); return VFB_ERR_ARG; }
    int rc;
    if ((rc = vfb_internal_partition_count(c, n_parts, 0xFFFFFFFFu, nullptr))) return rc;
    if ((rc = partition_fetch(c, n_parts))) return rc;
    for (uint32_t p = 0; p < n_parts; ++p) chunk_bytes[p] = chunk_bytes_for(c->h_part_rows[p], c->h_part_keys[p]);
    return VFB_OK;
}

int vfb_table_partition_fill(vfb_ctx *c, uint32_t n_parts, uint8_t *d_buf, const uint64_t *chunk_offsets)
{
    if (!c || !d_buf || !chunk_offsets || n_parts == 0 || c->h_part_rows.size() != n_parts || c->m_self != 0xFFFFFFFFu) {
        set_error("call vfb_table_partition_sizes with the same n_parts first");
        return VFB_ERR_ARG;
    }
    int rc = vfb_internal_partition_fill(c, n_parts, 0xFFFFFFFFu, false, d_buf, chunk_offsets);
    if (rc) return rc;
    VFB_CUDA(cudaStreamSynchronize(c->st_compute));
    return VFB_OK;
}

uint64_t vfb_hash_key(const uint8_t *key, uint32_t len) { return vfb_hash_bytes(key, len); }
uint32_t vfb_key_owner(uint64_t hash, uint32_t n_parts) { return n_parts ? vfb_hash_owner(hash, n_parts) : 0; }

int vfb_chunk_rows(const uint8_t *h_chunk, uint64_t chunk_bytes, uint64_t *rows)
{
    if (!h_chunk || !rows || chunk_bytes < sizeof(ChunkHeader)) { set_error("bad chunk"); return VFB_ERR_ARG; }
    ChunkHeader h;
    memcpy(&h, h_chunk, sizeof h);
    if (h.magic != VFB_CHUNK_MAGIC || chunk_bytes_for(h.rows, h.key_bytes) > chunk_bytes) { set_error("bad chunk header"); return VFB_ERR_FORMAT; }
    *rows = h.rows;
    return VFB_OK;
}

int vfb_table_absorb(vfb_ctx *c, const uint8_t *d_chunk, uint64_t chunk_bytes)
{
    if (!c || !d_chunk || chunk_bytes < sizeof(ChunkHeader)) { set_error("bad argument"); return VFB_ERR_ARG; }
    VFB_CUDA(cudaSetDevice(c->device));
    ChunkHeader h;
    VFB_CUDA(cudaMemcpyAsync(&h, d_chunk, sizeof h, cudaMemcpyDeviceToHost, c->st_compute));
    VFB_CUDA(cudaStreamSynchronize(c->st_compute));
    if (h.magic != VFB_CHUNK_MAGIC || chunk_bytes_for(h.rows, h.key_bytes) > chunk_bytes) { set_error("bad chunk header"); return VFB_ERR_FORMAT; }
    return vfb_internal_absorb_known(c, d_chunk, h.rows, h.key_bytes);
}

// ------------------------------------------------------------------------------------ synth + misc
int vfb_synth_adapters(const vfb_synth_cfg *cfg, uint8_t *prefix, uint8_t *suffix)
{
    if (!cfg || !prefix || !suffix) { set_error("null argument"); return VFB_ERR_ARG; }
    vfs_adapter(cfg->seed, 0, cfg->adapter_len, prefix);
    vfs_adapter(cfg->seed, 1, cfg->adapter_len, suffix);
    return VFB_OK;
}

int vfb_synth_host(const vfb_synth_cfg *cfg, uint64_t first, uint64_t n, uint8_t *text, vfb_span *spans)
{
    if (!cfg || (n && (!text || !spans))) { set_error("null argument"); return VFB_ERR_ARG; }
    if (cfg->adapter_len > 61 || cfg->adapter_len == 0 || cfg->read_len == 0 || cfg->read_len > 700 ||
        n * (uint64_t)cfg->read_len > 0xFFFFFFFFull) {
        set_error("synth: adapter_len must be 1..61, read_len 1..700, at most 4 GiB per call");
        return VFB_ERR_ARG;
    }
    uint8_t pre[64], suf[64];
    vfs_adapter(cfg->seed, 0, cfg->adapter_len, pre);
    vfs_adapter(cfg->seed, 1, cfg->adapter_len, suf);
    for (uint64_t i = 0; i < n; ++i) {
        vfs_read(cfg, first + i, pre, suf, text + i * cfg->read_len);
        spans[i] = vfb_span{(uint32_t)(i * cfg->read_len), cfg->read_len};
    }
    return VFB_OK;
}

int vfb_synth_device(const vfb_synth_cfg *cfg, uint64_t first, uint64_t n, uint8_t *d_text, vfb_span *d_spans, int device)
{
    if (!cfg || (n && (!d_text || !d_spans))) { set_error("null argument"); return VFB_ERR_ARG; }
    if (device >= 0) VFB_CUDA(cudaSetDevice(device));
    int rc = launch_synth(*cfg, first, n, d_text, d_spans, 0);
    if (rc) return rc;
    VFB_CUDA(cudaStreamSynchronize(0));
    return VFB_OK;
}

int vfb_debug_gpu_inflate(const uint8_t *z, uint64_t z_bytes, const uint32_t *members, uint32_t n_members,
                          uint8_t *out, uint64_t out_bytes, int device, uint32_t *first_bad, double *kernel_ms)
{
    if (!z || !members || !out || !first_bad) { set_error("null argument"); return VFB_ERR_ARG; }
    if (device >= 0) VFB_CUDA(cudaSetDevice(device));
    uint8_t *d_z = nullptr, *d_out = nullptr;
    vfb_member *d_m = nullptr;
    uint32_t *d_bad = nullptr;
    VFB_CUDA(cudaMalloc(&d_z, z_bytes + 16));
    VFB_CUDA(cudaMalloc(&d_out, out_bytes + 16));
    VFB_CUDA(cudaMalloc(&d_m, (size_t)n_members * sizeof(vfb_member) + 16));
    VFB_CUDA(cudaMalloc(&d_bad, 4));
    VFB_CUDA(cudaMemcpy(d_z, z, z_bytes, cudaMemcpyHostToDevice));
    VFB_CUDA(cudaMemcpy(d_m, members, (size_t)n_members * sizeof(vfb_member), cudaMemcpyHostToDevice));
    VFB_CUDA(cudaMemset(d_bad, 0xFF, 4));
    VFB_CUDA(cudaMemset(d_out, 0, out_bytes));
    cudaEvent_t e0, e1;
    VFB_CUDA(cudaEventCreate(&e0));
    VFB_CUDA(cudaEventCreate(&e1));
    VFB_CUDA(cudaEventRecord(e0, 0));
    int rc = launch_inflate(d_z, d_m, n_members, d_out, d_bad, 0);
    VFB_CUDA(cudaEventRecord(e1, 0));
    VFB_CUDA(cudaDeviceSynchronize());
    float ms = 0;
    VFB_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    if (kernel_ms) *kernel_ms = ms;
    VFB_CUDA(cudaMemcpy(out, d_out, out_bytes, cudaMemcpyDeviceToHost));
    VFB_CUDA(cudaMemcpy(first_bad, d_bad, 4, cudaMemcpyDeviceToHost));
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    cudaFree(d_z); cudaFree(d_out); cudaFree(d_m); cudaFree(d_bad);
    return rc;
}

int vfb_measure_int_peak(int device, double *alu_gops, double *dual_gops)
{
    return measure_int_peak(device, alu_gops, dual_gops);
}

int vfb_debug_window_plan(int32_t match_score, int32_t mismatch_score, int32_t gap_open_penalty, int32_t gap_extend_penalty,
                          uint32_t adapter_len, double accept_alignment, int32_t *accept_bound_out, int32_t *max_edits_out)
{
    if (!accept_bound_out || !max_edits_out || adapter_len == 0) { set_error("bad argument"); return VFB_ERR_ARG; }
    const int t = accept_bound(accept_alignment, match_score, adapter_len);
    const DpScoring sc{match_score, mismatch_score, gap_open_penalty, gap_extend_penalty};
    *accept_bound_out = t;
    *max_edits_out = dpw_max_edits(sc, adapter_len, t);
    return VFB_OK;
}

int vfb_debug_dp_layout(int32_t match_score, int32_t mismatch_score, int32_t gap_open_penalty, int32_t gap_extend_penalty,
                        uint32_t adapter_len, double accept_alignment, int32_t dp_mode, vfb_dp_layout_info *out)
{
    if (!out || adapter_len == 0) { set_error("bad argument"); return VFB_ERR_ARG; }
    memset(out, 0, sizeof *out);
    const DpScoring sc{match_score, mismatch_score, gap_open_penalty, gap_extend_penalty};
    out->accept_bound = accept_bound(accept_alignment, match_score, adapter_len);
    DpLayout l;
    uint32_t lcap = 0;
    int K = -1;
    out->packed = plan_packed_dp(sc, adapter_len, out->accept_bound, dp_mode != 1, &l, &lcap, &K) ? 1 : 0;
    out->max_edits = out->packed ? K : -1;
    if (!out->packed) return VFB_OK;
    out->S0 = l.S0; out->LB = l.LB; out->XB = l.XB;
    out->c_eopen = l.c_eopen; out->c_eext = l.c_eext; out->c_fopen = l.c_fopen; out->c_fext = l.c_fext;
    out->hmask = l.hmask; out->lowmask = l.lowmask; out->lenmask = l.lenmask;
    out->neg_e = l.neg_e; out->neg_f = l.neg_f;
    out->w_match = l.w_match; out->w_mismatch = l.w_mismatch; out->w_wild = l.w_wild;
    out->lcap = lcap;
    return VFB_OK;
}

int vfb_host_alloc(void **p, uint64_t bytes)
{
    if (!p) { set_error("null argument"); return VFB_ERR_ARG; }
    VFB_CUDA(cudaMallocHost(p, bytes ? bytes : 1));
    return VFB_OK;
}

int vfb_host_free(void *p)
{
    if (p) VFB_CUDA(cudaFreeHost(p));
    return VFB_OK;
}

int vfb_pinned_pool_trim(void)
{
    pinned_pool_trim();
    return VFB_OK;
}

int vfb_device_pool_trim(void)
{
    device_pool_trim();
    return VFB_OK;
}

}  // extern "C"
