// Ingest: gzip (multi-member) FASTQ file -> inflate -> pinned chunks -> async H2D -> GPU parse
// -> the hot loop.
//
// Replaces `File::open(fq_path).map(MultiGzDecoder::new)` + `seq_io::fastq::Reader` +
// `parallel_fastq` of /root/reference/src/lib.rs:233-234, :271-308 (flate2 1.1.1 /
// seq_io 0.3.4).  Grammar (SURVEY Q11): gzip only; strict 4-line records — '@' header, one
// sequence line, '+' line, quality of the same length; "\r\n" trimmed; a missing final
// newline and trailing blank lines are tolerated.
//
// Pipeline: a producer thread fills one of three pinned chunk buffers with inflated text,
// counts newlines as it goes and cuts the chunk at the last 4-line boundary (the remainder is
// carried into the next chunk).  The calling thread queues each chunk on the GPU: H2D copy on
// the copy stream, record framing / validation / span extraction on the device
// (kernels_parse.cu), then K1..K4.  The host never looks at a record.
//
// Inflate: a plain gzip stream is serial (one zlib stream, ~0.3 GB/s).  Block-gzip files
// (BGZF: every member carries its compressed size in a "BC" extra field, as written by
// bgzip / htslib and most sequencer pipelines) are inflated member-parallel on `n_threads`
// host threads — the reference's n_threads knob (src/lib.rs:228) keeps its meaning of
// "worker threads".
#include <unistd.h>
#include <zlib.h>

#include <algorithm>
#include <atomic>
#include <cerrno>
#include <chrono>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "ctx.cuh"
#include "gunzip_gpu.h"
#include "pgunzip.h"

using namespace vfb;

namespace {

size_t count_nl(const uint8_t *p, size_t n)
{
    // eight bytes at a time: x = word ^ 0x0A.. has a zero byte where the text has '\n'; ((x & 0x7F..) + 0x7F..) | x
    // sets the high bit of every NON-zero byte without carries between bytes, so the cleared high bits count
    size_t c = 0, i = 0;
    const uint64_t k = 0x0A0A0A0A0A0A0A0Aull, lo7 = 0x7F7F7F7F7F7F7F7Full;
    for (; i + 8 <= n; i += 8) {
        uint64_t w;
        memcpy(&w, p + i, 8);
        const uint64_t x = w ^ k;
        // per byte: high bit set iff the byte of x is non-zero (no cross-byte carries)
        const uint64_t nz = ((x & lo7) + lo7) | x;
        c += (size_t)__builtin_popcountll(~nz & ~lo7);
    }
    for (; i < n; ++i) c += p[i] == '\n';
    return c;
}

// Serial multi-member gzip stream (flate2 MultiGzDecoder semantics).
struct Inflater {
    FILE *f = nullptr;
    z_stream z;
    bool z_open = false;
    bool eof = false;          // no more compressed input
    bool member_done = true;   // between members
    std::vector<uint8_t> in;
    Inflater() : in(1 << 20) { memset(&z, 0, sizeof z); }
    ~Inflater()
    {
        if (z_open) inflateEnd(&z);
    }
    // Fill out[0..cap) with inflated bytes; returns bytes produced (0 at end) or -1 on error.
    long long read(uint8_t *out, size_t cap, std::string *err)
    {
        size_t produced = 0;
        while (produced < cap) {
            if (z.avail_in == 0 && !eof) {
                size_t got = fread(in.data(), 1, in.size(), f);
                if (got == 0) eof = true;
                z.next_in = in.data();
                z.avail_in = (uInt)got;
            }
            if (member_done) {
                if (z.avail_in == 0 && eof) break;     // clean end between members
                if (z_open) inflateEnd(&z);
                Bytef *ni = z.next_in;
                uInt ai = z.avail_in;
                memset(&z, 0, sizeof z);
                z.next_in = ni;
                z.avail_in = ai;
                if (inflateInit2(&z, 15 + 16) != Z_OK) { *err = "zlib init failed"; return -1; }
                z_open = true;
                member_done = false;
            }
            if (z.avail_in == 0 && eof) { *err = "truncated gzip stream"; return -1; }
            z.next_out = out + produced;
            size_t room = cap - produced;
            z.avail_out = (uInt)(room > (1u << 30) ? (1u << 30) : room);
            const uInt out0 = z.avail_out;
            int rc = inflate(&z, Z_NO_FLUSH);
            produced += out0 - z.avail_out;
            if (rc == Z_STREAM_END) { member_done = true; continue; }
            if (rc != Z_OK && rc != Z_BUF_ERROR) { *err = std::string("invalid gzip data: ") + (z.msg ? z.msg : "?"); return -1; }
            if (rc == Z_BUF_ERROR && z.avail_in == 0 && eof) { *err = "truncated gzip stream"; return -1; }
        }
        return (long long)produced;
    }
};

// One BGZF member read from the file but not yet inflated.
struct Member {
    size_t in_off = 0, in_len = 0;   // whole member inside the compressed staging buffer
    size_t out_off = 0;
    uint32_t isize = 0;
    size_t lines = 0;
};

// pread of a large range split over `threads` threads (page-cache copies into pinned memory run
// at a few GB/s per core).  Returns the bytes read from `off` on (short only at end of file), -1 on error.
ssize_t pread_parallel(int fd, uint8_t *buf, size_t want, off_t off, int threads)
{
    const size_t min_part = (size_t)4 << 20;
    int parts = threads < 1 ? 1 : threads;
    if ((size_t)parts > want / min_part) parts = (int)(want / min_part);
    if (parts <= 1) {
        size_t done = 0;
        while (done < want) {
            const ssize_t got = pread(fd, buf + done, want - done, off + (off_t)done);
            if (got < 0) { if (errno == EINTR) continue; return -1; }
            if (got == 0) break;
            done += (size_t)got;
        }
        return (ssize_t)done;
    }
    const size_t part = ((want / (size_t)parts) + 4095) & ~(size_t)4095;
    std::vector<ssize_t> got((size_t)parts, 0);
    std::vector<std::thread> pool;
    auto run = [&](int i) {
        const size_t lo = (size_t)i * part, hi = std::min(want, lo + part);
        got[(size_t)i] = lo < hi ? pread_parallel(fd, buf + lo, hi - lo, off + (off_t)lo, 1) : 0;
    };
    for (int i = 1; i < parts; ++i) pool.emplace_back(run, i);
    run(0);
    for (auto &t : pool) t.join();
    size_t total = 0;
    for (int i = 0; i < parts; ++i) {
        if (got[(size_t)i] < 0) return -1;
        const size_t lo = (size_t)i * part, hi = std::min(want, lo + part);
        total += (size_t)got[(size_t)i];
        if ((size_t)got[(size_t)i] < hi - lo) break;       // end of file inside this part
    }
    return (ssize_t)total;
}

// Reads the next gzip member header at the current file position.  Returns 1 and the total
// member size if it is a BGZF member, 0 if it is some other gzip member (position restored),
// -1 at a clean end of file.
int peek_bgzf(FILE *f, size_t *member_size)
{
    const long pos = ftell(f);
    uint8_t h[12];
    const size_t got = fread(h, 1, 12, f);
    if (got == 0) return -1;
    int is_bgzf = 0;
    if (got == 12 && h[0] == 0x1f && h[1] == 0x8b && h[2] == 8 && (h[3] & 4)) {
        const uint32_t xlen = h[10] | (h[11] << 8);
        std::vector<uint8_t> x(xlen);
        if (xlen >= 6 && fread(x.data(), 1, xlen, f) == xlen) {
            for (uint32_t p = 0; p + 4 <= xlen;) {
                const uint32_t slen = x[p + 2] | (x[p + 3] << 8);
                if (x[p] == 'B' && x[p + 1] == 'C' && slen == 2 && p + 6 <= xlen) {
                    *member_size = (size_t)(x[p + 4] | (x[p + 5] << 8)) + 1;
                    is_bgzf = 1;
                    break;
                }
                p += 4 + slen;
            }
        }
    }
    fseek(f, pos, SEEK_SET);
    return is_bgzf;
}

// Fills chunk buffers with inflated text and cuts them at record boundaries.
struct ChunkProducer {
    FILE *f = nullptr;
    ParallelGunzip pgz;         // plain gzip streams on `threads` > 1 host threads
    GpuGunzip ggz;              // ... or on the device (gpu_device >= 0): block-start search, marker decode, resolve
    int gpu_device = -1;
    int pgz_state = 0;          // 0 = not decided, 1 = host threads, 2 = device, -1 = zlib stream
    uint64_t file_size = 0;
    std::atomic<uint64_t> consumed{0};   // compressed bytes read so far (progress only)
    Inflater serial;
    bool bgzf = false;          // still reading BGZF members
    bool plain = false;         // uncompressed FASTQ text (vfb_run_file_ex with VFB_INPUT_ALLOW_TEXT only)
    int threads = 1;
    std::vector<uint8_t> carry;
    std::vector<uint8_t> dev_tail;
    std::vector<uint8_t> zbuf;  // compressed members of the current chunk
    bool at_end = false;
    std::string err;

    ~ChunkProducer()
    {
        if (f) fclose(f);
    }

    bool open(const char *path, int n_threads, std::string *e, bool allow_text = false)
    {
        f = fopen(path, "rb");
        if (!f) { *e = std::string("cannot open ") + path + ": " + strerror(errno); return false; }
        serial.f = f;
        fseek(f, 0, SEEK_END);
        file_size = (uint64_t)ftell(f);
        fseek(f, 0, SEEK_SET);
        threads = n_threads < 1 ? 1 : n_threads;
        size_t ms = 0;
        bgzf = peek_bgzf(f, &ms) == 1;
        if (allow_text && !bgzf) {
            uint8_t m[2] = {0, 0};
            const size_t got = fread(m, 1, 2, f);
            fseek(f, 0, SEEK_SET);
            plain = !(got == 2 && m[0] == 0x1f && m[1] == 0x8b);
        }
        return true;
    }

    // Member-parallel fill of buf[used..cap).  Returns false on error.
    bool fill_bgzf(uint8_t *buf, size_t cap, size_t &used, size_t &lines)
    {
        std::vector<Member> ms;
        zbuf.clear();
        while (used < cap) {
            size_t msize = 0;
            const int k = peek_bgzf(f, &msize);
            if (k < 0) { at_end = true; break; }
            if (k == 0) { bgzf = false; break; }          // the rest is plain gzip: serial from here
            if (msize < 26) { err = "invalid BGZF member"; return false; }
            const size_t zo = zbuf.size();
            zbuf.resize(zo + msize);
            const long pos = ftell(f);
            if (fread(zbuf.data() + zo, 1, msize, f) != msize) { err = "truncated gzip stream"; return false; }
            const uint8_t *t = zbuf.data() + zo + msize - 4;
            const uint32_t isize = t[0] | (t[1] << 8) | (t[2] << 16) | ((uint32_t)t[3] << 24);
            if (isize > cap - used) {
                fseek(f, pos, SEEK_SET);                   // does not fit: first member of the next chunk
                zbuf.resize(zo);
                if (ms.empty()) { err = "ingest chunk too small for a gzip member plus a carried record"; return false; }
                break;
            }
            Member m;
            m.in_off = zo; m.in_len = msize; m.out_off = used; m.isize = isize;
            ms.push_back(m);
            used += isize;
        }
        if (ms.empty()) return true;
        std::atomic<size_t> next{0};
        std::atomic<bool> bad{false};
        auto work = [&]() {
            z_stream z;
            for (;;) {
                const size_t i = next.fetch_add(1);
                if (i >= ms.size() || bad.load()) return;
                Member &m = ms[i];
                memset(&z, 0, sizeof z);
                if (inflateInit2(&z, 15 + 16) != Z_OK) { bad = true; return; }
                z.next_in = zbuf.data() + m.in_off;
                z.avail_in = (uInt)m.in_len;
                z.next_out = buf + m.out_off;
                z.avail_out = m.isize;
                const int rc = inflate(&z, Z_FINISH);
                const bool ok = rc == Z_STREAM_END && z.avail_out == 0 && z.avail_in == 0;
                inflateEnd(&z);
                if (!ok) { bad = true; return; }
                m.lines = count_nl(buf + m.out_off, m.isize);
            }
        };
        const int nt = (int)std::min<size_t>((size_t)threads, ms.size());
        std::vector<std::thread> pool;
        for (int t = 1; t < nt; ++t) pool.emplace_back(work);
        work();
        for (auto &t : pool) t.join();
        if (bad.load()) { err = "invalid gzip data in a BGZF member"; return false; }
        for (const Member &m : ms) lines += m.lines;
        return true;
    }

    // Produce the next chunk into buf (capacity cap, plus 64 spare bytes).  On success sets
    // cut (bytes to submit) and keep_lines (complete lines in [0,cut)); *last when the input is
    // exhausted.  Returns VFB_OK or an error code with `err` set.
    // dev_out (optional): the chunk may be [carry in buf | text that stays on the device] — see Chunk::dev.
    int next(uint8_t *buf, size_t cap, size_t *cut_out, size_t *lines_out, bool *last, GpuGunzip::DeviceRange *dev_out = nullptr,
             size_t *dev_len_out = nullptr)
    {
        if (carry.size() >= cap) { err = "a FASTQ record is larger than the ingest chunk"; return VFB_ERR_FORMAT; }
        size_t used = carry.size();
        if (used) memcpy(buf, carry.data(), used);
        size_t lines = count_nl(buf, used);
        if (dev_out) { *dev_out = GpuGunzip::DeviceRange(); *dev_len_out = 0; }
        if (dev_out && pgz_state == 2 && !at_end && cap - used > ((size_t)8 << 20)) {
            // decoded on the device: hand the text on without a round trip through host memory.  Only the range's tail
            // comes over, to find the last record boundary; what follows it is the next chunk's carry.
            const size_t tail_cap = (size_t)256 << 10;
            GpuGunzip::DeviceRange r;
            if (ggz.peek_device(cap - used, tail_cap, &r)) {
                const size_t total = lines + r.newlines, rem = total % 4, keep = total - rem;
                const size_t tn = std::min(r.len, tail_cap);
                dev_tail.resize(tn);
                if (!ggz.range_tail(r, dev_tail.data(), tn, &err)) return VFB_ERR_CUDA;
                // just behind newline number `keep`: walk back over the last rem + 1 newlines
                size_t end = tn;
                bool found = keep != 0;
                for (size_t sft = 0; sft <= rem && found; ++sft) {
                    const void *q = end ? memrchr(dev_tail.data(), '\n', end) : nullptr;
                    if (!q) found = false;
                    else end = (size_t)((const uint8_t *)q - dev_tail.data());
                }
                if (found) {
                    const size_t cut_in_tail = end + 1;
                    ggz.commit_device(r);
                    *dev_out = r;
                    *dev_len_out = r.len - (tn - cut_in_tail);
                    carry.assign(dev_tail.data() + cut_in_tail, dev_tail.data() + tn);
                    *cut_out = used;
                    *lines_out = keep;
                    *last = false;
                    return VFB_OK;
                }
                // (a record longer than the tail: this stretch goes through host memory)
            }
        }
        while (used < cap && !at_end) {
            if (bgzf) {
                if (!fill_bgzf(buf, cap, used, lines)) return VFB_ERR_FORMAT;
                if (bgzf && !at_end) break;                   // as full as whole members allow
            } else {
                if (!plain && pgz_state == 0) {
                    // a plain gzip stream: on the device when there is one (VFB_GPU_GUNZIP=0: never; files under
                    // 4 MB are not worth the set-up), else in parallel on the host threads, else one zlib stream
                    const char *g = getenv("VFB_GPU_GUNZIP");
                    const bool want_gpu = gpu_device >= 0 && !(g && g[0] == '0') && (file_size >= ((uint64_t)4 << 20) || (g && g[0] == '2'));
                    std::string ge;
                    if (want_gpu && ggz.init(f, gpu_device, &ge)) pgz_state = 2;
                    else {
                        const char *e = getenv("VFB_PGUNZIP");
                        pgz_state = threads > 1 && !(e && e[0] == '0') ? 1 : -1;
                        if (pgz_state == 1) pgz.init(f, threads);
                    }
                }
                if (!plain && pgz_state == 2) {
                    const size_t want = cap - used;
                    size_t nl = 0;
                    // (with the hand-off on the device, host memory only takes what is left of the current segment — its
                    // tail — so that the next segment can be handed on from its first, piece-aligned byte)
                    const long long got = ggz.read_counting(buf + used, want, &nl, &err, dev_out != nullptr);
                    if (got < 0) return VFB_ERR_FORMAT;
                    lines += nl;
                    used += (size_t)got;
                    if ((size_t)got < want && dev_out && !ggz.member_ended()) break;      // a segment's tail: cut the chunk here
                    if ((size_t)got < want) {
                        // the member has ended (trailer checked): further members go through the zlib stream
                        long off = 0;
                        if (ggz.handover(&off) && (uint64_t)off < file_size) { fseek(f, off, SEEK_SET); pgz_state = -1; }
                        else at_end = true;
                    }
                    continue;
                }
                if (!plain && pgz_state == 1) {
                    // already decoded in the background: take all the chunk has room for, copied and counted in parallel
                    const size_t want = cap - used;
                    size_t nl = 0;
                    const long long got = pgz.read_counting(buf + used, want, &nl, &err);
                    if (got < 0) return VFB_ERR_FORMAT;
                    if ((size_t)got < want) at_end = true;
                    lines += nl;
                    used += (size_t)got;
                    continue;
                }
                const size_t want = cap - used < ((size_t)4 << 20) ? cap - used : ((size_t)4 << 20);
                const long long got = plain ? (long long)fread(buf + used, 1, want, f) : serial.read(buf + used, want, &err);
                if (got < 0) return VFB_ERR_FORMAT;
                if ((size_t)got < want) at_end = true;
                lines += count_nl(buf + used, (size_t)got);
                used += (size_t)got;
            }
        }
        size_t cut = used, keep = lines;
        if (at_end) {
            // trailing blank lines are tolerated, and so is a missing final newline
            while (used && (buf[used - 1] == '\n' || buf[used - 1] == '\r')) --used;
            if (used) buf[used++] = '\n';
            lines = count_nl(buf, used);
            if (lines % 4) { err = "truncated FASTQ record at the end of the input"; return VFB_ERR_FORMAT; }
            cut = used;
            keep = lines;
            carry.clear();
        } else {
            const size_t rem = lines % 4;
            keep = lines - rem;
            // cut just after newline number `keep`: walk back over the last `rem` newlines
            size_t end = used;
            for (size_t s = 0; s <= rem && keep; ++s) {
                const void *q = end ? memrchr(buf, '\n', end) : nullptr;
                end = q ? (size_t)((const uint8_t *)q - buf) : 0;
            }
            cut = keep ? end + 1 : 0;
            carry.assign(buf + cut, buf + used);
        }
        *cut_out = cut;
        *lines_out = keep;
        *last = at_end;
        consumed = (uint64_t)ftell(f);
        return VFB_OK;
    }
};

size_t pick_chunk(FILE *f)
{
    fseek(f, 0, SEEK_END);
    const long fsz = ftell(f);
    fseek(f, 0, SEEK_SET);
    size_t cap = (size_t)128 << 20;
    if (const char *e = getenv("VFB_INGEST_CHUNK")) cap = (size_t)strtoull(e, nullptr, 10);
    else if (fsz >= 0 && (size_t)fsz * 12 + 65536 < cap) cap = (size_t)fsz * 12 + 65536;
    if (cap < 256) cap = 256;
    return cap;
}

struct Chunk {
    uint8_t *buf = nullptr;
    size_t buf_cap = 0;
    size_t cut = 0;        // bytes to submit (ends at a record boundary)
    size_t lines = 0;      // complete lines in [0, cut)
    cudaEvent_t copied = nullptr;
    // text that never left the device follows buf[0..cut) (plain gzip decoded on the device): lines counts both parts
    GpuGunzip::DeviceRange dev;
    size_t dev_len = 0;    // bytes of dev.d_ptr to submit (its rest is the next chunk's carry)
};

struct Pipe {
    std::mutex mu;
    std::condition_variable cv;
    std::deque<int> free_q, ready_q;
    bool done = false, failed = false, abort = false;
    std::string err;
    int err_code = VFB_OK;
};

// ---- GPU inflate phase: block-gzip members are shipped compressed and inflated on the device(s).
//
//   reader threads   pread fixed-size raw blocks of the file into a ring of pinned buffers, in parallel and
//                    without looking at the bytes (a block boundary falls anywhere);
//   indexer thread   walks the member headers across the raw blocks in file order and cuts segments of about
//                    `text_target` bytes of text: a list of members plus the pieces of raw blocks that hold them;
//   one worker per   takes every n-th segment: phase 1 (vfb_internal_bgzf_begin: H2D of the pieces + inflate) for up
//   device           to two segments ahead, then phase 2 (vfb_internal_bgzf_finish) in segment order;
//   the chain        a record may straddle two segments, so phase 2 of segment s needs the text after the last
//                    complete record of segment s-1 (and the number of records before it, for error messages):
//                    each worker publishes that when its phase 2 has framed the records, about half a
//                    millisecond of small kernels per segment — the only serial part of the pipeline.
// The calling thread waits, reports progress and collects errors.
static inline double now_ms()
{
    return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

struct RawRing {
    struct Block {
        uint8_t *p = nullptr;
        size_t cap = 0, len = 0;
        uint64_t idx = UINT64_MAX;
        int state = 0;                 // 0 free, 1 being read, 2 ready
        int refs = 0;                  // the indexer while it walks the block + one per segment with a piece in it
    };
    int fd = -1;
    uint64_t base = 0, end = 0;        // file range [base, end)
    size_t block = 0;
    uint64_t n_blocks = 0, next_idx = 0;
    std::vector<Block> ring;
    std::vector<std::thread> threads;
    std::mutex mu;
    std::condition_variable cv;
    bool abort = false;
    std::string err;
    double t_read_ms = 0, t_wait_ms = 0;          // summed over the reader threads (trace)

    bool start(int fd_, uint64_t base_, uint64_t end_, size_t block_, int n_ring, int n_threads)
    {
        fd = fd_; base = base_; end = end_; block = block_;
        n_blocks = (end - base + block - 1) / block;
        if ((uint64_t)n_ring > n_blocks) n_ring = (int)n_blocks;
        if (n_ring < 1) n_ring = 1;
        ring.resize((size_t)n_ring);
        for (auto &b : ring) {
            b.p = (uint8_t *)pinned_acquire(block, &b.cap);
            if (!b.p) return false;
        }
        if ((uint64_t)n_threads > n_blocks) n_threads = (int)n_blocks;
        for (int t = 0; t < n_threads; ++t) threads.emplace_back([this] { run(); });
        return true;
    }
    void run()
    {
        for (;;) {
            uint64_t idx;
            Block *b;
            {
                const double w0 = now_ms();
                std::unique_lock<std::mutex> lk(mu);
                cv.wait(lk, [&] { return abort || next_idx >= n_blocks || ring[next_idx % ring.size()].state == 0; });
                t_wait_ms += now_ms() - w0;
                if (abort || next_idx >= n_blocks) return;
                idx = next_idx++;
                b = &ring[idx % ring.size()];
                b->state = 1; b->idx = idx; b->refs = 0;
            }
            const uint64_t lo = base + idx * block;
            const size_t want = (size_t)std::min<uint64_t>(block, end - lo);
            size_t done = 0;
            bool bad = false;
            const double r0 = now_ms();
            while (done < want) {
                const ssize_t got = pread(fd, b->p + done, want - done, (off_t)(lo + done));
                if (got < 0) { if (errno == EINTR) continue; bad = true; break; }
                if (got == 0) break;                       // the file shrank: the indexer reports the truncation
                done += (size_t)got;
            }
            std::lock_guard<std::mutex> lk(mu);
            t_read_ms += now_ms() - r0;
            if (bad) { abort = true; err = std::string("read error: ") + strerror(errno); }
            b->len = done;
            b->state = 2;
            cv.notify_all();
        }
    }
    // Block idx, ready, with one more reference (nullptr after an abort).
    Block *acquire(uint64_t idx)
    {
        std::unique_lock<std::mutex> lk(mu);
        Block *b = &ring[idx % ring.size()];
        cv.wait(lk, [&] { return abort || (b->state == 2 && b->idx == idx); });
        if (abort) return nullptr;
        ++b->refs;
        return b;
    }
    void ref(uint64_t idx)
    {
        std::lock_guard<std::mutex> lk(mu);
        ++ring[idx % ring.size()].refs;
    }
    void unref(uint64_t idx)
    {
        std::lock_guard<std::mutex> lk(mu);
        Block &b = ring[idx % ring.size()];
        if (--b.refs == 0) { b.state = 0; cv.notify_all(); }
    }
    void stop()
    {
        {
            std::lock_guard<std::mutex> lk(mu);
            abort = true;
            cv.notify_all();
        }
        for (auto &t : threads) t.join();
        threads.clear();
        for (auto &b : ring) pinned_release(b.p, b.cap);
        ring.clear();
    }
};

struct Segment {
    uint64_t seq = 0;
    std::vector<vfb_zpiece> pieces;
    std::vector<uint64_t> blocks;      // raw blocks the pieces live in (one reference each)
    std::vector<vfb_member> members;
    uint64_t text_bytes = 0, z_bytes = 0;
    RawRing *ring = nullptr;
    int slot = -1;
    double t_pushed = 0, t_begin = 0, t_fin0 = 0;     // trace
};

void segment_release_blocks(void *arg)        // runs on a driver thread once the pieces are on the device
{
    Segment *g = static_cast<Segment *>(arg);
    for (uint64_t b : g->blocks) g->ring->unref(b);
}

struct GpuPhase {
    // where the threads spent their time (ms; VFB_INGEST_TRACE prints them)
    double ix_wait_block = 0, ix_wait_queue = 0, ix_total = 0;
    double sum_queue_ms = 0, sum_begin_to_fin_ms = 0, sum_fin_ms = 0;     // per segment: queued -> begun -> finish starts -> ends
    std::vector<double> w_wait_seg, w_wait_chain, w_begin, w_finish;
    std::mutex mu;
    std::condition_variable cv;
    bool abort = false, indexed = false;       // indexed: the indexer has queued its last segment
    int rc = VFB_OK;
    std::string err;
    uint64_t n_segments = 0;                   // valid once indexed
    std::vector<std::deque<Segment *>> queues; // per device
    // the chain: link s = text carried into segment s + records before it
    struct Link { bool ready = false; std::vector<uint8_t> carry; uint64_t records = 0; };
    std::deque<Link> links;                    // links[s - link_base]
    uint64_t link_base = 0;
    uint64_t records_done = 0, z_done = 0, segments_done = 0;
    uint64_t stop_off = 0;                     // file offset where the GPU phase ended (valid once indexed)
    bool hit_plain = false;                    // ... because a member that is not block gzip follows

    void fail(int code, const std::string &msg)
    {
        std::lock_guard<std::mutex> lk(mu);
        if (rc == VFB_OK) { rc = code; err = msg; }
        abort = true;
        cv.notify_all();
    }
    Link &link(uint64_t s)                     // mu held
    {
        while (links.size() <= s - link_base) links.emplace_back();
        return links[s - link_base];
    }
};

// Walks member headers over the raw blocks and deals segments to the device queues.
void index_members(RawRing &ring, GpuPhase &gp, size_t text_target, size_t mcap, size_t max_blocks, int n_dev, size_t queue_depth)
{
    uint64_t bi = 0;                           // current raw block
    size_t bo = 0;                             // offset inside it
    RawRing::Block *cur = ring.n_blocks ? ring.acquire(0) : nullptr;
    RawRing::Block *nxt = nullptr;             // block bi + 1 when a header / trailer straddles the boundary
    if (ring.n_blocks && !cur) { gp.fail(VFB_ERR_IO, ring.err.empty() ? "read aborted" : ring.err); return; }
    uint64_t seq = 0;
    Segment *g = nullptr;
    std::string err;
    bool plain = false, at_end = false;
    auto file_off = [&] { return ring.base + bi * ring.block + bo; };
    // bytes [bo + at, bo + at + n) of the stream that starts at block bi, copied out (they may straddle a block end)
    auto peek = [&](size_t at, size_t n, uint8_t *out) -> int {          // 1 ok, 0 end of file inside, -1 abort
        size_t pos = bo + at, got = 0;
        uint64_t b = bi;
        while (got < n) {
            RawRing::Block *blk;
            if (b == bi) blk = cur;
            else if (b == bi + 1) {
                if (!nxt) {
                    if (b >= ring.n_blocks) return 0;
                    const double w0 = now_ms();
                    nxt = ring.acquire(b);
                    gp.ix_wait_block += now_ms() - w0;
                    if (!nxt) return -1;
                }
                blk = nxt;
            } else return 0;                   // members are at most 64 KiB: never more than two blocks
            if (pos >= blk->len) {
                if (blk->len < ring.block) return 0;                     // short block = end of file
                pos -= blk->len; ++b;
                continue;
            }
            const size_t take = std::min(n - got, blk->len - pos);
            memcpy(out + got, blk->p + pos, take);
            got += take; pos += take;
        }
        return 1;
    };
    auto discard = [&](Segment *seg) {
        for (uint64_t b : seg->blocks) ring.unref(b);
        delete seg;
    };
    const double ix_t0 = now_ms();
    auto push = [&](Segment *seg) -> bool {            // takes the segment either way
        {
            const double w0 = now_ms();
            std::unique_lock<std::mutex> lk(gp.mu);
            auto &q = gp.queues[seg->seq % (uint64_t)n_dev];
            gp.cv.wait(lk, [&] { return gp.abort || q.size() < queue_depth; });
            gp.ix_wait_queue += now_ms() - w0;
            if (!gp.abort) {
                seg->t_pushed = now_ms();
                q.push_back(seg);
                gp.cv.notify_all();
                return true;
            }
        }
        discard(seg);
        return false;
    };
    while (cur) {
        if (bo >= cur->len) {
            // next block (or the end of the file)
            const bool short_block = cur->len < ring.block;
            if (short_block || bi + 1 >= ring.n_blocks) { at_end = true; break; }
            const double w0 = now_ms();
            RawRing::Block *n2 = nxt ? nxt : ring.acquire(bi + 1);
            gp.ix_wait_block += now_ms() - w0;
            if (!n2) { err = ring.err.empty() ? "read aborted" : ring.err; break; }
            bo -= cur->len;
            ring.unref(bi);
            cur = n2; nxt = nullptr; ++bi;
            continue;
        }
        size_t msize = 0;
        uint32_t isize = 0;
        bool is_bgzf = false;
        const uint8_t *hp = cur->p + bo;
        if (cur->len - bo >= 18 && hp[0] == 0x1f && hp[1] == 0x8b && hp[2] == 8 && hp[3] == 4 && hp[10] == 6 && hp[11] == 0 &&
            hp[12] == 'B' && hp[13] == 'C' && hp[14] == 2 && hp[15] == 0 &&
            bo + ((size_t)(hp[16] | (hp[17] << 8)) + 1) <= cur->len && (size_t)(hp[16] | (hp[17] << 8)) + 1 >= 26) {
            // the usual member: the standard 18-byte header, all of it inside this block
            msize = (size_t)(hp[16] | (hp[17] << 8)) + 1;
            const uint8_t *t = hp + msize - 4;
            isize = t[0] | (t[1] << 8) | (t[2] << 16) | ((uint32_t)t[3] << 24);
            is_bgzf = true;
        } else {
            uint8_t h[18];
            int k = peek(0, 18, h);
            if (k < 0) { err = ring.err.empty() ? "read aborted" : ring.err; break; }
            if (k == 1 && h[0] == 0x1f && h[1] == 0x8b && h[2] == 8 && (h[3] & 4)) {
                const uint32_t xlen = h[10] | (h[11] << 8);
                std::vector<uint8_t> x(xlen);
                const int kx = xlen >= 6 ? peek(12, xlen, x.data()) : 0;
                if (kx < 0) { err = "read aborted"; break; }
                if (kx == 1)
                    for (uint32_t p = 0; p + 4 <= xlen;) {
                        const uint32_t slen = x[p + 2] | (x[p + 3] << 8);
                        if (x[p] == 'B' && x[p + 1] == 'C' && slen == 2 && p + 6 <= xlen) { msize = (size_t)(x[p + 4] | (x[p + 5] << 8)) + 1; is_bgzf = true; break; }
                        p += 4 + slen;
                    }
                else if (xlen >= 6) { err = "truncated gzip stream"; break; }
            }
            if (k == 0) { err = "truncated gzip stream"; break; }      // fewer than 18 bytes left: no gzip member is that short
            if (!is_bgzf) { plain = true; break; }     // some other gzip member (or garbage): the host path decides
            if (msize < 26) { err = "invalid BGZF member"; break; }
            uint8_t t[4];
            k = peek(msize - 4, 4, t);
            if (k < 0) { err = "read aborted"; break; }
            if (k == 0) { err = "truncated gzip stream"; break; }
            isize = t[0] | (t[1] << 8) | (t[2] << 16) | ((uint32_t)t[3] << 24);
        }
        if (g && (g->text_bytes + isize > text_target || g->members.size() >= mcap || g->blocks.size() >= max_blocks)) {
            Segment *full = g;
            g = nullptr;
            if (!push(full)) break;
        }
        if (!g) {
            g = new Segment;
            g->seq = seq++;
            g->ring = &ring;
        }
        g->members.push_back(vfb_member{(uint32_t)g->z_bytes, (uint32_t)msize, (uint32_t)g->text_bytes, isize});
        // the member's bytes: in this block, and the next one if it straddles the boundary
        size_t left = msize, pos = bo;
        uint64_t b = bi;
        while (left) {
            RawRing::Block *blk = b == bi ? cur : nxt;
            const size_t take = std::min(left, blk->len - pos);
            // (a piece never crosses from one raw block into another: two pinned allocations may be neighbours in the
            // address space, but one copy must not span them)
            const bool same_block = !g->blocks.empty() && g->blocks.back() == b;
            if (!same_block) { g->blocks.push_back(b); ring.ref(b); }
            if (same_block && !g->pieces.empty() && g->pieces.back().p + g->pieces.back().len == blk->p + pos) g->pieces.back().len += take;
            else g->pieces.push_back(vfb_zpiece{blk->p + pos, take});
            left -= take; pos = 0; ++b;
        }
        g->z_bytes += msize;
        g->text_bytes += isize;
        bo += msize;                           // may run past the block: the loop head moves on
    }
    if (nxt) ring.unref(bi + 1);
    const uint64_t stop = cur ? file_off() : ring.base;
    if (cur) ring.unref(bi);
    if (g && err.empty() && !g->members.empty()) { push(g); g = nullptr; }
    if (g) { discard(g); --seq; }
    if (!err.empty()) { gp.fail(VFB_ERR_FORMAT, err); return; }
    std::lock_guard<std::mutex> lk(gp.mu);
    gp.ix_total = now_ms() - ix_t0;
    gp.indexed = true;
    gp.n_segments = seq;
    gp.stop_off = stop;
    gp.hit_plain = plain && !at_end;
    gp.cv.notify_all();
}

// One device: phase 1 up to two segments ahead, phase 2 in segment order.
void device_worker(vfb_ctx *ctx, int dev_index, GpuPhase &gp)
{
    std::deque<Segment *> pending;
    std::vector<uint8_t> tail(VFB_TAIL_CAP);
    auto drop = [&](Segment *g) { delete g; };
    for (;;) {
        // phase 1 for what is queued (wait only when nothing is pending)
        bool finished = false;
        while (pending.size() < VFB_SEG_SLOTS - 1) {
            Segment *g = nullptr;
            {
                const double w0 = now_ms();
                std::unique_lock<std::mutex> lk(gp.mu);
                auto &q = gp.queues[(size_t)dev_index];
                if (pending.empty()) gp.cv.wait(lk, [&] { return gp.abort || !q.empty() || gp.indexed; });
                gp.w_wait_seg[(size_t)dev_index] += now_ms() - w0;
                if (gp.abort) break;
                if (!q.empty()) { g = q.front(); q.pop_front(); gp.cv.notify_all(); }
                else { finished = gp.indexed; }
            }
            if (!g) break;
            const double b0 = now_ms();
            g->t_begin = b0;
            const int rc = vfb_internal_bgzf_begin(ctx, g->pieces.data(), (uint32_t)g->pieces.size(), g->members.data(),
                                                   (uint32_t)g->members.size(), g->text_bytes, segment_release_blocks, g, &g->slot);
            if (rc) {
                for (uint64_t b : g->blocks) g->ring->unref(b);
                gp.fail(rc, vfb_last_error());
                drop(g);
                break;
            }
            pending.push_back(g);
            gp.w_begin[(size_t)dev_index] += now_ms() - b0;
        }
        {
            std::lock_guard<std::mutex> lk(gp.mu);
            if (gp.abort) break;
        }
        if (pending.empty()) { if (finished) break; else continue; }
        Segment *g = pending.front();
        pending.pop_front();
        std::vector<uint8_t> carry;
        uint64_t record_base = 0;
        {
            const double w0 = now_ms();
            std::unique_lock<std::mutex> lk(gp.mu);
            gp.cv.wait(lk, [&] { return gp.abort || gp.link(g->seq).ready; });
            gp.w_wait_chain[(size_t)dev_index] += now_ms() - w0;
            if (gp.abort) { drop(g); break; }
            GpuPhase::Link &l = gp.link(g->seq);
            carry.swap(l.carry);
            record_base = l.records;
            while (gp.link_base < g->seq && !gp.links.empty()) { gp.links.pop_front(); ++gp.link_base; }
        }
        uint64_t n_rec = 0, tail_len = 0;
        uint32_t bad = 0xFFFFFFFFu;
        const double f0 = now_ms();
        int rc = vfb_internal_bgzf_finish(ctx, g->slot, carry.data(), carry.size(), record_base, &n_rec, tail.data(), &tail_len, &bad);
        if (rc == VFB_OK && bad != 0xFFFFFFFFu) {
            set_error("invalid gzip data in a BGZF member (deflate stream, CRC-32 or size mismatch)");
            rc = VFB_ERR_FORMAT;
        }
        if (rc) { gp.fail(rc, vfb_last_error()); drop(g); break; }
        gp.w_finish[(size_t)dev_index] += now_ms() - f0;
        {
            std::lock_guard<std::mutex> lk(gp.mu);
            gp.sum_queue_ms += g->t_begin - g->t_pushed;
            gp.sum_begin_to_fin_ms += f0 - g->t_begin;
            gp.sum_fin_ms += now_ms() - f0;
            GpuPhase::Link &l = gp.link(g->seq + 1);
            l.carry.assign(tail.data(), tail.data() + tail_len);
            l.records = record_base + n_rec;
            l.ready = true;
            gp.records_done += n_rec;
            gp.z_done += g->z_bytes;
            ++gp.segments_done;
            gp.cv.notify_all();
        }
        drop(g);
    }
    // an abort may leave segments behind whose release callback is still queued: wait for the stream, then free
    if (!pending.empty()) {
        cudaSetDevice(ctx->device);
        cudaStreamSynchronize(ctx->st_copy);
        cudaStreamSynchronize(ctx->st_ingest);
        for (Segment *g : pending) delete g;
    }
}

// Consumes BGZF members from prod.f until the end of the file or the first member that is not
// BGZF.  On return prod.carry holds the text after the last complete record, prod.at_end /
// prod.bgzf say what is left for the host path (which also applies the end-of-input rules).
int run_bgzf_gpu(vfb_ctx **ctxs, int n_dev, ChunkProducer &prod, size_t text_target, uint64_t *n_total, bool trace)
{
    const int fd = fileno(prod.f);
    const uint64_t here = (uint64_t)ftell(prod.f);
    fseek(prod.f, 0, SEEK_END);
    const uint64_t fsz = (uint64_t)ftell(prod.f);
    fseek(prod.f, (long)here, SEEK_SET);
    if (fsz <= here) { prod.at_end = true; return VFB_OK; }
    // segments: about text_target bytes of text, smaller when the file would not give every device a few of them
    if (!getenv("VFB_INGEST_CHUNK")) {
        const uint64_t est_text = (fsz - here) * 4;
        uint64_t per = est_text / ((uint64_t)n_dev * 4);
        if (per < ((uint64_t)16 << 20)) per = (uint64_t)16 << 20;
        if (per < text_target) text_target = (size_t)per;
    }
    // raw blocks of 8 MB; the ring holds 288 MB for one or two devices, up to 768 MB for eight (page-locked once per
    // process: the buffers come from the pinned pool); a segment may hold a third of the ring
    size_t block = (size_t)8 << 20;
    if (const char *e = getenv("VFB_RAW_BLOCK")) block = (size_t)strtoull(e, nullptr, 10);
    if (block < 131072) block = 131072;                     // a member (<= 64 KiB) spans at most two blocks
    if (block > fsz - here) block = (size_t)((fsz - here + 4095) & ~(uint64_t)4095);
    if (block < 131072) block = 131072;
    size_t ring_bytes = (size_t)128 << 20;
    ring_bytes *= (size_t)n_dev;
    if (ring_bytes < ((size_t)288 << 20)) ring_bytes = (size_t)288 << 20;
    if (ring_bytes > ((size_t)768 << 20)) ring_bytes = (size_t)768 << 20;
    int n_ring = (int)(ring_bytes / block);
    if (n_ring < 6) n_ring = 6;
    int n_threads = prod.threads < 1 ? 1 : prod.threads;
    if (n_threads > n_ring / 2) n_threads = n_ring / 2;
    const size_t max_blocks = (size_t)(n_ring / 3);
    RawRing ring;
    GpuPhase gp;
    gp.queues.resize((size_t)n_dev);
    gp.w_wait_seg.assign((size_t)n_dev, 0); gp.w_wait_chain.assign((size_t)n_dev, 0);
    gp.w_begin.assign((size_t)n_dev, 0); gp.w_finish.assign((size_t)n_dev, 0);
    const double phase_t0 = now_ms();
    gp.link(0).ready = true;
    gp.link(0).carry = prod.carry;
    gp.link(0).records = *n_total;
    if (!ring.start(fd, here, fsz, block, n_ring, n_threads)) {
        ring.stop();
        set_error("cannot allocate pinned ingest buffers");
        return VFB_ERR_NOMEM;
    }
    vfb::trace("ingest: %d raw blocks of %zu MB, %d reader threads, %d device(s), segments of %zu MB of text", (int)ring.ring.size(),
               block >> 20, n_threads, n_dev, text_target >> 20);
    const size_t mcap = text_target / 512 + 4096;
    std::thread indexer([&] { index_members(ring, gp, text_target, mcap, max_blocks, n_dev, 2); });
    std::vector<std::thread> workers;
    for (int d = 0; d < n_dev; ++d) workers.emplace_back([&, d] { device_worker(ctxs[d], d, gp); });
    // the calling thread: progress and the end
    const uint64_t base_records = *n_total;
    {
        std::unique_lock<std::mutex> lk(gp.mu);
        for (;;) {
            gp.cv.wait_for(lk, std::chrono::milliseconds(100), [&] { return gp.abort || (gp.indexed && gp.segments_done == gp.n_segments); });
            if (gp.abort || (gp.indexed && gp.segments_done == gp.n_segments)) break;
            const uint64_t r = base_records + gp.records_done, z = here + gp.z_done;
            lk.unlock();
            vfb_internal_progress(ctxs[0], r, z, prod.file_size, false);
            lk.lock();
        }
    }
    {
        // an abort must reach the threads that wait on the ring, too
        std::lock_guard<std::mutex> lk(gp.mu);
        if (gp.abort) { std::lock_guard<std::mutex> l2(ring.mu); ring.abort = true; ring.cv.notify_all(); }
    }
    indexer.join();
    for (auto &t : workers) t.join();
    int rc = gp.rc;
    std::string keep = gp.err;
    for (int d = 0; d < n_dev; ++d) {
        const int src = vfb_sync(ctxs[d]);     // the raw blocks are about to go away
        if (src && rc == VFB_OK) { rc = src; keep = vfb_last_error(); }
    }
    for (auto &q : gp.queues) for (Segment *g : q) { for (uint64_t b : g->blocks) ring.unref(b); delete g; }
    ring.stop();
    const double ring_read_ms = ring.t_read_ms, ring_wait_ms = ring.t_wait_ms;
    if (rc) { set_error(keep); return rc; }
    GpuPhase::Link &last = gp.link(gp.n_segments);
    prod.carry = last.carry;
    *n_total = last.records;
    if (trace) {
        fprintf(stderr, "[vfb ingest] gpu phase %.1f ms; indexer %.1f ms (waited %.1f for blocks, %.1f for queue room)\n",
                now_ms() - phase_t0, gp.ix_total, gp.ix_wait_block, gp.ix_wait_queue);
        fprintf(stderr, "[vfb ingest]   readers (summed over %d threads): %.1f ms in pread, %.1f ms waiting for a free block of %d\n",
                n_threads, ring_read_ms, ring_wait_ms, n_ring);
        if (gp.n_segments)
            fprintf(stderr, "[vfb ingest]   per segment: %.2f ms queued, %.2f ms from begin to the start of finish, %.2f ms in finish\n",
                    gp.sum_queue_ms / gp.n_segments, gp.sum_begin_to_fin_ms / gp.n_segments, gp.sum_fin_ms / gp.n_segments);
        for (int d = 0; d < n_dev; ++d)
            fprintf(stderr, "[vfb ingest]   device %d: waited %.1f ms for segments, %.1f ms for the chain; begin %.1f ms, finish %.1f ms\n",
                    ctxs[d]->device, gp.w_wait_seg[(size_t)d], gp.w_wait_chain[(size_t)d], gp.w_begin[(size_t)d], gp.w_finish[(size_t)d]);
    }
    if (trace) fprintf(stderr, "[vfb ingest] gpu phase: %llu segments, %llu records, stopped at offset %llu of %llu%s\n",
                       (unsigned long long)gp.n_segments, (unsigned long long)(*n_total - base_records),
                       (unsigned long long)gp.stop_off, (unsigned long long)fsz, gp.hit_plain ? " (a plain gzip member follows)" : "");
    fseek(prod.f, (long)gp.stop_off, SEEK_SET);      // the host path continues where the GPU phase stopped
    if (gp.hit_plain) prod.bgzf = false;
    else prod.at_end = true;
    prod.consumed = gp.stop_off;
    vfb_internal_progress(ctxs[0], *n_total, gp.stop_off, prod.file_size, false);
    return VFB_OK;
}

}  // namespace

// Host-only view of the ingest front half (no GPU): inflates `path` chunk by chunk exactly as
// vfb_run_file does and returns the concatenated submitted text, the number of complete lines
// and the number of chunks.  For CPU tests of the inflate / cut / carry logic.
extern "C" int vfb_debug_inflate_file(const char *path, uint32_t n_threads, uint8_t *out, uint64_t out_cap,
                                      uint64_t *n_bytes, uint64_t *n_lines, uint64_t *n_chunks)
{
    if (!path || !n_bytes || !n_lines) { set_error("null argument"); return VFB_ERR_ARG; }
    ChunkProducer prod;
    std::string e;
    if (!prod.open(path, (int)n_threads, &e)) { set_error(e); return VFB_ERR_IO; }
    {
        // the device decoder for plain gzip takes part when asked for (VFB_GPU_GUNZIP=1 / 2) and a device is there
        const char *g = getenv("VFB_GPU_GUNZIP");
        int nd = 0;
        if (g && g[0] != '0' && cudaGetDeviceCount(&nd) == cudaSuccess && nd > 0) prod.gpu_device = 0;
        else cudaGetLastError();
    }
    const size_t cap = pick_chunk(prod.f);
    std::vector<uint8_t> buf(cap + 64);
    uint64_t total = 0, lines = 0, chunks = 0;
    for (;;) {
        size_t cut = 0, kl = 0;
        bool last = false;
        const int rc = prod.next(buf.data(), cap, &cut, &kl, &last);
        if (rc) { set_error(prod.err); return rc; }
        if (out) {
            if (total + cut > out_cap) { set_error("output buffer too small"); return VFB_ERR_ARG; }
            memcpy(out + total, buf.data(), cut);
        }
        total += cut;
        lines += kl;
        ++chunks;
        if (last) break;
    }
    *n_bytes = total;
    *n_lines = lines;
    if (n_chunks) *n_chunks = chunks;
    return VFB_OK;
}

extern "C" int vfb_run_file(vfb_ctx *ctx, const char *path, uint64_t *n_reads_out)
{
    return vfb_run_file_ex(ctx, path, 0, n_reads_out);
}

extern "C" int vfb_run_file_ex(vfb_ctx *ctx, const char *path, uint32_t flags, uint64_t *n_reads_out)
{
    if (!ctx || !path) { set_error("null argument"); return VFB_ERR_ARG; }
    return vfb_internal_run_file(&ctx, 1, path, flags, n_reads_out);
}

// One file over n_ctx contexts (one per device; vfb_multi_run_file): block-gzip segments and host-inflated
// chunks are dealt round robin, every context counts what it is given into its own table.
int vfb_internal_run_file(vfb_ctx **ctxs, uint32_t n_ctx, const char *path, uint32_t flags, uint64_t *n_reads_out)
{
    vfb_ctx *ctx = ctxs[0];
    ChunkProducer prod;
    {
        std::string e;
        if (!prod.open(path, vfb_internal_ingest_threads(ctx), &e, (flags & VFB_INPUT_ALLOW_TEXT) != 0)) { set_error(e); return VFB_ERR_IO; }
        prod.gpu_device = ctx->device;
    }
    size_t cap = pick_chunk(prod.f);
    const bool trace = getenv("VFB_INGEST_TRACE") != nullptr;
    const auto t_start = std::chrono::steady_clock::now();
    uint64_t n_total = 0;
    int rc = VFB_OK;
    // Block-gzip input is inflated on the GPU (VFB_GPU_INFLATE=0 keeps it on the host threads);
    // whatever follows — plain gzip members, the end-of-input rules — goes through the host path.
    const char *gi = getenv("VFB_GPU_INFLATE");
    if (prod.bgzf && !(gi && gi[0] == '0')) {
        if (trace) fprintf(stderr, "[vfb ingest] %s: block gzip, inflating on the GPU\n", path);
        // (segments of about 6500 members: the inflate kernel keeps 44 warps = members per SM in flight, and a launch
        // takes as long as its slowest member whether the SMs are full or not — measured 48 GB/s of text at 4096
        // members per launch, 55.6 GB/s at 6500)
        rc = run_bgzf_gpu(ctxs, (int)n_ctx, prod, getenv("VFB_INGEST_CHUNK") ? cap : ((size_t)416 << 20), &n_total, trace);
        if (rc) return rc;
        // only the text after the last complete record may be left: no need for big chunks
        if (prod.at_end) cap = prod.carry.size() * 2 + 65536;
    }

    constexpr int NCH = 3;
    Chunk ch[NCH];
    std::vector<cudaEvent_t> ch_events((size_t)NCH * n_ctx, nullptr);     // [chunk][context]: an event belongs to a device
    int ch_ctx[NCH] = {0, 0, 0};
    Pipe pp;
    for (int i = 0; i < NCH; ++i) {
        void *p = pinned_acquire(cap + 64, &ch[i].buf_cap);
        if (!p) { set_error("cannot allocate pinned ingest buffers"); rc = VFB_ERR_NOMEM; }
        ch[i].buf = (uint8_t *)p;
        pp.free_q.push_back(i);
        for (uint32_t d = 0; d < n_ctx && rc == VFB_OK; ++d)
            if (cudaSetDevice(ctxs[d]->device) != cudaSuccess ||
                cudaEventCreateWithFlags(&ch_events[(size_t)i * n_ctx + d], cudaEventDisableTiming) != cudaSuccess) {
                cudaGetLastError();
                set_error("cannot create ingest events");
                rc = VFB_ERR_CUDA;
            }
    }

    auto ms_since = [&](std::chrono::steady_clock::time_point t) {
        return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t).count();
    };
    if (trace) fprintf(stderr, "[vfb ingest] %s: %s, chunk %zu bytes, %d inflate threads\n", path,
                       prod.plain ? "plain text" : (prod.bgzf ? "block gzip (member-parallel)" : "gzip stream (serial)"), cap, prod.threads);
    std::thread producer;
    if (rc == VFB_OK) producer = std::thread([&]() {
        for (;;) {
            int k;
            {
                std::unique_lock<std::mutex> lk(pp.mu);
                pp.cv.wait(lk, [&] { return !pp.free_q.empty() || pp.abort; });
                if (pp.abort) return;
                k = pp.free_q.front();
                pp.free_q.pop_front();
            }
            bool last = false;
            const auto t0 = std::chrono::steady_clock::now();
            const int prc = prod.next(ch[k].buf, cap, &ch[k].cut, &ch[k].lines, &last, &ch[k].dev, &ch[k].dev_len);
            if (trace) fprintf(stderr, "[vfb ingest] chunk %zu bytes %zu lines inflated in %.1f ms\n", ch[k].cut, ch[k].lines,
                               std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count());
            std::lock_guard<std::mutex> lk(pp.mu);
            if (prc) {
                pp.failed = true; pp.err = prod.err; pp.err_code = prc; pp.done = true;
                pp.cv.notify_all();
                return;
            }
            pp.ready_q.push_back(k);
            if (last) pp.done = true;
            pp.cv.notify_all();
            if (last) return;
        }
    });

    std::deque<int> in_flight;
    uint64_t n_chunks = 0;
    while (rc == VFB_OK) {
        int k = -1;
        {
            std::unique_lock<std::mutex> lk(pp.mu);
            pp.cv.wait(lk, [&] { return !pp.ready_q.empty() || pp.done; });
            if (!pp.ready_q.empty()) { k = pp.ready_q.front(); pp.ready_q.pop_front(); }
            else if (pp.failed) { set_error(pp.err); rc = pp.err_code; break; }
            else break;     // done and drained
        }
        Chunk &c = ch[k];
        const uint32_t d = (uint32_t)(n_chunks++ % n_ctx);
        ch_ctx[k] = (int)d;
        c.copied = ch_events[(size_t)k * n_ctx + d];
        if (c.lines) {
            const auto t0 = std::chrono::steady_clock::now();
            if (c.dev_len) {
                rc = vfb_internal_submit_fastq_dev(ctxs[d], c.buf, c.cut, c.dev.d_ptr, c.dev_len, c.dev.device, c.lines, n_total, c.copied);
                prod.ggz.release_device(c.dev);       // (the copy out of the range has completed)
                c.dev_len = 0;
            } else
            rc = vfb_internal_submit_fastq(ctxs[d], c.buf, c.cut, c.lines, n_total, c.copied);
            if (trace) fprintf(stderr, "[vfb ingest] submit at %.1f ms took %.1f ms\n", ms_since(t_start), ms_since(t0));
            n_total += c.lines / 4;
            vfb_internal_progress(ctx, n_total, prod.consumed.load(), prod.file_size, false);
        } else if (cudaSetDevice(ctxs[d]->device) != cudaSuccess || cudaEventRecord(c.copied, ctxs[d]->st_copy) != cudaSuccess) {
            cudaGetLastError();
        }
        in_flight.push_back(k);
        // hand buffers back to the producer once their H2D copy has finished; the newest copy
        // stays outstanding so that inflating the next chunk overlaps it
        while (rc == VFB_OK && in_flight.size() > 1) {
            const int o = in_flight.front();
            cudaSetDevice(ctxs[ch_ctx[o]]->device);
            if (cudaEventSynchronize(ch[o].copied) != cudaSuccess) { rc = cuda_fail(cudaGetLastError(), "ingest event", __FILE__, __LINE__); break; }
            in_flight.pop_front();
            std::lock_guard<std::mutex> lk(pp.mu);
            pp.free_q.push_back(o);
            pp.cv.notify_all();
        }
    }
    {
        std::lock_guard<std::mutex> lk(pp.mu);
        pp.abort = true;
        pp.cv.notify_all();
    }
    if (producer.joinable()) producer.join();
    if (rc == VFB_OK && pp.failed) { set_error(pp.err); rc = pp.err_code; }
    // the malformed-record flag comes back from the device
    std::string keep = rc ? std::string(vfb_last_error()) : std::string();
    if (trace) fprintf(stderr, "[vfb ingest] all chunks queued at %.1f ms\n", ms_since(t_start));
    for (uint32_t d = 0; d < n_ctx; ++d) {
        const int src = vfb_sync(ctxs[d]);
        if (src && rc == VFB_OK) { rc = src; keep = vfb_last_error(); }
    }
    if (trace) fprintf(stderr, "[vfb ingest] device drained at %.1f ms\n", ms_since(t_start));
    if (rc) set_error(keep);
    if (rc == VFB_OK) {
        uint64_t bad = UINT64_MAX;
        for (uint32_t d = 0; d < n_ctx && rc == VFB_OK; ++d) {
            uint64_t b = UINT64_MAX;
            rc = vfb_internal_parse_error(ctxs[d], &b);
            if (b < bad) bad = b;
        }
        if (rc == VFB_OK && bad != UINT64_MAX) {
            set_error("FASTQ record " + std::to_string(bad) +
                      ": malformed (expected '@' header, '+' separator, sequence and quality of equal length)");
            rc = VFB_ERR_FORMAT;
        }
    }
    for (int i = 0; i < NCH; ++i) pinned_release(ch[i].buf, ch[i].buf_cap);
    for (size_t i = 0; i < ch_events.size(); ++i)
        if (ch_events[i]) { cudaSetDevice(ctxs[i % n_ctx]->device); cudaEventDestroy(ch_events[i]); }
    if (n_reads_out) *n_reads_out = n_total;
    if (rc == VFB_OK) vfb_internal_progress(ctx, n_total, prod.file_size, prod.file_size, true);
    if (trace) fprintf(stderr, "[vfb ingest] %llu records in %.1f ms\n", (unsigned long long)n_total,
                       std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_start).count());
    return rc;
}
