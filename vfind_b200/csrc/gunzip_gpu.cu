// Single-stream gzip decoded on the device: the host side (segments, candidate selection, hand-over to zlib).
// Kernels and the scheme: kernels_inflate.cu ("Single-stream gzip on the device").  Replaces flate2's MultiGzDecoder
// (/root/reference/src/lib.rs:233) for the FIRST member of a plain gzip file; whatever the device cannot take — further
// members, a chunk that runs out of room, a stream without usable block starts — is inflated by zlib from the exact bit
// where the device stopped (raw inflate primed with the bits of the first byte and the text before it, up to 32 KiB, as
// dictionary), so every valid gzip file decodes to the same bytes either way.  CRC-32 and ISIZE are checked as flate2 does.
#include "gunzip_gpu.h"

#include <unistd.h>
#include <zlib.h>

#include <algorithm>
#include <chrono>
#include <condition_variable>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <thread>
#include <vector>

#include "ctx.cuh"

namespace vfb {

namespace {

struct CudaCheck {
    std::string *err;
    bool ok(cudaError_t e, const char *what)
    {
        if (e == cudaSuccess) return true;
        *err = std::string("CUDA error in the gzip decoder (") + what + "): " + cudaGetErrorString(e);
        cudaGetLastError();
        return false;
    }
};

}  // namespace

struct GpuGunzip::Impl {
    FILE *f = nullptr;
    int fd = -1;
    int device = 0;
    cudaStream_t st = nullptr;
    uint64_t file_size = 0;
    // where the deflate stream continues: file byte offset and bit inside that byte
    uint64_t byte_pos = 0;
    uint32_t bit_in_byte = 0;
    uint32_t hist = 0;                       // bytes of text before byte_pos/bit_in_byte, at most VFB_GZ_WIN
    std::vector<uint8_t> window;             // the 32 KiB before byte_pos/bit_in_byte: the last `hist` bytes are text
    uint32_t crc = 0;                        // of the member's text so far
    uint64_t text_total = 0;
    // parameters
    size_t seg_bytes = (size_t)224 << 20;    // compressed bytes per segment (a chunk is one warp: thousands are wanted at once)
    size_t ovl_bytes = (size_t)2 << 20;      // looked at beyond the segment for a landing spot
    uint32_t min_gap_bits = 32u * 1024u * 8u;   // chunk starts at least this far apart: the chain is serial over the chunks
    uint32_t cap_syms = 768u * 1024u;        // symbols per chunk region (a chunk may have to run over a block start the search missed)
    // buffers
    PinBuf h_small;
    DevBuf d_starts, d_res, d_out16, d_live, d_text_off, d_win_store, d_win_in, d_win_out, d_chain, d_nl,
        d_crc, d_flags;
    // The front half of a segment — read the compressed bytes, copy them in, search the candidates — does not depend on
    // where exactly the stream enters the segment (a candidate inside the first `ovl_bytes`), so the NEXT segment's front runs
    // on a thread and a stream of its own while this segment is decoded, chained and resolved.
    struct Front {
        PinBuf h_z, h_cand;
        DevBuf d_z, d_cand, d_list;
        cudaStream_t st = nullptr;
        std::thread th;
        bool started = false, ok = false;
        std::string err;
        uint64_t base_byte = 0;              // file offset of the buffer's first byte
        size_t want = 0;
        bool last_segment = false;
        uint32_t n_words = 0, n_cand = 0;
        double t_read = 0, t_search = 0;
    };
    Front fronts[2];
    int front_cur = 0;

    // Segments are produced by a thread of their own, two ahead of the reader at most: a slot is a segment's text on the
    // device with its newline counts.
    struct Slot {
        DevBuf d_text;
        uint64_t text = 0;
        std::vector<uint32_t> nl;            // newlines per VFB_GZ_PIECE
        uint32_t outstanding = 0;            // ranges handed out with peek / commit_device and not released yet
    };
    static constexpr int N_SLOTS = 2;
    Slot slots[N_SLOTS];
    std::mutex mu;
    std::condition_variable cv;
    uint64_t produced_seq = 0, consumed_seq = 0;     // slots [consumed_seq, produced_seq) are ready, in order
    bool producer_done = false, stop = false;
    std::string producer_err;
    std::thread producer;
    cudaStream_t st_out = nullptr;           // the reader's copies
    uint64_t cur_served = 0;                 // bytes of slot consumed_seq % N_SLOTS already handed out
    // state
    enum { GPU, HOST, TRAILER_DONE, FAILED } mode = GPU;
    z_stream zs;
    bool zs_open = false;
    std::vector<uint8_t> zin;
    bool member_final_seen = false;
    long handover_off = -1;
    uint64_t n_segments = 0, n_chunks_total = 0, n_live_total = 0, host_bytes = 0, host_takeovers = 0;
    uint64_t host_since = 0;                 // text bytes zlib has produced since it last took over
    bool trace = false;
    std::chrono::steady_clock::time_point t_init = std::chrono::steady_clock::now();
    double since_init() const { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_init).count(); }

    ~Impl()
    {
        {
            std::lock_guard<std::mutex> lk(mu);
            stop = true;
            cv.notify_all();
        }
        if (producer.joinable()) producer.join();
        if (zs_open) inflateEnd(&zs);
        cudaSetDevice(device);
        if (st) { cudaStreamSynchronize(st); cudaStreamDestroy(st); }
        if (st_out) { cudaStreamSynchronize(st_out); cudaStreamDestroy(st_out); }
        for (auto &fr : fronts) {
            if (fr.th.joinable()) fr.th.join();
            if (fr.st) { cudaStreamSynchronize(fr.st); cudaStreamDestroy(fr.st); }
            fr.d_z.release(); fr.d_cand.release(); fr.d_list.release();
            fr.h_z.release(); fr.h_cand.release();
        }
        DevBuf *db[] = {&d_starts, &d_res, &d_out16, &d_live, &d_text_off, &d_win_store, &d_win_in, &d_win_out,
                        &d_chain, &d_nl, &d_crc, &d_flags, &slots[0].d_text, &slots[1].d_text};
        for (auto *b : db) b->release();
        h_small.release();
    }

    bool parse_header(std::string *err)
    {
        // gzip member header (RFC 1952) at the current file position
        uint8_t h[10];
        const long pos = ftell(f);
        if (fread(h, 1, 10, f) != 10 || h[0] != 0x1f || h[1] != 0x8b || h[2] != 8) { fseek(f, pos, SEEK_SET); *err = "not a gzip member"; return false; }
        const int flg = h[3];
        if (flg & 4) {
            uint8_t x[2];
            if (fread(x, 1, 2, f) != 2) { fseek(f, pos, SEEK_SET); return false; }
            if (fseek(f, x[0] | (x[1] << 8), SEEK_CUR) != 0) { fseek(f, pos, SEEK_SET); return false; }
        }
        for (int bit : {8, 16})
            if (flg & bit) {
                int c;
                while ((c = fgetc(f)) != EOF && c != 0) {}
                if (c == EOF) { fseek(f, pos, SEEK_SET); return false; }
            }
        if (flg & 2) fseek(f, 2, SEEK_CUR);
        byte_pos = (uint64_t)ftell(f);
        bit_in_byte = 0;
        fseek(f, pos, SEEK_SET);
        return true;
    }

    // Read [base, base + seg + ovl), copy it in, search every bit offset: on a thread of its own.
    void front_start(Front &fr, uint64_t base)
    {
        if (fr.th.joinable()) fr.th.join();
        fr.started = true;
        fr.ok = false;
        fr.err.clear();
        fr.base_byte = base;
        const uint64_t avail = file_size - base;
        fr.want = (size_t)std::min<uint64_t>(avail, seg_bytes + ovl_bytes);
        fr.last_segment = avail <= seg_bytes + ovl_bytes;
        fr.th = std::thread([this, &fr]() {
            CudaCheck ck{&fr.err};
            const auto t0 = std::chrono::steady_clock::now();
            auto ms = [&]() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count(); };
            if (!ck.ok(cudaSetDevice(device), "set device")) return;
            if (!fr.st && !ck.ok(cudaStreamCreateWithFlags(&fr.st, cudaStreamNonBlocking), "stream")) return;
            const size_t want = fr.want;
            if (fr.h_z.ensure(want + 64)) { fr.err = "cannot allocate pinned memory"; return; }
            {
                // the page cache hands a few GB/s to one thread: read in parallel
                const int parts = want >= ((size_t)32 << 20) ? 8 : 1;
                const size_t part = ((want / parts) + 4095) & ~(size_t)4095;
                std::vector<int> bad((size_t)parts, 0);
                auto rd = [&](int i) {
                    const size_t lo = (size_t)i * part, hi = std::min(want, lo + part);
                    size_t got = lo;
                    while (got < hi) {
                        const ssize_t r = pread(fd, (uint8_t *)fr.h_z.p + got, hi - got, (off_t)(fr.base_byte + got));
                        if (r <= 0) { bad[(size_t)i] = 1; return; }
                        got += (size_t)r;
                    }
                };
                std::vector<std::thread> pool;
                for (int i = 1; i < parts; ++i) pool.emplace_back(rd, i);
                rd(0);
                for (auto &t : pool) t.join();
                for (int b : bad) if (b) { fr.err = "truncated gzip stream"; return; }
            }
            fr.t_read = ms();
            fr.n_words = (uint32_t)((want + 3) / 4);
            memset((uint8_t *)fr.h_z.p + want, 0, 8);
            if (fr.d_z.ensure((size_t)fr.n_words * 4 + 64)) { fr.err = vfb_last_error(); return; }
            if (!ck.ok(cudaMemcpyAsync(fr.d_z.p, fr.h_z.p, (size_t)fr.n_words * 4, cudaMemcpyHostToDevice, fr.st), "copy in")) return;
            const uint32_t total_bits = (uint32_t)(want * 8);
            const uint32_t cand_cap = (uint32_t)(want / 256) + 1024;
            if (fr.d_cand.ensure((size_t)(cand_cap + 4) * 4)) { fr.err = vfb_last_error(); return; }
            uint32_t *d_ncand = fr.d_cand.as<uint32_t>() + cand_cap;
            if (!ck.ok(cudaMemsetAsync(d_ncand, 0, 4, fr.st), "memset")) return;
            const uint32_t list_cap = (uint32_t)(want / 16) + 4096;       // about one offset in 500 passes the first test
            if (fr.d_list.ensure((size_t)(list_cap + 4) * 4)) { fr.err = vfb_last_error(); return; }
            if (launch_gz_search(fr.d_z.as<uint32_t>(), fr.n_words, 0, total_bits, fr.d_cand.as<uint32_t>(), d_ncand, cand_cap,
                                 fr.d_list.as<uint32_t>(), list_cap, fr.st)) { fr.err = vfb_last_error(); return; }
            if (fr.h_cand.ensure((size_t)(cand_cap + 4) * 4)) { fr.err = "cannot allocate pinned memory"; return; }
            uint32_t *h_cand = (uint32_t *)fr.h_cand.p;
            if (!ck.ok(cudaMemcpyAsync(h_cand, fr.d_cand.p, (size_t)(cand_cap + 4) * 4, cudaMemcpyDeviceToHost, fr.st), "copy candidates")) return;
            if (!ck.ok(cudaStreamSynchronize(fr.st), "search")) return;
            fr.n_cand = std::min(h_cand[cand_cap], cand_cap);   // (more than one per 256 bytes: keep what fits; they only bound chunk sizes)
            std::sort(h_cand, h_cand + fr.n_cand);
            fr.t_search = ms();
            fr.ok = true;
        });
    }

    // ---- one segment on the device.  Returns false with *err set on a CUDA / IO error; otherwise the segment's text is
    // in d_text (seg_text bytes, possibly 0) and the state has moved on (mode may have changed).
    bool run_segment(Slot &slot, std::string *err)
    {
        CudaCheck ck{err};
        if (!ck.ok(cudaSetDevice(device), "set device")) return false;
        slot.text = 0;
        const auto t0 = std::chrono::steady_clock::now();
        auto ms = [&]() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count(); };
        double t_read = 0, t_search = 0, t_decode = 0, t_resolve = 0;
        // ---- the front: prefetched (the buffer then starts seg_bytes behind the previous one's, the stream enters it a
        // little later), or done now (the first segment, and after zlib has handed the stream back)
        Front *fr = &fronts[front_cur];
        if (fr->started && !(fr->base_byte <= byte_pos && byte_pos - fr->base_byte < ovl_bytes)) {
            if (fr->th.joinable()) fr->th.join();
            fr->started = false;                              // not where the stream is: drop it
        }
        if (!fr->started) front_start(*fr, byte_pos);
        if (fr->th.joinable()) fr->th.join();
        fr->started = false;
        if (!fr->ok) { *err = fr->err; return false; }
        const uint64_t base = fr->base_byte;
        const size_t want = fr->want;
        const bool last_segment = fr->last_segment;
        const uint32_t n_words = fr->n_words;
        DevBuf &d_z = fr->d_z;
        const uint32_t start_bit = (uint32_t)((byte_pos - base) * 8u) + bit_in_byte;
        t_read = fr->t_read;
        t_search = fr->t_search;
        const uint32_t limit_bit = last_segment ? 0xFFFFFFFFu : (uint32_t)(seg_bytes * 8);
        // the next segment's front starts right away
        if (!last_segment) {
            front_cur ^= 1;
            front_start(fronts[front_cur], base + seg_bytes);
        }
        const uint32_t cand_cap = (uint32_t)(want / 256) + 1024;
        if (h_small.ensure(VFB_GZ_WIN + 256)) { *err = "cannot allocate pinned memory"; return false; }
        const uint32_t *h_cand = (const uint32_t *)fr->h_cand.p;
        const uint32_t n_cand = fr->n_cand;
        std::vector<uint32_t> starts;
        starts.push_back(start_bit);
        for (uint32_t i = 0; i < n_cand; ++i)
            if (h_cand[i] > start_bit && h_cand[i] >= starts.back() + min_gap_bits) starts.push_back(h_cand[i]);
        const uint32_t n_chunks = (uint32_t)starts.size();
        // ---- decode
        if (d_starts.ensure((size_t)n_chunks * 4) || d_res.ensure((size_t)n_chunks * VFB_GZ_RES_BYTES)) { *err = vfb_last_error(); return false; }
        if (d_out16.ensure((size_t)n_chunks * ((size_t)VFB_GZ_WIN + cap_syms) * 2)) { *err = "out of device memory for the gzip decoder"; return false; }
        if (d_live.ensure((size_t)(n_chunks + 1) * 4) || d_text_off.ensure((size_t)(n_chunks + 2) * 8) ||
            d_win_store.ensure((size_t)n_chunks * VFB_GZ_WIN) || d_win_in.ensure(VFB_GZ_WIN) || d_win_out.ensure(VFB_GZ_WIN) ||
            d_chain.ensure(64) || d_flags.ensure(16)) { *err = vfb_last_error(); return false; }
        (void)cand_cap;
        uint8_t *h_win = (uint8_t *)h_small.p;
        memcpy(h_win, window.data(), VFB_GZ_WIN);
        if (!ck.ok(cudaMemcpyAsync(d_win_in.p, h_win, VFB_GZ_WIN, cudaMemcpyHostToDevice, st), "copy window")) return false;
        if (!ck.ok(cudaMemcpyAsync(d_starts.p, starts.data(), (size_t)n_chunks * 4, cudaMemcpyHostToDevice, st), "copy starts")) return false;
        if (!ck.ok(cudaMemsetAsync(d_flags.p, 0, 16, st), "memset")) return false;
        // chunks that start at or beyond the limit are landing spots only
        uint32_t n_decode = n_chunks;
        while (n_decode > 1 && starts[n_decode - 1] >= limit_bit) --n_decode;
        if (n_decode < n_chunks)
            if (!ck.ok(cudaMemsetAsync((uint8_t *)d_res.p + (size_t)n_decode * VFB_GZ_RES_BYTES, 0xFF,
                                       (size_t)(n_chunks - n_decode) * VFB_GZ_RES_BYTES, st), "memset")) return false;
        const uint32_t max_span = (uint32_t)std::min<uint64_t>(0x7FFFFFFFull, (uint64_t)cap_syms * 8ull);
        // (the starts handed to the kernel include the landing spots; only the first n_decode are decoded)
        cudaEvent_t ev[3] = {nullptr, nullptr, nullptr};
        if (trace) { for (auto &e : ev) cudaEventCreate(&e); cudaEventRecord(ev[0], st); }
        if (launch_gz_decode_n(d_z, n_decode, n_chunks, n_words, max_span)) { *err = vfb_last_error(); return false; }
        if (trace) cudaEventRecord(ev[1], st);
        if (launch_gz_chain(d_res.p, d_starts.as<uint32_t>(), n_chunks, d_out16.as<uint16_t>(), cap_syms, limit_bit,
                            d_win_in.as<uint8_t>(), d_live.as<uint32_t>(), d_text_off.as<unsigned long long>(),
                            d_win_store.as<uint8_t>(), d_win_out.as<uint8_t>(), d_chain.p, st)) { *err = vfb_last_error(); return false; }
        if (trace) cudaEventRecord(ev[2], st);
        vfb_gz_chain_out co;
        if (!ck.ok(cudaMemcpyAsync(&co, d_chain.p, sizeof co, cudaMemcpyDeviceToHost, st), "copy chain")) return false;
        if (!ck.ok(cudaMemcpyAsync(h_win, d_win_out.p, VFB_GZ_WIN, cudaMemcpyDeviceToHost, st), "copy window")) return false;
        if (!ck.ok(cudaStreamSynchronize(st), "decode")) return false;
        t_decode = ms();
        if (trace) {
            float a = 0, b = 0;
            cudaEventElapsedTime(&a, ev[0], ev[1]);
            cudaEventElapsedTime(&b, ev[1], ev[2]);
            fprintf(stderr, "[vfb gunzip]   decode kernel %.1f ms, chain kernel %.1f ms\n", a, b);
            for (auto &e : ev) cudaEventDestroy(e);
        }
        ++n_segments;
        n_chunks_total += n_decode;
        n_live_total += co.n_live;
        // ---- text
        const uint64_t total = co.total_text;
        std::vector<uint32_t> piece_crc;
        if (total) {
            const size_t np = (size_t)((total + VFB_GZ_PIECE - 1) / VFB_GZ_PIECE), nc = (size_t)((total + VFB_GZ_CRC_PIECE - 1) / VFB_GZ_CRC_PIECE);
            if (slot.d_text.ensure(total + 64) || d_nl.ensure(np * 4) || d_crc.ensure(nc * 4)) { *err = "out of device memory for the gzip decoder"; return false; }
            if (launch_gz_resolve(d_live.as<uint32_t>(), d_text_off.as<unsigned long long>(), co.n_live, total, d_out16.as<uint16_t>(),
                                  cap_syms, d_win_store.as<uint8_t>(), slot.d_text.as<uint8_t>(), d_nl.as<uint32_t>(), d_crc.as<uint32_t>(),
                                  hist, d_flags.as<uint32_t>(), st)) { *err = vfb_last_error(); return false; }
            slot.nl.resize(np);
            piece_crc.resize(nc);
            uint32_t flag = 0;
            if (!ck.ok(cudaMemcpyAsync(slot.nl.data(), d_nl.p, np * 4, cudaMemcpyDeviceToHost, st), "copy counts")) return false;
            if (!ck.ok(cudaMemcpyAsync(piece_crc.data(), d_crc.p, nc * 4, cudaMemcpyDeviceToHost, st), "copy crc")) return false;
            if (!ck.ok(cudaMemcpyAsync(&flag, d_flags.p, 4, cudaMemcpyDeviceToHost, st), "copy flag")) return false;
            if (!ck.ok(cudaStreamSynchronize(st), "resolve")) return false;
            if (flag) { *err = "invalid gzip data: invalid distance too far back"; mode = FAILED; return false; }
            // CRC of the segment's text, appended to the member's
            uLong op = crc32_combine_gen((z_off_t)VFB_GZ_CRC_PIECE);
            for (size_t i = 0; i < nc; ++i) {
                const uint64_t len = std::min<uint64_t>(VFB_GZ_CRC_PIECE, total - (uint64_t)i * VFB_GZ_CRC_PIECE);
                crc = len == VFB_GZ_CRC_PIECE ? (uint32_t)crc32_combine_op(crc, piece_crc[i], op)
                                              : (uint32_t)crc32_combine(crc, piece_crc[i], (z_off_t)len);
            }
            text_total += total;
            window.assign(h_win, h_win + VFB_GZ_WIN);
            hist = (uint32_t)std::min<uint64_t>((uint64_t)hist + total, VFB_GZ_WIN);
        }
        slot.text = total;
        t_resolve = ms();
        if (trace)
            fprintf(stderr, "[vfb gunzip]   front (ahead of time when prefetched): read %.1f ms, copy + search %.1f; decode + chain %.1f, resolve + crc %.1f\n",
                    t_read, t_search - t_read, t_decode, t_resolve - t_decode);
        if (trace)
            fprintf(stderr, "[vfb gunzip] segment %llu: %zu compressed bytes, %u candidates, %u chunks, %u visited, %llu text bytes, end %u at bit %u (code %u)\n",
                    (unsigned long long)n_segments, want, n_cand, n_decode, co.n_live, (unsigned long long)total, co.end_kind, co.end_bit, co.reserved);
        // ---- where the stream goes on
        byte_pos = base + (co.end_bit >> 3);
        bit_in_byte = co.end_bit & 7u;
        if (co.end_kind == 1) {
            // the final block: trailer at the next byte boundary
            const uint64_t tr = base + ((uint64_t)co.end_bit + 7) / 8;
            return finish_member(tr, err);
        }
        if (co.end_kind == 2 || (co.end_kind == 0 && co.n_live == 0)) {
            // a chunk the device could not take (or no progress): zlib carries on from its first bit
            return start_host(err);
        }
        return true;
    }

    int launch_gz_decode_n(const DevBuf &d_z, uint32_t n_decode, uint32_t n_chunks, uint32_t n_words, uint32_t max_span)
    {
        // the kernel looks landings up in all n_chunks starts and decodes the first n_decode chunks
        return launch_gz_decode(d_z.as<uint32_t>(), n_words, d_starts.as<uint32_t>(), n_chunks, n_decode, d_out16.as<uint16_t>(), cap_syms,
                                max_span, d_res.p, st);
    }

    bool finish_member(uint64_t trailer_off, std::string *err)
    {
        uint8_t t[8];
        if (trailer_off + 8 > file_size || pread(fd, t, 8, (off_t)trailer_off) != 8) { *err = "truncated gzip stream"; mode = FAILED; return false; }
        const uint32_t want_crc = t[0] | (t[1] << 8) | (t[2] << 16) | ((uint32_t)t[3] << 24);
        const uint32_t want_len = t[4] | (t[5] << 8) | (t[6] << 16) | ((uint32_t)t[7] << 24);
        if (want_crc != crc) { *err = "invalid gzip data: incorrect data check"; mode = FAILED; return false; }
        if (want_len != (uint32_t)(text_total & 0xFFFFFFFFu)) { *err = "invalid gzip data: incorrect length check"; mode = FAILED; return false; }
        handover_off = (long)(trailer_off + 8);
        mode = TRAILER_DONE;
        return true;
    }

    // zlib from (byte_pos, bit_in_byte) with the text in `window` as dictionary (so that zlib, too, rejects a distance
    // that reaches before the stream's first byte)
    bool start_host(std::string *err)
    {
        memset(&zs, 0, sizeof zs);
        if (inflateInit2(&zs, -15) != Z_OK) { *err = "zlib init failed"; mode = FAILED; return false; }
        zs_open = true;
        if (hist && inflateSetDictionary(&zs, window.data() + (VFB_GZ_WIN - hist), hist) != Z_OK) { *err = "zlib dictionary failed"; mode = FAILED; return false; }
        zin.resize(1 << 20);
        uint64_t off = byte_pos;
        if (bit_in_byte) {
            uint8_t b0;
            if (pread(fd, &b0, 1, (off_t)off) != 1) { *err = "truncated gzip stream"; mode = FAILED; return false; }
            if (inflatePrime(&zs, 8 - (int)bit_in_byte, b0 >> bit_in_byte) != Z_OK) { *err = "zlib prime failed"; mode = FAILED; return false; }
            ++off;
        }
        byte_pos = off;                 // next byte to feed
        zs.avail_in = 0;
        mode = HOST;
        host_since = 0;
        ++host_takeovers;
        if (trace) fprintf(stderr, "[vfb gunzip] zlib takes over at byte %llu\n", (unsigned long long)off);
        return true;
    }

    // zlib carries the stream block by block (Z_BLOCK) and hands it back to the device at a block boundary once it has
    // produced a few megabytes: a chunk the device could not take costs milliseconds, not the rest of the file.
    long long host_read(uint8_t *out, size_t cap, size_t *nl, std::string *err)
    {
        size_t produced = 0;
        while (produced < cap && mode == HOST) {
            if (zs.avail_in == 0) {
                const size_t want = (size_t)std::min<uint64_t>(zin.size(), file_size - byte_pos);
                if (want == 0) { *err = "truncated gzip stream"; mode = FAILED; return -1; }
                if (pread(fd, zin.data(), want, (off_t)byte_pos) != (ssize_t)want) { *err = "read error"; mode = FAILED; return -1; }
                byte_pos += want;
                zs.next_in = zin.data();
                zs.avail_in = (uInt)want;
            }
            zs.next_out = out + produced;
            const size_t room = std::min<size_t>(cap - produced, (size_t)1 << 30);
            zs.avail_out = (uInt)room;
            const int rc = inflate(&zs, Z_BLOCK);
            const size_t n = room - zs.avail_out;
            crc = (uint32_t)crc32(crc, out + produced, (uInt)n);
            text_total += n;
            host_bytes += n;
            host_since += n;
            produced += n;
            if (rc == Z_STREAM_END) {
                const uint64_t tr = byte_pos - zs.avail_in;
                inflateEnd(&zs);
                zs_open = false;
                if (!finish_member(tr, err)) return -1;
                break;
            }
            if (rc != Z_OK && rc != Z_BUF_ERROR) { *err = std::string("invalid gzip data: ") + (zs.msg ? zs.msg : "?"); mode = FAILED; return -1; }
            // at the end of a block that is not the last: back to the device?
            if ((zs.data_type & 128) && !(zs.data_type & 64) && host_since >= host_quota && file_size - (byte_pos - zs.avail_in) > ((uint64_t)1 << 20)) {
                const uint32_t unused = (uint32_t)(zs.data_type & 7);
                uint64_t next = byte_pos - zs.avail_in;          // first byte zlib has not taken
                std::vector<uint8_t> dict(VFB_GZ_WIN);
                uInt dl = 0;
                if (inflateGetDictionary(&zs, dict.data(), &dl) != Z_OK) continue;
                window.assign(VFB_GZ_WIN, 0);
                memcpy(window.data() + (VFB_GZ_WIN - dl), dict.data(), dl);
                hist = dl;
                if (unused) { byte_pos = next - 1; bit_in_byte = 8 - unused; }
                else { byte_pos = next; bit_in_byte = 0; }
                inflateEnd(&zs);
                zs_open = false;
                mode = GPU;
                if (trace) fprintf(stderr, "[vfb gunzip] back to the device at byte %llu bit %u after %llu bytes of text from zlib\n",
                                   (unsigned long long)byte_pos, bit_in_byte, (unsigned long long)host_since);
            }
        }
        if (nl) for (size_t i = 0; i < produced; ++i) *nl += out[i] == '\n';
        return (long long)produced;
    }
    uint64_t host_quota = (uint64_t)8 << 20;
};

GpuGunzip::GpuGunzip() : impl_(nullptr) {}
GpuGunzip::~GpuGunzip() { delete impl_; }

bool GpuGunzip::init(FILE *f, int device, std::string *err)
{
    delete impl_;
    impl_ = new Impl;
    Impl &m = *impl_;
    m.f = f;
    m.fd = fileno(f);
    m.device = device;
    m.trace = getenv("VFB_GUNZIP_TRACE") != nullptr;
    const long pos = ftell(f);
    fseek(f, 0, SEEK_END);
    m.file_size = (uint64_t)ftell(f);
    fseek(f, pos, SEEK_SET);
    if (!m.parse_header(err)) return false;
    if (const char *e = getenv("VFB_GUNZIP_SEGMENT")) m.seg_bytes = std::max<size_t>(4096, (size_t)strtoull(e, nullptr, 10));
    if (const char *e = getenv("VFB_GUNZIP_GAP")) m.min_gap_bits = (uint32_t)std::max<unsigned long long>(64, strtoull(e, nullptr, 10)) * 8u;
    if (const char *e = getenv("VFB_GUNZIP_CAP")) m.cap_syms = (uint32_t)std::max<unsigned long long>(1024, strtoull(e, nullptr, 10));
    if (const char *e = getenv("VFB_GUNZIP_HOST_QUOTA")) m.host_quota = strtoull(e, nullptr, 10);
    if (m.seg_bytes > ((size_t)240 << 20)) m.seg_bytes = (size_t)240 << 20;         // bit positions are 32-bit
    m.ovl_bytes = std::min<size_t>(m.ovl_bytes, std::max<size_t>(m.seg_bytes / 4, 65536));
    m.window.assign(VFB_GZ_WIN, 0);
    if (cudaSetDevice(device) != cudaSuccess || cudaStreamCreateWithFlags(&m.st, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&m.st_out, cudaStreamNonBlocking) != cudaSuccess) {
        cudaGetLastError();
        *err = "no CUDA device for the gzip decoder";
        return false;
    }
    return true;
}

// The producer: segment after segment while the device decoder is in charge.
static void gz_producer(GpuGunzip::Impl *m);

long long GpuGunzip::read_counting(uint8_t *out, size_t cap, size_t *newlines, std::string *err, bool stop_at_segment)
{
    Impl &m = *impl_;
    size_t produced = 0;
    if (newlines) *newlines = 0;
    if (!m.producer.joinable() && !m.producer_done) m.producer = std::thread(gz_producer, impl_);
    while (produced < cap) {
        // the next ready slot, or the end of the device phase
        Impl::Slot *slot = nullptr;
        {
            std::unique_lock<std::mutex> lk(m.mu);
            m.cv.wait(lk, [&] { return m.consumed_seq < m.produced_seq || m.producer_done; });
            if (m.consumed_seq < m.produced_seq) slot = &m.slots[m.consumed_seq % Impl::N_SLOTS];
        }
        if (slot) {
            const size_t n = (size_t)std::min<uint64_t>(cap - produced, slot->text - m.cur_served);
            if (n) {
                if (cudaSetDevice(m.device) != cudaSuccess ||
                    cudaMemcpyAsync(out + produced, slot->d_text.as<uint8_t>() + m.cur_served, n, cudaMemcpyDeviceToHost, m.st_out) != cudaSuccess ||
                    cudaStreamSynchronize(m.st_out) != cudaSuccess) {
                    cudaGetLastError();
                    *err = "CUDA error in the gzip decoder (copy out)";
                    return -1;
                }
                if (newlines) {
                    // whole pieces from the device's counts, the ragged ends by looking
                    const uint64_t lo = m.cur_served, hi = lo + n;
                    const uint64_t p0 = (lo + VFB_GZ_PIECE - 1) / VFB_GZ_PIECE, p1 = hi / VFB_GZ_PIECE;
                    size_t c = 0;
                    if (p0 > p1) { for (size_t i = 0; i < n; ++i) c += out[produced + i] == '\n'; }
                    else {
                        for (uint64_t i = lo; i < p0 * VFB_GZ_PIECE; ++i) c += out[produced + (i - lo)] == '\n';
                        for (uint64_t p = p0; p < p1; ++p) c += slot->nl[(size_t)p];
                        for (uint64_t i = p1 * VFB_GZ_PIECE; i < hi; ++i) c += out[produced + (i - lo)] == '\n';
                    }
                    *newlines += c;
                }
                m.cur_served += n;
                produced += n;
            }
            if (m.cur_served >= slot->text) {
                std::unique_lock<std::mutex> lk(m.mu);
                m.cv.wait(lk, [&] { return slot->outstanding == 0; });      // ranges still being copied out of the slot
                if (m.trace) fprintf(stderr, "[vfb gunzip] reader: segment %llu handed out at %.1f ms\n", (unsigned long long)m.consumed_seq, m.since_init());
                ++m.consumed_seq;
                m.cur_served = 0;
                m.cv.notify_all();
                if (stop_at_segment) return (long long)produced;      // (the next segment starts piece-aligned: peek_device again)
            }
            continue;
        }
        // the producer has finished and everything it made has been handed out
        if (m.producer.joinable()) m.producer.join();
        if (m.mode == Impl::FAILED) { *err = m.producer_err.empty() ? "gzip decoder failed" : m.producer_err; return -1; }
        if (m.mode == Impl::TRAILER_DONE) break;
        if (m.mode == Impl::HOST) {
            const long long got = m.host_read(out + produced, cap - produced, newlines, err);
            if (got < 0) return -1;
            produced += (size_t)got;
            continue;
        }
        if (m.mode == Impl::GPU) {
            // zlib has handed the stream back
            {
                std::lock_guard<std::mutex> lk(m.mu);
                m.producer_done = false;
            }
            m.producer = std::thread(gz_producer, impl_);
            continue;
        }
        *err = "gzip decoder: unexpected state";
        return -1;
    }
    return (long long)produced;
}

static void gz_producer(GpuGunzip::Impl *mp)
{
    GpuGunzip::Impl &m = *mp;
    for (;;) {
        GpuGunzip::Impl::Slot *slot;
        {
            std::unique_lock<std::mutex> lk(m.mu);
            m.cv.wait(lk, [&] { return m.stop || m.produced_seq - m.consumed_seq < (uint64_t)GpuGunzip::Impl::N_SLOTS; });
            if (m.stop) break;
            slot = &m.slots[m.produced_seq % GpuGunzip::Impl::N_SLOTS];
        }
        std::string e;
        const double t_begin = m.since_init();
        const bool ok = m.run_segment(*slot, &e);
        if (m.trace) fprintf(stderr, "[vfb gunzip] producer: segment ran %.1f .. %.1f ms\n", t_begin, m.since_init());
        std::lock_guard<std::mutex> lk(m.mu);
        if (!ok) { m.mode = GpuGunzip::Impl::FAILED; m.producer_err = e; break; }
        if (slot->text) ++m.produced_seq;
        m.cv.notify_all();
        if (m.mode != GpuGunzip::Impl::GPU) break;
    }
    std::lock_guard<std::mutex> lk(m.mu);
    m.producer_done = true;
    m.cv.notify_all();
}

bool GpuGunzip::peek_device(size_t max_len, size_t keep_tail, DeviceRange *out)
{
    Impl &m = *impl_;
    if (!m.producer.joinable() && !m.producer_done) m.producer = std::thread(gz_producer, impl_);
    Impl::Slot *slot = nullptr;
    {
        std::unique_lock<std::mutex> lk(m.mu);
        m.cv.wait(lk, [&] { return m.consumed_seq < m.produced_seq || m.producer_done; });
        if (m.consumed_seq < m.produced_seq) slot = &m.slots[m.consumed_seq % Impl::N_SLOTS];
    }
    if (!slot) return false;
    if (m.cur_served % VFB_GZ_PIECE) return false;                   // (only after a read_counting inside the segment)
    const uint64_t left = slot->text - m.cur_served;
    if (left <= keep_tail + VFB_GZ_PIECE) return false;
    uint64_t n = std::min<uint64_t>(max_len, left - keep_tail);
    n -= n % VFB_GZ_PIECE;
    if (n == 0) return false;
    size_t nl = 0;
    for (uint64_t p = m.cur_served / VFB_GZ_PIECE; p < (m.cur_served + n) / VFB_GZ_PIECE; ++p) nl += slot->nl[(size_t)p];
    out->d_ptr = slot->d_text.as<uint8_t>() + m.cur_served;
    out->len = (size_t)n;
    out->newlines = nl;
    out->device = m.device;
    out->seq = m.consumed_seq;
    return true;
}

bool GpuGunzip::range_tail(const DeviceRange &r, uint8_t *out_host, size_t n, std::string *err)
{
    Impl &m = *impl_;
    if (n > r.len) n = r.len;
    if (cudaSetDevice(m.device) != cudaSuccess ||
        cudaMemcpyAsync(out_host, r.d_ptr + (r.len - n), n, cudaMemcpyDeviceToHost, m.st_out) != cudaSuccess ||
        cudaStreamSynchronize(m.st_out) != cudaSuccess) {
        cudaGetLastError();
        *err = "CUDA error in the gzip decoder (copy out)";
        return false;
    }
    return true;
}

void GpuGunzip::commit_device(const DeviceRange &r)
{
    Impl &m = *impl_;
    std::lock_guard<std::mutex> lk(m.mu);
    Impl::Slot &slot = m.slots[r.seq % Impl::N_SLOTS];
    m.cur_served += r.len;
    ++slot.outstanding;
}

void GpuGunzip::release_device(const DeviceRange &r)
{
    Impl &m = *impl_;
    std::lock_guard<std::mutex> lk(m.mu);
    Impl::Slot &slot = m.slots[r.seq % Impl::N_SLOTS];
    if (slot.outstanding) --slot.outstanding;
    m.cv.notify_all();
}

bool GpuGunzip::member_ended() const
{
    if (!impl_) return true;
    std::lock_guard<std::mutex> lk(impl_->mu);
    return impl_->mode == Impl::TRAILER_DONE && impl_->producer_done && impl_->consumed_seq >= impl_->produced_seq;
}

bool GpuGunzip::handover(long *file_off) const
{
    if (!impl_ || impl_->mode != Impl::TRAILER_DONE) return false;
    *file_off = impl_->handover_off;
    return true;
}

void GpuGunzip::stats(uint64_t *segments, uint64_t *chunks, uint64_t *visited, uint64_t *host_bytes) const
{
    if (segments) *segments = impl_ ? impl_->n_segments : 0;
    if (chunks) *chunks = impl_ ? impl_->n_chunks_total : 0;
    if (visited) *visited = impl_ ? impl_->n_live_total : 0;
    if (host_bytes) *host_bytes = impl_ ? impl_->host_bytes : 0;
}

}  // namespace vfb
