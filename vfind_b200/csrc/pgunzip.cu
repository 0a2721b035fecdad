// Parallel decoding of ONE gzip stream on the host threads (ingest of plain `gzip` / `fastp` output).
//
// Replaces the single zlib stream behind `MultiGzDecoder` (/root/reference/src/lib.rs:233) for input
// that is not block-gzip: a deflate stream has no index, so a worker that starts in the middle has
// to (1) FIND a block start and (2) decode without knowing the 32 KiB of text before it.
//   find    from a byte boundary, every bit offset is tried as the start of a non-final dynamic
//           block: header fields in range, complete code-length code, valid run-length stream,
//           complete literal/length and distance codes, then the whole block must decode and be
//           followed by a legal block type.  Random bits pass with negligible probability, and a
//           false start cannot survive the chain check below.
//   decode  to 16-bit symbols: values < 256 are bytes, 256 + p stands for "byte p of the unknown
//           32 KiB window before my first output".  Matches copy symbols, so unknown bytes
//           propagate as markers.  A worker stops when a block starts exactly at a later worker's
//           start; workers nobody lands on are dropped (false starts, or starts inside a stored /
//           fixed block), so the surviving chain is exactly the serial decode.
//   resolve the window is carried from worker to worker (32 KiB each, serial, cheap), then all
//           workers translate their symbols to bytes in parallel and CRC-32 them; the per-member
//           CRC-32 / ISIZE trailer is checked as flate2 does (crc32_combine over the pieces).
// Member ends, stored and fixed blocks, multi-member streams and truncated input follow the
// serial decoder's behaviour; VFB_PGUNZIP=0 keeps the zlib stream.
#include <zlib.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "pgunzip.h"

namespace vfb {
namespace {

constexpr int MAXBITS = 15, MAXL = 288, MAXD = 30;
constexpr int LBITS = 11, DBITS = 9;
constexpr uint32_t WSIZE = 32768;

const uint16_t LBASE[29] = {3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258};
const uint8_t LEXT[29] = {0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0};
const uint16_t DBASE[30] = {1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097, 6145, 8193, 12289, 16385, 24577};
const uint8_t DEXT[30] = {0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13};
const uint8_t ORDER[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};

// Bit reader over a buffer that is padded with >= 16 readable bytes behind `nbits`.
struct Bits {
    const uint8_t *p;
    uint64_t nbits;      // valid bits in the buffer
    uint64_t pos;        // next bit
    uint64_t buf = 0;
    int cnt = 0;
    uint64_t loaded = 0;     // bit position up to which the buffer has been loaded
    void seek(uint64_t bit)
    {
        pos = bit;
        loaded = bit & ~7ull;
        buf = 0;
        cnt = 0;
        refill();
        const int skip = (int)(bit & 7u);
        buf >>= skip;
        cnt -= skip;
    }
    inline void refill()
    {
        // top up to >= 56 bits with whole bytes
        uint64_t w;
        memcpy(&w, p + (loaded >> 3), 8);
        buf |= w << cnt;
        const int take = (63 - cnt) >> 3;
        loaded += (uint64_t)take * 8;
        cnt += take * 8;
    }
    inline uint32_t peek(int n) const { return (uint32_t)buf & ((1u << n) - 1u); }
    inline void drop(int n) { buf >>= n; cnt -= n; pos += (uint64_t)n; }
    inline uint32_t get(int n)
    {
        if (cnt < n) refill();
        const uint32_t v = peek(n);
        drop(n);
        return v;
    }
    inline bool past_end() const { return pos > nbits; }
};

struct Huff {
    uint16_t count[MAXBITS + 1];
    uint16_t symbol[MAXL];
};

// <0 over-subscribed, >0 incomplete, 0 complete
int construct(Huff &h, const uint8_t *length, int n)
{
    uint16_t offs[MAXBITS + 1];
    for (int l = 0; l <= MAXBITS; ++l) h.count[l] = 0;
    for (int s = 0; s < n; ++s) h.count[length[s]]++;
    if (h.count[0] == n) return 0;
    int left = 1;
    for (int l = 1; l <= MAXBITS; ++l) {
        left <<= 1;
        left -= h.count[l];
        if (left < 0) return left;
    }
    offs[1] = 0;
    for (int l = 1; l < MAXBITS; ++l) offs[l + 1] = offs[l] + h.count[l];
    for (int s = 0; s < n; ++s)
        if (length[s]) h.symbol[offs[length[s]]++] = (uint16_t)s;
    return left;
}

inline int slow_decode(uint32_t bits, const Huff &h, int maxlen, int *len_out)
{
    int code = 0, first = 0, index = 0;
    for (int len = 1; len <= maxlen; ++len) {
        code |= (int)(bits & 1u);
        bits >>= 1;
        const int c = h.count[len];
        if (code - c < first) {
            *len_out = len;
            return h.symbol[index + (code - first)];
        }
        index += c;
        first += c;
        first <<= 1;
        code <<= 1;
    }
    return -1;
}

// table entries: nbits | kind << 4 | value << 8 | extra << 24 ; kind 0 literal, 1 length, 2 end of block, 3 invalid
inline uint32_t lit_entry(int sym, int nbits)
{
    if (sym < 256) return (uint32_t)nbits | ((uint32_t)sym << 8);
    if (sym == 256) return (uint32_t)nbits | (2u << 4);
    if (sym > 285) return (uint32_t)nbits | (3u << 4);
    return (uint32_t)nbits | (1u << 4) | ((uint32_t)LBASE[sym - 257] << 8) | ((uint32_t)LEXT[sym - 257] << 24);
}
inline uint32_t dist_entry(int sym, int nbits)
{
    if (sym > 29) return (uint32_t)nbits | (15u << 4);
    return (uint32_t)nbits | ((uint32_t)DEXT[sym] << 4) | ((uint32_t)DBASE[sym] << 8);
}

struct Tables {
    Huff lh, dh;
    uint32_t ltab[1 << LBITS], dtab[1 << DBITS];
    void build()
    {
        // fill by enumerating the codes: a code of length l <= LBITS owns 2^(LBITS-l) entries
        memset(ltab, 0, sizeof ltab);
        memset(dtab, 0, sizeof dtab);
        fill(lh, ltab, LBITS, true);
        fill(dh, dtab, DBITS, false);
    }
    static void fill(const Huff &h, uint32_t *tab, int tbits, bool lit)
    {
        int code = 0, index = 0;
        for (int len = 1; len <= tbits; ++len) {
            for (int k = 0; k < h.count[len]; ++k, ++code, ++index) {
                // canonical code `code` of `len` bits, MSB first in the stream -> reverse for the LSB-first peek
                uint32_t r = 0;
                for (int b = 0; b < len; ++b) r |= ((uint32_t)(code >> b) & 1u) << (len - 1 - b);
                const uint32_t e = lit ? lit_entry(h.symbol[index], len) : dist_entry(h.symbol[index], len);
                for (uint32_t x = r; x < (1u << tbits); x += 1u << len) tab[x] = e;
            }
            code <<= 1;
        }
    }
};

// Reads a dynamic block header (after the 3 header bits).  strict = candidate search (every defect rejects).
bool read_dynamic(Bits &b, Tables &T)
{
    const int nlen = (int)b.get(5) + 257, ndist = (int)b.get(5) + 1, ncode = (int)b.get(4) + 4;
    if (nlen > 286 || ndist > 30) return false;
    uint8_t lens[MAXL + MAXD + 2];
    uint8_t cl[19];
    memset(cl, 0, sizeof cl);
    for (int i = 0; i < ncode; ++i) cl[ORDER[i]] = (uint8_t)b.get(3);
    Huff ch;
    if (construct(ch, cl, 19) != 0) return false;
    int idx = 0;
    while (idx < nlen + ndist) {
        if (b.cnt < 16) b.refill();
        int l = 0;
        const int sym = slow_decode((uint32_t)b.buf, ch, 7, &l);
        if (sym < 0) return false;
        b.drop(l);
        if (sym < 16) {
            lens[idx++] = (uint8_t)sym;
        } else {
            int len = 0, rep;
            if (sym == 16) {
                if (idx == 0) return false;
                len = lens[idx - 1];
                rep = 3 + (int)b.get(2);
            } else if (sym == 17) rep = 3 + (int)b.get(3);
            else rep = 11 + (int)b.get(7);
            if (idx + rep > nlen + ndist) return false;
            while (rep--) lens[idx++] = (uint8_t)len;
        }
        if (b.past_end()) return false;
    }
    if (lens[256] == 0) return false;
    // an incomplete code is accepted only as a single code of length 1 (zlib's inflate_table)
    int e = construct(T.lh, lens, nlen);
    if (e < 0 || (e > 0 && !(nlen - T.lh.count[0] == 1 && T.lh.count[1] == 1))) return false;
    e = construct(T.dh, lens + nlen, ndist);
    if (e < 0 || (e > 0 && !(ndist - T.dh.count[0] == 1 && T.dh.count[1] == 1))) return false;
    T.build();
    return true;
}

void fixed_tables(Tables &T)
{
    uint8_t lens[MAXL + MAXD];
    int s = 0;
    for (; s < 144; ++s) lens[s] = 8;
    for (; s < 256; ++s) lens[s] = 9;
    for (; s < 280; ++s) lens[s] = 7;
    for (; s < 288; ++s) lens[s] = 8;
    construct(T.lh, lens, 288);
    for (s = 0; s < 30; ++s) lens[s] = 5;
    construct(T.dh, lens, 30);
    T.build();
}

// Symbols of one Huffman block until its end-of-block.  out == nullptr: validate only (candidate search).
// `avail` = symbols of known history in front of out[0] for this worker (0 = none: everything before is
// the unknown window).  Returns 0 ok, -1 invalid data, -2 input exhausted.
struct OutBuf {
    uint16_t *p = nullptr;
    size_t cap = 0, n = 0;
    OutBuf() = default;
    OutBuf(const OutBuf &) = delete;
    OutBuf &operator=(const OutBuf &) = delete;
    ~OutBuf() { free(p); }
    void reserve(size_t want)
    {
        if (want <= cap) return;
        size_t ncap = std::max(cap * 2, want);
        uint16_t *np = static_cast<uint16_t *>(realloc(p, ncap * sizeof(uint16_t)));
        if (!np) abort();
        p = np;
        cap = ncap;
    }
    inline void need(size_t more)
    {
        if (n + more > cap) reserve(n + more + (1u << 16));
    }
};

template <bool WRITE>
int huffman_block_t(Bits &bb, const Tables &T, OutBuf *out, uint64_t *n_virtual, uint64_t member_out)
{
    // member_out: bytes this member has produced before this worker's first output, or UINT64_MAX when
    // unknown (a worker that started mid-stream) — then a distance may reach up to 32 KiB back into the
    // unknown window.  The bit reader and the output cursor live in locals for the duration of the block.
    Bits b = bb;
    uint16_t *base = WRITE ? out->p : nullptr;
    size_t n = WRITE ? out->n : 0, cap = WRITE ? out->cap : 0;
    uint64_t nv = *n_virtual;
    int rc;
    for (;;) {
        if (b.cnt < 48) {
            b.refill();
            if (b.past_end()) { rc = -2; break; }
        }
        uint32_t e = T.ltab[b.peek(LBITS)];
        if (e == 0) {
            int l = 0;
            const int sym = slow_decode((uint32_t)b.buf, T.lh, MAXBITS, &l);
            if (sym < 0) { rc = -1; break; }
            e = lit_entry(sym, l);
        }
        b.drop((int)(e & 15u));
        const uint32_t kind = (e >> 4) & 3u;
        if (kind == 0) {
            if (WRITE) {
                if (n + 1 > cap) { out->n = n; out->need(1); base = out->p; cap = out->cap; }
                base[n++] = (uint16_t)(e >> 8);
            }
            ++nv;
            continue;
        }
        if (kind == 2) { rc = b.past_end() ? -2 : 0; break; }
        if (kind == 3) { rc = -1; break; }
        const int xb = (int)(e >> 24);
        const uint32_t len = ((e >> 8) & 0xFFFFu) + b.peek(xb);
        b.drop(xb);
        if (b.cnt < 32) b.refill();
        uint32_t d = T.dtab[b.peek(DBITS)];
        if (d == 0) {
            int l = 0;
            const int ds = slow_decode((uint32_t)b.buf, T.dh, MAXBITS, &l);
            if (ds < 0) { rc = -1; break; }
            d = dist_entry(ds, l);
        }
        const int dx = (int)((d >> 4) & 15u);
        if (dx == 15) { rc = -1; break; }
        b.drop((int)(d & 15u));
        const uint32_t dist = (d >> 8) + b.peek(dx);
        b.drop(dx);
        if (dist > nv) {
            const uint64_t back = dist - nv;           // how far before this worker's first output
            if (back > WSIZE || (member_out != UINT64_MAX && back > member_out)) {
                rc = b.past_end() ? -2 : -1;
                break;
            }
        }
        if (WRITE) {
            if (n + len + 16 > cap) { out->n = n; out->need(len + 16); base = out->p; cap = out->cap; }
            uint16_t *o = base + n;
            if (dist <= n) {
                const uint16_t *f = o - dist;
                if (dist >= 16) {
                    // fixed 16-symbol pieces (two vector moves each, no call): a piece never overlaps its own source,
                    // pieces are written in order, and the up to 15 symbols written past the match are overwritten by
                    // what follows (the buffer keeps 16 symbols of slack).  Most matches in read text are a few bases.
                    uint32_t done = 0;
                    do { memcpy(o + done, f + done, 32); done += 16; } while (done < len);
                } else if (dist >= len) memcpy(o, f, (size_t)len * 2);
                else for (uint32_t i = 0; i < len; ++i) o[i] = f[i];
            } else {
                for (uint32_t i = 0; i < len; ++i) {
                    const int64_t src = (int64_t)(n + i) - (int64_t)dist;
                    o[i] = src >= 0 ? base[src] : (uint16_t)(256 + (int64_t)WSIZE + src);
                }
            }
            n += len;
        }
        nv += len;
    }
    if (WRITE) out->n = n;
    *n_virtual = nv;
    bb = b;
    return rc;
}

int huffman_block(Bits &b, const Tables &T, OutBuf *out, uint64_t *n_virtual, uint64_t member_out)
{
    return out ? huffman_block_t<true>(b, T, out, n_virtual, member_out) : huffman_block_t<false>(b, T, nullptr, n_virtual, member_out);
}

// A non-final dynamic block at bit `q` that decodes completely and is followed by a legal block type.
bool plausible_block_start(const uint8_t *z, uint64_t nbits, uint64_t q, Tables &T)
{
    Bits b{z, nbits, 0};
    b.seek(q);
    const uint32_t hdr = b.get(3);
    if (hdr != 4u) return false;                 // BFINAL = 0, BTYPE = 2 (bits: 0, then 0 1)
    {
        // cheap screen before the full header: field ranges and the Kraft sum of the code-length code
        const uint32_t f = b.peek(14);
        const int nlen = (int)(f & 31u) + 257, ndist = (int)((f >> 5) & 31u) + 1, ncode = (int)((f >> 10) & 15u) + 4;
        if (nlen > 286 || ndist > 30) return false;
        Bits c = b;
        c.drop(14);
        int kraft = 0;
        for (int i = 0; i < ncode; ++i) {
            const uint32_t l = c.get(3);
            if (l) kraft += 128 >> l;
        }
        if (kraft != 128) return false;
    }
    if (!read_dynamic(b, T)) return false;
    uint64_t nv = 0;
    if (huffman_block(b, T, nullptr, &nv, UINT64_MAX) != 0) return false;
    if (b.cnt < 3) b.refill();
    if (b.past_end()) return false;
    return ((b.peek(3) >> 1) & 3u) != 3u;
}

struct MemberEnd {
    uint64_t out_pos;        // symbols of this worker produced when the member ended
    uint32_t crc, isize;
};

struct Worker {
    uint64_t start_bit = 0;
    bool found = false;
    size_t out_hint = 0;     // symbols to reserve up front
    bool at_header = false;  // starts at a gzip member header (worker 0 only)
    OutBuf *outp = nullptr;  // symbol buffer, kept across segments (no fresh pages to fault in)
    uint64_t end_bit = 0;    // first bit not consumed (a block start, or the byte after a member trailer)
    int landed = -1;         // index of the worker whose start this one reached
    bool hit_member_end = false, hit_eof = false, exhausted = false;
    MemberEnd mend{};
    int error = 0;           // 1 = invalid data
    std::string msg;
    uint64_t out_off = 0;    // offset of the resolved bytes in the segment text
    uint32_t crc = 0;
};

// gzip member header at byte offset `p`; returns the deflate start byte or 0 when incomplete / -1 invalid
long long parse_gzip_header(const uint8_t *z, size_t zlen, size_t p)
{
    if (p + 10 > zlen) return 0;
    if (z[p] != 0x1f || z[p + 1] != 0x8b) return -1;
    if (z[p + 2] != 8) return -1;
    const uint32_t flg = z[p + 3];
    if (flg & 0xE0) return -1;
    size_t q = p + 10;
    if (flg & 4) {
        if (q + 2 > zlen) return 0;
        q += 2 + (size_t)(z[q] | (z[q + 1] << 8));
        if (q > zlen) return 0;
    }
    if (flg & 8) { while (q < zlen && z[q]) ++q; if (q >= zlen) return 0; ++q; }
    if (flg & 16) { while (q < zlen && z[q]) ++q; if (q >= zlen) return 0; ++q; }
    if (flg & 2) { q += 2; if (q > zlen) return 0; }
    return (long long)q;
}

}  // namespace

struct ParallelGunzip::Impl {
    FILE *f = nullptr;
    int threads = 1;
    bool eof = false;                 // no more compressed bytes in the file
    bool finished = false;            // clean end of the stream reached
    std::vector<uint8_t> z;           // compressed bytes not yet consumed (+ padding)
    size_t zlen = 0;
    uint64_t start_bit = 0;           // where the next segment starts in z
    bool in_member = false;           // start_bit is a block start inside a member (else: a member header / end of input)
    std::vector<uint8_t> window;      // last <= 32 KiB of text of the current member
    uint64_t member_out = 0;          // bytes the current member has produced
    uint32_t member_crc = 0;
    uint8_t *text = nullptr;          // text of the segment being decoded (malloc'd, never zero-filled)
    size_t text_cap = 0, text_len = 0, text_pos = 0;
    // the segment being handed out by read(), while the next one is decoded in the background
    uint8_t *cur = nullptr;
    size_t cur_cap = 0, cur_len = 0, cur_pos = 0;
    std::thread bg;
    bool bg_running = false, bg_ok = true, drained = false;
    size_t seg_bytes = (size_t)24 << 20;
    std::vector<OutBuf *> bufs;       // one symbol buffer per worker slot
    double ratio = 0;                 // text bytes per compressed byte, last segment
    bool serial_mode = false;         // many small members: decode them one by one without the block search
    std::string err;
    uint64_t n_segments = 0, n_workers_used = 0, n_workers_dropped = 0;
    double t_fill = 0, t_find = 0, t_decode = 0, t_window = 0, t_resolve = 0;

    bool fill()
    {
        // keep the unconsumed tail, append up to seg_bytes more
        const size_t keep_from = (size_t)(start_bit >> 3);
        if (keep_from) {
            memmove(z.data(), z.data() + keep_from, zlen - keep_from);
            zlen -= keep_from;
            start_bit &= 7u;
        }
        const size_t want = seg_bytes;
        z.resize(zlen + want + 64);
        while (!eof && zlen < want) {
            const size_t got = fread(z.data() + zlen, 1, want - zlen, f);
            if (got == 0) { eof = true; break; }
            zlen += got;
        }
        memset(z.data() + zlen, 0, 64);
        return true;
    }

    void decode_worker(Worker &w, const std::vector<Worker> &all, int self);
    bool segment();
};

void ParallelGunzip::Impl::decode_worker(Worker &w, const std::vector<Worker> &all, int self)
{
    const uint64_t nbits = (uint64_t)zlen * 8;
    Bits b{z.data(), nbits, 0};
    Tables *T = new Tables;
    uint64_t member_known = self == 0 ? member_out : UINT64_MAX;
    uint64_t nv = 0;
    uint64_t pos = w.start_bit;
    bool need_header = w.at_header;
    w.outp->reserve(w.out_hint ? w.out_hint : ((size_t)1 << 20));
    for (;;) {
        if (need_header) {
            const size_t byte = (size_t)((pos + 7) >> 3);
            if (byte >= zlen && eof) { w.hit_eof = true; w.end_bit = (uint64_t)byte * 8; break; }
            const long long ds = parse_gzip_header(z.data(), zlen, byte);
            if (ds < 0) { w.error = 1; w.msg = "invalid gzip header"; break; }
            if (ds == 0) {
                if (eof) { w.error = 1; w.msg = "truncated gzip stream"; }
                else { w.exhausted = true; w.end_bit = (uint64_t)byte * 8; }
                break;
            }
            pos = (uint64_t)ds * 8;
            need_header = false;
            member_known = 0;
            // a new member: this worker's earlier output is not reachable any more
            // (handled by stopping at the member end, see below)
        }
        // a block starts at `pos`: is it somebody's start?
        if (pos != w.start_bit || nv) {
            int hit = -1;
            for (size_t k = (size_t)self + 1; k < all.size(); ++k)
                if (all[k].found && all[k].start_bit == pos) { hit = (int)k; break; }
            if (hit >= 0) { w.landed = hit; w.end_bit = pos; break; }
        }
        const uint64_t block_start = pos;
        const size_t n_at_block = w.outp->n;
        const uint64_t nv_at_block = nv;
        b.seek(pos);
        const uint32_t last = b.get(1), type = b.get(2);
        int rc = 0;
        if (b.past_end()) rc = -2;
        else if (type == 0) {
            const int drop = b.cnt & 7;
            b.drop(drop);
            const uint32_t len = b.get(16), nlen = b.get(16);
            if (b.past_end()) rc = -2;
            else if ((len ^ 0xFFFFu) != nlen) rc = -1;
            else {
                const uint64_t src = b.pos >> 3;
                if (src + len > zlen) rc = -2;
                else {
                    w.outp->need(len);
                    for (uint32_t i = 0; i < len; ++i) w.outp->p[w.outp->n++] = z[src + i];
                    nv += len;
                    b.seek((src + len) * 8);
                }
            }
        } else if (type == 1) {
            fixed_tables(*T);
            rc = huffman_block(b, *T, w.outp, &nv, member_known);
        } else if (type == 2) {
            if (!read_dynamic(b, *T)) rc = b.past_end() ? -2 : -1;
            else rc = huffman_block(b, *T, w.outp, &nv, member_known);
        } else rc = -1;
        if (rc != 0 && b.past_end()) rc = -2;          // whatever went wrong, it went wrong in the padding
        if (rc == -2 || (rc == 0 && b.past_end())) {
            // ran out of input inside this block: give it back
            w.outp->n = n_at_block;
            nv = nv_at_block;
            if (eof) { w.error = 1; w.msg = "truncated gzip stream"; }
            else { w.exhausted = true; w.end_bit = block_start; }
            break;
        }
        if (rc != 0) { w.error = 1; w.msg = "invalid gzip data: corrupt deflate stream"; break; }
        pos = b.pos;
        if (last) {
            // member trailer at the next byte boundary
            const size_t t = (size_t)((pos + 7) >> 3);
            if (t + 8 > zlen) {
                if (eof) { w.error = 1; w.msg = "truncated gzip stream"; break; }
                w.outp->n = n_at_block;
                w.exhausted = true;
                w.end_bit = block_start;
                break;
            }
            const uint8_t *tr = z.data() + t;
            w.mend.out_pos = w.outp->n;
            w.mend.crc = tr[0] | (tr[1] << 8) | (tr[2] << 16) | ((uint32_t)tr[3] << 24);
            w.mend.isize = tr[4] | (tr[5] << 8) | (tr[6] << 16) | ((uint32_t)tr[7] << 24);
            w.hit_member_end = true;
            w.end_bit = (uint64_t)(t + 8) * 8;
            break;
        }
    }
    delete T;
}

bool ParallelGunzip::Impl::segment()
{
    text_len = 0;
    text_pos = 0;
    if (finished) return true;
    auto now = [] { return std::chrono::steady_clock::now(); };
    auto secs = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) { return std::chrono::duration<double>(b - a).count(); };
    auto t0 = now();
    fill();
    auto t1 = now();
    t_fill += secs(t0, t1);
    const uint64_t nbits = (uint64_t)zlen * 8;
    if (!in_member) {
        // between members: a clean end, or the next header
        const size_t byte = (size_t)((start_bit + 7) >> 3);
        if (byte >= zlen && eof) { finished = true; return true; }
    }
    ++n_segments;
    // ---- phase 1: starts
    const int T = serial_mode ? 1 : std::max(1, threads);
    std::vector<Worker> ws((size_t)T);
    while (bufs.size() < (size_t)T) bufs.push_back(new OutBuf);
    for (int t = 0; t < T; ++t) { ws[(size_t)t].outp = bufs[(size_t)t]; bufs[(size_t)t]->n = 0; }
    ws[0].start_bit = start_bit;
    ws[0].found = true;
    ws[0].at_header = !in_member;
    const size_t first_byte = (size_t)(start_bit >> 3);
    const size_t span = zlen > first_byte ? zlen - first_byte : 0;
    {
        std::vector<std::thread> pool;
        auto find = [&](int t) {
            const size_t lo = first_byte + span * (size_t)t / (size_t)T;
            const size_t hi = first_byte + span * (size_t)(t + 1) / (size_t)T;
            Tables *tab = new Tables;
            for (uint64_t q = (uint64_t)lo * 8; q < (uint64_t)hi * 8 && q + 64 < nbits; ++q) {
                // two cheap bits first: BFINAL = 0 and BTYPE = 2
                const uint32_t three = (uint32_t)(z[q >> 3] | (z[(q >> 3) + 1] << 8)) >> (q & 7u) & 7u;
                if (three != 4u) continue;
                if (plausible_block_start(z.data(), nbits, q, *tab)) { ws[(size_t)t].start_bit = q; ws[(size_t)t].found = true; break; }
            }
            delete tab;
        };
        for (int t = 2; t < T; ++t) pool.emplace_back(find, t);
        if (T > 1) find(1);
        for (auto &th : pool) th.join();
    }
    auto t2 = now();
    t_find += secs(t1, t2);
    // ---- phase 2: decode
    {
        const size_t hint = (size_t)((double)(span / (size_t)T) * (ratio > 1.0 ? ratio : 6.0) * 1.15) + (1u << 16);
        for (auto &w : ws) w.out_hint = hint;
        std::vector<std::thread> pool;
        auto run = [&](int t) { if (ws[(size_t)t].found) decode_worker(ws[(size_t)t], ws, t); };
        for (int t = 1; t < T; ++t) pool.emplace_back(run, t);
        run(0);
        for (auto &th : pool) th.join();
    }
    auto t3 = now();
    t_decode += secs(t2, t3);
    // ---- the chain
    std::vector<int> chain;
    for (int k = 0; k >= 0; k = ws[(size_t)k].landed) {
        chain.push_back(k);
        if (ws[(size_t)k].error) { err = ws[(size_t)k].msg; return false; }
    }
    n_workers_used += chain.size();
    n_workers_dropped += (uint64_t)T - chain.size();
    Worker &tail = ws[(size_t)chain.back()];
    if (tail.exhausted && chain.size() == 1 && tail.outp->n == 0 && !tail.hit_member_end) {
        // not even one block fits: read more next time
        if (eof) { err = "truncated gzip stream"; return false; }
        seg_bytes *= 2;
        return segment();
    }
    // ---- phase 3: windows (serial), then bytes + CRC (parallel)
    uint64_t total = 0;
    for (int k : chain) { ws[(size_t)k].out_off = total; total += ws[(size_t)k].outp->n; }
    if (total > text_cap) {
        free(text);
        text_cap = total + total / 8 + 4096;
        text = static_cast<uint8_t *>(malloc(text_cap));
        if (!text) { err = "out of memory"; return false; }
    }
    text_len = total;
    std::vector<std::vector<uint8_t>> wins(chain.size());
    {
        std::vector<uint8_t> cur(WSIZE, 0);
        uint64_t avail = std::min<uint64_t>(member_out, WSIZE);
        if (!window.empty()) memcpy(cur.data() + WSIZE - window.size(), window.data(), window.size());
        for (size_t c = 0; c < chain.size(); ++c) {
            Worker &w = ws[(size_t)chain[c]];
            wins[c] = cur;
            // resolve the last 32 KiB of this worker to get the next window
            const size_t n = w.outp->n, take = std::min<size_t>(n, WSIZE);
            std::vector<uint8_t> nxt(WSIZE, 0);
            if (take < WSIZE) memcpy(nxt.data(), cur.data() + take, WSIZE - take);
            for (size_t i = 0; i < take; ++i) {
                const uint16_t s = w.outp->p[n - take + i];
                if (s >= 256) {
                    const uint32_t p = s - 256u;
                    if ((uint64_t)(WSIZE - p) > avail) { err = "invalid gzip data: distance too far back"; return false; }
                    nxt[WSIZE - take + i] = cur[p];
                } else nxt[WSIZE - take + i] = (uint8_t)s;
            }
            cur.swap(nxt);
            avail = std::min<uint64_t>(avail + n, WSIZE);
        }
        window.assign(cur.end() - (ptrdiff_t)avail, cur.end());
    }
    auto t4 = now();
    t_window += secs(t3, t4);
    std::atomic<bool> bad{false};
    {
        std::vector<std::thread> pool;
        const uint64_t avail0 = std::min<uint64_t>(member_out, WSIZE);
        auto resolve = [&](size_t c) {
            Worker &w = ws[(size_t)chain[c]];
            const uint8_t *win = wins[c].data();
            uint8_t *dst = text + w.out_off;
            const uint16_t *src = w.outp->p;
            // history available in front of this worker (for the range check of its markers)
            const uint64_t avail = std::min<uint64_t>(avail0 + w.out_off, WSIZE);
            // cache-sized pieces: narrow 64 symbols at a time (vectorises; a block that held a marker is gone
            // over again symbol by symbol), then CRC the piece while it is still in cache
            const size_t n = w.outp->n;
            // In read text markers do not die out (a quality line copied from the previous record's keeps them
            // alive for the whole stream), so most blocks take the second pass: it goes through one table --
            // symbol -> byte, literals and the 32 KiB window behind each other -- without a branch per symbol;
            // a marker that points in front of the member's first byte is caught by one compare (none can once
            // the member has produced a full window).
            std::vector<uint8_t> lut(256 + WSIZE);
            for (int b = 0; b < 256; ++b) lut[(size_t)b] = (uint8_t)b;
            memcpy(lut.data() + 256, win, WSIZE);
            const uint8_t *tab = lut.data();
            const uint16_t n_invalid = (uint16_t)(WSIZE - avail);       // markers 256 .. 256 + n_invalid - 1 are out of range
            uLong c32 = crc32(0L, Z_NULL, 0);
            for (size_t p0 = 0; p0 < n; p0 += (size_t)1 << 16) {
                const size_t p1 = std::min(n, p0 + ((size_t)1 << 16));
                size_t i = p0;
                bool markers = true;            // the previous block held one: skip the narrowing attempt
                for (; i + 64 <= p1; i += 64) {
                    if (!markers) {
                        uint16_t any = 0;
                        for (int k = 0; k < 64; ++k) { any |= src[i + k]; dst[i + k] = (uint8_t)src[i + k]; }
                        if (any < 256) continue;
                    }
                    uint16_t inval = 0, any = 0;
                    if (n_invalid) {
                        for (int k = 0; k < 64; ++k) {
                            const uint16_t s = src[i + k];
                            dst[i + k] = tab[s];
                            any |= s;
                            inval |= (uint16_t)((uint16_t)(s - 256u) < n_invalid);
                        }
                    } else {
                        for (int k = 0; k < 64; ++k) {
                            const uint16_t s = src[i + k];
                            dst[i + k] = tab[s];
                            any |= s;
                        }
                    }
                    if (inval) { bad = true; return; }
                    markers = any >= 256;
                }
                for (; i < p1; ++i) {
                    const uint16_t s = src[i];
                    if ((uint16_t)(s - 256u) < n_invalid) { bad = true; return; }
                    dst[i] = tab[s];
                }
                c32 = crc32(c32, dst + p0, (uInt)(p1 - p0));
            }
            w.crc = (uint32_t)c32;
        };
        for (size_t c = 1; c < chain.size(); ++c) pool.emplace_back(resolve, c);
        resolve(0);
        for (auto &th : pool) th.join();
    }
    t_resolve += secs(t4, now());
    if (getenv("VFB_PGUNZIP_TRACE")) fprintf(stderr, "[pgunzip] segment %llu: chain %zu of %d workers, %llu bytes; cumulative fill %.3f find %.3f decode %.3f window %.3f resolve %.3f s\n", (unsigned long long)n_segments, chain.size(), T, (unsigned long long)total, t_fill, t_find, t_decode, t_window, t_resolve);
    if (bad.load()) { err = "invalid gzip data: distance too far back"; return false; }
    // ---- member bookkeeping
    for (int k : chain) {
        Worker &w = ws[(size_t)k];
        member_crc = (uint32_t)crc32_combine(member_crc, w.crc, (z_off_t)w.outp->n);
        member_out += w.outp->n;
    }
    if (tail.end_bit > start_bit) ratio = (double)total / ((double)(tail.end_bit - start_bit) / 8.0);
    start_bit = tail.end_bit;
    in_member = true;
    // a stream of small members gains nothing from the block search (everything behind the first
    // member end is thrown away): decode those serially until a segment is worth splitting again
    serial_mode = tail.hit_member_end ? total < ((uint64_t)8 << 20) : (serial_mode && total < ((uint64_t)8 << 20));
    if (tail.hit_member_end) {
        if (member_crc != tail.mend.crc) { err = "invalid gzip data: CRC-32 mismatch"; return false; }
        if ((uint32_t)member_out != tail.mend.isize) { err = "invalid gzip data: size mismatch"; return false; }
        in_member = false;
        member_out = 0;
        member_crc = 0;
        window.clear();
    } else if (tail.hit_eof) {
        finished = true;
        in_member = false;
    }
    return true;
}

ParallelGunzip::ParallelGunzip() : impl_(new Impl) {}
ParallelGunzip::~ParallelGunzip()
{
    if (impl_->bg_running) impl_->bg.join();
    for (OutBuf *b : impl_->bufs) delete b;
    free(impl_->text);
    free(impl_->cur);
    delete impl_;
}

void ParallelGunzip::init(FILE *f, int threads)
{
    impl_->f = f;
    impl_->threads = threads < 1 ? 1 : (threads > 64 ? 64 : threads);
    if (const char *e = getenv("VFB_PGUNZIP_SEGMENT")) impl_->seg_bytes = std::max<size_t>(4096, (size_t)strtoull(e, nullptr, 10));
}

namespace {
size_t copy_count(uint8_t *dst, const uint8_t *src, size_t n)
{
    memcpy(dst, src, n);
    size_t c = 0, i = 0;
    const uint64_t k = 0x0A0A0A0A0A0A0A0Aull, lo7 = 0x7F7F7F7F7F7F7F7Full;
    for (; i + 8 <= n; i += 8) {
        uint64_t w;
        memcpy(&w, dst + i, 8);
        const uint64_t x = w ^ k, nz = ((x & lo7) + lo7) | x;      // high bit of every non-'\n' byte
        c += (size_t)__builtin_popcountll(~nz & ~lo7);
    }
    for (; i < n; ++i) c += dst[i] == '\n';
    return c;
}
}  // namespace

long long ParallelGunzip::read(uint8_t *out, size_t cap, std::string *err) { return read_counting(out, cap, nullptr, err); }

long long ParallelGunzip::read_counting(uint8_t *out, size_t cap, size_t *newlines, std::string *err)
{
    Impl &m = *impl_;
    size_t produced = 0;
    if (newlines) *newlines = 0;
    while (produced < cap) {
        if (m.cur_pos == m.cur_len) {
            if (m.drained) break;
            if (!m.bg_running) {
                m.bg = std::thread([&m] { m.bg_ok = m.segment(); });
                m.bg_running = true;
            }
            m.bg.join();
            m.bg_running = false;
            if (!m.bg_ok) { *err = m.err; m.drained = true; return -1; }
            std::swap(m.cur, m.text);
            std::swap(m.cur_cap, m.text_cap);
            m.cur_len = m.text_len;
            m.cur_pos = 0;
            m.text_len = 0;
            if (m.finished) {
                if (m.cur_len == 0) { m.drained = true; break; }
                m.drained = true;                 // this is the last text; nothing left to decode
            } else {
                // decode the next segment while the caller consumes this one
                m.bg = std::thread([&m] { m.bg_ok = m.segment(); });
                m.bg_running = true;
            }
            if (m.cur_len == 0) { if (m.drained) break; continue; }
        }
        const size_t n = std::min(cap - produced, m.cur_len - m.cur_pos);
        if (!newlines) {
            memcpy(out + produced, m.cur + m.cur_pos, n);
        } else {
            // split over the threads (the background decode of the next segment shares the cores: fine)
            const size_t min_part = (size_t)2 << 20;
            int parts = (int)std::min<size_t>((size_t)m.threads, n / min_part);
            if (parts <= 1) {
                *newlines += copy_count(out + produced, m.cur + m.cur_pos, n);
            } else {
                std::vector<size_t> cnt((size_t)parts, 0);
                std::vector<std::thread> pool;
                const size_t per = n / (size_t)parts;
                auto run = [&](int t) {
                    const size_t lo = (size_t)t * per, hi = t + 1 == parts ? n : lo + per;
                    cnt[(size_t)t] = copy_count(out + produced + lo, m.cur + m.cur_pos + lo, hi - lo);
                };
                for (int t = 1; t < parts; ++t) pool.emplace_back(run, t);
                run(0);
                for (auto &th : pool) th.join();
                for (size_t c : cnt) *newlines += c;
            }
        }
        m.cur_pos += n;
        produced += n;
    }
    return (long long)produced;
}

void ParallelGunzip::stats(uint64_t *segments, uint64_t *workers_used, uint64_t *workers_dropped) const
{
    if (segments) *segments = impl_->n_segments;
    if (workers_used) *workers_used = impl_->n_workers_used;
    if (workers_dropped) *workers_dropped = impl_->n_workers_dropped;
}

}  // namespace vfb
